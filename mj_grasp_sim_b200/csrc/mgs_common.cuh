// mgs_common.cuh - types shared by the sm_100a kernels and the C-ABI glue.
//
// Execution model: ONE ENVIRONMENT PER WARP.  All per-environment state lives in that warp's
// slice of dynamic shared memory for the whole rollout (thousands of steps); HBM is touched only
// for the read-only model constants (L1/L2 resident, shared by every warp) and for the
// candidate inputs / labels at the two ends of the rollout.
//
// The device code is written against a tiny "lane" abstraction (PFOR / warp reductions).  With
// -DMGS_HOST the same source builds as a 1-lane scalar program; that build exists ONLY so the
// CPU-only test tier can check the kernel's arithmetic against the fp64 oracle before GPU time is
// spent.  It is compiled into tests/hostsim/, never into the product library, which has no CPU
// path at all.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#ifdef MGS_REAL_DOUBLE
typedef double real;
#define R_(x) x
#define REAL_EPS 2.2e-16
#else
typedef float real;
#define R_(x) x##f
#define REAL_EPS 1.2e-7f
#endif
#define MGS_MINVAL R_(1e-15)
// fp32 build: qpos carries a low-order companion word (qpos = hi + lo, integrated in double): with h = 1 ms a slow creep
// (|qvel| < ~1e-4) moves a coordinate by less than one fp32 ulp per step, so plain fp32 accumulation either stalls or rounds
// the creep to whole ulps - which is what decides marginal grasps over thousands of steps (DESIGN.md 5).
#if !defined(MGS_REAL_DOUBLE) && !defined(MGS_NO_QPOS_COMP)
#define MGS_QPOS_COMP 1
#define MGS_NQ_LO(nq) (nq)
#else
#define MGS_NQ_LO(nq) 0
#endif

#ifdef MGS_HOST
#define MGS_DEV static inline
#define MGS_DEVN static
#define LANES 1
#define MGS_LANE 0
#define WSYNC() ((void)0)
#define LDG(p) (*(p))
#define MGS_STAGE_BARRIER(k) ((void)0)
#elif defined(MGS_WIDE)
// ENVIRONMENT PER CTA ("wide" variant, -DMGS_WIDE=<threads>): the same device source with the lane abstraction widened to a
// whole thread block - every PFOR loop is strided over MGS_WIDE threads, WSYNC is a CTA barrier and the "warp" collectives
// (wsum, wany, wrank, ...) are block-level.  For scenes whose per-environment state fills most of an SM's shared memory
// (BASELINE configs[4]: Shadow hand + 10 objects, nv = 94, ~220 KB): with one warp per environment a single warp would run on
// the SM; here 8 warps share the environment's rows / pairs / matrix entries.  No stage barriers: there is nothing to align.
#include <cuda_runtime.h>
#define MGS_DEV __device__ __forceinline__
#define MGS_DEVN static __device__ __noinline__
#define LANES MGS_WIDE
#define MGS_LANE ((int)threadIdx.x)
#define WSYNC() __syncthreads()
#define LDG(p) __ldg(p)
#define MGS_STAGE_BARRIER(k) ((void)0)
#else
#include <cuda_runtime.h>
#define MGS_DEV __device__ __forceinline__
#define MGS_DEVN static __device__ __noinline__
#define LANES 32
#define MGS_LANE ((int)(threadIdx.x & 31))
#define WSYNC() __syncwarp()
#define LDG(p) __ldg(p)
// CTA-wide STAGE barrier.  The step is ~250 KB of SASS that every warp walks through once per step;
// with independent warps on an SM each sits in a different part of it and the instruction caches thrash
// (ncu r1_a / r1_c: "no instruction" = 12-17 of the 18-24 stall cycles per issue).  One CTA per SM whose
// warps enter every stage together share the fetches.  The barriers carry no data dependency (warps
// never touch each other's environment); they only align code position, and every warp executes the
// same number of them per step, whatever its contact count or solver path.  -DMGS_BAR_MASK=0 turns
// them off for A/B measurements.
// MGS_BAR_MASK selects which of the six per-step barriers are compiled in (bit k = barrier k):
// 0 step start, 1 before collision, 2 after collision, 3 after constraint assembly, 4 after Newton,
// 5 before integration.
#ifndef MGS_BAR_MASK
#define MGS_BAR_MASK 63
#endif
// (Taking the barriers only every K-th step was measured too: K=2 -3 %, K=4 -34 %, K=8 -47 %.)
#define MGS_STAGE_BARRIER(k) do { if ((MGS_BAR_MASK >> (k)) & 1) __syncthreads(); } while (0)
#endif

// Innermost multiply-accumulate loops: unrolled by MGS_INNER_UNROLL (the stage-level loops stay `#pragma unroll 1`
// to keep the instruction footprint small; at unroll 1 an inner MAC costs 2 loads + FMA + 3-4 loop-control
// instructions with a serial dependence - ncu r1_i: 20 % of stall samples were fixed-latency "wait").
#ifndef MGS_INNER_UNROLL
#define MGS_INNER_UNROLL 4
#endif
#define MGS_PRAGMA_(x) _Pragma(#x)
#define MGS_PRAGMA(x) MGS_PRAGMA_(x)
#define MGS_UNROLL_INNER MGS_PRAGMA(unroll MGS_INNER_UNROLL)

// lane-strided loop: on the GPU lane L handles i = L, L+32, ...; on the host build one lane does all
#define PFOR(i, n) for (int i = MGS_LANE; i < (n); i += LANES)

enum { JNT_FREE = 0, JNT_BALL = 1, JNT_SLIDE = 2, JNT_HINGE = 3 };
enum { GEOM_SPHERE = 2, GEOM_CAPSULE = 3, GEOM_CYLINDER = 5, GEOM_BOX = 6, GEOM_MESH = 7 };
enum { EQ_CONNECT = 0, EQ_WELD = 1, EQ_JOINT = 2 };
enum { CT_EQUALITY = 0, CT_FRICTION_DOF = 1, CT_LIMIT = 2, CT_CONTACT = 3 };
enum { ST_SATISFIED = 0, ST_QUADRATIC = 1, ST_LINEARNEG = 2, ST_LINEARPOS = 3, ST_CONE = 4 };
enum { MGS_MODE_STEP = 0, MGS_MODE_COLLISION = 1, MGS_MODE_STABILITY = 2, MGS_MODE_CLUTTER_COLLISION = 3, MGS_MODE_CLUTTER_STABLE = 4 };

// Model constants on the device (all pointers into one read-only blob).
struct DevModel {
  int nq, nv, nu, nbody, njnt, neq, nmocap, ntendon, nwrap, ncgeom, npair, nhull;
  int maxdepth, max_tree_dofs, nM, ntree, ne_rows, nf_rows, ngravcomp, dofmask_words, cone_elliptic, iterations, ls_iterations, noslip_iterations, mpr_iterations, ground_geomid;
  real timestep, impratio, tolerance, ls_tolerance, noslip_tolerance, mpr_tolerance, meaninertia, gravity[3];
  const int *body_parentid, *body_rootid, *body_mocapid, *body_jntadr, *body_jntnum, *body_dofadr, *body_dofnum, *body_depth;
  const real *body_pos, *body_quat, *body_ipos, *body_iquat, *body_mass, *body_inertia, *body_invweight0, *body_subtreemass, *body_gravcomp;
  const int *jnt_type, *jnt_bodyid, *jnt_qposadr, *jnt_dofadr, *jnt_limited;
  const real *jnt_pos, *jnt_axis, *jnt_range, *jnt_stiffness, *jnt_solref, *jnt_solimp, *jnt_margin, *qpos0, *qpos_spring;
  const int *dof_bodyid, *dof_jntid, *dof_parentid, *dof_treeadr, *dof_treenum;
  const real *dof_armature, *dof_damping, *dof_frictionloss, *dof_solref, *dof_solimp, *dof_invweight0;
  const int *cgeom_geomid, *cgeom_type, *cgeom_bodyid, *cgeom_hullid;
  const real *cgeom_pos, *cgeom_quat, *cgeom_size, *cgeom_rbound;
  const int *hull_vertadr, *hull_vertnum, *hull_faceadr, *hull_facenum, *hull_facevertadr, *hull_facevertnum, *hull_facevert;
  const int *hull_nbradr, *hull_nbrnum, *hull_nbr;
  const real *hull_vert, *hull_facenormal;
  const int *pair_geom1, *pair_geom2, *pair_condim;
  const real *pair_friction, *pair_solref, *pair_solimp, *pair_margin;
  const int *tendon_adr, *tendon_num, *wrap_dofadr, *wrap_qposadr;
  const real *wrap_coef;
  const int *actuator_trntype, *actuator_trnid, *actuator_ctrllimited, *actuator_forcelimited;
  const real *actuator_gainprm, *actuator_biasprm, *actuator_ctrlrange, *actuator_forcerange, *actuator_gear;
  const int *eq_type, *eq_obj1id, *eq_obj2id, *eq_active, *eq_rowadr, *tri_ab;
  const int *dof_frictionrank;       // [nv]: rank of dof d among the dofs with frictionloss > 0 (its row is ne_rows + rank), -1 if none
  // Block storage of the per-tree matrices (M, M^-1, the blocked uses of the H scratch): the block of a kinematic tree with t dofs
  // is a dense t x t row-major tile, tiles back to back (nM = sum t^2 words instead of nv^2).  Entry (i, j) of one tree lives at
  // dof_rowoff[i] + j; rows of one tree are dof_treenum apart.
  const int *dof_rowoff;             // [nv]
  const int *dof_blk;                // [nv]: dof_rowoff | dof_treeadr << 16 | dof_treenum << 24 (one load instead of three)
  const int *blk_ij;                 // [nM]: (i << 8) | j of every stored entry
  const int *dof_treeid, *body_treeid;  // kinematic tree index of a dof / of the dofs that move a body (-1: static body)
  const int *tri_madr;               // [nv (nv + 1) / 2], parallel to tri_ab: address of M(a, b), -1 when a and b are in different trees
  const unsigned int *body_dofmask;  // [nbody][dofmask_words]: bit d set = dof d is on the path from the body to its root
  const real *eq_data, *eq_solref, *eq_solimp;
  const real *mocap_pos0, *mocap_quat0;
};

// Per-environment scratch layout (offsets in `real` units into the warp's shared-memory slice).
// Three groups: PERSIST lives for the whole rollout; TRANSIENT (kinematics/collision/inertia/RNE
// temporaries) and SOLVER (constraint rows) are never live at the same time, so they OVERLAY each
// other - shared memory per environment is what bounds the number of resident warps per SM.
#define MGS_LAYOUT_PERSIST(X)                                                                                      \
  X(hdr, 8) X(qpos, nq) X(qpos_lo, MGS_NQ_LO(nq)) X(qvel, nv) X(qacc_ws, nv) X(ctrl, nu) X(mocap, 7 * nmocap)                                          \
  X(xpos, 3 * nbody) X(xquat, 4 * nbody) X(xmat, 9 * nbody) X(rootcom, 3 * nbody) X(cdof, 6 * nv)                  \
  X(M, nM) X(Minv, nM) X(H, nv * nv)                                                                     \
  X(ten_length, ntendon) X(ten_J, ntendon * nv) X(act_moment, nu * nv) X(act_force, nu) X(act_length, nu)          \
  X(qfrc_smooth, nv) X(qacc_smooth, nv) X(qacc, nv) X(qfrc_constraint, nv) X(Ma, nv) X(grad, nv) X(search, nv)     \
  X(Mv, nv) X(wvec, nv) X(con_pos, 3 * ncon_max) X(con_normal, 3 * ncon_max) X(con_dist, ncon_max)                 \
  X(con_mu, ncon_max) X(con_pair, ncon_max) X(con_efc, ncon_max) X(nsB, 3 * nv) X(nsS, lanes + (lanes > 32 ? 8 : 0)) X(mpr_cache, 4 * ncache)
#define MGS_LAYOUT_TRANSIENT(X)                                                                                    \
  X(xipos, 3 * nbody) X(ximat, 9 * nbody) X(xanchor, 3 * njnt) X(xaxis, 3 * njnt) X(gxpos, 3 * ncgeom)             \
  X(gxmat, 9 * ncgeom) X(cinert, 10 * nbody) X(crb, 10 * nbody) X(cdof_dot, 6 * nv) X(cvel, 6 * nbody)             \
  X(cacc, 6 * nbody) X(cfrc, 6 * nbody)
#define MGS_LAYOUT_SOLVER(X)                                                                                       \
  X(J, nefc_max * nv) X(efc_D, nefc_max) X(efc_R, nefc_max) X(efc_aref, nefc_max) X(efc_aux, nefc_max)             \
  X(efc_force, nefc_max) X(efc_jar, nefc_max) X(efc_jv, nefc_max) X(efc_tsi, nefc_max)                                       \
  X(efc_key, (lanes > 32 ? nefc_max : 0)) X(efc_list, (lanes > 32 ? nefc_max : 0))
#define MGS_LAYOUT_FIELDS(X) MGS_LAYOUT_PERSIST(X) MGS_LAYOUT_TRANSIENT(X) MGS_LAYOUT_SOLVER(X)

struct Layout {
#define X(name, cnt) int name;
  MGS_LAYOUT_FIELDS(X)
#undef X
  int total, ncon_max, nefc_max, ncache;
  int req_off;          // env-per-CTA variant: request / answer records of the face search (6 words per thread), behind the clipping slots
  int clip_off, nclip;  // face-clipping scratch: `nclip` slots of MGS_CLIP_STRIDE reals in the part of the SOLVER overlay that lies beyond the
                        // TRANSIENT arrays (free during collision: the constraint rows are built afterwards)
};

// one clipping slot: reference polygon (8 x 3), two ping-pong polygons (12 x 3 each), depths (12); odd stride = no bank conflicts
#define MGS_CLIP_STRIDE 109
#define MGS_MPR_CACHE_MAX 128  // geom pairs (the first ones of the list: the object pairs) whose last MPR result is remembered:
                               // 4 words per pair - portal vertex pairs or separating axis (words 0-2), hill-climb start vertices (3)
// `lanes`: threads that share one environment (32 for the warp-per-environment variants, MGS_WIDE for the env-per-CTA one)
static inline void layout_compute(Layout *L, int nq, int nv, int nu, int nbody, int njnt, int nmocap, int ntendon, int ncgeom,
                                  int ncon_max, int nefc_max, int npair, int nM, int lanes = 32, int ncache_max = MGS_MPR_CACHE_MAX) {
  int off = 0;
  const int ncache = npair < ncache_max ? npair : ncache_max;  // the pairs beyond it keep their warm start in the global (L2) cache
  L->ncache = ncache;
  // arrays are packed back to back (no vector loads anywhere: word alignment is enough); padding every array to 16 bytes cost
  // ~270 bytes per environment, which is the difference between 10 and 9 resident Robotiq environments per SM
#define X(name, cnt) L->name = off; off += (cnt);
  MGS_LAYOUT_PERSIST(X)
  const int overlay = off;
  MGS_LAYOUT_TRANSIENT(X)
  const int end_t = off;
  off = overlay;
  MGS_LAYOUT_SOLVER(X)
#undef X
  L->total = off > end_t ? off : end_t;
  L->clip_off = end_t;
  L->nclip = (L->total - end_t) / MGS_CLIP_STRIDE;
  if (L->nclip < 1) { L->nclip = 1; L->total = end_t + MGS_CLIP_STRIDE; }
  if (L->nclip > 32) L->nclip = 32;
  L->req_off = L->clip_off + L->nclip * MGS_CLIP_STRIDE;
  if (lanes > 32 && L->total < L->req_off + 6 * lanes) L->total = L->req_off + 6 * lanes;
  L->total = (L->total + 3) & ~3;  // every environment's slice starts 16-byte aligned
  L->ncon_max = ncon_max;
  L->nefc_max = nefc_max;
}

// Rollout parameters (reference: gravityless_object_grasping.py:127-137 defaults and the
// per-gripper close_gripper_at control vectors).
#define MGS_MAX_NU 24
#define MGS_MAX_NJ 24
struct RolloutParams {
  int mode, n, nj, base_qposadr, nstep, nstep_close, nstep_lift, shake_steps, repose_on_close;
  real lift_dist, shake_dist;
  real qvel_clip;  // MGS_MODE_STEP only: clamp qvel to +-qvel_clip before every step (0 = off); clutter_table.py:215-221
  int joint_qposadr[MGS_MAX_NJ];
  real close_ctrl[MGS_MAX_NU];
};

// Per-call device I/O.  All arrays are env-major (one contiguous record per environment): with one
// warp per environment that is the coalesced layout - lane k reads element k of its env's record.
struct BatchIO {
  const float *pose7;   // [n][7]  processed base pose (pos, quat wxyz), fp32 like SE3Pose
  const float *joints;  // [n][nj]
  uint8_t *labels;      // [n]
  int *steps;           // [n] env-steps executed
  // generic state in/out (MGS_MODE_STEP and diagnostics): [n][state_stride]
  // record = qpos(nq) qvel(nv) qacc_ws(nv) ctrl(nu) mocap(7*nmocap)
  const real *state_in;
  real *state_out;
  real *diag_out;  // optional [n][diag_stride]: ncon, nefc, niter, then contacts/qacc (tests)
  float *aux;      // optional [n][4]: flags (bit 0 capacity overflow, bit 1 state blew up), object drift over the close phase
                   // (position [m], rotation [deg]; gravityless_object_grasping.py:175-200), reserved
  int state_stride, diag_stride;
  unsigned int *work_counter;
  // per-pair MPR cache of the pairs beyond the shared-memory one (4 words per pair, one slab of npair pairs per environment slot of the
  // persistent grid; L2 resident) - null for models whose pairs all fit the shared-memory cache
  int *mpr_cache_g;
  // environment-per-CTA variant with the state in global memory (csrc/mgs_kernel_wide_g.cu): one Layout.total slice per CTA of the
  // persistent grid - null for the variants that keep it in shared memory.  Last member: the constant-bank offsets of the fields
  // above stay where they were.
  real *env_state;
  // Clutter modes over several scenes of one model (appended after env_state for the same reason).  Candidate i starts from the
  // record state_in + scene_index[i] * state_stride; null = every candidate starts from scene 0 (nscene is then not read, so a
  // zero-filled BatchIO behaves as before these members existed).  An index outside [0, nscene) gets label 0 and aux bit 1 without
  // any read at that index.
  const int *scene_index;  // [n]
  int nscene;
  // Device enough_stable early stop: non-overflowed successes per scene, counted during the launch; a candidate whose scene already
  // counts >= enough_stable when it is pulled is not simulated (label 0, aux bit 2).  Null = no early stop.
  unsigned int *scene_success;  // [nscene]
  int enough_stable;
};
