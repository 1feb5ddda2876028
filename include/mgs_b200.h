/* mgs_b200.h - C ABI of libmgs_b200.so, the B200-native replacement for the grasp-evaluation
 * rollout hot path of freiberg-roman/mj-grasp-sim.
 *
 * What each entry point replaces in the reference (paths under /root/reference):
 *   mgs_model_create          MjModel.from_xml_string + MjData  (mgs/env/gravityless_object_grasping.py:67-70)
 *                             - the MJCF itself is compiled on the host (mj_grasp_sim_b200/compiler);
 *                             this call uploads the flat result to the GPU.
 *   mgs_grasp_collision_mask  the per-candidate loop of GravitylessObjectGrasping.grasp_collision_mask
 *                             (mgs/env/gravityless_object_grasping.py:112-122: mj_resetData, set_qpos, set_pose,
 *                             mj_forward, ncon != 0)
 *   mgs_grasp_stability       the per-candidate loop of grasp_stability_evaluation_from_joints
 *                             (mgs/env/gravityless_object_grasping.py:158-277) including close_gripper_at
 *                             (mgs/gripper/panda.py:225-241 and siblings): up to 8000 mj_step per candidate
 *   mgs_step_*                mujoco.mj_step(model, data, nstep) / mj_forward on a batch of explicit states
 *                             (mgs/core/simualtion.py:45-61 state get/set + mj_step) - used by parity tests
 *
 * Conventions: every function returns 0 on success, <0 on error (message via mgs_last_error(),
 * thread-local).  No torch types; plain pointers and sizes.  "_device" variants take CUDA device
 * pointers (e.g. torch tensor .data_ptr()) and a cudaStream_t passed as void*; the plain variants
 * take host pointers and perform the host<->device copies themselves (pinned staging).
 * Buffers are owned by the caller; the model handle owns only the model constants and scratch.
 * One host thread per model handle at a time; different handles may be driven from different threads (launches are
 * serialised internally).  There is no CPU fallback: without a CUDA device every call
 * fails with an error.
 */
#ifndef MGS_B200_H
#define MGS_B200_H
#include <stdint.h>

#include "mgs_model_desc.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct MgsModel MgsModel;

/* rollout schedule: defaults of grasp_stability_evaluation_from_joints (:131-135) are
 * {3000, 3000, 500, 0, 0.1, 0.02}; repose_on_close=1 for Allegro/LEAP (their close_gripper_at
 * calls set_pose again, allegro.py:354-357). */
typedef struct MgsRolloutCfg {
  int nstep_close, nstep_lift, shake_steps, repose_on_close;
  double lift_dist, shake_dist;
} MgsRolloutCfg;

typedef struct MgsModelInfo {
  int nq, nv, nu, nmocap, state_stride, diag_stride, ncon_max, nefc_max,
      smem_bytes_per_env, /* size of one environment's state: shared memory, or global memory when mgs_model_state_in_global() is 1 */
      warps_per_block, /* environments per CTA */
      blocks_per_sm, num_sms, real_bytes,
      lanes_per_env; /* threads that share one environment: 32 (warp per environment) or 256 (environment per CTA) */
} MgsModelInfo;

int mgs_model_create(const MgsModelDesc *desc, int device, MgsModel **out);
/* Same, with explicit per-environment capacities (0 = default: 32-64 contacts depending on the number of object
 * pairs - 32 for models with more than 24 dofs - and static rows + 4 rows per contact slot).  Shared memory per environment - and so the number of environments resident per SM - follows
 * from them.  Contacts beyond capacity are dropped and counted in the diagnostics' overflow field. */
int mgs_model_create_ex(const MgsModelDesc *desc, int device, int ncon_max, int nefc_max, MgsModel **out);
/* Same as mgs_model_create_ex (same kernel selection, same capacities), except that a model whose environment state does not fit one
 * CTA's shared memory - where _ex fails - is created on the environment-per-CTA variant with the state in a global-memory slab
 * (one slice per CTA of the persistent grid, allocated here, freed by mgs_model_destroy).  mgs_model_create / _ex keep failing
 * there, so a caller can still probe for the largest capacity that fits shared memory. */
int mgs_model_create_any(const MgsModelDesc *desc, int device, int ncon_max, int nefc_max, MgsModel **out);
/* 1: the model's environment state lives in global memory (variant wide_g), 0: in shared memory, <0: error */
int mgs_model_state_in_global(const MgsModel *model);
void mgs_model_destroy(MgsModel *model);
int mgs_model_info(const MgsModel *model, MgsModelInfo *info);

/* pose7: [n][7] processed base pose (pos xyz, quat wxyz) in float32 exactly as SE3Pose holds it;
 * joints: [n][nj] float32; joint_qposadr: [nj] qpos addresses of the actuated joints
 * (MjSimulation.get_joint_idxs); base_qposadr: qpos address of the gripper's free joint. */
int mgs_grasp_collision_mask(MgsModel *model, int n, const float *pose7, const float *joints, int nj,
                             const int *joint_qposadr, int base_qposadr, uint8_t *collision_free_out);
int mgs_grasp_stability(MgsModel *model, int n, const float *pose7, const float *joints, int nj,
                        const int *joint_qposadr, int base_qposadr, const double *close_ctrl,
                        const MgsRolloutCfg *cfg, uint8_t *stable_out, int *steps_out);
/* mode: 1 = collision mask, 2 = stability.  d_* are device pointers; steps may be NULL. */
int mgs_rollout_device(MgsModel *model, int mode, int n, const float *d_pose7, const float *d_joints, int nj,
                       const int *joint_qposadr, int base_qposadr, const double *close_ctrl,
                       const MgsRolloutCfg *cfg, uint8_t *d_labels, int *d_steps, void *stream);

/* Clutter table (reference: mgs/env/clutter_table.py).  `scene` is the settled scene every candidate starts
 * from - what the reference restores with mj_setState(..., mjSTATE_INTEGRATION) at the top of each iteration
 * (:291, :356) - as one state record of MgsModelInfo.state_stride values:
 * qpos[nq] qvel[nv] qacc_warmstart[nv] ctrl[nu] mocap_pos[3] mocap_quat[4].
 *   mgs_clutter_collision_mask  the loop body of ClutterTableEnv.grasp_collision_mask (:356-364); the workspace
 *                               bounds test on the unprocessed pose (:344-354) stays on the host
 *   mgs_clutter_stable_mask     the loop body of ClutterTableEnv.grasp_stable_mask (:288-317): close nstep_close,
 *                               lift lift_dist over nstep_lift with check_gripper_contact every 100 steps
 *                               (cfg.shake_* are ignored)
 * The model's ground_geomid must be the id of "geom:table". */
int mgs_clutter_collision_mask(MgsModel *model, int n, const double *scene, const float *pose7, const float *joints, int nj,
                               const int *joint_qposadr, int base_qposadr, uint8_t *collision_free_out);
int mgs_clutter_stable_mask(MgsModel *model, int n, const double *scene, const float *pose7, const float *joints, int nj,
                            const int *joint_qposadr, int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg,
                            uint8_t *stable_out, int *steps_out);
/* device-pointer variant: mode 3 = clutter collision mask, 4 = clutter stable mask; d_scene holds the record
 * in the library's compute type (float, or double in the ablation build) */
int mgs_clutter_device(MgsModel *model, int mode, int n, const void *d_scene, const float *d_pose7, const float *d_joints, int nj,
                       const int *joint_qposadr, int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg,
                       uint8_t *d_labels, int *d_steps, void *stream);

/* Many scenes of one model in one launch.  `scenes` holds nscene state records back to back ([nscene][state_stride]); candidate i
 * starts from scene scene_index[i].  The plain variants reject an index outside [0, nscene); the device variant cannot check on the
 * host, so such a candidate gets label 0, 0 steps and aux flag bit 1, and nothing is read at that index.  d_scene_index may be NULL
 * (every candidate uses scene 0).  mgs_clutter_device is the nscene = 1, no-index, no-early-stop case of the same launch.
 *
 * enough_stable > 0 switches on the early stop of the reference's loop per scene (ClutterTableEnv.grasp_stable_mask, :293-296): the
 * launch counts, per scene, the candidates that finished with label 1 and no capacity overflow; a candidate whose scene already
 * counts >= enough_stable when it is pulled from the work queue is not simulated (label 0, 0 steps, aux flag bit 2).  Candidates are
 * pulled in index order, so when each scene's candidates are in that scene's sequential order, a skipped candidate is one the
 * sequential loop labels False; the others get their true label.  The caller still applies the prefix rule per scene (after
 * re-running overflowed candidates at larger capacities): candidates after a scene's enough_stable-th success that were not
 * skipped - they were in flight when the count was reached - keep their true label here.  Ordering candidates round-robin across
 * scenes keeps that waste small.  The counters belong to the model (zeroed on the launch stream before every launch). */
int mgs_clutter_scenes_collision_mask(MgsModel *model, int n, int nscene, const double *scenes, const int *scene_index,
                                      const float *pose7, const float *joints, int nj, const int *joint_qposadr, int base_qposadr,
                                      uint8_t *collision_free_out);
int mgs_clutter_scenes_stable_mask(MgsModel *model, int n, int nscene, const double *scenes, const int *scene_index, const float *pose7,
                                   const float *joints, int nj, const int *joint_qposadr, int base_qposadr, int enough_stable,
                                   const double *close_ctrl, const MgsRolloutCfg *cfg, uint8_t *stable_out, int *steps_out);
int mgs_clutter_scenes_device(MgsModel *model, int mode, int n, int nscene, const void *d_scenes, const int *d_scene_index,
                              int enough_stable, const float *d_pose7, const float *d_joints, int nj, const int *joint_qposadr,
                              int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg, uint8_t *d_labels, int *d_steps,
                              void *stream);

/* Batched mj_step on explicit states.  State record (state_stride reals, env-major):
 * qpos[nq] qvel[nv] qacc_warmstart[nv] ctrl[nu] mocap_pos[3] mocap_quat[4].  nstep = 0 runs
 * mj_forward only.  diag (may be NULL) receives diag_stride reals per env: header
 * {ncon, nefc, niter, bad, overflow, ne, nf, nl}, qacc, qacc_smooth, qfrc_smooth, M, xpos, xquat,
 * contacts {dist,pos3,pair} x ncon_max, rows {aref,D,force,jar} x nefc_max.  Reals are float
 * (double in the -DMGS_REAL_DOUBLE ablation build; see MgsModelInfo.real_bytes). */
int mgs_step_host(MgsModel *model, int n, int nstep, const void *state_in, void *state_out, void *diag_out);
int mgs_step_device(MgsModel *model, int n, int nstep, const void *d_state_in, void *d_state_out, void *d_diag_out,
                    void *stream);

/* environments of the most recent launch on this model that dropped contacts for lack of capacity
 * (synchronises the device); re-run with larger capacities if non-zero and exactness matters */
int mgs_overflow_count(MgsModel *model);

/* Per-candidate auxiliary results of the most recent launch on this model (synchronises the device): 4 floats per candidate -
 * [0] flags: bit 0 = the environment dropped contacts / constraint rows for lack of capacity (its label was computed on a
 *     truncated contact set: re-run it on a model created with larger capacities), bit 1 = the state blew up, or (clutter
 *     scenes) the candidate's scene index was out of range (label False), bit 2 = skipped by the enough_stable early stop of
 *     mgs_clutter_scenes_* (not simulated: its scene already had enough stable grasps; label False);
 * [1], [2] stability rollouts: displacement [m] and rotation [deg] of the grasped object over the close phase - what the
 *     reference computes as positional / rotational drift (mgs/env/gravityless_object_grasping.py:175-200) - NaN when the
 *     candidate lost contact before that point; [3] reserved (0). */
int mgs_last_aux(MgsModel *model, int n, float *aux_out);

/* mgs_step_*: clamp qvel to [-clip, clip] before every step (ClutterTableEnv.gen_clutter does that around each mj_step,
 * mgs/env/clutter_table.py:215-221); 0 switches it off (default) */
int mgs_set_qvel_clip(MgsModel *model, double clip);

/* identifies the sources this library was built from (sha256 prefix of csrc/ + include/, set by lib.build()) */
const char *mgs_build_stamp(void);

/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
long long mgs_launch_count(void);
const char *mgs_last_error(void);

/* Ray casting of the antipodal grasp sampler (replaces the per-point trimesh ray queries of
 * /root/reference/mgs/sampler/antipodal.py:115-151).  For every point i: rays from p1[i] along +dirs[i] and -dirs[i] against the
 * nface triangles tri[nface][3][3] (host arrays, float64); hits closer than eps are dropped; of the nvalid_out[i] remaining hits
 * (ordered: +dir faces 0..nface-1, then -dir faces) number floor(pick_u[i] * nvalid) is chosen and its signed distance along dirs[i]
 * is written to signed_t_out[i] (NaN when there is no valid hit).  One warp per point, triangles staged through shared memory. */
int mgs_antipodal_hits(int device, int n, const double *p1, const double *dirs, int nface, const double *tri, double eps,
                       const double *pick_u, double *signed_t_out, int *nvalid_out);

#ifdef __cplusplus
}
#endif
#endif
