// mgs_sim.cuh - warp-per-environment rigid-body step (sm_100a device code).
//
// Replaces, for the batched rollout, what the reference gets from mujoco.mj_step / mj_forward
// (/root/reference/mgs/gripper/panda.py:241, /root/reference/mgs/env/gravityless_object_grasping.py
// :159-165,214,244,258,273).  Stage list per step (SURVEY.md 8(a-MJ)):
//   kinematics -> CoM frames/CRBA mass matrix -> M^-1 -> broadphase+narrowphase (MPR + face
//   clipping, lane per geom pair) -> constraint rows (weld/connect/joint equality, dof friction,
//   limits, elliptic contacts) -> smooth forces (RNE bias, passive, actuators) -> primal Newton with
//   exact line search (warp-cooperative dense Cholesky in shared memory) -> noslip -> implicitfast.
// Lanes split the work inside one environment (dofs, bodies of one tree level, constraint rows,
// geom pairs); warp shuffles do the reductions.  No global-memory traffic for state inside a step.
#pragma once
#include "mgs_common.cuh"

// ---------------------------------------------------------------------------------- warp helpers
#ifdef MGS_HOST
MGS_DEV real wsum(real x) { return x; }
MGS_DEV int wsumi(int x) { return x; }
MGS_DEV int wany(int p) { return p; }
MGS_DEV int wscan_excl(int x, int *total) { *total = x; return 0; }
MGS_DEV real wbcast(real x, int src) { (void)src; return x; }
MGS_DEV int wbcasti(int x, int src) { (void)src; return x; }
MGS_DEV void wargmax(real &v, int &idx) { (void)v; (void)idx; }
MGS_DEV int wrank(int p, int *total) { *total = p ? 1 : 0; return 0; }
MGS_DEV int wfirst(int p) { return p ? 0 : -1; }
MGS_DEV void wsum3(real &a, real &b, real &c) { (void)a; (void)b; (void)c; }
#elif defined(MGS_WIDE)
// block-level versions (environment per CTA).  Every collective is called by ALL threads of the CTA from converged code, like
// the full-mask warp intrinsics of the warp variant; results are identical on every thread and do not depend on timing
// (partial results are combined in warp order).  The trailing barrier of each lets the scratch be reused by the next call.
#define MGS_NWARP (MGS_WIDE / 32)
static __shared__ real mgs_cta_r[3 * MGS_NWARP];
static __shared__ int mgs_cta_i[MGS_NWARP];
// three sums with the two barriers of one
MGS_DEV void wsum3(real &a, real &b, real &c) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); c += __shfl_xor_sync(0xffffffffu, c, o);
  }
  if ((threadIdx.x & 31) == 0) { mgs_cta_r[threadIdx.x >> 5] = a; mgs_cta_r[MGS_NWARP + (threadIdx.x >> 5)] = b; mgs_cta_r[2 * MGS_NWARP + (threadIdx.x >> 5)] = c; }
  __syncthreads();
  a = mgs_cta_r[0]; b = mgs_cta_r[MGS_NWARP]; c = mgs_cta_r[2 * MGS_NWARP];
#pragma unroll
  for (int w = 1; w < MGS_NWARP; w++) { a += mgs_cta_r[w]; b += mgs_cta_r[MGS_NWARP + w]; c += mgs_cta_r[2 * MGS_NWARP + w]; }
  __syncthreads();
}
MGS_DEV real wsum(real x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  if ((threadIdx.x & 31) == 0) mgs_cta_r[threadIdx.x >> 5] = x;
  __syncthreads();
  real s = mgs_cta_r[0];
#pragma unroll
  for (int w = 1; w < MGS_NWARP; w++) s += mgs_cta_r[w];
  __syncthreads();
  return s;
}
MGS_DEV int wsumi(int x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  if ((threadIdx.x & 31) == 0) mgs_cta_i[threadIdx.x >> 5] = x;
  __syncthreads();
  int s = mgs_cta_i[0];
#pragma unroll
  for (int w = 1; w < MGS_NWARP; w++) s += mgs_cta_i[w];
  __syncthreads();
  return s;
}
MGS_DEV int wany(int p) { return __syncthreads_or(p); }
MGS_DEV real wbcast(real x, int src) {
  if ((int)threadIdx.x == src) mgs_cta_r[0] = x;
  __syncthreads();
  const real r = mgs_cta_r[0];
  __syncthreads();
  return r;
}
MGS_DEV int wbcasti(int x, int src) {
  if ((int)threadIdx.x == src) mgs_cta_i[0] = x;
  __syncthreads();
  const int r = mgs_cta_i[0];
  __syncthreads();
  return r;
}
// number of threads below this one with `p` set (and the CTA total)
MGS_DEV int wrank(int p, int *total) {
  const unsigned m = __ballot_sync(0xffffffffu, p);
  if ((threadIdx.x & 31) == 0) mgs_cta_i[threadIdx.x >> 5] = __popc(m);
  __syncthreads();
  int below = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < MGS_NWARP; w++) { const int c = mgs_cta_i[w]; if (w < (int)(threadIdx.x >> 5)) below += c; tot += c; }
  __syncthreads();
  *total = tot;
  return below + __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
}
// smallest thread index with `p` set, -1 if none
MGS_DEV int wfirst(int p) {
  const unsigned m = __ballot_sync(0xffffffffu, p);
  if ((threadIdx.x & 31) == 0) mgs_cta_i[threadIdx.x >> 5] = m ? (int)(threadIdx.x & ~31u) + __ffs(m) - 1 : 0x7fffffff;
  __syncthreads();
  int f = mgs_cta_i[0];
#pragma unroll
  for (int w = 1; w < MGS_NWARP; w++) f = min(f, mgs_cta_i[w]);
  __syncthreads();
  return f == 0x7fffffff ? -1 : f;
}
// arg-max over the CTA; ties go to the smaller index
MGS_DEV void wargmax(real &v, int &idx) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const real v2 = __shfl_xor_sync(0xffffffffu, v, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
    if (v2 > v || (v2 == v && i2 < idx)) { v = v2; idx = i2; }
  }
  if ((threadIdx.x & 31) == 0) { mgs_cta_r[threadIdx.x >> 5] = v; mgs_cta_i[threadIdx.x >> 5] = idx; }
  __syncthreads();
  v = mgs_cta_r[0]; idx = mgs_cta_i[0];
#pragma unroll
  for (int w = 1; w < MGS_NWARP; w++) {
    const real v2 = mgs_cta_r[w];
    const int i2 = mgs_cta_i[w];
    if (v2 > v || (v2 == v && i2 < idx)) { v = v2; idx = i2; }
  }
  __syncthreads();
}
MGS_DEV int wscan_excl(int x, int *total) {
  const int lane = threadIdx.x & 31;
  int v = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  if (lane == 31) mgs_cta_i[threadIdx.x >> 5] = v;
  __syncthreads();
  int below = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < MGS_NWARP; w++) { const int c = mgs_cta_i[w]; if (w < (int)(threadIdx.x >> 5)) below += c; tot += c; }
  __syncthreads();
  *total = tot;
  return below + v - x;
}
#else
MGS_DEV real wsum(real x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}
MGS_DEV int wsumi(int x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}
MGS_DEV int wany(int p) { return __any_sync(0xffffffffu, p); }
MGS_DEV int wfirst(int p) { return __ffs(__ballot_sync(0xffffffffu, p)) - 1; }
MGS_DEV void wsum3(real &a, real &b, real &c) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); c += __shfl_xor_sync(0xffffffffu, c, o);
  }
}
MGS_DEV real wbcast(real x, int src) { return __shfl_sync(0xffffffffu, x, src); }
MGS_DEV int wbcasti(int x, int src) { return __shfl_sync(0xffffffffu, x, src); }
// number of lanes below this one with `p` set (and the warp total)
MGS_DEV int wrank(int p, int *total) {
  const unsigned m = __ballot_sync(0xffffffffu, p);
  *total = __popc(m);
  return __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
}
// warp arg-max; ties go to the smaller index (= the first maximum of a sequential scan)
MGS_DEV void wargmax(real &v, int &idx) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const real v2 = __shfl_xor_sync(0xffffffffu, v, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
    if (v2 > v || (v2 == v && i2 < idx)) { v = v2; idx = i2; }
  }
}
MGS_DEV int wscan_excl(int x, int *total) {
  int lane = MGS_LANE, v = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  *total = __shfl_sync(0xffffffffu, v, 31);
  return v - x;
}
#endif

// ---------------------------------------------------------------------------------- small math
MGS_DEV real rsqrt_(real x) { return R_(1.0) / sqrt(x); }
MGS_DEV real dot3(const real *a, const real *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
MGS_DEV void cross3(real *r, const real *a, const real *b) {
  real x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
MGS_DEV void copy3(real *r, const real *a) { r[0] = a[0]; r[1] = a[1]; r[2] = a[2]; }
MGS_DEV void add3(real *r, const real *a, const real *b) { r[0] = a[0] + b[0]; r[1] = a[1] + b[1]; r[2] = a[2] + b[2]; }
MGS_DEV void sub3(real *r, const real *a, const real *b) { r[0] = a[0] - b[0]; r[1] = a[1] - b[1]; r[2] = a[2] - b[2]; }
MGS_DEV void scl3(real *r, const real *a, real s) { r[0] = a[0] * s; r[1] = a[1] * s; r[2] = a[2] * s; }
MGS_DEV void addscl3(real *r, const real *a, real s) { r[0] += a[0] * s; r[1] += a[1] * s; r[2] += a[2] * s; }
MGS_DEV real normalize3(real *a) {
  real n = sqrt(dot3(a, a));
  if (n < MGS_MINVAL) { a[0] = 1; a[1] = 0; a[2] = 0; return 0; }
  real i = R_(1.0) / n;
  a[0] *= i; a[1] *= i; a[2] *= i;
  return n;
}
MGS_DEV void mulquat(real *r, const real *a, const real *b) {
  real w = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  real x = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  real y = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  real z = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = w; r[1] = x; r[2] = y; r[3] = z;
}
MGS_DEV void normquat(real *q) {
  real n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < MGS_MINVAL) { q[0] = 1; q[1] = q[2] = q[3] = 0; return; }
  real i = R_(1.0) / n;
  q[0] *= i; q[1] *= i; q[2] *= i; q[3] *= i;
}
MGS_DEV void quat2mat(real *R, const real *q) {
  real w = q[0], x = q[1], y = q[2], z = q[3];
  R[0] = w * w + x * x - y * y - z * z; R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
  R[3] = 2 * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = 2 * (y * z - w * x);
  R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
}
MGS_DEV void mulmatvec3(real *r, const real *R, const real *v) {
  real x = R[0] * v[0] + R[1] * v[1] + R[2] * v[2], y = R[3] * v[0] + R[4] * v[1] + R[5] * v[2],
       z = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
MGS_DEV void mulmatTvec3(real *r, const real *R, const real *v) {
  real x = R[0] * v[0] + R[3] * v[1] + R[6] * v[2], y = R[1] * v[0] + R[4] * v[1] + R[7] * v[2],
       z = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
MGS_DEV void ld3(real *r, const real *g) { r[0] = LDG(g); r[1] = LDG(g + 1); r[2] = LDG(g + 2); }
MGS_DEV void ld4(real *r, const real *g) { r[0] = LDG(g); r[1] = LDG(g + 1); r[2] = LDG(g + 2); r[3] = LDG(g + 3); }

// ---------------------------------------------------------------------------------- environment
// Model constants, the scratch layout, the rollout parameters and the I/O pointers live in
// __constant__ memory (uniform loads through the constant cache; nothing is copied to the stack when
// the non-inlined stage functions are called).
struct KernelConsts { DevModel m; Layout L; RolloutParams prm; BatchIO io; };
#ifdef MGS_HOST
static KernelConsts g_k;
#define MGS_K g_k
#else
static __constant__ KernelConsts c_k;  // one copy per kernel variant (translation unit)
#define MGS_K c_k
#endif
#define MD (MGS_K.m)
#define LY (MGS_K.L)
#define PRM (MGS_K.prm)
#define IO (MGS_K.io)
// per-environment scratch arrays: slice base + constant offset.  On the device the slice base is recomputed
// from the warp index (two integer instructions) instead of being read from `Env`: the Env object is passed by
// reference to the non-inlined stage functions, so every field access was a local-memory load (ncu r1_h:
// ~1900 LDL per env-step).  The per-environment counters live in the slice itself (`hdr`), i.e. in shared
// memory; every lane writes the same value, so no lane ever reads a counter it has not written itself or that
// was not published by a WSYNC.
struct EnvHdr { int ncon, nefc, ne, nf, nl, niter, bad, overflow; };
struct Env { real *base; };
#ifdef MGS_HOST
#define EBASE (e.base)
#else
extern __shared__ __align__(16) unsigned char mgs_smem_raw[];
#if defined(MGS_WIDE) && defined(MGS_ENV_GLOBAL)
// environment per CTA with the slice in a global-memory slab (one slice per CTA of the persistent grid, BatchIO.env_state): scenes
// whose state does not fit one CTA's shared memory.  Every access to the slice is a plain (coherent) load or store - nothing reads it
// through LDG / __ldg - and WSYNC = __syncthreads() orders global memory within the CTA as it does shared memory, so no fence is needed.
#define EBASE (IO.env_state + (size_t)blockIdx.x * LY.total)
#define MGS_ENV_SLOT ((int)blockIdx.x)
#elif defined(MGS_WIDE)
#define EBASE (reinterpret_cast<real *>(mgs_smem_raw))
#define MGS_ENV_SLOT ((int)blockIdx.x)  // index of this environment slot in the persistent grid
#else
#define EBASE (reinterpret_cast<real *>(mgs_smem_raw) + (size_t)(threadIdx.x >> 5) * LY.total)
#define MGS_ENV_SLOT ((int)(blockIdx.x * MGS_MAX_WARPS_PER_BLOCK + (threadIdx.x >> 5)))
#endif
#endif
#define EF(name) (EBASE + LY.name)
#define EH (*reinterpret_cast<EnvHdr *>(EF(hdr)))
MGS_DEV void env_bind(Env &e, real *base) {
  e.base = base;
  EH.ncon = EH.nefc = EH.ne = EH.nf = EH.nl = EH.niter = EH.bad = EH.overflow = 0;
  WSYNC();
}
#define IARR(p) ((int *)(p))
// -DMGS_STAGE_CLOCKS (profiling builds only): cycles per stage of the step, accumulated by thread 0 of each CTA and printed for
// environment 0 at the end of its rollout (tools/README.md).  MGS_CLK(k) closes the interval that belongs to stage k.
#if defined(MGS_STAGE_CLOCKS) && !defined(MGS_HOST)
#include <stdio.h>
static __shared__ long long mgs_clk_acc[16];
static __shared__ long long mgs_clk_last;
#define MGS_CLK(k) do { if (threadIdx.x == 0) { const long long t_ = clock64(); mgs_clk_acc[k] += t_ - mgs_clk_last; mgs_clk_last = t_; } } while (0)
#define MGS_CLK_RESET() do { if (threadIdx.x == 0) { for (int q_ = 0; q_ < 16; q_++) mgs_clk_acc[q_] = 0; mgs_clk_last = clock64(); } } while (0)
#define MGS_CLK_PRINT(env, steps) do { if (threadIdx.x == 0 && (env) == 0) { printf("stage cycles per step (env 0, %d steps):", (steps)); \
  for (int q_ = 0; q_ < 12; q_++) printf(" [%d] %lld", q_, mgs_clk_acc[q_] / ((steps) > 0 ? (steps) : 1)); printf("\n"); } } while (0)
#else
#define MGS_CLK(k) ((void)0)
#define MGS_CLK_RESET() ((void)0)
#define MGS_CLK_PRINT(env, steps) ((void)0)
#endif
#ifdef MGS_QPOS_COMP
#define QPOS_LO_CLEAR(i) (EF(qpos_lo)[i] = 0)
#else
#define QPOS_LO_CLEAR(i) ((void)0)
#endif

// ---------------------------------------------------------------------------------- dense linear algebra (warp)
// `blocked` != 0: the matrix is block diagonal with one block per kinematic tree (the mass matrix M and the implicit-integration
// matrix M - h dF/dv) and is STORED as such (DevModel.dof_rowoff: a t x t tile per tree, nM words in all).  Lane i works on row i
// of ITS tree's block, all blocks advance one column per step together, so the number of column steps is the largest tree, not nv.
// `blocked` == 0: dense n x n row-major (the Newton Hessian).  Both cases address through (ro, s): entry (i, k) of lane i's own row
// is A[ro + k], entry (k, j) of another row of the same tile / matrix is A[ro + (k - i) * s + j].
// In-place lower Cholesky (only the lower triangle is read).
// (row offset, first dof, number of dofs) of dof i's tree tile: one packed word
MGS_DEV void blk_row(int i, int &ro, int &lo, int &tn) {
  const unsigned w = (unsigned)LDG(MD.dof_blk + i);
  ro = (int)(w & 0xffffu); lo = (int)((w >> 16) & 255u); tn = (int)(w >> 24);
}
MGS_DEV void row_addr(int i, int n, int blocked, int &ro, int &s, int &tadr, int &tnum) {
  if (blocked) { blk_row(i, ro, tadr, tnum); s = tnum; }
  else { ro = i * n; s = n; tadr = 0; tnum = n; }
}
#ifdef MGS_HOST
// 1-lane host build: the same factorisation written serially (per block)
MGS_DEVN void chol_factor_w(real *A, int n, int blocked, real *colbuf = (real *)0) {
  for (int j = 0; j < n; j++) {
    int ro, s, tadr, tnum;
    row_addr(j, n, blocked, ro, s, tadr, tnum);
    const int hi = tadr + tnum;
    real d = A[ro + j];
    d = sqrt(d > MGS_MINVAL ? d : MGS_MINVAL);
    const real inv = R_(1.0) / d;
    A[ro + j] = d;
    for (int i = j + 1; i < hi; i++) A[ro + (i - j) * s + j] *= inv;
    for (int i = j + 1; i < hi; i++) {
      const real lij = A[ro + (i - j) * s + j];
      for (int k = j + 1; k <= i; k++) A[ro + (i - j) * s + k] -= lij * A[ro + (k - j) * s + j];
    }
  }
}
MGS_DEVN void chol_solve_w(const real *L, real *x, int n, int blocked) {
  for (int k = 0; k < n; k++) {
    int ro, s, tadr, tnum;
    row_addr(k, n, blocked, ro, s, tadr, tnum);
    const int hi = tadr + tnum;
    const real xk = x[k] / L[ro + k];
    x[k] = xk;
    for (int i = k + 1; i < hi; i++) x[i] -= L[ro + (i - k) * s + k] * xk;
  }
  for (int k = n - 1; k >= 0; k--) {
    int ro, s, tadr, tnum;
    row_addr(k, n, blocked, ro, s, tadr, tnum);
    const real xk = x[k] / L[ro + k];
    x[k] = xk;
    for (int i = tadr; i < k; i++) x[i] -= L[ro + i] * xk;
  }
}
#elif defined(MGS_WIDE)
// ENVIRONMENT PER CTA.  Dense factor (the Newton Hessian, n up to 255): right-looking, the trailing update of every column spread
// over all threads as a 16 x 16 grid over (row, column), ONE barrier per column: the column is used unscaled
// (A[i][k] -= A[i][j] A[k][j] / A[j][j]) and scaled to L afterwards, while the next column's update runs (nobody reads it again).
// ncu / stage clocks of the round-2 capture (Shadow + 10 objects, nv = 94): the row-per-lane version with three barriers per column
// was 27 % of the step (3.4 k cycles per column).  Block-diagonal factor: rows per lane like the warp variants, same single barrier.
MGS_DEVN void chol_factor_w(real *A, int n, int blocked, real *colbuf = (real *)0) {
  WSYNC();
  (void)colbuf;
  if (!blocked) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    real dprev = 1;
    #pragma unroll 1
    for (int j = 0; j < n; j++) {
      real d2 = A[j * n + j];
      d2 = d2 > MGS_MINVAL ? d2 : MGS_MINVAL;
      const real inv = R_(1.0) / d2;
      // this thread's column entries A[k][j] (k = j + 1 + tx + 16 m) are the same for all of its rows: loaded once, four at a
      // time, so that the read-modify-writes of a row are independent (a serial LDS-FFMA-STS chain per entry was 1.5 k cycles per column)
      #pragma unroll 1
      for (int k0 = j + 1 + tx; k0 < n; k0 += 64) {
        const int k1 = k0 + 16, k2 = k0 + 32, k3 = k0 + 48;
        const real c0 = A[k0 * n + j], c1 = k1 < n ? A[k1 * n + j] : R_(0.0), c2 = k2 < n ? A[k2 * n + j] : R_(0.0), c3 = k3 < n ? A[k3 * n + j] : R_(0.0);
        int i = j + 1 + ty;
        while (i < k0) i += 16;  // rows above the diagonal entry of the first column have nothing to update
        #pragma unroll 1
        for (; i < n; i += 16) {
          real *row = A + i * n;
          const real lij = row[j] * inv;
          const real r0 = row[k0], r1 = k1 <= i ? row[k1] : R_(0.0), r2 = k2 <= i ? row[k2] : R_(0.0), r3 = k3 <= i ? row[k3] : R_(0.0);
          row[k0] = r0 - lij * c0;
          if (k1 <= i) row[k1] = r1 - lij * c1;
          if (k2 <= i) row[k2] = r2 - lij * c2;
          if (k3 <= i) row[k3] = r3 - lij * c3;
        }
      }
      if (j > 0) {  // deferred scaling of column j - 1
        const real sd = sqrt(dprev), rs = R_(1.0) / sd;
        #pragma unroll 1
        for (int i = j - 1 + (int)threadIdx.x; i < n; i += LANES) A[i * n + j - 1] = (i == j - 1) ? sd : A[i * n + j - 1] * rs;
      }
      dprev = d2;
      WSYNC();
    }
    if (threadIdx.x == 0 && n > 0) A[(n - 1) * n + n - 1] = sqrt(dprev);
    WSYNC();
    return;
  }
  // block diagonal (n <= LANES: one row per thread): every tile advances one column per step, one barrier per step
  const int nsteps = MD.max_tree_dofs, i = threadIdx.x;
  int ro = 0, tadr = 0, tnum = 0;
  if (i < n) blk_row(i, ro, tadr, tnum);
  const int s = tnum;
  #pragma unroll 1
  for (int t = 0; t < nsteps; t++) {
    const int j = tadr + t, act = (i < n) && (t < tnum) && (i >= j);
    real d2 = 1, aij = 0;
    if (act) {
      d2 = A[ro + (j - i) * s + j];  // the pivot, unscaled (final: the previous step's trailing update is behind a barrier)
      d2 = d2 > MGS_MINVAL ? d2 : MGS_MINVAL;
      if (i > j) {
        aij = A[ro + j];
        const real lij = aij / d2;
        const real *col = A + ro + (j + 1 - i) * s + j;
        real *row = A + ro + j + 1;
        const int cnt = i - j;
        #pragma unroll 2
        for (int k = 0; k < cnt; k++) row[k] -= lij * col[k * s];
      }
    }
    WSYNC();  // every read of column j is done: scale it (the next step only reads column j + 1)
    if (act) A[ro + j] = (i == j) ? sqrt(d2) : aij / sqrt(d2);
  }
  WSYNC();
}
// x <- (L L')^-1 x, one row per thread (n <= LANES), in blocks of 32 rows = one warp: the warp that owns a block solves its 32 x 32
// diagonal triangle with shuffles (no CTA barrier inside, like the warp variants' solve), publishes the block's values, ONE barrier,
// and every later (earlier, in the backward pass) row absorbs the whole block with 32 multiply-adds.  2 x ceil(n / 32) barriers per
// solve instead of one per pivot (stage clocks of config 5: 188 pivots x ~230 cycles per 94 x 94 solve before).
MGS_DEVN void chol_solve_w(const real *L, real *x, int n, int blocked) {
  if (blocked) {
    // block-diagonal factor: every tile advances one pivot per step TOGETHER (max_tree_dofs steps, not n), one barrier per pivot:
    // the thread of row k + 1 finishes its own entry (last update, then the division by its diagonal) inside step k
    const int i = threadIdx.x;
    int ro = 0, s = n, lo = 0, tn = n;
    if (i < n) row_addr(i, n, blocked, ro, s, lo, tn);
    const int hi = lo + tn, nsteps = MD.max_tree_dofs;
    WSYNC();
    real xi = i < n ? x[i] : R_(0.0);
    if (i < n && i == lo) { xi = xi / L[ro + i]; x[i] = xi; }
    WSYNC();
    #pragma unroll 1
    for (int t = 0; t + 1 < nsteps; t++) {
      const int k = lo + t;
      if (i < n && i > k && k < hi) {
        xi -= L[ro + k] * x[k];
        if (i == k + 1) { xi = xi / L[ro + i]; x[i] = xi; }
      }
      WSYNC();
    }
    if (i < n && i == hi - 1) { xi = xi / L[ro + i]; x[i] = xi; }
    WSYNC();
    #pragma unroll 1
    for (int t = 0; t + 1 < nsteps; t++) {
      const int k = hi - 1 - t;
      if (i < n && i < k && k >= lo) {
        xi -= L[ro + (k - i) * s + i] * x[k];
        if (i == k - 1) { xi = xi / L[ro + i]; x[i] = xi; }
      }
      WSYNC();
    }
    WSYNC();
    return;
  }
  const int i = threadIdx.x, wb = i >> 5, nblk = (n + 31) >> 5;
  int ro = 0, s = n, lo = 0, tn = n;
  if (i < n) row_addr(i, n, blocked, ro, s, lo, tn);
  const int hi = lo + tn;
  WSYNC();
  real xi = i < n ? x[i] : R_(0.0);
  #pragma unroll 1
  for (int B = 0; B < nblk; B++) {  // forward: L y = x
    const int k0 = B << 5, k1 = min(n, k0 + 32);
    if (wb == B) {
      #pragma unroll 1
      for (int k = k0; k < k1; k++) {
        if (i == k) xi = xi / L[ro + i];
        const real xk = __shfl_sync(0xffffffffu, xi, k - k0);
        if (i < n && i > k && k >= lo) xi -= L[ro + k] * xk;
      }
      if (i < n) x[i] = xi;
    }
    WSYNC();
    if (i < n && wb > B) {
      #pragma unroll 4
      for (int k = max(k0, lo); k < k1; k++) xi -= L[ro + k] * x[k];
    }
  }
  #pragma unroll 1
  for (int B = nblk - 1; B >= 0; B--) {  // backward: L' z = y
    const int k0 = B << 5, k1 = min(n, k0 + 32);
    if (wb == B) {
      #pragma unroll 1
      for (int k = k1 - 1; k >= k0; k--) {
        if (i == k) xi = xi / L[ro + i];
        const real xk = __shfl_sync(0xffffffffu, xi, k - k0);
        if (i < k && k < hi) xi -= L[ro + (k - i) * s + i] * xk;
      }
      if (i < n) x[i] = xi;
    }
    WSYNC();
    if (i < n && wb < B) {
      const int kk = min(k1, hi);
      #pragma unroll 4
      for (int k = k0; k < kk; k++) xi -= L[ro + (k - i) * s + i] * x[k];
    }
  }
  WSYNC();
}
#else
// GPU: lanes own rows (row i on lane i % LANES); every diagonal block advances one pivot column per step.
// Warp variants, n <= 32 (every in-scope single-object model except Shadow): one row per lane, pivots kept in registers.
MGS_DEVN void chol_factor_w(real *A, int n, int blocked, real *colbuf = (real *)0) {
  const int nsteps = blocked ? MD.max_tree_dofs : n;
  if (LANES == 32 && n <= LANES) {  // (warp variants only: pivots by shuffle)
    const int i = MGS_LANE;
    int tadr = 0, tnum = n, ro = i * n, s = n;
    if (i < n) row_addr(i, n, blocked, ro, s, tadr, tnum);
    WSYNC();
    #pragma unroll 1
    for (int t = 0; t < nsteps; t++) {
      const int j = tadr + t;
      const int live = (i < n) && (t < tnum);
      // the pivot A[j][j] is final (previous trailing update + WSYNC); every lane of the block reads it, the pivot
      // lane writes its square root back only after the column has been scaled (second phase)
      real d = 1, lij = 0;
      if (live) {
        d = A[ro + (j - i) * s + j];
        d = sqrt(d > MGS_MINVAL ? d : MGS_MINVAL);
        // (IEEE sqrt and division on purpose: replacing them by MUFU.RSQ / __fdividef (<= 2 ulp) was measured - no speed-up on
        // Panda, +3 % on Robotiq, but the fp32 trajectory error of the 16-dof hands over the first 50 steps grew 4-13x)
        if (i > j) { lij = A[ro + j] * (R_(1.0) / d); A[ro + j] = lij; }
      }
      WSYNC();
      if (live) {
        if (i == j) A[ro + j] = d;
        else if (i > j) {
          const real *col = A + ro + (j + 1 - i) * s + j;  // A[k][j], k = j + 1 ..
          real *row = A + ro + j + 1;
          const int cnt = i - j;
          MGS_UNROLL_INNER
          for (int k = 0; k < cnt; k++) row[k] -= lij * col[k * s];
        }
      }
      WSYNC();
    }
    WSYNC();
    return;
  }
  #pragma unroll 1
  for (int t = 0; t < nsteps; t++) {
    WSYNC();
    #pragma unroll 1
    PFOR(i, n) {  // pivot rows: sqrt of the diagonal
      int ro, s, tadr, tnum;
      row_addr(i, n, blocked, ro, s, tadr, tnum);
      if (i == tadr + t) { const real d = A[ro + i]; A[ro + i] = sqrt(d > MGS_MINVAL ? d : MGS_MINVAL); }
    }
    WSYNC();
    #pragma unroll 1
    PFOR(i, n) {  // scale the pivot column
      int ro, s, tadr, tnum;
      row_addr(i, n, blocked, ro, s, tadr, tnum);
      const int j = tadr + t;
      if (t < tnum && i > j) A[ro + j] /= A[ro + (j - i) * s + j];
    }
    WSYNC();
    #pragma unroll 1
    PFOR(i, n) {  // trailing update of this lane's rows
      int ro, s, tadr, tnum;
      row_addr(i, n, blocked, ro, s, tadr, tnum);
      const int j = tadr + t;
      if (t < tnum && i > j) {
        const real lij = A[ro + j];
        const real *col = A + ro + (j + 1 - i) * s + j;
        real *row = A + ro + j + 1;
        const int cnt = i - j;
        MGS_UNROLL_INNER
        for (int k = 0; k < cnt; k++) row[k] -= lij * col[k * s];
      }
    }
  }
  WSYNC();
}
// x <- (L L')^-1 x (column-oriented substitution)
MGS_DEVN void chol_solve_w(const real *L, real *x, int n, int blocked) {
  const int nsteps = blocked ? MD.max_tree_dofs : n;
  if (LANES == 32 && n <= LANES) {
    const int i = MGS_LANE;
    int tadr = 0, tnum = n, ro = i * n, s = n;
    if (i < n) row_addr(i, n, blocked, ro, s, tadr, tnum);
    // the right-hand side lives in registers (lane i owns x[i]); x[k] travels by shuffle: no shared-memory
    // round trip and no warp barrier per column
    WSYNC();
    real xi = (i < n) ? x[i] : R_(0.0);
    #pragma unroll 1
    for (int t = 0; t < nsteps; t++) {
      const int k = tadr + t, live = (i < n) && (t < tnum);
      const real xs = __shfl_sync(0xffffffffu, xi, live ? k : i);
      if (live) {
        const real xk = xs / L[ro + (k - i) * s + k];
        if (i == k) xi = xk;
        else if (i > k) xi -= L[ro + k] * xk;
      }
    }
    #pragma unroll 1
    for (int t = nsteps - 1; t >= 0; t--) {
      const int k = tadr + t, live = (i < n) && (t < tnum);
      const real xs = __shfl_sync(0xffffffffu, xi, live ? k : i);
      if (live) {
        const real xk = xs / L[ro + (k - i) * s + k];
        if (i == k) xi = xk;
        else if (i < k) xi -= L[ro + (k - i) * s + i] * xk;
      }
    }
    if (i < n) x[i] = xi;
    WSYNC();
    return;
  }
  #pragma unroll 1
  for (int pass = 0; pass < 2; pass++) {
    #pragma unroll 1
    for (int tt = 0; tt < nsteps; tt++) {
      const int t = pass == 0 ? tt : nsteps - 1 - tt;
      WSYNC();
      #pragma unroll 1
      PFOR(i, n) {
        int ro, s, tadr, tnum;
        row_addr(i, n, blocked, ro, s, tadr, tnum);
        if (i == tadr + t) x[i] /= L[ro + i];
      }
      WSYNC();
      #pragma unroll 1
      PFOR(i, n) {
        int ro, s, tadr, tnum;
        row_addr(i, n, blocked, ro, s, tadr, tnum);
        const int k = tadr + t;
        if (t >= tnum) continue;
        if (pass == 0 && i > k) x[i] -= L[ro + k] * x[k];
        else if (pass == 1 && i < k) x[i] -= L[ro + (k - i) * s + i] * x[k];
      }
    }
  }
  WSYNC();
}
#endif
// Ainv <- (L L')^-1 of a block-diagonal factor, both in block storage; one column per lane (serial substitution inside the lane)
MGS_DEVN void chol_inverse_w(const real *L, real *Ainv, int n) {
  #pragma unroll 1
  PFOR(c, n) {
    int roc, lo, t;
    blk_row(c, roc, lo, t);
    const int bo = roc - (c - lo) * t + lo;  // first word of the tile
    const real *Lt = L + bo;
    real *At = Ainv + bo;
    const int cl = c - lo;
    #pragma unroll 1
    for (int i = 0; i < t; i++) {
      real sacc = (i == cl) ? R_(1.0) : R_(0.0);
      MGS_UNROLL_INNER
      for (int k = 0; k < i; k++) sacc -= Lt[i * t + k] * At[k * t + cl];
      At[i * t + cl] = sacc / Lt[i * t + i];
    }
    #pragma unroll 1
    for (int i = t - 1; i >= 0; i--) {
      real sacc = At[i * t + cl];
      MGS_UNROLL_INNER
      for (int k = i + 1; k < t; k++) sacc -= Lt[k * t + i] * At[k * t + cl];
      At[i * t + cl] = sacc / Lt[i * t + i];
    }
  }
  WSYNC();
}
// y <- A x for a block-diagonal A in block storage (lane per row; only the row's own tree contributes)
MGS_DEVN void matvec_w(real *y, const real *A, const real *x, int n) {
  #pragma unroll 1
  PFOR(i, n) {
    int ro, lo, tn;
    blk_row(i, ro, lo, tn);
    const int hi = lo + tn;
    const real *row = A + ro;
    real t = 0;
    MGS_UNROLL_INNER
    for (int j = lo; j < hi; j++) t += row[j] * x[j];
    y[i] = t;
  }
  WSYNC();
}

// ---------------------------------------------------------------------------------- kinematics
MGS_DEVN void kinematics_w(Env &e) {
  #pragma unroll 1
  PFOR(i, 1) {
    EF(xpos)[0] = EF(xpos)[1] = EF(xpos)[2] = 0;
    EF(xquat)[0] = 1; EF(xquat)[1] = EF(xquat)[2] = EF(xquat)[3] = 0;
    for (int k = 0; k < 9; k++) EF(xmat)[k] = EF(ximat)[k] = (k % 4 == 0) ? R_(1.0) : R_(0.0);
    EF(xipos)[0] = EF(xipos)[1] = EF(xipos)[2] = 0;
  }
  WSYNC();
  #pragma unroll 1
  for (int lvl = 1; lvl <= MD.maxdepth; lvl++) {
    #pragma unroll 1
    PFOR(b, MD.nbody) {
      if (LDG(MD.body_depth + b) != lvl) continue;
      int p = LDG(MD.body_parentid + b);
      real xp[3], xq[4], t[3], bq[4];
      int mid = LDG(MD.body_mocapid + b);
      if (mid >= 0) {
        copy3(xp, EF(mocap) + 7 * mid);
        xq[0] = EF(mocap)[7 * mid + 3]; xq[1] = EF(mocap)[7 * mid + 4]; xq[2] = EF(mocap)[7 * mid + 5]; xq[3] = EF(mocap)[7 * mid + 6];
        normquat(xq);
      } else {
        ld3(t, MD.body_pos + 3 * b);
        mulmatvec3(xp, EF(xmat) + 9 * p, t);
        add3(xp, xp, EF(xpos) + 3 * p);
        ld4(bq, MD.body_quat + 4 * b);
        mulquat(xq, EF(xquat) + 4 * p, bq);
      }
      int ja = LDG(MD.body_jntadr + b), jn = LDG(MD.body_jntnum + b);
      #pragma unroll 1
      for (int j = ja; j < ja + jn; j++) {
        int qa = LDG(MD.jnt_qposadr + j), jt = LDG(MD.jnt_type + j);
        real *anchor = EF(xanchor) + 3 * j, *axis = EF(xaxis) + 3 * j;
        if (jt == JNT_FREE) {
          copy3(xp, EF(qpos) + qa);
#ifdef MGS_QPOS_COMP
          // the integrator keeps hi + lo normalised (in double); only an externally written quaternion is renormalised in place
          xq[0] = EF(qpos)[qa + 3]; xq[1] = EF(qpos)[qa + 4]; xq[2] = EF(qpos)[qa + 5]; xq[3] = EF(qpos)[qa + 6];
          if (fabs(xq[0] * xq[0] + xq[1] * xq[1] + xq[2] * xq[2] + xq[3] * xq[3] - R_(1.0)) > R_(1e-5)) {
            normquat(EF(qpos) + qa + 3);
            for (int k = 3; k < 7; k++) { xq[k - 3] = EF(qpos)[qa + k]; QPOS_LO_CLEAR(qa + k); }
          } else normquat(xq);
#else
          normquat(EF(qpos) + qa + 3);
          xq[0] = EF(qpos)[qa + 3]; xq[1] = EF(qpos)[qa + 4]; xq[2] = EF(qpos)[qa + 5]; xq[3] = EF(qpos)[qa + 6];
#endif
          copy3(anchor, xp);
          axis[0] = 0; axis[1] = 0; axis[2] = 1;
          continue;
        }
        real Rm[9], ja3[3], jp3[3];
        quat2mat(Rm, xq);
        ld3(ja3, MD.jnt_axis + 3 * j); ld3(jp3, MD.jnt_pos + 3 * j);
        mulmatvec3(axis, Rm, ja3);
        mulmatvec3(anchor, Rm, jp3);
        add3(anchor, anchor, xp);
        real dq = EF(qpos)[qa] - LDG(MD.qpos0 + qa);
        if (jt == JNT_SLIDE) {
          addscl3(xp, axis, dq);
        } else {
          real sn = sin(R_(0.5) * dq), cs = cos(R_(0.5) * dq);
          real ql[4] = {cs, sn * ja3[0], sn * ja3[1], sn * ja3[2]};
          mulquat(xq, xq, ql);
          quat2mat(Rm, xq);
          mulmatvec3(t, Rm, jp3);
          sub3(xp, anchor, t);
        }
      }
      normquat(xq);
      copy3(EF(xpos) + 3 * b, xp);
      EF(xquat)[4 * b] = xq[0]; EF(xquat)[4 * b + 1] = xq[1]; EF(xquat)[4 * b + 2] = xq[2]; EF(xquat)[4 * b + 3] = xq[3];
      quat2mat(EF(xmat) + 9 * b, xq);
      ld3(t, MD.body_ipos + 3 * b);
      mulmatvec3(t, EF(xmat) + 9 * b, t);
      add3(EF(xipos) + 3 * b, xp, t);
      ld4(bq, MD.body_iquat + 4 * b);
      real qi[4];
      mulquat(qi, xq, bq);
      quat2mat(EF(ximat) + 9 * b, qi);
    }
    WSYNC();
  }
  #pragma unroll 1
  PFOR(g, MD.ncgeom) {
    int b = LDG(MD.cgeom_bodyid + g);
    real t[3], q[4], gq[4];
    ld3(t, MD.cgeom_pos + 3 * g);
    mulmatvec3(t, EF(xmat) + 9 * b, t);
    add3(EF(gxpos) + 3 * g, EF(xpos) + 3 * b, t);
    ld4(gq, MD.cgeom_quat + 4 * g);
    mulquat(q, EF(xquat) + 4 * b, gq);
    quat2mat(EF(gxmat) + 9 * g, q);
  }
  WSYNC();
}

// spatial inertia helpers (CoM-based 10-vector: Ixx Iyy Izz Ixy Ixz Iyz, m*c, m)
MGS_DEV void mul_inert_vec(real *res, const real *I, const real *v) {
  real t[3];
  res[0] = I[0] * v[0] + I[3] * v[1] + I[4] * v[2];
  res[1] = I[3] * v[0] + I[1] * v[1] + I[5] * v[2];
  res[2] = I[4] * v[0] + I[5] * v[1] + I[2] * v[2];
  cross3(t, I + 6, v + 3);
  add3(res, res, t);
  cross3(t, I + 6, v);
  res[3] = I[9] * v[3] - t[0]; res[4] = I[9] * v[4] - t[1]; res[5] = I[9] * v[5] - t[2];
}
MGS_DEV void cross_motion(real *res, const real *vel, const real *v) {
  real t[3];
  cross3(res, vel, v);
  cross3(res + 3, vel, v + 3);
  cross3(t, vel + 3, v);
  add3(res + 3, res + 3, t);
}
MGS_DEV void cross_force(real *res, const real *vel, const real *f) {
  real t[3];
  cross3(res, vel, f);
  cross3(t, vel + 3, f + 3);
  add3(res, res, t);
  cross3(res + 3, vel, f + 3);
}

// CoM frames, composite inertias, motion axes, mass matrix, M^-1
MGS_DEVN void inertia_w(Env &e) {
  const int nb = MD.nbody, nv = MD.nv;
  // centre of mass of every kinematic tree (origin of its spatial quantities)
  #pragma unroll 1
  PFOR(b, nb) {
    if (b == 0 || LDG(MD.body_parentid + b) != 0) continue;
    real c[3] = {0, 0, 0}, mt = LDG(MD.body_subtreemass + b);
    if (mt < MGS_MINVAL) copy3(c, EF(xipos) + 3 * b);
    else {
      #pragma unroll 1
      for (int k = b; k < nb; k++)
        if (LDG(MD.body_rootid + k) == b) addscl3(c, EF(xipos) + 3 * k, LDG(MD.body_mass + k));
      scl3(c, c, R_(1.0) / mt);
    }
    copy3(EF(rootcom) + 3 * b, c);
  }
  WSYNC();
  #pragma unroll 1
  PFOR(b, nb) {
    real *ci = EF(cinert) + 10 * b;
    if (b == 0) { for (int k = 0; k < 10; k++) ci[k] = 0; continue; }
    real dif[3], diag[3], mass = LDG(MD.body_mass + b);
    const real *Rm = EF(ximat) + 9 * b;
    sub3(dif, EF(xipos) + 3 * b, EF(rootcom) + 3 * LDG(MD.body_rootid + b));
    ld3(diag, MD.body_inertia + 3 * b);
    real I[6];  // xx yy zz xy xz yz
    I[0] = Rm[0] * diag[0] * Rm[0] + Rm[1] * diag[1] * Rm[1] + Rm[2] * diag[2] * Rm[2];
    I[1] = Rm[3] * diag[0] * Rm[3] + Rm[4] * diag[1] * Rm[4] + Rm[5] * diag[2] * Rm[5];
    I[2] = Rm[6] * diag[0] * Rm[6] + Rm[7] * diag[1] * Rm[7] + Rm[8] * diag[2] * Rm[8];
    I[3] = Rm[0] * diag[0] * Rm[3] + Rm[1] * diag[1] * Rm[4] + Rm[2] * diag[2] * Rm[5];
    I[4] = Rm[0] * diag[0] * Rm[6] + Rm[1] * diag[1] * Rm[7] + Rm[2] * diag[2] * Rm[8];
    I[5] = Rm[3] * diag[0] * Rm[6] + Rm[4] * diag[1] * Rm[7] + Rm[5] * diag[2] * Rm[8];
    real d2 = dot3(dif, dif);
    ci[0] = I[0] + mass * (d2 - dif[0] * dif[0]);
    ci[1] = I[1] + mass * (d2 - dif[1] * dif[1]);
    ci[2] = I[2] + mass * (d2 - dif[2] * dif[2]);
    ci[3] = I[3] - mass * dif[0] * dif[1];
    ci[4] = I[4] - mass * dif[0] * dif[2];
    ci[5] = I[5] - mass * dif[1] * dif[2];
    ci[6] = mass * dif[0]; ci[7] = mass * dif[1]; ci[8] = mass * dif[2]; ci[9] = mass;
    for (int k = 0; k < 10; k++) EF(crb)[10 * b + k] = ci[k];
  }
  #pragma unroll 1
  PFOR(j, MD.njnt) {
    int b = LDG(MD.jnt_bodyid + j), da = LDG(MD.jnt_dofadr + j), jt = LDG(MD.jnt_type + j);
    real off[3];
    sub3(off, EF(rootcom) + 3 * LDG(MD.body_rootid + b), EF(xanchor) + 3 * j);
    if (jt == JNT_FREE) {
      for (int k = 0; k < 36; k++) EF(cdof)[6 * da + k] = 0;
      for (int k = 0; k < 3; k++) EF(cdof)[6 * (da + k) + 3 + k] = 1;
      for (int k = 0; k < 3; k++) {
        real ax[3] = {EF(xmat)[9 * b + k], EF(xmat)[9 * b + 3 + k], EF(xmat)[9 * b + 6 + k]};
        real *c = EF(cdof) + 6 * (da + 3 + k);
        copy3(c, ax);
        cross3(c + 3, ax, off);
      }
    } else if (jt == JNT_SLIDE) {
      real *c = EF(cdof) + 6 * da;
      c[0] = c[1] = c[2] = 0;
      copy3(c + 3, EF(xaxis) + 3 * j);
    } else {
      real *c = EF(cdof) + 6 * da;
      copy3(c, EF(xaxis) + 3 * j);
      cross3(c + 3, EF(xaxis) + 3 * j, off);
    }
  }
  #pragma unroll 1
  PFOR(i, MD.nM) EF(M)[i] = 0;
  WSYNC();
  // composite inertias: parents absorb their children, deepest level first
  #pragma unroll 1
  for (int lvl = MD.maxdepth - 1; lvl >= 1; lvl--) {
    #pragma unroll 1
    PFOR(b, nb) {
      if (LDG(MD.body_depth + b) != lvl) continue;
      #pragma unroll 1
      for (int c = b + 1; c < nb; c++)
        if (LDG(MD.body_parentid + c) == b)
          for (int k = 0; k < 10; k++) EF(crb)[10 * b + k] += EF(crb)[10 * c + k];
    }
    WSYNC();
  }
  #pragma unroll 1
  PFOR(i, nv) {
    real buf[6];
    mul_inert_vec(buf, EF(crb) + 10 * LDG(MD.dof_bodyid + i), EF(cdof) + 6 * i);
    #pragma unroll 1
    for (int j = i; j >= 0; j = LDG(MD.dof_parentid + j)) {
      real v = 0;
      for (int k = 0; k < 6; k++) v += EF(cdof)[6 * j + k] * buf[k];
      if (j == i) v += LDG(MD.dof_armature + i);
      EF(M)[LDG(MD.dof_rowoff + i) + j] = v;
      EF(M)[LDG(MD.dof_rowoff + j) + i] = v;
    }
  }
  WSYNC();
  #pragma unroll 1
  PFOR(i, MD.nM) EF(H)[i] = EF(M)[i];  // (block storage in the H scratch)
  chol_factor_w(EF(H), nv, 1);
  chol_inverse_w(EF(H), EF(Minv), nv);
}

// fixed tendons + actuator transmission
MGS_DEVN void transmission_w(Env &e) {
  const int nv = MD.nv;
  #pragma unroll 1
  PFOR(i, MD.ntendon * nv) EF(ten_J)[i] = 0;
  #pragma unroll 1
  PFOR(i, MD.nu * nv) EF(act_moment)[i] = 0;
  WSYNC();
  #pragma unroll 1
  PFOR(t, MD.ntendon) {
    real L = 0;
    int a = LDG(MD.tendon_adr + t), n = LDG(MD.tendon_num + t);
    #pragma unroll 1
    for (int w = a; w < a + n; w++) {
      real c = LDG(MD.wrap_coef + w);
      L += c * EF(qpos)[LDG(MD.wrap_qposadr + w)];
      EF(ten_J)[t * nv + LDG(MD.wrap_dofadr + w)] += c;
    }
    EF(ten_length)[t] = L;
  }
  WSYNC();
  #pragma unroll 1
  PFOR(a, MD.nu) {
    real gear = LDG(MD.actuator_gear + a);
    int id = LDG(MD.actuator_trnid + a);
    if (LDG(MD.actuator_trntype + a) == 0) {
      EF(act_length)[a] = gear * EF(qpos)[LDG(MD.jnt_qposadr + id)];
      EF(act_moment)[a * nv + LDG(MD.jnt_dofadr + id)] = gear;
    } else {
      EF(act_length)[a] = gear * EF(ten_length)[id];
      #pragma unroll 1
      for (int d = 0; d < nv; d++) EF(act_moment)[a * nv + d] = gear * EF(ten_J)[id * nv + d];
    }
  }
  WSYNC();
}

// velocities, bias (RNE without acceleration), passive and actuator forces -> qfrc_smooth, qacc_smooth
MGS_DEVN void smooth_forces_w(Env &e) {
  const int nb = MD.nbody, nv = MD.nv;
  #pragma unroll 1
  PFOR(k, 6) { EF(cvel)[k] = 0; EF(cfrc)[k] = 0; EF(cacc)[k] = (k < 3) ? R_(0.0) : -MD.gravity[k - 3]; }
  WSYNC();
  #pragma unroll 1
  for (int lvl = 1; lvl <= MD.maxdepth; lvl++) {
    #pragma unroll 1
    PFOR(b, nb) {
      if (LDG(MD.body_depth + b) != lvl) continue;
      int p = LDG(MD.body_parentid + b);
      real cv[6], ca[6];
      for (int k = 0; k < 6; k++) { cv[k] = EF(cvel)[6 * p + k]; ca[k] = EF(cacc)[6 * p + k]; }
      int ja = LDG(MD.body_jntadr + b), jn = LDG(MD.body_jntnum + b);
      #pragma unroll 1
      for (int j = ja; j < ja + jn; j++) {
        int da = LDG(MD.jnt_dofadr + j);
        if (LDG(MD.jnt_type + j) == JNT_FREE) {
          for (int k = 0; k < 18; k++) EF(cdof_dot)[6 * da + k] = 0;
          for (int k = 0; k < 3; k++)
            for (int c = 0; c < 6; c++) cv[c] += EF(cdof)[6 * (da + k) + c] * EF(qvel)[da + k];
          for (int k = 3; k < 6; k++) cross_motion(EF(cdof_dot) + 6 * (da + k), cv, EF(cdof) + 6 * (da + k));
          for (int k = 3; k < 6; k++)
            for (int c = 0; c < 6; c++) cv[c] += EF(cdof)[6 * (da + k) + c] * EF(qvel)[da + k];
          for (int k = 3; k < 6; k++)
            for (int c = 0; c < 6; c++) ca[c] += EF(cdof_dot)[6 * (da + k) + c] * EF(qvel)[da + k];
        } else {
          cross_motion(EF(cdof_dot) + 6 * da, cv, EF(cdof) + 6 * da);
          for (int c = 0; c < 6; c++) { cv[c] += EF(cdof)[6 * da + c] * EF(qvel)[da]; ca[c] += EF(cdof_dot)[6 * da + c] * EF(qvel)[da]; }
        }
      }
      real t1[6], t2[6];
      mul_inert_vec(t1, EF(cinert) + 10 * b, cv);
      cross_force(t2, cv, t1);
      mul_inert_vec(t1, EF(cinert) + 10 * b, ca);
      for (int k = 0; k < 6; k++) { EF(cvel)[6 * b + k] = cv[k]; EF(cacc)[6 * b + k] = ca[k]; EF(cfrc)[6 * b + k] = t1[k] + t2[k]; }
    }
    WSYNC();
  }
  #pragma unroll 1
  for (int lvl = MD.maxdepth - 1; lvl >= 1; lvl--) {
    #pragma unroll 1
    PFOR(b, nb) {
      if (LDG(MD.body_depth + b) != lvl) continue;
      #pragma unroll 1
      for (int c = b + 1; c < nb; c++)
        if (LDG(MD.body_parentid + c) == b)
          for (int k = 0; k < 6; k++) EF(cfrc)[6 * b + k] += EF(cfrc)[6 * c + k];
    }
    WSYNC();
  }
  // actuator forces (lane per actuator), then per-dof totals
  #pragma unroll 1
  PFOR(a, MD.nu) {
    real c = EF(ctrl)[a], vel = 0;
    if (LDG(MD.actuator_ctrllimited + a)) c = fmax(LDG(MD.actuator_ctrlrange + 2 * a), fmin(LDG(MD.actuator_ctrlrange + 2 * a + 1), c));
    #pragma unroll 1
    for (int d = 0; d < nv; d++) vel += EF(act_moment)[a * nv + d] * EF(qvel)[d];
    real f = LDG(MD.actuator_gainprm + 3 * a) * c + LDG(MD.actuator_biasprm + 3 * a) + LDG(MD.actuator_biasprm + 3 * a + 1) * EF(act_length)[a] +
             LDG(MD.actuator_biasprm + 3 * a + 2) * vel;
    if (LDG(MD.actuator_forcelimited + a)) f = fmax(LDG(MD.actuator_forcerange + 2 * a), fmin(LDG(MD.actuator_forcerange + 2 * a + 1), f));
    EF(act_force)[a] = f;
  }
  WSYNC();
  #pragma unroll 1
  PFOR(d, nv) {
    real bias = 0;
    int b = LDG(MD.dof_bodyid + d);
    for (int c = 0; c < 6; c++) bias += EF(cdof)[6 * d + c] * EF(cfrc)[6 * b + c];
    real f = -LDG(MD.dof_damping + d) * EF(qvel)[d] - bias;
    int j = LDG(MD.dof_jntid + d);
    if (LDG(MD.jnt_type + j) != JNT_FREE) {
      real k = LDG(MD.jnt_stiffness + j);
      int qa = LDG(MD.jnt_qposadr + j);
      if (k != 0) f -= k * (EF(qpos)[qa] - LDG(MD.qpos_spring + qa));
    }
    #pragma unroll 1
    for (int a = 0; a < MD.nu; a++) f += EF(act_moment)[a * nv + d] * EF(act_force)[a];
    EF(qfrc_smooth)[d] = f;
  }
  WSYNC();
  if (MD.ngravcomp > 0) {
    // gravity compensation (clutter scenes: the camera body): -gravity * mass * gravcomp at the body CoM.
    // Rare and tiny, so one lane walks the dof chains.
    #pragma unroll 1
    PFOR(one, 1) {
      #pragma unroll 1
      for (int b = 1; b < nb; b++) {
        const real gc = LDG(MD.body_gravcomp + b), mass = LDG(MD.body_mass + b);
        if (gc == 0 || mass == 0) continue;
        real off[3], f[3] = {-MD.gravity[0] * mass * gc, -MD.gravity[1] * mass * gc, -MD.gravity[2] * mass * gc};
        // body CoM relative to the tree origin: cinert holds mass * offset
        off[0] = EF(cinert)[10 * b + 6] / mass; off[1] = EF(cinert)[10 * b + 7] / mass; off[2] = EF(cinert)[10 * b + 8] / mass;
        int bb = b;
        while (bb > 0 && LDG(MD.body_dofnum + bb) == 0) bb = LDG(MD.body_parentid + bb);
        if (bb == 0) continue;
        #pragma unroll 1
        for (int d = LDG(MD.body_dofadr + bb) + LDG(MD.body_dofnum + bb) - 1; d >= 0; d = LDG(MD.dof_parentid + d)) {
          const real *c = EF(cdof) + 6 * d;
          real lin[3];
          cross3(lin, c, off);
          EF(qfrc_smooth)[d] += (lin[0] + c[3]) * f[0] + (lin[1] + c[4]) * f[1] + (lin[2] + c[5]) * f[2];
        }
      }
    }
    WSYNC();
  }
  matvec_w(EF(qacc_smooth), EF(Minv), EF(qfrc_smooth), nv);
}
