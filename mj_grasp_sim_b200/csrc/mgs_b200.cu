// mgs_b200.cu - the C ABI (include/mgs_b200.h) + the 16-warp variant of the persistent warp-per-environment rollout
// kernel (mgs_kernel.cuh; the 12-warp variant lives in mgs_kernel_w12.cu).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/mgs_b200.h"
#include "mgs_model_build.h"
#ifndef MGS_MAX_WARPS_PER_BLOCK
#define MGS_MAX_WARPS_PER_BLOCK 16
#endif
#define MGS_KERNEL_TAG w16
#include "mgs_kernel.cuh"

// ---------------------------------------------------------------------------------- host side
static thread_local std::string g_err;
static std::atomic<long long> g_launches{0};
// One lock for everything that touches per-kernel-variant global state: the variant's __constant__ block (rewritten per
// launch), its dynamic-shared-memory attribute (per kernel function, so shared by all models on the variant) and the
// per-device "previous launch finished" events.  Host threads may call into different model handles concurrently
// (ctypes releases the GIL); launches are enqueued under the lock, they do not execute under it.
static std::mutex g_launch_mu;
static std::vector<cudaEvent_t> g_last_done;  // [device], created on first use, never destroyed
static std::vector<char> g_have_last;
#ifndef MGS_BUILD_STAMP
#define MGS_BUILD_STAMP "unstamped"
#endif

static int fail(const std::string &msg) { g_err = msg; return -1; }
int mgs_set_error(const char *msg) { return fail(msg); }  // for the other translation units of the library
#define CU(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess) return fail(std::string(#call) + ": " + cudaGetErrorString(e_));       \
  } while (0)

struct MgsModel {
  int device;
  DevModel dm;
  Layout L;
  char *d_blob;
  unsigned int *d_counter;
  int num_sms, blocks_per_sm, smem_per_block, warps_per_block;
  const MgsKernelOps *ops;  // the kernel variant this model runs on
  int state_stride, diag_stride;
  // staging for the host-pointer entry points (grown on demand)
  void *d_stage, *h_stage;
  size_t stage_bytes;
  int *d_mpr_cache;  // global MPR cache (models with more pairs than the shared-memory cache holds): npair x 4 words per environment slot
  float *d_aux;  // [aux_cap][4] per-candidate auxiliary results of the most recent rollout launch (flags, drift)
  int aux_cap, aux_n;
  double qvel_clip;
  cudaStream_t stream;
  real *d_env_state;  // wide_g variant: the environments' state, one Layout.total slice per CTA of the persistent grid (else null)
  unsigned int *d_scene_success;  // [scene_cap] successes per scene of the enough_stable early stop (grown on demand)
  int scene_cap;
};

extern "C" const char *mgs_last_error(void) { return g_err.c_str(); }
extern "C" long long mgs_launch_count(void) { return g_launches.load(); }
extern "C" const char *mgs_build_stamp(void) { return MGS_BUILD_STAMP; }

extern "C" int mgs_model_create(const MgsModelDesc *desc, int device, MgsModel **out) {
  return mgs_model_create_ex(desc, device, 0, 0, out);
}

// allow_global: a model whose environment state does not fit one CTA's shared memory runs on the wide_g variant (state in a global
// slab) instead of failing - mgs_model_create_any.  mgs_model_create / _ex keep failing there: callers (EscalatingSim) probe for the
// largest capacity that fits shared memory that way.
static int model_create(const MgsModelDesc *desc, int device, int ncon_max, int nefc_max, bool allow_global, MgsModel **out) {
  if (!desc || !out) return fail("null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("no CUDA device: libmgs_b200 has no CPU path");
  if (device < 0 || device >= ndev) return fail("bad device index");
  CU(cudaSetDevice(device));
  ModelBlob blob;
  std::string err;
  if (!build_model_blob(desc, blob, err)) return fail("model: " + err);
  if (ncon_max > 0) {
    blob.ncon_max = (ncon_max + 3) & ~3;
    blob.nefc_max = blob.rows_static + blob.ncon_max * blob.rows_per_contact;  // the default for this contact capacity
  }
  if (nefc_max > 0) blob.nefc_max = nefc_max;
  if (blob.ncon_max > 256 || blob.nefc_max < desc->nv || 6 * blob.ncon_max > 2 * blob.nefc_max ||
      blob.nefc_max < blob.dm.ne_rows + blob.dm.nf_rows)
    return fail("bad contact capacities (need ncon_max <= 256, nefc_max >= 3 * ncon_max and room for the equality / dof-friction rows)");
  MgsModel *M = new MgsModel();
  memset(M, 0, sizeof(*M));
  M->device = device;
  CU(cudaMalloc(&M->d_blob, blob.bytes.size()));
  CU(cudaMemcpy(M->d_blob, blob.bytes.data(), blob.bytes.size(), cudaMemcpyHostToDevice));
  M->dm = blob.dm;
  rebase_model(M->dm, M->d_blob);
  CU(cudaMalloc(&M->d_counter, 2 * sizeof(unsigned int)));  // [0] work queue head, [1] environments that overflowed a capacity
  int ncache_max = MGS_MPR_CACHE_MAX;
  auto make_layout = [&](int lanes) {
    layout_compute(&M->L, desc->nq, desc->nv, desc->nu, desc->nbody, desc->njnt, desc->nmocap, desc->ntendon, desc->ncgeom, blob.ncon_max,
                   blob.nefc_max, desc->npair, blob.dm.nM, lanes, ncache_max);
    return (int)(M->L.total * sizeof(real));
  };
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  M->num_sms = prop.multiProcessorCount;
  int env_bytes = 0;
  // Warp-per-environment variants: CTA size = the warps-per-block that gives the most resident warps per SM (shared memory per
  // environment and the per-CTA reservation decide).  First with the 16-warp variant; if at most 12 environments fit per SM
  // anyway, the 12-warp variant (more registers per thread) takes over.  Scenes that leave room for fewer than
  // MGS_WIDE_BELOW_ENVS environments per SM (or for none) run the environment-per-CTA variant instead.
  const char *force_wpb = getenv("MGS_WARPS_PER_BLOCK");  // tuning knobs: force the CTA size / the variant
  const char *force_var = getenv("MGS_KERNEL_VARIANT");
  const bool force_wide_g = force_var && std::string(force_var) == "wide_g";
  const bool force_wide = (force_var && std::string(force_var) == "wide") || force_wide_g;
  std::lock_guard<std::mutex> lock(g_launch_mu);  // the occupancy sweep changes the variants' shared-memory attribute
  const MgsKernelOps *variants[2] = {mgs_kernel_ops_w16(), mgs_kernel_ops_w12()};
  int best_warps = 0;
  // FIRST-PASS CAPACITY of single-object scenes, when the caller left the capacities to the library: if the default contact
  // capacity leaves room for fewer than MGS_WIDE_BELOW_ENVS warp-environments per SM, smaller ones are tried (24, 20, 16 contacts,
  // then 16 and 12 with the shared-memory MPR cache cut to 32 pairs - the rest of the pairs use the global cache) and the first
  // that fits that many is taken.  Measured on the Allegro hand in the fp64 build (its product path): 32 contacts =
  // 90 KB per environment = the environment-per-CTA variant at 0.54 M env-steps/s; 16 contacts = 57 KB = four warp-environments
  // per SM at 0.94 M, no environment of 1,024 over capacity, identical labels (profiles/caps_sweep_r2c_f64_hands.log).  An
  // environment that does exceed its capacity is flagged per candidate as always and re-run on larger capacities by the callers
  // (mgs.env EscalatingSim, tools/label_agreement.py).  MGS_NO_AUTO_CAPS=1 keeps the default capacity.
  const bool auto_caps = ncon_max <= 0 && nefc_max <= 0 && !force_var && !force_wpb && blob.nfreeobj <= 1 && !getenv("MGS_NO_AUTO_CAPS");
  const int default_nc = blob.ncon_max, default_ne = blob.nefc_max;
  const int ntry = 6, try_nc[ntry] = {default_nc, 24, 20, 16, 16, 12}, try_cache[ntry] = {MGS_MPR_CACHE_MAX, MGS_MPR_CACHE_MAX, MGS_MPR_CACHE_MAX, MGS_MPR_CACHE_MAX, 32, 32};
  for (int attempt = 0; attempt < ntry; attempt++) {
    if (attempt > 0) {
      if (!auto_caps || force_wide) break;
      if (try_nc[attempt] >= default_nc) continue;
      blob.ncon_max = try_nc[attempt];
      blob.nefc_max = blob.rows_static + blob.ncon_max * blob.rows_per_contact;
      ncache_max = try_cache[attempt];
    }
    env_bytes = make_layout(32);
    best_warps = 0;
    for (int v = 0; v < 2 && !force_wide && (size_t)env_bytes <= prop.sharedMemPerBlockOptin; v++) {
      const MgsKernelOps *ops = variants[v];
      if (force_var && std::string(force_var) != (v == 0 ? "w16" : "w12")) continue;
      if (v == 1 && !force_var && (best_warps == 0 || best_warps > ops->max_warps || M->blocks_per_sm != 1)) break;
      int vb = 0, vw = 0, vo = 0;
      for (int w = 1; w <= ops->max_warps; w++) {
        if (force_wpb && atoi(force_wpb) != w) continue;
        if ((size_t)env_bytes * w > prop.sharedMemPerBlockOptin) break;
        CU(ops->prepare(env_bytes * w));
        int occ = 0;
        CU(ops->occupancy(&occ, w * 32, (size_t)env_bytes * w));
        if (occ * w >= vb && occ > 0) { vb = occ * w; vw = w; vo = occ; }  // ties go to the LARGER CTA: one CTA per SM keeps all resident warps stage-aligned
      }
      if (vb >= best_warps && vb > 0) { best_warps = vb; M->warps_per_block = vw; M->blocks_per_sm = vo; M->ops = ops; }
    }
    if (best_warps >= MGS_WIDE_BELOW_ENVS) break;
  }
  if (best_warps < MGS_WIDE_BELOW_ENVS && blob.ncon_max != default_nc) {  // no smaller capacity helped: back to the default (wide variant)
    blob.ncon_max = default_nc;
    blob.nefc_max = default_ne;
    ncache_max = MGS_MPR_CACHE_MAX;
    env_bytes = make_layout(32);
  }
  bool in_global = false;
  if (force_wide || (!force_var && best_warps < MGS_WIDE_BELOW_ENVS)) {
    const MgsKernelOps *ops = mgs_kernel_ops_wide();
    env_bytes = make_layout(ops->lanes_per_env);
    in_global = force_wide_g || (allow_global && (size_t)env_bytes > prop.sharedMemPerBlockOptin);
    if (in_global) ops = mgs_kernel_ops_wide_g();  // same lanes per environment, so the same layout
    if (!in_global && (size_t)env_bytes > prop.sharedMemPerBlockOptin) {
      delete M;
      return fail("model needs more shared memory per environment than one CTA can have: lower ncon_max / nefc_max");
    }
    const int dyn_smem = in_global ? 0 : env_bytes;
    CU(ops->prepare(dyn_smem));
    int occ = 0;
    CU(ops->occupancy(&occ, ops->lanes_per_env, (size_t)dyn_smem));
    best_warps = occ;
    M->warps_per_block = 1; M->blocks_per_sm = occ; M->ops = ops;
  }
  if (best_warps > 0 && desc->npair > M->L.ncache) {
    // global MPR cache: one slab per environment slot (CTA of the wide variant, warp slot of the warp variants)
    const size_t slots = (size_t)M->num_sms * M->blocks_per_sm * (M->ops->lanes_per_env > 32 ? 1 : M->ops->max_warps);
    CU(cudaMalloc(&M->d_mpr_cache, slots * desc->npair * 4 * sizeof(int)));
  }
  if (best_warps == 0) { delete M; return fail("kernel does not fit on this device"); }
  if (in_global) {  // one slice per CTA of the persistent grid (launch() never starts more CTAs than that)
    const size_t slab = (size_t)M->num_sms * M->blocks_per_sm * env_bytes;
    if (cudaMalloc(&M->d_env_state, slab) != cudaSuccess) {
      cudaGetLastError();
      M->d_env_state = nullptr;
      mgs_model_destroy(M);
      return fail("cannot allocate the global-memory environment state (" + std::to_string(slab >> 20) + " MiB)");
    }
  }
  M->smem_per_block = in_global ? 0 : env_bytes * M->warps_per_block;
  // (the attribute is set again before every launch: it belongs to the kernel function, not to this model)
  M->state_stride = desc->nq + 2 * desc->nv + desc->nu + 7 * desc->nmocap;
  M->diag_stride = mgs_diag_stride(desc->nv, desc->nbody, blob.ncon_max, blob.nefc_max);
  CU(cudaStreamCreateWithFlags(&M->stream, cudaStreamNonBlocking));
  *out = M;
  return 0;
}

extern "C" int mgs_model_create_ex(const MgsModelDesc *desc, int device, int ncon_max, int nefc_max, MgsModel **out) {
  return model_create(desc, device, ncon_max, nefc_max, false, out);
}

extern "C" int mgs_model_create_any(const MgsModelDesc *desc, int device, int ncon_max, int nefc_max, MgsModel **out) {
  return model_create(desc, device, ncon_max, nefc_max, true, out);
}

extern "C" int mgs_model_state_in_global(const MgsModel *M) {
  if (!M) return fail("null model");
  return M->d_env_state ? 1 : 0;
}

extern "C" void mgs_model_destroy(MgsModel *M) {
  if (!M) return;
  cudaSetDevice(M->device);
  cudaFree(M->d_blob);
  cudaFree(M->d_counter);
  if (M->d_mpr_cache) cudaFree(M->d_mpr_cache);
  if (M->d_env_state) cudaFree(M->d_env_state);
  if (M->d_aux) cudaFree(M->d_aux);
  if (M->d_scene_success) cudaFree(M->d_scene_success);
  if (M->d_stage) cudaFree(M->d_stage);
  if (M->h_stage) cudaFreeHost(M->h_stage);
  if (M->stream) cudaStreamDestroy(M->stream);
  delete M;
}

extern "C" int mgs_overflow_count(MgsModel *M) {
  if (!M) return fail("null model");
  unsigned int v[2] = {0, 0};
  if (cudaSetDevice(M->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
      cudaMemcpy(v, M->d_counter, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess)
    return fail("mgs_overflow_count: CUDA error");
  return (int)v[1];
}

extern "C" int mgs_last_aux(MgsModel *M, int n, float *aux_out) {
  if (!M || !aux_out) return fail("null argument");
  if (n > M->aux_n) return fail("mgs_last_aux: the most recent launch had fewer candidates");
  if (n <= 0) return 0;
  if (cudaSetDevice(M->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
      cudaMemcpy(aux_out, M->d_aux, (size_t)n * 4 * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess)
    return fail("mgs_last_aux: CUDA error");
  return 0;
}

extern "C" int mgs_set_qvel_clip(MgsModel *M, double clip) {
  if (!M) return fail("null model");
  M->qvel_clip = clip > 0 ? clip : 0;
  return 0;
}

extern "C" int mgs_model_info(const MgsModel *M, MgsModelInfo *info) {
  if (!M || !info) return fail("null argument");
  info->nq = M->dm.nq; info->nv = M->dm.nv; info->nu = M->dm.nu; info->nmocap = M->dm.nmocap;
  info->state_stride = M->state_stride; info->diag_stride = M->diag_stride;
  info->ncon_max = M->L.ncon_max; info->nefc_max = M->L.nefc_max;
  info->smem_bytes_per_env = (int)(M->L.total * sizeof(real));
  info->warps_per_block = M->warps_per_block; info->blocks_per_sm = M->blocks_per_sm; info->num_sms = M->num_sms;
  info->real_bytes = (int)sizeof(real);
  info->lanes_per_env = M->ops->lanes_per_env;
  return 0;
}

static int launch(MgsModel *M, const RolloutParams &prm, const BatchIO &io_in, cudaStream_t st) {
  if (prm.n <= 0) return 0;
  BatchIO io = io_in;
  io.work_counter = M->d_counter;
  if (prm.n > M->aux_cap) {
    CU(cudaDeviceSynchronize());
    if (M->d_aux) cudaFree(M->d_aux);
    M->d_aux = nullptr; M->aux_cap = 0;
    const int cap = (prm.n + 1023) & ~1023;
    CU(cudaMalloc(&M->d_aux, (size_t)cap * 4 * sizeof(float)));
    M->aux_cap = cap;
  }
  io.aux = M->d_aux;
  io.mpr_cache_g = M->d_mpr_cache;
  io.env_state = M->d_env_state;
  M->aux_n = prm.n;
  // Wave quantisation: every candidate of a batch costs about the same, so what matters is the number of
  // "waves" of resident environments.  If fewer warps per CTA give the same number of waves, use fewer: each
  // environment then shares its SM with fewer neighbours (4096 candidates: 2 waves of 14 warps/SM beat
  // 1.73 waves of 16 by 3.5 % on B200).
  int wpb = M->warps_per_block;
  if (M->blocks_per_sm == 1 && !getenv("MGS_WARPS_PER_BLOCK")) {
    const int slots = M->num_sms * wpb;
    const int waves = (prm.n + slots - 1) / slots;
    const int need = (prm.n + M->num_sms * waves - 1) / (M->num_sms * waves);
    if (need < wpb) wpb = need < 1 ? 1 : need;
  }
  int blocks_needed = (prm.n + wpb - 1) / wpb;
  int grid = M->num_sms * M->blocks_per_sm;
  if (grid > blocks_needed) grid = blocks_needed;
  // The constants of this launch (model pointers, layout, parameters, I/O) go to the variant's __constant__ block,
  // stream-ordered: the stream first waits for the previous launch on this device (any model, any stream), THEN resets this
  // model's work queue / overflow counter, sets the variant's shared-memory attribute for this model and launches.
  std::lock_guard<std::mutex> lock(g_launch_mu);
  if ((size_t)M->device >= g_last_done.size()) { g_last_done.resize(M->device + 1); g_have_last.resize(M->device + 1, 0); }
  if (!g_have_last[M->device]) {
    CU(cudaEventCreateWithFlags(&g_last_done[M->device], cudaEventDisableTiming));
    g_have_last[M->device] = 1;
  } else CU(cudaStreamWaitEvent(st, g_last_done[M->device], 0));
  CU(cudaMemsetAsync(M->d_counter, 0, 2 * sizeof(unsigned int), st));
  if (io.scene_success) CU(cudaMemsetAsync(io.scene_success, 0, (size_t)io.nscene * sizeof(unsigned int), st));
  CU(M->ops->prepare(M->smem_per_block));
  KernelConsts kc;
  kc.m = M->dm; kc.L = M->L; kc.prm = prm; kc.io = io;
  CU(M->ops->launch(&kc, grid, wpb * M->ops->lanes_per_env, (size_t)(M->smem_per_block / M->warps_per_block) * wpb, st));
  g_launches++;
  CU(cudaEventRecord(g_last_done[M->device], st));
  return 0;
}

static int fill_params(const MgsModel *M, RolloutParams &prm, int mode, int n, int nj, const int *joint_qposadr, int base_qposadr,
                       const double *close_ctrl, const MgsRolloutCfg *cfg) {
  memset(&prm, 0, sizeof(prm));
  if (nj > MGS_MAX_NJ) return fail("too many actuated joints");
  if (base_qposadr < 0 || base_qposadr + 7 > M->dm.nq) return fail("bad base_qposadr");
  prm.mode = mode; prm.n = n; prm.nj = nj; prm.base_qposadr = base_qposadr;
  for (int k = 0; k < nj; k++) {
    if (joint_qposadr[k] < 0 || joint_qposadr[k] >= M->dm.nq) return fail("bad joint_qposadr");
    prm.joint_qposadr[k] = joint_qposadr[k];
  }
  if (mode == MGS_MODE_STABILITY || mode == MGS_MODE_CLUTTER_STABLE) {
    if (!cfg || !close_ctrl) return fail("stability rollout needs cfg and close_ctrl");
    prm.nstep_close = cfg->nstep_close; prm.nstep_lift = cfg->nstep_lift; prm.shake_steps = cfg->shake_steps;
    prm.repose_on_close = cfg->repose_on_close; prm.lift_dist = (real)cfg->lift_dist; prm.shake_dist = (real)cfg->shake_dist;
    for (int u = 0; u < M->dm.nu; u++) prm.close_ctrl[u] = (real)close_ctrl[u];
  }
  return 0;
}

extern "C" int mgs_rollout_device(MgsModel *M, int mode, int n, const float *d_pose7, const float *d_joints, int nj,
                                  const int *joint_qposadr, int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg,
                                  uint8_t *d_labels, int *d_steps, void *stream) {
  if (!M) return fail("null model");
  if (mode != MGS_MODE_COLLISION && mode != MGS_MODE_STABILITY) return fail("bad mode");
  CU(cudaSetDevice(M->device));
  RolloutParams prm;
  if (fill_params(M, prm, mode, n, nj, joint_qposadr, base_qposadr, close_ctrl, cfg)) return -1;
  BatchIO io;
  memset(&io, 0, sizeof(io));
  io.pose7 = d_pose7; io.joints = d_joints; io.labels = d_labels; io.steps = d_steps;
  return launch(M, prm, io, (cudaStream_t)stream);
}

extern "C" int mgs_clutter_scenes_device(MgsModel *M, int mode, int n, int nscene, const void *d_scenes, const int *d_scene_index,
                                         int enough_stable, const float *d_pose7, const float *d_joints, int nj, const int *joint_qposadr,
                                         int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg, uint8_t *d_labels, int *d_steps,
                                         void *stream) {
  if (!M) return fail("null model");
  if (mode != MGS_MODE_CLUTTER_COLLISION && mode != MGS_MODE_CLUTTER_STABLE) return fail("bad mode");
  if (!d_scenes) return fail("clutter rollouts need the scene state record");
  if (nscene < 1) return fail("nscene must be >= 1");
  CU(cudaSetDevice(M->device));
  RolloutParams prm;
  if (fill_params(M, prm, mode, n, nj, joint_qposadr, base_qposadr, close_ctrl, cfg)) return -1;
  BatchIO io;
  memset(&io, 0, sizeof(io));
  io.pose7 = d_pose7; io.joints = d_joints; io.labels = d_labels; io.steps = d_steps;
  io.state_in = (const real *)d_scenes; io.state_stride = M->state_stride;
  io.scene_index = d_scene_index; io.nscene = nscene;
  if (enough_stable > 0 && n > 0) {  // the model's per-scene counters; launch() zeroes them on the launch stream
    if (nscene > M->scene_cap) {
      CU(cudaDeviceSynchronize());  // an earlier launch may still count into the old array
      if (M->d_scene_success) cudaFree(M->d_scene_success);
      M->d_scene_success = nullptr; M->scene_cap = 0;
      const int cap = (nscene + 255) & ~255;
      CU(cudaMalloc(&M->d_scene_success, (size_t)cap * sizeof(unsigned int)));
      M->scene_cap = cap;
    }
    io.scene_success = M->d_scene_success;
    io.enough_stable = enough_stable;
  }
  return launch(M, prm, io, (cudaStream_t)stream);
}

// one scene, no index, no early stop
extern "C" int mgs_clutter_device(MgsModel *M, int mode, int n, const void *d_scene, const float *d_pose7, const float *d_joints, int nj,
                                  const int *joint_qposadr, int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg,
                                  uint8_t *d_labels, int *d_steps, void *stream) {
  return mgs_clutter_scenes_device(M, mode, n, 1, d_scene, nullptr, 0, d_pose7, d_joints, nj, joint_qposadr, base_qposadr, close_ctrl, cfg,
                                   d_labels, d_steps, stream);
}

static int ensure_stage(MgsModel *M, size_t bytes) {
  if (bytes <= M->stage_bytes) return 0;
  if (M->d_stage) cudaFree(M->d_stage);
  if (M->h_stage) cudaFreeHost(M->h_stage);
  M->d_stage = M->h_stage = nullptr;
  M->stage_bytes = 0;
  CU(cudaMalloc(&M->d_stage, bytes));
  CU(cudaMallocHost(&M->h_stage, bytes));
  M->stage_bytes = bytes;
  return 0;
}

static size_t up256(size_t x) { return (x + 255) & ~size_t(255); }

static int rollout_host(MgsModel *M, int mode, int n, const float *pose7, const float *joints, int nj, const int *joint_qposadr,
                        int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg, uint8_t *labels, int *steps,
                        const double *scene = nullptr, int nscene = 1, const int *scene_index = nullptr, int enough_stable = 0) {
  if (!M) return fail("null model");
  if (n <= 0) return 0;
  if (scene && nscene < 1) return fail("nscene must be >= 1");
  if (scene_index)
    for (int i = 0; i < n; i++)
      if (scene_index[i] < 0 || scene_index[i] >= nscene) return fail("scene_index out of range [0, nscene)");
  CU(cudaSetDevice(M->device));
  const size_t scene_bytes = scene ? (size_t)nscene * M->state_stride * sizeof(real) : 0, index_bytes = scene_index ? (size_t)n * 4 : 0;
  size_t o_pose = 0, o_joint = up256(o_pose + (size_t)n * 7 * 4), o_scene = up256(o_joint + (size_t)n * (nj > 0 ? nj : 1) * 4),
         o_index = up256(o_scene + scene_bytes), o_lab = up256(o_index + index_bytes), o_steps = up256(o_lab + (size_t)n),
         total = up256(o_steps + (size_t)n * 4);
  if (ensure_stage(M, total)) return -1;
  char *h = (char *)M->h_stage, *d = (char *)M->d_stage;
  memcpy(h + o_pose, pose7, (size_t)n * 7 * 4);
  memcpy(h + o_joint, joints, (size_t)n * nj * 4);
  if (scene) { real *sr = (real *)(h + o_scene); for (size_t i = 0; i < (size_t)nscene * M->state_stride; i++) sr[i] = (real)scene[i]; }
  if (scene_index) memcpy(h + o_index, scene_index, index_bytes);
  CU(cudaMemcpyAsync(d + o_pose, h + o_pose, o_lab, cudaMemcpyHostToDevice, M->stream));
  int rc;
  if (scene) rc = mgs_clutter_scenes_device(M, mode, n, nscene, d + o_scene, scene_index ? (const int *)(d + o_index) : nullptr, enough_stable,
                                            (const float *)(d + o_pose), (const float *)(d + o_joint), nj, joint_qposadr, base_qposadr,
                                            close_ctrl, cfg, (uint8_t *)(d + o_lab), (int *)(d + o_steps), M->stream);
  else rc = mgs_rollout_device(M, mode, n, (const float *)(d + o_pose), (const float *)(d + o_joint), nj, joint_qposadr, base_qposadr,
                               close_ctrl, cfg, (uint8_t *)(d + o_lab), (int *)(d + o_steps), M->stream);
  if (rc) return rc;
  CU(cudaMemcpyAsync(h + o_lab, d + o_lab, total - o_lab, cudaMemcpyDeviceToHost, M->stream));
  CU(cudaStreamSynchronize(M->stream));
  memcpy(labels, h + o_lab, (size_t)n);
  if (steps) memcpy(steps, h + o_steps, (size_t)n * 4);
  return 0;
}

extern "C" int mgs_grasp_collision_mask(MgsModel *M, int n, const float *pose7, const float *joints, int nj, const int *joint_qposadr,
                                        int base_qposadr, uint8_t *collision_free_out) {
  return rollout_host(M, MGS_MODE_COLLISION, n, pose7, joints, nj, joint_qposadr, base_qposadr, nullptr, nullptr, collision_free_out, nullptr);
}

extern "C" int mgs_grasp_stability(MgsModel *M, int n, const float *pose7, const float *joints, int nj, const int *joint_qposadr,
                                   int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg, uint8_t *stable_out,
                                   int *steps_out) {
  return rollout_host(M, MGS_MODE_STABILITY, n, pose7, joints, nj, joint_qposadr, base_qposadr, close_ctrl, cfg, stable_out, steps_out);
}

extern "C" int mgs_clutter_collision_mask(MgsModel *M, int n, const double *scene, const float *pose7, const float *joints, int nj,
                                          const int *joint_qposadr, int base_qposadr, uint8_t *collision_free_out) {
  if (!scene) return fail("null scene");
  return rollout_host(M, MGS_MODE_CLUTTER_COLLISION, n, pose7, joints, nj, joint_qposadr, base_qposadr, nullptr, nullptr, collision_free_out,
                      nullptr, scene);
}

extern "C" int mgs_clutter_stable_mask(MgsModel *M, int n, const double *scene, const float *pose7, const float *joints, int nj,
                                       const int *joint_qposadr, int base_qposadr, const double *close_ctrl, const MgsRolloutCfg *cfg,
                                       uint8_t *stable_out, int *steps_out) {
  if (!scene) return fail("null scene");
  return rollout_host(M, MGS_MODE_CLUTTER_STABLE, n, pose7, joints, nj, joint_qposadr, base_qposadr, close_ctrl, cfg, stable_out, steps_out, scene);
}

extern "C" int mgs_clutter_scenes_collision_mask(MgsModel *M, int n, int nscene, const double *scenes, const int *scene_index,
                                                 const float *pose7, const float *joints, int nj, const int *joint_qposadr, int base_qposadr,
                                                 uint8_t *collision_free_out) {
  if (!scenes || !scene_index) return fail("null scenes / scene_index");
  return rollout_host(M, MGS_MODE_CLUTTER_COLLISION, n, pose7, joints, nj, joint_qposadr, base_qposadr, nullptr, nullptr, collision_free_out,
                      nullptr, scenes, nscene, scene_index, 0);
}

extern "C" int mgs_clutter_scenes_stable_mask(MgsModel *M, int n, int nscene, const double *scenes, const int *scene_index, const float *pose7,
                                              const float *joints, int nj, const int *joint_qposadr, int base_qposadr, int enough_stable,
                                              const double *close_ctrl, const MgsRolloutCfg *cfg, uint8_t *stable_out, int *steps_out) {
  if (!scenes || !scene_index) return fail("null scenes / scene_index");
  return rollout_host(M, MGS_MODE_CLUTTER_STABLE, n, pose7, joints, nj, joint_qposadr, base_qposadr, close_ctrl, cfg, stable_out, steps_out,
                      scenes, nscene, scene_index, enough_stable);
}

extern "C" int mgs_step_device(MgsModel *M, int n, int nstep, const void *d_state_in, void *d_state_out, void *d_diag_out, void *stream) {
  if (!M) return fail("null model");
  CU(cudaSetDevice(M->device));
  RolloutParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.mode = MGS_MODE_STEP; prm.n = n; prm.nstep = nstep; prm.qvel_clip = (real)M->qvel_clip;
  BatchIO io;
  memset(&io, 0, sizeof(io));
  io.state_in = (const real *)d_state_in; io.state_out = (real *)d_state_out; io.diag_out = (real *)d_diag_out;
  io.state_stride = M->state_stride; io.diag_stride = M->diag_stride;
  return launch(M, prm, io, (cudaStream_t)stream);
}

extern "C" int mgs_step_host(MgsModel *M, int n, int nstep, const void *state_in, void *state_out, void *diag_out) {
  if (!M) return fail("null model");
  if (n <= 0) return 0;
  CU(cudaSetDevice(M->device));
  size_t sb = (size_t)n * M->state_stride * sizeof(real), db = diag_out ? (size_t)n * M->diag_stride * sizeof(real) : 0;
  size_t o_in = 0, o_out = up256(sb), o_diag = up256(o_out + sb), total = up256(o_diag + db);
  if (ensure_stage(M, total)) return -1;
  char *h = (char *)M->h_stage, *d = (char *)M->d_stage;
  memcpy(h + o_in, state_in, sb);
  CU(cudaMemcpyAsync(d + o_in, h + o_in, sb, cudaMemcpyHostToDevice, M->stream));
  int rc = mgs_step_device(M, n, nstep, d + o_in, d + o_out, diag_out ? d + o_diag : nullptr, M->stream);
  if (rc) return rc;
  CU(cudaMemcpyAsync(h + o_out, d + o_out, total - o_out, cudaMemcpyDeviceToHost, M->stream));
  CU(cudaStreamSynchronize(M->stream));
  memcpy(state_out, h + o_out, sb);
  if (diag_out) memcpy(diag_out, h + o_diag, db);
  return 0;
}
