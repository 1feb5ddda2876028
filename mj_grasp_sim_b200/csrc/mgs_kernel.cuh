// mgs_kernel.cuh - the persistent rollout kernel, instantiated once per translation unit.
// Expects MGS_KERNEL_TAG (w16, w12, wide, wide_g) and MGS_MAX_WARPS_PER_BLOCK to be defined by the including .cu file (MGS_WIDE for
// the environment-per-CTA variants, MGS_ENV_GLOBAL for the one whose environment state lives in global memory).
//
// Launch shape: a persistent grid of (blocks_per_sm x 148) CTAs, each up to MGS_MAX_WARPS_PER_BLOCK warps; every warp
// pulls candidate indices from a global atomic work queue, so warps that finish early (candidates that fail the
// post-close contact test after 3000 of 8000 steps) immediately start the next candidate.
#include "mgs_kernel_ops.h"
#include "mgs_rollout.cuh"

#define MGS_CAT_(a, b) a##b
#define MGS_CAT(a, b) MGS_CAT_(a, b)
#define MGS_STR_(x) #x
#define MGS_STR(x) MGS_STR_(x)
#define MGS_KERNEL MGS_CAT(mgs_rollout_kernel_, MGS_KERNEL_TAG)

#ifdef MGS_WIDE
// environment per CTA: the whole block works on one candidate at a time, pulled from the same global queue
__global__ void __launch_bounds__(MGS_WIDE, 1)
MGS_KERNEL() {
  __shared__ unsigned int s_env;
#ifdef MGS_ENV_GLOBAL
  real *base = IO.env_state + (size_t)blockIdx.x * LY.total;
#else
  real *base = reinterpret_cast<real *>(mgs_smem_raw);
#endif
  Env e;
  for (;;) {
    if (threadIdx.x == 0) s_env = atomicAdd(IO.work_counter, 1u);
    __syncthreads();
    const unsigned int env = s_env;
    __syncthreads();
    if (env >= (unsigned int)PRM.n) break;
    env_bind(e, base);
    run_env_w(e, (int)env);
  }
}
#else
__global__ void __launch_bounds__(MGS_MAX_WARPS_PER_BLOCK * 32, 1)
MGS_KERNEL() {
  real *base = reinterpret_cast<real *>(mgs_smem_raw) + (size_t)(threadIdx.x >> 5) * LY.total;
  const int lane = threadIdx.x & 31;
  Env e;
  for (;;) {
    unsigned int env = 0;
    if (lane == 0) env = atomicAdd(IO.work_counter, 1u);
    env = __shfl_sync(0xffffffffu, env, 0);
    if (env >= (unsigned int)PRM.n) break;
    env_bind(e, base);
    run_env_w(e, (int)env);
  }
  // a warp that runs out of work leaves; exited warps no longer count towards the CTA barrier
}

#endif

namespace {
#ifdef MGS_ENV_GLOBAL
// No dynamic shared memory (the environment's state is in the global slab): the carveout goes to L1, which caches the slab.
// MGS_CARVEOUT=default keeps the driver's choice instead (A/B knob).
cudaError_t ops_prepare(int) {
  const char *c = getenv("MGS_CARVEOUT");
  const int carveout = (c && std::string(c) == "default") ? (int)cudaSharedmemCarveoutDefault : (int)cudaSharedmemCarveoutMaxL1;
  cudaError_t rc = cudaFuncSetAttribute(MGS_KERNEL, cudaFuncAttributePreferredSharedMemoryCarveout, carveout);
  if (rc != cudaSuccess) return rc;
  return cudaFuncSetAttribute(MGS_KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, 0);
}
#else
cudaError_t ops_prepare(int smem_bytes) {
  cudaError_t rc = cudaFuncSetAttribute(MGS_KERNEL, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (rc != cudaSuccess) return rc;
  return cudaFuncSetAttribute(MGS_KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
}
#endif
cudaError_t ops_occupancy(int *blocks_per_sm, int threads, size_t smem_bytes) {
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, MGS_KERNEL, threads, smem_bytes);
}
cudaError_t ops_launch(const KernelConsts *kc, int grid, int threads, size_t smem_bytes, cudaStream_t st) {
  // the constants of this launch (model pointers, layout, parameters, I/O) go to this variant's __constant__ block
  cudaError_t rc = cudaMemcpyToSymbolAsync(c_k, kc, sizeof(KernelConsts), 0, cudaMemcpyHostToDevice, st);
  if (rc != cudaSuccess) return rc;
  MGS_KERNEL<<<grid, threads, smem_bytes, st>>>();
  return cudaGetLastError();
}
#ifdef MGS_WIDE
const MgsKernelOps g_ops = {1, MGS_WIDE, "mgs_rollout_kernel_" MGS_STR(MGS_KERNEL_TAG), ops_prepare, ops_occupancy, ops_launch};
#else
const MgsKernelOps g_ops = {MGS_MAX_WARPS_PER_BLOCK, 32, "mgs_rollout_kernel_" MGS_STR(MGS_KERNEL_TAG), ops_prepare, ops_occupancy, ops_launch};
#endif
}  // namespace

const MgsKernelOps *MGS_CAT(mgs_kernel_ops_, MGS_KERNEL_TAG)() { return &g_ops; }
