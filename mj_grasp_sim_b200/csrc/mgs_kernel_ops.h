// mgs_kernel_ops.h - host-side handle of one compiled variant of the rollout kernel.
//
// The same kernel source is compiled more than once with different launch bounds (one translation unit per variant):
// 16 warps per CTA caps the kernel at 128 registers per thread, which the small models need to keep 14-16
// environments resident per SM; models that fit at most 12 environments per SM (Robotiq, VX300 at default capacities,
// the 16-dof hands, clutter scenes) run the 12-warp variant, which may use 168 registers (fewer spills, +4 % on Robotiq).
#pragma once
#include <cuda_runtime.h>

struct KernelConsts;

struct MgsKernelOps {
  int max_warps;      // environments per CTA at most (warp variants: one warp each; wide variant: 1)
  int lanes_per_env;  // threads that share one environment: 32, or MGS_WIDE for the environment-per-CTA variant
  const char *name;
  cudaError_t (*prepare)(int smem_bytes);                                   // carve-out + max dynamic shared memory
  cudaError_t (*occupancy)(int *blocks_per_sm, int threads, size_t smem_bytes);
  cudaError_t (*launch)(const KernelConsts *kc, int grid, int threads, size_t smem_bytes, cudaStream_t st);
};

const MgsKernelOps *mgs_kernel_ops_w16();
const MgsKernelOps *mgs_kernel_ops_w12();
// environment per CTA (csrc/mgs_kernel_wide.cu): scenes whose state leaves room for fewer than MGS_WIDE_BELOW_ENVS
// warp-environments per SM (Shadow hand in 10-object clutter: one)
const MgsKernelOps *mgs_kernel_ops_wide();
// the same with the environment's state in a global-memory slab (csrc/mgs_kernel_wide_g.cu): scenes whose state does not fit one CTA's
// shared memory at all (fp64 Shadow hand over four or more clutter objects, clutter escalation capacities); mgs_model_create_any only
const MgsKernelOps *mgs_kernel_ops_wide_g();
#define MGS_WIDE_BELOW_ENVS 4
