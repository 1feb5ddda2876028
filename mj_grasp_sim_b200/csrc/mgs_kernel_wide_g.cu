// mgs_kernel_wide_g.cu - the environment-per-CTA variant with the environment's state in a global-memory slab instead of shared
// memory (same source as mgs_kernel_wide.cu): for scenes whose state is larger than one CTA's shared memory (the fp64 Shadow hand
// over a cluttered table, escalation capacities of clutter scenes); see mgs_sim.cuh (MGS_ENV_GLOBAL) and mgs_kernel_ops.h
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string>
#define MGS_WIDE 256
#define MGS_ENV_GLOBAL 1
#define MGS_MAX_WARPS_PER_BLOCK 8
#define MGS_KERNEL_TAG wide_g
#include "mgs_kernel.cuh"
