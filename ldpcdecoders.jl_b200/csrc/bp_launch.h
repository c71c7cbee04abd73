// bp_launch.h -- entry points of the batch BP kernels.  Each variant's instantiations live in their own translation
// units so that they compile in parallel: one per (MODE, BIG) pair of the persistent kernel (bp_launch_inst.cuh) and
// one for the shared-memory-resident kernel (bp_smem_inst.cuh).  The host sets attributes and launches through these
// tables (ldpcb200.cu).
#pragma once
#include <cuda_runtime.h>

#include "bp_filter.cuh"

namespace bp {

// Launch shapes: (threads <= 256, 2 CTAs/SM, <= 128 regs), (<= 384, 2 CTAs/SM, <= 80 regs; not for
// the local-memory degree path), (<= 512, 1 CTA/SM, <= 128 regs; mode 0 only).
// (<= 320, 2 CTAs/SM, <= 96 regs; HBM modes only: ten warps without the spills of the 80-register shape)
enum KernelShape { kShape256x2 = 0, kShape384x2 = 1, kShape512x1 = 2, kShape320x2 = 3, kShapes = 4 };

// bp_persistent_kernel<M, B, ...> by KernelShape for memory mode M, degree path B (1 = local-memory degrees),
// variant V; nullptr where no instantiation exists
#define BP_DECLARE_MODE(M, B, V) extern const void *const persistent_kernels_##M##_##B##_##V[kShapes];
BP_DECLARE_MODE(0, 0, 0) BP_DECLARE_MODE(0, 1, 0) BP_DECLARE_MODE(1, 0, 0) BP_DECLARE_MODE(1, 1, 0) BP_DECLARE_MODE(2, 0, 0) BP_DECLARE_MODE(2, 1, 0)
BP_DECLARE_MODE(0, 0, 1) BP_DECLARE_MODE(1, 0, 1) BP_DECLARE_MODE(2, 0, 1)
BP_DECLARE_MODE(0, 0, 2) BP_DECLARE_MODE(1, 0, 2) BP_DECLARE_MODE(2, 0, 2)
#undef BP_DECLARE_MODE

// bp_smem_kernel of one variant: [KernelShape or kSmemDual][eb64], and the phase-timing builds (option kernel_profile)
// of the 256 x 2 shape and of the dual-team form without eb64 (nullptr elsewhere: the normal kernel runs there)
constexpr int kSmemDual = kShapes;          // dual-team form: one CTA of 2 x W warps per SM
struct SmemKernels {
    const void *kernel[kShapes + 1][2];
    const void *prof[kShapes + 1];
};
#define BP_DECLARE_SMEM(V)                  \
    extern const SmemKernels smem_kernels_##V; \
    cudaError_t filter_setup_##V(const FilterSetup &q, cudaStream_t st);
BP_DECLARE_SMEM(0) BP_DECLARE_SMEM(1) BP_DECLARE_SMEM(2)
#undef BP_DECLARE_SMEM

}  // namespace bp
