// bp_smem_inst.cuh -- body of one BP_VARIANT translation unit of the shared-memory-resident kernel (bp_smem.cuh).
#define BP_FILTER_SETUP 1      // (before the first inclusion of bp_filter.cuh, which bp_launch.h pulls in)
#include "bp_launch.h"
#include "bp_smem.cuh"

#define BPS_CAT(a, v) a##v
#define BPS_NAME2(prefix, v) BPS_CAT(prefix, v)
#define BPS_NAME(prefix) BPS_NAME2(prefix, BP_VARIANT)

namespace bp {

template <int MAXT, int MINB, bool EB64, bool PROF = false, bool DUAL = false>
static const void *entry() { return reinterpret_cast<const void *>(bp_smem_kernel<MAXT, MINB, EB64, PROF, DUAL>); }

const SmemKernels BPS_NAME(smem_kernels_) = {
    {{entry<256, 2, false>(), entry<256, 2, true>()},
     {entry<384, 2, false>(), entry<384, 2, true>()},
     {entry<512, 1, false>(), entry<512, 1, true>()},
     {nullptr, nullptr},                                                          // kShape320x2: HBM modes only
     {entry<512, 1, false, false, true>(), entry<512, 1, true, false, true>()}},  // kSmemDual
    {entry<256, 2, false, true>(), nullptr, nullptr, nullptr, entry<512, 1, false, true, true>()},
};

// ---- tables of the first-iteration filter, computed with this variant's node updates (bp_filter.cuh)
cudaError_t BPS_NAME(filter_setup_)(const FilterSetup &q, cudaStream_t st)
{
    first_iter_check_table_kernel<<<1, 32, 0, st>>>(q);
    first_iter_truth_table_kernel<<<(q.n + 127) / 128, 128, 0, st>>>(q);
    return cudaGetLastError();
}

}  // namespace bp
