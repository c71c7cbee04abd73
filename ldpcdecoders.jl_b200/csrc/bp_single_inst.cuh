// bp_single_inst.cuh -- body of one BP_VARIANT translation unit of the node-parallel small-batch kernel and the
// grid-wide kernel (bp_single.cuh).
#include "bp_single.cuh"

#define BPN_CAT(a, v) a##v
#define BPN_NAME2(prefix, v) BPN_CAT(prefix, v)
#define BPN_NAME(prefix) BPN_NAME2(prefix, BP_VARIANT)

namespace bp {

const SingleKernels BPN_NAME(single_kernels_) = {
    reinterpret_cast<const void *>(bp_node_parallel_kernel<kSingleThreads>),
    reinterpret_cast<const void *>(bp_grid_kernel<kGridThreads>),
};

}  // namespace bp
