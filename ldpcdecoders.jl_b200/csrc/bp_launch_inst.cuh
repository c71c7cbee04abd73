// bp_launch_inst.cuh -- body of one (BP_INST_MODE, BP_INST_BIG, BP_VARIANT) translation unit.
#include "bp_launch.h"
#include "bp_kernel.cuh"

#define BP_CAT4(a, b, c, d) a##b##_##c##_##d
#define BP_NAME4(prefix, m, b, v) BP_CAT4(prefix, m, b, v)
#define BP_NAME(prefix, m, b) BP_NAME4(prefix, m, b, BP_VARIANT)

namespace bp {

template <int MAXT, int MINB>
static const void *entry() { return reinterpret_cast<const void *>(bp_persistent_kernel<BP_INST_MODE, BP_INST_BIG != 0, MAXT, MINB>); }

// (the #if blocks keep the absent shapes from being instantiated at all)
const void *const BP_NAME(persistent_kernels_, BP_INST_MODE, BP_INST_BIG)[kShapes] = {
    entry<256, 2>(),
#if !BP_INST_BIG
    entry<384, 2>(),
#else
    nullptr,
#endif
#if BP_INST_MODE == 0
    entry<512, 1>(),
#else
    nullptr,
#endif
#if !BP_INST_BIG && BP_INST_MODE >= 1
    entry<320, 2>(),
#else
    nullptr,
#endif
};

}  // namespace bp
