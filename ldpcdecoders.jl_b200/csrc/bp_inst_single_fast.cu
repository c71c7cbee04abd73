#define BP_VARIANT 2
#include "bp_single_inst.cuh"
