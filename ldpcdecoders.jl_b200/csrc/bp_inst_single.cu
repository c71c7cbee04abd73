#define BP_VARIANT 0
#include "bp_single_inst.cuh"
