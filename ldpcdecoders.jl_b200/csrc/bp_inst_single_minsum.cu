#define BP_VARIANT 1
#include "bp_single_inst.cuh"
