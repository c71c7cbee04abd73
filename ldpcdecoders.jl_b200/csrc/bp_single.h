// bp_single.h -- host-visible part of the node-parallel small-batch kernel (bp_single.cuh).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bp {

struct SingleParams {
    int s, n, E, SW, NW, max_iters, early_stop, regular_p0, ratio_last_only;
    double p0;         // prior ratio p/(1-p); min-sum variant: prior log-likelihood ratio
    double check_aux;  // min-sum variant: normalisation factor
    long long B;
    const int *rowptr, *colptr, *ve_slot, *ve_chk;
    const uint32_t *syn_words;
    uint32_t *err_words;
    uint8_t *conv;
    int32_t *iters;
    double *ratio;
    unsigned long long *counters;
    int off_syn, off_resid, off_dec;      // shared-memory byte offsets behind the E message slots
};

// the grid-wide form (bp_grid_kernel): one syndrome at a time over all CTAs of a cooperative launch, messages in global memory
struct GridParams {
    int s, n, E, SW, NW, max_iters, early_stop, regular_p0, ratio_last_only;
    double p0, check_aux;
    long long B;
    const int *rowptr, *colptr, *ve_slot, *ve_chk;
    const uint32_t *syn_words;
    uint32_t *err_words;
    uint8_t *conv;
    int32_t *iters;
    double *ratio;
    unsigned long long *counters;
    double *msg;            // [E]
    uint32_t *resid, *dec;  // [SW], [NW]
    int *work;              // [2] unsatisfied checks of even / odd syndromes (zero on entry and on exit)
    unsigned int *bar;      // [2] barrier counters (zero on entry and on exit)
};
constexpr int kGridThreads = 256;
constexpr int kSingleThreads = 512;

// Entry points of one variant's bp_node_parallel_kernel<kSingleThreads> and bp_grid_kernel<kGridThreads>
// (bp_single_inst.cuh).  The grid kernel needs a cooperative launch with no more CTAs than can be co-resident.
struct SingleKernels {
    const void *node_parallel, *grid;
};
extern const SingleKernels single_kernels_0, single_kernels_1, single_kernels_2;   // exact, min-sum, fast FP32 variant

}  // namespace bp
