/*
 * ldpcb200.h -- C ABI of libldpcb200.so, the B200-native belief-propagation decoder that
 * stands behind LDPCDecoders.jl's BeliefPropagationDecoder / decode! / batchdecode!.
 *
 * The reference has no FFI layer (it is pure Julia); the entry points below are what a
 * Julia `ccall` shim for this path binds.  Each one cites the reference interface it
 * replaces (paths relative to /root/reference/).  INTEGRATION.md shows the Julia-side stub.
 *
 * Conventions
 *   - every function returns 0 on success, a nonzero LDPCB200_E* code otherwise; nothing
 *     throws or aborts; ldpcb200_last_error() gives a thread-local message.
 *   - the caller owns every host buffer for the duration of the call (Julia: GC.@preserve);
 *     the library owns all device memory, streams and events inside the handle.
 *   - one in-flight call per handle (the reference decoder is non-reentrant too: shared
 *     scratch, src/decoders/belief_propagation.jl:125); different handles are independent.
 *   - there is NO CPU fallback: without a usable CUDA device ldpcb200_create fails.
 */
#ifndef LDPCB200_H
#define LDPCB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ldpcb200 ldpcb200_t;

/* error codes */
#define LDPCB200_OK            0
#define LDPCB200_EINVAL        1   /* bad argument (shape, format, null pointer, unsorted CSC ...) */
#define LDPCB200_ECUDA         2   /* CUDA runtime error, see ldpcb200_last_error() */
#define LDPCB200_ENODEVICE     3   /* no CUDA device / requested device missing */
#define LDPCB200_EUNSUPPORTED  4   /* e.g. node degree above LDPCB200_MAX_DEGREE */
#define LDPCB200_ENOMEM        5

#define LDPCB200_MAX_DEGREE  128   /* largest check / variable degree the kernels accept */
#define LDPCB200_MAX_EDGES   8388607 /* nnz(H) limit: edge slot * 256 B must stay below 2^31 */

/* element formats of host matrices at the boundary (column = one syndrome / one error vector,
 * exactly the shapes batchdecode! takes: belief_propagation.jl:220, test_bp_decoder.jl:24-26) */
#define LDPCB200_FMT_U8       0   /* column-major bytes 0/1: Matrix{Bool}, Matrix{UInt8}; ld in elements */
#define LDPCB200_FMT_I64      1   /* column-major int64 0/1: Matrix{Int} (test_bp_decoder.jl:24) */
#define LDPCB200_FMT_BITS     2   /* Julia BitMatrix chunks: bit (c*rows + r) of a little-endian bit stream; ld ignored */
#define LDPCB200_FMT_PACKED32 3   /* native: one row of ceil(rows/32) uint32 per column, bit r%32 of word r/32; ld ignored */
#define LDPCB200_FMT_F64      4   /* column-major Float64 0.0/1.0 (scratch.err, belief_propagation.jl:17,187); outputs only */

/* kernel variants */
#define LDPCB200_VARIANT_EXACT  0 /* FP64 likelihood-ratio sum-product, op-for-op with belief_propagation.jl:135-178 */
#define LDPCB200_VARIANT_MINSUM 1 /* min-sum on FP64 log-likelihood ratios; NO reference equivalent (the package's BP is
                                     sum-product): a faster, non-bit-compatible option.  Same schedule, early stop and
                                     outputs; posterior_ratio then carries the posterior LLR log(P0/P1). */
#define LDPCB200_VARIANT_FAST32 2 /* FP32 tanh/atanh sum-product on log-likelihood ratios with the special-function unit (MUFU
                                     EX2 / RCP / LG2); the clamped textbook form of bpots_decoder.jl:182-211 on the BP decoder's
                                     schedule.  Fast, NOT bit-compatible with the reference: judged by mismatch rate and logical
                                     error rate against the exact variant (bench.py reports both).  posterior_ratio = posterior LLR. */

/* kernel families (ldpcb200_info_t.family, option "family") */
#define LDPCB200_FAMILY_AUTO   0
#define LDPCB200_FAMILY_SMEM   1  /* persistent kernel, messages resident in shared memory, lane = syndrome */
#define LDPCB200_FAMILY_GLOBAL 2  /* same kernel, messages (and for very large codes state/tables) in HBM/L2 */

typedef struct {
    int64_t s, n, E;            /* checks, variables, edges (nnz of H) */
    int32_t max_check_degree, max_var_degree;
    int32_t family;             /* LDPCB200_FAMILY_* actually selected */
    int32_t ndev;               /* devices the batch is sharded over */
    int32_t sm_count;           /* SMs of device 0 */
    int32_t ctas_per_sm;        /* family SMEM: resident CTAs per SM */
    int32_t threads_per_cta;
    int32_t smem_bytes;         /* dynamic shared memory per CTA (family SMEM) */
    int32_t slots;              /* resident syndrome slots per device (32 x resident CTAs) */
    int32_t syn_words, err_words; /* uint32 words per packed syndrome / error row */
    int64_t message_bytes;      /* device bytes of the message store per device (family GLOBAL) */
    int32_t kernel_mode;        /* 0: all in shared memory, 1: messages in HBM/L2, 2: messages + state + tables in HBM/L2 */
    int32_t prefetch_distance;  /* cp.async ring depth of modes 1/2 (0 = messages read directly) */
    int32_t kernel_rev;         /* 2: round-2 shared-memory kernel (bp_smem.cuh); 3: the same kernel with two teams per CTA taking turns
                                   in the check pass (option "dual" = 1); 1: the general persistent kernel (bp_kernel.cuh, option "lean" = 0) */
    int32_t counters_via_nccl;  /* 1: the per-device counters of a multi-device handle are summed with ncclAllReduce */
    int64_t bpots_workspace_bytes; /* device bytes of the BP-OTS workspace of device 0 (codes beyond shared memory; allocated by
                                      the first BP-OTS call that needs it, 0 before) */
} ldpcb200_info_t;

/* counters[] layout of the decode calls (summed over all devices of the handle) */
#define LDPCB200_CTR_DECODED     0  /* syndromes decoded */
#define LDPCB200_CTR_CONVERGED   1  /* of which converged */
#define LDPCB200_CTR_ITERATIONS  2  /* sum of executed BP iterations */
#define LDPCB200_CTR_FILTERED    3  /* of which finished by the first-iteration filter (1 iteration each, no messages) */
#define LDPCB200_NUM_COUNTERS    4

/* OSD-0 statistics (ldpcb200_bposd_decode_batch / ldpcb200_osd0_device) */
#define LDPCB200_OSD_PROCESSED   0  /* syndromes that went through OSD-0 (= BP did not converge) */
#define LDPCB200_OSD_PIVOTS      1  /* sum of pivots taken */
#define LDPCB200_OSD_COLUMNS     2  /* sum of sorted columns visited before the target vanished */
#define LDPCB200_NUM_OSD_STATS   3

const char *ldpcb200_last_error(void);
int ldpcb200_version(void);
int ldpcb200_device_count(int32_t *out);

/* Replaces the constructor BeliefPropagationDecoder(H, per, max_iters)
 * (src/decoders/belief_propagation.jl:61-67): takes sparse_H's CSC arrays
 * (colptr n+1, rowval E, row indices ascending inside a column -- the SparseMatrixCSC invariant)
 * and builds the device-resident Tanner graph once.  index_base = 1 for Julia arrays, 0 for C.
 * devices/ndev: shard set (NULL/0 -> device 0).  Messages need no reset between calls
 * (reset!, belief_propagation.jl:83-91, becomes a no-op). */
int ldpcb200_create(int64_t s, int64_t n, const int64_t *colptr, const int64_t *rowval,
                    int32_t index_base, double per, int32_t max_iters, int32_t variant,
                    const int32_t *devices, int32_t ndev, ldpcb200_t **out);
int ldpcb200_destroy(ldpcb200_t *h);
int ldpcb200_info(const ldpcb200_t *h, ldpcb200_info_t *out);

/* Tunables, set before the first decode (all optional):
 *   "family" (LDPCB200_FAMILY_*), "warps" (warps per CTA), "prefetch" (cp.async prefetch distance of the
 *   HBM modes, 0..3), "lean" (family SMEM: 1 = round-2 kernel where the code fits its envelope (default),
 *   0 = always the general persistent kernel),
 *   "minsum_scale_permille" (min-sum variant: normalisation factor x 1000, default 875),
 *   "early_stop" (1 = reference semantics, default; 0 = always run max_iters -- benchmarking only,
 *   outputs are then those of the last iteration), "chunk" (syndromes per host<->device chunk),
 *   "small_batch" (batches of at most this many syndromes run on the node-parallel kernel, one CTA per syndrome:
 *   the low-latency path of decode!; -1 = number of SMs (default), 0 = never),
 *   "osd_order" (ldpcb200_bposd_decode_batch and the sampling harness: 0 (default) = OSD-0 on the syndromes BP left
 *   unconverged; 1..12 = the order-O exhaustive search of belief_propagation_osd.jl:127-209 on EVERY syndrome, as the
 *   reference's decode! does for osd_order > 0),
 *   "ratio_last_only" (ldpcb200_decode_device writes d_posterior_ratio only in iteration max_iters: all an OSD
 *   stage needs, since it only reads the ratios of syndromes that did not converge; default 0),
 *   "grid_kernel" (1, default: small batches of codes whose messages exceed one SM's shared memory run on the grid-wide
 *   cooperative kernel, one syndrome at a time over all SMs; 0 = persistent kernel),
 *   "first_iteration_filter" (1, default: family SMEM evaluates iteration 1 of every syndrome from per-variable truth
 *   tables and decodes only the syndromes that did not converge there; results are identical either way),
 *   "ring_mult" (HBM modes: ring slot = this many times the rows of the widest node, i.e. nodes per loop trip; 0 = auto),
 *   "overlap_chunks" (host batches on the shared-memory kernel: decoding kernels of consecutive chunks may overlap; 1, default:
 *   with pinned buffers and BitMatrix output, or once the previous batch averaged >= 2 iterations per syndrome; 0 never;
 *   2 always), "direct_bits" (1, default: with BitMatrix output the shared-memory kernel writes the caller's bit stream itself),
 *   "dynamic_queue" (1, default: the CTAs of the persistent kernels claim 32-syndrome chunks of the batch from a global
 *   counter; 0 = static shares c, c+G, ...),
 *   "stage_pageable" (1, default: pageable host buffers are staged through pinned blocks), "nccl" (1, default: a
 *   multi-device handle sums its counters with ncclAllReduce), "time_kernels" (see ldpcb200_kernel_time),
 *   "kernel_profile" (see ldpcb200_kernel_profile), "osd_profile"; experiments that measured no gain and stay off:
 *   "dual" (two teams per CTA), "max_ctas_per_sm";
 *   "contiguous_variables" (1, default: the shared-memory kernel gives every warp a contiguous block of variables where the
 *   code has a uniform variable degree; 0 = round-robin ownership),
 *   "bpots_memory" (where BP-OTS keeps the 16 E + 23 n + 4 s bytes of per-syndrome arrays: 0, default = shared memory when
 *   they fit, otherwise a per-device workspace in global memory with one slice per resident CTA; 1 = shared memory only,
 *   LDPCB200_EUNSUPPORTED when they do not fit; 2 = always the global workspace.  Outputs are bit-identical either way). */
int ldpcb200_set_option(ldpcb200_t *h, const char *key, int64_t value);

/* Replaces batchdecode!(decoder, syndromes, errors, success)
 * (src/decoders/belief_propagation.jl:220-231; 3-argument form abstract_decoder.jl:44-48) and,
 * with B = 1, decode!(decoder, syndrome) (belief_propagation.jl:121-188).
 *   syndromes : s x B host matrix in syn_fmt (syn_ld = leading dimension in elements for U8/I64)
 *   errors    : n x B host matrix in err_fmt, overwritten (errors[:, i] .= guess, :227)
 *   converged : B bytes (Julia Vector{Bool}), overwritten (success[i] = conv, :226)
 *   iters     : nullable, B int32 -- executed iterations per syndrome
 *   posterior_ratio : nullable, n x B column-major doubles R_j = P(e_j=1)/P(e_j=0) after the
 *               last executed iteration; scratch.log_probabs[j] = log(1/R_j) (belief_propagation.jl:163),
 *               which is what BeliefPropagationOSDDecoder reads (belief_propagation_osd.jl:52)
 *   counters  : nullable, LDPCB200_NUM_COUNTERS int64
 * Blocks until all outputs are in host memory. */
int ldpcb200_decode_batch(ldpcb200_t *h, int64_t B,
                          const void *syndromes, int32_t syn_fmt, int64_t syn_ld,
                          void *errors, int32_t err_fmt, int64_t err_ld,
                          uint8_t *converged, int32_t *iters, double *posterior_ratio,
                          int64_t *counters);

/* Same decode with inputs/outputs already resident on one device of the handle, native packed
 * format (LDPCB200_FMT_PACKED32).  Asynchronous on `stream` (a cudaStream_t; NULL = the handle's
 * own stream).  d_counters: nullable device pointer to LDPCB200_NUM_COUNTERS uint64 that the
 * kernels ADD to.  Used by the device-resident benchmark and by sample->decode->score loops. */
int ldpcb200_decode_device(ldpcb200_t *h, int32_t dev_slot, int64_t B,
                           const uint32_t *d_syn_words, uint32_t *d_err_words,
                           uint8_t *d_converged, int32_t *d_iters, double *d_posterior_ratio,
                           unsigned long long *d_counters, void *stream);

/* Replaces decode!(::BeliefPropagationOSDDecoder, syndrome) with osd_order = 0
 * (src/decoders/belief_propagation_osd.jl:49-61, osd(..., Val(0)) :63-125), applied to every column of a
 * batch: BP as ldpcb200_decode_batch, then OSD-0 on the syndromes BP left unconverged (the reference returns
 * BP's own decision for the converged ones, :72-74); with option "osd_order" = O > 0, osd(..., Val{O}) (:127-209) on every
 * column instead.  errors receives the OSD result, converged BP's flag
 * (:60 returns BP's `converged`).  osd_stats: nullable, LDPCB200_NUM_OSD_STATS int64.  Exact variant only;
 * the bit-packed s x (n+1) matrix must fit in shared memory (LDPCB200_EUNSUPPORTED otherwise).
 * Sort key: max(r, 1-r) with r = RN(1/R_j) where the reference has exp(log(1/R_j)) (see DESIGN.md 3.4). */
int ldpcb200_bposd_decode_batch(ldpcb200_t *h, int64_t B,
                                const void *syndromes, int32_t syn_fmt, int64_t syn_ld,
                                void *errors, int32_t err_fmt, int64_t err_ld,
                                uint8_t *converged, int32_t *iters, int64_t *counters, int64_t *osd_stats);

/* Replaces decode!(::BPOTSDecoder, syndrome) (src/decoders/bpots_decoder.jl:226-340; constructor BPOTSDecoder(H, per, max_iters;
 * T = 9, C = 2.0) :90-111) applied to every column of a batch, which is what the generic batchdecode! (abstract_decoder.jl:31-42)
 * does with it.  The handle supplies H, per and max_iters (its variant is irrelevant: BP-OTS has its own Float64 LLR-domain
 * tanh/atanh updates, depolarising prior log((1 - 2 per/3)/(2 per/3)), oscillation counting, best-so-far tracking and bias -C every
 * T iterations).  errors receives best_decisions, converged the flag decode! returns, iters (nullable) the executed iterations.
 * One CTA per syndrome; its arrays live in shared memory or in the global workspace (option "bpots_memory").
 * tanh / atanh / log are CUDA's where the reference uses Julia's: outcomes agree except where a last-bit difference gets amplified. */
int ldpcb200_bpots_decode_batch(ldpcb200_t *h, int64_t B,
                                const void *syndromes, int32_t syn_fmt, int64_t syn_ld,
                                void *errors, int32_t err_fmt, int64_t err_ld,
                                uint8_t *converged, int32_t *iters, int32_t T, double C);

/* The same BP-OTS decode on buffers already resident on one device of the handle, native packed rows
 * (LDPCB200_FMT_PACKED32): d_syn_words [B][syn_words], d_err_words [B][err_words] receives best_decisions, d_converged
 * B bytes, d_iters nullable B int32.  d_counters: nullable device pointer to LDPCB200_NUM_COUNTERS uint64; the kernel ADDS
 * the decoded syndromes, converged ones and executed iterations to [LDPCB200_CTR_DECODED / _CONVERGED / _ITERATIONS].
 * Asynchronous on `stream` (a cudaStream_t; NULL = the handle's own stream).  One in-flight call per handle applies in
 * full here: codes beyond shared memory decode in a workspace shared by all BP-OTS calls on the device, so a call must have
 * completed on its stream before another BP-OTS call of the handle is issued on a different stream. */
int ldpcb200_bpots_device(ldpcb200_t *h, int32_t dev_slot, int64_t B,
                          const uint32_t *d_syn_words, uint32_t *d_err_words,
                          uint8_t *d_converged, int32_t *d_iters, unsigned long long *d_counters,
                          int32_t T, double C, void *stream);

/* The OSD-0 stage alone on device-resident buffers (native packed rows), after ldpcb200_decode_device with a
 * posterior-ratio output: d_err_words holds BP's decisions on entry and the OSD result on return;
 * d_posterior_ratio is [B][n].  d_stats: nullable device pointer to LDPCB200_NUM_OSD_STATS uint64 the kernel
 * ADDS to (8 uint64 when the option "osd_profile" is set: [3..7] then receive SM cycles of the kernel's sort /
 * build / pivot search / row update / solve phases).  Asynchronous on `stream`. */
int ldpcb200_osd0_device(ldpcb200_t *h, int32_t dev_slot, int64_t B,
                         const uint32_t *d_syn_words, uint32_t *d_err_words, const uint8_t *d_converged,
                         const double *d_posterior_ratio, unsigned long long *d_stats, void *stream);

/* Harness helpers (pattern of test/test_bp_decoder.jl:19-30 moved on-device).
 * sample: i.i.d. Bernoulli(per) errors from Philox4x32-10 keyed by the global syndrome index
 * (first .. first+B-1) and their syndromes H*e mod 2, both in packed rows.
 * score : counts rows where decoded == true error (out[0]) and rows whose decoded error
 * reproduces the syndrome (out[1]); ADDS into d_out[2] (uint64). */
int ldpcb200_sample_device(ldpcb200_t *h, int32_t dev_slot, int64_t B, int64_t first,
                           uint64_t seed, double per,
                           uint32_t *d_true_err_words, uint32_t *d_syn_words, void *stream);
int ldpcb200_score_device(ldpcb200_t *h, int32_t dev_slot, int64_t B,
                          const uint32_t *d_true_err_words, const uint32_t *d_err_words,
                          const uint32_t *d_syn_words, unsigned long long *d_out, void *stream);

/* Logical operators for failure counting: L is k x n over GF(2), k <= 64, given like H by its CSC arrays.  A decoded error
 * e' fails on the true error e when H*e' != syndrome or L*(e xor e') != 0.  k = 0 removes them (failure = e' != e, the
 * criterion of test/test_bp_decoder.jl:27-28). */
int ldpcb200_set_logicals(ldpcb200_t *h, int64_t k, const int64_t *colptr, const int64_t *rowval, int32_t index_base);

/* ldpcb200_score_device with failure counting: ADDS into d_out[4] (uint64): [0] exact matches, [1] rows whose decoded error
 * reproduces the syndrome, [2] failures (see ldpcb200_set_logicals), [3] total weight of e xor e'. */
int ldpcb200_score_logical_device(ldpcb200_t *h, int32_t dev_slot, int64_t B, const uint32_t *d_true_err_words,
                                  const uint32_t *d_err_words, const uint32_t *d_syn_words, unsigned long long *d_out,
                                  void *stream);

/* Prior of an existing handle (channel_probs of belief_propagation.jl:8,89): lets an error-rate sweep reuse the
 * device-resident Tanner graph.  Same rules as the `per` of ldpcb200_create. */
int ldpcb200_set_per(ldpcb200_t *h, double per);

/* The sampling + scoring harness (SURVEY 8(f) rank 2; pattern of test/test_bp_decoder.jl:19-30 with the batch generated where it
 * is decoded): `shots` i.i.d. Bernoulli(per_channel) errors from the Philox stream (seed, global indices first ..
 * first+shots-1), their syndromes, BP with the handle's prior and max_iters (followed by OSD-0 on the unconverged ones when
 * osd != 0), scoring against the true errors -- sharded over the handle's devices in device-resident tiles; nothing but the
 * counters crosses PCIe.  The per-device counters are summed with one ncclAllReduce when the handle has communicators, else
 * on the host.  out[8]: [0] shots decoded, [1] converged, [2] BP iterations, [3] exact matches, [4] syndrome satisfied,
 * [5] failures (logical failures when logical operators are set), [6] weight of e xor e', [7] syndromes sent to OSD-0. */
#define LDPCB200_NUM_HARNESS_COUNTERS 8
int ldpcb200_sample_decode_score(ldpcb200_t *h, int64_t shots, int64_t first, uint64_t seed, double per_channel,
                                 int32_t osd, int64_t *out);

/* The same harness with BP-OTS (ldpcb200_bpots_decode_batch's decoder, biasing period T and constant C) in place of BP:
 * same sampling, tiles, device shards, scoring and counter summation.  out[8] as above, with [2] the BP-OTS iterations and
 * [7] = 0. */
int ldpcb200_sample_bpots_score(ldpcb200_t *h, int64_t shots, int64_t first, uint64_t seed, double per_channel,
                                int32_t T, double C, int64_t *out);

/* Self-test of the kernels' branch-free division sequences against the stock IEEE routines
 * (__drcp_rn / __ddiv_rn) on n pseudo-random operands of envelope `mode` (0: t = 2/(1+q)-1,
 * 1: r = (1-x)/(1+x)).  mismatches[4]: [0] node map vs stock IEEE form, [1] refined reciprocal vs
 * __drcp_rn, [2] __drcp_rn vs __ddiv_rn(1,d), [3] bits of one offending operand; [0..2] must come
 * back 0.  Test hook, not part of the decode path. */
int ldpcb200_selftest_division(int32_t device, int32_t mode, uint64_t n, uint64_t seed, uint64_t *mismatches);

/* Phase timing of the shared-memory kernel (option "kernel_profile" = 1 before the decodes): out8 receives SM cycles
 * summed over all warps since the last reset -- [0] check pass, [1] wait at the barrier after it, [2] variable pass,
 * [3] residual-syndrome updates of flipped decisions, [4] wait at the second barrier, [5] syndrome re-check + outputs,
 * [6] refill -- and [7] the number of warp-iterations.  Synchronises the device.  Diagnostics, not part of the path. */
int ldpcb200_kernel_profile(ldpcb200_t *h, int32_t dev_slot, int64_t *out8, int32_t reset);

/* Duration of the decoding kernel itself (option "time_kernels" = 1 before the decodes): every launch of the persistent
 * BP kernel is bracketed by CUDA events on the stream it is launched on; ms receives the sum of the elapsed times and
 * launches their number since the last reset.  Synchronises the device.  bench.py's roofline uses it (the kernel's
 * own time, not the step's).  Diagnostics, not part of the path. */
int ldpcb200_kernel_time(ldpcb200_t *h, int32_t dev_slot, double *ms, int64_t *launches, int32_t reset);

/* Number of kernels of this library launched through the handle so far (bench bookkeeping). */
int ldpcb200_launch_count(const ldpcb200_t *h, int64_t *out);

#ifdef __cplusplus
}
#endif
#endif /* LDPCB200_H */
