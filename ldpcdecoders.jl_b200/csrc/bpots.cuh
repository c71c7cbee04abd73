// bpots.cuh -- BP-OTS decoder (SURVEY.md section 8(f) rank 3): decode!(::BPOTSDecoder, syndrome) of
// /root/reference/src/decoders/bpots_decoder.jl:226-340 with its message updates (:161-211) and beliefs (:113-129).
//
// A different algorithm from the BP decoder: Float64 log-likelihood ratios, tanh/atanh check update with the clamps of
// :186-206, depolarising prior log((1 - 2p/3)/(2p/3)) (:231), oscillation counters, best-so-far tracking by
// (syndrome mismatch, weight) and a bias of -C on the most oscillating / least certain variables every T iterations
// (:294-336).  The bias step is a sequential arg-max per syndrome, so the mapping is one CTA per syndrome with threads
// over the nodes (as bp_single.cuh), block-wide lexicographic reductions for the two arg-max selections.  The per-syndrome
// arrays (both message arrays, node state, decisions) live in shared memory when they fit (GLOBAL = false); otherwise
// (GLOBAL = true) each resident CTA works in its own slice of a device workspace, with the same layout and the same
// operations in the same order, so both instantiations return bit-identical outputs.  The reduction scratch is in shared
// memory either way.  Summation and product orders follow the reference (neighbour order, from 0.0 / 1.0), so
// given equal tanh/atanh/log values every discrete outcome is the reference's; those three functions are CUDA's here,
// Julia's there (see oracle/bpots_oracle.c on what that means for parity).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bp {

struct BpotsParams {
    int s, n, E, SW, NW, max_iters, T;
    double prior, C;                 // Pi = log((1 - 2p/3)/(2p/3)), bias constant
    long long B;
    const int *rowptr, *colptr, *ve_slot, *ve_chk;   // CSR check -> slots, CSC variable -> edges, slot / check of each CSC edge
    const uint32_t *syn_words;
    uint32_t *err_words;
    uint8_t *conv;
    int32_t *iters;
    unsigned long long *counters;    // nullable: decoded, converged and executed iterations are ADDED to [0..2]
    unsigned char *ws;               // GLOBAL: the workspace, one slice of slice_bytes per CTA of the grid
    long long slice_bytes;
    int off_cv, off_omega, off_llr, off_osc, off_par, off_dec, off_red;   // byte offsets in the per-syndrome arrays (vc at 0);
                                                                          // off_red: of the reduction scratch in shared memory
};

constexpr int kBpotsThreads = 256;

struct OtsPick { int osc; double a; int idx; };
// better = more oscillations, then smaller |llr|, then smaller index (the strict comparisons of :303-312 keep the first)
__device__ __forceinline__ bool ots_better_j1(const OtsPick &x, const OtsPick &y)
{
    if (x.osc != y.osc) return x.osc > y.osc;
    if (x.a != y.a) return x.a < y.a;
    return x.idx < y.idx;
}
__device__ __forceinline__ bool ots_better_j2(const OtsPick &x, const OtsPick &y)
{
    if (x.a != y.a) return x.a < y.a;
    return x.idx < y.idx;
}

template <bool J1>
__device__ __forceinline__ OtsPick ots_block_pick(OtsPick v, unsigned char *red_raw)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o > 0; o >>= 1) {
        OtsPick w;
        w.osc = __shfl_xor_sync(0xffffffffu, v.osc, o);
        w.a = __shfl_xor_sync(0xffffffffu, v.a, o);
        w.idx = __shfl_xor_sync(0xffffffffu, v.idx, o);
        if (J1 ? ots_better_j1(w, v) : ots_better_j2(w, v)) v = w;
    }
    OtsPick *red = reinterpret_cast<OtsPick *>(red_raw);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    OtsPick best = red[0];
    for (int w = 1; w < kBpotsThreads / 32; ++w)
        if (J1 ? ots_better_j1(red[w], best) : ots_better_j2(red[w], best)) best = red[w];
    return best;
}

__device__ __forceinline__ int ots_block_sum(int v, unsigned char *red_raw)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = __reduce_add_sync(0xffffffffu, v);
    int *red = reinterpret_cast<int *>(red_raw);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    int t = 0;
    for (int w = 0; w < kBpotsThreads / 32; ++w) t += red[w];
    return t;
}

template <bool GLOBAL>
__global__ void __launch_bounds__(kBpotsThreads, 1) bpots_kernel(const BpotsParams p)
{
    extern __shared__ __align__(16) unsigned char ots_smem[];
    // (64-bit slice offset: grid x slice_bytes exceeds 2^31 on large codes; offsets inside a slice are below 2^31)
    unsigned char *base = GLOBAL ? p.ws + static_cast<long long>(blockIdx.x) * p.slice_bytes : ots_smem;
    double *vc = reinterpret_cast<double *>(base);                           // [E] variable->check, then the clamped tanh of it
    double *cv = reinterpret_cast<double *>(base + p.off_cv);                // [E] check->variable   (both in check-major slots)
    double *omega = reinterpret_cast<double *>(base + p.off_omega);          // [n]
    double *llr = reinterpret_cast<double *>(base + p.off_llr);              // [n]
    int *osc = reinterpret_cast<int *>(base + p.off_osc);                    // [n]
    int *par = reinterpret_cast<int *>(base + p.off_par);                    // [s] parity of the decisions on each check
    uint8_t *dec = base + p.off_dec;                                         // [n] current, [n] previous, [n] best decisions
    uint8_t *prior = dec + p.n, *best = dec + 2 * p.n;
    unsigned char *red = ots_smem + p.off_red;
    const int tid = threadIdx.x;
    constexpr double MAX_TANH = 0.99999, MAX_MSG = 100.0;

    for (long long b = blockIdx.x; b < p.B; b += gridDim.x) {
        const uint32_t *srow = p.syn_words + b * p.SW;
        for (int k = tid; k < p.E; k += kBpotsThreads) { vc[k] = 0.0; cv[k] = 0.0; }                       // reset! :144-156
        for (int j = tid; j < p.n; j += kBpotsThreads) { osc[j] = 0; prior[j] = 0; best[j] = 0; omega[j] = p.prior; }
        __syncthreads();
        int best_mismatch = p.s, best_weight = p.n, it = 0, converged = 0;
        for (int iter = 1; iter <= p.max_iters; ++iter) {
            it = iter;
            for (int j = tid; j < p.n; j += kBpotsThreads) {                                               // :161-174
                const int e0 = p.colptr[j], e1 = p.colptr[j + 1];
                for (int e = e0; e < e1; ++e) {
                    double msg_sum = 0.0;
                    for (int e2 = e0; e2 < e1; ++e2)
                        if (e2 != e) msg_sum = __dadd_rn(msg_sum, cv[p.ve_slot[e2]]);
                    vc[p.ve_slot[e]] = __dadd_rn(omega[j], msg_sum);
                }
            }
            __syncthreads();
            for (int k = tid; k < p.E; k += kBpotsThreads) {                                               // :187-189, once per edge
                const double t = tanh(__dmul_rn(0.5, vc[k]));
                vc[k] = fmin(MAX_TANH, fmax(-MAX_TANH, t));
            }
            __syncthreads();
            for (int i = tid; i < p.s; i += kBpotsThreads) {                                               // :180-211
                const int k0 = p.rowptr[i], k1 = p.rowptr[i + 1];
                const bool neg = (srow[i >> 5] >> (i & 31)) & 1u;
                for (int k = k0; k < k1; ++k) {
                    double prod = 1.0;
                    for (int k2 = k0; k2 < k1; ++k2)
                        if (k2 != k) prod = __dmul_rn(prod, vc[k2]);
                    if (neg) prod = -prod;
                    if (fabs(prod) >= MAX_TANH) prod = prod > 0 ? MAX_TANH : -MAX_TANH;
                    double msg = __dmul_rn(2.0, atanh(prod));
                    msg = fmin(MAX_MSG, fmax(-MAX_MSG, msg));
                    cv[k] = msg;
                }
                par[i] = 0;
            }
            __syncthreads();
            int weight = 0;
            for (int j = tid; j < p.n; j += kBpotsThreads) {                                               // :113-129, :257-262
                double l = omega[j];
                const int e0 = p.colptr[j], e1 = p.colptr[j + 1];
                for (int e = e0; e < e1; ++e) l = __dadd_rn(l, cv[p.ve_slot[e]]);
                llr[j] = l;
                const uint8_t d = l < 0.0 ? 1 : 0;
                if (iter > 1) osc[j] += d ^ prior[j];
                prior[j] = d;
                dec[j] = d;
                weight += d;
                if (d)
                    for (int e = e0; e < e1; ++e) atomicXor(&par[p.ve_chk[e]], 1);
            }
            weight = ots_block_sum(weight, red);           // (its barriers also complete the parities)
            int mismatch = 0;
            for (int i = tid; i < p.s; i += kBpotsThreads) mismatch += par[i] != static_cast<int>((srow[i >> 5] >> (i & 31)) & 1u);
            mismatch = ots_block_sum(mismatch, red);
            if (mismatch < best_mismatch || (mismatch == best_mismatch && weight < best_weight)) {          // :283-292
                best_mismatch = mismatch; best_weight = weight;
                for (int j = tid; j < p.n; j += kBpotsThreads) best[j] = dec[j];
                if (mismatch == 0) { converged = 1; break; }
            }
            if (mismatch > 0 && iter % p.T == 0) {                                                         // :294-336
                OtsPick m1{0, 0.0, 0x7fffffff}, m2{0, 1.0 / 0.0, 0x7fffffff};
                bool have = false;
                for (int j = tid; j < p.n; j += kBpotsThreads) {
                    omega[j] = p.prior;
                    const OtsPick c{osc[j], fabs(llr[j]), j};
                    if (!have || ots_better_j1(c, m1)) m1 = c;
                    if (!have || ots_better_j2(c, m2)) m2 = c;
                    have = true;
                }
                if (!have) { m1 = OtsPick{-1, 1.0 / 0.0, 0x7fffffff}; m2 = m1; }
                const OtsPick j1 = ots_block_pick<true>(m1, red);
                const OtsPick j2 = ots_block_pick<false>(m2, red);
                __syncthreads();
                if (tid == 0 && j1.osc > 0) {              // maximum(oscillations) > 0
                    osc[j1.idx] = 0;
                    omega[j1.idx] = -p.C;
                    omega[j2.idx] = -p.C;
                }
            }
            __syncthreads();
        }
        __syncthreads();
        // outputs: best_decisions (packed), converged, executed iterations
        for (int w = tid; w < p.NW; w += kBpotsThreads) {
            uint32_t v = 0;
            for (int k = 0; k < 32 && w * 32 + k < p.n; ++k) v |= static_cast<uint32_t>(best[w * 32 + k]) << k;
            p.err_words[b * p.NW + w] = v;
        }
        if (tid == 0) {
            p.conv[b] = static_cast<uint8_t>(converged);
            if (p.iters) p.iters[b] = it;
            if (p.counters) {
                atomicAdd(&p.counters[0], 1ull);
                atomicAdd(&p.counters[1], static_cast<unsigned long long>(converged));
                atomicAdd(&p.counters[2], static_cast<unsigned long long>(it));
            }
        }
        __syncthreads();
    }
}

}  // namespace bp
