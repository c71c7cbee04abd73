// osd.cuh -- OSD-0 post-processing of the syndromes BP left unconverged (SURVEY.md section 8(f) rank 1).
//
// Replaces, for osd_order = 0, what decode!(::BeliefPropagationOSDDecoder, syndrome) does after its BP call
// (/root/reference/src/decoders/belief_propagation_osd.jl:52-60) and osd(H, syndrome, bp_err, Val(0)) (:63-125):
//   * order the columns by max(r, 1-r) descending, r = 1/R the posterior ratio P0/P1, stable (:53-55);
//   * eliminate over GF(2) in that order until the remaining target is zero (:81-107), solve (:110-121),
//     un-permute (:60).
// For a syndrome in the column space of H that is: with S the first linearly independent columns (in sorted
// order) up to the point where the residual syndrome lies in their span, bp_err on the columns outside S and
// bp_err xor d on S, d the unique solution of H_S d = syndrome xor H bp_err -- whatever rows are taken as pivot
// rows.  For a syndrome OUTSIDE the column space the outcome depends on which equations become pivot rows, so
// the kernel takes the reference's: the first hit row in its physically swapped row order, which is tracked as
// a position per row (the rows themselves never move; a row becomes "used" instead).  Back substitution over
// the pivots as in the reference; tests compare bit for bit with the literal restatement in oracle/bp_oracle.c.
// Converged syndromes are returned unchanged by the reference (:72-74) and are skipped here.
//
// One CTA per syndrome (work queue over the unconverged list).  Shared memory holds the whole augmented
// matrix bit-packed by rows over the SORTED column positions: m rows x NWr words, the last bit of a row is
// its target bit; NWr is 4 x odd so that 16-byte row accesses of 8 consecutive rows are bank-conflict-free.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bp {

struct OsdParams {
    int m, n;              // checks, variables
    int NWr;               // words per augmented row (multiple of 4, odd multiple)
    int NP;                // sort length: power of two >= n
    int SW, NW;            // packed words per syndrome / error row
    const int *colptr;     // [n+1] original CSC
    const int *rowval;     // [E]   check of every CSC edge, ascending per column
    const uint32_t *syn_words;   // [B][SW]
    uint32_t *err_words;         // [B][NW]  in: BP decisions, out: OSD result
    const double *ratio;         // [B][n]   posterior ratios R_j of the last BP iteration
    const int *list;             // unconverged syndrome indices
    const int *count;            // how many
    int *queue;                  // work counter (zeroed before the launch)
    unsigned long long *stats;   // [0] syndromes processed, [1] pivots, [2] column steps; with `profile`
                                 // also SM cycles of [3] sort [4] build [5] pivot search [6] row updates [7] solve
    int profile;
    // shared-memory byte offsets
    int off_key, off_idx, off_piv, off_red;
};

__global__ void osd_collect_kernel(const uint8_t *conv, long long B, int *list, int *count)
{
    const long long b = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (b < B && !conv[b]) list[atomicAdd(count, 1)] = static_cast<int>(b);
}

__global__ void osd_fill_ones_kernel(double *p, long long nelem)
{
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nelem;
         i += static_cast<long long>(gridDim.x) * blockDim.x)
        p[i] = 1.0;
}

constexpr int kOsdMaxRowsPerThread = 8;     // rows a thread owns: m <= 8 * T

// Reliability keys of the columns (:53-54), padded to NP with the largest key: descending max(r, 1-r), ties by index
// == ascending (~bits(max(r, 1-r)), index).  Stated deviation (as in the oracle): r = RN(1/R) instead of Julia's
// exp(log(1/R)).
template <int T>
__device__ __forceinline__ void osd_keys(int tid, const double *R, int n, int NP, unsigned long long *key, int *idx)
{
    for (int j = tid; j < NP; j += T) {
        unsigned long long kb = ~0ull;
        if (j < n) {
            const double r = __ddiv_rn(1.0, R[j]);
            const double q = __dsub_rn(1.0, r);
            kb = ~static_cast<unsigned long long>(__double_as_longlong(r > q ? r : q));
        }
        key[j] = kb;
        idx[j] = j;
    }
}

// Bitonic sort of the NP (key, idx) pairs into ascending order, which is the stable descending order of :55 (every
// thread of the CTA calls it after a barrier that follows osd_keys; it ends with a barrier)
template <int T>
__device__ __forceinline__ void osd_sort(int tid, int NP, unsigned long long *key, int *idx)
{
    for (int k = 2; k <= NP; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int q = tid; q < NP / 2; q += T) {        // one compare-exchange per thread and trip, no idle lanes
                const int i = ((q & ~(j - 1)) << 1) | (q & (j - 1)), x = i | j;
                const unsigned long long ka = key[i], kb = key[x];
                const int ia = idx[i], ib = idx[x];
                const bool gt = ka > kb || (ka == kb && ia > ib);
                if (gt == ((i & k) == 0)) {
                    key[i] = kb; key[x] = ka;
                    idx[i] = ib; idx[x] = ia;
                }
            }
            __syncthreads();
        }
    }
}

template <int T, int RPT>                   // RPT = ceil(m / T)
__global__ void __launch_bounds__(T, 1) osd0_kernel(const OsdParams p)
{
    extern __shared__ __align__(16) unsigned char osd_smem[];
    uint32_t *Hs = reinterpret_cast<uint32_t *>(osd_smem);
    unsigned long long *key = reinterpret_cast<unsigned long long *>(osd_smem + p.off_key);
    int *idx = reinterpret_cast<int *>(osd_smem + p.off_idx);
    int *piv = reinterpret_cast<int *>(osd_smem + p.off_piv);          // [m] pivot number of a row, or -1
    int *prow = piv + p.m, *pcol = piv + 2 * p.m;                      // [m] row / sorted column of the q-th pivot
    int *list = piv + 3 * p.m;                                         // [m] rows to eliminate in the current step
    int *rowat = piv + 4 * p.m;                                        // [m] row standing at a position of the reference's
                                                                       //     (physically swapped) row order
    int *ctl = reinterpret_cast<int *>(osd_smem + p.off_red);          // [16] block-wide control words (see below)
    uint32_t *invtab = reinterpret_cast<uint32_t *>(ctl) + 16 + 192;   // [NWr/4 + 1] 2^32 / ng rounded up
    int *wcnts = ctl + 16;                                             // [2][96] per-warp hit counts / candidates / later bits
    __shared__ int s_work;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m = p.m, n = p.n, NWr = p.NWr, NP = p.NP;
    const int augw = NWr - 1;
    const uint32_t augm = 0x80000000u;

    for (int g = tid + 2; g <= NWr / 4; g += T) invtab[g] = 0xffffffffu / static_cast<uint32_t>(g) + 1u;
    for (;;) {
        if (tid == 0) s_work = atomicAdd(p.queue, 1);
        __syncthreads();
        const int work = s_work;
        if (work >= *p.count) break;
        const long long b = p.list[work];
        const double *R = p.ratio + b * n;
        uint32_t *erow = p.err_words + b * p.NW;
        const uint32_t *srow = p.syn_words + b * p.SW;

        long long t0 = 0, c_sort = 0, c_build = 0, c_scan = 0, c_xor = 0, c_solve = 0;
        const bool prof = p.profile != 0 && tid == 0;
        if (prof) t0 = clock64();
        // ---- reliability sort (:53-55)
        osd_keys<T>(tid, R, n, NP, key, idx);
        for (int i = tid; i < m * (NWr / 4); i += T) reinterpret_cast<uint4 *>(Hs)[i] = make_uint4(0, 0, 0, 0);
        for (int r = tid; r < m; r += T) { piv[r] = -1; rowat[r] = r; }
        if (tid == 0) { ctl[2] = 0; ctl[12] = -1; }   // target count / solve round 0
        __syncthreads();
        osd_sort<T>(tid, NP, key, idx);
        if (prof) { const long long t = clock64(); c_sort = t - t0; t0 = t; }
        // ---- H_sorted (:56) with the target column syndrome xor H*bp_err (:66-71) as the last bit of a row
        for (int r = tid; r < m; r += T)
            if ((srow[r >> 5] >> (r & 31)) & 1u) atomicXor(&Hs[r * NWr + augw], augm);
        for (int q = tid; q < n; q += T) {
            const int c = idx[q];
            const bool e1 = (erow[c >> 5] >> (c & 31)) & 1u;
            const uint32_t bit = 1u << (q & 31);
            const int wq = q >> 5;
            for (int e = p.colptr[c]; e < p.colptr[c + 1]; ++e) {
                const int r = p.rowval[e];
                atomicOr(&Hs[r * NWr + wq], bit);
                if (e1) atomicXor(&Hs[r * NWr + augw], augm);
            }
        }
        __syncthreads();

        if (prof) { const long long t = clock64(); c_build = t - t0; t0 = t; }
        // ---- forward elimination over the sorted columns (:81-107), no row swaps.  Thread t owns rows t, t+T, ...
        // (bit k of umask: row t+k*T is not a pivot row yet).  Every step: the owners ballot their unused rows
        // that have bit j set; every warp leaves its hit count and smallest hit row; after the barrier the
        // smallest of all is the pivot row, the hit rows are compacted into a list (prefix over the per-warp
        // counts) and, after a second barrier, the (row, 16-byte group) pairs of the listed rows are spread
        // over all threads.
        // ctl[2]: number of unused rows whose target bit is set.
        uint32_t umask = 0;
        int posr[RPT];                                    // position of the thread's rows in the reference's row order
#pragma unroll
        for (int k = 0; k < RPT; ++k) posr[k] = tid + k * T;
        {
            int mine_t = 0;
            for (int r = tid, k = 0; r < m; r += T, ++k) {
                umask |= 1u << k;
                mine_t += (Hs[r * NWr + augw] & augm) ? 1 : 0;
            }
            if (mine_t) atomicAdd(&ctl[2], mine_t);
        }
        __syncthreads();
        int npiv = 0, steps = 0;
        int tog = 0;                                      // exchange buffer of this trip: flips on EVERY trip (a column skip may
                                                          // land on a column of the same parity, so `j & 1` would reuse the buffer
                                                          // a slow warp is still reading)
        for (int j = 0; j < n; ++j) {
            const int wj = j >> 5;
            const uint32_t bj = 1u << (j & 31);
            int *wb = wcnts + tog * 96;                   // per warp: [0..31] hits, [32..63] smallest hit row, [64..95] later bits
            tog ^= 1;
            int cand = 0x7fffffff, total = 0;
            uint32_t hbs[RPT], later = 0;                 // later: bits above j (same word) set in any unused row
#pragma unroll
            for (int k = 0; k < RPT; ++k) {
                const int r = tid + k * T;
                const uint32_t w = (r < m && ((umask >> k) & 1u)) ? Hs[r * NWr + wj] : 0u;
                const bool hit = (w & bj) != 0u;
                later |= w;
                hbs[k] = __ballot_sync(0xffffffffu, hit);
                total += __popc(hbs[k]);
                if (hit) cand = min(cand, (posr[k] << 12) | r);
            }
            cand = __reduce_min_sync(0xffffffffu, cand);
            later = __reduce_or_sync(0xffffffffu, later & ~(bj | (bj - 1u)));
            if (lane == 0) { wb[warp] = total; wb[32 + warp] = cand; wb[64 + warp] = static_cast<int>(later); }
            __syncthreads();
            // every warp redoes the small cross-warp reduction: pivot row, list offsets (prefix over the counts)
            int c = 0, mn = 0x7fffffff;
            if (lane < T / 32) { c = wb[lane]; mn = wb[32 + lane]; }
            const int best = __reduce_min_sync(0xffffffffu, mn);
            if (prof) { const long long t = clock64(); c_scan += t - t0; t0 = t; }
            if (ctl[2] == 0) break;                  // :82  remaining target is all zero
            ++steps;
            if (best == 0x7fffffff) {                  // :87  no pivot in this column; nothing changes until the next
                uint32_t lw = lane < T / 32 ? static_cast<uint32_t>(wb[64 + lane]) : 0u;   // column some unused row has
                lw = __reduce_or_sync(0xffffffffu, lw);
                const int nj = min(lw ? (wj << 5) + __ffs(static_cast<int>(lw)) - 1 : ((wj + 1) << 5), n);
                steps += nj - (j + 1);               // the skipped columns count as visited
                j = nj - 1;
                continue;
            }
            int base = __reduce_add_sync(0xffffffffu, lane < warp ? c : 0);   // exclusive prefix of this warp
            const int cnt = __reduce_add_sync(0xffffffffu, c);
#pragma unroll
            for (int k = 0; k < RPT; ++k) {
                if ((hbs[k] >> lane) & 1u) list[base + __popc(hbs[k] & ((1u << lane) - 1u))] = tid + k * T;
                base += __popc(hbs[k]);
            }
            // pivot row = the hit row standing first in the reference's row order (:88 findfirst); the reference then swaps
            // it with the row at position npiv (:94-98): that row, still unused, takes over the pivot row's old position
            const int pr = best & 4095, kpos = best >> 12;
            const int ri = rowat[npiv];
#pragma unroll
            for (int k = 0; k < RPT; ++k)
                if (tid + k * T == ri) posr[k] = kpos;
            const uint32_t ptgt = Hs[pr * NWr + augw] & augm;
            if (tid == 0) { prow[npiv] = pr; pcol[npiv] = j; }
            if ((pr % T) == tid) { umask &= ~(1u << (pr / T)); piv[pr] = npiv; }
            __syncthreads();
            if (tid == 0) rowat[kpos] = ri;          // (every thread has read rowat[npiv] before the barrier)
            ++npiv;
            const int g0 = wj >> 2, ng = (NWr >> 2) - g0;
            const uint32_t inv = invtab[ng];         // q / ng by multiplication
            const uint4 *prow4 = reinterpret_cast<const uint4 *>(Hs + pr * NWr) + g0;
            int dt = (ptgt && tid == 0) ? -1 : 0;    // the pivot row leaves the set of unused rows
            for (int q = tid; q < cnt * ng; q += T) {
                const int li = ng > 1 ? static_cast<int>(__umulhi(static_cast<uint32_t>(q), inv)) : q;
                const int g = q - li * ng;
                const int r = list[li];
                if (r == pr) continue;
                uint4 *row = reinterpret_cast<uint4 *>(Hs + r * NWr) + g0 + g;
                uint4 v = *row;
                const uint4 u = prow4[g];
                v.x ^= u.x; v.y ^= u.y; v.z ^= u.z; v.w ^= u.w;
                *row = v;
                if (ptgt && g == ng - 1) dt += (v.w & augm) ? 1 : -1;   // its target bit flipped
            }
            if (ptgt) {                              // block-uniform
                dt = __reduce_add_sync(0xffffffffu, dt);
                if (lane == 0 && dt) atomicAdd(&ctl[2], dt);
            }
            __syncthreads();
            if (prof) { const long long t = clock64(); c_xor += t - t0; t0 = t; }
        }
        if (prof) t0 = clock64();
        // ---- back substitution (:110-121): d_c of the q-th pivot = its row's target bit once the later pivots are
        // folded in.  Only pivots whose bit is set change anything: find the next one below q_hi with a block-wide
        // search, fold its column into the earlier pivot rows, repeat.
        __syncthreads();
        for (int q_hi = npiv, it = 0;; ++it) {
            int *slot = ctl + 12 + (it & 1);
            if (tid == 0) ctl[12 + ((it + 1) & 1)] = -1;
            int mine = -1;
            for (int qq = q_hi - 1 - tid; qq >= 0; qq -= T)
                if (Hs[prow[qq] * NWr + augw] & augm) { mine = qq; break; }
            mine = __reduce_max_sync(0xffffffffu, mine);
            if (lane == 0 && mine >= 0) atomicMax(slot, mine);
            __syncthreads();
            const int q = *slot;
            if (q < 0) break;
            const int c = pcol[q];
            const int wc = c >> 5;
            const uint32_t bc = 1u << (c & 31);
            for (int rr = tid; rr < m; rr += T) {
                const int o = piv[rr];
                if (o >= 0 && o < q && (Hs[rr * NWr + wc] & bc)) Hs[rr * NWr + augw] ^= augm;
            }
            if (tid == 0) {                              // correction = bp_err xor d  (:60 un-permutes)
                const int cc = idx[c];
                atomicXor(&erow[cc >> 5], 1u << (cc & 31));
            }
            q_hi = q;
            __syncthreads();
        }
        if (prof) {
            c_solve = clock64() - t0;
            atomicAdd(&p.stats[3], static_cast<unsigned long long>(c_sort));
            atomicAdd(&p.stats[4], static_cast<unsigned long long>(c_build));
            atomicAdd(&p.stats[5], static_cast<unsigned long long>(c_scan));
            atomicAdd(&p.stats[6], static_cast<unsigned long long>(c_xor));
            atomicAdd(&p.stats[7], static_cast<unsigned long long>(c_solve));
        }
        if (tid == 0) {
            atomicAdd(&p.stats[0], 1ull);
            atomicAdd(&p.stats[1], static_cast<unsigned long long>(npiv));
            atomicAdd(&p.stats[2], static_cast<unsigned long long>(steps));
        }
        __syncthreads();                             // shared memory is reused by the next syndrome
    }
}


// ---- OSD of order O > 0 (SURVEY 8(f) rank 4): osd(H_sorted, syndrome, bp_err_sorted, Val{O}) of
// /root/reference/src/decoders/belief_propagation_osd.jl:127-209 behind the sort of :53-57 and the un-permutation of :60.
// decode! applies it to EVERY syndrome (no shortcut for converged ones), so the kernel takes all B columns.
//   1. reliability sort and bit-packed [H_sorted | syndrome] in shared memory, as in osd0_kernel;
//   2. Gauss-Jordan: forward elimination in the reference's PHYSICAL row order (position -> row table instead of moving
//      rows: `findfirst(H[i:end, j])` is the smallest position >= i whose row has bit j, :140-146), then the
//      back-elimination over the pivots in reverse (:163-170).  Pivot q stands at position q;
//   3. the exhaustive search (:182-206): with E the bp_err bits on the non-pivot columns, a pivot row q gives
//      err[pivot col] = s_q xor <row_q, E>; only the first O non-pivot columns change between trials, so per pivot one
//      precomputed bit a_q (everything but the trial columns) and an O-bit mask b_q (the row on the trial columns) make a
//      trial a parity of b_q & x.  Trial x = 0 keeps bp_err's own bits on the trial columns (the reference only writes
//      them for x != 0); weights are compared with `<` in ascending x, so the smallest x among the lightest wins.
// One CTA per syndrome; O <= kOsdMaxOrder.
constexpr int kOsdMaxOrder = 12;

template <int T>
__global__ void __launch_bounds__(T, 1) osdk_kernel(const OsdParams p, const int order_req, const long long B)
{
    extern __shared__ __align__(16) unsigned char osd_smem[];
    uint32_t *Hs = reinterpret_cast<uint32_t *>(osd_smem);
    unsigned long long *key = reinterpret_cast<unsigned long long *>(osd_smem + p.off_key);
    int *idx = reinterpret_cast<int *>(osd_smem + p.off_idx);
    int *piv_r = reinterpret_cast<int *>(osd_smem + p.off_piv);        // [m] row of the q-th pivot
    int *piv_c = piv_r + p.m;                                          // [m] sorted column of the q-th pivot
    int *rowat = piv_r + 2 * p.m;                                      // [m] row standing at a position
    uint32_t *ab = reinterpret_cast<uint32_t *>(piv_r + 3 * p.m);      // [m] a_q | b_q << 1
    uint32_t *ev = reinterpret_cast<uint32_t *>(piv_r + 4 * p.m);      // [NWr] bp_err over the sorted positions (then: the answer)
    int *ctl = reinterpret_cast<int *>(osd_smem + p.off_red);          // [16] control words, [16..] per-warp scratch
    __shared__ int s_work;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m = p.m, n = p.n, NWr = p.NWr, NP = p.NP;
    const int augw = NWr - 1;
    const uint32_t augm = 0x80000000u;
    constexpr int NWARP = T / 32;

    for (;;) {
        if (tid == 0) s_work = atomicAdd(p.queue, 1);
        __syncthreads();
        const long long b = s_work;
        if (b >= B) break;
        const double *R = p.ratio + b * n;
        uint32_t *erow = p.err_words + b * p.NW;
        const uint32_t *srow = p.syn_words + b * p.SW;
        // ---- reliability sort (:53-55)
        osd_keys<T>(tid, R, n, NP, key, idx);
        for (int i = tid; i < m * (NWr / 4); i += T) reinterpret_cast<uint4 *>(Hs)[i] = make_uint4(0, 0, 0, 0);
        for (int r = tid; r < m; r += T) rowat[r] = r;
        for (int w = tid; w < NWr; w += T) ev[w] = 0u;
        __syncthreads();
        osd_sort<T>(tid, NP, key, idx);
        // ---- [H_sorted | syndrome] (:56, :137) and bp_err over the sorted positions (:57)
        for (int r = tid; r < m; r += T)
            if ((srow[r >> 5] >> (r & 31)) & 1u) atomicOr(&Hs[r * NWr + augw], augm);
        for (int q = tid; q < n; q += T) {
            const int c = idx[q];
            if ((erow[c >> 5] >> (c & 31)) & 1u) atomicOr(&ev[q >> 5], 1u << (q & 31));
            const uint32_t bit = 1u << (q & 31);
            const int wq = q >> 5;
            for (int e = p.colptr[c]; e < p.colptr[c + 1]; ++e) atomicOr(&Hs[p.rowval[e] * NWr + wq], bit);
        }
        __syncthreads();
        // ---- forward elimination (:139-160)
        int np = 0;
        for (int j = 0; j < n && np < m; ++j) {
            const int wj = j >> 5;
            const uint32_t bj = 1u << (j & 31);
            int cand = 0x7fffffff;                         // smallest position >= np whose row has bit j
            for (int pos = np + tid; pos < m; pos += T)
                if (Hs[rowat[pos] * NWr + wj] & bj) { cand = pos; break; }
            cand = __reduce_min_sync(0xffffffffu, cand);
            int *wb = ctl + 16 + (j & 1) * NWARP;
            if (lane == 0) wb[warp] = cand;
            __syncthreads();
            int best = lane < NWARP ? wb[lane] : 0x7fffffff;
            best = __reduce_min_sync(0xffffffffu, best);
            if (best == 0x7fffffff) continue;              // :142 no pivot in this column
            const int pr = rowat[best], other = rowat[np];
            __syncthreads();                               // everybody has read rowat[best], rowat[np]
            if (tid == 0) { rowat[np] = pr; rowat[best] = other; piv_r[np] = pr; piv_c[np] = j; }   // :144-148 the swap
            __syncthreads();
            const uint32_t *prow = Hs + pr * NWr;
            for (int pos = np + 1 + tid; pos < m; pos += T) {                                        // :149-154
                uint32_t *row = Hs + rowat[pos] * NWr;
                if (row[wj] & bj)
                    for (int w = wj; w < NWr; ++w) row[w] ^= prow[w];
            }
            ++np;
            __syncthreads();
        }
        // ---- back-elimination over the pivots in reverse (:163-170): pivot q stands at position q
        for (int q = np - 1; q > 0; --q) {
            const int pj = piv_c[q], wj = pj >> 5;
            const uint32_t bj = 1u << (pj & 31);
            const uint32_t *prow = Hs + piv_r[q] * NWr;
            for (int qq = tid; qq < q; qq += T) {
                uint32_t *row = Hs + piv_r[qq] * NWr;
                if (row[wj] & bj)
                    for (int w = wj; w < NWr; ++w) row[w] ^= prow[w];
            }
            __syncthreads();
        }
        // ---- the search (:172-206)
        const int order = min(min(order_req, kOsdMaxOrder), n - np);
        // trial columns = the first `order` non-pivot columns; pivot columns are cleared from ev (err is overwritten there)
        if (tid == 0) {
            int q = 0, nt = 0;
            uint32_t e0t = 0;
            for (int c = 0; c < n && (nt < order || q < np); ++c) {
                if (q < np && piv_c[q] == c) { ev[c >> 5] &= ~(1u << (c & 31)); ++q; continue; }
                if (nt < order) {
                    ctl[16 + 2 * NWARP + nt] = c;                                  // trial column list
                    if ((ev[c >> 5] >> (c & 31)) & 1u) e0t |= 1u << nt;
                    ev[c >> 5] &= ~(1u << (c & 31));
                    ++nt;
                }
            }
            ctl[0] = static_cast<int>(e0t);                // bp_err on the trial columns (what trial x = 0 uses)
        }
        __syncthreads();
        const int *tcol = ctl + 16 + 2 * NWARP;
        const uint32_t e0t = static_cast<uint32_t>(ctl[0]);
        for (int q = tid; q < np; q += T) {
            const uint32_t *row = Hs + piv_r[q] * NWr;
            uint32_t par = (row[augw] & augm) ? 1u : 0u;
            for (int w = 0; w < NWr; ++w) par ^= __popc(row[w] & ev[w] & (w == augw ? ~augm : 0xffffffffu)) & 1u;
            uint32_t bq = 0;
            for (int t = 0; t < order; ++t) bq |= ((row[tcol[t] >> 5] >> (tcol[t] & 31)) & 1u) << t;
            ab[q] = par | (bq << 1);
        }
        int wbase = 0;
        for (int w = lane; w < NWr; w += 32) wbase += __popc(ev[w] & (w == augw ? ~augm : 0xffffffffu));
        wbase = __reduce_add_sync(0xffffffffu, wbase);
        __syncthreads();
        unsigned long long mine = ~0ull;                   // (weight << 32) | x, smallest wins = lightest, then smallest x
        for (uint32_t x = tid; x < (1u << order); x += T) {
            const uint32_t v = x == 0u ? e0t : x;
            int wgt = wbase + __popc(v);
            for (int q = 0; q < np; ++q) {
                const uint32_t a = ab[q];
                wgt += (a ^ __popc((a >> 1) & v)) & 1u;
            }
            const unsigned long long cnd = (static_cast<unsigned long long>(wgt) << 32) | x;
            mine = cnd < mine ? cnd : mine;
        }
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long oth = __shfl_xor_sync(0xffffffffu, mine, o);
            mine = oth < mine ? oth : mine;
        }
        int *red = ctl + 16 + 2 * NWARP + kOsdMaxOrder;    // per warp: weight, x
        if (lane == 0) { red[2 * warp] = static_cast<int>(mine >> 32); red[2 * warp + 1] = static_cast<int>(mine & 0xffffffffu); }
        __syncthreads();
        unsigned long long bestc = ~0ull;
        for (int w = 0; w < NWARP; ++w) {
            const unsigned long long c2 = (static_cast<unsigned long long>(static_cast<uint32_t>(red[2 * w])) << 32) | static_cast<uint32_t>(red[2 * w + 1]);
            bestc = c2 < bestc ? c2 : bestc;
        }
        const uint32_t xb = static_cast<uint32_t>(bestc);
        const uint32_t vb = xb == 0u ? e0t : xb;
        __syncthreads();
        // ---- the winning error over the sorted positions, then back to the caller's column order (:60)
        for (int t = tid; t < order; t += T)
            if ((vb >> t) & 1u) atomicOr(&ev[tcol[t] >> 5], 1u << (tcol[t] & 31));
        for (int q = tid; q < np; q += T) {
            const uint32_t a = ab[q];
            if ((a ^ __popc((a >> 1) & vb)) & 1u) atomicOr(&ev[piv_c[q] >> 5], 1u << (piv_c[q] & 31));
        }
        for (int w = tid; w < p.NW; w += T) erow[w] = 0u;
        __syncthreads();
        for (int c = tid; c < n; c += T)
            if ((ev[c >> 5] >> (c & 31)) & 1u) {
                const int cc = idx[c];
                atomicOr(&erow[cc >> 5], 1u << (cc & 31));
            }
        if (tid == 0) {
            atomicAdd(&p.stats[0], 1ull);
            atomicAdd(&p.stats[1], static_cast<unsigned long long>(np));
            atomicAdd(&p.stats[2], static_cast<unsigned long long>(1u << order));
        }
        __syncthreads();
    }
}

}  // namespace bp
