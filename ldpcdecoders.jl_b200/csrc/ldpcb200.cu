// ldpcb200.cu -- host side of libldpcb200.so: Tanner-graph builder, device contexts, kernel
// dispatch and the C ABI declared in include/ldpcb200.h.
//
// Path replaced: BeliefPropagationDecoder / decode! / batchdecode! of
// /root/reference/src/decoders/belief_propagation.jl:38-67,121-188,220-231.
// No CPU fallback exists in this file: every decode runs the CUDA kernels or fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>          // types and prototypes only: libnccl.so.2 is bound with dlopen when a handle spans several devices

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/ldpcb200.h"
#define BP_WITH_SELFTEST 1
#define BP_FILTER_KERNEL 1
#include "bp_kernel.cuh"
#include "bp_launch.h"
#include "bp_single.h"
#include "formats.cuh"
#include "osd.cuh"
#include "bpots.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(e_ == cudaErrorMemoryAllocation ? LDPCB200_ENOMEM : LDPCB200_ECUDA,        \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// ---- NCCL, bound at run time (SURVEY section 5 / 8(e): one ncclAllReduce of the counters per batch).  The library
// has no link-time dependency on NCCL: a single-device handle never touches it, and inside a process that already
// carries an NCCL (PyTorch bundles one) dlopen by SONAME binds to that copy.
struct NcclApi {
    bool tried = false, ok = false;
    std::string why;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
};
NcclApi g_nccl;
std::mutex g_nccl_mutex;

bool nccl_load()
{
    std::lock_guard<std::mutex> lock(g_nccl_mutex);
    if (g_nccl.tried) return g_nccl.ok;
    g_nccl.tried = true;
    void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) { g_nccl.why = std::string("dlopen(libnccl.so.2): ") + dlerror(); return false; }
    auto sym = [&](const char *name) { void *p = dlsym(lib, name); if (!p) g_nccl.why = std::string("missing symbol ") + name; return p; };
    g_nccl.CommInitAll = reinterpret_cast<decltype(&ncclCommInitAll)>(sym("ncclCommInitAll"));
    g_nccl.CommDestroy = reinterpret_cast<decltype(&ncclCommDestroy)>(sym("ncclCommDestroy"));
    g_nccl.AllReduce = reinterpret_cast<decltype(&ncclAllReduce)>(sym("ncclAllReduce"));
    g_nccl.GroupStart = reinterpret_cast<decltype(&ncclGroupStart)>(sym("ncclGroupStart"));
    g_nccl.GroupEnd = reinterpret_cast<decltype(&ncclGroupEnd)>(sym("ncclGroupEnd"));
    g_nccl.GetErrorString = reinterpret_cast<decltype(&ncclGetErrorString)>(sym("ncclGetErrorString"));
    g_nccl.ok = g_nccl.CommInitAll && g_nccl.CommDestroy && g_nccl.AllReduce && g_nccl.GroupStart && g_nccl.GroupEnd && g_nccl.GetErrorString;
    return g_nccl.ok;
}

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        CU(cudaMalloc(&p, bytes));
        cap = bytes;
        return 0;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T *as() const { return static_cast<T *>(p); }
};

struct PinnedBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        CU(cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
        cap = bytes;
        return 0;
    }
    void release()
    {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

struct DeviceCtx {
    int device = 0;
    int sm_count = 0;
    int smem_optin = 0, smem_per_sm = 0;
    cudaStream_t stream = nullptr;
    // graph tables
    int *d_rowptr = nullptr, *d_colptr = nullptr, *d_ve_slot = nullptr, *d_ve_chk = nullptr;
    unsigned char *d_tables = nullptr;
    // decoder tables in the kernels' node order (mode 2 reads them from global memory)
    int *d_p_rowptr = nullptr, *d_p_colptr = nullptr, *d_corig = nullptr, *d_vorig = nullptr;
    uint32_t *d_ve_off = nullptr, *d_vflip = nullptr;
    // family GLOBAL stores: per resident CTA messages (+ syndrome state / decision fields when those are global)
    DevBuf msg, state, efield;
    // host-batch staging: two buffer sets / streams so that the copies of one chunk overlap the
    // decode of the other
    struct StageSet {
        cudaStream_t stream = nullptr;
        DevBuf raw_in, raw_out, syn_words, err_words, conv, iters, ratio;
        DevBuf osd_list, osd_ctl;            // OSD-0: unconverged list, {count, queue}
        DevBuf f_list, f_count;              // first-iteration filter: this set's own work list, so that the decoding kernels
                                             // of consecutive chunks may overlap (shared-memory kernel: nothing else is shared)
        // pageable caller memory is staged through pinned blocks so that the copies stay asynchronous: the chunk's
        // input is gathered into pin_in by the host thread while the GPU works on the previous chunk; outputs land in
        // pin_out and are handed to the caller (`pending`) when this set comes round again
        PinnedBuf pin_in, pin_out;
        size_t pin_out_used = 0;
        struct Pending { void *dst; const void *src; size_t bytes; };
        std::vector<Pending> pending;
    } set[2];
    cudaEvent_t decode_done = nullptr;
    DevBuf counters, scratch, osd_stats, kprof, ctr_sum;
    DevBuf f_vars, f_edeg, f_epos, f_ctab, f_list, f_count;   // first-iteration filter: tables, work list
    bool f_ready = false;                                     // ... tables valid for the handle's current prior
    DevBuf lmask;                                         // logical operators: one 64-bit mask per variable (or empty)
    DevBuf hs_truth, hs_syn, hs_err, hs_conv, hs_iters, hs_ratio, hs_ctr, hs_sum;   // sampling + scoring harness tiles
    // option "time_kernels": CUDA event pairs around every launch of the decoding kernel, on the launching stream
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ktime_events;
    double ktime_ms = 0.0;
    long long ktime_launches = 0;
    DevBuf gk_msg, gk_state;   // grid-wide small-batch kernel (bp_grid_kernel): messages [E], resid | dec | work[2] | bar[2]
    int gk_blocks_per_sm = -1; // its co-resident CTAs per SM (-1: not asked yet, 0: unavailable)
    DevBuf bpots_ws;        // BP-OTS arrays of codes beyond shared memory: one slice per resident CTA (see bpots_on_device)
    DevBuf tiny;            // small-batch host calls: one device block ...
    PinnedBuf tiny_host;    // ... mirrored by one pinned block (one copy each way, one synchronisation)
};

}  // namespace

struct ldpcb200 {
    int64_t s = 0, n = 0, E = 0;
    double per = 0, p0 = 0;
    int regular_p0 = 0;
    int max_iters = 0, variant = 0;
    int max_cdeg = 0, max_vdeg = 0;
    int uni_cdeg = 0, uni_vdeg = 0;   // common degree when every check / variable has the same one (<= 12)
    bool big = false;
    int SW = 0, NW = 0;
    std::vector<int> rowptr, colptr, ve_slot, ve_chk;      // original node order (sampler / scorer)
    // decoder tables in degree-sorted node order (kernels); corig/vorig map back to original ids
    std::vector<int> p_rowptr, p_colptr, p_ve_slot, p_ve_chk, corig, vorig;
    bool perm_c = false, perm_v = false;
    bp::Segments segs{};
    std::vector<unsigned char> tables;   // SMEM-family blob
    int off_colptr = 0, off_ve = 0, off_vflip = 0, off_corig = 0, off_vorig = 0;
    int cv_cpw = 0, cv_stride = 0;       // contiguous variable ownership of bp_smem_kernel: variables per warp, bytes per warp in the ve table
    int tables_cv_warps = 0;             // layout the device copies of `tables` currently have
    bool tables_dirty = false;           // host blob rebuilt, device copies stale
    int opt_cv = 1;                      // bp_smem_kernel: contiguous variable ownership where the code allows it
    int opt_filter = 1;                  // shared-memory kernel: first-iteration filter (bp_filter.cuh) where the code allows it
    int opt_osd_order = 0;               // ldpcb200_bposd_decode_batch / the harness: OSD order (0: OSD-0 on the unconverged syndromes)
    int opt_stage_pageable = 1;          // host batches: stage pageable caller memory through pinned blocks (0: copy it directly)
    // options
    int opt_family = LDPCB200_FAMILY_AUTO, opt_warps = 0, opt_slots = 0, opt_early_stop = 1;
    int64_t opt_chunk = 0;
    double ms_scale = 0.875;     // min-sum normalisation factor (option "minsum_scale_permille")
    int64_t opt_small_batch = -1; // batches up to this size take the node-parallel kernel (-1: one CTA per SM, 0: never)
    int opt_osd_profile = 0;     // OSD kernel adds per-phase SM cycle counts to stats[3..7] (d_stats must then hold 8 uint64)
    int opt_ratio_last_only = 0; // ldpcb200_decode_device: write posterior ratios only in iteration max_iters (OSD pipelines)
    int opt_dynamic_queue = 1;   // shared-memory kernel: CTAs claim 32-syndrome chunks from a global counter (0: static shares)
    int opt_direct_bits = 1;     // host batches with BitMatrix output: the shared-memory kernel writes the bit stream itself
    int opt_overlap_chunks = 1;  // host batches, shared-memory kernel: decoding kernels of consecutive chunks may overlap (2: always)
    std::atomic<int> last_milli_iters{0};   // mean BP iterations per syndrome of the previous host batch x 1000 (0: none yet)
    int opt_grid_kernel = 1;     // small batches of codes too large for the one-CTA kernel: the grid-wide cooperative kernel
    int opt_ring_mult = 0;       // ring slot = this many times the rows of the widest node (more nodes per loop trip of the HBM modes; 0 = auto)
    int opt_pd = -1;             // cp.async prefetch distance of the HBM modes (-1: as deep as fits, 0: no staging)
    int opt_kernel_profile = 0;  // bp_smem_kernel adds per-phase SM cycles to the handle's profile block (ldpcb200_kernel_profile)
    int opt_time_kernels = 0;    // bracket every launch of the decoding kernel with CUDA events (ldpcb200_kernel_time)
    int opt_max_ctas = 0;        // cap on resident CTAs per SM (0: whatever fits; experiments)
    int opt_lean = 1;            // family SMEM: use the round-2 kernel (bp_smem.cuh) when the code fits its envelope
    int opt_bpots_memory = 0;    // BP-OTS arrays: 0 shared memory where they fit, else the global workspace; 1 shared only; 2 global
    // resolved configuration
    bool configured = false;
    int family = 0, mode = 0, warps = 0, ctas_per_sm = 0, smem_bytes = 0, slots = 0, shape = 0;
    int nfw = 0;                 // decision-field words per thread (0: fields live in registers)
    bool efield_global = false;
    bool lean = false, eb64 = false;   // bp_smem_kernel selected / its decision fields are 64 bits wide
    bool dual = false;                 // ... in its two-teams-per-CTA form
    int opt_dual = 0;                  // (measured equal to two independent CTAs per SM on C3: kept as an option, see DESIGN.md)
    const void *kernel = nullptr;      // entry point of the batch kernel configure() selected ...
    const void *kernel_prof = nullptr; // ... and the one that runs with option kernel_profile (its phase-timing build, if any)
    bp::KernelParams kp_proto{};
    std::vector<DeviceCtx> dev;
    std::atomic<long long> launches{0};
    // counters of a multi-device handle: ncclAllReduce over the handle's own communicators (one per device) when NCCL
    // is available and the devices are distinct; otherwise (or with option "nccl" = 0) the host adds the per-device values
    int opt_nccl = 1;
    int nccl_state = 0;                 // 0 not tried, 1 communicators ready, -1 unavailable (see nccl_why)
    std::string nccl_why;
    std::vector<ncclComm_t> comms;
    std::vector<unsigned long long> lmask;   // logical operators as per-variable bit masks (empty: none)
    int n_logicals = 0;
};

namespace {

inline int align_up(int x, int a) { return (x + a - 1) / a * a; }

inline int grid_for(long long work, int sm) { return static_cast<int>(std::max<long long>(1, std::min<long long>((work + 255) / 256, static_cast<long long>(sm) * 16))); }

// channel_probs[j] / (1 - channel_probs[j]) (belief_propagation.jl:129,153), IEEE double on the host
void set_prior(ldpcb200 *h, double per)
{
    volatile double one_minus = 1.0 - per;
    volatile double q = per / one_minus;
    h->per = per;
    for (DeviceCtx &d : h->dev) d.f_ready = false;        // the first-iteration tables depend on the prior
    h->p0 = q;
    h->regular_p0 = std::isnormal(h->p0) && h->p0 > 0.0;
    if (h->variant != LDPCB200_VARIANT_EXACT) {         // the kernels' prior slot carries L0 = log((1-p)/p)
        volatile double r = one_minus / per;
        h->p0 = std::log(r);
        if (h->variant == LDPCB200_VARIANT_FAST32) h->p0 = static_cast<double>(static_cast<float>(h->p0));
    }
}

// shared-memory carve-up for a kernel mode / thread count; returns total bytes
//   mode 0: messages | syn | resid | stage | nnz | [efield] | tables | mbar
//   mode 1:            syn | resid | stage | nnz | [efield] | tables | mbar
//   mode 2:                                  nnz                      | mbar
int smem_layout(const ldpcb200 *h, int mode, int threads, int nfw, bool efield_in_smem, int pd, bp::KernelParams &p)
{
    long long off = 0;
    if (mode == 0) off = static_cast<long long>(h->E) * 32 * 8;
    if (mode <= 1) {
        p.off_syn = static_cast<int>(off);    off += h->SW * 128;
        p.off_resid = static_cast<int>(off);  off += h->SW * 128;
        p.off_stage = static_cast<int>(off);  off += 2 * h->SW * 128;      // double-buffered
    }
    p.off_nnz = static_cast<int>(off);    off += 2 * 32 * 4;
    p.off_efield = static_cast<int>(off);
    if (efield_in_smem) off += static_cast<long long>(nfw) * threads * 4;
    off = (off + 15) / 16 * 16;
    p.off_tables = static_cast<int>(off);
    if (mode <= 1) off += static_cast<long long>(h->tables.size());
    off = (off + 7) / 8 * 8;
    p.off_mbar = static_cast<int>(off);   off += 8 + 16;              // mbarrier + the dynamic queue's four claimed chunk ids
    off = (off + 127) / 128 * 128;
    // cp.async ring (modes 1/2): per warp pd+1 slots of one node's rows (max register degree)
    const int maxdeg = std::min(std::max(h->max_cdeg, h->max_vdeg), bp::kMaxRegDegree);
    p.pd = (mode >= 1) ? pd : 0;
    // (a slot holds several nodes of a trip; measured best: two nodes' worth with tables in shared memory -- C4 0.87 -> 0.91
    // of the HBM roofline -- one with tables in global memory, where a ring depth of 2 wins instead: C5 0.69 -> 0.74)
    const int mult = h->opt_ring_mult > 0 ? h->opt_ring_mult : (mode == 1 ? 2 : 1);
    p.ring_slot_bytes = std::max(maxdeg, 1) * 256 * mult;
    p.ring_warp_bytes = (p.pd + 1) * p.ring_slot_bytes;
    p.off_ring = static_cast<int>(off);
    if (p.pd > 0) off += static_cast<long long>(threads / 32) * p.ring_warp_bytes;
    off = (off + 15) / 16 * 16;
    return off > 0x7fffffff ? 0x7fffffff : static_cast<int>(off);
}

// shared-memory carve-up of bp_smem_kernel (bp_smem.cuh):
//   messages | syn [SW][32] | resid [2][SW][32] | stage [2][SW][32] | sidq [2][32] | tables | mbar
//   dual: the first four arrays twice (one group per team, group_stride apart), then tables | mbar | team flags
int smem_layout_lean(const ldpcb200 *h, bp::KernelParams &p, bool dual = false)
{
    long long off = static_cast<long long>(h->E) * 32 * 8;
    p.off_syn = static_cast<int>(off);    off += h->SW * 128;
    p.off_resid = static_cast<int>(off);  off += 2 * h->SW * 128;      // per-lane double buffer
    p.off_stage = static_cast<int>(off);  off += 2 * h->SW * 128;      // double-buffered queue window
    p.off_sidq = static_cast<int>(off);   off += 2 * 128;              // ... and the syndrome index of each of its entries
    p.off_nnz = p.off_efield = 0;
    p.group_stride = 0;
    if (dual) {
        off = (off + 127) / 128 * 128;
        p.group_stride = static_cast<int>(off);
        off *= 2;
    }
    off = (off + 15) / 16 * 16;
    p.off_tables = static_cast<int>(off);
    off += static_cast<long long>(h->tables.size());
    off = (off + 7) / 8 * 8;
    p.off_mbar = static_cast<int>(off);   off += 8 + 16;                // mbarrier + team_done[2] + team_seen[2]
    off = (off + 127) / 128 * 128;
    p.pd = 0; p.ring_slot_bytes = 0; p.ring_warp_bytes = 0; p.off_ring = static_cast<int>(off);
    return off > 0x7fffffff ? 0x7fffffff : static_cast<int>(off);
}

// SMEM-family table blob (copied to shared memory by one TMA bulk copy): rowptr u16[s+1] | colptr u16[n+1] |
// ve_off u32 (slot * 256 bytes per edge, variable-major) | vflip u16[E] | corig u16[s] | vorig u16[n], all in the
// kernels' node order.  cv_warps > 0 (bp_smem_kernel with contiguous variable ownership, uniform variable degree D):
// the ve_off section is laid out per warp -- warp w's cpw = ceil(n / cv_warps) variables start at
// w * cv_stride bytes, cv_stride a multiple of 16 -- so that the offsets of four variables are D aligned 16-byte loads.
void build_tables(ldpcb200 *h, int cv_warps)
{
    const int64_t s = h->s, n = h->n, E = h->E;
    h->tables.clear();
    h->cv_cpw = 0; h->cv_stride = 0;
    if (!(E <= 0xffff && s <= 16384 && n <= 0xffff)) return;
    int ve_bytes = static_cast<int>(4 * E);
    if (cv_warps > 0) {
        h->cv_cpw = static_cast<int>((n + cv_warps - 1) / cv_warps);
        h->cv_stride = align_up(h->cv_cpw * h->uni_vdeg * 4, 16);
        ve_bytes = cv_warps * h->cv_stride;
    }
    // (the contiguous-ownership layout is only read by bp_smem_kernel in its uniform-degree form, which needs neither
    // rowptr nor colptr: those sections are left out -- on the gross code that is what makes room for the queue's
    // staged syndrome indices next to two resident CTAs)
    const bool ptrs = cv_warps <= 0;
    const int o_col = ptrs ? align_up(static_cast<int>(2 * (s + 1)), 4) : 0;
    const int o_ve = ptrs ? align_up(o_col + static_cast<int>(2 * (n + 1)), 16) : 0;
    const int o_fl = o_ve + ve_bytes;
    const int o_co = align_up(o_fl + static_cast<int>(2 * E), 4);
    const int o_vo = o_co + (h->perm_c ? static_cast<int>(2 * s) : 0);
    const int total = align_up(o_vo + (h->perm_v ? static_cast<int>(2 * n) : 0), 16);
    h->tables.assign(std::max(total, 16), 0);
    uint16_t *rp = reinterpret_cast<uint16_t *>(h->tables.data());
    uint16_t *cp = reinterpret_cast<uint16_t *>(h->tables.data() + o_col);
    uint32_t *ve = reinterpret_cast<uint32_t *>(h->tables.data() + o_ve);
    if (ptrs) {
        for (int64_t i = 0; i <= s; ++i) rp[i] = static_cast<uint16_t>(h->p_rowptr[i]);
        for (int64_t j = 0; j <= n; ++j) cp[j] = static_cast<uint16_t>(h->p_colptr[j]);
    }
    uint16_t *fl = reinterpret_cast<uint16_t *>(h->tables.data() + o_fl);
    for (int64_t e = 0; e < E; ++e) {
        // residual-syndrome word (byte offset of its 128 B row) | bit: needs s <= 16384
        fl[e] = static_cast<uint16_t>((h->p_ve_chk[e] >> 5) * 128 + (h->p_ve_chk[e] & 31));
    }
    if (cv_warps > 0) {
        const int D = h->uni_vdeg;
        for (int64_t j = 0; j < n; ++j) {
            const int w = static_cast<int>(j / h->cv_cpw), i = static_cast<int>(j % h->cv_cpw);
            uint32_t *dst = reinterpret_cast<uint32_t *>(h->tables.data() + o_ve + w * h->cv_stride) + i * D;
            for (int k = 0; k < D; ++k) dst[k] = static_cast<uint32_t>(h->p_ve_slot[j * D + k]) * 256u;
        }
    } else {
        for (int64_t e = 0; e < E; ++e) ve[e] = static_cast<uint32_t>(h->p_ve_slot[e]) * 256u;
    }
    if (h->perm_c) {
        uint16_t *co = reinterpret_cast<uint16_t *>(h->tables.data() + o_co);
        for (int64_t i = 0; i < s; ++i) co[i] = static_cast<uint16_t>(h->corig[i]);
    }
    if (h->perm_v) {
        uint16_t *vo = reinterpret_cast<uint16_t *>(h->tables.data() + o_vo);
        for (int64_t j = 0; j < n; ++j) vo[j] = static_cast<uint16_t>(h->vorig[j]);
    }
    h->off_colptr = o_col;
    h->off_ve = o_ve;
    h->off_vflip = o_fl;
    h->off_corig = o_co;
    h->off_vorig = o_vo;
}

int build_graph(ldpcb200 *h, const int64_t *colptr, const int64_t *rowval, int base)
{
    const int64_t s = h->s, n = h->n;
    if (colptr[0] - base != 0) return fail(LDPCB200_EINVAL, "colptr[0] must equal index_base");
    const int64_t E = colptr[n] - base;
    // message rows are addressed as slot * 256 in 32-bit arithmetic inside the kernels
    if (E < 0 || E > LDPCB200_MAX_EDGES) return fail(LDPCB200_EUNSUPPORTED, "edge count %lld exceeds LDPCB200_MAX_EDGES", (long long)E);
    h->E = E;
    h->colptr.assign(n + 1, 0);
    h->rowptr.assign(s + 1, 0);
    h->ve_slot.assign(std::max<int64_t>(E, 1), 0);
    h->ve_chk.assign(std::max<int64_t>(E, 1), 0);
    for (int64_t j = 0; j < n; ++j) {
        const int64_t a = colptr[j] - base, b = colptr[j + 1] - base;
        if (b < a || b > E) return fail(LDPCB200_EINVAL, "colptr not monotone at column %lld", (long long)j);
        h->colptr[j + 1] = static_cast<int>(b);
        h->max_vdeg = std::max<int>(h->max_vdeg, static_cast<int>(b - a));
        for (int64_t e = a; e < b; ++e) {
            const int64_t r = rowval[e] - base;
            if (r < 0 || r >= s) return fail(LDPCB200_EINVAL, "row index out of range at entry %lld", (long long)e);
            if (e > a && rowval[e] <= rowval[e - 1])
                return fail(LDPCB200_EINVAL, "row indices must be strictly ascending inside column %lld", (long long)j);
            h->ve_chk[e] = static_cast<int>(r);
            h->rowptr[r + 1]++;
        }
    }
    for (int64_t i = 0; i < s; ++i) {
        h->max_cdeg = std::max(h->max_cdeg, h->rowptr[i + 1]);
        h->rowptr[i + 1] += h->rowptr[i];
    }
    // check-major edge slots: visiting columns in ascending order makes the variables of every
    // check ascending, the order nzrange(sparse_HT, i) walks (belief_propagation.jl:137)
    std::vector<int> fill(h->rowptr.begin(), h->rowptr.end() - 1);
    for (int64_t j = 0; j < n; ++j)
        for (int e = h->colptr[j]; e < h->colptr[j + 1]; ++e) h->ve_slot[e] = fill[h->ve_chk[e]]++;
    if (h->max_cdeg > LDPCB200_MAX_DEGREE || h->max_vdeg > LDPCB200_MAX_DEGREE)
        return fail(LDPCB200_EUNSUPPORTED, "node degree %d exceeds LDPCB200_MAX_DEGREE=%d",
                    std::max(h->max_cdeg, h->max_vdeg), LDPCB200_MAX_DEGREE);
    h->big = std::max(h->max_cdeg, h->max_vdeg) > bp::kMaxRegDegree;
    {
        bool uc = s > 0, uv = n > 0;
        for (int64_t i = 0; i < s; ++i) uc &= (h->rowptr[i + 1] - h->rowptr[i]) == h->max_cdeg;
        for (int64_t j = 0; j < n; ++j) uv &= (h->colptr[j + 1] - h->colptr[j]) == h->max_vdeg;
        h->uni_cdeg = (uc && h->max_cdeg >= 1 && h->max_cdeg <= bp::kMaxRegDegree) ? h->max_cdeg : 0;
        h->uni_vdeg = (uv && h->max_vdeg >= 1 && h->max_vdeg <= bp::kMaxRegDegree) ? h->max_vdeg : 0;
    }
    h->SW = static_cast<int>((s + 31) / 32);
    h->NW = static_cast<int>((n + 31) / 32);
    if (h->SW == 0) h->SW = 1;
    if (h->NW == 0) h->NW = 1;
    // ---- degree-sorted node order for the kernels: nodes of equal degree become contiguous
    // "segments", so the per-node degree switch and table reads are hoisted out of the node
    // loops.  Inside a node the edge order stays ascending in ORIGINAL indices (the order the
    // reference multiplies in); corig/vorig translate syndrome bits and output positions.
    {
        std::vector<int> cdeg(s), vdeg(n);
        for (int64_t i = 0; i < s; ++i) cdeg[i] = h->rowptr[i + 1] - h->rowptr[i];
        for (int64_t j = 0; j < n; ++j) vdeg[j] = h->colptr[j + 1] - h->colptr[j];
        h->corig.resize(s); h->vorig.resize(n);
        for (int64_t i = 0; i < s; ++i) h->corig[i] = static_cast<int>(i);
        for (int64_t j = 0; j < n; ++j) h->vorig[j] = static_cast<int>(j);
        std::stable_sort(h->corig.begin(), h->corig.end(), [&](int a, int b) { return cdeg[a] < cdeg[b]; });
        std::stable_sort(h->vorig.begin(), h->vorig.end(), [&](int a, int b) { return vdeg[a] < vdeg[b]; });
        auto count_runs = [](const std::vector<int> &order, const std::vector<int> &deg) {
            int runs = 0;
            for (size_t k = 0; k < order.size(); ++k) runs += (k == 0 || deg[order[k]] != deg[order[k - 1]]);
            return runs;
        };
        // codes with many distinct degrees keep the original order and the per-node path
        if (count_runs(h->corig, cdeg) > bp::kMaxSeg) for (int64_t i = 0; i < s; ++i) h->corig[i] = static_cast<int>(i);
        if (count_runs(h->vorig, vdeg) > bp::kMaxSeg) for (int64_t j = 0; j < n; ++j) h->vorig[j] = static_cast<int>(j);
        h->perm_c = h->perm_v = false;
        for (int64_t i = 0; i < s; ++i) h->perm_c |= h->corig[i] != i;
        for (int64_t j = 0; j < n; ++j) h->perm_v |= h->vorig[j] != j;
        std::vector<int> inv_c(s);
        for (int64_t i = 0; i < s; ++i) inv_c[h->corig[i]] = static_cast<int>(i);
        h->p_rowptr.assign(s + 1, 0);
        for (int64_t i = 0; i < s; ++i) h->p_rowptr[i + 1] = h->p_rowptr[i] + cdeg[h->corig[i]];
        // slot of every original CSC edge: columns visited in ascending original order => inside a
        // check, variables ascend in original index (nzrange(sparse_HT, i), belief_propagation.jl:137)
        std::vector<int> slot_of(std::max<int64_t>(E, 1), 0), fill2(s);
        for (int64_t r = 0; r < s; ++r) fill2[r] = h->p_rowptr[inv_c[r]];
        for (int64_t j = 0; j < n; ++j)
            for (int e = h->colptr[j]; e < h->colptr[j + 1]; ++e) slot_of[e] = fill2[h->ve_chk[e]]++;
        h->p_colptr.assign(n + 1, 0);
        h->p_ve_slot.assign(std::max<int64_t>(E, 1), 0);
        h->p_ve_chk.assign(std::max<int64_t>(E, 1), 0);
        for (int64_t jp = 0; jp < n; ++jp) {
            const int j = h->vorig[jp];
            h->p_colptr[jp + 1] = h->p_colptr[jp] + vdeg[j];
            for (int k = 0; k < vdeg[j]; ++k) {      // ascending original check index (:155)
                h->p_ve_slot[h->p_colptr[jp] + k] = slot_of[h->colptr[j] + k];
                h->p_ve_chk[h->p_colptr[jp] + k] = h->ve_chk[h->colptr[j] + k];
            }
        }
        // segments (only used when they cover the node order with <= kMaxSeg runs)
        bp::Segments &sg = h->segs;
        sg.ncseg = sg.nvseg = 0;
        if (count_runs(h->corig, cdeg) <= bp::kMaxSeg && s > 0) {
            for (int64_t i = 0; i < s; ++i) {
                const int dg = cdeg[h->corig[i]];
                if (i == 0 || dg != sg.cdeg[sg.ncseg - 1]) {
                    sg.cdeg[sg.ncseg] = dg; sg.cfirst[sg.ncseg] = static_cast<int>(i); sg.cslot[sg.ncseg] = h->p_rowptr[i];
                    ++sg.ncseg;
                }
                sg.cend[sg.ncseg - 1] = static_cast<int>(i + 1);
            }
        }
        if (count_runs(h->vorig, vdeg) <= bp::kMaxSeg && n > 0) {
            for (int64_t j = 0; j < n; ++j) {
                const int dg = vdeg[h->vorig[j]];
                if (j == 0 || dg != sg.vdeg[sg.nvseg - 1]) {
                    sg.vdeg[sg.nvseg] = dg; sg.vfirst[sg.nvseg] = static_cast<int>(j); sg.vedge[sg.nvseg] = h->p_colptr[j];
                    ++sg.nvseg;
                }
                sg.vend[sg.nvseg - 1] = static_cast<int>(j + 1);
            }
        }
    }
    build_tables(h, 0);
    return 0;
}

int init_device(ldpcb200 *h, DeviceCtx &d)
{
    CU(cudaSetDevice(d.device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, d.device));
    if (prop.major < 10)
        return fail(LDPCB200_ENODEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", d.device,
                    prop.major, prop.minor);
    d.sm_count = prop.multiProcessorCount;
    d.smem_optin = static_cast<int>(prop.sharedMemPerBlockOptin);
    d.smem_per_sm = static_cast<int>(prop.sharedMemPerMultiprocessor);
    CU(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
    d.set[0].stream = d.stream;
    CU(cudaStreamCreateWithFlags(&d.set[1].stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&d.decode_done, cudaEventDisableTiming));
    auto up = [&](int **dst, const std::vector<int> &v) -> int {
        CU(cudaMalloc(dst, sizeof(int) * v.size()));
        CU(cudaMemcpy(*dst, v.data(), sizeof(int) * v.size(), cudaMemcpyHostToDevice));
        return 0;
    };
    int rc;
    if ((rc = up(&d.d_rowptr, h->rowptr))) return rc;
    if ((rc = up(&d.d_colptr, h->colptr))) return rc;
    if ((rc = up(&d.d_ve_slot, h->ve_slot))) return rc;
    if ((rc = up(&d.d_ve_chk, h->ve_chk))) return rc;
    if (!h->tables.empty()) {
        CU(cudaMalloc(&d.d_tables, h->tables.size()));
        CU(cudaMemcpy(d.d_tables, h->tables.data(), h->tables.size(), cudaMemcpyHostToDevice));
    }
    if ((rc = up(&d.d_p_rowptr, h->p_rowptr))) return rc;
    if ((rc = up(&d.d_p_colptr, h->p_colptr))) return rc;
    if (!h->corig.empty() && (rc = up(&d.d_corig, h->corig))) return rc;
    if (!h->vorig.empty() && (rc = up(&d.d_vorig, h->vorig))) return rc;
    {   // wide tables: slot byte offsets and residual (word, bit) of every edge, kernels' node order
        std::vector<uint32_t> off(h->p_ve_slot.size()), fl(h->p_ve_slot.size());
        for (size_t e = 0; e < off.size(); ++e) {
            off[e] = static_cast<uint32_t>(h->p_ve_slot[e]) * 256u;
            fl[e] = static_cast<uint32_t>((h->p_ve_chk[e] >> 5) * 128 + (h->p_ve_chk[e] & 31));
        }
        CU(cudaMalloc(&d.d_ve_off, sizeof(uint32_t) * off.size()));
        CU(cudaMemcpy(d.d_ve_off, off.data(), sizeof(uint32_t) * off.size(), cudaMemcpyHostToDevice));
        CU(cudaMalloc(&d.d_vflip, sizeof(uint32_t) * fl.size()));
        CU(cudaMemcpy(d.d_vflip, fl.data(), sizeof(uint32_t) * fl.size(), cudaMemcpyHostToDevice));
    }
    return 0;
}

void destroy_device(DeviceCtx &d)
{
    cudaSetDevice(d.device);
    if (d.stream) cudaStreamSynchronize(d.stream);
    cudaFree(d.d_rowptr); cudaFree(d.d_colptr); cudaFree(d.d_ve_slot); cudaFree(d.d_ve_chk);
    cudaFree(d.d_tables); cudaFree(d.d_ve_off); cudaFree(d.d_vflip);
    cudaFree(d.d_p_rowptr); cudaFree(d.d_p_colptr); cudaFree(d.d_corig); cudaFree(d.d_vorig);
    if (d.set[1].stream) cudaStreamSynchronize(d.set[1].stream);
    for (DevBuf *b : {&d.gk_msg, &d.gk_state, &d.msg, &d.state, &d.efield, &d.counters, &d.scratch, &d.osd_stats, &d.tiny, &d.kprof, &d.ctr_sum, &d.f_vars, &d.f_edeg, &d.f_epos, &d.f_ctab, &d.f_list, &d.f_count, &d.lmask, &d.hs_truth, &d.hs_syn, &d.hs_err,
                       &d.hs_conv, &d.hs_iters, &d.hs_ratio, &d.hs_ctr, &d.hs_sum, &d.bpots_ws}) b->release();
    d.tiny_host.release();
    for (auto &S : d.set)
        for (DevBuf *b : {&S.raw_in, &S.raw_out, &S.syn_words, &S.err_words, &S.conv, &S.iters, &S.ratio, &S.osd_list, &S.osd_ctl, &S.f_list, &S.f_count})
            b->release();
    for (auto &S : d.set) { S.pin_in.release(); S.pin_out.release(); }
    for (auto &pr : d.ktime_events) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }   // not yet read by ldpcb200_kernel_time
    d.ktime_events.clear();
    if (d.decode_done) cudaEventDestroy(d.decode_done);
    if (d.set[1].stream) cudaStreamDestroy(d.set[1].stream);
    if (d.stream) cudaStreamDestroy(d.stream);
}

using bp::kShape256x2;
using bp::kShape384x2;
using bp::kShape512x1;
using bp::kShape320x2;

int kernel_shape(bool two_ctas, int threads, int mode = 0, bool big = false)
{
    if (!two_ctas) return kShape512x1;
    if (threads <= 256) return kShape256x2;
    if (threads <= 320 && mode >= 1 && !big) return kShape320x2;
    return kShape384x2;
}

// The compiled kernels of one variant.  The instantiations live in their own translation units (bp_inst_*.cu); the
// persistent kernel's are indexed [mode][big][shape], nullptr where none exists (the min-sum and fast variants have
// no local-memory degree path: ldpcb200_create refuses those codes).
struct VariantKernels {
    const void *const *persistent[3][2];
    const bp::SmemKernels *smem;
    cudaError_t (*filter_setup)(const bp::FilterSetup &, cudaStream_t);
    const bp::SingleKernels *single;
};

const VariantKernels kVariantKernels[3] = {
    {{{bp::persistent_kernels_0_0_0, bp::persistent_kernels_0_1_0}, {bp::persistent_kernels_1_0_0, bp::persistent_kernels_1_1_0},
      {bp::persistent_kernels_2_0_0, bp::persistent_kernels_2_1_0}},
     &bp::smem_kernels_0, bp::filter_setup_0, &bp::single_kernels_0},
    {{{bp::persistent_kernels_0_0_1, nullptr}, {bp::persistent_kernels_1_0_1, nullptr}, {bp::persistent_kernels_2_0_1, nullptr}},
     &bp::smem_kernels_1, bp::filter_setup_1, &bp::single_kernels_1},
    {{{bp::persistent_kernels_0_0_2, nullptr}, {bp::persistent_kernels_1_0_2, nullptr}, {bp::persistent_kernels_2_0_2, nullptr}},
     &bp::smem_kernels_2, bp::filter_setup_2, &bp::single_kernels_2},
};

// (indexed by LDPCB200_VARIANT_*, which ldpcb200_create checks)
const VariantKernels &kernels_of(int variant) { return kVariantKernels[variant]; }

// Shared-memory limit (and, where the messages live in shared memory, the carveout) of a kernel instantiation on the
// current device, then how many of its CTAs an SM holds.  A nullptr entry is no instantiation: configure never picks one.
cudaError_t kernel_attrs(const void *k, bool carveout, int smem_bytes, int threads, int *blocks_per_sm)
{
    if (!k) return cudaErrorInvalidDeviceFunction;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    if (e == cudaSuccess && carveout)
        e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, k, threads, smem_bytes);
    return e;
}

// The dynamic-shared-memory limit is an attribute of the kernel instantiation on the current device, not of a decoder
// handle: two live handles that share an instantiation but need different sizes would otherwise lower each other's
// limit.  It is therefore (re)set before every launch (a host-side call of about a microsecond).
template <class P>
cudaError_t launch_kernel(const void *k, int grid, int threads, int smem_bytes, cudaStream_t st, const P &p)
{
    if (!k) return cudaErrorInvalidDeviceFunction;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    if (e != cudaSuccess) return e;
    void *args[] = {const_cast<P *>(&p)};
    return cudaLaunchKernel(k, dim3(grid), dim3(threads), args, smem_bytes, st);
}

// Warps per CTA: warp w owns checks w, w+W, ... and variables w, w+W, ...; pick the W whose two
// round-robin splits waste the fewest warp-slots (ties -> more warps, better latency hiding).
int pick_warps(int64_t s, int64_t n, int wmin, int wmax, bool forced = false)
{
    double best = -1.0;
    int best_w = wmax;
    for (int w = wmin; w <= wmax; ++w) {
        const double ec = s > 0 ? static_cast<double>(s) / (w * ((s + w - 1) / w)) : 1.0;
        const double ev = n > 0 ? static_cast<double>(n) / (w * ((n + w - 1) / w)) : 1.0;
        // equally even splits: more warps up to 8 (the 256-thread shape, <= 128 registers); the 384-thread shape
        // is capped at 80 registers and spills per-iteration state, measured 2.7 % slower on C3 at the same evenness
        // (without the early-stop bookkeeping -- option early_stop = 0 set before the first decode -- occupancy wins:
        // forced-32 runs are 10 % faster with 12 warps)
        const double score = 0.6 * ec + 0.4 * ev + (forced ? 0.004 * w : 0.004 * std::min(w, 8) - 0.002 * std::max(0, w - 8));
        if (score > best) { best = score; best_w = w; }
    }
    return best_w;
}

// Resolve family / kernel mode / launch shape from the code size, the options and device 0's limits.
int configure(ldpcb200 *h)
{
    if (h->configured) return 0;
    DeviceCtx &d0 = h->dev[0];
    CU(cudaSetDevice(d0.device));
    const bool narrow = !h->tables.empty();
    const int per_cta_2 = d0.smem_per_sm / 2 - 1024;          // budget per CTA with two resident CTAs
    auto fields = [&](int warps) { return h->n <= 64ll * warps ? 0 : static_cast<int>(((h->n + warps - 1) / warps + 31) / 32); };

    int family = h->opt_family;
    int mode = -1, warps = 0, shape = 0, need = 0, nfw = 0;
    bool two = false, ef_global = false;
    bp::KernelParams kp{};

    // ---- family SMEM (mode 0): messages of 32 syndromes + state + tables in shared memory
    if (family != LDPCB200_FAMILY_GLOBAL && narrow && h->E > 0) {
        const int wmax_two = h->big ? 8 : 12, wmax_one = 16;   // the local-memory degree path has no 384-thread kernel
        int w = h->opt_warps > 0 ? h->opt_warps : 0;
        // try two CTAs per SM first
        int w2 = w ? std::min(w, wmax_two) : pick_warps(h->s, h->n, 4, wmax_two, h->opt_early_stop == 0);
        int f2 = fields(w2);
        int need2 = smem_layout(h, 0, w2 * 32, f2, true, 0, kp);
        if (need2 <= per_cta_2) {
            mode = 0; warps = w2; two = true; need = need2; nfw = f2;
        } else {
            int w1 = w ? std::min(w, wmax_one) : pick_warps(h->s, h->n, 8, wmax_one);
            int f1 = fields(w1);
            int need1 = smem_layout(h, 0, w1 * 32, f1, true, 0, kp);
            if (need1 <= d0.smem_optin) { mode = 0; warps = w1; two = false; need = need1; nfw = f1; }
        }
        if (mode == 0) family = LDPCB200_FAMILY_SMEM;
    }
    if (family == LDPCB200_FAMILY_SMEM && mode != 0)
        return fail(LDPCB200_EUNSUPPORTED, "family SMEM: messages of 32 syndromes (%lld B) + tables do not fit in shared memory",
                    static_cast<long long>(h->E) * 256);
    // ---- family GLOBAL: messages in HBM/L2; state + tables in shared memory (mode 1) if they fit, else global (mode 2)
    if (mode < 0) {
        family = LDPCB200_FAMILY_GLOBAL;
        const int pd_max = h->opt_pd >= 0 ? std::min(h->opt_pd, bp::kMaxPrefetch) : 3;
        const int pd_max2 = h->opt_pd >= 0 ? pd_max : 2;     // mode 2 (two variables per trip): depth 2 measured best
        // HBM-bound: the depth of the cp.async ring matters more than the warp count, so take the
        // widest CTA (12, 10, 8 warps; two CTAs per SM) whose ring still reaches the full depth,
        // else the one with the deepest ring.  mode 1 (state + tables in shared memory) if it fits.
        std::vector<int> cand;
        if (h->opt_warps > 0) cand.push_back(std::min(h->opt_warps, h->big ? 8 : 12));
        else if (h->big) cand = {8};
        else if (narrow) cand = {12, 10, 8};
        else cand = {10, 12, 8};       // mode 2 for certain: ten warps (96 registers, few spills) measured best on C5 (+3 % over twelve)
        int best_pd = -1;
        for (int w : cand) {
            const bool two_w = w <= 12;
            const int budget = two_w ? per_cta_2 : d0.smem_optin;
            const int f = fields(w);
            int m = -1, pd_fit = -1, need_w = 0;
            bool efg = false;
            bp::KernelParams kw{};
            if (narrow) {
                const long long ef_bytes = static_cast<long long>(f) * w * 32 * 4;
                const bool ef_smem = ef_bytes <= 32 * 1024;
                for (int pd = pd_max; pd >= 0 && m < 0; --pd) {
                    need_w = smem_layout(h, 1, w * 32, f, ef_smem, pd, kw);
                    if (need_w <= budget) { m = 1; pd_fit = pd; efg = f > 0 && !ef_smem; }
                }
            }
            if (m < 0) {
                for (int pd = pd_max2; pd >= 0 && m < 0; --pd) {
                    need_w = smem_layout(h, 2, w * 32, f, false, pd, kw);
                    if (need_w <= budget) { m = 2; pd_fit = pd; }
                }
                efg = f > 0;
            }
            if (m >= 0 && pd_fit > best_pd) {
                best_pd = pd_fit; mode = m; warps = w; two = two_w; nfw = f; need = need_w; ef_global = efg; kp = kw;
            }
            if (best_pd == (mode == 2 ? pd_max2 : pd_max)) break;
        }
        if (mode < 0) return fail(LDPCB200_EUNSUPPORTED, "no kernel configuration fits in shared memory");
    }
    shape = kernel_shape(two, warps * 32, mode, h->big);
    // round-2 kernel for the shared-memory family: regular-enough codes whose decisions fit in a register per warp
    bool lean = false, eb64 = false, dual = false;
    int want_cv = 0;                 // contiguous variable ownership (uniform variable degree, caller's variable order)
    if (mode == 0 && h->opt_lean && !h->big && nfw == 0 && h->segs.ncseg > 0 && h->segs.nvseg > 0) {
        const int budget = two ? per_cta_2 : d0.smem_optin;
        if (h->uni_vdeg && !h->perm_v && h->opt_cv) want_cv = warps;
        for (int attempt = 0; attempt < 2 && !lean; ++attempt) {
            if (h->tables_cv_warps != want_cv) { build_tables(h, want_cv); h->tables_cv_warps = want_cv; h->tables_dirty = true; }
            bp::KernelParams kl{};
            const int need_l = smem_layout_lean(h, kl);
            if (need_l <= budget) {
                lean = true; need = need_l; kp = kl;
                eb64 = (h->n + warps - 1) / warps > 32;
                // two groups in one CTA per SM taking turns in the check pass (see bp_smem.cuh) instead of two independent CTAs
                bp::KernelParams kd{};
                const int need_d = smem_layout_lean(h, kd, true);
                if (two && h->opt_dual && warps <= 8 && need_d <= d0.smem_optin) { dual = true; need = need_d; kp = kd; }
            } else if (want_cv) {
                want_cv = 0;          // the padded table does not fit: interleaved ownership
            } else {
                break;
            }
        }
    }
    if (!lean && h->tables_cv_warps != 0) { build_tables(h, 0); h->tables_cv_warps = 0; h->tables_dirty = true; }
    if (h->tables_dirty) {
        for (DeviceCtx &d : h->dev) {
            CU(cudaSetDevice(d.device));
            CU(cudaStreamSynchronize(d.stream));
            if (d.d_tables) CU(cudaFree(d.d_tables));
            d.d_tables = nullptr;
            if (!h->tables.empty()) {
                CU(cudaMalloc(&d.d_tables, h->tables.size()));
                CU(cudaMemcpy(d.d_tables, h->tables.data(), h->tables.size(), cudaMemcpyHostToDevice));
            }
        }
        h->tables_dirty = false;
        CU(cudaSetDevice(d0.device));
    }
    const VariantKernels &K = kernels_of(h->variant);
    const int form = dual ? bp::kSmemDual : shape;
    const void *const *persistent = K.persistent[mode][h->big];
    const void *kernel = lean ? K.smem->kernel[form][eb64] : persistent ? persistent[shape] : nullptr;
    int bps = 0;
    for (DeviceCtx &d : h->dev) {
        CU(cudaSetDevice(d.device));
        const cudaError_t e = kernel_attrs(kernel, mode == 0, need, (dual ? 2 : 1) * warps * 32, &bps);
        if (e != cudaSuccess && lean) return fail(LDPCB200_ECUDA, "kernel attributes (shared-memory kernel): %s", cudaGetErrorString(e));
        if (e != cudaSuccess) return fail(LDPCB200_ECUDA, "kernel attributes (mode %d): %s", mode, cudaGetErrorString(e));
    }
    if (bps < 1) return fail(LDPCB200_EUNSUPPORTED, "BP kernel (mode %d, %d threads, %d B smem) does not fit on an SM", mode, warps * 32, need);
    if (h->opt_max_ctas > 0) bps = std::min(bps, h->opt_max_ctas);
    h->family = family; h->mode = mode; h->warps = warps; h->shape = shape; h->ctas_per_sm = bps;
    h->smem_bytes = need; h->nfw = nfw; h->efield_global = ef_global; h->kp_proto = kp;
    h->lean = lean; h->eb64 = eb64; h->dual = dual;
    h->kernel = kernel;
    h->kernel_prof = lean && !eb64 && K.smem->prof[form] ? K.smem->prof[form] : kernel;
    h->slots = (dual ? 64 : 32) * bps * d0.sm_count;
    h->configured = true;
    return 0;
}

__global__ void add_counters_kernel(unsigned long long *c, unsigned long long decoded)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) atomicAdd(c, decoded);
}

// Tables of the first-iteration filter for the handle's current prior (bp_filter.cuh), built on the device with the
// variant's own node updates.
int filter_prepare(ldpcb200 *h, DeviceCtx &d, cudaStream_t st)
{
    const int64_t n = h->n, E = h->E;
    std::vector<bp::FilterVar> vars(std::max<int64_t>(n, 1));
    std::vector<uint8_t> edeg(std::max<int64_t>(E, 1)), epos(std::max<int64_t>(E, 1));
    memset(vars.data(), 0, vars.size() * sizeof(bp::FilterVar));
    // position of every edge inside its check: slot - first slot of the check (slots are check-major, variables ascending)
    for (int64_t j = 0; j < n; ++j) {
        const int e0 = h->colptr[j], deg = h->colptr[j + 1] - e0;
        vars[j].deg = static_cast<uint8_t>(deg);
        for (int k = 0; k < deg; ++k) {
            const int chk = h->ve_chk[e0 + k];
            vars[j].chk[k] = static_cast<uint16_t>(chk);
            edeg[e0 + k] = static_cast<uint8_t>(h->rowptr[chk + 1] - h->rowptr[chk]);
            epos[e0 + k] = static_cast<uint8_t>(h->ve_slot[e0 + k] - h->rowptr[chk]);
        }
    }
    int rc;
    if ((rc = d.f_vars.reserve(vars.size() * sizeof(bp::FilterVar))) || (rc = d.f_edeg.reserve(edeg.size())) || (rc = d.f_epos.reserve(epos.size())) ||
        (rc = d.f_ctab.reserve((bp::kMaxRegDegree + 1) * 2 * bp::kMaxRegDegree * 8)))
        return rc;
    CU(cudaMemcpyAsync(d.f_vars.p, vars.data(), vars.size() * sizeof(bp::FilterVar), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.f_edeg.p, edeg.data(), edeg.size(), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.f_epos.p, epos.data(), epos.size(), cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(d.f_ctab.p, 0, (bp::kMaxRegDegree + 1) * 2 * bp::kMaxRegDegree * 8, st));
    CU(cudaStreamSynchronize(st));              // the host vectors go out of scope
    bp::FilterSetup q{};
    q.n = static_cast<int>(n); q.p0 = h->p0; q.check_aux = h->ms_scale; q.regular_p0 = h->regular_p0;
    q.colptr = d.d_colptr; q.e_deg = d.f_edeg.as<uint8_t>(); q.e_pos = d.f_epos.as<uint8_t>();
    q.ctab = d.f_ctab.as<double>(); q.vars = d.f_vars.as<bp::FilterVar>();
    cudaError_t e = kernels_of(h->variant).filter_setup(q, st);
    if (e != cudaSuccess) return fail(LDPCB200_ECUDA, "first-iteration tables: %s", cudaGetErrorString(e));
    CU(cudaStreamSynchronize(st));              // (other streams of the device read the tables from now on)
    h->launches += 2;
    d.f_ready = true;
    return 0;
}

// Option "time_kernels": the decoding kernel's own duration, by CUDA events recorded on the launching stream right
// before and after it (read back by ldpcb200_kernel_time once the stream is idle).
struct KernelTimer {
    DeviceCtx &d;
    cudaStream_t st;
    cudaEvent_t e1 = nullptr;
    KernelTimer(ldpcb200 *h, DeviceCtx &d_, cudaStream_t st_) : d(d_), st(st_)
    {
        if (!h->opt_time_kernels || d.ktime_events.size() >= 4096) return;
        cudaEvent_t e0 = nullptr;
        if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) { cudaGetLastError(); e1 = nullptr; return; }
        cudaEventRecord(e0, st);
        d.ktime_events.emplace_back(e0, e1);
    }
    ~KernelTimer() { if (e1) cudaEventRecord(e1, st); }
};

// Decode B syndromes resident on device `d` (native packed rows); stream-ordered, one launch.
int decode_on_device(ldpcb200 *h, DeviceCtx &d, int64_t B, const uint32_t *syn_words, uint32_t *err_words,
                     uint8_t *conv, int32_t *iters, double *ratio, unsigned long long *counters, cudaStream_t st,
                     bool ratio_last_only = false, DeviceCtx::StageSet *set = nullptr, uint32_t *err_bits = nullptr,
                     bool *used_bits = nullptr)
{
    // err_bits (nullable): a buffer of ceil(B*n/32) words; when the shared-memory kernel runs, the decisions are written there
    // as the caller's bit stream (bit b*n + j) instead of packed rows in err_words, and *used_bits is set
    DevBuf &f_list = set ? set->f_list : d.f_list, &f_count = set ? set->f_count : d.f_count;
    if (used_bits) *used_bits = false;
    if (B <= 0) return 0;
    CU(cudaSetDevice(d.device));
    if (h->max_iters <= 0) {
        // loop at belief_propagation.jl:134 never runs: err stays zero, converged = false
        CU(cudaMemsetAsync(err_words, 0, static_cast<size_t>(B) * h->NW * 4, st));
        CU(cudaMemsetAsync(conv, 0, static_cast<size_t>(B), st));
        if (iters) CU(cudaMemsetAsync(iters, 0, static_cast<size_t>(B) * 4, st));
        if (ratio) return fail(LDPCB200_EINVAL, "posterior_ratio is undefined for max_iters = 0");
        if (counters) {
            add_counters_kernel<<<1, 32, 0, st>>>(counters, static_cast<unsigned long long>(B));
            h->launches++;
        }
        return 0;
    }
    const VariantKernels &K = kernels_of(h->variant);
    // ---- small batches: one CTA per syndrome, threads over the nodes (bp_single.cuh)
    {
        const int64_t limit = h->opt_small_batch < 0 ? d.sm_count : h->opt_small_batch;
        const int off_syn = static_cast<int>((std::max<int64_t>(h->E, 1) * 8 + 15) / 16 * 16);
        const int smem = off_syn + 2 * h->SW * 4 + h->NW * 4;
        auto common = [&](auto &q) {        // the fields bp::SingleParams and bp::GridParams share
            q.s = static_cast<int>(h->s); q.n = static_cast<int>(h->n); q.E = static_cast<int>(h->E);
            q.SW = h->SW; q.NW = h->NW; q.max_iters = h->max_iters; q.early_stop = h->opt_early_stop;
            q.regular_p0 = h->regular_p0; q.ratio_last_only = ratio_last_only ? 1 : 0; q.p0 = h->p0; q.check_aux = h->ms_scale; q.B = B;
            q.rowptr = d.d_rowptr; q.colptr = d.d_colptr; q.ve_slot = d.d_ve_slot; q.ve_chk = d.d_ve_chk;
            q.syn_words = syn_words; q.err_words = err_words; q.conv = conv; q.iters = iters; q.ratio = ratio; q.counters = counters;
        };
        // ... or, when the messages of one syndrome do not fit in an SM's shared memory, the whole grid per syndrome
        // (cooperative launch, messages in L2): otherwise a lone decode! on a large code walks every edge on ONE lane
        if (B <= limit && !h->big && (smem > d.smem_optin || h->opt_grid_kernel == 2) && h->E > 0) {   // (2: always, a test hook)
            if (d.gk_blocks_per_sm < 0) {
                int coop = 0, bps = 0;
                cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, d.device);
                cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, K.single->grid, bp::kGridThreads, 0);
                if (e != cudaSuccess) { cudaGetLastError(); bps = 0; }
                d.gk_blocks_per_sm = coop ? bps : 0;
            }
            const long long nodes = std::max(h->s, h->n);
            const int grid = static_cast<int>(std::min<long long>(static_cast<long long>(d.gk_blocks_per_sm) * d.sm_count,
                                                                   (nodes + bp::kGridThreads - 1) / bp::kGridThreads));
            // barrier counter: (2 * max_iters + 2) arrivals per syndrome and CTA, 32 bits
            if (grid >= 1 && h->opt_grid_kernel && (2.0 * h->max_iters + 2.0) * static_cast<double>(B) * grid < 2.0e9) {
                int rc;
                const size_t st_bytes = static_cast<size_t>(h->SW + h->NW) * 4 + 16;
                const bool fresh_state = d.gk_state.cap < st_bytes;
                if ((rc = d.gk_msg.reserve(static_cast<size_t>(h->E) * 8)) || (rc = d.gk_state.reserve(st_bytes))) return rc;
                if (fresh_state) CU(cudaMemsetAsync(d.gk_state.p, 0, st_bytes, st));      // counters start at zero; the kernel leaves them so
                bp::GridParams q{};
                common(q);
                q.msg = d.gk_msg.as<double>();
                q.resid = d.gk_state.as<uint32_t>(); q.dec = q.resid + h->SW;
                q.work = reinterpret_cast<int *>(q.dec + h->NW); q.bar = reinterpret_cast<unsigned int *>(q.work + 2);
                // cooperative launch: the runtime guarantees that all CTAs are co-resident (the kernel spins on a grid-wide barrier)
                void *args[] = {&q};
                CU(cudaLaunchCooperativeKernel(K.single->grid, dim3(grid), dim3(bp::kGridThreads), args, 0, st));
                h->launches++;
                return 0;
            }
        }
        if (B <= limit && !h->big && smem <= d.smem_optin && h->E * 8 < (1 << 30)) {
            bp::SingleParams q{};
            common(q);
            q.off_syn = off_syn; q.off_resid = off_syn + h->SW * 4; q.off_dec = off_syn + 2 * h->SW * 4;
            CU(launch_kernel(K.single->node_parallel, static_cast<int>(B), bp::kSingleThreads, smem, st, q));
            h->launches++;
            return 0;
        }
    }
    const long long nchunks = (B + 31) / 32;
    const int grid = static_cast<int>(std::min<long long>(nchunks, static_cast<long long>(d.sm_count) * h->ctas_per_sm));
    const int thr = h->warps * 32;
    bp::KernelParams p = h->kp_proto;
    p.s = static_cast<int>(h->s); p.n = static_cast<int>(h->n); p.E = static_cast<int>(h->E);
    p.SW = h->SW; p.NW = h->NW; p.uni_cdeg = h->uni_cdeg; p.uni_vdeg = h->uni_vdeg;
    p.max_iters = h->max_iters; p.early_stop = h->opt_early_stop; p.p0 = h->p0; p.B = B;
    p.regular_p0 = h->regular_p0;
    p.check_aux = h->ms_scale;
    p.syn_words = syn_words; p.err_words = err_words; p.conv = conv; p.iters = iters; p.ratio = ratio;
    p.ratio_last_only = ratio_last_only ? 1 : 0;
    p.counters = counters;
    p.tables = d.d_tables; p.tables_bytes = static_cast<int>(h->tables.size());
    p.off_colptr = h->off_colptr; p.off_ve = h->off_ve; p.off_vflip = h->off_vflip;
    p.cv_cpw = h->lean ? h->cv_cpw : 0; p.cv_stride = h->cv_stride;
    p.g_rowptr = d.d_p_rowptr; p.g_colptr = d.d_p_colptr; p.g_ve_off = d.d_ve_off; p.g_vflip = d.d_vflip;
    p.g_corig = d.d_corig; p.g_vorig = d.d_vorig;
    p.perm_c = h->perm_c; p.perm_v = h->perm_v; p.off_corig = h->off_corig; p.off_vorig = h->off_vorig;
    p.seg = h->segs;
    p.nfw = h->nfw;
    int rc;
    if (h->mode >= 1) {
        if ((rc = d.msg.reserve(static_cast<size_t>(grid) * std::max<int64_t>(h->E, 1) * 32 * 8))) return rc;
        p.msg_global = d.msg.as<double>();
    }
    if (h->mode == 2) {
        if ((rc = d.state.reserve(static_cast<size_t>(grid) * 2 * h->SW * 128))) return rc;
        p.state_global = d.state.as<uint32_t>();
    }
    if (h->efield_global) {
        if ((rc = d.efield.reserve(static_cast<size_t>(grid) * h->nfw * thr * 4))) return rc;
        p.efield_global = d.efield.as<uint32_t>();
    }
    // finished lanes OR their set decision bits into the row: rows start out zero
    const bool bits_out = err_bits != nullptr && h->lean;
    if (bits_out) {
        CU(cudaMemsetAsync(err_bits, 0, static_cast<size_t>((B * h->n + 31) / 32) * 4, st));
        if (used_bits) *used_bits = true;
    } else {
        CU(cudaMemsetAsync(err_words, 0, static_cast<size_t>(B) * h->NW * 4, st));
    }
    if (h->lean && h->opt_kernel_profile) {
        if (!d.kprof.p) {
            if ((rc = d.kprof.reserve(64))) return rc;
            CU(cudaMemsetAsync(d.kprof.p, 0, 64, st));
        }
        p.prof = d.kprof.as<unsigned long long>();
    }
    // first-iteration filter: iteration 1 of every syndrome with integer instructions; only the rest is decoded for real
    const bool filter = h->lean && h->opt_filter && h->opt_early_stop && h->max_iters >= 2 && h->max_vdeg <= bp::kFilterMaxVarDeg &&
                        !h->big && h->s <= 0xffff && (2 * h->SW + h->NW) * 32 * 4 * bp::kFilterWarps <= d.smem_optin && (!ratio || ratio_last_only);
    if (filter && !d.f_ready) {
        if ((rc = filter_prepare(h, d, st))) return rc;
    }
    if (h->lean) {
        // 32-bit queue arithmetic inside the kernel: at most 2^30 syndromes per launch
        const int64_t kMaxLaunch = 1ll << 30;
        for (int64_t b0 = 0; b0 < B; b0 += kMaxLaunch) {
            const int64_t Bl = std::min(kMaxLaunch, B - b0);
            bp::KernelParams q = p;
            q.B = Bl;
            q.syn_words = syn_words + b0 * h->SW; q.conv = conv + b0;
            q.err_words = bits_out ? err_bits + (b0 * h->n) / 32 : err_words + b0 * h->NW;      // (b0 is a multiple of 2^30)
            q.out_bits = bits_out ? 1 : 0;
            q.iters = iters ? iters + b0 : nullptr; q.ratio = ratio ? ratio + b0 * h->n : nullptr;
            // f_count: [0] length of the filter's work list, [2] chunks of the batch claimed by the CTAs (dynamic queue)
            if ((rc = f_count.reserve(16))) return rc;
            CU(cudaMemsetAsync(f_count.p, 0, 16, st));
            q.queue_ctr = h->opt_dynamic_queue ? f_count.as<unsigned int>() + 2 : nullptr;
            if (filter) {
                if ((rc = f_list.reserve(static_cast<size_t>(Bl) * 4))) return rc;
                bp::FilterParams f{};
                f.s = static_cast<int>(h->s); f.n = static_cast<int>(h->n); f.SW = h->SW; f.NW = h->NW; f.B = Bl;
                f.vars = d.f_vars.as<bp::FilterVar>();
                f.syn_words = q.syn_words; f.err_words = q.err_words; f.out_bits = q.out_bits; f.conv = q.conv; f.iters = q.iters;
                f.list = f_list.as<int>(); f.list_count = f_count.as<int>(); f.counters = counters;
                const int fsmem = (2 * h->SW + h->NW) * 32 * 4 * bp::kFilterWarps;
                const int fgrid = static_cast<int>(std::min<int64_t>((Bl + bp::kFilterThreads - 1) / bp::kFilterThreads, static_cast<int64_t>(d.sm_count) * 16));
                if (fsmem > 48 * 1024) CU(cudaFuncSetAttribute(bp::first_iter_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fsmem));
                bp::first_iter_filter_kernel<<<fgrid, bp::kFilterThreads, fsmem, st>>>(f);
                h->launches++;
                q.list = f_list.as<int>(); q.list_count = f_count.as<int>();
            }
            const long long groups = (Bl + 31) / 32;
            KernelTimer timer(h, d, st);
            const int teams = h->dual ? 2 : 1;
            const int gl = static_cast<int>(std::min<long long>((groups + teams - 1) / teams, static_cast<long long>(d.sm_count) * h->ctas_per_sm));
            CU(launch_kernel(q.prof ? h->kernel_prof : h->kernel, gl, teams * thr, h->smem_bytes, st, q));
            h->launches++;
        }
    } else {
        if (h->opt_dynamic_queue) {                       // CTAs claim 32-syndrome chunks from a zeroed counter
            if ((rc = f_count.reserve(16))) return rc;
            CU(cudaMemsetAsync(f_count.p, 0, 16, st));
            p.queue_ctr = f_count.as<unsigned int>() + 2;
        }
        KernelTimer timer(h, d, st);
        CU(launch_kernel(h->kernel, grid, thr, h->smem_bytes, st, p));
        h->launches++;
    }
    CU(cudaGetLastError());
    return 0;
}

// ---- OSD (osd.cuh)
constexpr int kOsdThreads = 256;

int osd_layout(const ldpcb200 *h, bp::OsdParams &p)
{
    const int m = static_cast<int>(h->s), n = static_cast<int>(h->n);
    int g = (n + 1 + 127) / 128;              // 16-byte groups per augmented row
    if ((g & 1) == 0) ++g;                    // odd: 8 consecutive rows hit 8 distinct bank quads
    p.m = m; p.n = n; p.NWr = 4 * g;
    int np = 2;
    while (np < n) np <<= 1;
    p.NP = np;
    p.SW = h->SW; p.NW = h->NW;
    long long off = static_cast<long long>(m) * p.NWr * 4;
    off = (off + 15) / 16 * 16;
    p.off_key = static_cast<int>(off); off += static_cast<long long>(np) * 8;
    p.off_idx = static_cast<int>(off); off += static_cast<long long>(np) * 4;
    p.off_piv = static_cast<int>(off); off += static_cast<long long>(std::max(m, 1)) * 4 * 5 + static_cast<long long>(p.NWr) * 4;   // piv, prow, pcol, list, rowat (+ the order-O kernel's error words)
    p.off_red = static_cast<int>(off); off += (16 + 192 + p.NWr / 4 + 1) * 4;
    return off > 0x7fffffffLL ? 0x7fffffff : static_cast<int>(off);
}

// OSD of order `order`, stream-ordered; err_words: BP decisions in, OSD result out.  Order 0 (OSD-0, osd0_kernel) runs
// on the syndromes BP left unconverged, a higher order (osdk_kernel) on every syndrome of the batch.
int osd_on_device(ldpcb200 *h, DeviceCtx &d, DeviceCtx::StageSet &S, int64_t B, int order, const uint32_t *syn_words,
                  uint32_t *err_words, const uint8_t *conv, const double *ratio, unsigned long long *stats, cudaStream_t st)
{
    if (B <= 0) return 0;
    const char *what = order > 0 ? "OSD" : "OSD-0";
    if (h->variant != LDPCB200_VARIANT_EXACT)
        return fail(LDPCB200_EUNSUPPORTED, "%s is defined on the posterior ratios of the exact variant", what);
    if (order < 0 || order > bp::kOsdMaxOrder) return fail(LDPCB200_EUNSUPPORTED, "osd_order must be between 0 and %d", bp::kOsdMaxOrder);
    if (B > 0x7fffffffLL) return fail(LDPCB200_EINVAL, "%s: at most 2^31-1 syndromes per call", what);
    if (order == 0 && h->s > static_cast<int64_t>(bp::kOsdMaxRowsPerThread) * kOsdThreads)
        return fail(LDPCB200_EUNSUPPORTED, "OSD-0: more than %d checks", bp::kOsdMaxRowsPerThread * kOsdThreads);
    CU(cudaSetDevice(d.device));
    bp::OsdParams p{};
    const int smem = osd_layout(h, p);
    if (smem > d.smem_optin)
        return fail(LDPCB200_EUNSUPPORTED, "%s: the bit-packed %lld x %lld matrix (%d bytes) does not fit in shared memory", what,
                    static_cast<long long>(h->s), static_cast<long long>(h->n), smem);
    int rc;
    if (order == 0 && (rc = S.osd_list.reserve(static_cast<size_t>(B) * 4))) return rc;
    if ((rc = S.osd_ctl.reserve(16))) return rc;
    if (!stats) {
        if ((rc = d.osd_stats.reserve(64))) return rc;
        stats = d.osd_stats.as<unsigned long long>();
    }
    CU(cudaMemsetAsync(S.osd_ctl.p, 0, 16, st));
    p.colptr = d.d_colptr; p.rowval = d.d_ve_chk;
    p.syn_words = syn_words; p.err_words = err_words; p.ratio = ratio;
    p.queue = S.osd_ctl.as<int>() + 1;
    p.stats = stats;
    const int per_sm = std::max(1, std::min(4, d.smem_per_sm / (smem + 1024)));
    const int grid = static_cast<int>(std::min<int64_t>(B, static_cast<int64_t>(d.sm_count) * per_sm));
    auto launch = [&](auto kern, auto... args) -> cudaError_t {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        kern<<<grid, kOsdThreads, smem, st>>>(args...);
        return cudaSuccess;
    };
    if (order > 0) {
        CU(launch(bp::osdk_kernel<kOsdThreads>, p, order, static_cast<long long>(B)));
        h->launches++;
    } else {
        p.list = S.osd_list.as<int>(); p.count = S.osd_ctl.as<int>();
        p.profile = h->opt_osd_profile;
        bp::osd_collect_kernel<<<static_cast<unsigned>((B + 255) / 256), 256, 0, st>>>(conv, B, S.osd_list.as<int>(), S.osd_ctl.as<int>());
        switch ((p.m + kOsdThreads - 1) / kOsdThreads) {
            case 0: case 1: CU(launch(bp::osd0_kernel<kOsdThreads, 1>, p)); break;
            case 2: CU(launch(bp::osd0_kernel<kOsdThreads, 2>, p)); break;
            case 3: CU(launch(bp::osd0_kernel<kOsdThreads, 3>, p)); break;
            case 4: CU(launch(bp::osd0_kernel<kOsdThreads, 4>, p)); break;
            default: CU(launch(bp::osd0_kernel<kOsdThreads, 8>, p)); break;
        }
        h->launches += 2;
    }
    CU(cudaGetLastError());
    return 0;
}

// OSD of the handle's order after BP: where BP ran no iteration, log_probabs stays zero (reset!, belief_propagation.jl:86)
// and the ratios are 1 everywhere.  Statistics go to d.osd_stats.
int osd_after_bp(ldpcb200 *h, DeviceCtx &d, DeviceCtx::StageSet &S, int64_t B, const uint32_t *syn_words, uint32_t *err_words,
                 const uint8_t *conv, double *ratio, cudaStream_t st)
{
    if (h->max_iters <= 0) {
        bp::osd_fill_ones_kernel<<<grid_for(B * h->n, d.sm_count), 256, 0, st>>>(ratio, B * h->n);
        h->launches++;
    }
    return osd_on_device(h, d, S, B, h->opt_osd_order, syn_words, err_words, conv, ratio, d.osd_stats.as<unsigned long long>(), st);
}

// ---- BP-OTS (bpots.cuh): one CTA per syndrome.  Stream-ordered.
// The per-syndrome arrays (16 E + 23 n + 4 s bytes) live in shared memory when they fit; otherwise every CTA of the grid
// gets its own slice of the device's workspace d.bpots_ws.  That workspace is shared by all BP-OTS launches on the device:
// launches that use it must not overlap (host-batch chunks are ordered by decode_done; device-resident calls follow the
// one-in-flight-call-per-handle rule).
struct BpotsArgs { int T; double C; };

int bpots_on_device(ldpcb200 *h, DeviceCtx &d, int64_t B, const uint32_t *syn_words, uint32_t *err_words, uint8_t *conv, int32_t *iters,
                    const BpotsArgs &a, unsigned long long *counters, cudaStream_t st)
{
    if (B <= 0) return 0;
    CU(cudaSetDevice(d.device));
    if (a.T < 1) return fail(LDPCB200_EINVAL, "BP-OTS: the biasing period T must be at least 1");
    bp::BpotsParams p{};
    p.s = static_cast<int>(h->s); p.n = static_cast<int>(h->n); p.E = static_cast<int>(h->E);
    p.SW = h->SW; p.NW = h->NW; p.max_iters = h->max_iters; p.T = a.T; p.C = a.C; p.B = B;
    {   // log.((1 .- (2*per/3)) ./ (2*per/3))  (bpots_decoder.jl:231), IEEE double on the host
        volatile double q = 2 * h->per / 3;
        volatile double r = (1 - q) / q;
        p.prior = std::log(r);
    }
    long long off = static_cast<long long>(std::max<int64_t>(h->E, 1)) * 8;
    p.off_cv = static_cast<int>(off);     off *= 2;
    p.off_omega = static_cast<int>(off);  off += static_cast<long long>(std::max<int64_t>(h->n, 1)) * 8;
    p.off_llr = static_cast<int>(off);    off += static_cast<long long>(std::max<int64_t>(h->n, 1)) * 8;
    p.off_osc = static_cast<int>(off);    off += static_cast<long long>(std::max<int64_t>(h->n, 1)) * 4;
    p.off_par = static_cast<int>(off);    off += static_cast<long long>(std::max<int64_t>(h->s, 1)) * 4;
    p.off_dec = static_cast<int>(off);    off += 3 * std::max<int64_t>(h->n, 1);
    off = (off + 15) / 16 * 16;
    const long long arrays = off;                     // bytes of the per-syndrome arrays
    if (arrays > 0x7fffffffLL)
        return fail(LDPCB200_EUNSUPPORTED, "BP-OTS: the arrays of one syndrome (%lld bytes) exceed 2^31 bytes", arrays);
    const bool fits = arrays + 512 <= d.smem_optin;
    if (h->opt_bpots_memory == 1 && !fits)
        return fail(LDPCB200_EUNSUPPORTED, "BP-OTS: the two message arrays of one syndrome (%lld bytes with state) do not fit in shared memory "
                    "(option bpots_memory = 1)", arrays + 512);
    p.rowptr = d.d_rowptr; p.colptr = d.d_colptr; p.ve_slot = d.d_ve_slot; p.ve_chk = d.d_ve_chk;
    p.syn_words = syn_words; p.err_words = err_words; p.conv = conv; p.iters = iters; p.counters = counters;
    if (fits && h->opt_bpots_memory != 2) {
        p.off_red = static_cast<int>(arrays);
        const int smem = static_cast<int>(arrays + 512);
        const int per_sm = std::max(1, std::min(8, d.smem_per_sm / (smem + 1024)));
        const int grid = static_cast<int>(std::min<int64_t>(B, static_cast<int64_t>(d.sm_count) * per_sm));
        CU(cudaFuncSetAttribute(bp::bpots_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        bp::bpots_kernel<false><<<grid, bp::kBpotsThreads, smem, st>>>(p);
    } else {
        // grid: resident CTAs, at most one per syndrome, and at most a quarter of the free device memory in slices
        const long long slice = (arrays + 255) / 256 * 256;
        int occ = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bp::bpots_kernel<true>, bp::kBpotsThreads, 512));
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        const long long cap = static_cast<long long>((free_b + d.bpots_ws.cap) / 4);
        if (slice > cap)
            return fail(LDPCB200_ENOMEM, "BP-OTS: the workspace of one syndrome (%lld bytes) exceeds a quarter of the free device memory", slice);
        const int grid = static_cast<int>(std::min<int64_t>({B, static_cast<int64_t>(d.sm_count) * std::max(occ, 1), cap / slice}));
        int rc = d.bpots_ws.reserve(static_cast<size_t>(grid) * static_cast<size_t>(slice));
        if (rc) return rc;
        p.ws = d.bpots_ws.as<unsigned char>();
        p.slice_bytes = slice;
        p.off_red = 0;
        bp::bpots_kernel<true><<<grid, bp::kBpotsThreads, 512, st>>>(p);
    }
    h->launches++;
    CU(cudaGetLastError());
    return 0;
}

size_t fmt_bytes(int fmt, int64_t rows, int64_t ld, int64_t B, int RW)
{
    switch (fmt) {
        case LDPCB200_FMT_U8: return static_cast<size_t>(B ? (B - 1) * ld + rows : 0);
        case LDPCB200_FMT_I64: return static_cast<size_t>(B ? (B - 1) * ld + rows : 0) * 8;
        case LDPCB200_FMT_F64: return static_cast<size_t>(B ? (B - 1) * ld + rows : 0) * 8;
        case LDPCB200_FMT_BITS: return static_cast<size_t>((B * rows + 31) / 32) * 4;
        case LDPCB200_FMT_PACKED32: return static_cast<size_t>(B) * RW * 4;
    }
    return 0;
}

// Packed rows from B syndromes in the caller's format, already on the device at `raw` (U8 / I64: column stride ld).
// PACKED32 needs no kernel: those rows are copied to syn_words as they are.
void pack_syndromes(ldpcb200 *h, DeviceCtx &d, int fmt, const void *raw, int64_t ld, int64_t B, uint32_t *syn_words, cudaStream_t st)
{
    if (fmt == LDPCB200_FMT_PACKED32) return;
    const int g = grid_for(B * h->SW, d.sm_count), s = static_cast<int>(h->s);
    if (fmt == LDPCB200_FMT_BITS)
        bp::pack_bits<<<g, 256, 0, st>>>(static_cast<const uint32_t *>(raw), (B * h->s + 31) / 32, s, h->SW, B, syn_words);
    else if (fmt == LDPCB200_FMT_U8)
        bp::pack_elems<uint8_t><<<g, 256, 0, st>>>(static_cast<const uint8_t *>(raw), ld, s, h->SW, B, syn_words);
    else
        bp::pack_elems<long long><<<g, 256, 0, st>>>(static_cast<const long long *>(raw), ld, s, h->SW, B, syn_words);
    h->launches++;
}

// The caller's error format (BITS, U8, I64 or F64; column stride ld for the element formats) from B packed rows, on the device.
void unpack_errors(ldpcb200 *h, DeviceCtx &d, int fmt, const uint32_t *err_words, int64_t B, void *raw, int64_t ld, cudaStream_t st)
{
    const int g = grid_for(B * h->NW, d.sm_count), n = static_cast<int>(h->n);
    if (fmt == LDPCB200_FMT_BITS) {
        const long long nw = (B * h->n + 31) / 32;
        bp::unpack_bits<<<grid_for(nw, d.sm_count), 256, 0, st>>>(err_words, n, h->NW, B, static_cast<uint32_t *>(raw), nw);
    } else if (fmt == LDPCB200_FMT_U8) {
        bp::unpack_elems<uint8_t><<<g, 256, 0, st>>>(err_words, n, h->NW, B, static_cast<uint8_t *>(raw), ld);
    } else if (fmt == LDPCB200_FMT_I64) {
        bp::unpack_elems<long long><<<g, 256, 0, st>>>(err_words, n, h->NW, B, static_cast<long long *>(raw), ld);
    } else {
        bp::unpack_elems<double><<<g, 256, 0, st>>>(err_words, n, h->NW, B, static_cast<double *>(raw), ld);
    }
    h->launches++;
}

// Small host batch (decode! and a handful of columns): everything goes through ONE device block and its pinned
// mirror -- one host->device copy, the kernels, one device->host copy, one synchronisation -- instead of the
// chunked double-buffered pipeline below, whose fixed cost (~10 API calls and 4 blocking copies) dominates here.
int decode_host_tiny(ldpcb200 *h, DeviceCtx &d, int64_t B, const void *syndromes, int syn_fmt, int64_t syn_ld, void *errors,
                     int err_fmt, int64_t err_ld, uint8_t *converged, int32_t *iters, double *ratio, int64_t *counters_out)
{
    const int64_t s = h->s, n = h->n;
    cudaStream_t st = d.set[0].stream;
    auto up16 = [](size_t x) { return (x + 15) / 16 * 16; };
    const size_t in_bytes = fmt_bytes(syn_fmt, s, syn_ld, B, h->SW), out_bytes = fmt_bytes(err_fmt, n, err_ld, B, h->NW);
    const size_t synw_bytes = static_cast<size_t>(B) * h->SW * 4, errw_bytes = static_cast<size_t>(B) * h->NW * 4;
    // device block:  [in_raw | syn_words | err_words]  then the part copied back: [out_raw | conv | iters | ratio | counters]
    const size_t o_in = 0, o_synw = up16(in_bytes), o_errw = o_synw + up16(synw_bytes), o_out = o_errw + up16(errw_bytes);
    const size_t o_conv = o_out + up16(out_bytes), o_iters = o_conv + up16(static_cast<size_t>(B));
    const size_t o_ratio = o_iters + up16(static_cast<size_t>(B) * 4);
    const size_t o_ctr = o_ratio + (ratio ? up16(static_cast<size_t>(B) * n * 8) : 0);
    const size_t total = o_ctr + LDPCB200_NUM_COUNTERS * 8;
    int rc;
    if ((rc = d.tiny.reserve(total)) || (rc = d.tiny_host.reserve(total))) return rc;
    unsigned char *D = d.tiny.as<unsigned char>(), *P = static_cast<unsigned char *>(d.tiny_host.p);
    uint32_t *syn_words = reinterpret_cast<uint32_t *>(D + o_synw), *err_words = reinterpret_cast<uint32_t *>(D + o_errw);
    // ---- in
    const bool in_packed = syn_fmt == LDPCB200_FMT_PACKED32;
    memcpy(P + o_in, syndromes, in_bytes);
    CU(cudaMemcpyAsync(in_packed ? static_cast<void *>(syn_words) : static_cast<void *>(D + o_in), P + o_in, in_bytes,
                       cudaMemcpyHostToDevice, st));
    pack_syndromes(h, d, syn_fmt, D + o_in, syn_ld, B, syn_words, st);
    // ---- decode
    CU(cudaMemsetAsync(D + o_out, 0, total - o_out, st));
    rc = decode_on_device(h, d, B, syn_words, err_words, D + o_conv, reinterpret_cast<int32_t *>(D + o_iters),
                          ratio ? reinterpret_cast<double *>(D + o_ratio) : nullptr,
                          reinterpret_cast<unsigned long long *>(D + o_ctr), st);
    if (rc) return rc;
    // ---- out
    if (err_fmt == LDPCB200_FMT_PACKED32) CU(cudaMemcpyAsync(D + o_out, err_words, errw_bytes, cudaMemcpyDeviceToDevice, st));
    else unpack_errors(h, d, err_fmt, err_words, B, D + o_out, err_ld, st);
    CU(cudaMemcpyAsync(P + o_out, D + o_out, total - o_out, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const bool elems = err_fmt == LDPCB200_FMT_U8 || err_fmt == LDPCB200_FMT_I64 || err_fmt == LDPCB200_FMT_F64;
    if (elems && err_ld != n) {          // strided destination: only the n rows of each column belong to the caller
        const size_t esz = err_fmt == LDPCB200_FMT_U8 ? 1 : 8;
        for (int64_t b = 0; b < B; ++b)
            memcpy(static_cast<unsigned char *>(errors) + static_cast<size_t>(b) * err_ld * esz, P + o_out + static_cast<size_t>(b) * err_ld * esz,
                   static_cast<size_t>(n) * esz);
    } else {
        memcpy(errors, P + o_out, out_bytes);
    }
    memcpy(converged, P + o_conv, static_cast<size_t>(B));
    if (iters) memcpy(iters, P + o_iters, static_cast<size_t>(B) * 4);
    if (ratio) memcpy(ratio, P + o_ratio, static_cast<size_t>(B) * n * 8);
    unsigned long long hc[LDPCB200_NUM_COUNTERS];
    memcpy(hc, P + o_ctr, sizeof(hc));
    for (int k = 0; k < LDPCB200_NUM_COUNTERS; ++k) counters_out[k] = static_cast<int64_t>(hc[k]);
    return 0;
}

// memcpy between caller memory and a pinned staging block, split over a few host threads when it is large
void par_memcpy(void *dst, const void *src, size_t bytes)
{
    const size_t kSlice = 8u << 20;
    if (bytes < 2 * kSlice) { memcpy(dst, src, bytes); return; }
    const int nt = static_cast<int>(std::min<size_t>(4, bytes / kSlice));
    const size_t per = (bytes / nt + 63) / 64 * 64;
    std::vector<std::thread> th;
    for (int t = 1; t < nt; ++t) {
        const size_t o = per * t, len = std::min(per, bytes - std::min(bytes, o));
        if (len) th.emplace_back([=] { memcpy(static_cast<char *>(dst) + o, static_cast<const char *>(src) + o, len); });
    }
    memcpy(dst, src, std::min(per, bytes));
    for (auto &t : th) t.join();
}

// Ordinary (pageable) host memory?  cudaMemcpyAsync from/to it is staged by the driver and blocks the calling thread,
// which serialises the two-stream pipeline below; pinned or registered memory (cudaHostAlloc, cudaHostRegister,
// CUDA.jl's pinned arrays) is copied directly.
bool is_pageable(const void *p)
{
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

// One device's share [b0, b0+Bd) of a host batch, processed in chunks.
int decode_host_range(ldpcb200 *h, DeviceCtx &d, int64_t b0, int64_t Bd, int64_t Btot, const void *syndromes,
                      int syn_fmt, int64_t syn_ld, void *errors, int err_fmt, int64_t err_ld, uint8_t *converged,
                      int32_t *iters, double *ratio, int64_t *counters_out, bool osd = false, int64_t *osd_stats_out = nullptr,
                      const BpotsArgs *ots = nullptr)
{
    CU(cudaSetDevice(d.device));
    const int64_t s = h->s, n = h->n;
    {
        const int64_t limit = h->opt_small_batch < 0 ? d.sm_count : h->opt_small_batch;
        if (!osd && !ots && b0 == 0 && Bd == Btot && Bd <= limit && h->opt_chunk <= 0 &&
            static_cast<double>(Bd) * (static_cast<double>(n) * 8.0 * (ratio ? 2 : 1) + static_cast<double>(s) * 8.0) < 64.0 * 1048576.0)
            return decode_host_tiny(h, d, Bd, syndromes, syn_fmt, syn_ld, errors, err_fmt, err_ld, converged, iters, ratio, counters_out);
    }
    // chunk size: bound the staging footprint (two sets are in flight)
    const double per_syn = static_cast<double>(fmt_bytes(syn_fmt, s, syn_ld, 2, h->SW) - fmt_bytes(syn_fmt, s, syn_ld, 1, h->SW)) +
                           static_cast<double>(fmt_bytes(err_fmt, n, err_ld, 2, h->NW) - fmt_bytes(err_fmt, n, err_ld, 1, h->NW)) +
                           (h->SW + h->NW) * 4.0 + 5.0 + ((ratio || osd) ? 8.0 * n : 0.0) + (osd ? 4.0 : 0.0);
    // about four chunks per call (every chunk ends with a tail of slow syndromes, so fewer is better, but
    // at least two are needed to overlap copies with decoding); never less than two waves of the
    // resident slots (a smaller chunk leaves SMs idle); staging bounded by 256 MB per set, or what
    // two waves need (<= 2 GB)
    const double two_waves = 2.0 * h->slots * std::max(per_syn, 1.0);
    // (the OSD pipeline keeps n posterior ratios per syndrome on the device: its chunks are bounded by 2 GB, and two
    // chunks per call are enough to overlap the copies -- every chunk pays a BP tail and an OSD tail)
    const double budget = osd ? 2048.0 * 1048576.0 : std::min(std::max(256.0 * 1048576.0, two_waves), 2048.0 * 1048576.0);
    // pageable caller buffers are staged through pinned memory by this thread: more, smaller chunks keep the part of
    // that host-side copying that cannot overlap GPU work (first chunk in, last chunk out) small
    const bool pg_in = h->opt_stage_pageable && is_pageable(syndromes);
    const bool pg_out = h->opt_stage_pageable && is_pageable(errors);
    const bool pg_conv = h->opt_stage_pageable && is_pageable(converged), pg_iters = h->opt_stage_pageable && is_pageable(iters),
               pg_ratio = h->opt_stage_pageable && is_pageable(ratio);
    // (where the decoding kernels of consecutive chunks may overlap -- shared-memory kernel -- a chunk's tail of slow
    //  syndromes costs nothing, and six chunks measured best: C3 10 M BitMatrix 3.49e8 -> 3.65e8 syndromes/s end to end)
    // (BitMatrix output written by the decoding kernel itself needs no conversion kernel after the decode: overlapping is
    //  then safe in every regime; otherwise see the comment at `ordered` below)
    const bool direct_out = err_fmt == LDPCB200_FMT_BITS && h->lean && !osd && !ots && h->opt_direct_bits;
    const bool may_overlap = h->lean && !osd && !ots && h->opt_overlap_chunks && !pg_in && !pg_out &&
                             (h->opt_overlap_chunks == 2 || direct_out || h->last_milli_iters.load() >= 2000);
    const int nchunk_target = osd ? 2 : ((pg_in || pg_out) ? 8 : (may_overlap ? 6 : 4));
    int64_t CH = h->opt_chunk > 0 ? h->opt_chunk
                                  : std::max<int64_t>({(Bd + nchunk_target - 1) / nchunk_target, 32768, 2 * static_cast<int64_t>(h->slots)});
    CH = std::min<int64_t>(CH, static_cast<int64_t>(budget / std::max(per_syn, 1.0)));
    CH = std::max<int64_t>(32, (CH + 31) / 32 * 32);
    int rc;
    if ((rc = d.counters.reserve(LDPCB200_NUM_COUNTERS * 8))) return rc;
    CU(cudaMemsetAsync(d.counters.p, 0, LDPCB200_NUM_COUNTERS * 8, d.set[0].stream));
    if (osd) {
        if ((rc = d.osd_stats.reserve(64))) return rc;
        CU(cudaMemsetAsync(d.osd_stats.p, 0, 64, d.set[0].stream));
    }
    CU(cudaStreamSynchronize(d.set[0].stream));
    bool have_prev_decode = false;
    int64_t chunk_no = 0;
    for (int64_t c0 = 0; c0 < Bd; c0 += CH, ++chunk_no) {
        DeviceCtx::StageSet &S = d.set[chunk_no & 1];
        cudaStream_t st = S.stream;
        CU(cudaStreamSynchronize(st));                    // the chunk that used this set two steps ago has landed
        for (const auto &pd : S.pending) par_memcpy(pd.dst, pd.src, pd.bytes);      // ... hand its staged outputs to the caller
        S.pending.clear();
        S.pin_out_used = 0;
        const int64_t Bc = std::min(CH, Bd - c0);
        const int64_t g0 = b0 + c0;                       // first global column of this chunk
        // copies between the caller's memory and the device, through the pinned staging blocks when that memory is pageable
        auto h2d = [&](void *dst_dev, const void *src_host, size_t bytes, bool staged) -> int {
            if (staged) {
                int r_ = S.pin_in.reserve(bytes);
                if (r_) return r_;
                par_memcpy(S.pin_in.p, src_host, bytes);
                src_host = S.pin_in.p;
            }
            CU(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, st));
            return 0;
        };
        auto d2h = [&](void *dst_host, const void *src_dev, size_t bytes, bool staged) -> int {
            if (staged) {
                unsigned char *q = static_cast<unsigned char *>(S.pin_out.p) + S.pin_out_used;
                S.pin_out_used += (bytes + 255) / 256 * 256;
                S.pending.push_back({dst_host, q, bytes});
                dst_host = q;
            }
            CU(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, st));
            return 0;
        };
        {   // one pinned output block per chunk, sized before the first copy is issued (it must not move afterwards)
            size_t need_out = 0;
            auto up = [](size_t x) { return (x + 255) / 256 * 256; };
            if (pg_out) need_out += up(fmt_bytes(err_fmt, n, err_ld, Bc, h->NW) + 8);
            if (pg_conv) need_out += up(static_cast<size_t>(Bc));
            if (pg_iters) need_out += up(static_cast<size_t>(Bc) * 4);
            if (pg_ratio) need_out += up(static_cast<size_t>(Bc) * n * 8);
            if (need_out && (rc = S.pin_out.reserve(need_out))) return rc;
        }
        if ((rc = S.syn_words.reserve(static_cast<size_t>(Bc) * h->SW * 4))) return rc;
        if ((rc = S.err_words.reserve(static_cast<size_t>(Bc) * h->NW * 4))) return rc;
        if ((rc = S.conv.reserve(static_cast<size_t>(Bc)))) return rc;
        if ((rc = S.iters.reserve(static_cast<size_t>(Bc) * 4))) return rc;
        if ((ratio || osd) && (rc = S.ratio.reserve(static_cast<size_t>(Bc) * n * 8))) return rc;
        // ---- syndromes -> device -> packed rows
        uint32_t *syn_words = S.syn_words.as<uint32_t>();
        if (syn_fmt == LDPCB200_FMT_PACKED32) {
            if ((rc = h2d(syn_words, static_cast<const uint32_t *>(syndromes) + g0 * h->SW, static_cast<size_t>(Bc) * h->SW * 4, pg_in))) return rc;
        } else {
            // column g0 of the caller's buffer (g0 is a multiple of 32: whole words of the bit stream)
            const size_t at = syn_fmt == LDPCB200_FMT_BITS ? static_cast<size_t>(g0 * s / 8)
                                                           : static_cast<size_t>(g0 * syn_ld) * (syn_fmt == LDPCB200_FMT_I64 ? 8 : 1);
            const size_t bytes = fmt_bytes(syn_fmt, s, syn_ld, Bc, h->SW);
            if ((rc = S.raw_in.reserve(bytes))) return rc;
            if ((rc = h2d(S.raw_in.p, static_cast<const uint8_t *>(syndromes) + at, bytes, pg_in))) return rc;
            pack_syndromes(h, d, syn_fmt, S.raw_in.p, syn_ld, Bc, syn_words, st);
        }
        // BitMatrix output: the shared-memory kernel writes the caller's bit stream itself (no conversion kernel between the
        // decode and the copy out)
        uint32_t *direct_bits = nullptr;
        bool bits_done = false;
        if (direct_out) {
            const size_t nwb = static_cast<size_t>((Bc * n + 31) / 32);
            if ((rc = S.raw_out.reserve(nwb * 4))) return rc;
            direct_bits = S.raw_out.as<uint32_t>();
        }
        // ---- decode (kernels of consecutive chunks share the per-device message store: keep them ordered)
        // (the shared-memory kernel keeps everything on chip and its filter list is per set: there the next chunk's kernel
        //  may start while the previous one is still finishing its slowest syndromes)
        // That only pays when the call is compute-bound and the caller's buffers are pinned: a decoding kernel that starts
        // early holds every SM until it ends, so the previous chunk's conversion kernel and copy out wait for it -- in a
        // copy- or host-bound call (low error rate, pageable buffers) that delay is the whole call (measured: -25 % / -20 %).
        // The handle therefore looks at the mean iteration count of its previous host batch: overlap from 2 iterations up.
        const bool ordered = !may_overlap;
        if (have_prev_decode && ordered) CU(cudaStreamWaitEvent(st, d.decode_done, 0));
        // (OSD-0 only reads the ratios of unconverged syndromes: those of iteration max_iters; a higher order post-processes
        //  every syndrome, so the ratios of each syndrome's own last iteration are needed)
        if (ots)
            rc = bpots_on_device(h, d, Bc, syn_words, S.err_words.as<uint32_t>(), S.conv.as<uint8_t>(), S.iters.as<int32_t>(), *ots,
                                 nullptr, st);
        else
        rc = decode_on_device(h, d, Bc, syn_words, S.err_words.as<uint32_t>(), S.conv.as<uint8_t>(), S.iters.as<int32_t>(),
                              (ratio || (osd && h->max_iters > 0)) ? S.ratio.as<double>() : nullptr,
                              d.counters.as<unsigned long long>(), st, osd && !ratio && h->opt_osd_order == 0, &S, direct_bits, &bits_done);
        if (rc) return rc;
        CU(cudaEventRecord(d.decode_done, st));
        have_prev_decode = true;
        if (osd && (rc = osd_after_bp(h, d, S, Bc, syn_words, S.err_words.as<uint32_t>(), S.conv.as<uint8_t>(), S.ratio.as<double>(), st)))
            return rc;
        // ---- packed rows -> caller's format -> host
        if (err_fmt == LDPCB200_FMT_PACKED32) {
            if ((rc = d2h(static_cast<uint32_t *>(errors) + g0 * h->NW, S.err_words.p, static_cast<size_t>(Bc) * h->NW * 4, pg_out))) return rc;
        } else {
            const bool bits = err_fmt == LDPCB200_FMT_BITS;
            const size_t bytes = fmt_bytes(err_fmt, n, err_ld, Bc, h->NW), esz = err_fmt == LDPCB200_FMT_U8 ? 1 : 8;
            // column g0 of the caller's buffer (g0 is a multiple of 32: whole words of the bit stream)
            uint8_t *dst = static_cast<uint8_t *>(errors) + (bits ? static_cast<size_t>(g0 * n / 8) : static_cast<size_t>(g0) * err_ld * esz);
            if ((rc = S.raw_out.reserve(bytes))) return rc;
            if (!bits && err_ld != n) CU(cudaMemsetAsync(S.raw_out.p, 0, bytes, st));
            if (!bits_done) unpack_errors(h, d, err_fmt, S.err_words.as<uint32_t>(), Bc, S.raw_out.p, err_ld, st);
            // (the last word of a chunk may hold bits of the next chunk's first column only when Bc*n is not a multiple
            //  of 32, i.e. in the final chunk of the batch: chunk boundaries are multiples of 32 columns)
            if (bits || err_ld == n) {
                if ((rc = d2h(dst, S.raw_out.p, bytes, pg_out))) return rc;
            } else {   // strided destination: only the n rows of each column belong to the caller
                CU(cudaMemcpy2DAsync(dst, err_ld * esz, S.raw_out.p, err_ld * esz, n * esz, Bc, cudaMemcpyDeviceToHost, st));
            }
        }
        if ((rc = d2h(converged + g0, S.conv.p, static_cast<size_t>(Bc), pg_conv))) return rc;
        if (iters && (rc = d2h(iters + g0, S.iters.p, static_cast<size_t>(Bc) * 4, pg_iters))) return rc;
        if (ratio && (rc = d2h(ratio + g0 * n, S.ratio.p, static_cast<size_t>(Bc) * n * 8, pg_ratio))) return rc;
    }
    {   // drain both sets, the older chunk first, and hand the staged outputs to the caller
        const int last = static_cast<int>((chunk_no + 1) & 1), prev = static_cast<int>(chunk_no & 1);   // chunk_no = chunks issued
        for (int k : {prev, last}) {
            DeviceCtx::StageSet &S = d.set[k];
            CU(cudaStreamSynchronize(S.stream));
            for (const auto &pd : S.pending) par_memcpy(pd.dst, pd.src, pd.bytes);
            S.pending.clear();
            S.pin_out_used = 0;
        }
    }
    cudaStream_t st = d.set[0].stream;
    unsigned long long hc[LDPCB200_NUM_COUNTERS];
    CU(cudaMemcpyAsync(hc, d.counters.p, sizeof(hc), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int k = 0; k < LDPCB200_NUM_COUNTERS; ++k) counters_out[k] = static_cast<int64_t>(hc[k]);
    if (hc[0] > 0) h->last_milli_iters.store(static_cast<int>(std::min<unsigned long long>(1000ull * hc[2] / hc[0], 1000000ull)));
    if (osd && osd_stats_out) {
        unsigned long long ho[4] = {0, 0, 0, 0};
        CU(cudaMemcpyAsync(ho, d.osd_stats.p, sizeof(ho), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        for (int k = 0; k < LDPCB200_NUM_OSD_STATS; ++k) osd_stats_out[k] = static_cast<int64_t>(ho[k]);
    }
    return 0;
}

// Communicators for the handle's device set (lazy: the first multi-device batch that asks for counters).
void nccl_prepare(ldpcb200 *h)
{
    if (h->nccl_state != 0) return;
    h->nccl_state = -1;
    const int nd = static_cast<int>(h->dev.size());
    if (nd < 2 || !h->opt_nccl) { h->nccl_why = nd < 2 ? "single device" : "disabled by option"; return; }
    std::vector<int> devs;
    for (const DeviceCtx &d : h->dev) {
        if (std::find(devs.begin(), devs.end(), d.device) != devs.end()) { h->nccl_why = "a device is listed twice (NCCL needs distinct devices)"; return; }
        devs.push_back(d.device);
    }
    if (!nccl_load()) { h->nccl_why = g_nccl.why; return; }
    h->comms.assign(nd, nullptr);
    ncclResult_t r = g_nccl.CommInitAll(h->comms.data(), nd, devs.data());
    if (r != ncclSuccess) { h->nccl_why = std::string("ncclCommInitAll: ") + g_nccl.GetErrorString(r); h->comms.clear(); return; }
    h->nccl_state = 1;
}

// Sum per-device counter blocks (`count` x uint64 at src(d), complete on d.set[0].stream) over all devices of the
// handle with one grouped ncclAllReduce; the result of device 0 goes to `out`.
template <class Src>
int nccl_sum_block(ldpcb200 *h, int count, Src src, int64_t *out)
{
    const int nd = static_cast<int>(h->dev.size());
    for (int k = 0; k < nd; ++k) {
        DeviceCtx &d = h->dev[k];
        CU(cudaSetDevice(d.device));
        int rc = d.ctr_sum.reserve(16 * 8);
        if (rc) return rc;
    }
    ncclResult_t r = g_nccl.GroupStart();
    for (int k = 0; k < nd && r == ncclSuccess; ++k) {
        DeviceCtx &d = h->dev[k];
        r = g_nccl.AllReduce(src(d), d.ctr_sum.p, count, ncclUint64, ncclSum, h->comms[k], d.set[0].stream);
    }
    ncclResult_t r2 = g_nccl.GroupEnd();
    if (r == ncclSuccess) r = r2;
    if (r != ncclSuccess) return fail(LDPCB200_ECUDA, "ncclAllReduce of the counters: %s", g_nccl.GetErrorString(r));
    unsigned long long hc[16];
    for (int k = 0; k < nd; ++k) {
        DeviceCtx &d = h->dev[k];
        CU(cudaSetDevice(d.device));
        if (k == 0) CU(cudaMemcpyAsync(hc, d.ctr_sum.p, sizeof(unsigned long long) * count, cudaMemcpyDeviceToHost, d.set[0].stream));
        CU(cudaStreamSynchronize(d.set[0].stream));
    }
    for (int c = 0; c < count; ++c) out[c] = static_cast<int64_t>(hc[c]);
    return 0;
}

// Per-device blocks of `count` values each, added on the host into out
void host_sum(const std::vector<int64_t> &per_dev, int count, int64_t *out)
{
    for (size_t i = 0; i < per_dev.size(); ++i) out[i % count] += per_dev[i];
}

// Split `total` columns into contiguous per-device ranges, boundaries multiples of 32 (bit formats stay word aligned),
// and run work(k, first, count) for every device k: inline for one device, on one thread per device otherwise.
// Returns the first failing device's code, with its message.
template <class Work>
int fan_out(ldpcb200 *h, int64_t total, Work work)
{
    const int nd = static_cast<int>(h->dev.size());
    std::vector<int64_t> lo(nd + 1, 0);
    const int64_t blocks = (total + 31) / 32;
    for (int k = 0; k <= nd; ++k) lo[k] = std::min<int64_t>(total, (blocks * k / nd) * 32);
    lo[nd] = total;
    std::vector<int> rcs(nd, 0);
    std::vector<std::string> errs(nd);
    auto run = [&](int k) {
        rcs[k] = work(k, lo[k], lo[k + 1] - lo[k]);
        if (rcs[k]) errs[k] = g_err;
    };
    if (nd == 1) {
        run(0);
    } else {
        std::vector<std::thread> th;
        for (int k = 0; k < nd; ++k) th.emplace_back(run, k);
        for (auto &t : th) t.join();
    }
    for (int k = 0; k < nd; ++k)
        if (rcs[k]) { g_err = errs[k]; return rcs[k]; }
    return 0;
}

// B error rows with independent flips of probability per (rows first .. first+B-1 of the stream `seed`) and their syndromes,
// as packed rows on the device
int sample_on_device(ldpcb200 *h, DeviceCtx &d, int64_t B, int64_t first, uint64_t seed, double per, uint32_t *err_words,
                     uint32_t *syn_words, cudaStream_t st)
{
    const double t = std::floor(per * 4294967296.0);
    const uint32_t thr = !(t > 0) ? 0u : (t >= 4294967295.0 ? 0xFFFFFFFFu : static_cast<uint32_t>(t));
    CU(cudaMemsetAsync(syn_words, 0, static_cast<size_t>(B) * h->SW * 4, st));
    bp::sample_errors<<<grid_for(B * h->NW, d.sm_count), 256, 0, st>>>(static_cast<int>(h->n), h->NW, B, first, static_cast<uint32_t>(seed),
                                                                      static_cast<uint32_t>(seed >> 32), thr, err_words);
    bp::syndrome_of<<<grid_for(B * h->NW, d.sm_count), 256, 0, st>>>(d.d_colptr, d.d_ve_chk, h->NW, h->SW, B, err_words, syn_words);
    h->launches += 2;
    return 0;
}

// One device's share of the sampling + scoring harness: tiles of device-resident shots.
// ots: BP-OTS instead of BP (osd is then false).
int harness_on_device(ldpcb200 *h, DeviceCtx &d, int64_t first, int64_t shots, uint64_t seed, double per_channel, bool osd,
                      const BpotsArgs *ots, int64_t *out8)
{
    CU(cudaSetDevice(d.device));
    cudaStream_t st = d.set[0].stream;
    int rc;
    // [0..7] the harness counters, [8..11] the decode calls' own block (its slot 3 counts filter-finished syndromes)
    if ((rc = d.hs_ctr.reserve((LDPCB200_NUM_HARNESS_COUNTERS + LDPCB200_NUM_COUNTERS) * 8))) return rc;
    CU(cudaMemsetAsync(d.hs_ctr.p, 0, (LDPCB200_NUM_HARNESS_COUNTERS + LDPCB200_NUM_COUNTERS) * 8, st));
    if (shots > 0) {
        // tile: bounded by 64 MB of packed rows (and 1 GB of posterior ratios when OSD follows)
        int64_t tile = std::max<int64_t>(32, (64ll << 20) / (static_cast<int64_t>(h->SW + 2 * h->NW) * 4 + 5));
        if (osd) tile = std::min<int64_t>(tile, std::max<int64_t>(32, (1ll << 30) / (h->n * 8)));
        tile = std::min<int64_t>(std::max<int64_t>(tile, 2 * static_cast<int64_t>(h->slots)), shots);
        if ((rc = d.hs_truth.reserve(static_cast<size_t>(tile) * h->NW * 4)) || (rc = d.hs_err.reserve(static_cast<size_t>(tile) * h->NW * 4)) ||
            (rc = d.hs_syn.reserve(static_cast<size_t>(tile) * h->SW * 4)) || (rc = d.hs_conv.reserve(static_cast<size_t>(tile))) ||
            (rc = d.hs_iters.reserve(static_cast<size_t>(tile) * 4)) || (rc = d.scratch.reserve(static_cast<size_t>(tile) * h->SW * 4)))
            return rc;
        if (osd && (rc = d.hs_ratio.reserve(static_cast<size_t>(tile) * h->n * 8))) return rc;
        if (osd && (rc = d.osd_stats.reserve(64))) return rc;
        if (osd) CU(cudaMemsetAsync(d.osd_stats.p, 0, 64, st));
        if (!h->lmask.empty() && !d.lmask.p) {
            if ((rc = d.lmask.reserve(h->lmask.size() * 8))) return rc;
            CU(cudaMemcpyAsync(d.lmask.p, h->lmask.data(), h->lmask.size() * 8, cudaMemcpyHostToDevice, st));
        }
        unsigned long long *ctr = d.hs_ctr.as<unsigned long long>();
        for (int64_t t0 = 0; t0 < shots; t0 += tile) {
            const int64_t bt = std::min(tile, shots - t0);
            if ((rc = sample_on_device(h, d, bt, first + t0, seed, per_channel, d.hs_truth.as<uint32_t>(), d.hs_syn.as<uint32_t>(), st)))
                return rc;
            const bool want_ratio = osd && h->max_iters > 0;
            if (ots)
                rc = bpots_on_device(h, d, bt, d.hs_syn.as<uint32_t>(), d.hs_err.as<uint32_t>(), d.hs_conv.as<uint8_t>(), d.hs_iters.as<int32_t>(),
                                     *ots, ctr + LDPCB200_NUM_HARNESS_COUNTERS, st);
            else
                rc = decode_on_device(h, d, bt, d.hs_syn.as<uint32_t>(), d.hs_err.as<uint32_t>(), d.hs_conv.as<uint8_t>(), d.hs_iters.as<int32_t>(),
                                      want_ratio ? d.hs_ratio.as<double>() : nullptr, ctr + LDPCB200_NUM_HARNESS_COUNTERS, st, h->opt_osd_order == 0);
            if (rc) return rc;
            if (osd && (rc = osd_after_bp(h, d, d.set[0], bt, d.hs_syn.as<uint32_t>(), d.hs_err.as<uint32_t>(), d.hs_conv.as<uint8_t>(),
                                          d.hs_ratio.as<double>(), st)))
                return rc;
            bp::score_rows_logical<<<grid_for(bt * 32, d.sm_count), 256, 0, st>>>(
                d.d_colptr, d.d_ve_chk, h->NW, h->SW, bt, d.hs_truth.as<uint32_t>(), d.hs_err.as<uint32_t>(), d.hs_syn.as<uint32_t>(),
                d.scratch.as<uint32_t>(), h->lmask.empty() ? nullptr : d.lmask.as<unsigned long long>(), ctr + 3);
            h->launches++;
            CU(cudaGetLastError());
        }
        CU(cudaMemcpyAsync(ctr, ctr + LDPCB200_NUM_HARNESS_COUNTERS, 3 * 8, cudaMemcpyDeviceToDevice, st));   // decoded, converged, iterations
        if (osd) CU(cudaMemcpyAsync(ctr + 7, d.osd_stats.p, 8, cudaMemcpyDeviceToDevice, st));
    }
    unsigned long long hc[LDPCB200_NUM_HARNESS_COUNTERS];
    CU(cudaMemcpyAsync(hc, d.hs_ctr.p, sizeof(hc), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int k = 0; k < LDPCB200_NUM_HARNESS_COUNTERS; ++k) out8[k] = static_cast<int64_t>(hc[k]);
    return 0;
}

// The device of a call on device-resident buffers, and its stream: the caller's, or the device's own when that is null
int device_of(ldpcb200 *h, int32_t dev_slot, void *stream, DeviceCtx *&d, cudaStream_t &st)
{
    if (!h) return fail(LDPCB200_EINVAL, "null handle");
    if (dev_slot < 0 || dev_slot >= static_cast<int>(h->dev.size())) return fail(LDPCB200_EINVAL, "bad dev_slot");
    d = &h->dev[dev_slot];
    st = stream ? static_cast<cudaStream_t>(stream) : d->stream;
    return 0;
}

}  // namespace

// ================================================================================ C ABI
extern "C" {

const char *ldpcb200_last_error(void) { return g_err.c_str(); }

int ldpcb200_version(void) { return 100; }

int ldpcb200_device_count(int32_t *out)
{
    if (!out) return fail(LDPCB200_EINVAL, "out is null");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        *out = 0;
        return fail(LDPCB200_ENODEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *out = c;
    return 0;
}

int ldpcb200_create(int64_t s, int64_t n, const int64_t *colptr, const int64_t *rowval, int32_t index_base, double per,
                    int32_t max_iters, int32_t variant, const int32_t *devices, int32_t ndev, ldpcb200_t **out)
{
    if (!out) return fail(LDPCB200_EINVAL, "out is null");
    *out = nullptr;
    if (s < 0 || n < 0 || !colptr || (index_base != 0 && index_base != 1))
        return fail(LDPCB200_EINVAL, "bad shape / null colptr / index_base not 0 or 1");
    if (s > 0x3fffffff || n > 0x3fffffff) return fail(LDPCB200_EINVAL, "matrix too large");
    if (!rowval && colptr[n] - index_base != 0) return fail(LDPCB200_EINVAL, "rowval is null");
    if (variant != LDPCB200_VARIANT_EXACT && variant != LDPCB200_VARIANT_MINSUM && variant != LDPCB200_VARIANT_FAST32)
        return fail(LDPCB200_EUNSUPPORTED, "variant %d not available", variant);
    if (variant != LDPCB200_VARIANT_EXACT && !(per > 0.0 && per < 1.0))
        return fail(LDPCB200_EINVAL, "the log-likelihood-ratio variants need 0 < per < 1 (finite prior)");
    if (max_iters < 0) max_iters = 0;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(LDPCB200_ENODEVICE, "no CUDA device available (%s); libldpcb200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    ldpcb200 *h = new ldpcb200();
    h->s = s; h->n = n; h->max_iters = max_iters; h->variant = variant;
    set_prior(h, per);
    int rc = build_graph(h, colptr, rowval, index_base);
    if (rc) { delete h; return rc; }
    if (variant != LDPCB200_VARIANT_EXACT && h->big) {
        delete h;
        return fail(LDPCB200_EUNSUPPORTED, "the min-sum and fast variants support node degrees up to %d", bp::kMaxRegDegree);
    }
    std::vector<int> devs;
    if (devices && ndev > 0) devs.assign(devices, devices + ndev); else devs.push_back(0);
    for (int dv : devs) {
        if (dv < 0 || dv >= count) { delete h; return fail(LDPCB200_ENODEVICE, "device %d not present (%d devices)", dv, count); }
    }
    h->dev.resize(devs.size());
    for (size_t k = 0; k < devs.size(); ++k) {
        h->dev[k].device = devs[k];
        rc = init_device(h, h->dev[k]);
        if (rc) { ldpcb200_destroy(h); return rc; }
    }
    *out = h;
    return 0;
}

int ldpcb200_destroy(ldpcb200_t *h)
{
    if (!h) return 0;
    if (h->nccl_state == 1)
        for (ncclComm_t cm : h->comms)
            if (cm) g_nccl.CommDestroy(cm);
    for (DeviceCtx &d : h->dev) destroy_device(d);
    delete h;
    return 0;
}

int ldpcb200_set_option(ldpcb200_t *h, const char *key, int64_t value)
{
    if (!h || !key) return fail(LDPCB200_EINVAL, "null handle or key");
    const std::string k(key);
    if (k == "small_batch") { h->opt_small_batch = value; return 0; }
    if (k == "osd_order") {
        if (value < 0 || value > bp::kOsdMaxOrder) return fail(LDPCB200_EUNSUPPORTED, "osd_order must be between 0 and %d", bp::kOsdMaxOrder);
        h->opt_osd_order = static_cast<int>(value);
        return 0;
    }
    if (k == "stage_pageable") { h->opt_stage_pageable = value ? 1 : 0; return 0; }
    if (k == "nccl") { h->opt_nccl = value ? 1 : 0; return 0; }      // before the first multi-device batch
    if (k == "osd_profile") { h->opt_osd_profile = value ? 1 : 0; return 0; }
    if (k == "ratio_last_only") { h->opt_ratio_last_only = value ? 1 : 0; return 0; }
    if (k == "early_stop") { h->opt_early_stop = value ? 1 : 0; return 0; }   // run-time switch, no reconfiguration
    if (k == "chunk") { h->opt_chunk = value; return 0; }
    if (k == "minsum_scale_permille") {
        h->ms_scale = static_cast<double>(value) / 1000.0;
        for (DeviceCtx &d : h->dev) d.f_ready = false;
        return 0;
    }
    if (k == "family") h->opt_family = static_cast<int>(value);
    else if (k == "warps") h->opt_warps = static_cast<int>(value);
    else if (k == "dynamic_queue") { h->opt_dynamic_queue = value ? 1 : 0; return 0; }
    else if (k == "direct_bits") { h->opt_direct_bits = value ? 1 : 0; return 0; }
    else if (k == "overlap_chunks") { h->opt_overlap_chunks = value == 2 ? 2 : (value ? 1 : 0); return 0; }
    else if (k == "grid_kernel") { h->opt_grid_kernel = value == 2 ? 2 : (value ? 1 : 0); return 0; }
    else if (k == "prefetch") h->opt_pd = static_cast<int>(value);
    else if (k == "ring_mult") h->opt_ring_mult = static_cast<int>(std::min<int64_t>(std::max<int64_t>(value, 0), 4));
    else if (k == "lean") h->opt_lean = value ? 1 : 0;
    else if (k == "bpots_memory") {
        if (value < 0 || value > 2) return fail(LDPCB200_EINVAL, "bpots_memory must be 0 (auto), 1 (shared) or 2 (global)");
        h->opt_bpots_memory = static_cast<int>(value);
        return 0;
    }
    else if (k == "first_iteration_filter") { h->opt_filter = value ? 1 : 0; return 0; }
    else if (k == "dual") h->opt_dual = value ? 1 : 0;
    else if (k == "contiguous_variables") h->opt_cv = value ? 1 : 0;
    else if (k == "kernel_profile") { h->opt_kernel_profile = value ? 1 : 0; return 0; }
    else if (k == "time_kernels") { h->opt_time_kernels = value ? 1 : 0; return 0; }
    else if (k == "max_ctas_per_sm") h->opt_max_ctas = static_cast<int>(value);
    else if (k == "slots") h->opt_slots = static_cast<int>(value);   // accepted for compatibility, unused
    else return fail(LDPCB200_EINVAL, "unknown option '%s'", key);
    h->configured = false;
    return 0;
}

int ldpcb200_info(const ldpcb200_t *hc, ldpcb200_info_t *out)
{
    if (!hc || !out) return fail(LDPCB200_EINVAL, "null argument");
    ldpcb200 *h = const_cast<ldpcb200 *>(hc);
    int rc = configure(h);
    if (rc) return rc;
    memset(out, 0, sizeof(*out));
    out->s = h->s; out->n = h->n; out->E = h->E;
    out->max_check_degree = h->max_cdeg; out->max_var_degree = h->max_vdeg;
    out->family = h->family; out->ndev = static_cast<int>(h->dev.size());
    out->sm_count = h->dev[0].sm_count;
    out->ctas_per_sm = h->ctas_per_sm; out->threads_per_cta = h->warps * 32 * (h->dual ? 2 : 1);
    out->smem_bytes = h->smem_bytes; out->slots = h->slots;
    out->syn_words = h->SW; out->err_words = h->NW;
    out->message_bytes = h->family == LDPCB200_FAMILY_SMEM
                             ? 0
                             : static_cast<int64_t>(h->slots) * std::max<int64_t>(h->E, 1) * 8;
    out->kernel_mode = h->mode;
    out->prefetch_distance = h->kp_proto.pd;
    out->kernel_rev = h->lean ? (h->dual ? 3 : 2) : 1;
    nccl_prepare(h);
    out->counters_via_nccl = h->nccl_state == 1 ? 1 : 0;
    out->bpots_workspace_bytes = static_cast<int64_t>(h->dev[0].bpots_ws.cap);
    return 0;
}

int ldpcb200_decode_device(ldpcb200_t *h, int32_t dev_slot, int64_t B, const uint32_t *d_syn_words, uint32_t *d_err_words,
                           uint8_t *d_converged, int32_t *d_iters, double *d_posterior_ratio,
                           unsigned long long *d_counters, void *stream)
{
    DeviceCtx *d;
    cudaStream_t st;
    int rc = device_of(h, dev_slot, stream, d, st);
    if (rc) return rc;
    if (B < 0 || (B > 0 && (!d_syn_words || !d_err_words || !d_converged))) return fail(LDPCB200_EINVAL, "null device buffer");
    if ((rc = configure(h))) return rc;
    return decode_on_device(h, *d, B, d_syn_words, d_err_words, d_converged, d_iters, d_posterior_ratio, d_counters, st,
                            h->opt_ratio_last_only != 0);
}

static int decode_batch_impl(ldpcb200_t *h, int64_t B, const void *syndromes, int32_t syn_fmt, int64_t syn_ld, void *errors,
                             int32_t err_fmt, int64_t err_ld, uint8_t *converged, int32_t *iters, double *posterior_ratio,
                             int64_t *counters, bool osd, int64_t *osd_stats, const BpotsArgs *ots = nullptr)
{
    if (!h) return fail(LDPCB200_EINVAL, "null handle");
    if (osd_stats) memset(osd_stats, 0, sizeof(int64_t) * LDPCB200_NUM_OSD_STATS);
    if (osd && h->variant != LDPCB200_VARIANT_EXACT)
        return fail(LDPCB200_EUNSUPPORTED, "OSD-0 is defined on the posterior ratios of the exact variant");
    if (B < 0) return fail(LDPCB200_EINVAL, "negative batch");
    if (counters) memset(counters, 0, sizeof(int64_t) * LDPCB200_NUM_COUNTERS);
    if (B == 0) return 0;
    if (!syndromes || !errors || !converged) return fail(LDPCB200_EINVAL, "null host buffer");
    if (syn_fmt == LDPCB200_FMT_F64) return fail(LDPCB200_EINVAL, "FMT_F64 is an output-only format");
    if (syn_fmt < LDPCB200_FMT_U8 || syn_fmt > LDPCB200_FMT_PACKED32) return fail(LDPCB200_EINVAL, "unsupported syndrome format %d", syn_fmt);
    if (err_fmt < LDPCB200_FMT_U8 || err_fmt > LDPCB200_FMT_F64) return fail(LDPCB200_EINVAL, "unsupported error format %d", err_fmt);
    if ((syn_fmt == LDPCB200_FMT_U8 || syn_fmt == LDPCB200_FMT_I64) && syn_ld < h->s) return fail(LDPCB200_EINVAL, "syn_ld < s");
    if ((err_fmt == LDPCB200_FMT_U8 || err_fmt == LDPCB200_FMT_I64 || err_fmt == LDPCB200_FMT_F64) && err_ld < h->n)
        return fail(LDPCB200_EINVAL, "err_ld < n");
    int rc = configure(h);
    if (rc) return rc;
    const int nd = static_cast<int>(h->dev.size());
    std::vector<int64_t> ctr(static_cast<size_t>(nd) * LDPCB200_NUM_COUNTERS, 0);
    std::vector<int64_t> ost(static_cast<size_t>(nd) * LDPCB200_NUM_OSD_STATS, 0);
    rc = fan_out(h, B, [&](int k, int64_t b0, int64_t Bd) {
        return Bd <= 0 ? 0 : decode_host_range(h, h->dev[k], b0, Bd, B, syndromes, syn_fmt, syn_ld, errors, err_fmt, err_ld, converged,
                                               iters, posterior_ratio, &ctr[static_cast<size_t>(k) * LDPCB200_NUM_COUNTERS], osd,
                                               &ost[static_cast<size_t>(k) * LDPCB200_NUM_OSD_STATS], ots);
    });
    if (rc) return rc;
    if (counters) {
        if (nd > 1) nccl_prepare(h);
        // NCCL only when every device decoded a share -- fan_out gives each one 32 columns or more when there are at least
        // nd blocks of 32 -- so that its counter block holds this call's values; a smaller batch is summed on the host
        if (h->nccl_state == 1 && (B + 31) / 32 >= nd) {
            if ((rc = nccl_sum_block(h, LDPCB200_NUM_COUNTERS, [](DeviceCtx &d) { return d.counters.p; }, counters))) return rc;
        } else {
            host_sum(ctr, LDPCB200_NUM_COUNTERS, counters);
        }
    }
    if (osd_stats) host_sum(ost, LDPCB200_NUM_OSD_STATS, osd_stats);
    return 0;
}

int ldpcb200_decode_batch(ldpcb200_t *h, int64_t B, const void *syndromes, int32_t syn_fmt, int64_t syn_ld, void *errors,
                          int32_t err_fmt, int64_t err_ld, uint8_t *converged, int32_t *iters, double *posterior_ratio,
                          int64_t *counters)
{
    return decode_batch_impl(h, B, syndromes, syn_fmt, syn_ld, errors, err_fmt, err_ld, converged, iters, posterior_ratio,
                             counters, false, nullptr);
}

int ldpcb200_bposd_decode_batch(ldpcb200_t *h, int64_t B, const void *syndromes, int32_t syn_fmt, int64_t syn_ld, void *errors,
                                int32_t err_fmt, int64_t err_ld, uint8_t *converged, int32_t *iters, int64_t *counters,
                                int64_t *osd_stats)
{
    return decode_batch_impl(h, B, syndromes, syn_fmt, syn_ld, errors, err_fmt, err_ld, converged, iters, nullptr, counters,
                             true, osd_stats);
}

int ldpcb200_bpots_decode_batch(ldpcb200_t *h, int64_t B, const void *syndromes, int32_t syn_fmt, int64_t syn_ld, void *errors,
                                int32_t err_fmt, int64_t err_ld, uint8_t *converged, int32_t *iters, int32_t T, double C)
{
    const BpotsArgs a{T, C};
    return decode_batch_impl(h, B, syndromes, syn_fmt, syn_ld, errors, err_fmt, err_ld, converged, iters, nullptr, nullptr, false, nullptr, &a);
}

int ldpcb200_bpots_device(ldpcb200_t *h, int32_t dev_slot, int64_t B, const uint32_t *d_syn_words, uint32_t *d_err_words,
                          uint8_t *d_converged, int32_t *d_iters, unsigned long long *d_counters, int32_t T, double C, void *stream)
{
    DeviceCtx *d;
    cudaStream_t st;
    int rc = device_of(h, dev_slot, stream, d, st);
    if (rc) return rc;
    if (B < 0 || (B > 0 && (!d_syn_words || !d_err_words || !d_converged))) return fail(LDPCB200_EINVAL, "null device buffer");
    const BpotsArgs a{T, C};
    return bpots_on_device(h, *d, B, d_syn_words, d_err_words, d_converged, d_iters, a, d_counters, st);
}

int ldpcb200_osd0_device(ldpcb200_t *h, int32_t dev_slot, int64_t B, const uint32_t *d_syn_words, uint32_t *d_err_words,
                         const uint8_t *d_converged, const double *d_posterior_ratio, unsigned long long *d_stats, void *stream)
{
    DeviceCtx *d;
    cudaStream_t st;
    int rc = device_of(h, dev_slot, stream, d, st);
    if (rc) return rc;
    if (B < 0 || (B > 0 && (!d_syn_words || !d_err_words || !d_converged || !d_posterior_ratio)))
        return fail(LDPCB200_EINVAL, "null device buffer");
    return osd_on_device(h, *d, d->set[0], B, 0, d_syn_words, d_err_words, d_converged, d_posterior_ratio, d_stats, st);
}

int ldpcb200_sample_device(ldpcb200_t *h, int32_t dev_slot, int64_t B, int64_t first, uint64_t seed, double per,
                           uint32_t *d_true_err_words, uint32_t *d_syn_words, void *stream)
{
    DeviceCtx *d;
    cudaStream_t st;
    int rc = device_of(h, dev_slot, stream, d, st);
    if (rc) return rc;
    if (B <= 0) return 0;
    if (!d_true_err_words || !d_syn_words) return fail(LDPCB200_EINVAL, "null device buffer");
    CU(cudaSetDevice(d->device));
    if ((rc = sample_on_device(h, *d, B, first, seed, per, d_true_err_words, d_syn_words, st))) return rc;
    CU(cudaGetLastError());
    return 0;
}

int ldpcb200_score_device(ldpcb200_t *h, int32_t dev_slot, int64_t B, const uint32_t *d_true_err_words,
                          const uint32_t *d_err_words, const uint32_t *d_syn_words, unsigned long long *d_out, void *stream)
{
    DeviceCtx *d;
    cudaStream_t st;
    int rc = device_of(h, dev_slot, stream, d, st);
    if (rc) return rc;
    if (B <= 0) return 0;
    if (!d_true_err_words || !d_err_words || !d_syn_words || !d_out) return fail(LDPCB200_EINVAL, "null device buffer");
    CU(cudaSetDevice(d->device));
    if ((rc = d->scratch.reserve(static_cast<size_t>(B) * h->SW * 4))) return rc;
    bp::score_rows<<<grid_for(B * 32, d->sm_count), 256, 0, st>>>(d->d_rowptr, d->d_colptr, d->d_ve_chk, h->NW, h->SW, B,
                                                                 d_true_err_words, d_err_words, d_syn_words,
                                                                 d->scratch.as<uint32_t>(), d_out);
    h->launches++;
    CU(cudaGetLastError());
    return 0;
}

int ldpcb200_set_logicals(ldpcb200_t *h, int64_t k, const int64_t *colptr, const int64_t *rowval, int32_t index_base)
{
    if (!h) return fail(LDPCB200_EINVAL, "null handle");
    if (k < 0 || k > 64) return fail(LDPCB200_EUNSUPPORTED, "between 0 and 64 logical operators are supported (got %lld)", (long long)k);
    if (k > 0 && (!colptr || (index_base != 0 && index_base != 1))) return fail(LDPCB200_EINVAL, "null colptr / bad index_base");
    std::vector<unsigned long long> m;
    if (k > 0) {
        m.assign(std::max<int64_t>(h->n, 1), 0ull);
        for (int64_t j = 0; j < h->n; ++j)
            for (int64_t e = colptr[j] - index_base; e < colptr[j + 1] - index_base; ++e) {
                const int64_t r = rowval[e] - index_base;
                if (r < 0 || r >= k) return fail(LDPCB200_EINVAL, "logical operator index out of range at entry %lld", (long long)e);
                m[j] ^= 1ull << r;
            }
    }
    h->lmask.swap(m);
    h->n_logicals = static_cast<int>(k);
    for (DeviceCtx &d : h->dev) {
        CU(cudaSetDevice(d.device));
        CU(cudaStreamSynchronize(d.set[0].stream));
        d.lmask.release();
        if (!h->lmask.empty()) {
            int rc = d.lmask.reserve(h->lmask.size() * 8);
            if (rc) return rc;
            CU(cudaMemcpy(d.lmask.p, h->lmask.data(), h->lmask.size() * 8, cudaMemcpyHostToDevice));
        }
    }
    return 0;
}

int ldpcb200_score_logical_device(ldpcb200_t *h, int32_t dev_slot, int64_t B, const uint32_t *d_true_err_words,
                                  const uint32_t *d_err_words, const uint32_t *d_syn_words, unsigned long long *d_out, void *stream)
{
    DeviceCtx *d;
    cudaStream_t st;
    int rc = device_of(h, dev_slot, stream, d, st);
    if (rc) return rc;
    if (B <= 0) return 0;
    if (!d_true_err_words || !d_err_words || !d_syn_words || !d_out) return fail(LDPCB200_EINVAL, "null device buffer");
    CU(cudaSetDevice(d->device));
    if ((rc = d->scratch.reserve(static_cast<size_t>(B) * h->SW * 4))) return rc;
    bp::score_rows_logical<<<grid_for(B * 32, d->sm_count), 256, 0, st>>>(d->d_colptr, d->d_ve_chk, h->NW, h->SW, B, d_true_err_words, d_err_words,
                                                                         d_syn_words, d->scratch.as<uint32_t>(),
                                                                         h->lmask.empty() ? nullptr : d->lmask.as<unsigned long long>(), d_out);
    h->launches++;
    CU(cudaGetLastError());
    return 0;
}

int ldpcb200_set_per(ldpcb200_t *h, double per)
{
    if (!h) return fail(LDPCB200_EINVAL, "null handle");
    if (h->variant != LDPCB200_VARIANT_EXACT && !(per > 0.0 && per < 1.0))
        return fail(LDPCB200_EINVAL, "the log-likelihood-ratio variants need 0 < per < 1 (finite prior)");
    set_prior(h, per);
    return 0;
}

static int sample_score_impl(ldpcb200_t *h, int64_t shots, int64_t first, uint64_t seed, double per_channel, int32_t osd,
                             const BpotsArgs *ots, int64_t *out)
{
    if (!h || !out) return fail(LDPCB200_EINVAL, "null argument");
    memset(out, 0, sizeof(int64_t) * LDPCB200_NUM_HARNESS_COUNTERS);
    if (shots < 0) return fail(LDPCB200_EINVAL, "negative shot count");
    if (osd && h->variant != LDPCB200_VARIANT_EXACT) return fail(LDPCB200_EUNSUPPORTED, "OSD-0 is defined on the posterior ratios of the exact variant");
    if (shots == 0) return 0;
    int rc = configure(h);
    if (rc) return rc;
    const int nd = static_cast<int>(h->dev.size());
    std::vector<int64_t> ctr(static_cast<size_t>(nd) * LDPCB200_NUM_HARNESS_COUNTERS, 0);
    // every device runs, even with no shots: that zeroes its counter block for the sum below
    rc = fan_out(h, shots, [&](int k, int64_t s0, int64_t count) {
        return harness_on_device(h, h->dev[k], first + s0, count, seed, per_channel, osd != 0, ots,
                                 &ctr[static_cast<size_t>(k) * LDPCB200_NUM_HARNESS_COUNTERS]);
    });
    if (rc) return rc;
    if (nd > 1) nccl_prepare(h);
    if (h->nccl_state == 1)                                // one grouped ncclAllReduce of the 8 counters (K7 of SURVEY section 2)
        return nccl_sum_block(h, LDPCB200_NUM_HARNESS_COUNTERS, [](DeviceCtx &d) { return d.hs_ctr.p; }, out);
    host_sum(ctr, LDPCB200_NUM_HARNESS_COUNTERS, out);
    return 0;
}

int ldpcb200_sample_decode_score(ldpcb200_t *h, int64_t shots, int64_t first, uint64_t seed, double per_channel, int32_t osd,
                                 int64_t *out)
{
    return sample_score_impl(h, shots, first, seed, per_channel, osd, nullptr, out);
}

int ldpcb200_sample_bpots_score(ldpcb200_t *h, int64_t shots, int64_t first, uint64_t seed, double per_channel, int32_t T, double C,
                                int64_t *out)
{
    const BpotsArgs a{T, C};
    return sample_score_impl(h, shots, first, seed, per_channel, 0, &a, out);
}

int ldpcb200_selftest_division(int32_t device, int32_t mode, uint64_t n, uint64_t seed, uint64_t *mismatches)
{
    if (!mismatches || (mode != 0 && mode != 1)) return fail(LDPCB200_EINVAL, "bad selftest arguments");
    CU(cudaSetDevice(device));
    unsigned long long *d = nullptr;
    CU(cudaMalloc(&d, 32));
    CU(cudaMemset(d, 0, 32));
    bp::selftest_division<<<148 * 8, 256>>>(mode, n, seed, d);
    unsigned long long hcount[4] = {0, 0, 0, 0};
    cudaError_t e = cudaMemcpy(hcount, d, 32, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(LDPCB200_ECUDA, "selftest: %s", cudaGetErrorString(e));
    for (int k = 0; k < 4; ++k) mismatches[k] = hcount[k];
    return 0;
}

int ldpcb200_kernel_profile(ldpcb200_t *h, int32_t dev_slot, int64_t *out8, int32_t reset)
{
    DeviceCtx *d;
    cudaStream_t st;
    int rc = device_of(h, dev_slot, nullptr, d, st);
    if (rc) return rc;
    if (!out8) return fail(LDPCB200_EINVAL, "out8 is null");
    CU(cudaSetDevice(d->device));
    CU(cudaDeviceSynchronize());
    unsigned long long v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (d->kprof.p) {
        CU(cudaMemcpy(v, d->kprof.p, 64, cudaMemcpyDeviceToHost));
        if (reset) CU(cudaMemset(d->kprof.p, 0, 64));
    }
    for (int k = 0; k < 8; ++k) out8[k] = static_cast<int64_t>(v[k]);
    return 0;
}

int ldpcb200_kernel_time(ldpcb200_t *h, int32_t dev_slot, double *ms, int64_t *launches, int32_t reset)
{
    DeviceCtx *d;
    cudaStream_t st;
    int rc = device_of(h, dev_slot, nullptr, d, st);
    if (rc) return rc;
    if (!ms || !launches) return fail(LDPCB200_EINVAL, "null argument");
    CU(cudaSetDevice(d->device));
    CU(cudaDeviceSynchronize());
    for (auto &pr : d->ktime_events) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, pr.first, pr.second) == cudaSuccess) { d->ktime_ms += t; d->ktime_launches++; }
        else cudaGetLastError();
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    d->ktime_events.clear();
    *ms = d->ktime_ms;
    *launches = d->ktime_launches;
    if (reset) { d->ktime_ms = 0.0; d->ktime_launches = 0; }
    return 0;
}

int ldpcb200_launch_count(const ldpcb200_t *h, int64_t *out)
{
    if (!h || !out) return fail(LDPCB200_EINVAL, "null argument");
    *out = h->launches.load();
    return 0;
}

}  // extern "C"
