"""OSD-0 and order-O OSD (csrc/osd.cuh) across their envelope, bit for bit against the CPU oracle.

The named codes reach the OSD kernels only with m <= 900 checks, at ordinary error rates, and with BP's own consistent
outputs.  The graphs here are built from chosen degree sequences so that each row-ownership instantiation of osd0_kernel
runs (rows per thread RPT = ceil(m / 256) in {1, 2, 3, 8}, the last one up to 2048 checks and about 218 KB of shared
memory), the padded sort length and the 128-bit row groups sit on both sides of a boundary, equal columns leave the pivot
choice to the sort alone, and order-O OSD runs beyond OSD-0's row limit.  OSD-0 is also fed crafted inputs directly:
posterior ratios whose sort keys are +inf (R = 0 or subnormal), exactly 1 (R = 1, inf, DBL_MAX), 0.5 (R = 2), ulp
neighbours and heavy ties, and converged flags whose decisions do not satisfy the syndrome (those rows must come back
untouched).  Order-O OSD runs orders 1 to 12, the clamp to n - rank and the tie rule of the trial search (smallest x
among the lightest).  Every GPU case must equal the oracle in decisions, converged flags and pivot counts."""
import functools

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import bp_dense
from test_kernel_paths import PRIORS, configuration_model, degrees, designed as designed_bp

OSD_THREADS = 256           # kOsdThreads
OSD_MAX_ROWS = 8 * 256      # kOsdMaxRowsPerThread * kOsdThreads: OSD-0's row limit
B200_SMEM_OPTIN = 232448    # shared memory per block (opt-in) of a B200
MAX_ITERS = 12

DBL_MAX = float(np.finfo(np.float64).max)


# ---------------------------------------------------------------------------------------------------------------------
# designed graphs
OSPECS = {
    # RPT 2; degree-0 variables and empty checks
    "O1": ({0: 4, 1: 10, 2: 30, 3: 126, 4: 80, 5: 40, 6: 10}, {0: 8, 2: 188, 3: 164, 4: 40}, 201),
    # RPT 2 / 3 boundary; n = 2^9 + 1 and 2^9 (sort length NP 1024 and 512)
    "O2a": ({2: 140, 3: 229, 4: 143}, {3: 513}, 202),
    "O2b": ({2: 144, 3: 228, 4: 141}, {3: 512}, 203),
    # RPT 8 at its lower end, m > n
    "O3": ({2: 519, 3: 506}, {4: 639}, 204),
    # RPT 8 at the row limit: 2048 x 639 needs 218,024 B of shared memory
    "O4": ({2: 1671, 3: 377}, {7: 639}, 205),
    # n + 1 = 128 bits (one 16-byte group per row) and 129 bits (two, rounded up to three)
    "O5a": ({2: 257}, {4: 121, 5: 6}, 206),
    "O5b": ({2: 257}, {4: 126, 5: 2}, 207),
    # order-O OSD beyond OSD-0's row limit
    "O6": ({1: 2400, 2: 600}, {12: 300}, 208),
}
O7_BASE = ({2: 56, 3: 144}, {2: 80, 3: 128}, 209)       # 200 x 208, then 12 duplicated columns appended
# sample rate of the syndrome set: where BP leaves many unconverged (the m > n graphs converge on every sampled syndrome,
# there the uniformly random columns, mostly outside the column space, are the unconverged ones)
SAMPLE_RATE = {"O1": 0.15, "O2a": 0.25, "O2b": 0.25, "O3": 0.3, "O4": 0.3, "O5a": 0.3, "O5b": 0.3, "O6": 0.3, "O7": 0.25,
               "G1": 0.1, "G3": 0.06, "C2": 0.08, "C3": 0.08}


@functools.lru_cache(maxsize=None)
def ograph(name):
    if name == "O7":
        H = configuration_model(*O7_BASE).tolil()
        cols = np.random.default_rng(210).choice(H.shape[1], 12, replace=False)
        return sp.csc_matrix(sp.hstack([H, H[:, cols]]))
    if name in OSPECS:
        return configuration_model(*OSPECS[name])
    return designed_bp(name)


def graph(codes, name):
    """(H, max_iters) of a designed graph or a named code."""
    if name in ("C2", "C3"):
        H, _, mi = codes.config_matrix(name)
        return sp.csc_matrix(H), mi
    return ograph(name), MAX_ITERS


def gf2_rank(H):
    M = np.asarray(sp.csc_matrix(H).todense()).astype(bool)
    r = 0
    for c in range(M.shape[1]):
        nz = np.nonzero(M[r:, c])[0]
        if nz.size == 0:
            continue
        M[[r, r + nz[0]]] = M[[r + nz[0], r]]
        rows = np.nonzero(M[:, c])[0]
        M[rows[rows != r]] ^= M[r]
        r += 1
        if r == M.shape[0]:
            break
    return r


def osd_layout(m, n):
    """Shared-memory bytes of one OSD CTA: osd_layout() of ldpcb200.cu restated."""
    g = (n + 1 + 127) // 128
    if g % 2 == 0:
        g += 1
    nwr = 4 * g
    np_ = 2
    while np_ < n:
        np_ <<= 1
    off = (m * nwr * 4 + 15) // 16 * 16
    off += np_ * 8 + np_ * 4
    off += max(m, 1) * 4 * 5 + nwr * 4
    off += (16 + 192 + nwr // 4 + 1) * 4
    return off


def straddle(budget, m=OSD_MAX_ROWS):
    """(largest n whose m x n layout fits the budget, smallest n that does not)."""
    n = 1
    while osd_layout(m, n + 1) <= budget:
        n += 1
    return n, n + 1


_SYN = {}


def syndromes_of(oracle, name, H, sampled=96, rnd=64):
    """Columns: `sampled` errors at SAMPLE_RATE[name], then `rnd` uniformly random syndromes."""
    key = (name, sampled, rnd)
    if key not in _SYN:
        _, a = oracle.sample(H, SAMPLE_RATE[name], 17, 0, sampled)
        r = (np.random.default_rng(18).random((H.shape[0], rnd)) < 0.5).astype(np.uint8)
        _SYN[key] = np.asfortranarray(np.column_stack([a, r]).astype(np.uint8))
    return _SYN[key]


# ---------------------------------------------------------------------------------------------------------------------
# crafted OSD-0 inputs
RATIO_CLASSES = ("ones", "specials", "ulp", "pool", "loguniform")


def crafted_inputs(H, syn, seed):
    """(bp_err, ratio, conv) for every column of syn: ratio class = column % 5, bp_err all-zero / all-one / random by
    (column // 5) % 3, about a quarter of the columns flagged converged (whatever their bp_err)."""
    m, n = H.shape
    B = syn.shape[1]
    rng = np.random.default_rng(seed)
    ratio = np.empty((n, B), dtype=np.float64, order="F")
    specials = np.array([0.0, 5e-324, 1e-310, 1.0, 2.0, DBL_MAX, np.inf])
    ulps = np.array([np.nextafter(2.0, 0.0), 2.0, np.nextafter(2.0, 3.0), np.nextafter(1.0, 0.0), 1.0, np.nextafter(1.0, 2.0)])
    pool = 10.0 ** rng.uniform(-6, 6, 5)
    for b in range(B):
        cls = RATIO_CLASSES[b % 5]
        if cls == "ones":
            ratio[:, b] = 1.0
        elif cls == "specials":
            ratio[:, b] = rng.choice(specials, n)
        elif cls == "ulp":
            ratio[:, b] = rng.choice(ulps, n)
        elif cls == "pool":
            ratio[:, b] = rng.choice(pool, n)
        else:
            ratio[:, b] = 10.0 ** rng.uniform(-12, 12, n)
    mode = (np.arange(B) // 5) % 3
    bp_err = np.where(mode[None, :] == 0, 0, np.where(mode[None, :] == 1, 1, rng.random((n, B)) < 0.3)).astype(np.uint8)
    bp_err = np.asfortranarray(bp_err)
    conv = rng.random(B) < 0.25
    return bp_err, ratio, conv


# ---------------------------------------------------------------------------------------------------------------------
# CPU: profiles of the designed graphs
def test_osd_graph_profiles(oracle):
    """Each designed graph has the shape, row-ownership instantiation, rank and degenerate nodes it is meant to hit; the
    syndrome sets leave a third or more unconverged at the sample rate."""
    rpt = lambda m: -(-m // OSD_THREADS)
    expect = {"O1": (300, 400, 2), "O2a": (512, 513, 2), "O2b": (513, 512, 3), "O3": (1025, 639, 8), "O4": (2048, 639, 8),
              "O5a": (257, 127, 2), "O5b": (257, 128, 2), "O6": (3000, 300, None), "O7": (200, 220, 1)}
    for name, (m, n, r) in expect.items():
        H = ograph(name)
        assert H.shape == (m, n), name
        if r is not None:
            assert rpt(m) == r or (r == 8 and 4 < rpt(m) <= 8), name
        assert H.max() == 1 and (H.data == 1).all(), name
    cd, vd = degrees(ograph("O1"))
    assert (cd == 0).sum() == 4 and (vd == 0).sum() == 8
    assert gf2_rank(ograph("O1")) == 296
    assert gf2_rank(ograph("O2a")) == 512 and gf2_rank(ograph("O2b")) == 511
    # m > n: rank n, so a uniformly random syndrome is almost never in the column space
    for name in ("O3", "O4", "O5a", "O5b", "O6"):
        m, n = ograph(name).shape
        assert gf2_rank(ograph(name)) >= n - 1 and m > n, name
    # sort lengths: n = 512 pads to 512, n = 513 to 1024; row groups: n + 1 = 128 bits is one, 129 bits three
    for name, npad in (("O2a", 1024), ("O2b", 512)):
        n = ograph(name).shape[1]
        assert 1 << (n - 1).bit_length() == npad
    assert osd_layout(257, 127) < osd_layout(257, 128)
    assert (127 + 1 + 127) // 128 == 1 and (128 + 1 + 127) // 128 == 2
    # the shared-memory limit at 2048 checks on a B200: 639 columns fit (218,024 B), 640 do not (283,600 B)
    assert osd_layout(2048, 639) == 218024 and osd_layout(2048, 640) == 283600
    assert straddle(B200_SMEM_OPTIN) == (639, 640)
    # O7: 12 columns equal to an earlier one
    H7 = ograph("O7").toarray()
    assert sum(any((H7[:, j] == H7[:, k]).all() for k in range(j)) for j in range(H7.shape[1])) == 12
    for name in ("O1", "O2a", "O2b", "O3", "O4", "O5a", "O5b", "O7"):
        H = ograph(name)
        syn = syndromes_of(oracle, name, H)
        r = oracle.batch_decode(H, SAMPLE_RATE[name], MAX_ITERS, syn, nthreads=oracle.num_threads())
        assert (~r["converged"]).mean() >= 1 / 3, name


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the oracle's OSD-0 on given inputs
@pytest.mark.parametrize("name", ["C2", "C3"])
def test_osd0_given_reproduces_bposd(oracle, codes, name):
    """BP's own outputs fed to osd0_given give what bposd_decode gives, bit for bit, pivots included."""
    H, mi = graph(codes, name)
    _, syn = oracle.sample(H, 0.08, 55, 0, 300)
    bp = oracle.batch_decode(H, 0.08, mi, syn, nthreads=oracle.num_threads(), want_ratio=True)
    ref = oracle.bposd_decode(H, 0.08, mi, syn, nthreads=oracle.num_threads())
    got = oracle.osd0_given(H, syn, bp["errors"], bp["ratio"], nthreads=oracle.num_threads())
    assert (~bp["converged"]).sum() > 30
    assert np.array_equal(got["errors"], ref["errors"]) and np.array_equal(got["pivots"], ref["pivots"])


def small_designed(seed):
    """Small shapes (n <= 64) for the dense transliteration: square, tall, wide, with duplicated and empty columns."""
    rng = np.random.default_rng(seed)
    out = []
    for m, n in ((12, 16), (24, 20), (31, 64), (40, 33)):
        H = (rng.random((m, n)) < 0.15).astype(np.uint8)
        H[:, 1] = H[:, 0]                              # equal columns
        H[:, 5] = 0                                    # an empty column
        out.append(H)
    return out


def test_osd0_given_equals_dense_transliteration_on_crafted_keys(oracle):
    """osd0_given against bp_dense.osd0_dense at every crafted ratio class (keys +inf, exactly 1 and 0.5, ulp neighbours,
    ties): pins the oracle itself where the GPU is compared with it.  (NaN ratios are excluded: BP never produces them
    and the comparison sort has no total order on NaN.)"""
    for k, H in enumerate(small_designed(5)):
        m, n = H.shape
        syn = np.asfortranarray(np.column_stack([(H @ (np.random.default_rng(k).random((n, 20)) < 0.2)) % 2,
                                                 np.random.default_rng(k + 9).random((m, 20)) < 0.5]).astype(np.uint8))
        bp_err, ratio, _ = crafted_inputs(H, syn, 100 + k)
        assert not np.isnan(ratio).any()
        got = oracle.osd0_given(H, syn, bp_err, ratio)
        for b in range(syn.shape[1]):
            want, npiv = bp_dense.osd0_dense(H, syn[:, b], bp_err[:, b], ratio[:, b], return_pivots=True)
            assert np.array_equal(got["errors"][:, b], want), (k, b, RATIO_CLASSES[b % 5])
            assert got["pivots"][b] == npiv, (k, b)


GOLDEN_OSD_KEY_DIFFS = {"gallager1000_p03": 0, "gross_p05": 0, "hgp_p05": 0, "surface15_p03": 1}


@pytest.mark.parametrize("fixture", sorted(GOLDEN_OSD_KEY_DIFFS))
def test_osd_key_deviation_count_on_golden_fixtures(oracle, fixture):
    """The stated deviation of the OSD sort key (RN(1/R) instead of the reference's exp(log(1/R))), counted: columns of
    the golden fixtures whose OSD-0 output changes with the key."""
    import os
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", fixture + ".npz"))
    zo = np.load(os.path.join(os.path.dirname(__file__), "golden", fixture + ".osd.npz"))
    H = sp.csc_matrix((np.ones(len(z["rowval"]), dtype=np.uint8), z["rowval"], z["colptr"]), shape=tuple(z["shape"]))
    a = oracle.bposd_decode(H, float(z["per"]), int(zo["max_iters"]), z["syndromes"], nthreads=oracle.num_threads(), key_mode=0)
    b = oracle.bposd_decode(H, float(z["per"]), int(zo["max_iters"]), z["syndromes"], nthreads=oracle.num_threads(), key_mode=1)
    differ = int((a["errors"] != b["errors"]).any(axis=0).sum())
    assert differ == GOLDEN_OSD_KEY_DIFFS[fixture], (
        "%s: %d columns change with the key (expected %d); key mode 1 uses this C library's exp and log, so a different "
        "libm can move this count" % (fixture, differ, GOLDEN_OSD_KEY_DIFFS[fixture]))


# ---------------------------------------------------------------------------------------------------------------------
# GPU runners
def pack_rows(bits, words):
    """(rows, B) 0/1 -> [B][words] int32 rows, bit j of a row at word j // 32, bit j % 32 (the library's packed rows)."""
    rows, B = bits.shape
    pad = np.zeros((B, words * 32), dtype=np.uint8)
    pad[:, :rows] = bits.T
    return np.packbits(pad, axis=1, bitorder="little").view(np.int32).copy()


def unpack_rows(words, rows):
    return np.asfortranarray(np.unpackbits(words.view(np.uint8), axis=1, bitorder="little")[:, :rows].T)


def osd0_on_device(pkg, H, syn, bp_err, ratio, conv):
    """ldpcb200_osd0_device on crafted inputs, bracketed by device synchronisations (the library's stream does not order
    itself after torch's).  Returns (errors (n,B), stats[0..2])."""
    import torch
    dec = pkg.BeliefPropagationDecoder(H, 0.05, MAX_ITERS)
    info = dec.info()
    n, B = H.shape[1], syn.shape[1]
    dev = torch.device("cuda:0")
    synw = torch.from_numpy(pack_rows(syn, info["syn_words"])).to(dev)
    errw = torch.from_numpy(pack_rows(bp_err, info["err_words"])).to(dev)
    cv = torch.from_numpy(conv.astype(np.uint8)).to(dev)
    rt = torch.from_numpy(np.ascontiguousarray(ratio.T)).to(dev)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    dec.osd0_device(B, synw.data_ptr(), errw.data_ptr(), cv.data_ptr(), rt.data_ptr(), stats.data_ptr())
    torch.cuda.synchronize()
    out = unpack_rows(errw.cpu().numpy(), n), stats.cpu().numpy()[:3]
    dec.close()
    return out


def bposd_host(pkg, H, per, mi, syn, **opts):
    """batchdecode! of BeliefPropagationOSDDecoder (OSD-0, or order O with osd_order = O)."""
    dec = pkg.BeliefPropagationOSDDecoder(H, per, mi, **opts)
    n, B = H.shape[1], syn.shape[1]
    errors = np.full((n, B), 1, dtype=np.uint8, order="F")
    _, success = pkg.batchdecode_b(dec, np.asfortranarray(syn), errors)
    out = dict(errors=errors, converged=success.copy(), stats=dec.last_osd_stats.copy(), info=dec.bp_decoder.info())
    dec.close()
    return out


def bposd_device_pipeline(pkg, H, per, mi, syn):
    """ldpcb200_decode_device with ratio_last_only = 1, then ldpcb200_osd0_device on the same handle."""
    import torch
    dec = pkg.BeliefPropagationDecoder(H, per, mi, ratio_last_only=1)
    info = dec.info()
    n, B = H.shape[1], syn.shape[1]
    dev = torch.device("cuda:0")
    synw = torch.from_numpy(pack_rows(syn, info["syn_words"])).to(dev)
    errw = torch.full((B, info["err_words"]), -1, dtype=torch.int32, device=dev)
    conv = torch.full((B,), 7, dtype=torch.uint8, device=dev)
    ratio = torch.zeros((B, n), dtype=torch.float64, device=dev)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    dec.decode_device(B, synw.data_ptr(), errw.data_ptr(), conv.data_ptr(), None, ratio.data_ptr() if mi > 0 else None, None)
    if mi <= 0:
        ratio.fill_(1.0)                   # max_iters = 0: log_probabs stays zero, ratio 1 everywhere
    torch.cuda.synchronize()
    dec.osd0_device(B, synw.data_ptr(), errw.data_ptr(), conv.data_ptr(), ratio.data_ptr(), stats.data_ptr())
    torch.cuda.synchronize()
    out = dict(errors=unpack_rows(errw.cpu().numpy(), n), converged=conv.cpu().numpy().astype(bool), stats=stats.cpu().numpy()[:3])
    dec.close()
    return out


def assert_osd_same(g, ref, cols, what, order=0):
    re, rc = ref["errors"][:, cols], ref["converged"][cols]
    bad = np.nonzero((g["errors"] != re).any(axis=0) | (g["converged"] != rc))[0]
    assert bad.size == 0, "%s: mismatching syndromes %s of %d" % (what, bad[:10], re.shape[1])
    if order == 0:
        assert g["stats"][0] == int((~rc).sum()), (what, g["stats"])
        assert g["stats"][1] == int(ref["pivots"][cols].sum()), (what, g["stats"], int(ref["pivots"][cols].sum()))
    else:
        assert g["stats"][0] == re.shape[1], (what, g["stats"])      # every syndrome goes through the search


# ---------------------------------------------------------------------------------------------------------------------
# GPU: OSD-0 on crafted inputs
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["O1", "O2a", "O2b", "O3", "O4", "O5a", "O5b", "O7"])
def test_osd0_device_on_crafted_inputs(pkg, oracle, name):
    """ldpcb200_osd0_device as a function of (syndrome, bp_err, ratio) alone: every ratio class, all-zero / all-one /
    random decisions, converged flags on decisions that do not satisfy the syndrome.  Unconverged columns equal
    osd0_given bit for bit, converged ones come back untouched; stats = (unconverged, the oracle's pivot sum)."""
    H = ograph(name)
    syn = syndromes_of(oracle, name, H)
    bp_err, ratio, conv = crafted_inputs(H, syn, sum(map(ord, name)))
    unsat = ((H @ bp_err) % 2 != syn).any(axis=0)
    assert (conv & unsat).sum() >= 10 and (~conv).sum() >= 100
    ref = oracle.osd0_given(H, syn, bp_err, ratio, nthreads=oracle.num_threads())
    got, stats = osd0_on_device(pkg, H, syn, bp_err, ratio, conv)
    unc = np.nonzero(~conv)[0]
    bad = unc[(got[:, unc] != ref["errors"][:, unc]).any(axis=0)]
    assert bad.size == 0, "%s: OSD-0 differs on syndromes %s (ratio classes %s)" % (
        name, bad[:10], sorted({RATIO_CLASSES[b % 5] for b in bad}))
    assert np.array_equal(got[:, conv], bp_err[:, conv]), name
    assert stats[0] == unc.size and stats[1] == int(ref["pivots"][unc].sum()), (name, stats)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: BP -> OSD-0 and BP -> OSD-k at every prior, on every BP path that feeds them
def osd0_paths(B):
    small = np.unique(np.r_[0, 1, np.linspace(0, B - 1, 98).astype(int)])          # <= SM count: node-parallel kernel
    tiny = np.unique(np.r_[0, np.linspace(0, B - 1, 7).astype(int)])
    allc = np.arange(B)
    return [("default", {}, allc), ("node_parallel", {}, small), ("small_batch0", {"small_batch": 0}, small),
            ("global", {"family": 2}, allc), ("grid", {"grid_kernel": 2}, tiny), ("chunk64", {"chunk": 64}, allc),
            ("two_devices", {"devices": [0, 0]}, allc), ("device_pipeline", None, allc)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["O1", "O3", "O4", "G1", "G3", "C2", "C3"])
def test_bp_osd0_every_path_at_every_prior(pkg, oracle, codes, name):
    """BP -> OSD-0 against bposd_decode at every prior of the BP sweep, on every BP path that can feed OSD-0: the host
    batch (lean kernel with ratio_last_only and the filter), the node-parallel and the grid kernel, the persistent kernel
    on a small batch, the global family, two staging sets, two device slots, the device-resident pipeline."""
    H, mi = graph(codes, name)
    syn = syndromes_of(oracle, name, H)
    B = syn.shape[1]
    assert B > 148
    for per in PRIORS:
        ref = oracle.bposd_decode(H, per, mi, syn, nthreads=oracle.num_threads())
        for label, opts, cols in osd0_paths(B):
            what = "%s per=%r path=%s" % (name, per, label)
            sub = np.asfortranarray(syn[:, cols])
            if opts is None:
                g = bposd_device_pipeline(pkg, H, per, mi, sub)
            else:
                g = bposd_host(pkg, H, per, mi, sub, **opts)
            assert_osd_same(g, ref, cols, what)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["O1", "O3", "O4", "G1", "G3", "C2", "C3"])
def test_bp_osdk_host_batch_at_every_prior(pkg, oracle, codes, name):
    """BP -> order-O OSD (orders 2 and 7) through the host batch at every prior, against bposd_order_decode."""
    H, mi = graph(codes, name)
    syn = syndromes_of(oracle, name, H)
    cols = np.arange(syn.shape[1]) if H.shape[0] < 1000 else np.r_[0:12, 96:108]
    sub = np.asfortranarray(syn[:, cols])
    for per in PRIORS:
        for order in (2, 7):
            ref = oracle.bposd_order_decode(H, per, mi, order, sub, nthreads=oracle.num_threads())
            g = bposd_host(pkg, H, per, mi, sub, osd_order=order)
            assert_osd_same(g, ref, slice(None), "%s per=%r order=%d" % (name, per, order), order=order)


@pytest.mark.gpu
def test_sampling_harness_with_order_o_osd(pkg, oracle, codes):
    """ldpcb200_sample_decode_score(osd = 1) with osd_order set (BP without ratio_last_only, then the order-O search on
    every syndrome): the counters equal numpy scoring of the oracle's BP -> OSD-k output on the same samples."""
    H = codes.gross_x()
    L = codes.css_logicals(H, codes.gross_z())
    shots, first, seed, per = 3000, 500, 4321, 0.08
    truth, syn = oracle.sample(H, per, seed, first, shots)
    bpref = oracle.batch_decode(H, per, 32, syn, nthreads=oracle.num_threads())
    for order in (2, 7):
        ref = oracle.bposd_order_decode(H, per, 32, order, syn, nthreads=oracle.num_threads())
        resid = ref["errors"] ^ truth
        sat = ((H @ ref["errors"]) % 2 == syn).all(axis=0)
        logical = ((L @ resid) % 2 != 0).any(axis=0)
        want = dict(shots=shots, converged=int(bpref["converged"].sum()), iterations=int(bpref["iters"].sum()),
                    exact_matches=int((resid == 0).all(axis=0).sum()), syndrome_satisfied=int(sat.sum()),
                    failures=int((~sat | logical).sum()), residual_weight=int(resid.sum()), osd_processed=shots)
        dec = pkg.BeliefPropagationDecoder(H, per, 32, osd_order=order)
        dec.set_logicals(L)
        got = dec.sample_decode_score(shots, first, seed, per, osd=True)
        dec.close()
        assert got == want, (order, got, want)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the order-O search
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "O1"])
def test_osd_orders_1_to_12(pkg, oracle, codes, name):
    """Every order the library accepts; orders 9..12 run 512..4096 trials, several passes of the 256-thread CTA."""
    H, mi = graph(codes, name)
    assert H.shape[1] - gf2_rank(H) >= 12
    syn = syndromes_of(oracle, name, H)
    for order in range(1, 13):
        cols = np.r_[0:8, 96:104] if order < 10 else np.r_[0:3, 96:99]
        sub = np.asfortranarray(syn[:, cols])
        per = SAMPLE_RATE[name]
        ref = oracle.bposd_order_decode(H, per, mi, order, sub, nthreads=oracle.num_threads())
        g = bposd_host(pkg, H, per, mi, sub, osd_order=order)
        assert_osd_same(g, ref, slice(None), "%s order=%d" % (name, order), order=order)


def full_rank(m, extra, seed):
    """m x (m + extra) of rank m: a unit upper-triangular block, then `extra` random columns."""
    rng = np.random.default_rng(seed)
    T = np.triu((rng.random((m, m)) < 0.1).astype(np.uint8), 1) | np.eye(m, dtype=np.uint8)
    return sp.csc_matrix(np.hstack([T, (rng.random((m, extra)) < 0.2).astype(np.uint8)]))


@pytest.mark.gpu
def test_osd_order_clamp_and_trial_ties(pkg, oracle, codes):
    """order = min(order, n - rank) with n - rank = 0, 1 and 5; and trials that tie on weight (every key equal: per = 0.5
    or max_iters = 0), where the smallest x among the lightest must win."""
    for extra in (0, 1, 5):
        H = full_rank(40, extra, 7 + extra)
        assert gf2_rank(H) == 40
        _, syn = oracle.sample(H, 0.1, 3, 0, 24)
        for order in (1, 6, 12):
            ref = oracle.bposd_order_decode(H, 0.1, 5, order, syn)
            g = bposd_host(pkg, H, 0.1, 5, syn, osd_order=order)
            assert_osd_same(g, ref, slice(None), "n-rank=%d order=%d" % (extra, order), order=order)
    from test_gpu_parity import _cycle_matrix
    rng = np.random.default_rng(11)
    for H in (_cycle_matrix(9), sp.csc_matrix(codes.surface_x(5))):
        syn = np.asfortranarray((rng.random((H.shape[0], 32)) < 0.3).astype(np.uint8))
        for per, mi in ((0.5, 3), (0.1, 0)):
            for order in (3, 8, 12):
                ref = oracle.bposd_order_decode(H, per, mi, order, syn)
                g = bposd_host(pkg, H, per, mi, syn, osd_order=order)
                assert_osd_same(g, ref, slice(None), "ties %s per=%r mi=%d order=%d" % (H.shape, per, mi, order), order=order)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the limits
def tall(m, n, seed):
    """m x n, variables of degree 7, checks of degree 2 and 3 (needs 2m <= 7n <= 3m)."""
    k3 = 7 * n - 2 * m
    return configuration_model({2: m - k3, 3: k3}, {7: n}, seed)


@pytest.mark.gpu
def test_order_o_osd_beyond_the_osd0_row_limit(pkg, oracle):
    """3000 checks: OSD-0 refuses (EUNSUPPORTED), orders 1 and 4 decode bit for bit."""
    H = ograph("O6")
    syn = np.asfortranarray(syndromes_of(oracle, "O6", H)[:, np.r_[0:12, 96:108]])
    with pytest.raises(pkg._lib.LibraryError) as e:
        bposd_host(pkg, H, 0.1, MAX_ITERS, syn)
    assert e.value.code == pkg._lib.EUNSUPPORTED
    for order in (1, 4):
        ref = oracle.bposd_order_decode(H, 0.1, MAX_ITERS, order, syn, nthreads=oracle.num_threads())
        g = bposd_host(pkg, H, 0.1, MAX_ITERS, syn, osd_order=order)
        assert_osd_same(g, ref, slice(None), "O6 order=%d" % order, order=order)


@pytest.mark.gpu
def test_osd0_shared_memory_and_row_limits(pkg, oracle):
    """At 2048 checks the widest matrix that fits the device's shared memory decodes, one column more is refused; 2049
    checks are refused; a refused call leaves the handle able to decode plain BP."""
    import torch
    budget = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    fit_n, over_n = straddle(budget)
    if budget == B200_SMEM_OPTIN:
        assert (fit_n, over_n) == (639, 640)
    Hf = ograph("O4") if fit_n == 639 else tall(OSD_MAX_ROWS, fit_n, 211)
    syn = np.asfortranarray(syndromes_of(oracle, "O4", ograph("O4"))[:, 90:110]) if fit_n == 639 else \
        np.asfortranarray((np.random.default_rng(3).random((OSD_MAX_ROWS, 20)) < 0.5).astype(np.uint8))
    ref = oracle.bposd_decode(Hf, 0.3, MAX_ITERS, syn, nthreads=oracle.num_threads())
    assert_osd_same(bposd_host(pkg, Hf, 0.3, MAX_ITERS, syn), ref, slice(None), "%d x %d" % Hf.shape)
    for H in (tall(OSD_MAX_ROWS, over_n, 212), tall(OSD_MAX_ROWS + 1, 639, 213)):
        s = np.asfortranarray((np.random.default_rng(4).random((H.shape[0], 20)) < 0.5).astype(np.uint8))
        dec = pkg.BeliefPropagationOSDDecoder(H, 0.3, MAX_ITERS)
        errors = np.zeros((H.shape[1], 20), dtype=np.uint8, order="F")
        with pytest.raises(pkg._lib.LibraryError) as e:
            pkg.batchdecode_b(dec, s, errors)
        assert e.value.code == pkg._lib.EUNSUPPORTED, H.shape
        ref = oracle.batch_decode(H, 0.3, MAX_ITERS, s)
        _, conv = pkg.batchdecode_b(dec.bp_decoder, s, errors)
        assert np.array_equal(errors, ref["errors"]) and np.array_equal(conv, ref["converged"]), H.shape
        dec.close()
