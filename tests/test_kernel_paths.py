"""Every decoding path of the BP kernels on designed irregular Tanner graphs and at degenerate priors.

The named codes are regular or nearly so and are decoded at ordinary error rates.  The graphs here are built from chosen
degree sequences so that each branch of the kernel selector is taken on purpose: degree-sorted node segments with empty
rows and columns, 64-bit decision fields, contiguous variable ownership with a ragged last group of four, a check of
degree exactly 12 or 13, more than eight distinct check degrees.  The priors include 0, a subnormal and a saturating
ratio, the neighbours of 0.5 and 1, and 1 itself (the only ones for which the kernels' `regular_p0` is false).

Each GPU case forces its path through public options, confirms it from info(), the launch count, the timed persistent
launches and the counters, and must equal the CPU oracle bit for bit (decisions, flags, iterations, posterior-ratio bits
where requested).  counters[3] pins the first-iteration filter (bp_filter.cuh): it must equal the number of syndromes the
oracle finishes and converges in iteration 1 wherever the filter is eligible, and 0 elsewhere, so a filter that silently
switched itself off, or on, fails."""
import functools

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import bp_dense

SMEM, GLOBAL = 1, 2
MAX_SEG = 8               # bp::kMaxSeg: distinct degrees the lean kernel's segments can cover
FILTER_MAX_VDEG = 5       # bp::kFilterMaxVarDeg
MAX_REG_DEG = 12          # bp::kMaxRegDegree: larger nodes take the general kernel's local-memory path
MAX_ITERS = 12            # designed graphs (the named codes keep their own)

PRIORS = [0.0, 1e-310, 1e-300, 0.01, 0.05, float(np.nextafter(0.5, 0.0)), 0.5, float(np.nextafter(0.5, 1.0)),
          1.0 - 2.0 ** -53, 1.0]
DEGENERATE = [0.0, 1e-310, 1e-300, 0.5, 1.0 - 2.0 ** -53, 1.0]
VARIANT_PRIORS = [1e-300, 0.01, 0.5, 1.0 - 2.0 ** -53]


# ---------------------------------------------------------------------------------------------------------------------
# designed graphs
def configuration_model(check_degs, var_degs, seed):
    """H with exactly the given check and variable degree counts ({degree: count}): edge stubs of the checks are
    matched to those of the variables in random order; matchings with a double edge are rejected and redrawn."""
    rng = np.random.default_rng(seed)
    cd = rng.permutation(np.repeat(list(check_degs), list(check_degs.values())))
    vd = rng.permutation(np.repeat(list(var_degs), list(var_degs.values())))
    assert cd.sum() == vd.sum(), (cd.sum(), vd.sum())
    s, n = len(cd), len(vd)
    v_stubs = np.repeat(np.arange(n), vd)
    for _ in range(20000):
        c_stubs = rng.permutation(np.repeat(np.arange(s), cd))
        if len(np.unique(c_stubs * n + v_stubs)) == len(v_stubs):
            return sp.csc_matrix((np.ones(len(v_stubs), dtype=np.uint8), (c_stubs, v_stubs)), shape=(s, n))
    raise RuntimeError("no simple graph drawn for this degree sequence")


G1_VARS = {0: 6, 1: 150, 2: 76, 3: 18, 5: 10}
SPECS = {
    # eight distinct check degrees (0, 1 and 12 among them), five variable degrees including 0
    "G1": ({0: 3, 1: 15, 2: 55, 3: 47, 4: 20, 5: 6, 6: 3, 12: 1}, G1_VARS, 101),
    # uniform variable degree 3, irregular checks
    "G3": ({3: 17, 4: 31, 5: 29, 6: 20, 7: 15, 8: 8}, {3: 203}, 103),
    # one check of degree exactly 12 (register path) / 13 (local-memory path)
    "G4a": ({2: 1, 3: 14, 4: 8, 12: 1}, {1: 16, 2: 24, 3: 8}, 104),
    "G4b": ({2: 1, 3: 15, 4: 7, 13: 1}, {1: 16, 2: 24, 3: 8}, 105),
    # ten distinct check degrees, all <= 12: no segments
    "G5": ({1: 40, 2: 30, 3: 48, 4: 20, 5: 4, 6: 3, 7: 2, 8: 1, 10: 1, 12: 1}, G1_VARS, 106),
}


@functools.lru_cache(maxsize=None)
def designed(name):
    if name == "G2":
        # G1 plus one variable of degree 6 (filter ineligible); its checks had degree 2..4, so the set of check degrees
        # stays the same
        H = designed("G1").tolil()
        cdeg = np.asarray(H.sum(axis=1)).ravel()
        rng = np.random.default_rng(102)
        rows = np.concatenate([rng.choice(np.nonzero(cdeg == d)[0], 2, replace=False) for d in (2, 3, 4)])
        col = sp.lil_matrix((H.shape[0], 1), dtype=np.uint8)
        col[rows, 0] = 1
        return sp.csc_matrix(sp.hstack([H, col]))
    checks, vars_, seed = SPECS[name]
    return configuration_model(checks, vars_, seed)


def degrees(H):
    H = sp.csc_matrix(H)
    return np.asarray(H.sum(axis=1)).ravel().astype(int), np.asarray(H.sum(axis=0)).ravel().astype(int)


def graph(codes, name):
    """(H, max_iters) of a designed graph or a named code."""
    if name in ("C2", "C3"):
        H, _, mi = codes.config_matrix(name)
        return sp.csc_matrix(H), mi
    return designed(name), MAX_ITERS


# What the kernel selector must pick for each graph by default (confirmed from info() in every GPU case):
#   lean     the shared-memory kernel of bp_smem.cuh (kernel_rev 2): <= 8 distinct degrees each side, no node above 12
#   filter   first-iteration filter eligible on the lean paths: additionally no variable above degree 5
#   dual     the two-team form fits (two CTAs of 8 warps per SM at most)
META = {
    "G1": dict(lean=True, filter=True, dual=True),
    "G2": dict(lean=True, filter=False, dual=True),
    "G3": dict(lean=True, filter=True, dual=False),      # 609 edges: one CTA per SM
    "G4a": dict(lean=True, filter=True, dual=True),
    "G4b": dict(lean=False, filter=False, dual=False),   # big: general kernel, local-memory degree path
    "G5": dict(lean=False, filter=False, dual=False),    # > 8 distinct check degrees: no segments
    "C2": dict(lean=True, filter=True, dual=True),
    "C3": dict(lean=True, filter=True, dual=True),
}


# A 4 x 11 graph (degree-0 variables included) and a prior at which one first-iteration decision is decided by the last
# bit of a check output that depends on the position inside the check (see test_near_tie_...); every syndrome of it.
NEAR_TIE = (np.array([[0, 0, 0, 0, 0, 0, 1, 0, 1, 0, 0],
                      [0, 0, 1, 1, 0, 0, 1, 0, 1, 1, 0],
                      [0, 0, 0, 1, 0, 1, 0, 0, 0, 1, 0],
                      [0, 1, 0, 1, 0, 0, 1, 0, 0, 1, 1]], dtype=np.uint8), 0.13992169903478202, 10)
NEAR_TIE_SYN = np.array([[(b >> i) & 1 for b in range(16)] for i in range(4)], dtype=np.uint8)

_SYN = {}
_REF = {}


def syndromes_of(oracle, name, H):
    """Columns: zero, H*1 (the syndrome of the all-ones error), 256 sampled at 0.005 and 256 at 0.02 (the oracle
    finishes most of the first and about a quarter of the second in iteration 1), 64 uniformly random (mostly outside
    the column space)."""
    if name not in _SYN:
        s = H.shape[0]
        ones = (np.asarray(H.sum(axis=1)).ravel() % 2).astype(np.uint8)
        _, a = oracle.sample(H, 0.005, 7, 0, 256)
        _, b = oracle.sample(H, 0.02, 8, 0, 256)
        rnd = (np.random.default_rng(9).random((s, 64)) < 0.5).astype(np.uint8)
        _SYN[name] = np.asfortranarray(np.column_stack([np.zeros(s, np.uint8), ones, a, b, rnd]).astype(np.uint8))
    return _SYN[name]


def reference(oracle, name, H, per, mi, syn, variant="exact"):
    """Oracle outputs (ratios included) once per (graph, prior, variant); every path of a case is compared with it."""
    key = (name, per, mi, variant)
    if key not in _REF:
        _REF[key] = oracle.batch_decode(H, per, mi, syn, nthreads=oracle.num_threads(), want_ratio=True, variant=variant)
    return _REF[key]


def finished_in_iteration_1(ref, cols=slice(None)):
    return int((ref["converged"][cols] & (ref["iters"][cols] == 1)).sum())


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the graphs have the promised profiles; the oracle is sound at the degenerate priors
def test_designed_graph_profiles():
    cd, vd = degrees(designed("G1"))
    assert designed("G1").shape == (150, 260)
    assert set(vd) == {0, 1, 2, 3, 5} and len(set(cd)) <= MAX_SEG and {0, 1, 12} <= set(cd) and cd.max() == 12
    assert (cd == 0).sum() >= 2 and (vd == 0).sum() >= 3
    # decision fields: 64-bit with 8 warps (ceil(n / warps) > 32), 32-bit with 12
    assert -(-260 // 8) > 32 and -(-260 // 12) <= 32
    # G1 fits two CTAs of the lean kernel per SM (and its two-team form): at most ~420 edges
    assert designed("G1").nnz <= 410

    cd2, vd2 = degrees(designed("G2"))
    assert designed("G2").shape == (150, 261) and (designed("G2")[:, :260] != designed("G1")).nnz == 0
    assert vd2.max() == 6 > FILTER_MAX_VDEG and set(vd2) == {0, 1, 2, 3, 5, 6}
    assert set(cd2) == set(cd) and cd2.max() == 12
    assert designed("G2").nnz <= 420

    cd3, vd3 = degrees(designed("G3"))
    assert designed("G3").shape == (120, 203) and set(vd3) == {3}
    assert 2 <= len(set(cd3)) <= MAX_SEG and cd3.max() <= MAX_REG_DEG
    cpw = -(-203 // 8)                     # contiguous ownership at 8 warps: variables per warp, last warp's share
    assert cpw % 4 != 0 and (203 - 7 * cpw) % 4 != 0

    for name, top in (("G4a", 12), ("G4b", 13)):
        cd4, vd4 = degrees(designed(name))
        assert cd4.max() == top and (cd4 == top).sum() == 1 and vd4.max() <= 3 and len(set(cd4)) <= MAX_SEG

    cd5, vd5 = degrees(designed("G5"))
    assert designed("G5").shape == (150, 260)
    assert len(set(cd5)) > MAX_SEG and cd5.max() <= MAX_REG_DEG and vd5.max() <= FILTER_MAX_VDEG


@pytest.mark.parametrize("name", ["G1", "C2"])
def test_dense_transliteration_agrees_at_degenerate_priors(oracle, codes, name):
    """The C oracle against the independent dense restatement (oracle/bp_dense.py) at every degenerate prior:
    decisions, flags, iterations and the bits of the posterior ratios."""
    H, mi = graph(codes, name)
    syn = syndromes_of(oracle, name, H)[:, [0, 1, 2, 3, 258, 259, 514, 515]]
    Hd = H.toarray()
    for per in DEGENERATE:
        r = oracle.batch_decode(H, per, mi, syn, want_ratio=True)
        for b in range(syn.shape[1]):
            e, c, ratio, it = bp_dense.decode_dense(Hd, per, mi, syn[:, b])
            assert np.array_equal(e.astype(np.uint8), r["errors"][:, b]), (per, b)
            assert c == bool(r["converged"][b]) and it == r["iters"][b], (per, b)
            assert np.array_equal(ratio.view(np.uint64), r["ratio"][:, b].view(np.uint64)), (per, b)


def test_near_tie_graph_hinges_on_the_position_inside_a_check(oracle):
    """In iteration 1 every input of a check is the prior, so its outputs differ by position only through rounding: the
    middle output of a degree-5 check is a product of the same four factors in another association than the end ones.
    NEAR_TIE is a graph and a prior (found by search) where that last bit decides a first decision: variable 6 sits at
    position 2 of both degree-5 checks and in a degree-2 check whose output cancels the prior, and its ratio for
    syndrome 0b0011 is 1 - 2^-52 -- the oracle decides 0 and converges in iteration 1.  A filter table built with
    another position would decide 1 there."""
    H, per, _ = NEAR_TIE
    r = oracle.batch_decode(H, per, 1, NEAR_TIE_SYN[:, [3]], want_ratio=True)
    assert r["ratio"][6, 0] == 1.0 - 2.0 ** -52 and r["errors"][6, 0] == 0 and r["converged"][0]
    assert np.nonzero(H[1])[0].tolist().index(6) == 2 and np.nonzero(H[3])[0].tolist().index(6) == 2
    assert H[:, 6].sum() == 3 and H[0].sum() == 2 and H[1].sum() == H[3].sum() == 5


@pytest.mark.parametrize("name", ["G1", "G2", "G3", "G4a", "G4b", "G5", "C2", "C3"])
def test_oracle_ratios_have_no_nan(oracle, codes, name):
    """Bitwise comparison of posterior ratios is well defined only without NaN (whose payload a GPU need not
    reproduce).  At every prior of the GPU sweep the oracle's ratios are free of NaN; they do contain +-Inf and zeros."""
    H, mi = graph(codes, name)
    syn = syndromes_of(oracle, name, H)
    for per in PRIORS:
        r = reference(oracle, name, H, per, mi, syn)
        nan = np.isnan(r["ratio"])
        assert not nan.any(), "%s, per %r: %d NaN posterior ratios (columns %s): bitwise ratio checks are void here" % (
            name, per, int(nan.sum()), np.nonzero(nan.any(axis=0))[0][:10])


# ---------------------------------------------------------------------------------------------------------------------
# GPU runners
def decode_host(pkg, H, per, mi, syn, variant="exact", want_ratio=False, **opts):
    """batchdecode! through the host entry point; returns outputs, info, counters and how the work was launched."""
    dec = pkg.BeliefPropagationDecoder(H, per, mi, variant=variant, time_kernels=1, **opts)
    n, B = H.shape[1], syn.shape[1]
    errors = np.full((n, B), 7, dtype=np.uint8, order="F")
    iters = np.full(B, -1, dtype=np.int32)
    ratio = np.zeros((n, B), dtype=np.float64, order="F") if want_ratio else None
    _, conv = pkg.batchdecode_b(dec, np.asfortranarray(syn), errors, iters=iters, posterior_ratio=ratio)
    out = dict(errors=errors, converged=conv, iters=iters, ratio=ratio, info=dec.info(), counters=dec.last_counters.copy(),
               launches=dec.launch_count(), persistent=dec.kernel_time()[1])
    dec.close()
    return out


def decode_device(pkg, H, per, mi, syn, **opts):
    """ldpcb200_decode_device on packed device rows with option ratio_last_only = 1 (the OSD pipeline's call): ratios of
    iteration max_iters only, so the filter stays eligible."""
    import torch
    dec = pkg.BeliefPropagationDecoder(H, per, mi, time_kernels=1, ratio_last_only=1, **opts)
    info = dec.info()
    s, n = H.shape
    B = syn.shape[1]
    SW, NW = info["syn_words"], info["err_words"]
    pad = np.zeros((B, SW * 32), dtype=np.uint8)
    pad[:, :s] = syn.T
    dev = torch.device("cuda:0")
    synw = torch.from_numpy(np.packbits(pad, axis=1, bitorder="little").view(np.int32).copy()).to(dev)
    errw = torch.full((B, NW), -1, dtype=torch.int32, device=dev)
    conv = torch.full((B,), 7, dtype=torch.uint8, device=dev)
    iters = torch.full((B,), -1, dtype=torch.int32, device=dev)
    ratio = torch.zeros((B, n), dtype=torch.float64, device=dev)
    ctr = torch.zeros(4, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()                          # (the library's stream does not order itself after torch's)
    dec.decode_device(B, synw.data_ptr(), errw.data_ptr(), conv.data_ptr(), iters.data_ptr(), ratio.data_ptr(), ctr.data_ptr())
    torch.cuda.synchronize()
    errors = np.unpackbits(errw.cpu().numpy().view(np.uint8), axis=1, bitorder="little")[:, :n].T
    out = dict(errors=np.asfortranarray(errors), converged=conv.cpu().numpy().astype(bool), iters=iters.cpu().numpy(),
               ratio=np.asfortranarray(ratio.cpu().numpy().T), info=info, counters=ctr.cpu().numpy(),
               launches=dec.launch_count(), persistent=dec.kernel_time()[1])
    dec.close()
    return out


def assert_same(g, r, cols=slice(None), ratio_cols=None, what=""):
    """Bit-exact against the oracle (restricted to `cols`); ratios compared on `ratio_cols` (None: not requested);
    counters [0..2] equal to the oracle's sums."""
    re, rc, ri = r["errors"][:, cols], r["converged"][cols], r["iters"][cols]
    bad = np.nonzero((g["errors"] != re).any(axis=0) | (g["converged"] != rc) | (g["iters"] != ri))[0]
    assert bad.size == 0, "%s: mismatching syndromes %s of %d" % (what, bad[:10], re.shape[1])
    if ratio_cols is not None:
        a = g["ratio"][:, ratio_cols].view(np.uint64)
        b = r["ratio"][:, cols][:, ratio_cols].view(np.uint64)
        badr = np.nonzero((a != b).any(axis=0))[0]
        assert badr.size == 0, "%s: posterior-ratio bits differ on syndromes %s" % (what, badr[:10])
    c = g["counters"]
    assert c[0] == re.shape[1] and c[1] == int(rc.sum()) and c[2] == int(ri.sum()), (what, c)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every path of the exact variant at every prior
def paths_for(name, meta, B):
    """(label, runner, options, columns, expectations) of every path that applies to the graph."""
    all_cols = np.arange(B)
    small = np.unique(np.r_[0, 1, np.linspace(0, B - 1, 98).astype(int)])        # <= SM count: node-parallel kernel
    tiny = np.unique(np.r_[0, 1, np.linspace(0, B - 1, 22).astype(int)])
    lean_rev = 2 if meta["lean"] else 1
    P = [
        ("default", "host", {}, all_cols, dict(family=SMEM, rev=lean_rev, filt=meta["filter"], persistent=1)),
        ("ratios", "host", {}, all_cols, dict(family=SMEM, rev=lean_rev, filt=False, persistent=1, ratio=True)),
        ("ratio_last_only", "device", {}, all_cols, dict(family=SMEM, rev=lean_rev, filt=meta["filter"], persistent=1)),
        ("static_queue", "host", {"dynamic_queue": 0}, all_cols, dict(family=SMEM, rev=lean_rev, filt=meta["filter"], persistent=1)),
        ("global_pf0", "host", {"family": GLOBAL, "prefetch": 0}, all_cols, dict(family=GLOBAL, mode=1, rev=1, filt=False, persistent=1, pd=0)),
        ("global", "host", {"family": GLOBAL}, all_cols, dict(family=GLOBAL, mode=1, rev=1, filt=False, persistent=1)),
    ]
    if meta["lean"]:
        P += [
            ("no_filter", "host", {"first_iteration_filter": 0}, all_cols, dict(family=SMEM, rev=2, filt=False, persistent=1)),
            ("general", "host", {"lean": 0}, all_cols, dict(family=SMEM, rev=1, filt=False, persistent=1)),
        ]
    if meta["dual"]:
        P.append(("dual", "host", {"dual": 1, "warps": 8}, all_cols, dict(family=SMEM, rev=3, filt=meta["filter"], persistent=1)))
    if name in ("G1", "G2"):
        P += [("warps8_eb64", "host", {"warps": 8}, all_cols, dict(family=SMEM, rev=2, filt=meta["filter"], persistent=1, warps=8)),
              ("warps12_eb32", "host", {"warps": 12}, all_cols, dict(family=SMEM, rev=2, filt=meta["filter"], persistent=1, warps=12))]
    if name == "G3":
        P += [("contiguous", "host", {"warps": 8}, all_cols, dict(family=SMEM, rev=2, filt=True, persistent=1, warps=8)),
              ("interleaved", "host", {"warps": 8, "contiguous_variables": 0}, all_cols, dict(family=SMEM, rev=2, filt=True, persistent=1, warps=8))]
    if name != "G4b":        # (nodes above degree 12 always take the persistent kernel)
        P += [("node_parallel", "host", {}, small, dict(filt=False, persistent=0)),
              ("grid", "host", {"grid_kernel": 2}, tiny, dict(filt=False, persistent=0))]
    return P


GPU_GRAPHS = ["G1", "G2", "G3", "G4a", "G4b", "G5", "C2", "C3"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_GRAPHS)
def test_every_path_at_every_prior(pkg, oracle, codes, name):
    """Every applicable path (paths_for) at every prior, against one oracle run per prior.  (The node-parallel and the
    grid kernel both show no persistent launch; the grid kernel is only reachable through grid_kernel = 2 on graphs
    this small, so each of the two cases runs the kernel it names.)"""
    H, mi = graph(codes, name)
    syn = syndromes_of(oracle, name, H)
    meta = META[name]
    B = syn.shape[1]
    n = H.shape[1]
    for per in PRIORS:
        ref = reference(oracle, name, H, per, mi, syn)
        smem = {}
        for label, runner, opts, cols, ex in paths_for(name, meta, B):
            what = "%s per=%r path=%s" % (name, per, label)
            sub = np.asfortranarray(syn[:, cols])
            if runner == "device":
                g = decode_device(pkg, H, per, mi, sub, **opts)
                # ratios are written in iteration max_iters only: compare the syndromes that ran that long
                assert_same(g, ref, cols, ratio_cols=np.nonzero(ref["iters"][cols] == mi)[0], what=what)
                # one decoding kernel, plus the two table kernels and the filter kernel when the filter runs
                assert g["launches"] == 1 + (3 if ex["filt"] else 0), (what, g["launches"])
            else:
                g = decode_host(pkg, H, per, mi, sub, want_ratio=ex.get("ratio", False), **opts)
                assert_same(g, ref, cols, ratio_cols=np.arange(len(cols)) if ex.get("ratio") else None, what=what)
            info = g["info"]
            if "family" in ex:
                assert info["family"] == ex["family"] and info["kernel_mode"] == ex.get("mode", 0), (what, info)
                assert info["kernel_rev"] == ex["rev"], (what, info)
            if "pd" in ex:
                assert info["prefetch_distance"] == ex["pd"], (what, info)
            if "warps" in ex:
                assert info["threads_per_cta"] == 32 * ex["warps"], (what, info)
            assert g["persistent"] == ex["persistent"], (what, g["persistent"])
            want = finished_in_iteration_1(ref, cols) if ex["filt"] else 0
            assert g["counters"][3] == want, (what, g["counters"], want)
            smem[label] = info["smem_bytes"]
        if name == "G3":
            # contiguous ownership has its own table layout (no row / column pointers, per-warp padding)
            assert smem["contiguous"] != smem["interleaved"], smem
        if name in ("G1", "G2"):
            assert -(-n // 8) > 32 >= -(-n // 12)        # 64-bit decision fields at 8 warps, 32-bit at 12


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["G1", "C3"])
def test_set_per_walks_through_every_prior(pkg, oracle, codes, name):
    """One handle, the prior changed under it: regular_p0 goes false -> true -> false and the filter's tables are rebuilt
    each time; every result equals the oracle's, and returning to the first prior gives the first result again."""
    H, mi = graph(codes, name)
    syn = syndromes_of(oracle, name, H)
    B = syn.shape[1]
    dec = pkg.BeliefPropagationDecoder(H, 0.05, mi)

    def run():
        errors = np.zeros((H.shape[1], B), dtype=np.uint8, order="F")
        iters = np.zeros(B, dtype=np.int32)
        _, conv = pkg.batchdecode_b(dec, syn, errors, iters=iters)
        return dict(errors=errors, converged=conv.copy(), iters=iters, counters=dec.last_counters.copy())

    first = run()
    assert dec.info()["kernel_rev"] == 2
    for per in PRIORS + [0.05]:
        dec.set_per(per)
        g = run()
        ref = reference(oracle, name, H, per, mi, syn)
        assert_same(g, ref, what="%s set_per(%r)" % (name, per))
        assert g["counters"][3] == finished_in_iteration_1(ref), (name, per, g["counters"])
    for k in ("errors", "converged", "iters", "counters"):
        assert np.array_equal(g[k], first[k]), k
    dec.close()


@pytest.mark.gpu
def test_first_iteration_filter_near_tie(pkg, oracle):
    """Every syndrome of NEAR_TIE, 24 times over (beyond the node-parallel kernel's batch sizes), through the filter and
    without it: the filter must finish exactly the syndromes the oracle converges in iteration 1, with its decisions."""
    H, per, mi = NEAR_TIE
    syn = np.asfortranarray(np.tile(NEAR_TIE_SYN, 24))
    ref = oracle.batch_decode(H, per, mi, syn, want_ratio=True)
    assert ref["converged"][3] and ref["iters"][3] == 1
    for flt in (1, 0):
        g = decode_host(pkg, sp.csc_matrix(H), per, mi, syn, first_iteration_filter=flt)
        assert g["info"]["kernel_rev"] == 2 and g["persistent"] == 1, g["info"]
        assert_same(g, ref, what="near tie, filter %d" % flt)
        assert g["counters"][3] == (finished_in_iteration_1(ref) if flt else 0), (flt, g["counters"])


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the min-sum and fast variants on the designed graphs
def assert_fast_bar(g, ref, H, syn, what):
    """The statistical bar of test_fast32_variant_tracks_its_definition: at most 2 % of syndromes decoded differently,
    convergence rate within 0.5 % absolute, mean iterations within 2 %, every converged output satisfies its syndrome."""
    differ = ((g["errors"] != ref["errors"]).any(axis=0) | (g["converged"] != ref["converged"])).mean()
    assert differ <= 0.02, (what, differ)
    assert abs(g["converged"].mean() - ref["converged"].mean()) <= 0.005, what
    assert abs(g["iters"].mean() - ref["iters"].mean()) <= 0.02 * ref["iters"].mean() + 0.01, what
    sat = ((H @ g["errors"]) % 2 == syn).all(axis=0)
    assert (sat == g["converged"]).all(), what


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["G1", "G3", "G5"])
def test_llr_variants_on_designed_graphs(pkg, oracle, codes, name):
    H, mi = graph(codes, name)
    syn = syndromes_of(oracle, name, H)
    meta = META[name]
    for per in VARIANT_PRIORS:
        ref = reference(oracle, name, H, per, mi, syn, variant="minsum")
        what = "%s minsum per=%r" % (name, per)
        g = decode_host(pkg, H, per, mi, syn, variant="minsum")
        assert_same(g, ref, what=what + " filter")
        assert g["info"]["kernel_rev"] == (2 if meta["lean"] else 1), (what, g["info"])
        assert g["counters"][3] == (finished_in_iteration_1(ref) if meta["filter"] else 0), (what, g["counters"])
        g = decode_host(pkg, H, per, mi, syn, variant="minsum", want_ratio=True)
        assert_same(g, ref, ratio_cols=np.arange(syn.shape[1]), what=what + " ratios")
        assert g["counters"][3] == 0

        ref = reference(oracle, name, H, per, mi, syn, variant="fast")
        what = "%s fast per=%r" % (name, per)
        on = decode_host(pkg, H, per, mi, syn, variant="fast")
        off = decode_host(pkg, H, per, mi, syn, variant="fast", first_iteration_filter=0)
        for k in ("errors", "converged", "iters"):
            assert np.array_equal(on[k], off[k]), (what, k)     # the filter's tables come from the variant's own updates
        assert on["counters"][3] == (int((on["converged"] & (on["iters"] == 1)).sum()) if meta["filter"] else 0), what
        assert off["counters"][3] == 0
        assert_fast_bar(on, ref, H, syn, what)


@pytest.mark.gpu
def test_llr_variants_refuse_degenerate_priors_and_big_nodes(pkg):
    """The log-likelihood-ratio variants need 0 < per < 1 (EINVAL at create and at set_per) and nodes of degree <= 12
    (EUNSUPPORTED)."""
    H = designed("G1")
    for variant in ("minsum", "fast"):
        for per in (0.0, 1.0):
            with pytest.raises(pkg._lib.LibraryError) as e:
                pkg.BeliefPropagationDecoder(H, per, MAX_ITERS, variant=variant)
            assert e.value.code == pkg._lib.EINVAL, (variant, per)
            dec = pkg.BeliefPropagationDecoder(H, 0.05, MAX_ITERS, variant=variant)
            with pytest.raises(pkg._lib.LibraryError) as e:
                dec.set_per(per)
            assert e.value.code == pkg._lib.EINVAL, (variant, per)
            dec.close()
        with pytest.raises(pkg._lib.LibraryError) as e:
            pkg.BeliefPropagationDecoder(designed("G4b"), 0.05, MAX_ITERS, variant=variant)
        assert e.value.code == pkg._lib.EUNSUPPORTED, variant
