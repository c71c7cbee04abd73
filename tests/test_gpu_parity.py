"""Parity tests proper: the CUDA path, called through the C ABI (ctypes mirror), against the
CPU oracle on identical (H, per, max_iters, syndromes).  Bar: hard decisions, convergence flags,
executed iterations and posterior ratios are BIT-EXACT (the kernels replay the reference's FP64
operation sequence, so no tie tolerance is needed or used)."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

SMEM, GLOBAL = 1, 2


def run_gpu(pkg, H, per, max_iters, syn, family=0, want_ratio=False, fmt="u8", **opts):
    dec = pkg.BeliefPropagationDecoder(H, per, max_iters, family=family, **opts)
    s, n = H.shape
    B = syn.shape[1]
    dt = {"u8": np.uint8, "i64": np.int64, "bool": np.bool_}[fmt]
    errors = np.full((n, B), 7, dtype=dt, order="F") if fmt != "bool" else np.ones((n, B), dtype=dt, order="F")
    iters = np.full(B, -1, dtype=np.int32)
    ratio = np.zeros((n, B), dtype=np.float64, order="F") if want_ratio else None
    _, success = pkg.batchdecode_b(dec, np.asfortranarray(syn.astype(dt)), errors, iters=iters, posterior_ratio=ratio)
    info = dec.info()
    counters = dec.last_counters.copy()
    launches = dec.launch_count()
    persistent_launches = dec.kernel_time()[1]
    dec.close()
    return dict(errors=errors.astype(np.uint8), converged=success, iters=iters, ratio=ratio, info=info, counters=counters, launches=launches,
                persistent_launches=persistent_launches)


def assert_same(g, r, want_ratio=False):
    bad = np.nonzero((g["errors"] != r["errors"]).any(axis=0) | (g["converged"] != r["converged"]) | (g["iters"] != r["iters"]))[0]
    assert bad.size == 0, "mismatching syndromes: %s (of %d)" % (bad[:10], g["errors"].shape[1])
    if want_ratio:
        assert np.array_equal(g["ratio"].view(np.uint64), r["ratio"].view(np.uint64))
    B = g["errors"].shape[1]
    assert g["counters"][0] == B
    assert g["counters"][1] == int(r["converged"].sum())
    assert g["counters"][2] == int(r["iters"].sum())


CASES = [
    # name, per, B, families
    ("C3", 0.01, 3000, (SMEM, GLOBAL)),
    ("C3", 0.05, 3000, (SMEM, GLOBAL)),
    ("C3", 0.10, 2000, (SMEM, GLOBAL)),
    ("C2", 0.001, 2000, (SMEM,)),
    ("C2", 0.03, 3000, (SMEM, GLOBAL)),
    ("C2", 0.10, 2000, (SMEM,)),
    ("C4", 0.02, 600, (GLOBAL,)),
    ("C4", 0.05, 400, (GLOBAL,)),
    ("C1", 0.01, 200, (GLOBAL,)),
    ("C1", 0.04, 100, (GLOBAL,)),
]


@pytest.mark.parametrize("name,per,B,families", CASES)
def test_parity_configs(pkg, oracle, codes, name, per, B, families):
    H, _, mi = codes.config_matrix(name)
    _, syn = oracle.sample(H, per, 12345, 0, B)
    ref = oracle.batch_decode(H, per, mi, syn, nthreads=oracle.num_threads(), want_ratio=True)
    for fam in families:
        g = run_gpu(pkg, H, per, mi, syn, family=fam, want_ratio=True)
        assert g["info"]["family"] == fam
        assert_same(g, ref, want_ratio=True)
        if fam == SMEM:
            # the shared-memory family has three forms: the round-2 kernel (default where the code fits its envelope),
            # the same kernel with two teams per CTA taking turns in the check pass (dual = 1) and the general
            # persistent kernel (lean = 0); all must replay the reference bit for bit
            assert g["info"]["kernel_rev"] == 2, g["info"]
            # (posterior ratios of every iteration were requested above, which keeps the first-iteration filter off;
            #  without them the filter takes iteration 1 of every syndrome: same decisions, flags, iteration counts)
            assert_same(run_gpu(pkg, H, per, mi, syn, family=fam), ref)
            assert_same(run_gpu(pkg, H, per, mi, syn, family=fam, first_iteration_filter=0), ref)
            g = run_gpu(pkg, H, per, mi, syn, family=fam, want_ratio=True, dual=1)
            assert g["info"]["kernel_rev"] == 3
            assert_same(g, ref, want_ratio=True)
            g = run_gpu(pkg, H, per, mi, syn, family=fam, want_ratio=True, lean=0)
            assert g["info"]["kernel_rev"] == 1
            assert_same(g, ref, want_ratio=True)


def test_parity_c5_large_code(pkg, oracle, codes):
    H, per, mi = codes.config_matrix("C5")
    B = 40
    _, syn = oracle.sample(H, per, 12345, 0, B)
    ref = oracle.batch_decode(H, per, mi, syn, nthreads=oracle.num_threads())
    g = run_gpu(pkg, H, per, mi, syn, grid_kernel=0)         # (small batches would otherwise take the grid-wide kernel)
    assert g["info"]["family"] == GLOBAL
    assert_same(g, ref)
    # harder channel: some syndromes must run many iterations
    _, syn = oracle.sample(H, 0.07, 777, 0, 16)
    ref = oracle.batch_decode(H, 0.07, mi, syn, nthreads=oracle.num_threads())
    g = run_gpu(pkg, H, 0.07, mi, syn, slots=32, grid_kernel=0)
    assert_same(g, ref)


@pytest.mark.parametrize("variant", ["exact", "minsum"])
def test_grid_kernel_small_batches_of_a_large_code(pkg, oracle, codes, variant):
    """decode! / a handful of columns on a code whose messages do not fit in one SM's shared memory (n = 100 002) run on
    the grid-wide cooperative kernel (bp_single.cuh: bp_grid_kernel): bit-identical to the oracle, to the persistent
    kernel, across repeated launches (its barrier counters must come back to zero), with posterior ratios."""
    H, per, mi = codes.config_matrix("C5")
    for B, p_ch, seed in ((1, per, 5), (3, 0.07, 6), (20, 0.05, 7)):
        _, syn = oracle.sample(H, p_ch, seed, 0, B)
        ref = oracle.batch_decode(H, p_ch, mi, syn, nthreads=oracle.num_threads(), want_ratio=(B == 3), variant=variant)
        g = run_gpu(pkg, H, p_ch, mi, syn, want_ratio=(B == 3), variant=variant, time_kernels=1)
        assert g["persistent_launches"] == 0                   # (only launches of the persistent kernels are timed)
        assert_same(g, ref, want_ratio=(B == 3))
        if B == 3:
            g0 = run_gpu(pkg, H, p_ch, mi, syn, want_ratio=True, variant=variant, time_kernels=1, grid_kernel=0)
            assert g0["persistent_launches"] == 1
            assert_same(g0, ref, want_ratio=True)
    # one decoder, many calls: single decode! (host vectors in and out) and forced iterations
    dec = pkg.BeliefPropagationDecoder(H, 0.05, 6, variant=variant)
    _, syn = oracle.sample(H, 0.05, 8, 0, 4)
    ref = oracle.batch_decode(H, 0.05, 6, syn, nthreads=oracle.num_threads(), variant=variant)
    for rep in range(2):
        for c in range(4):
            guess, conv = pkg.decode_b(dec, syn[:, c])
            assert np.array_equal(np.asarray(guess != 0, dtype=np.uint8), ref["errors"][:, c]) and bool(conv) == bool(ref["converged"][c])
    dec.close()


def test_auto_family_selection(pkg, codes):
    for name, fam in (("C2", SMEM), ("C3", SMEM), ("C4", GLOBAL), ("C1", GLOBAL)):
        H, per, mi = codes.config_matrix(name)
        dec = pkg.BeliefPropagationDecoder(H, per, mi)
        info = dec.info()
        dec.close()
        assert info["family"] == fam, (name, info)
        if fam == SMEM:
            assert info["ctas_per_sm"] == 2 and info["slots"] == 64 * info["sm_count"], info


@pytest.mark.parametrize("B", [1, 2, 31, 32, 33, 95, 1000])
@pytest.mark.parametrize("fam", [SMEM, GLOBAL])
def test_ragged_batches(pkg, oracle, codes, B, fam):
    H, _, mi = codes.config_matrix("C3")
    _, syn = oracle.sample(H, 0.06, 99, 1000, B)
    ref = oracle.batch_decode(H, 0.06, mi, syn)
    # small_batch = 0: keep these small batches on the persistent (lane-per-syndrome) kernel
    assert_same(run_gpu(pkg, H, 0.06, mi, syn, family=fam, small_batch=0), ref)
    if fam == SMEM:
        assert_same(run_gpu(pkg, H, 0.06, mi, syn, family=fam, small_batch=0, dual=1), ref)
        assert_same(run_gpu(pkg, H, 0.06, mi, syn, family=fam, small_batch=0, lean=0), ref)


@pytest.mark.parametrize("fam", [SMEM, GLOBAL])
def test_semantic_edge_cases(pkg, oracle, codes, fam):
    H, _, _ = codes.config_matrix("C3")
    s, n = H.shape
    zero = np.zeros((s, 40), dtype=np.uint8)
    g = run_gpu(pkg, H, 0.01, 0, zero, family=fam)          # max_iters = 0
    assert not g["errors"].any() and not g["converged"].any() and (g["iters"] == 0).all()
    g = run_gpu(pkg, H, 0.01, 5, zero, family=fam, small_batch=0)   # zero syndrome: converged at iteration 1
    assert not g["errors"].any() and g["converged"].all() and (g["iters"] == 1).all()
    for per in (0.5, 0.7, 0.999):                           # prior ratio >= 1, ties -> 1
        _, syn = oracle.sample(H, 0.3, 5, 0, 64)
        ref = oracle.batch_decode(H, per, 7, syn, want_ratio=True)
        assert_same(run_gpu(pkg, H, per, 7, syn, family=fam, want_ratio=True, small_batch=0), ref, want_ratio=True)
    for mi in (1, 2, 3):                                    # non-converged outputs of iteration max_iters
        _, syn = oracle.sample(H, 0.1, 6, 0, 200)
        ref = oracle.batch_decode(H, 0.1, mi, syn, want_ratio=True)
        assert_same(run_gpu(pkg, H, 0.1, mi, syn, family=fam, want_ratio=True), ref, want_ratio=True)


@pytest.mark.parametrize("fam", [SMEM, GLOBAL])
def test_irregular_and_degenerate_graphs(pkg, oracle, fam):
    rng = np.random.default_rng(5)
    # empty rows / columns, degree-1 nodes, one heavy row (local-memory degree path) and one heavy column
    s, n = 40, 90
    H = (rng.random((s, n)) < 0.06).astype(np.uint8)
    H[3, :] = 0
    H[:, 7] = 0
    H[5, :] = 0
    H[5, 10] = 1
    H[9, 20:55] = 1          # check degree 35 > 12
    H[10:30, 60] = 1         # variable degree >= 20 > 12
    H = sp.csc_matrix(H)
    for per in (0.02, 0.2):
        e = (rng.random((n, 300)) < per).astype(np.uint8)
        syn = np.asarray((H @ e) % 2).astype(np.uint8)
        syn[3, ::7] = 1      # unsatisfiable empty check -> never converges
        ref = oracle.batch_decode(H, per, 20, syn, want_ratio=True)
        g = run_gpu(pkg, H, per, 20, syn, family=fam, want_ratio=True)
        assert_same(g, ref, want_ratio=True)
        assert not ref["converged"][::7].any()


def test_tiny_codes(pkg, oracle):
    for Hd in ([[1]], [[1, 1]], [[1, 1, 0], [0, 1, 1]], [[1, 1, 0, 0, 0], [0, 1, 1, 1, 0], [0, 0, 0, 1, 1]]):
        H = sp.csc_matrix(np.array(Hd, dtype=np.uint8))
        s, n = H.shape
        syn = np.array([[(b >> i) & 1 for b in range(1 << s)] for i in range(s)], dtype=np.uint8)
        for fam in (SMEM, GLOBAL):
            ref = oracle.batch_decode(H, 0.1, 10, syn, want_ratio=True)
            assert_same(run_gpu(pkg, H, 0.1, 10, syn, family=fam, want_ratio=True, small_batch=0), ref, want_ratio=True)
        assert_same(run_gpu(pkg, H, 0.1, 10, syn, want_ratio=True), ref, want_ratio=True)       # node-parallel kernel


@pytest.mark.parametrize("fmt", ["u8", "i64", "bool"])
def test_element_formats(pkg, oracle, codes, fmt):
    H, _, mi = codes.config_matrix("C2")
    _, syn = oracle.sample(H, 0.05, 31, 0, 777)
    ref = oracle.batch_decode(H, 0.05, mi, syn)
    assert_same(run_gpu(pkg, H, 0.05, mi, syn, fmt=fmt), ref)


def test_bit_formats_and_packed_rows(pkg, oracle, codes):
    """Julia BitMatrix chunks in and out (bit c*rows + r), and the native packed rows."""
    lib = pkg._lib
    for name in ("C3", "C2"):
        H, _, mi = codes.config_matrix(name)
        s, n = H.shape
        B = 1237
        _, syn = oracle.sample(H, 0.05, 8, 0, B)
        ref = oracle.batch_decode(H, 0.05, mi, syn)
        dec = pkg.BeliefPropagationDecoder(H, 0.05, mi, chunk=320)   # several chunks, word-aligned boundaries
        # BitMatrix: column-major bit stream, 64-bit chunks
        bits_in = np.packbits(syn.T.reshape(-1), bitorder="little")
        bits_in = np.concatenate([bits_in, np.zeros((-len(bits_in)) % 8, dtype=np.uint8)])
        out = np.zeros(((B * n + 63) // 64) * 8, dtype=np.uint8)
        conv = np.zeros(B, dtype=np.uint8)
        dec.decode_raw(B, bits_in, lib.FMT_BITS, 0, out, lib.FMT_BITS, 0, conv)
        got = np.unpackbits(out, bitorder="little")[: B * n].reshape(B, n).T
        assert np.array_equal(got, ref["errors"]) and np.array_equal(conv.astype(bool), ref["converged"])
        # packed rows
        SW, NW = (s + 31) // 32, (n + 31) // 32
        pin = np.zeros((B, SW * 32), dtype=np.uint8)
        pin[:, :s] = syn.T
        pin = np.packbits(pin, axis=1, bitorder="little").view(np.uint32).copy()
        pout = np.zeros((B, NW), dtype=np.uint32)
        dec.decode_raw(B, pin, lib.FMT_PACKED32, 0, pout, lib.FMT_PACKED32, 0, conv)
        got = np.unpackbits(pout.view(np.uint8), axis=1, bitorder="little")[:, :n].T
        assert np.array_equal(got, ref["errors"])
        # mixed: Matrix{Int} in, BitMatrix out (test_bp_decoder.jl:24-26)
        out[:] = 0
        dec.decode_raw(B, np.asfortranarray(syn.astype(np.int64)), lib.FMT_I64, s, out, lib.FMT_BITS, 0, conv)
        got = np.unpackbits(out, bitorder="little")[: B * n].reshape(B, n).T
        assert np.array_equal(got, ref["errors"])
        dec.close()


def test_direct_bit_stream_output_and_overlapping_chunks(pkg, oracle, codes):
    """BitMatrix output written by the decoding kernel and the filter themselves (option direct_bits) with the chunk kernels
    overlapping or ordered, on one device and split over two shards: identical to the converted output, and to the oracle.
    n = 225 (odd) and 144: syndromes share output words with their neighbours."""
    lib = pkg._lib
    for name, per in (("C2", 0.02), ("C3", 0.04)):
        H, _, mi = codes.config_matrix(name)
        s, n = H.shape
        B = 50_001
        _, syn = oracle.sample(H, per, 77, 0, B)
        bits_in = np.packbits(syn.T.reshape(-1), bitorder="little")
        bits_in = np.concatenate([bits_in, np.zeros((-len(bits_in)) % 8, dtype=np.uint8)])
        outs = []
        for direct, overlap, devices in ((1, 2, [0]), (0, 0, [0]), (1, 0, [0]), (1, 2, [0, 0]), (0, 2, [0, 0])):
            dec = pkg.BeliefPropagationDecoder(H, per, mi, devices=devices, direct_bits=direct, overlap_chunks=overlap, chunk=9984)
            out = np.full(((B * n + 63) // 64) * 8, 0xFF, dtype=np.uint8)        # stale contents must not leak through
            conv = np.zeros(B, dtype=np.uint8)
            iters = np.zeros(B, dtype=np.int32)
            dec.decode_raw(B, bits_in, lib.FMT_BITS, 0, out, lib.FMT_BITS, 0, conv, iters=iters)
            outs.append((np.unpackbits(out, bitorder="little")[: B * n].copy(), conv.copy(), iters.copy()))
            dec.close()
        for o in outs[1:]:
            assert all(np.array_equal(a, b) for a, b in zip(outs[0], o)), name
        ref = oracle.batch_decode(H, per, mi, syn[:, :4000], nthreads=oracle.num_threads())
        got = outs[0][0].reshape(B, n).T[:, :4000]
        assert np.array_equal(got, ref["errors"]) and np.array_equal(outs[0][1][:4000].astype(bool), ref["converged"])
        assert np.array_equal(outs[0][2][:4000], ref["iters"])


def test_decode_b_single_syndrome_api(pkg, oracle, codes):
    """decode!(decoder, syndrome): aliased Float64 scratch.err, converged flag, log_probabs."""
    H, per, mi = codes.config_matrix("C1")
    errs, syn = oracle.sample(H, per, 2024, 0, 5)
    ref = oracle.batch_decode(H, per, mi, syn, want_ratio=True)
    dec = pkg.BeliefPropagationDecoder(H, per, mi)
    for b in range(5):
        for s_in in (syn[:, b], syn[:, b].astype(np.int64), syn[:, b].astype(bool)):
            guess, success = pkg.decode_b(dec, s_in)
            assert guess is dec.scratch.err and guess.dtype == np.float64
            assert np.array_equal(guess.astype(np.uint8), ref["errors"][:, b]) and success == bool(ref["converged"][b])
            with np.errstate(all="ignore"):
                np.testing.assert_array_equal(dec.scratch.log_probabs, np.log(1.0 / ref["ratio"][:, b]))
    assert pkg.reset_b(dec) is dec and not dec.scratch.err.any()
    # 3-argument batchdecode! allocates success (abstract_decoder.jl:44-48); column-count asserts
    errors = np.zeros((H.shape[1], 5), dtype=np.bool_, order="F")
    out, success = pkg.batchdecode_b(dec, syn.astype(np.int64), errors)
    assert out is errors and success.dtype == np.bool_ and np.array_equal(errors.astype(np.uint8), ref["errors"])
    with pytest.raises(AssertionError):
        pkg.batchdecode_b(dec, syn, np.zeros((H.shape[1], 4), dtype=np.uint8, order="F"))
    with pytest.raises(AssertionError):
        pkg.batchdecode_b(dec, syn, errors, np.zeros(3, dtype=np.bool_))
    dec.close()


def test_reference_thresholds_on_gpu(pkg, oracle, codes):
    """test/test_bp_decoder.jl:46-51 against the GPU path."""
    H = codes.gallager(1000, 10, 9, seed=7)
    errs, syn = oracle.sample(H, 0.01, 4242, 0, 1100)
    g = run_gpu(pkg, H, 0.01, 100, syn)
    exact = (g["errors"] == errs).all(axis=0)
    assert exact[0]
    assert 1 - exact[:100].mean() < 0.005
    assert 1 - exact[100:].mean() < 0.001


def test_device_sampler_matches_oracle_and_full_size_properties(pkg, oracle, codes):
    """Device-resident sample -> decode -> score on the gross code at 2M syndromes: the sampler
    equals the oracle's Philox stream, every converged output reproduces its syndrome, counters
    agree with per-syndrome outputs, and results do not depend on how the batch is split."""
    H, _, mi = codes.config_matrix("C3")
    s, n = H.shape
    per = 0.03
    dec = pkg.BeliefPropagationDecoder(H, per, mi)
    info = dec.info()
    SW, NW = info["syn_words"], info["err_words"]
    B = 2_000_000
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    st = stream.cuda_stream
    truth = torch.empty((B, NW), dtype=torch.int32, device=dev)
    synw = torch.empty((B, SW), dtype=torch.int32, device=dev)
    errw = torch.empty((B, NW), dtype=torch.int32, device=dev)
    conv = torch.empty(B, dtype=torch.uint8, device=dev)
    iters = torch.empty(B, dtype=torch.int32, device=dev)
    ctr = torch.zeros(4, dtype=torch.int64, device=dev)
    score = torch.zeros(2, dtype=torch.int64, device=dev)
    dec.sample_device(B, 0, 12345, per, truth.data_ptr(), synw.data_ptr(), stream=st)
    dec.decode_device(B, synw.data_ptr(), errw.data_ptr(), conv.data_ptr(), iters.data_ptr(), None, ctr.data_ptr(), stream=st)
    dec.score_device(B, truth.data_ptr(), errw.data_ptr(), synw.data_ptr(), score.data_ptr(), stream=st)
    torch.cuda.synchronize()
    # sampler == oracle stream on a prefix and in the middle (sharding independence)
    for first, cnt in ((0, 500), (1_234_567, 300)):
        e_ref, s_ref = oracle.sample(H, per, 12345, first, cnt)
        e_gpu = np.unpackbits(truth[first:first + cnt].cpu().numpy().view(np.uint8), axis=1, bitorder="little")[:, :n].T
        s_gpu = np.unpackbits(synw[first:first + cnt].cpu().numpy().view(np.uint8), axis=1, bitorder="little")[:, :s].T
        assert np.array_equal(e_gpu, e_ref) and np.array_equal(s_gpu, s_ref)
        ref = oracle.batch_decode(H, per, mi, s_ref)
        d_gpu = np.unpackbits(errw[first:first + cnt].cpu().numpy().view(np.uint8), axis=1, bitorder="little")[:, :n].T
        assert np.array_equal(d_gpu, ref["errors"])
        assert np.array_equal(conv[first:first + cnt].cpu().numpy().astype(bool), ref["converged"])
        assert np.array_equal(iters[first:first + cnt].cpu().numpy(), ref["iters"])
    c = ctr.cpu().numpy()
    assert c[0] == B and c[1] == int(conv.sum().item()) and c[2] == int(iters.sum(dtype=torch.int64).item())
    sc = score.cpu().numpy()
    assert sc[1] == c[1]                     # converged <=> H*e == syndrome, over the whole batch
    assert sc[0] <= sc[1] and sc[0] > 0.5 * B
    assert int(iters.min().item()) >= 1 and int(iters.max().item()) <= mi
    assert bool(((iters == mi) | (conv == 1)).all().item())
    # a different split of the same batch gives the same bits
    errw2 = torch.empty_like(errw[:700_000])
    conv2 = torch.empty_like(conv[:700_000])
    dec.decode_device(700_000, synw[300_000:].data_ptr(), errw2.data_ptr(), conv2.data_ptr(), None, None, None, stream=st)
    torch.cuda.synchronize()
    assert torch.equal(errw2, errw[300_000:1_000_000]) and torch.equal(conv2, conv[300_000:1_000_000])
    assert dec.launch_count() > 0
    dec.close()


def test_fast_division_is_ieee(pkg):
    """The kernels' branch-free reciprocal / quotient sequences equal __drcp_rn / __ddiv_rn bit for
    bit on their operand envelopes (2^31 pseudo-random operands each, incl. values next to the
    envelope edges)."""
    import ctypes
    lib = pkg._lib.load()
    for mode in (0, 1):
        bad = (ctypes.c_uint64 * 4)(1, 1, 1, 1)
        pkg._lib.check(lib.ldpcb200_selftest_division(0, mode, 1 << 31, 2024 + mode, bad))
        assert list(bad)[:3] == [0, 0, 0], (mode, list(bad), np.array([bad[3]], dtype=np.uint64).view(np.float64))


def test_forced_iterations_mode_runs_max_iters(pkg, oracle, codes):
    H, _, mi = codes.config_matrix("C3")
    _, syn = oracle.sample(H, 0.01, 3, 0, 500)
    g = run_gpu(pkg, H, 0.01, mi, syn, early_stop=0)
    assert (g["iters"] == mi).all()


GOLDEN = __import__("os").path.join(__import__("os").path.dirname(__file__), "golden")


@pytest.mark.parametrize("fixture", sorted(f for f in __import__("os").listdir(GOLDEN) if f.endswith(".npz") and not f.endswith(".osd.npz")))
def test_golden_fixtures_on_gpu(pkg, fixture):
    """The committed fixtures (tests/golden/make_golden.py) decoded by the CUDA path."""
    z = np.load(__import__("os").path.join(GOLDEN, fixture))
    H = sp.csc_matrix((np.ones(len(z["rowval"]), dtype=np.uint8), z["rowval"], z["colptr"]), shape=tuple(z["shape"]))
    g = run_gpu(pkg, H, float(z["per"]), int(z["max_iters"]), z["syndromes"], want_ratio=True)
    assert np.array_equal(g["errors"], z["errors"])
    assert np.array_equal(g["converged"], z["converged"])
    assert np.array_equal(g["iters"], z["iters"])
    assert np.array_equal(g["ratio"].view(np.uint64), z["ratio_bits"])


def _random_code(rng, s, n, col_deg):
    rows = np.concatenate([rng.choice(s, size=col_deg, replace=False) for _ in range(n)])
    cols = np.repeat(np.arange(n), col_deg)
    return sp.csc_matrix((np.ones(len(rows), dtype=np.uint8), (rows, cols)), shape=(s, n))


def test_decision_fields_in_memory(pkg, oracle):
    """Codes where a warp owns more than 64 variables keep their decisions as bit fields in
    shared memory (modes 0/1) or in HBM (mode 1 with many variables, mode 2)."""
    rng = np.random.default_rng(11)
    cases = [
        # (H, warps option, expected family)   n / warps > 64 in every case
        (_random_code(rng, 60, 400, 1), 4, SMEM),        # mode 0, fields in shared memory
        (_random_code(rng, 300, 2000, 2), 8, GLOBAL),    # mode 1, fields in shared memory
        (_random_code(rng, 3000, 9000, 2), 12, GLOBAL),  # mode 1, fields in HBM
    ]
    for H, warps, fam in cases:
        s, n = H.shape
        e = (rng.random((n, 150)) < 0.01).astype(np.uint8)
        syn = np.asarray((H @ e) % 2).astype(np.uint8)
        ref = oracle.batch_decode(H, 0.01, 12, syn, want_ratio=True, nthreads=oracle.num_threads())
        g = run_gpu(pkg, H, 0.01, 12, syn, want_ratio=True, warps=warps)
        assert g["info"]["family"] == fam and n > 64 * (g["info"]["threads_per_cta"] // 32), g["info"]
        assert_same(g, ref, want_ratio=True)


def test_staging_depths_agree(pkg, oracle, codes):
    """HBM modes: the cp.async ring (prefetch 1..3) and the direct path give the same bits."""
    H, _, mi = codes.config_matrix("C4")
    _, syn = oracle.sample(H, 0.04, 21, 0, 300)
    ref = oracle.batch_decode(H, 0.04, mi, syn, nthreads=oracle.num_threads())
    for pf in (0, 1, 2, 3):
        assert_same(run_gpu(pkg, H, 0.04, mi, syn, prefetch=pf), ref)


def shard_device_sets():
    """Device lists for the in-library sharding tests.  With one visible GPU the same device is listed
    several times: the threaded split, the shard-boundary alignment of the bit formats and the counter
    summation run exactly as they do over distinct devices (each entry has its own streams and buffers)."""
    nd = torch.cuda.device_count()
    sets = [[0, 0], [0, 0, 0]]
    if nd >= 2:
        sets.append(list(range(min(nd, 8))))
    return sets


@pytest.mark.parametrize("fmt", ["u8", "bits", "packed", "i64"])
def test_in_library_sharding_over_devices(pkg, oracle, codes, fmt):
    """devices = [d0, d1, ...]: the library splits the batch into contiguous column ranges (boundaries
    multiples of 32) and sums the counters; results equal the single-device ones
    (batchdecode! semantics, belief_propagation.jl:220-231, for every boundary format)."""
    H, _, mi = codes.config_matrix("C3")
    s, n = H.shape
    B = 100_003
    _, syn = oracle.sample(H, 0.05, 77, 0, B)
    ref = oracle.batch_decode(H, 0.05, mi, syn, nthreads=oracle.num_threads())
    lib = pkg._lib
    for devs in shard_device_sets():
        dec = pkg.BeliefPropagationDecoder(H, 0.05, mi, devices=devs)
        info = dec.info()
        assert info["ndev"] == len(devs)
        iters = np.zeros(B, dtype=np.int32)
        if fmt in ("u8", "i64"):
            dt = np.uint8 if fmt == "u8" else np.int64
            errors = np.zeros((n, B), dtype=dt, order="F")
            _, success = pkg.batchdecode_b(dec, np.asfortranarray(syn.astype(dt)), errors, iters=iters)
            got = errors.astype(np.uint8)
        elif fmt == "bits":
            sin = np.packbits(syn.T.reshape(-1), bitorder="little")           # bit c*s + r of the stream
            sin = np.concatenate([sin, np.zeros((-len(sin)) % 8, np.uint8)])
            eout = np.zeros((B * n + 63) // 64 * 8, dtype=np.uint8)
            conv = np.zeros(B, dtype=np.uint8)
            dec.last_counters = dec.decode_raw(B, sin, lib.FMT_BITS, 0, eout, lib.FMT_BITS, 0, conv, iters)
            got = np.unpackbits(eout, bitorder="little")[:B * n].reshape(B, n).T
            success = conv.astype(bool)
        else:
            SW, NW = info["syn_words"], info["err_words"]
            pad = np.zeros((SW * 32, B), np.uint8)
            pad[:s] = syn
            sin = np.ascontiguousarray(np.packbits(np.ascontiguousarray(pad.T), axis=1, bitorder="little")).view(np.uint32).reshape(B, SW)
            eout = np.zeros((B, NW), dtype=np.uint32)
            conv = np.zeros(B, dtype=np.uint8)
            dec.last_counters = dec.decode_raw(B, np.ascontiguousarray(sin), lib.FMT_PACKED32, SW, eout, lib.FMT_PACKED32, NW, conv, iters)
            got = np.unpackbits(eout.view(np.uint8).reshape(B, NW * 4), axis=1, bitorder="little")[:, :n].T
            success = conv.astype(bool)
        g = dict(errors=got, converged=success, iters=iters, counters=dec.last_counters)
        dec.close()
        assert_same(g, ref)


def run_gpu_variant(pkg, H, per, max_iters, syn, variant, **opts):
    dec = pkg.BeliefPropagationDecoder(H, per, max_iters, variant=variant, **opts)
    n, B = H.shape[1], syn.shape[1]
    errors = np.zeros((n, B), dtype=np.uint8, order="F")
    iters = np.zeros(B, dtype=np.int32)
    llr = np.zeros((n, B), dtype=np.float64, order="F")
    _, success = pkg.batchdecode_b(dec, np.asfortranarray(syn), errors, iters=iters, posterior_ratio=llr)
    out = dict(errors=errors, converged=success, iters=iters, ratio=llr, info=dec.info(), counters=dec.last_counters.copy())
    dec.close()
    return out


@pytest.mark.parametrize("name,per,B", [("C3", 0.03, 3000), ("C3", 0.1, 1000), ("C2", 0.02, 2000), ("C4", 0.03, 400), ("C1", 0.03, 100)])
def test_minsum_variant_matches_its_definition(pkg, oracle, codes, name, per, B):
    """LDPCB200_VARIANT_MINSUM has no reference equivalent; the CUDA kernels must reproduce the
    CPU checker's min-sum definition (oracle/bp_oracle.c: decode_edge_minsum) bit for bit."""
    H, _, mi = codes.config_matrix(name)
    _, syn = oracle.sample(H, per, 4321, 0, B)
    ref = oracle.batch_decode(H, per, mi, syn, nthreads=oracle.num_threads(), variant="minsum", want_ratio=True)
    g = run_gpu_variant(pkg, H, per, mi, syn, "minsum")
    assert_same(g, ref, want_ratio=True)


def test_minsum_large_code_and_scale_option(pkg, oracle, codes):
    H, per, mi = codes.config_matrix("C5")
    _, syn = oracle.sample(H, per, 99, 0, 24)
    ref = oracle.batch_decode(H, per, mi, syn, nthreads=oracle.num_threads(), variant="minsum")
    g = run_gpu_variant(pkg, H, per, mi, syn, "minsum", grid_kernel=0)
    assert g["info"]["kernel_mode"] == 2
    assert np.array_equal(g["errors"], ref["errors"]) and np.array_equal(g["iters"], ref["iters"])
    # plain (unnormalised) min-sum through the scale option
    H, _, mi = codes.config_matrix("C3")
    _, syn = oracle.sample(H, 0.03, 98, 0, 500)
    ref = oracle.batch_decode(H, 0.03, mi, syn, variant="minsum", minsum_scale=1.0)
    g = run_gpu_variant(pkg, H, 0.03, mi, syn, "minsum", minsum_scale_permille=1000)
    assert np.array_equal(g["errors"], ref["errors"]) and np.array_equal(g["iters"], ref["iters"])


def test_minsum_quality_is_close_to_sum_product(pkg, oracle, codes):
    """Normalised min-sum (0.875) on the gross code: logical quality within a point of sum-product."""
    H, _, mi = codes.config_matrix("C3")
    errs, syn = oracle.sample(H, 0.03, 5, 0, 20000)
    ms = run_gpu_variant(pkg, H, 0.03, mi, syn, "minsum")
    sp = run_gpu_variant(pkg, H, 0.03, mi, syn, "exact")
    ok_ms = (ms["errors"] == errs).all(axis=0).mean()
    ok_sp = (sp["errors"] == errs).all(axis=0).mean()
    assert ok_ms > ok_sp - 0.01, (ok_ms, ok_sp)
    assert ms["converged"].mean() > 0.97


# ---------------------------------------------------------------------------------------------
# BP + OSD-0 (SURVEY 8(f) rank 1; reference belief_propagation_osd.jl:49-125) -- GPU Gauss-Jordan
# without row swaps against the literal restatement (row swaps, early break, back substitution)
def run_gpu_bposd(pkg, H, per, max_iters, syn, fmt=np.uint8, **opts):
    dec = pkg.BeliefPropagationOSDDecoder(H, per, max_iters, **opts)
    n, B = H.shape[1], syn.shape[1]
    errors = np.full((n, B), 1, dtype=fmt, order="F")
    _, success = pkg.batchdecode_b(dec, np.asfortranarray(syn.astype(fmt)), errors)
    out = dict(errors=errors.astype(np.uint8), converged=success.copy(), counters=dec.last_counters.copy(),
               stats=dec.last_osd_stats.copy())
    dec.close()
    return out


@pytest.mark.parametrize("name,per,B", [("C3", 0.06, 3000), ("C3", 0.12, 1500), ("C2", 0.05, 2000), ("C4", 0.04, 300),
                                        ("C4", 0.08, 150), ("C1", 0.09, 60)])
def test_bposd_matches_restated_reference(pkg, oracle, codes, name, per, B):
    H, _, mi = codes.config_matrix(name)
    _, syn = oracle.sample(H, per, 4242, 0, B)
    ref = oracle.bposd_decode(H, per, mi, syn, nthreads=oracle.num_threads())
    g = run_gpu_bposd(pkg, H, per, mi, syn)
    nonconv = int((~ref["converged"]).sum())
    assert nonconv > 0, "case does not exercise OSD"
    assert np.array_equal(g["converged"], ref["converged"])
    bad = np.nonzero((g["errors"] != ref["errors"]).any(axis=0))[0]
    assert bad.size == 0, "OSD results differ on syndromes %s (%d unconverged of %d)" % (bad[:10], nonconv, B)
    assert g["stats"][0] == nonconv
    assert g["stats"][1] == int(ref["pivots"].sum())
    # OSD-0 always returns an error that reproduces the syndrome when the syndrome is in the column space
    Hd = np.asarray(sp.csc_matrix(H).todense()).astype(np.int64)
    assert np.array_equal((Hd @ g["errors"].astype(np.int64)) % 2, syn.astype(np.int64))


def test_bposd_edge_cases(pkg, oracle, codes):
    H, _, _ = codes.config_matrix("C3")
    _, syn = oracle.sample(H, 0.08, 99, 0, 257)
    # max_iters = 0: BP returns zeros / not converged, log_probabs = 0 -> all keys tie -> index order
    for mi in (0, 1, 3):
        ref = oracle.bposd_decode(H, 0.08, mi, syn, nthreads=2)
        g = run_gpu_bposd(pkg, H, 0.08, mi, syn)
        assert np.array_equal(g["converged"], ref["converged"])
        assert np.array_equal(g["errors"], ref["errors"])
    # int64 matrices (Matrix{Int}) and the single-syndrome decode!
    ref = oracle.bposd_decode(H, 0.08, 8, syn, nthreads=2)
    g = run_gpu_bposd(pkg, H, 0.08, 8, syn, fmt=np.int64)
    assert np.array_equal(g["errors"], ref["errors"])
    dec = pkg.BeliefPropagationOSDDecoder(H, 0.08, 8)
    for b in (0, 5, 100):
        e, conv = pkg.decode_b(dec, syn[:, b])
        assert e.dtype == np.bool_ and np.array_equal(e.astype(np.uint8), ref["errors"][:, b]) and conv == ref["converged"][b]
    assert pkg.reset_b(dec) is dec
    dec.close()
    # a syndrome outside the column space (rank-deficient H with a redundant check violated): the reference
    # runs out of columns and returns whatever the elimination solved; same here
    Hs = np.asarray(sp.csc_matrix(codes.surface_x(5)).todense()).astype(np.uint8)
    Hr = np.vstack([Hs, Hs[0:1] ^ Hs[1:2]])            # last row = row0 + row1
    rng = np.random.default_rng(5)
    synr = (rng.random((Hr.shape[0], 64)) < 0.3).astype(np.uint8)
    ref = oracle.bposd_decode(Hr, 0.05, 6, synr, nthreads=2)
    g = run_gpu_bposd(pkg, Hr, 0.05, 6, synr)
    assert np.array_equal(g["errors"], ref["errors"]) and np.array_equal(g["converged"], ref["converged"])
    # min-sum posteriors are LLRs: OSD is refused, loudly
    decm = pkg.BeliefPropagationDecoder(H, 0.05, 8, variant="minsum")
    with pytest.raises(pkg._lib.LibraryError):
        decm.bposd_raw(1, np.zeros((72, 1), np.uint8, order="F"), pkg._lib.FMT_U8, 72, np.zeros((144, 1), np.uint8, order="F"),
                       pkg._lib.FMT_U8, 144, np.zeros(1, np.uint8))
    decm.close()


def test_bposd_large_batch_properties_and_host_device_agreement(pkg, oracle, codes):
    """200k gross-code syndromes at per = 0.08 (a third unconverged): the chunked host entry point (two staging sets,
    two streams) and the device-resident BP -> OSD-0 pipeline give the same bits; converged flags are BP's; every
    output reproduces its syndrome; converged rows are BP's own decisions; a sample equals the restated reference."""
    H, _, mi = codes.config_matrix("C3")
    s, n = H.shape
    per, B = 0.08, 200_000
    dec = pkg.BeliefPropagationOSDDecoder(H, per, mi, chunk=32768)
    bp = dec.bp_decoder
    info = bp.info()
    SW, NW = info["syn_words"], info["err_words"]
    dev = torch.device("cuda:0")
    truth = torch.empty((B, NW), dtype=torch.int32, device=dev)
    synw = torch.empty((B, SW), dtype=torch.int32, device=dev)
    bp.sample_device(B, 0, 777, per, truth.data_ptr(), synw.data_ptr())
    torch.cuda.synchronize()
    # host entry point, native packed rows
    syn_h = synw.cpu().numpy().view(np.uint32)
    err_h = np.zeros((B, NW), dtype=np.uint32)
    conv_h = np.zeros(B, dtype=np.uint8)
    ctr, stats = bp.bposd_raw(B, syn_h, pkg._lib.FMT_PACKED32, SW, err_h, pkg._lib.FMT_PACKED32, NW, conv_h)
    # device pipeline
    errw = torch.empty((B, NW), dtype=torch.int32, device=dev)
    bperr = torch.empty((B, NW), dtype=torch.int32, device=dev)
    conv = torch.empty(B, dtype=torch.uint8, device=dev)
    ratio = torch.empty((B, n), dtype=torch.float64, device=dev)
    st8 = torch.zeros(8, dtype=torch.int64, device=dev)
    score = torch.zeros(2, dtype=torch.int64, device=dev)
    bp.set_option("ratio_last_only", 1)
    bp.decode_device(B, synw.data_ptr(), errw.data_ptr(), conv.data_ptr(), None, ratio.data_ptr(), None)
    torch.cuda.synchronize()
    bperr.copy_(errw)
    bp.osd0_device(B, synw.data_ptr(), errw.data_ptr(), conv.data_ptr(), ratio.data_ptr(), st8.data_ptr())
    bp.score_device(B, truth.data_ptr(), errw.data_ptr(), synw.data_ptr(), score.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(errw.cpu().numpy().view(np.uint32), err_h)
    assert np.array_equal(conv.cpu().numpy(), conv_h)
    nonconv = int((conv == 0).sum().item())
    assert 0.1 * B < nonconv < 0.9 * B
    assert stats[0] == nonconv == int(st8[0].item()) and stats[1] == int(st8[1].item())
    assert ctr[0] == B and ctr[1] == B - nonconv
    assert int(score[1].item()) == B                       # H * e == syndrome for every syndrome after OSD-0
    cm = conv.bool()
    assert torch.equal(errw[cm], bperr[cm])                # converged: BP's own decision (:72-74)
    assert not torch.equal(errw[~cm], bperr[~cm])
    for first, cnt in ((0, 300), (150_000, 200)):
        _, s_ref = oracle.sample(H, per, 777, first, cnt)
        ref = oracle.bposd_decode(H, per, mi, s_ref, nthreads=oracle.num_threads())
        got = np.unpackbits(err_h[first:first + cnt].view(np.uint8), axis=1, bitorder="little")[:, :n].T
        assert np.array_equal(got, ref["errors"])
        assert np.array_equal(conv_h[first:first + cnt].astype(bool), ref["converged"])
    dec.close()


# ---------------------------------------------------------------------------------------------
# node-parallel small-batch kernel (bp_single.cuh): the low-latency path of decode! and of batches up to one
# CTA per SM; bit-identical to the oracle like the persistent kernel
@pytest.mark.parametrize("name,per,B", [("C1", 0.01, 5), ("C1", 0.04, 64), ("C3", 0.06, 148), ("C3", 0.12, 33),
                                        ("C2", 0.05, 100), ("C4", 0.03, 40), ("C4", 0.08, 7)])
def test_small_batch_kernel_parity(pkg, oracle, codes, name, per, B):
    H, _, mi = codes.config_matrix(name)
    _, syn = oracle.sample(H, per, 808, 0, B)
    ref = oracle.batch_decode(H, per, mi, syn, nthreads=oracle.num_threads(), want_ratio=True)
    g = run_gpu(pkg, H, per, mi, syn, want_ratio=True, small_batch=1000)
    assert_same(g, ref, want_ratio=True)
    g0 = run_gpu(pkg, H, per, mi, syn, want_ratio=True, small_batch=0)        # persistent kernel, same bits
    assert_same(g0, ref, want_ratio=True)


def test_small_batch_kernel_edge_cases(pkg, oracle, codes):
    H, _, _ = codes.config_matrix("C3")
    s, n = H.shape
    zero = np.zeros((s, 9), dtype=np.uint8)
    g = run_gpu(pkg, H, 0.01, 5, zero)                       # zero syndrome: converged at iteration 1
    assert not g["errors"].any() and g["converged"].all() and (g["iters"] == 1).all()
    for per in (0.5, 0.7, 0.999):                            # prior ratio >= 1, ties -> 1
        _, syn = oracle.sample(H, 0.3, 5, 0, 64)
        ref = oracle.batch_decode(H, per, 7, syn, want_ratio=True)
        assert_same(run_gpu(pkg, H, per, 7, syn, want_ratio=True), ref, want_ratio=True)
    for mi in (1, 2, 3):                                     # non-converged outputs of iteration max_iters
        _, syn = oracle.sample(H, 0.1, 6, 0, 100)
        ref = oracle.batch_decode(H, 0.1, mi, syn, want_ratio=True)
        assert_same(run_gpu(pkg, H, 0.1, mi, syn, want_ratio=True), ref, want_ratio=True)
    # forced iterations (early_stop = 0) and irregular graphs with empty rows/columns
    _, syn = oracle.sample(H, 0.05, 7, 0, 50)
    g = run_gpu(pkg, H, 0.05, 6, syn, early_stop=0)
    assert (g["iters"] == 6).all()
    rng = np.random.default_rng(9)
    Hd = (rng.random((30, 70)) < 0.08).astype(np.uint8)
    Hd[3, :] = 0
    Hd[:, 7] = 0
    Hi = sp.csc_matrix(Hd)
    e = (rng.random((70, 60)) < 0.05).astype(np.uint8)
    syn = np.asarray((Hi @ e) % 2).astype(np.uint8)
    syn[3, ::5] = 1
    ref = oracle.batch_decode(Hi, 0.05, 15, syn, want_ratio=True)
    assert_same(run_gpu(pkg, Hi, 0.05, 15, syn, want_ratio=True), ref, want_ratio=True)


def test_grid_kernel_forced_on_small_and_irregular_graphs(pkg, oracle, codes):
    """The grid-wide kernel forced (grid_kernel = 2) where the one-CTA kernel would normally run: configs C1-C4, semantic
    edge cases (max_iters 1..3, prior ratio >= 1, zero syndrome, forced iterations) and a graph with empty rows / columns
    and syndromes outside the column space, posterior ratios included -- bit for bit against the oracle."""
    for name, per, B in (("C3", 0.05, 40), ("C2", 0.03, 33), ("C4", 0.03, 12), ("C1", 0.03, 9)):
        H, _, mi = codes.config_matrix(name)
        _, syn = oracle.sample(H, per, 31, 0, B)
        ref = oracle.batch_decode(H, per, mi, syn, want_ratio=True)
        g = run_gpu(pkg, H, per, mi, syn, want_ratio=True, grid_kernel=2, time_kernels=1)
        assert g["persistent_launches"] == 0
        assert_same(g, ref, want_ratio=True)
    H, _, _ = codes.config_matrix("C3")
    zero = np.zeros((H.shape[0], 5), dtype=np.uint8)
    g = run_gpu(pkg, H, 0.01, 5, zero, grid_kernel=2)
    assert not g["errors"].any() and g["converged"].all() and (g["iters"] == 1).all()
    for per, mi in ((0.5, 7), (0.999, 4), (0.1, 1), (0.1, 2), (0.1, 3)):
        _, syn = oracle.sample(H, 0.2, 5, 0, 48)
        ref = oracle.batch_decode(H, per, mi, syn, want_ratio=True)
        assert_same(run_gpu(pkg, H, per, mi, syn, want_ratio=True, grid_kernel=2), ref, want_ratio=True)
    _, syn = oracle.sample(H, 0.05, 7, 0, 20)
    g = run_gpu(pkg, H, 0.05, 6, syn, early_stop=0, grid_kernel=2)
    assert (g["iters"] == 6).all()
    rng = np.random.default_rng(19)
    Hd = (rng.random((40, 90)) < 0.07).astype(np.uint8)
    Hd[5, :] = 0
    Hd[:, 11] = 0
    for r in range(Hd.shape[0]):                             # keep every degree within the register paths (<= 12)
        ones = np.nonzero(Hd[r])[0]
        Hd[r, ones[12:]] = 0
    assert Hd.sum(axis=0).max() <= 12
    Hi = sp.csc_matrix(Hd)
    e = (rng.random((90, 30)) < 0.05).astype(np.uint8)
    syn = np.asarray((Hi @ e) % 2).astype(np.uint8)
    syn[5, ::4] = 1
    for variant in ("exact", "minsum"):
        ref = oracle.batch_decode(Hi, 0.05, 15, syn, want_ratio=True, variant=variant)
        assert_same(run_gpu(pkg, Hi, 0.05, 15, syn, want_ratio=True, grid_kernel=2, variant=variant), ref, want_ratio=True)


@pytest.mark.parametrize("B", [1, 7, 64, 148])
def test_small_batch_host_path_all_formats(pkg, oracle, codes, B):
    """Small host batches go through one staging block each way (decode_host_tiny): every boundary format,
    strided matrices, iteration counts, posterior ratios and counters."""
    lib = pkg._lib
    H, _, mi = codes.config_matrix("C2")
    s, n = H.shape
    _, syn = oracle.sample(H, 0.04, 21, 0, B)
    ref = oracle.batch_decode(H, 0.04, mi, syn, want_ratio=True)
    dec = pkg.BeliefPropagationDecoder(H, 0.04, mi)
    conv = np.zeros(B, dtype=np.uint8)
    iters = np.zeros(B, dtype=np.int32)
    ratio = np.zeros((n, B), dtype=np.float64, order="F")
    # element formats, leading dimensions larger than the row count (views into bigger Julia matrices)
    for dt, fmt in ((np.uint8, lib.FMT_U8), (np.int64, lib.FMT_I64)):
        big_in = np.full((s + 5, B), 3, dtype=dt, order="F")
        big_in[:s] = syn
        for odt, ofmt in ((np.uint8, lib.FMT_U8), (np.int64, lib.FMT_I64), (np.float64, lib.FMT_F64)):
            big_out = np.full((n + 3, B), 9, dtype=odt, order="F")
            ctr = dec.decode_raw(B, big_in, fmt, s + 5, big_out, ofmt, n + 3, conv, iters, ratio)
            assert np.array_equal(big_out[:n].astype(np.uint8), ref["errors"]) and (big_out[n:] == 9).all()
            assert np.array_equal(conv.astype(bool), ref["converged"]) and np.array_equal(iters, ref["iters"])
            assert np.array_equal(ratio.view(np.uint64), ref["ratio"].view(np.uint64))
            assert ctr[0] == B and ctr[1] == int(ref["converged"].sum()) and ctr[2] == int(ref["iters"].sum())
    # BitMatrix stream and packed rows
    bits_in = np.packbits(syn.T.reshape(-1), bitorder="little")
    bits_in = np.concatenate([bits_in, np.zeros((-len(bits_in)) % 8, dtype=np.uint8)])
    out = np.zeros(((B * n + 63) // 64) * 8, dtype=np.uint8)
    dec.decode_raw(B, bits_in, lib.FMT_BITS, 0, out, lib.FMT_BITS, 0, conv)
    assert np.array_equal(np.unpackbits(out, bitorder="little")[: B * n].reshape(B, n).T, ref["errors"])
    SW, NW = (s + 31) // 32, (n + 31) // 32
    pin = np.zeros((B, SW * 32), dtype=np.uint8)
    pin[:, :s] = syn.T
    pin = np.packbits(pin, axis=1, bitorder="little").view(np.uint32).copy()
    pout = np.zeros((B, NW), dtype=np.uint32)
    dec.decode_raw(B, pin, lib.FMT_PACKED32, 0, pout, lib.FMT_PACKED32, 0, conv)
    assert np.array_equal(np.unpackbits(pout.view(np.uint8), axis=1, bitorder="little")[:, :n].T, ref["errors"])
    # the same through the chunked pipeline (small_batch = 0)
    dec.set_option("small_batch", 0)
    out2 = np.zeros((n, B), dtype=np.uint8, order="F")
    dec.decode_raw(B, np.asfortranarray(syn), lib.FMT_U8, s, out2, lib.FMT_U8, n, conv)
    assert np.array_equal(out2, ref["errors"])
    dec.close()
    # max_iters = 0 and the min-sum variant (persistent kernel behind the same host path)
    d0 = pkg.BeliefPropagationDecoder(H, 0.04, 0)
    e0 = np.ones((n, B), dtype=np.uint8, order="F")
    d0.decode_raw(B, np.asfortranarray(syn), lib.FMT_U8, s, e0, lib.FMT_U8, n, conv)
    assert not e0.any() and not conv.any()
    d0.close()
    refm = oracle.batch_decode(H, 0.04, mi, syn, variant="minsum")
    dm = pkg.BeliefPropagationDecoder(H, 0.04, mi, variant="minsum")
    em = np.zeros((n, B), dtype=np.uint8, order="F")
    dm.decode_raw(B, np.asfortranarray(syn), lib.FMT_U8, s, em, lib.FMT_U8, n, conv)
    assert np.array_equal(em, refm["errors"]) and np.array_equal(conv.astype(bool), refm["converged"])
    dm.close()


def test_bposd_in_library_sharding_over_devices(pkg, oracle, codes):
    H, _, mi = codes.config_matrix("C3")
    B = 5000
    _, syn = oracle.sample(H, 0.08, 1234, 0, B)
    ref = oracle.bposd_decode(H, 0.08, mi, syn, nthreads=oracle.num_threads())
    for devs in shard_device_sets():
        g = run_gpu_bposd(pkg, H, 0.08, mi, syn, devices=devs)
        assert np.array_equal(g["errors"], ref["errors"]) and np.array_equal(g["converged"], ref["converged"])
        assert g["stats"][0] == int((~ref["converged"]).sum()) and g["counters"][0] == B


def test_two_live_decoders_with_different_shared_memory_sizes(pkg, oracle, codes):
    """Two handles that share a kernel instantiation but need different dynamic shared-memory sizes (surface-15 and
    the gross code, both family SMEM, 256-thread shape) decode alternately: the limit is an attribute of the
    instantiation, not of a handle, so it must be set per launch."""
    Ha, _, mi = codes.config_matrix("C3")
    Hb, _, _ = codes.config_matrix("C2")
    for lean in (1, 0):
        da = pkg.BeliefPropagationDecoder(Ha, 0.05, mi, lean=lean, warps=8)
        db = pkg.BeliefPropagationDecoder(Hb, 0.03, mi, lean=lean, warps=8)
        assert da.info()["smem_bytes"] != db.info()["smem_bytes"]
        _, sa = oracle.sample(Ha, 0.05, 5, 0, 2000)
        _, sb = oracle.sample(Hb, 0.03, 6, 0, 2000)
        ra = oracle.batch_decode(Ha, 0.05, mi, sa, nthreads=oracle.num_threads())
        rb = oracle.batch_decode(Hb, 0.03, mi, sb, nthreads=oracle.num_threads())
        for _ in range(2):
            for dec, H, syn, ref in ((da, Ha, sa, ra), (db, Hb, sb, rb), (da, Ha, sa, ra)):
                errors = np.zeros((H.shape[1], syn.shape[1]), dtype=np.uint8, order="F")
                _, success = pkg.batchdecode_b(dec, syn, errors)
                assert np.array_equal(errors, ref["errors"]) and np.array_equal(success, ref["converged"])
        da.close()
        db.close()


@pytest.mark.parametrize("name,per,B", [("C3", 0.05, 60), ("C4", 0.04, 20), ("C1", 0.04, 9), ("C2", 0.03, 148)])
def test_minsum_small_batch_kernel(pkg, oracle, codes, name, per, B):
    """The node-parallel kernel of the min-sum variant against its CPU definition, and against the persistent kernel."""
    H, _, mi = codes.config_matrix(name)
    _, syn = oracle.sample(H, per, 606, 0, B)
    ref = oracle.batch_decode(H, per, mi, syn, variant="minsum", want_ratio=True)
    for sb in (-1, 0):
        g = run_gpu_variant(pkg, H, per, mi, syn, "minsum", small_batch=sb)
        assert np.array_equal(g["errors"], ref["errors"]) and np.array_equal(g["converged"], ref["converged"])
        assert np.array_equal(g["iters"], ref["iters"])
        assert np.array_equal(g["ratio"].view(np.uint64), ref["ratio"].view(np.uint64))


def test_bposd_syndromes_outside_the_column_space(pkg, oracle, codes):
    """Rank-deficient H and arbitrary syndromes: the elimination runs out of columns and which equations were made
    pivot rows decides the output, so the kernel has to follow the reference's (swapped) row order.  Found by
    tools/fuzz_parity.py; all posteriors tie at per = 0.5."""
    for (n, wr, wc, per, mi) in ((120, 6, 3, 0.5, 7), (100, 10, 5, 0.5, 7), (200, 8, 4, 0.1, 3), (96, 4, 3, 0.02, 5)):
        H = codes.gallager(n, wr, wc, seed=n + wr)
        s = H.shape[0]
        rng = np.random.default_rng(n)
        syn = (rng.random((s, 300)) < 0.5).astype(np.uint8)
        ref = oracle.bposd_decode(H, per, mi, syn, nthreads=oracle.num_threads())
        Hd = np.asarray(sp.csc_matrix(H).todense()).astype(np.int64)
        ok = ((Hd @ ref["errors"].astype(np.int64)) % 2 == syn).all(axis=0)
        assert 0 < ok.sum() < 300 or not ok.any()                      # most syndromes cannot be satisfied
        g = run_gpu_bposd(pkg, H, per, mi, syn)
        bad = np.nonzero((g["errors"] != ref["errors"]).any(axis=0))[0]
        assert bad.size == 0, (n, wr, wc, per, mi, bad[:10])
        assert np.array_equal(g["converged"], ref["converged"]) and g["stats"][1] == int(ref["pivots"].sum())


def test_pinned_and_pageable_host_memory_agree(pkg, oracle, codes):
    """The host-batch call stages pageable caller memory through pinned blocks and copies pinned (or registered)
    memory directly; both must give the oracle's answer, chunk by chunk (several chunks: chunk = 4096)."""
    H, _, mi = codes.config_matrix("C3")
    s, n = H.shape
    B = 50_000
    _, syn = oracle.sample(H, 0.05, 4242, 0, B)
    ref = oracle.batch_decode(H, 0.05, mi, syn, nthreads=oracle.num_threads())
    lib = pkg._lib
    for stage in (1, 0):
        dec = pkg.BeliefPropagationDecoder(H, 0.05, mi, chunk=4096, stage_pageable=stage)
        for pinned in (False, True):
            t_in = torch.from_numpy(np.ascontiguousarray(syn.T.astype(np.uint8)))          # [B][s] bytes == column-major s x B
            t_out = torch.zeros((B, n), dtype=torch.uint8)
            t_conv = torch.zeros(B, dtype=torch.uint8)
            t_it = torch.zeros(B, dtype=torch.int32)
            if pinned:
                t_in, t_out, t_conv, t_it = (x.pin_memory() for x in (t_in, t_out, t_conv, t_it))
            cnt = dec.decode_raw(B, t_in.numpy(), lib.FMT_U8, s, t_out.numpy(), lib.FMT_U8, n, t_conv.numpy(), t_it.numpy())
            assert np.array_equal(t_out.numpy().T, ref["errors"]), (stage, pinned)
            assert np.array_equal(t_conv.numpy().astype(bool), ref["converged"]) and np.array_equal(t_it.numpy(), ref["iters"])
            assert cnt[0] == B and cnt[1] == int(ref["converged"].sum())
        dec.close()


def test_sampling_and_scoring_harness_matches_host_recomputation(pkg, oracle, codes):
    """ldpcb200_sample_decode_score: sample -> decode -> score on the device equals the same steps done with the oracle's
    sampler/decoder and numpy scoring (failures against logical operators, and against plain equality without them);
    sharded handles give the same counters; set_per changes the prior only."""
    H = codes.gross_x()
    L = codes.css_logicals(H, codes.gross_z())
    s, n = H.shape
    shots, first, seed, per = 20_000, 1000, 777, 0.06
    truth, syn = oracle.sample(H, per, seed, first, shots)
    for prior, osd in ((per, False), (0.03, False), (per, True)):
        ref = (oracle.bposd_decode if osd else oracle.batch_decode)(H, prior, 32, syn, nthreads=oracle.num_threads())
        bpref = oracle.batch_decode(H, prior, 32, syn, nthreads=oracle.num_threads())
        dec_e = ref["errors"]
        resid = dec_e ^ truth
        sat = ((H @ dec_e) % 2 == syn).all(axis=0)
        logical = ((L @ resid) % 2 != 0).any(axis=0)
        want = dict(shots=shots, converged=int(bpref["converged"].sum()), iterations=int(bpref["iters"].sum()),
                    exact_matches=int((resid == 0).all(axis=0).sum()), syndrome_satisfied=int(sat.sum()),
                    failures=int((~sat | logical).sum()), residual_weight=int(resid.sum()),
                    osd_processed=int((~bpref["converged"]).sum()) if osd else 0)
        for devs in ([0], [0, 0, 0]):
            dec = pkg.BeliefPropagationDecoder(H, 0.5, 32, devices=devs)
            dec.set_per(prior)
            dec.set_logicals(L)
            got = dec.sample_decode_score(shots, first, seed, per, osd=osd)
            assert got == want, (prior, osd, devs, got, want)
            dec.set_logicals(None)                      # the reference test's criterion: decoded == truth
            got = dec.sample_decode_score(shots, first, seed, per, osd=osd)
            assert got["failures"] == shots - want["exact_matches"]
            dec.close()
    dec = pkg.BeliefPropagationDecoder(H, 0.01, 32)
    dec.set_logicals(L)
    rows = pkg.ler_curve(dec, [0.005, 0.02, 0.08], 30_000)
    assert [r["per"] for r in rows] == [0.005, 0.02, 0.08] and rows[0]["ler"] < rows[1]["ler"] < rows[2]["ler"]
    assert dec.per == 0.01
    dec.close()


@pytest.mark.parametrize("name,per,B", [("C3", 0.03, 20000), ("C3", 0.08, 8000), ("C2", 0.02, 8000), ("C4", 0.03, 1500), ("C1", 0.02, 300)])
def test_fast32_variant_tracks_its_definition(pkg, oracle, codes, name, per, B):
    """LDPCB200_VARIANT_FAST32 (FP32 tanh/atanh with the special-function unit) against its CPU definition
    (oracle: decode_edge_fast32, exp2f/log2f): the approximations differ in the last bits, BP amplifies that on a small
    fraction of hard syndromes, so the bar is statistical: at most 2 % of syndromes decoded differently, convergence
    rate within 0.5 % absolute, every converged output satisfies its syndrome, mean iterations within 2 %."""
    H, _, mi = codes.config_matrix(name)
    truth, syn = oracle.sample(H, per, 4711, 0, B)
    ref = oracle.batch_decode(H, per, mi, syn, nthreads=oracle.num_threads(), variant="fast")
    for opts in ({}, {"family": GLOBAL}):
        g = run_gpu_variant(pkg, H, per, mi, syn, "fast", **opts)
        differ = ((g["errors"] != ref["errors"]).any(axis=0) | (g["converged"] != ref["converged"])).mean()
        assert differ <= 0.02, (name, per, opts, differ)
        assert abs(g["converged"].mean() - ref["converged"].mean()) <= 0.005
        assert abs(g["iters"].mean() - ref["iters"].mean()) <= 0.02 * ref["iters"].mean() + 0.01
        sat = ((H @ g["errors"]) % 2 == syn).all(axis=0)
        assert (sat == g["converged"]).all()


def test_fast32_quality_is_close_to_exact(pkg, oracle, codes):
    """The fast variant is judged by decoding quality: exact-match rate within 0.5 % absolute of the exact kernels on
    the gross code at per 0.03, and the small-batch kernel agrees with the persistent one."""
    H, _, mi = codes.config_matrix("C3")
    B = 30000
    truth, syn = oracle.sample(H, 0.03, 99, 0, B)
    ex = run_gpu(pkg, H, 0.03, mi, syn)
    fa = run_gpu_variant(pkg, H, 0.03, mi, syn, "fast")
    em_ex = (ex["errors"] == truth).all(axis=0).mean()
    em_fa = (fa["errors"] == truth).all(axis=0).mean()
    assert abs(em_ex - em_fa) < 0.005, (em_ex, em_fa)
    small = run_gpu_variant(pkg, H, 0.03, mi, syn[:, :100], "fast")          # node-parallel kernel (B <= SM count)
    pers = run_gpu_variant(pkg, H, 0.03, mi, syn[:, :100], "fast", small_batch=0)
    assert np.array_equal(small["errors"], pers["errors"]) and np.array_equal(small["iters"], pers["iters"])


@pytest.mark.parametrize("name", ["gross_p05", "surface15_p03", "hgp_p05", "gallager1000_p03"])
def test_golden_osd_fixtures_on_gpu(pkg, name):
    """The committed BP+OSD-0 fixtures (what oracle/dump_golden.jl compares the real package with) through the CUDA path."""
    z = np.load(__import__("os").path.join(GOLDEN, name + ".npz"))
    zo = np.load(__import__("os").path.join(GOLDEN, name + ".osd.npz"))
    H = sp.csc_matrix((np.ones(len(z["rowval"]), dtype=np.uint8), z["rowval"], z["colptr"]), shape=tuple(z["shape"]))
    g = run_gpu_bposd(pkg, H, float(z["per"]), int(zo["max_iters"]), z["syndromes"])
    assert np.array_equal(g["errors"], zo["errors"]) and np.array_equal(g["converged"], zo["converged"])
    assert g["stats"][0] == int((~zo["converged"]).sum()) and g["stats"][1] == int(zo["pivots"][~zo["converged"]].sum())


@pytest.mark.parametrize("name,per,mi,B", [("C3", 0.08, 6, 600), ("C2", 0.05, 8, 400), ("C1", 0.05, 3, 24), ("C4", 0.04, 4, 40)])
def test_higher_order_osd_matches_restated_reference(pkg, oracle, codes, name, per, mi, B):
    """BeliefPropagationOSDDecoder(H, per, max_iters; osd_order = O > 0): osd(..., Val{O}) (belief_propagation_osd.jl:127-209)
    on every column -- bit for bit against the restated reference (physical row swaps, strict `<` in ascending trial order)."""
    H, _, _ = codes.config_matrix(name)
    _, syn = oracle.sample(H, per, 909, 0, B)
    for order in ((1, 3, 5) if name != "C4" else (2,)):
        ref = oracle.bposd_order_decode(H, per, mi, order, syn, nthreads=oracle.num_threads())
        g = run_gpu_bposd(pkg, H, per, mi, syn, osd_order=order)
        bad = np.nonzero((g["errors"] != ref["errors"]).any(axis=0) | (g["converged"] != ref["converged"]))[0]
        assert bad.size == 0, (name, order, bad[:10])
        assert ((H @ g["errors"]) % 2 == syn).all()
        assert g["stats"][0] == B            # every column goes through the search


def test_higher_order_osd_edge_cases(pkg, oracle, codes):
    """Order larger than the information set (clamped, :172-175), rank-deficient H with syndromes outside the column space
    (the outcome then depends on the reference's row order), max_iters = 0, single-syndrome decode!."""
    H = sp.csc_matrix(np.array([[1, 1, 0, 0], [0, 1, 1, 0], [1, 0, 1, 0]], dtype=np.uint8))
    syn = np.array([[1, 0, 1], [1, 1, 1], [0, 0, 1], [0, 0, 0], [1, 1, 0]], dtype=np.uint8).T
    for mi in (0, 3):
        for order in (1, 7):
            ref = oracle.bposd_order_decode(H, 0.1, mi, order, syn)
            g = run_gpu_bposd(pkg, H, 0.1, mi, syn, osd_order=order)
            assert np.array_equal(g["errors"], ref["errors"]) and np.array_equal(g["converged"], ref["converged"]), (mi, order)
    Hg = codes.gross_x()
    _, s2 = oracle.sample(Hg, 0.1, 4, 0, 20)
    ref = oracle.bposd_order_decode(Hg, 0.1, 4, 4, s2)
    dec = pkg.BeliefPropagationOSDDecoder(Hg, 0.1, 4, osd_order=4)
    for c in range(5):
        guess, conv = pkg.decode_b(dec, s2[:, c])
        assert np.array_equal(guess.astype(np.uint8), ref["errors"][:, c]) and conv == bool(ref["converged"][c])
    dec.close()


def _cycle_matrix(n):
    """create_cycle_matrix of /root/reference/test/test_bpots.jl:14-25."""
    r, c = [], []
    for j in range(n):
        r += [j, j]
        c += [(j + 1) % n, j]
    return sp.csc_matrix((np.ones(2 * n, dtype=np.uint8), (r, c)), shape=(n, n))


def _run_bpots(pkg, H, per, mi, syn, T=9, C=2.0, fmt=np.uint8, **opts):
    dec = pkg.BPOTSDecoder(H, per, mi, T=T, C=C, **opts)
    n, B = H.shape[1], syn.shape[1]
    errors = np.full((n, B), 1, dtype=fmt, order="F")
    iters = np.zeros(B, dtype=np.int32)
    _, success = pkg.batchdecode_b(dec, np.asfortranarray(syn.astype(fmt)), errors, iters=iters)
    dec.close()
    return dict(errors=errors.astype(np.uint8), converged=success.copy(), iters=iters)


@pytest.mark.parametrize("name,per,mi,T,C,B", [("C3", 0.05, 50, 9, 2.0, 3000), ("C3", 0.1, 40, 5, 3.0, 1500), ("C2", 0.05, 60, 9, 2.0, 1500),
                                               ("C1", 0.03, 30, 9, 2.0, 100), ("C4", 0.03, 30, 7, 5.0, 150)])
def test_bpots_matches_restated_reference(pkg, oracle, codes, name, per, mi, T, C, B):
    """BP-OTS (bpots_decoder.jl:226-340) on the GPU against the C restatement.  tanh / atanh / log come from two different
    math libraries (CUDA's and glibc's; the reference has Julia's), so a last-bit difference can be amplified on a hard
    syndrome: at least 99 % of the columns must agree in best_decisions, converged flag AND iteration count, the
    converged ones must reproduce their syndrome, and the rates must agree to 1 %."""
    H, _, _ = codes.config_matrix(name)
    _, syn = oracle.sample(H, per, 1357, 0, B)
    ref = oracle.bpots_decode(H, per, mi, syn, T=T, C=C, nthreads=oracle.num_threads())
    g = _run_bpots(pkg, H, per, mi, syn, T=T, C=C)
    same = (g["errors"] == ref["errors"]).all(axis=0) & (g["converged"] == ref["converged"]) & (g["iters"] == ref["iters"])
    assert same.mean() >= 0.99, (name, same.mean())
    sat = ((H @ g["errors"]) % 2 == syn).all(axis=0)
    assert (sat == g["converged"]).all()
    assert abs(g["converged"].mean() - ref["converged"].mean()) <= 0.01


def test_bpots_reference_test_cases(pkg, oracle):
    """The reference's own BP-OTS tests re-expressed (test/test_bpots.jl): cycle matrices n = 4, 8, 16 with random syndromes
    for several C (:56-114), the generic batchdecode! with a Matrix{Int} output (:139-153), a bool syndrome vector through
    decode! (:155-167) -- every decoded error must reproduce its syndrome, exactly what those tests assert."""
    rng = np.random.default_rng(5)
    for n in (4, 8, 16):
        H = _cycle_matrix(n)
        errs = rng.integers(0, 2, (n, 64)).astype(np.uint8)
        syn = (H @ errs) % 2
        for C in (1.0, 2.0, 5.0, 10.0):
            g = _run_bpots(pkg, H, 0.01, 100, syn, T=9, C=C, fmt=np.int64)
            ref = oracle.bpots_decode(H, 0.01, 100, syn, T=9, C=C)
            ok = ((H @ g["errors"]) % 2 == syn).all(axis=0)
            ok_ref = ((H @ ref["errors"]) % 2 == syn).all(axis=0)
            assert ok.mean() >= ok_ref.mean() - 0.05 and ok.mean() >= 0.9, (n, C, ok.mean(), ok_ref.mean())
            assert (ok == g["converged"]).all()
    H = _cycle_matrix(8)
    dec = pkg.BPOTSDecoder(H, 0.01, 100, T=9, C=3.0)
    e = np.zeros(8, dtype=bool)
    e[:2] = True
    syn = ((H @ e) % 2).astype(bool)
    guess, conv = pkg.decode_b(dec, syn)
    assert guess.dtype == np.int64 and conv and (((H @ guess) % 2).astype(bool) == syn).all()
    assert pkg.reset_b(dec) is dec
    dec.close()


def test_first_iteration_filter_properties(pkg, oracle, codes):
    """The first-iteration filter (bp_filter.cuh): with and without it the outputs are identical on a large batch at an
    error rate where most syndromes end in iteration 1, for all three variants, after set_per, and through the
    sampling harness; syndromes that end in iteration 1 really report one iteration."""
    H = codes.gross_x()
    B = 200_000
    for variant in ("exact", "minsum", "fast"):
        outs = []
        for flt in (1, 0):
            dec = pkg.BeliefPropagationDecoder(H, 0.2, 32, variant=variant, first_iteration_filter=flt)
            dec.set_per(0.01)                                   # tables must follow the prior
            errors = np.zeros((144, B), dtype=np.uint8, order="F")
            iters = np.zeros(B, dtype=np.int32)
            _, syn = oracle.sample(H, 0.01, 5, 0, B)
            _, success = pkg.batchdecode_b(dec, syn, errors, iters=iters)
            ctr = dec.last_counters.copy()
            # LDPCB200_CTR_FILTERED: syndromes the filter finished = those that report one iteration and converged
            assert ctr[3] == (int(((iters == 1) & (success != 0)).sum()) if flt else 0), (variant, flt, ctr)
            outs.append((errors.copy(), success.copy(), iters.copy(), ctr[:3]))
            dec.close()
        for a, b in zip(outs[0], outs[1]):
            assert np.array_equal(a, b), variant
        assert (outs[0][2] == 1).mean() > 0.8 and outs[0][3][0] == B and outs[0][3][2] == int(outs[0][2].sum())
    # the filtered fast-variant outputs (the last variant above, filter on) against the variant's CPU definition, with the
    # statistical bar of test_fast32_variant_tracks_its_definition
    syn_f = syn[:, :20000]
    ref_f = oracle.batch_decode(H, 0.01, 32, syn_f, nthreads=oracle.num_threads(), variant="fast")
    err_f, conv_f, it_f = outs[0][0][:, :20000], outs[0][1][:20000], outs[0][2][:20000]
    assert ((err_f != ref_f["errors"]).any(axis=0) | (conv_f != ref_f["converged"])).mean() <= 0.02
    assert abs(conv_f.mean() - ref_f["converged"].mean()) <= 0.005
    assert abs(it_f.mean() - ref_f["iters"].mean()) <= 0.02 * ref_f["iters"].mean() + 0.01
    assert (((H @ err_f) % 2 == syn_f).all(axis=0) == conv_f).all()
    ref = oracle.batch_decode(H, 0.01, 32, syn_f, nthreads=oracle.num_threads())
    dec = pkg.BeliefPropagationDecoder(H, 0.01, 32)
    errors = np.zeros((144, 20000), dtype=np.uint8, order="F")
    iters = np.zeros(20000, dtype=np.int32)
    _, success = pkg.batchdecode_b(dec, syn[:, :20000], errors, iters=iters)
    dec.close()
    assert np.array_equal(errors, ref["errors"]) and np.array_equal(success, ref["converged"]) and np.array_equal(iters, ref["iters"])
