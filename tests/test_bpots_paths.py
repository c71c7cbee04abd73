"""BP-OTS (csrc/bpots.cuh) on both memory paths, through every entry point.

One syndrome's BP-OTS arrays take 16 E + 23 n + 4 s bytes (two message arrays, node state, three decision arrays), rounded
up to 16, plus 512 bytes of reduction scratch.  Where that fits one CTA's shared memory the kernel keeps everything there;
beyond it (and always with option bpots_memory = 2) every CTA of the grid works in its own slice of a per-device workspace
in global memory, running the same operations in the same order.  The global path must therefore give the shared path's
outputs bit for bit: best decisions, converged flags and iteration counts.  Codes beyond shared memory are compared with
the CPU restatement by the criterion of test_bpots_matches_restated_reference (tanh / atanh / log differ between CUDA and
glibc in the last bit).  The device-resident call, the multi-device and single-syndrome host paths and the sampling
harness must each equal the single-device host batch."""
import functools

import numpy as np
import pytest
import scipy.sparse as sp

from test_kernel_paths import configuration_model, degrees

B200_SMEM_OPTIN = 232448    # shared memory per block (opt-in) of a B200


def ots_need(s, n, E):
    """Shared-memory bytes of one BP-OTS CTA (bpots_on_device's carve-up, empty graphs count one node / edge)."""
    s, n, E = max(s, 1), max(n, 1), max(E, 1)
    return (16 * E + 23 * n + 4 * s + 15) // 16 * 16 + 512


def need_of(H):
    H = sp.csc_matrix(H)
    return ots_need(H.shape[0], H.shape[1], H.nnz)


def cycle_matrix(n):
    """create_cycle_matrix of the reference's test/test_bpots.jl:14-25."""
    r, c = [], []
    for j in range(n):
        r += [j, j]
        c += [(j + 1) % n, j]
    return sp.csc_matrix((np.ones(2 * n, dtype=np.uint8), (r, c)), shape=(n, n))


# designed graphs ({check degree: count}, {variable degree: count}, seed)
QSPECS = {
    # irregular: empty rows, degree-0 variables, check degrees up to 64 (fits shared memory)
    "Q1": ({0: 5, 1: 20, 2: 30, 3: 40, 8: 20, 16: 10, 32: 5, 64: 3}, {0: 10, 1: 600, 2: 100, 3: 24}, 301),
    # check degrees 32..128, beyond shared memory
    "Q2": ({32: 100, 64: 50, 128: 20}, {1: 8000, 2: 480}, 302),
    # straddle pair: exactly the budget (16 E + 23 n + 4 s = 231,936), and one empty check more (the next 16-byte step)
    "S0": ({5: 132, 6: 1478}, {3: 3176}, 303),
    "S1": ({0: 1, 5: 132, 6: 1478}, {3: 3176}, 303),
}


@functools.lru_cache(maxsize=None)
def qgraph(name):
    return configuration_model(*QSPECS[name])


@functools.lru_cache(maxsize=None)
def named(codes, name):
    if name in ("C1", "C2", "C3", "C4", "C5"):
        return sp.csc_matrix(codes.config_matrix(name)[0])
    if name.startswith("cycle"):
        return cycle_matrix(int(name[5:]))
    if name.startswith("hgp"):
        return sp.csc_matrix(codes.hgp_x(codes.gallager(int(name[3:]), 4, 3)))
    return qgraph(name)


def run_batch(pkg, H, per, mi, syn, T, C, devices=None, **opts):
    dec = pkg.BPOTSDecoder(H, per, mi, T=T, C=C, devices=devices, **opts)
    n, B = H.shape[1], syn.shape[1]
    errors = np.full((n, B), 1, dtype=np.uint8, order="F")
    iters = np.full(B, -1, dtype=np.int32)
    _, success = pkg.batchdecode_b(dec, np.asfortranarray(syn.astype(np.uint8)), errors, iters=iters)
    ws = dec.info()["bpots_workspace_bytes"]
    dec.close()
    return dict(errors=errors, converged=success.copy(), iters=iters), ws


def assert_same(a, b, what):
    assert np.array_equal(a["errors"], b["errors"]), what
    assert np.array_equal(a["converged"], b["converged"]), what
    assert np.array_equal(a["iters"], b["iters"]), what


def oracle_agreement(H, syn, g, ref):
    """Fraction of columns equal to the restatement; converged columns must reproduce their syndrome and the rates must
    agree to 1 % (the bar of test_bpots_matches_restated_reference)."""
    same = (g["errors"] == ref["errors"]).all(axis=0) & (g["converged"] == ref["converged"]) & (g["iters"] == ref["iters"])
    sat = ((H @ g["errors"]) % 2 == syn).all(axis=0)
    assert (sat == g["converged"]).all()
    assert abs(g["converged"].mean() - ref["converged"].mean()) <= 0.01
    return same.mean()


# ---------------------------------------------------------------------------------------------------------------------
# CPU
def test_shared_memory_need_of_the_named_codes(codes):
    """The restated carve-up gives the shared memory each code needs; at most 232,448 bytes fit (the B200's opt-in)."""
    want = {"C1": 171120, "C4": 126400, "hgp40": 197216, "hgp44": 238528, "hgp64": 504064, "C5": 7300672}
    shapes = {"C1": (900, 1000, 9000), "C4": (768, 1600, 5376), "hgp40": (1200, 2500, 8400), "hgp44": (1452, 3025, 10164),
              "hgp64": (3072, 6400, 21504), "C5": (50001, 100002, 300006)}
    for name, need in want.items():
        H = named(codes, name)
        assert (H.shape[0], H.shape[1], H.nnz) == shapes[name], name
        assert need_of(H) == need, name
        assert (need <= B200_SMEM_OPTIN) == (name in ("C1", "C4", "hgp40")), name


def test_designed_graph_profiles():
    cd, vd = degrees(qgraph("Q1"))
    assert (cd == 0).sum() == 5 and cd.max() == 64 and (vd == 0).sum() == 10 and qgraph("Q1").shape == (133, 734)
    assert need_of(qgraph("Q1")) <= B200_SMEM_OPTIN
    cd, vd = degrees(qgraph("Q2"))
    assert sorted(set(cd)) == [32, 64, 128] and vd.max() == 2 and need_of(qgraph("Q2")) > B200_SMEM_OPTIN
    for name in ("S0", "S1"):
        H = qgraph(name)
        assert H.max() == 1 and H.nnz == 9528 and H.shape[1] == 3176
    assert (degrees(qgraph("S1"))[0] == 0).sum() == 1 and qgraph("S1").shape[0] == 1611


def test_straddle_pair_needs_exactly_the_budget_and_one_step_more():
    assert need_of(qgraph("S0")) == B200_SMEM_OPTIN
    assert need_of(qgraph("S1")) == B200_SMEM_OPTIN + 16


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# (name, per, max_iters, T, C, B): B = 2501 exceeds any grid of the global path (at most 148 SMs x 8 CTAs of 256 threads), so
# CTAs decode several syndromes in one workspace slice and the last wave is partial
EQUAL_CASES = [
    ("C1", 0.03, 30, 9, 2.0, 2501),
    ("C2", 0.05, 40, 1, 1.0, 2501),
    ("C3", 0.08, 0, 9, 2.0, 1300),
    ("C3", 0.08, 32, 5, 3.0, 2501),
    ("C4", 0.03, 30, 7, 5.0, 1500),
    ("cycle4", 0.01, 100, 9, 2.0, 64),
    ("cycle8", 0.01, 100, 9, 10.0, 64),
    ("cycle16", 0.01, 100, 9, 1.0, 64),
    ("hgp40", 0.03, 30, 9, 2.0, 300),
    ("Q1", 0.05, 40, 3, 3.0, 2501),
    ("Q1", 0.3, 12, 1, 2.0, 700),
    ("S0", 0.02, 20, 9, 2.0, 200),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,per,mi,T,C,B", EQUAL_CASES)
def test_global_path_equals_shared_path(pkg, oracle, codes, name, per, mi, T, C, B):
    H = named(codes, name)
    if name.startswith("cycle"):
        syn = (H @ np.random.default_rng(int(name[5:])).integers(0, 2, (H.shape[1], B))) % 2      # test_bpots.jl's syndromes
    else:
        _, syn = oracle.sample(H, per, 8080, 0, B)
    shared, ws_s = run_batch(pkg, H, per, mi, syn, T, C)
    glob, ws_g = run_batch(pkg, H, per, mi, syn, T, C, bpots_memory=2)
    assert ws_s == 0 and ws_g > 0                        # default = shared memory; option 2 = the workspace
    assert_same(shared, glob, name)
    assert (glob["iters"] <= mi).all() and (glob["iters"] >= min(mi, 1)).all()


# (name, per, max_iters, T, C, B)
BEYOND_CASES = [
    ("hgp44", 0.03, 30, 9, 2.0, 300),
    ("hgp64", 0.02, 32, 9, 2.0, 300),
    ("C5", 0.02, 20, 9, 2.0, 64),
    ("Q2", 0.01, 20, 5, 2.0, 300),
    ("S1", 0.02, 20, 9, 2.0, 200),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,per,mi,T,C,B", BEYOND_CASES)
def test_codes_beyond_shared_memory(pkg, oracle, codes, name, per, mi, T, C, B):
    """Auto mode runs these in the workspace; they agree with the restatement; shared-only mode refuses them on the same
    handle, which afterwards decodes again."""
    H = named(codes, name)
    assert need_of(H) > B200_SMEM_OPTIN
    _, syn = oracle.sample(H, per, 9090, 0, B)
    ref = oracle.bpots_decode(H, per, mi, syn, T=T, C=C, nthreads=oracle.num_threads())
    g, ws = run_batch(pkg, H, per, mi, syn, T, C)
    assert ws > 0
    agree = oracle_agreement(H, syn, g, ref)
    print("%s: %.4f of %d columns equal the restatement, converged %.4f" % (name, agree, B, g["converged"].mean()))
    assert agree >= 0.99, (name, agree)
    dec = pkg.BPOTSDecoder(H, per, mi, T=T, C=C)
    errors = np.zeros((H.shape[1], 8), dtype=np.uint8, order="F")
    dec.set_option("bpots_memory", 1)
    with pytest.raises(pkg._lib.LibraryError) as ei:
        pkg.batchdecode_b(dec, syn[:, :8], errors)
    assert ei.value.code == pkg._lib.EUNSUPPORTED
    dec.set_option("bpots_memory", 0)
    _, success = pkg.batchdecode_b(dec, syn[:, :8], errors)
    assert np.array_equal(errors, g["errors"][:, :8]) and np.array_equal(success, g["converged"][:8])
    dec.close()


def pack_rows(M):
    """(rows, B) 0/1 -> [B][ceil(rows/32)] uint32, bit r % 32 of word r / 32 (LDPCB200_FMT_PACKED32)."""
    rows, B = M.shape
    W = (rows + 31) // 32
    bits = np.zeros((B, W * 32), dtype=np.uint8)
    bits[:, :rows] = M.T
    return np.packbits(bits, axis=1, bitorder="little").view("<u4").reshape(B, W)


def unpack_rows(words, rows):
    return np.unpackbits(words.view(np.uint8), axis=1, bitorder="little")[:, :rows].T.copy()


@pytest.mark.gpu
def test_entry_points_equal_the_host_batch(pkg, oracle, codes):
    """Three devices of one GPU, decode_b of one column, and ldpcb200_bpots_device on torch buffers and a caller's stream
    (both memory paths, counters added) all give the single-device host batch's outputs."""
    import torch
    per, mi, T, C = 0.02, 32, 9, 2.0
    Hh = named(codes, "hgp64")
    _, syn = oracle.sample(Hh, per, 4343, 0, 250)
    ref, _ = run_batch(pkg, Hh, per, mi, syn, T, C)
    sharded, _ = run_batch(pkg, Hh, per, mi, syn, T, C, devices=[0, 0, 0])
    assert_same(ref, sharded, "devices=[0,0,0]")
    dec = pkg.BPOTSDecoder(Hh, per, mi, T=T, C=C)
    for c in (0, 7):
        guess, conv = pkg.decode_b(dec, syn[:, c])
        assert np.array_equal(guess.astype(np.uint8), ref["errors"][:, c]) and conv == bool(ref["converged"][c])
    dec.close()
    for name, mem in (("C4", 1), ("C4", 2), ("hgp64", 0)):
        H = named(codes, name)
        s, n = H.shape
        B = 333
        _, syn = oracle.sample(H, per, 5151, 0, B)
        want, _ = run_batch(pkg, H, per, mi, syn, T, C)
        dec = pkg.BPOTSDecoder(H, per, mi, T=T, C=C, bpots_memory=mem)
        dev = torch.device("cuda:0")
        d_syn = torch.from_numpy(pack_rows(syn).view(np.int32)).to(dev)
        d_err = torch.full((B, (n + 31) // 32), -1, dtype=torch.int32, device=dev)
        d_conv = torch.full((B,), 7, dtype=torch.uint8, device=dev)
        d_it = torch.zeros(B, dtype=torch.int32, device=dev)
        d_ctr = torch.tensor([5, 6, 7, 8], dtype=torch.int64, device=dev)
        st = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(st):
            dec.decode_device(B, d_syn.data_ptr(), d_err.data_ptr(), d_conv.data_ptr(), d_it.data_ptr(), d_ctr.data_ptr(),
                              stream=st.cuda_stream)
        st.synchronize()
        got_e = unpack_rows(d_err.cpu().numpy().view(np.uint32), n)
        got_c = d_conv.cpu().numpy()
        got_i = d_it.cpu().numpy()
        assert np.array_equal(got_e, want["errors"]), (name, mem)
        assert np.array_equal(got_c, want["converged"].astype(np.uint8)) and np.array_equal(got_i, want["iters"]), (name, mem)
        assert d_ctr.cpu().tolist() == [5 + B, 6 + int(got_c.sum()), 7 + int(got_i.sum()), 8], (name, mem)
        assert (dec.info()["bpots_workspace_bytes"] > 0) == (mem != 1), (name, mem)
        dec.close()


@pytest.mark.gpu
def test_sampling_harness_equals_host_recomputation(pkg, oracle, codes):
    """ldpcb200_sample_bpots_score draws the oracle's Philox shots, decodes them as the host batch does and scores them as
    numpy does, on one device and three, with and without logical operators, in shared memory and in the workspace."""
    T, C = 9, 2.0
    Hg = named(codes, "C3")
    Lg = codes.css_logicals(codes.gross_x(), codes.gross_z())
    cases = [("C3", Lg, 0.05, 3001, 1000, 32), ("C3", None, 0.08, 2999, 77, 20), ("hgp64", None, 0.02, 301, 64, 32)]
    for name, L, per, shots, first, mi in cases:
        H = named(codes, name)
        seed = 2468
        truth, syn = oracle.sample(H, per, seed, first, shots)
        g, _ = run_batch(pkg, H, per, mi, syn, T, C)
        resid = g["errors"] ^ truth
        sat = ((H @ g["errors"]) % 2 == syn).all(axis=0)
        fail = ~sat | ((L @ resid) % 2 != 0).any(axis=0) if L is not None else (resid != 0).any(axis=0)
        want = dict(shots=shots, converged=int(g["converged"].sum()), iterations=int(g["iters"].sum()),
                    exact_matches=int((resid == 0).all(axis=0).sum()), syndrome_satisfied=int(sat.sum()),
                    failures=int(fail.sum()), residual_weight=int(resid.sum()), osd_processed=0)
        for devs in ([0], [0, 0, 0]):
            dec = pkg.BPOTSDecoder(H, 0.5, mi, T=T, C=C, devices=devs)
            dec.set_per(per)
            dec.set_logicals(L)
            got = dec.sample_decode_score(shots, first, seed, per)
            assert got == want, (name, devs, got, want)
            assert (dec.info()["bpots_workspace_bytes"] > 0) == (name == "hgp64")
            dec.close()
    dec = pkg.BPOTSDecoder(Hg, 0.01, 32, T=T, C=C)
    dec.set_logicals(Lg)
    rows = pkg.ler_curve(dec, [0.01, 0.04, 0.1], 5000)
    assert [r["per"] for r in rows] == [0.01, 0.04, 0.1] and rows[0]["ler"] < rows[1]["ler"] < rows[2]["ler"]
    assert rows[0]["osd_processed"] == 0 and dec.per == 0.01
    dec.close()
