"""ctypes front-end of oracle/bp_oracle.c (TEST INFRASTRUCTURE ONLY).

Follows /root/reference/src/decoders/belief_propagation.jl:121-188,220-231 -- see the C file
for the line-by-line citations.
"""
import ctypes
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "bp_oracle.c")
_SRC_OTS = os.path.join(_HERE, "bpots_oracle.c")
_OUT_DIR = os.path.join(_HERE, "_build")
_SO = os.path.join(_OUT_DIR, "libbporacle.so")
_lib = None

# IEEE double, every op rounded separately: no contraction, no fast-math.
CFLAGS = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared", "-fPIC", "-std=c11"]


def build(force=False):
    """Compile the C restatement with gcc (build() of __graft_entry__ calls this)."""
    if not force and os.path.exists(_SO) and os.path.getmtime(_SO) >= max(os.path.getmtime(_SRC), os.path.getmtime(_SRC_OTS)):
        return _SO
    os.makedirs(_OUT_DIR, exist_ok=True)
    tmp = _SO + ".tmp.%d" % os.getpid()
    subprocess.check_call(["gcc"] + CFLAGS + [_SRC, _SRC_OTS, "-o", tmp, "-lm"])
    os.replace(tmp, _SO)
    return _SO


def load():
    global _lib
    if _lib is not None:
        return _lib
    build()
    lib = ctypes.CDLL(_SO)
    i64p = ctypes.POINTER(ctypes.c_int64)
    u8p = ctypes.POINTER(ctypes.c_uint8)
    lib.bp_oracle_batch.restype = ctypes.c_int
    lib.bp_oracle_batch.argtypes = [ctypes.c_int64, ctypes.c_int64, i64p, i64p, ctypes.c_double,
                                    ctypes.c_int32, ctypes.c_int64, u8p, u8p, u8p,
                                    ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_double),
                                    ctypes.c_int32, ctypes.c_int32]
    lib.bp_oracle_sample.restype = ctypes.c_int
    lib.bp_oracle_sample.argtypes = [ctypes.c_int64, ctypes.c_int64, i64p, i64p, ctypes.c_double,
                                     ctypes.c_uint64, ctypes.c_int64, ctypes.c_int64, u8p, u8p]
    lib.bp_oracle_bposd_batch.restype = ctypes.c_int
    lib.bp_oracle_bposd_batch.argtypes = [ctypes.c_int64, ctypes.c_int64, i64p, i64p, ctypes.c_double,
                                          ctypes.c_int32, ctypes.c_int64, u8p, u8p, u8p, u8p,
                                          ctypes.POINTER(ctypes.c_int32), ctypes.c_int32]
    lib.bp_oracle_bposd_order_batch.restype = ctypes.c_int
    lib.bp_oracle_bposd_order_batch.argtypes = [ctypes.c_int64, ctypes.c_int64, i64p, i64p, ctypes.c_double, ctypes.c_int32, ctypes.c_int32,
                                                ctypes.c_int64, u8p, u8p, u8p, ctypes.c_int32]
    lib.bp_oracle_osd0_given.restype = ctypes.c_int
    lib.bp_oracle_osd0_given.argtypes = [ctypes.c_int64, ctypes.c_int64, i64p, i64p, ctypes.c_int64, u8p, u8p,
                                         ctypes.POINTER(ctypes.c_double), u8p, ctypes.POINTER(ctypes.c_int32), ctypes.c_int32]
    lib.bpots_oracle_batch.restype = ctypes.c_int
    lib.bpots_oracle_batch.argtypes = [ctypes.c_int64, ctypes.c_int64, i64p, i64p, ctypes.c_double, ctypes.c_int32, ctypes.c_int32,
                                       ctypes.c_double, ctypes.c_int64, u8p, u8p, u8p, ctypes.POINTER(ctypes.c_int32), ctypes.c_int32]
    lib.bp_oracle_set_minsum_scale.argtypes = [ctypes.c_double]
    lib.bp_oracle_set_minsum_scale.restype = None
    lib.bp_oracle_set_osd_key_mode.argtypes = [ctypes.c_int]
    lib.bp_oracle_set_osd_key_mode.restype = None
    lib.bp_oracle_threshold.restype = ctypes.c_uint32
    lib.bp_oracle_threshold.argtypes = [ctypes.c_double]
    lib.bp_oracle_num_threads.restype = ctypes.c_int
    _lib = lib
    return lib


def csc_arrays(H):
    """(s, n, colptr0, rowval0) of a 0/1 matrix; rows ascending inside each column."""
    import scipy.sparse as sp
    Hc = sp.csc_matrix(H)
    Hc.eliminate_zeros()
    Hc.sort_indices()
    s, n = Hc.shape
    return (s, n, np.ascontiguousarray(Hc.indptr, dtype=np.int64),
            np.ascontiguousarray(Hc.indices, dtype=np.int64))


def _p(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


def batch_decode(H, per, max_iters, syndromes, nthreads=1, dense=False, want_ratio=False, variant="exact",
                 minsum_scale=0.875):
    """Restated batchdecode! (variant="minsum": the min-sum definition the CUDA min-sum kernels are
    checked against -- no reference equivalent).  syndromes: (s, B) array of 0/1 (column = syndrome).
    Returns dict(errors (n,B) uint8, converged (B,) bool, iters (B,) int32[, ratio (n,B) f64])."""
    lib = load()
    lib.bp_oracle_set_minsum_scale(float(minsum_scale))
    s, n, colptr, rowval = csc_arrays(H)
    syn = np.asfortranarray(np.asarray(syndromes).astype(np.uint8))
    if syn.ndim == 1:
        syn = np.asfortranarray(syn.reshape(s, 1))
    assert syn.shape[0] == s
    B = syn.shape[1]
    err = np.zeros((n, B), dtype=np.uint8, order="F")
    conv = np.zeros(B, dtype=np.uint8)
    iters = np.zeros(B, dtype=np.int32)
    ratio = np.zeros((n, B), dtype=np.float64, order="F") if want_ratio else None
    rc = lib.bp_oracle_batch(s, n, _p(colptr, ctypes.c_int64), _p(rowval, ctypes.c_int64),
                             float(per), int(max_iters), B, _p(syn, ctypes.c_uint8),
                             _p(err, ctypes.c_uint8), _p(conv, ctypes.c_uint8),
                             _p(iters, ctypes.c_int32),
                             _p(ratio, ctypes.c_double) if want_ratio else None,
                             int(nthreads), {"minsum": 2, "fast": 3}.get(variant, 1 if dense else 0))
    if rc != 0:
        raise RuntimeError("bp_oracle_batch failed: %d" % rc)
    out = dict(errors=err, converged=conv.astype(bool), iters=iters)
    if want_ratio:
        out["ratio"] = ratio
    return out


def bposd_decode(H, per, max_iters, syndromes, nthreads=1, key_mode=0):
    """Restated decode!(::BeliefPropagationOSDDecoder, syndrome) with osd_order = 0
    (belief_propagation_osd.jl:49-125) applied to every column.  Returns dict(errors (n,B) uint8 -- the
    OSD result, converged (B,) bool -- BP's flag, bp_errors (n,B) uint8, pivots (B,) int32).
    key_mode: 0 = sort key from RN(1/R) (what the kernel computes), 1 = from exp(log(1/R)) with libm (the reference's
    expression; used to measure the stated deviation)."""
    lib = load()
    lib.bp_oracle_set_osd_key_mode(int(key_mode))
    s, n, colptr, rowval = csc_arrays(H)
    syn = np.asfortranarray(np.asarray(syndromes).astype(np.uint8))
    if syn.ndim == 1:
        syn = np.asfortranarray(syn.reshape(s, 1))
    assert syn.shape[0] == s
    B = syn.shape[1]
    err = np.zeros((n, B), dtype=np.uint8, order="F")
    bp = np.zeros((n, B), dtype=np.uint8, order="F")
    conv = np.zeros(B, dtype=np.uint8)
    piv = np.zeros(B, dtype=np.int32)
    rc = lib.bp_oracle_bposd_batch(s, n, _p(colptr, ctypes.c_int64), _p(rowval, ctypes.c_int64),
                                   float(per), int(max_iters), B, _p(syn, ctypes.c_uint8),
                                   _p(err, ctypes.c_uint8), _p(conv, ctypes.c_uint8), _p(bp, ctypes.c_uint8),
                                   _p(piv, ctypes.c_int32), int(nthreads))
    if rc != 0:
        raise RuntimeError("bp_oracle_bposd_batch failed: %d" % rc)
    return dict(errors=err, converged=conv.astype(bool), bp_errors=bp, pivots=piv)


def osd0_given(H, syndromes, bp_err, ratio, nthreads=1):
    """osd(..., Val(0)) behind the reliability sort (belief_propagation_osd.jl:52-60, :63-125) on caller-supplied BP
    decisions bp_err (n,B) and posterior ratios ratio (n,B), every column -- no BP call, and no shortcut for columns BP
    would call converged (bp_err satisfying the syndrome comes back unchanged with 0 pivots).  Returns dict(errors (n,B)
    uint8, pivots (B,) int32)."""
    lib = load()
    lib.bp_oracle_set_osd_key_mode(0)                 # the kernel's key, RN(1/R)
    s, n, colptr, rowval = csc_arrays(H)
    syn = np.asfortranarray(np.asarray(syndromes).astype(np.uint8))
    if syn.ndim == 1:
        syn = np.asfortranarray(syn.reshape(s, 1))
    B = syn.shape[1]
    e =np.asfortranarray(np.asarray(bp_err).astype(np.uint8).reshape(n, B))
    r = np.asfortranarray(np.asarray(ratio, dtype=np.float64).reshape(n, B))
    assert syn.shape[0] == s
    err = np.zeros((n, B), dtype=np.uint8, order="F")
    piv = np.zeros(B, dtype=np.int32)
    rc = lib.bp_oracle_osd0_given(s, n, _p(colptr, ctypes.c_int64), _p(rowval, ctypes.c_int64), B, _p(syn, ctypes.c_uint8),
                                  _p(e, ctypes.c_uint8), _p(r, ctypes.c_double), _p(err, ctypes.c_uint8),
                                  _p(piv, ctypes.c_int32), int(nthreads))
    if rc != 0:
        raise RuntimeError("bp_oracle_osd0_given failed: %d" % rc)
    return dict(errors=err, pivots=piv)


def bposd_order_decode(H, per, max_iters, osd_order, syndromes, nthreads=1, key_mode=0):
    """Restated decode!(::BeliefPropagationOSDDecoder, syndrome) with osd_order > 0 (belief_propagation_osd.jl:49-61,
    osd(..., Val{O}) :127-209) applied to every column.  Returns dict(errors (n,B) uint8, converged (B,) bool -- BP's flag)."""
    lib = load()
    lib.bp_oracle_set_osd_key_mode(int(key_mode))
    s, n, colptr, rowval = csc_arrays(H)
    syn = np.asfortranarray(np.asarray(syndromes).astype(np.uint8))
    if syn.ndim == 1:
        syn = np.asfortranarray(syn.reshape(s, 1))
    B = syn.shape[1]
    err = np.zeros((n, B), dtype=np.uint8, order="F")
    conv = np.zeros(B, dtype=np.uint8)
    rc = lib.bp_oracle_bposd_order_batch(s, n, _p(colptr, ctypes.c_int64), _p(rowval, ctypes.c_int64), float(per), int(max_iters),
                                         int(osd_order), B, _p(syn, ctypes.c_uint8), _p(err, ctypes.c_uint8), _p(conv, ctypes.c_uint8),
                                         int(nthreads))
    if rc != 0:
        raise RuntimeError("bp_oracle_bposd_order_batch failed: %d" % rc)
    return dict(errors=err, converged=conv.astype(bool))


def bpots_decode(H, per, max_iters, syndromes, T=9, C=2.0, nthreads=1):
    """Restated decode!(::BPOTSDecoder, syndrome) (bpots_decoder.jl:226-340) applied to every column.
    Returns dict(errors (n,B) uint8 -- best_decisions, converged (B,) bool, iters (B,) int32)."""
    lib = load()
    s, n, colptr, rowval = csc_arrays(H)
    syn = np.asfortranarray(np.asarray(syndromes).astype(np.uint8))
    if syn.ndim == 1:
        syn = np.asfortranarray(syn.reshape(s, 1))
    B = syn.shape[1]
    err = np.zeros((n, B), dtype=np.uint8, order="F")
    conv = np.zeros(B, dtype=np.uint8)
    iters = np.zeros(B, dtype=np.int32)
    rc = lib.bpots_oracle_batch(s, n, _p(colptr, ctypes.c_int64), _p(rowval, ctypes.c_int64), float(per), int(max_iters), int(T), float(C),
                                B, _p(syn, ctypes.c_uint8), _p(err, ctypes.c_uint8), _p(conv, ctypes.c_uint8), _p(iters, ctypes.c_int32),
                                int(nthreads))
    if rc != 0:
        raise RuntimeError("bpots_oracle_batch failed: %d" % rc)
    return dict(errors=err, converged=conv.astype(bool), iters=iters)


def sample(H, per, seed, first, B):
    """Philox4x32-10 Bernoulli(per) errors and their syndromes for global indices first..first+B-1.
    Returns (errors (n,B) uint8, syndromes (s,B) uint8), both Fortran order."""
    lib = load()
    s, n, colptr, rowval = csc_arrays(H)
    errs = np.zeros((n, B), dtype=np.uint8, order="F")
    syn = np.zeros((s, B), dtype=np.uint8, order="F")
    lib.bp_oracle_sample(s, n, _p(colptr, ctypes.c_int64), _p(rowval, ctypes.c_int64), float(per),
                         ctypes.c_uint64(seed), int(first), int(B),
                         _p(errs, ctypes.c_uint8), _p(syn, ctypes.c_uint8))
    return errs, syn


def threshold(per):
    return int(load().bp_oracle_threshold(float(per)))


def num_threads():
    """Host threads available to this process (affinity-aware); NOT omp_get_max_threads(), which
    torchrun pins to 1 through OMP_NUM_THREADS."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)
