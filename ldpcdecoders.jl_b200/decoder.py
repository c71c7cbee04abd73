"""Host-side mirror of the reference's BP decoder interface, on top of the C ABI.

Julia is not available in the build image, so this Python module plays the role the Julia shim
(julia/LDPCDecodersB200.jl, see INTEGRATION.md) plays for real users: same names, argument
meaning and error behaviour as /root/reference/src/decoders/belief_propagation.jl, with `f!`
spelled `f_b` (PyJulia's convention):

    BeliefPropagationDecoder(H, per, max_iters)      belief_propagation.jl:61-67
    reset_b(decoder)                                 belief_propagation.jl:83-91  (no-op: no host scratch to clear)
    decode_b(decoder, syndrome) -> (err, converged)  belief_propagation.jl:121-188
    batchdecode_b(decoder, syndromes, errors[, success]) -> (errors, success)
                                                     belief_propagation.jl:220-231, abstract_decoder.jl:44-48

All arithmetic happens in libldpcb200.so on the GPU; nothing here computes messages.
"""
import ctypes

import numpy as np
import scipy.sparse as sp

from . import _lib


class BeliefPropagationScratchSpace:
    """What BP+OSD reads after decode! (belief_propagation_osd.jl:51-52): err and log_probabs."""

    def __init__(self, n):
        self.log_probabs = np.zeros(n, dtype=np.float64)
        self.err = np.zeros(n, dtype=np.float64)


def _fmt_of(a, what):
    if a.dtype == np.bool_ or a.dtype == np.uint8 or a.dtype == np.int8:
        return _lib.FMT_U8
    if a.dtype == np.int64:
        return _lib.FMT_I64
    if what == "errors" and a.dtype == np.float64:
        return _lib.FMT_F64
    raise TypeError("%s: unsupported element type %s (use bool/uint8/int64%s)" %
                    (what, a.dtype, "/float64" if what == "errors" else ""))


class BeliefPropagationDecoder:
    """BeliefPropagationDecoder(H, per, max_iters) -- fields per, max_iters, s, n, sparse_H,
    sparse_HT, scratch as in belief_propagation.jl:38-59; the Tanner graph lives on the GPU.
    variant="minsum" selects the (non-reference) min-sum kernels; default is the exact replica."""

    def __init__(self, H, per, max_iters, devices=None, variant="exact", **options):
        if not isinstance(per, float):
            raise TypeError("per must be a Float64 (belief_propagation.jl:61)")
        if isinstance(max_iters, bool) or not isinstance(max_iters, (int, np.integer)):
            raise TypeError("max_iters must be an Int (belief_propagation.jl:61)")
        Hc = sp.csc_matrix(H)
        Hc.eliminate_zeros()
        Hc.sort_indices()
        self.per = float(per)
        self.max_iters = int(max_iters)
        self.s, self.n = (int(x) for x in Hc.shape)
        self.sparse_H = Hc
        self.sparse_HT = Hc.T.tocsc()
        self.variant = variant
        self.scratch = BeliefPropagationScratchSpace(self.n)
        lib = _lib.load()
        colptr = np.ascontiguousarray(Hc.indptr, dtype=np.int64)
        rowval = np.ascontiguousarray(Hc.indices, dtype=np.int64)
        devs = None
        ndev = 0
        if devices is not None:
            devs = np.ascontiguousarray(devices, dtype=np.int32)
            ndev = len(devs)
        h = ctypes.c_void_p()
        _lib.check(lib.ldpcb200_create(self.s, self.n, colptr.ctypes.data, rowval.ctypes.data, 0,
                                       self.per, self.max_iters,
                                       {"exact": _lib.VARIANT_EXACT, "minsum": _lib.VARIANT_MINSUM, "fast": _lib.VARIANT_FAST32}[variant],
                                       devs.ctypes.data if devs is not None else None, ndev,
                                       ctypes.byref(h)))
        self._h = h
        self._lib = lib
        for k, v in options.items():
            self.set_option(k, v)

    # -- library plumbing -------------------------------------------------------------------
    def set_option(self, key, value):
        _lib.check(self._lib.ldpcb200_set_option(self._h, key.encode(), int(value)))

    def info(self):
        out = _lib.Info()
        _lib.check(self._lib.ldpcb200_info(self._h, ctypes.byref(out)))
        return {f: getattr(out, f) for f, _ in _lib.Info._fields_}

    def launch_count(self):
        out = ctypes.c_int64()
        _lib.check(self._lib.ldpcb200_launch_count(self._h, ctypes.byref(out)))
        return out.value

    # -- sampling + scoring harness (SURVEY 8(f) rank 2) ---------------------------------------
    def set_logicals(self, L):
        """Logical operators L (k x n, k <= 64, any 0/1 matrix; None removes them): a decoded error then counts as a
        failure when it does not reproduce the syndrome or differs from the true error by a logical operator."""
        if L is None:
            _lib.check(self._lib.ldpcb200_set_logicals(self._h, 0, None, None, 0))
            return
        Lc = sp.csc_matrix(L)
        Lc.data[:] = Lc.data % 2
        Lc.eliminate_zeros()
        Lc.sort_indices()
        assert Lc.shape[1] == self.n
        colptr = np.ascontiguousarray(Lc.indptr, dtype=np.int64)
        rowval = np.ascontiguousarray(Lc.indices, dtype=np.int64)
        _lib.check(self._lib.ldpcb200_set_logicals(self._h, Lc.shape[0], colptr.ctypes.data, rowval.ctypes.data, 0))

    def set_per(self, per):
        """New prior (channel_probs) for the same device-resident Tanner graph."""
        _lib.check(self._lib.ldpcb200_set_per(self._h, float(per)))
        self.per = float(per)

    def sample_decode_score(self, shots, first, seed, per_channel, osd=False):
        """`shots` synthetic errors of rate per_channel sampled, decoded and scored on the handle's devices
        (ldpcb200_sample_decode_score); returns a dict of the eight counters."""
        out = (ctypes.c_int64 * _lib.NUM_HARNESS_COUNTERS)()
        _lib.check(self._lib.ldpcb200_sample_decode_score(self._h, int(shots), int(first), ctypes.c_uint64(seed), float(per_channel),
                                                          1 if osd else 0, out))
        return dict(zip(_lib.HARNESS_FIELDS, [int(x) for x in out]))

    def score_logical_device(self, B, d_true_err_words, d_err_words, d_syn_words, d_out, stream=None, dev_slot=0):
        _lib.check(self._lib.ldpcb200_score_logical_device(self._h, dev_slot, int(B), d_true_err_words, d_err_words, d_syn_words,
                                                           d_out, stream))

    def kernel_profile(self, reset=True, dev_slot=0):
        """Per-phase SM cycles of the shared-memory kernel (option kernel_profile=1); see ldpcb200_kernel_profile."""
        out = (ctypes.c_int64 * 8)()
        _lib.check(self._lib.ldpcb200_kernel_profile(self._h, dev_slot, out, 1 if reset else 0))
        names = ("check", "wait_b1", "variable", "flips", "wait_b2", "done_emit", "refill", "warp_iterations")
        return dict(zip(names, [int(x) for x in out]))

    def kernel_time(self, reset=True, dev_slot=0):
        """(milliseconds, launches) of the decoding kernel itself since the last reset (option time_kernels=1):
        CUDA events on the launching stream around every launch; see ldpcb200_kernel_time."""
        ms = ctypes.c_double(0.0)
        nl = ctypes.c_int64(0)
        _lib.check(self._lib.ldpcb200_kernel_time(self._h, dev_slot, ctypes.byref(ms), ctypes.byref(nl), 1 if reset else 0))
        return float(ms.value), int(nl.value)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ldpcb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- device-resident entry points (bench / sampling loops) ------------------------------
    def decode_device(self, B, d_syn_words, d_err_words, d_conv, d_iters=None, d_ratio=None,
                      d_counters=None, stream=None, dev_slot=0):
        _lib.check(self._lib.ldpcb200_decode_device(self._h, dev_slot, int(B), d_syn_words, d_err_words,
                                                    d_conv, d_iters, d_ratio, d_counters, stream))

    def sample_device(self, B, first, seed, per, d_true_err_words, d_syn_words, stream=None, dev_slot=0):
        _lib.check(self._lib.ldpcb200_sample_device(self._h, dev_slot, int(B), int(first),
                                                    ctypes.c_uint64(seed), float(per),
                                                    d_true_err_words, d_syn_words, stream))

    def score_device(self, B, d_true_err_words, d_err_words, d_syn_words, d_out, stream=None, dev_slot=0):
        _lib.check(self._lib.ldpcb200_score_device(self._h, dev_slot, int(B), d_true_err_words,
                                                   d_err_words, d_syn_words, d_out, stream))

    def osd0_device(self, B, d_syn_words, d_err_words, d_conv, d_ratio, d_stats=None, stream=None, dev_slot=0):
        _lib.check(self._lib.ldpcb200_osd0_device(self._h, dev_slot, int(B), d_syn_words, d_err_words, d_conv,
                                                  d_ratio, d_stats, stream))

    # -- raw host-buffer calls --------------------------------------------------------------
    def bposd_raw(self, B, syn, syn_fmt, syn_ld, err, err_fmt, err_ld, conv, iters=None):
        counters = np.zeros(_lib.NUM_COUNTERS, dtype=np.int64)
        stats = np.zeros(_lib.NUM_OSD_STATS, dtype=np.int64)
        _lib.check(self._lib.ldpcb200_bposd_decode_batch(
            self._h, int(B), syn.ctypes.data, syn_fmt, int(syn_ld), err.ctypes.data, err_fmt, int(err_ld),
            conv.ctypes.data, iters.ctypes.data if iters is not None else None, counters.ctypes.data,
            stats.ctypes.data))
        return counters, stats

    def decode_raw(self, B, syn, syn_fmt, syn_ld, err, err_fmt, err_ld, conv, iters=None, ratio=None):
        counters = np.zeros(_lib.NUM_COUNTERS, dtype=np.int64)
        _lib.check(self._lib.ldpcb200_decode_batch(
            self._h, int(B), syn.ctypes.data, syn_fmt, int(syn_ld), err.ctypes.data, err_fmt, int(err_ld),
            conv.ctypes.data, iters.ctypes.data if iters is not None else None,
            ratio.ctypes.data if ratio is not None else None, counters.ctypes.data))
        return counters


class BeliefPropagationOSDDecoder:
    """Mirror of BeliefPropagationOSDDecoder(H, per, max_iters; osd_order=0)
    (/root/reference/src/decoders/belief_propagation_osd.jl:17-29): fields bp_decoder, H, osd_order.
    osd_order = 0 (the path BASELINE config 4 names) post-processes the syndromes BP left unconverged
    (osd(..., Val(0)), :63-125); osd_order > 0 runs the exhaustive search of osd(..., Val{O}) (:127-209) on every
    syndrome, as the reference's decode! does."""

    def __init__(self, H, per, max_iters, osd_order=0, devices=None, **options):
        if not 0 <= int(osd_order) <= 12:
            raise ValueError("osd_order must be between 0 and 12 on the GPU")
        self.bp_decoder = BeliefPropagationDecoder(H, per, max_iters, devices=devices, **options)
        self.H = H
        self.osd_order = int(osd_order)
        if self.osd_order:
            self.bp_decoder.set_option("osd_order", self.osd_order)
        self.s, self.n = self.bp_decoder.s, self.bp_decoder.n
        self.last_counters = None
        self.last_osd_stats = None

    def close(self):
        self.bp_decoder.close()


class BPOTSDecoder:
    """Mirror of BPOTSDecoder(H, per, max_iters; T=9, C=2.0) (/root/reference/src/decoders/bpots_decoder.jl:42-111):
    fields per, max_iters, s, n, T, C, sparse_H, sparse_HT; decode_b / batchdecode_b return (best_decisions, converged)."""

    def __init__(self, H, per, max_iters, T=9, C=2.0, devices=None, **options):
        self._bp = BeliefPropagationDecoder(H, per, max_iters, devices=devices, **options)     # graph tables + handle
        self.per, self.max_iters, self.s, self.n = self._bp.per, self._bp.max_iters, self._bp.s, self._bp.n
        self.sparse_H, self.sparse_HT = self._bp.sparse_H, self._bp.sparse_HT
        self.T, self.C = int(T), float(C)
        self.last_counters = None

    def decode_raw(self, B, syn, syn_fmt, syn_ld, err, err_fmt, err_ld, conv, iters=None):
        _lib.check(self._bp._lib.ldpcb200_bpots_decode_batch(
            self._bp._h, int(B), syn.ctypes.data, syn_fmt, int(syn_ld), err.ctypes.data, err_fmt, int(err_ld), conv.ctypes.data,
            iters.ctypes.data if iters is not None else None, self.T, self.C))

    def decode_device(self, B, d_syn_words, d_err_words, d_conv, d_iters=None, d_counters=None, stream=None, dev_slot=0):
        """BP-OTS on device-resident packed rows (ldpcb200_bpots_device), asynchronous on `stream`; d_counters (nullable,
        four uint64) receives ADDED decoded / converged / iteration counts."""
        _lib.check(self._bp._lib.ldpcb200_bpots_device(self._bp._h, dev_slot, int(B), d_syn_words, d_err_words, d_conv, d_iters,
                                                       d_counters, self.T, self.C, stream))

    def sample_decode_score(self, shots, first, seed, per_channel):
        """The sampling + scoring harness with BP-OTS as the decoder (ldpcb200_sample_bpots_score); returns a dict of the
        eight counters (iterations = BP-OTS iterations, osd_processed = 0)."""
        out = (ctypes.c_int64 * _lib.NUM_HARNESS_COUNTERS)()
        _lib.check(self._bp._lib.ldpcb200_sample_bpots_score(self._bp._h, int(shots), int(first), ctypes.c_uint64(seed),
                                                             float(per_channel), self.T, self.C, out))
        return dict(zip(_lib.HARNESS_FIELDS, [int(x) for x in out]))

    def set_per(self, per):
        """New prior for the same device-resident Tanner graph (the depolarising prior follows it)."""
        self._bp.set_per(per)
        self.per = self._bp.per

    def set_logicals(self, L):
        self._bp.set_logicals(L)

    def set_option(self, key, value):
        self._bp.set_option(key, value)

    def info(self):
        return self._bp.info()

    def close(self):
        self._bp.close()


def reset_b(decoder):
    """LDPCDecoders.reset!(decoder): the GPU path keeps no host scratch between calls."""
    if isinstance(decoder, BeliefPropagationOSDDecoder):
        reset_b(decoder.bp_decoder)
        return decoder
    if isinstance(decoder, BPOTSDecoder):
        return decoder                          # bpots_decoder.jl:144-156: all state is re-initialised inside the kernel
    decoder.scratch.log_probabs[:] = 0.0
    decoder.scratch.err[:] = 0.0
    return decoder


def _as_columns(a, rows, what):
    a = np.asarray(a)
    if a.ndim != 2 or a.shape[0] != rows:
        raise ValueError("%s must be a %d x B matrix" % (what, rows))
    return a


def batchdecode_b(decoder, syndromes, errors, success=None, iters=None, posterior_ratio=None):
    """batchdecode!(decoder, syndromes, errors[, success]) -> (errors, success).

    syndromes: s x B (column = syndrome), errors: n x B overwritten in place; both numpy arrays
    of bool / uint8 / int64 (errors also float64).  Fortran-ordered arrays (Julia's layout) are
    passed to the library without a copy."""
    syn = _as_columns(syndromes, decoder.s, "syndromes")
    if not isinstance(errors, np.ndarray):
        raise TypeError("errors must be a numpy array (it is written in place)")
    err = _as_columns(errors, decoder.n, "errors")
    B = syn.shape[1]
    # @assert size(syndromes, 2) == size(errors, 2)   (belief_propagation.jl:221)
    assert syn.shape[1] == err.shape[1]
    if success is None:
        success = np.empty(B, dtype=np.bool_)          # abstract_decoder.jl:44-48
    # @assert size(syndromes, 2) == length(success)   (belief_propagation.jl:222)
    assert B == len(success)
    if not (isinstance(success, np.ndarray) and success.dtype == np.bool_ and success.flags.c_contiguous):
        raise TypeError("success must be a contiguous numpy bool vector")
    syn_f = np.asfortranarray(syn)
    syn_fmt = _fmt_of(syn_f, "syndromes")
    err_fmt = _fmt_of(err, "errors")
    err_f = err if err.flags.f_contiguous else np.zeros(err.shape, dtype=err.dtype, order="F")
    ratio = None
    if posterior_ratio is not None:
        ratio = posterior_ratio
        assert ratio.shape == (decoder.n, B) and ratio.dtype == np.float64 and ratio.flags.f_contiguous
    if iters is not None:
        assert iters.shape == (B,) and iters.dtype == np.int32
    if isinstance(decoder, BPOTSDecoder):
        if ratio is not None:
            raise ValueError("posterior_ratio is not an output of the BP-OTS decoder")
        decoder.decode_raw(B, syn_f, syn_fmt, max(decoder.s, 1), err_f, err_fmt, max(decoder.n, 1), success.view(np.uint8), iters)
    elif isinstance(decoder, BeliefPropagationOSDDecoder):
        # generic batchdecode! (abstract_decoder.jl:31-42) over decode!(::BeliefPropagationOSDDecoder)
        if ratio is not None:
            raise ValueError("posterior_ratio is not an output of the BP+OSD decoder")
        decoder.last_counters, decoder.last_osd_stats = decoder.bp_decoder.bposd_raw(
            B, syn_f, syn_fmt, max(decoder.s, 1), err_f, err_fmt, max(decoder.n, 1), success.view(np.uint8), iters)
    else:
        decoder.last_counters = decoder.decode_raw(B, syn_f, syn_fmt, max(decoder.s, 1), err_f, err_fmt,
                                                   max(decoder.n, 1), success.view(np.uint8), iters, ratio)
    if err_f is not err:
        err[...] = err_f
    return errors, success


def decode_b(decoder, syndrome):
    """decode!(decoder, syndrome) -> (err, converged); err is decoder.scratch.err (aliased,
    Float64 0.0/1.0, belief_propagation.jl:187) and scratch.log_probabs is refreshed."""
    syn = np.asarray(syndrome)
    if syn.ndim != 1 or syn.shape[0] != decoder.s:
        raise ValueError("syndrome must be a vector of length %d" % decoder.s)
    if syn.dtype not in (np.bool_, np.uint8, np.int8, np.int64):
        syn = syn.astype(np.int64)
    syn_f = np.asfortranarray(syn.reshape(decoder.s, 1))
    if isinstance(decoder, BPOTSDecoder):
        # decode!(::BPOTSDecoder) returns best_decisions (a Vector{Int}) and the converged flag (bpots_decoder.jl:291,339)
        out = np.zeros((decoder.n, 1), dtype=np.int64, order="F")
        conv = np.zeros(1, dtype=np.uint8)
        decoder.decode_raw(1, syn_f, _fmt_of(syn_f, "syndrome"), max(decoder.s, 1), out, _lib.FMT_I64, max(decoder.n, 1), conv)
        return out[:, 0], bool(conv[0])
    if isinstance(decoder, BeliefPropagationOSDDecoder):
        # decode!(::BeliefPropagationOSDDecoder) returns a fresh Bool vector and BP's flag (:60)
        out = np.zeros((decoder.n, 1), dtype=np.bool_, order="F")
        conv = np.zeros(1, dtype=np.uint8)
        decoder.last_counters, decoder.last_osd_stats = decoder.bp_decoder.bposd_raw(
            1, syn_f, _fmt_of(syn_f, "syndrome"), max(decoder.s, 1), out, _lib.FMT_U8, max(decoder.n, 1), conv)
        return out[:, 0], bool(conv[0])
    err = decoder.scratch.err.reshape(decoder.n, 1, order="F")
    conv = np.zeros(1, dtype=np.uint8)
    ratio = None
    if decoder.max_iters > 0:
        ratio = np.ones((decoder.n, 1), dtype=np.float64, order="F")
    decoder.last_counters = decoder.decode_raw(1, syn_f, _fmt_of(syn_f, "syndrome"), max(decoder.s, 1), err,
                                               _lib.FMT_F64, max(decoder.n, 1), conv, None, ratio)
    if ratio is not None and decoder.variant in ("minsum", "fast"):
        decoder.scratch.log_probabs[:] = ratio[:, 0]                      # posterior LLR log(P0/P1)
    elif ratio is not None:
        with np.errstate(all="ignore"):
            decoder.scratch.log_probabs[:] = np.log(1.0 / ratio[:, 0])   # belief_propagation.jl:163
    else:
        decoder.scratch.log_probabs[:] = 0.0
    return decoder.scratch.err, bool(conv[0])


def ler_curve(decoder, pers, shots, seed=12345, osd=False, match_prior=True):
    """Logical-error-rate sweep on the GPU (the loop of test/test_bp_decoder.jl:19-30 per error rate, with the batch
    sampled, decoded and scored on the device): for each physical error rate the prior is set to it (match_prior), `shots`
    errors are drawn from the Philox stream, decoded (BP, or BP+OSD-0 with osd=True) and compared with the truth.
    A BPOTSDecoder is swept with BP-OTS as the decoder (osd does not apply).
    Returns one dict per rate: the eight counters plus ler (= failures / shots), converged_frac and mean_iters."""
    bp = decoder.bp_decoder if isinstance(decoder, BeliefPropagationOSDDecoder) else decoder
    ots = isinstance(decoder, BPOTSDecoder)
    if ots and osd:
        raise ValueError("osd does not apply to the BP-OTS decoder")
    osd = osd or isinstance(decoder, BeliefPropagationOSDDecoder)
    prior = bp.per
    rows = []
    for k, per in enumerate(pers):
        if match_prior:
            bp.set_per(per)
        if ots:
            c = bp.sample_decode_score(shots, k * int(shots), seed, per)
        else:
            c = bp.sample_decode_score(shots, k * int(shots), seed, per, osd=osd)
        c.update(per=float(per), ler=c["failures"] / max(c["shots"], 1), converged_frac=c["converged"] / max(c["shots"], 1),
                 mean_iters=c["iterations"] / max(c["shots"], 1))
        rows.append(c)
    if match_prior:
        bp.set_per(prior)
    return rows
