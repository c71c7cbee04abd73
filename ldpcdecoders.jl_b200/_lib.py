"""ctypes binding of libldpcb200.so -- exactly the symbols include/ldpcb200.h declares.

The library is the product: if it is missing or no CUDA device is usable, calls fail loudly.
There is no CPU fallback anywhere in this package.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LDPCB200_LIB") or os.path.join(HERE, "lib", "libldpcb200.so")   # (override: kernel experiments)

OK, EINVAL, ECUDA, ENODEVICE, EUNSUPPORTED, ENOMEM = range(6)
FMT_U8, FMT_I64, FMT_BITS, FMT_PACKED32, FMT_F64 = range(5)
FAMILY_AUTO, FAMILY_SMEM, FAMILY_GLOBAL = range(3)
VARIANT_EXACT, VARIANT_MINSUM, VARIANT_FAST32 = 0, 1, 2
NUM_COUNTERS = 4
NUM_OSD_STATS = 3      # processed, pivots, columns visited
CTR_DECODED, CTR_CONVERGED, CTR_ITERATIONS = 0, 1, 2

# every exported symbol of include/ldpcb200.h (tests check the .so against this list)
SYMBOLS = [
    "ldpcb200_last_error", "ldpcb200_version", "ldpcb200_device_count", "ldpcb200_create",
    "ldpcb200_destroy", "ldpcb200_info", "ldpcb200_set_option", "ldpcb200_decode_batch",
    "ldpcb200_decode_device", "ldpcb200_sample_device", "ldpcb200_score_device",
    "ldpcb200_launch_count", "ldpcb200_selftest_division",
    "ldpcb200_bposd_decode_batch", "ldpcb200_osd0_device", "ldpcb200_kernel_profile",
    "ldpcb200_set_logicals", "ldpcb200_score_logical_device", "ldpcb200_set_per", "ldpcb200_sample_decode_score", "ldpcb200_bpots_decode_batch",
    "ldpcb200_kernel_time", "ldpcb200_bpots_device", "ldpcb200_sample_bpots_score",
]
NUM_HARNESS_COUNTERS = 8
HARNESS_FIELDS = ("shots", "converged", "iterations", "exact_matches", "syndrome_satisfied", "failures", "residual_weight", "osd_processed")


class Info(ctypes.Structure):
    _fields_ = [("s", ctypes.c_int64), ("n", ctypes.c_int64), ("E", ctypes.c_int64),
                ("max_check_degree", ctypes.c_int32), ("max_var_degree", ctypes.c_int32),
                ("family", ctypes.c_int32), ("ndev", ctypes.c_int32), ("sm_count", ctypes.c_int32),
                ("ctas_per_sm", ctypes.c_int32), ("threads_per_cta", ctypes.c_int32),
                ("smem_bytes", ctypes.c_int32), ("slots", ctypes.c_int32),
                ("syn_words", ctypes.c_int32), ("err_words", ctypes.c_int32),
                ("message_bytes", ctypes.c_int64), ("kernel_mode", ctypes.c_int32), ("prefetch_distance", ctypes.c_int32),
                ("kernel_rev", ctypes.c_int32), ("counters_via_nccl", ctypes.c_int32),
                ("bpots_workspace_bytes", ctypes.c_int64)]


class LibraryError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libldpcb200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load():
    """Load the shared library (built in-tree by build.py).  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            "%s not found: build it with `python __graft_entry__.py build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, u64, dbl = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double
    lib.ldpcb200_last_error.restype = ctypes.c_char_p
    lib.ldpcb200_last_error.argtypes = []
    lib.ldpcb200_version.restype = ctypes.c_int
    lib.ldpcb200_device_count.argtypes = [ctypes.POINTER(i32)]
    lib.ldpcb200_create.argtypes = [i64, i64, vp, vp, i32, dbl, i32, i32, vp, i32, ctypes.POINTER(vp)]
    lib.ldpcb200_destroy.argtypes = [vp]
    lib.ldpcb200_info.argtypes = [vp, ctypes.POINTER(Info)]
    lib.ldpcb200_set_option.argtypes = [vp, ctypes.c_char_p, i64]
    lib.ldpcb200_decode_batch.argtypes = [vp, i64, vp, i32, i64, vp, i32, i64, vp, vp, vp, vp]
    lib.ldpcb200_decode_device.argtypes = [vp, i32, i64, vp, vp, vp, vp, vp, vp, vp]
    lib.ldpcb200_bposd_decode_batch.argtypes = [vp, i64, vp, i32, i64, vp, i32, i64, vp, vp, vp, vp]
    lib.ldpcb200_osd0_device.argtypes = [vp, i32, i64, vp, vp, vp, vp, vp, vp]
    lib.ldpcb200_sample_device.argtypes = [vp, i32, i64, i64, u64, dbl, vp, vp, vp]
    lib.ldpcb200_score_device.argtypes = [vp, i32, i64, vp, vp, vp, vp, vp]
    lib.ldpcb200_bpots_decode_batch.argtypes = [vp, i64, vp, i32, i64, vp, i32, i64, vp, vp, i32, dbl]
    lib.ldpcb200_bpots_device.argtypes = [vp, i32, i64, vp, vp, vp, vp, vp, i32, dbl, vp]
    lib.ldpcb200_sample_bpots_score.argtypes = [vp, i64, i64, u64, dbl, i32, dbl, ctypes.POINTER(i64)]
    lib.ldpcb200_set_logicals.argtypes = [vp, i64, vp, vp, i32]
    lib.ldpcb200_score_logical_device.argtypes = [vp, i32, i64, vp, vp, vp, vp, vp]
    lib.ldpcb200_set_per.argtypes = [vp, dbl]
    lib.ldpcb200_sample_decode_score.argtypes = [vp, i64, i64, u64, dbl, i32, ctypes.POINTER(i64)]
    lib.ldpcb200_kernel_profile.argtypes = [vp, i32, ctypes.POINTER(i64), i32]
    lib.ldpcb200_kernel_time.argtypes = [vp, i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i64), i32]
    lib.ldpcb200_launch_count.argtypes = [vp, ctypes.POINTER(i64)]
    lib.ldpcb200_selftest_division.argtypes = [i32, i32, u64, u64, ctypes.POINTER(u64)]   # mismatches[4]
    for name in SYMBOLS:
        if name != "ldpcb200_last_error":
            getattr(lib, name).restype = ctypes.c_int
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise LibraryError(rc, load().ldpcb200_last_error().decode("utf-8", "replace"))
