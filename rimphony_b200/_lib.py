"""ctypes loader for the C-ABI shared library (include/rimphony_b200.h).

There is no Python or CPU implementation behind this package: if the CUDA
library is missing or no B200 is visible, the calls fail loudly.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# RIMPHONY_B200_LIB: an alternative build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("RIMPHONY_B200_LIB") or os.path.join(HERE, "librimphony_b200.so")

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int32_p = ctypes.POINTER(ctypes.c_int32)
c_uint32_p = ctypes.POINTER(ctypes.c_uint32)


class Options(ctypes.Structure):
    """struct rimphony_b200_options"""
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("mode", ctypes.c_int32),
        ("coeff_mask", ctypes.c_uint32),
        ("param_broadcast_mask", ctypes.c_uint32),
        ("device_plus_one", ctypes.c_int32),
        ("reserved0", ctypes.c_int32),
        ("epsrel_gamma", ctypes.c_double),
        ("epsrel_n", ctypes.c_double),
        ("epsrel_heyvaerts_inner", ctypes.c_double),
        ("epsrel_heyvaerts_outer", ctypes.c_double),
    ]


class Extras(ctypes.Structure):
    """struct rimphony_b200_extras"""
    _fields_ = [
        ("lobes4", c_double_p),
        ("counters", c_uint32_p),
        ("norm", c_double_p),
    ]


# every symbol include/rimphony_b200.h declares
EXPORTED_SYMBOLS = (
    "rimphony_b200_compute_all_dimensionless",
    "rimphony_b200_compute_all_dimensionless_ex",
    "rimphony_b200_compute_all_dimensionless_device",
    "rimphony_b200_compute_all_dimensionless_multi",
    "rimphony_b200_compute_dimensionless",
    "rimphony_b200_compute_cgs",
    "rimphony_b200_diagnostic_symphony",
    "rimphony_b200_bessel_jn",
    "rimphony_b200_dist_eval",
    "rimphony_b200_transfer",
    "rimphony_b200_transfer_device",
    "rimphony_b200_compute_stokes_cgs",
    "rimphony_b200_last_kernel_ms",
    "rimphony_b200_fp64_peak_tflops",
    "rimphony_b200_kernel_launch_count",
    "rimphony_b200_device_count",
    "rimphony_b200_abi_version",
    "rimphony_b200_last_error",
    "rimphony_b200_shutdown",
)

_lib = None


class RimphonyB200Error(RuntimeError):
    """Infrastructure error reported by the CUDA library (never a numerical one)."""


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RimphonyB200Error(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C rimphony_b200/csrc).  There is no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    i32, i64, dbl, vp = ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p
    pp = ctypes.POINTER(c_double_p)
    OP, EP = ctypes.POINTER(Options), ctypes.POINTER(Extras)
    L.rimphony_b200_compute_all_dimensionless.argtypes = [i32, i64, c_double_p, c_double_p, pp, i32, OP, c_double_p, c_int32_p]
    L.rimphony_b200_compute_all_dimensionless_ex.argtypes = [i32, i64, c_double_p, c_double_p, pp, i32, OP, c_double_p, c_int32_p, EP]
    # device-pointer variant: raw addresses
    L.rimphony_b200_compute_all_dimensionless_device.argtypes = [i32, i64, vp, vp, ctypes.POINTER(vp), i32, OP, vp, vp, EP, vp, i32]
    L.rimphony_b200_compute_all_dimensionless_multi.argtypes = [i32, i64, c_double_p, c_double_p, pp, i32, OP, c_double_p, c_int32_p, i32]
    L.rimphony_b200_compute_dimensionless.argtypes = [i32, c_double_p, i32, i32, i32, dbl, dbl, c_double_p]
    L.rimphony_b200_compute_cgs.argtypes = [i32, c_double_p, i32, i32, i32, dbl, dbl, dbl, dbl, c_double_p]
    L.rimphony_b200_diagnostic_symphony.argtypes = [i32, c_double_p, i32, i32, i32, dbl, dbl, i32, i64, c_double_p,
                                                    c_double_p, c_double_p, c_int32_p]
    L.rimphony_b200_bessel_jn.argtypes = [i64, c_double_p, c_double_p, c_double_p, c_double_p]
    L.rimphony_b200_dist_eval.argtypes = [i32, c_double_p, i32, i64, c_double_p, c_double_p, c_double_p]
    L.rimphony_b200_transfer.argtypes = [i64, i64, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_int32_p]
    L.rimphony_b200_transfer_device.argtypes = [i64, i64, vp, vp, vp, vp, vp, vp, vp, i32]
    L.rimphony_b200_compute_stokes_cgs.argtypes = [i32, i64, i64, c_double_p, c_double_p, c_double_p, c_double_p,
                                                   c_double_p, c_double_p, pp, i32, OP, c_double_p, c_double_p,
                                                   c_int32_p]
    L.rimphony_b200_last_kernel_ms.argtypes = [i32, ctypes.POINTER(ctypes.c_float)]
    L.rimphony_b200_fp64_peak_tflops.argtypes = [i32, c_double_p]
    L.rimphony_b200_kernel_launch_count.restype = ctypes.c_uint64
    L.rimphony_b200_last_error.restype = ctypes.c_char_p
    L.rimphony_b200_shutdown.restype = None
    _lib = L
    return L


class current_device:
    """Within the block, the calling thread's current CUDA device (of the CUDA runtime the library uses) is
    `device`; -1 leaves it as it is.  The entry points without an options struct run there."""

    def __init__(self, device):
        self.device, self.saved = int(device), None

    def __enter__(self):
        if self.device >= 0:
            L, cur = load(), ctypes.c_int(-1)
            if L.cudaGetDevice(ctypes.byref(cur)) != 0 or L.cudaSetDevice(self.device) != 0:
                raise RimphonyB200Error(f"cannot select CUDA device {self.device}")
            self.saved = cur.value
        return self

    def __exit__(self, *exc):
        if self.saved is not None:
            load().cudaSetDevice(self.saved)
        return False


def check(rc):
    if rc != 0:
        raise RimphonyB200Error(load().rimphony_b200_last_error().decode("utf-8", "replace"))
