"""ctypes binding of the CPU oracle -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product package
``rimphony_b200`` never does (``tests/test_no_oracle_in_product.py`` checks).

``oracle/Makefile`` builds ``oracle/_build/liboracle.so``, the restatement of
``src/symphony.rs`` / ``src/heyvaerts.rs`` / the four distributions.  It links the
reference's own ``leung-bessel/src/bessel.c`` (``oracle/_ref/libleung_ref.so``, prebuilt
or compiled in place from the reference) and, where neither is at hand, ``leung_bessel.c``,
a C restatement of it; ``bessel_source()`` says which.
"""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "liboracle.so")

POWER_LAW, THERMAL_JUETTNER, PITCHY_PL, PITCHY_KAPPA = 0, 1, 2, 3
EMISSION, ABSORPTION, FARADAY = 0, 1, 2
STOKES_I, STOKES_Q, STOKES_V = 0, 1, 2

_c_double_p = ctypes.POINTER(ctypes.c_double)


class Dist(ctypes.Structure):
    _fields_ = [
        ("kind", ctypes.c_int),
        ("p", ctypes.c_double),
        ("k", ctypes.c_double),
        ("gamma_min", ctypes.c_double),
        ("gamma_max", ctypes.c_double),
        ("inv_gamma_cutoff", ctypes.c_double),
        ("kappa", ctypes.c_double),
        ("width", ctypes.c_double),
        ("inv_kappa_width", ctypes.c_double),
        ("neg_inverse_t", ctypes.c_double),
        ("norm", ctypes.c_double),
    ]


class Stats(ctypes.Structure):
    _fields_ = [
        ("n_symphony_integrand", ctypes.c_uint64),
        ("n_gamma_qag", ctypes.c_uint64),
        ("n_gamma_qag_failed", ctypes.c_uint64),
        ("n_chunks", ctypes.c_uint64),
        ("max_gamma_intervals", ctypes.c_uint64),
        ("max_n_intervals", ctypes.c_uint64),
        ("n_heyvaerts_element", ctypes.c_uint64),
        ("n_heyvaerts_qag", ctypes.c_uint64),
        ("n_heyvaerts_jy", ctypes.c_uint64),
        ("hey_nr_val", ctypes.c_double),
        ("hey_qr_val", ctypes.c_double),
        ("hey_fail_stage", ctypes.c_int),
        ("hey_fail_outer_status", ctypes.c_int),
        ("hey_fail_inner_status", ctypes.c_int),
        ("hey_fail_inner_kind", ctypes.c_int),
        ("hey_fail_lo", ctypes.c_double),
        ("hey_fail_hi", ctypes.c_double),
        ("hey_fail_inner_var", ctypes.c_double),
        ("hey_nan_kind", ctypes.c_int),   # 0 none, 1 NR, 2 QR
        ("hey_nan_sigma", ctypes.c_double),
        ("hey_nan_pomega", ctypes.c_double),
        ("hey_nan_x", ctypes.c_double),
        ("hey_nan_gamma", ctypes.c_double),
        ("hey_nan_mu", ctypes.c_double),
        ("hey_nan_value", ctypes.c_double),
    ]


def build(force=False):
    """Run oracle/Makefile unless liboracle.so is already built."""
    if force or not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", HERE, "-s"])
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = ctypes.CDLL(LIB_PATH)
    D = ctypes.POINTER(Dist)
    S = ctypes.POINTER(Stats)
    dbl, i32 = ctypes.c_double, ctypes.c_int
    L.orc_dist_init.argtypes = [D, i32, _c_double_p, i32]
    L.orc_dist_init.restype = i32
    L.orc_calc_f.argtypes = [D, dbl, dbl]
    L.orc_calc_f.restype = dbl
    L.orc_calc_f_derivatives.argtypes = [D, dbl, dbl, _c_double_p, _c_double_p]
    L.orc_calc_f_derivatives.restype = None
    L.orc_symphony.argtypes = [D, i32, i32, dbl, dbl, S]
    L.orc_symphony.restype = dbl
    L.orc_symphony_lobes.argtypes = [D, i32, i32, dbl, dbl, S, _c_double_p]
    L.orc_symphony_lobes.restype = dbl
    L.orc_heyvaerts.argtypes = [D, i32, dbl, dbl, S]
    L.orc_heyvaerts.restype = dbl
    L.orc_compute_dimensionless.argtypes = [D, i32, i32, dbl, dbl, S]
    L.orc_compute_dimensionless.restype = dbl
    L.orc_compute_cgs.argtypes = [D, i32, i32, dbl, dbl, dbl, dbl, S]
    L.orc_compute_cgs.restype = dbl
    L.orc_compute_all_dimensionless.argtypes = [D, dbl, dbl, _c_double_p, _c_double_p, S]
    L.orc_compute_all_dimensionless.restype = None
    L.orc_batch_compute_all_dimensionless.argtypes = [
        i32, ctypes.c_int64, _c_double_p, _c_double_p, ctypes.POINTER(_c_double_p), i32,
        ctypes.c_uint, _c_double_p, _c_double_p, i32]
    L.orc_batch_compute_all_dimensionless.restype = i32
    L.orc_num_threads.restype = i32
    L.orc_set_epsrel.argtypes = [dbl, dbl]
    L.orc_set_epsrel.restype = None
    for name in ("orc_ref_bessel_j", "orc_ref_bessel_dj", "orc_test_bessel_i"):
        getattr(L, name).argtypes = [dbl, dbl]
        getattr(L, name).restype = dbl
    L.orc_test_bessel_jy.argtypes = [dbl, dbl, _c_double_p, _c_double_p]
    L.orc_test_bessel_jy.restype = None
    L.orc_test_bessel_k2.argtypes = [dbl]
    L.orc_test_bessel_k2.restype = dbl
    L.orc_test_pitch_angle_integral.argtypes = [dbl]
    L.orc_test_pitch_angle_integral.restype = dbl
    L.orc_test_qag.argtypes = [i32, dbl, dbl, dbl, dbl, _c_double_p, _c_double_p,
                               ctypes.POINTER(i32)]
    L.orc_test_qag.restype = i32
    L.orc_test_deriv.argtypes = [i32, dbl, dbl, dbl]
    L.orc_test_deriv.restype = dbl
    L.orc_symphony_diagnostic.argtypes = [ctypes.POINTER(Dist), i32, i32, dbl, dbl, i32, dbl, dbl]
    L.orc_symphony_diagnostic.restype = dbl
    L.orc_gk31_tables.argtypes = [_c_double_p, _c_double_p, _c_double_p]
    L.orc_gk31_tables.restype = None
    _lib = L
    return L


def make_dist(kind, params):
    d = Dist()
    arr = (ctypes.c_double * len(params))(*[float(p) for p in params])
    status = lib().orc_dist_init(ctypes.byref(d), kind, arr, len(params))
    if status != 0:
        raise ValueError(f"oracle: distribution init failed (status {status})")
    return d


def compute_dimensionless(dist, coeff, stokes, s, theta, stats=None):
    sp = ctypes.byref(stats) if stats is not None else None
    return lib().orc_compute_dimensionless(ctypes.byref(dist), coeff, stokes, s, theta, sp)


DIAG_GAMMA_INTEGRAND, DIAG_GAMMA_INTEGRAL, DIAG_N_INTEGRAL, DIAG_GAMMA_CONTRIBUTION = range(4)


def symphony_diagnostic(dist, coeff, stokes, s, theta, what, a, b=0.0):
    """FullSynchrotronCalculator::diagnostic_symphony_* (src/lib.rs:254-298)."""
    return lib().orc_symphony_diagnostic(ctypes.byref(dist), coeff, stokes, s, theta, what, a, b)


def compute_cgs(dist, coeff, stokes, nu, b, n_e, theta):
    return lib().orc_compute_cgs(ctypes.byref(dist), coeff, stokes, nu, b, n_e, theta, None)


def compute_all_dimensionless(dist, s, theta, stats=None):
    out = (ctypes.c_double * 8)()
    lobes = (ctypes.c_double * 4)()
    sp = ctypes.byref(stats) if stats is not None else None
    lib().orc_compute_all_dimensionless(ctypes.byref(dist), s, theta, out, lobes, sp)
    return np.array(out[:]), np.array(lobes[:])


def batch(kind, s, theta, params, coeff_mask=0xFF, n_threads=0):
    """All eight coefficients for each point.  Returns (out[8, n], lobes[4, n]).

    ``params`` is a sequence of per-point arrays in the C-ABI order documented in
    include/rimphony_b200.h.
    """
    s = np.ascontiguousarray(s, dtype=np.float64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    n = s.shape[0]
    cols = [np.ascontiguousarray(np.broadcast_to(np.asarray(p, dtype=np.float64), (n,))) for p in params]
    ptrs = (_c_double_p * len(cols))(*[c.ctypes.data_as(_c_double_p) for c in cols])
    out = np.full((8, n), np.nan)
    lobes = np.full((4, n), np.nan)
    lib().orc_batch_compute_all_dimensionless(
        kind, n, s.ctypes.data_as(_c_double_p), theta.ctypes.data_as(_c_double_p), ptrs, len(cols),
        coeff_mask, out.ctypes.data_as(_c_double_p), lobes.ctypes.data_as(_c_double_p), n_threads)
    return out, lobes


def set_epsrel(symphony=0.0, heyvaerts=0.0):
    """Stability studies only (tests/golden/make_stability.py): the epsrel of the oracle's QAG calls;
    0 restores the reference's 1e-3."""
    lib().orc_set_epsrel(symphony, heyvaerts)


def num_threads():
    return lib().orc_num_threads()


def bessel_source():
    """"reference" when liboracle.so runs the reference's own bessel.c (oracle/_ref/libleung_ref.so),
    "restatement" when it runs oracle/leung_bessel.c."""
    lib()
    with open("/proc/self/maps") as f:
        return "reference" if "libleung_ref.so" in f.read() else "restatement"


def ref_bessel_j(n, x):
    return lib().orc_ref_bessel_j(n, x)


def ref_bessel_dj(n, x):
    return lib().orc_ref_bessel_dj(n, x)
