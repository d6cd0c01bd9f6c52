"""ctypes binding of the CPU oracle with the pitchy broken power law -- TEST INFRASTRUCTURE ONLY.

``Makefile`` builds ``_build/libbpl_oracle.so``: oracle/rimphony_oracle.c unchanged, with its distribution
functions extended by PITCHY_BROKEN_PL (bpl_oracle.c), so that the reference's Symphony and Heyvaerts
algorithms run on the new distribution function.  Every other kind gives what ``oracle.oracle`` gives.
The functions below take and return what their namesakes in ``oracle.oracle`` do.
"""
import ctypes
import os
import subprocess

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "libbpl_oracle.so")

POWER_LAW, THERMAL_JUETTNER, PITCHY_PL, PITCHY_KAPPA, PITCHY_BROKEN_PL = 0, 1, 2, 3, 4

_lib = None


def lib():
    global _lib
    if _lib is None:
        base = O.lib()   # builds the oracle first: its choice of J_n evaluator is linked here as well
        subprocess.check_call(["make", "-C", HERE, "-s"])
        L = ctypes.CDLL(LIB_PATH)
        for name in ("orc_dist_init", "orc_calc_f", "orc_calc_f_derivatives", "orc_compute_all_dimensionless",
                     "orc_batch_compute_all_dimensionless", "orc_num_threads", "orc_set_epsrel"):
            f, g = getattr(L, name), getattr(base, name)
            f.argtypes, f.restype = g.argtypes, g.restype
        _lib = L
    return _lib


def make_dist(kind, params):
    d = O.Dist()
    arr = (ctypes.c_double * len(params))(*[float(p) for p in params])
    status = lib().orc_dist_init(ctypes.byref(d), kind, arr, len(params))
    if status != 0:
        raise ValueError(f"oracle: distribution init failed (status {status})")
    return d


def calc_f(dist, gamma, cos_xi):
    return lib().orc_calc_f(ctypes.byref(dist), gamma, cos_xi)


def calc_f_derivatives(dist, gamma, cos_xi):
    a, b = ctypes.c_double(), ctypes.c_double()
    lib().orc_calc_f_derivatives(ctypes.byref(dist), gamma, cos_xi, ctypes.byref(a), ctypes.byref(b))
    return a.value, b.value


def compute_all_dimensionless(dist, s, theta):
    out = (ctypes.c_double * 8)()
    lobes = (ctypes.c_double * 4)()
    lib().orc_compute_all_dimensionless(ctypes.byref(dist), s, theta, out, lobes, None)
    return np.array(out[:]), np.array(lobes[:])


def batch(kind, s, theta, params, coeff_mask=0xFF, n_threads=0):
    s = np.ascontiguousarray(s, dtype=np.float64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    n = s.shape[0]
    cols = [np.ascontiguousarray(np.broadcast_to(np.asarray(p, dtype=np.float64), (n,))) for p in params]
    dp = ctypes.POINTER(ctypes.c_double)
    ptrs = (dp * len(cols))(*[c.ctypes.data_as(dp) for c in cols])
    out = np.full((8, n), np.nan)
    lobes = np.full((4, n), np.nan)
    lib().orc_batch_compute_all_dimensionless(kind, n, s.ctypes.data_as(dp), theta.ctypes.data_as(dp), ptrs, len(cols),
                                              coeff_mask, out.ctypes.data_as(dp), lobes.ctypes.data_as(dp), n_threads)
    return out, lobes


def set_epsrel(symphony=0.0, heyvaerts=0.0):
    lib().orc_set_epsrel(symphony, heyvaerts)


def num_threads():
    return lib().orc_num_threads()
