"""rimphony_b200 -- B200-native evaluation of rimphony's eight polarized
synchrotron transfer coefficients.

Host-side mirror of the reference's public interface for this path (pkgw/rimphony):

* ``Coefficient``, ``Stokes``                      src/lib.rs:75-107
* ``PI, TWO_PI, MASS_ELECTRON, SPEED_LIGHT, ELECTRON_CHARGE``   src/lib.rs:55-67
* ``PowerLawDistribution(p).gamma_limits(..)``      src/power_law.rs:71-87
* ``ThermalJuettnerDistribution(t)``                src/thermal_juettner.rs:45-50
* ``PitchyPowerLawDistribution(p, k).gamma_limits(..)``  src/pitchy_pl.rs:73-90
* ``PitchyKappaDistribution(kappa, width, k).gamma_cutoff(..)``  src/pitchy_kappa.rs:70-85
* ``PitchyBrokenPowerLawDistribution(p1, p2, gamma_break, k).gamma_limits(..)``  a broken power law
  built as src/pitchy_pl.rs builds its single one (no counterpart in the reference)
* ``.full_calculation(logger)`` -> ``FullSynchrotronCalculator`` with the trait
  methods ``compute_dimensionless``, ``compute_cgs``, ``compute_all_dimensionless``,
  ``compute_all_cgs``                               src/lib.rs:150-247

Beyond the reference: ``transfer`` / ``transfer_device`` solve the polarized transfer equation
through rays of cells with the eight cgs coefficients, and
``FullSynchrotronCalculator.compute_stokes_cgs`` runs coefficients and transfer in one call
(the convention is in ``include/rimphony_b200.h`` and DESIGN.md section 13).

Same names, argument order and error behaviour (numerical failure = NaN in the
slot, never an exception).  What is new is that every distribution parameter,
``s`` and ``theta`` may be arrays: one call then evaluates a whole batch of
independent points on the GPU, which is the workload of
``examples/crank-out-pitchypl.rs:157-195``.

Everything here calls the C ABI of ``librimphony_b200.so``
(``include/rimphony_b200.h``); there is no CPU implementation.
"""
import ctypes
import enum
import math

import numpy as np

from . import _lib
from ._lib import RimphonyB200Error  # noqa: F401

# src/lib.rs:55-67
PI = math.pi
TWO_PI = 2.0 * math.pi
MASS_ELECTRON = 9.1093826e-28
SPEED_LIGHT = 2.99792458e10
ELECTRON_CHARGE = 4.80320680e-10

POWER_LAW, THERMAL_JUETTNER, PITCHY_PL, PITCHY_KAPPA, PITCHY_BROKEN_PL = 0, 1, 2, 3, 4

MODE_FAST, MODE_FAITHFUL, MODE_FUSED_ALL, MODE_FUSED = 0, 1, 2, 3

STATUS_NAN, STATUS_CAP_HIT, STATUS_NORM_FAILED, STATUS_REROUTED, STATUS_REFERENCE_DIVERGES = 1, 2, 4, 8, 16
DIAG_GAMMA_INTEGRAND, DIAG_GAMMA_INTEGRAL, DIAG_N_INTEGRAL, DIAG_GAMMA_CONTRIBUTION = 0, 1, 2, 3

COEFFICIENT_NAMES = ("j_I", "alpha_I", "j_Q", "alpha_Q", "j_V", "alpha_V", "rho_Q", "rho_V")


class Stokes(enum.IntEnum):
    """src/lib.rs:75-87"""
    I = 0  # noqa: E741
    Q = 1
    V = 2


class Coefficient(enum.IntEnum):
    """src/lib.rs:92-107"""
    Emission = 0
    Absorption = 1
    Faraday = 2


def output_slot(coeff, stokes):
    """Index into the ``[j_I, a_I, j_Q, a_Q, j_V, a_V, rho_Q, rho_V]`` vector (lib.rs:176-177)."""
    coeff, stokes = Coefficient(coeff), Stokes(stokes)
    if coeff == Coefficient.Faraday:
        return {Stokes.Q: 6, Stokes.V: 7}.get(stokes, -1)
    return 2 * int(stokes) + int(coeff)


def _as_column(x, n):
    a = np.asarray(x, dtype=np.float64)
    if a.ndim == 0:
        return a.reshape(1), True
    if a.shape != (n,):
        raise ValueError(f"parameter array has shape {a.shape}, expected ({n},) or a scalar")
    return np.ascontiguousarray(a), False


def make_options(mode=MODE_FAST, coeff_mask=0xFF, broadcast_mask=0, device=-1, epsrel_gamma=0.0,
                 epsrel_n=0.0, epsrel_heyvaerts_inner=0.0, epsrel_heyvaerts_outer=0.0):
    o = _lib.Options()
    o.struct_size = ctypes.sizeof(_lib.Options)
    o.mode = int(mode)
    o.coeff_mask = int(coeff_mask)
    o.param_broadcast_mask = int(broadcast_mask)
    o.device_plus_one = int(device) + 1 if int(device) >= 0 else 0
    o.epsrel_gamma = float(epsrel_gamma)
    o.epsrel_n = float(epsrel_n)
    o.epsrel_heyvaerts_inner = float(epsrel_heyvaerts_inner)
    o.epsrel_heyvaerts_outer = float(epsrel_heyvaerts_outer)
    return o


class BatchResult:
    """What one batched call returns.

    ``values`` is ``[8, n]`` in the order of ``COEFFICIENT_NAMES``; ``status`` is the
    per-point status word; ``lobes`` (``[4, n]``: j_V(+), j_V(-), alpha_V(+),
    alpha_V(-)), ``counters`` (``[2, n]``) and ``norm`` are present when asked for.
    """

    def __init__(self, values, status, lobes=None, counters=None, norm=None, kernel_ms=None):
        self.values = values
        self.status = status
        self.lobes = lobes
        self.counters = counters
        self.norm = norm
        self.kernel_ms = kernel_ms

    def rows(self):
        """``[n, 8]``: one ``compute_all_dimensionless`` vector per point."""
        return np.ascontiguousarray(self.values.T)


def compute_all_dimensionless_batch(kind, s, theta, params, *, mode=MODE_FAST, coeff_mask=0xFF, device=-1,
                                    extras=False, n_devices=None, **tolerances):
    """All eight dimensionless coefficients for ``n`` independent points (host arrays).

    ``params`` follows the column order of ``include/rimphony_b200.h``; scalars are
    broadcast on the device without being expanded on the host.  With
    ``n_devices`` the batch is sharded over that many GPUs of this box.
    """
    L = _lib.load()
    s = np.ascontiguousarray(np.atleast_1d(np.asarray(s, dtype=np.float64)))
    n = s.shape[0]
    theta = np.atleast_1d(np.asarray(theta, dtype=np.float64))
    if theta.shape == (1,) and n != 1:
        theta = np.full(n, theta[0])
    theta = np.ascontiguousarray(theta)
    if theta.shape != (n,):
        raise ValueError("s and theta must have the same length")
    cols, bmask = [], 0
    for j, p in enumerate(params):
        col, scalar = _as_column(p, n)
        cols.append(col)
        if scalar:
            bmask |= 1 << j
    ptrs = (_lib.c_double_p * max(len(cols), 1))(*[c.ctypes.data_as(_lib.c_double_p) for c in cols])
    opts = make_options(mode=mode, coeff_mask=coeff_mask, broadcast_mask=bmask, device=device, **tolerances)
    out = np.empty((8, n), dtype=np.float64)
    status = np.zeros(n, dtype=np.int32)
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)  # noqa: E731

    if n_devices is not None:
        rc = L.rimphony_b200_compute_all_dimensionless_multi(
            kind, n, dp(s), dp(theta), ptrs, len(cols), ctypes.byref(opts), dp(out),
            status.ctypes.data_as(_lib.c_int32_p), int(n_devices))
        _lib.check(rc)
        return BatchResult(out, status)

    lobes = counters = norm = None
    ex = None
    if extras:
        lobes = np.full((4, n), np.nan)
        counters = np.zeros((2, n), dtype=np.uint32)
        norm = np.full(n, np.nan)
        ex = _lib.Extras(dp(lobes), counters.ctypes.data_as(_lib.c_uint32_p), dp(norm))
    rc = L.rimphony_b200_compute_all_dimensionless_ex(
        kind, n, dp(s), dp(theta), ptrs, len(cols), ctypes.byref(opts), dp(out),
        status.ctypes.data_as(_lib.c_int32_p), ctypes.byref(ex) if ex is not None else None)
    _lib.check(rc)
    return BatchResult(out, status, lobes, counters, norm, last_kernel_ms(device))


def compute_all_dimensionless_device(kind, s, theta, params, out8, status=None, *, mode=MODE_FAST, coeff_mask=0xFF,
                                     stream=None, synchronize=True, **tolerances):
    """Device-resident variant: every argument is a CUDA ``torch.Tensor`` (float64,
    contiguous; ``status`` int32) already in HBM on the current device; nothing is
    copied.  ``stream`` is a ``torch.cuda.Stream`` (default: the library's own)."""
    import torch

    L = _lib.load()
    n = s.numel()
    for t in (s, theta, out8, *params):
        if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
            raise ValueError("device path needs contiguous float64 CUDA tensors")
    if theta.numel() != n or out8.numel() != 8 * n:
        raise ValueError("theta must have n elements and out8 8 n")
    bmask = 0
    for j, p in enumerate(params):
        if p.numel() == 1 and n != 1:
            bmask |= 1 << j
        elif p.numel() != n:
            raise ValueError("parameter column length mismatch")
    ptrs = (ctypes.c_void_p * max(len(params), 1))(*[p.data_ptr() for p in params])
    opts = make_options(mode=mode, coeff_mask=coeff_mask, broadcast_mask=bmask, device=s.device.index, **tolerances)
    rc = L.rimphony_b200_compute_all_dimensionless_device(
        kind, n, s.data_ptr(), theta.data_ptr(), ptrs, len(params), ctypes.byref(opts), out8.data_ptr(),
        status.data_ptr() if status is not None else None, None,
        stream.cuda_stream if stream is not None else None, 1 if synchronize else 0)
    _lib.check(rc)


def last_kernel_ms(device=-1):
    """Device time (ms) of the last batched call: normalise, Symphony, Heyvaerts, total."""
    buf = (ctypes.c_float * 4)()
    _lib.check(_lib.load().rimphony_b200_last_kernel_ms(int(device), buf))
    return tuple(buf)


def fp64_peak_tflops(device=-1):
    """Measured FP64 FMA throughput of the device in TFLOP/s (roofline denominator)."""
    out = ctypes.c_double()
    _lib.check(_lib.load().rimphony_b200_fp64_peak_tflops(int(device), ctypes.byref(out)))
    return out.value


def kernel_launch_count():
    return int(_lib.load().rimphony_b200_kernel_launch_count())


def device_count():
    return int(_lib.load().rimphony_b200_device_count())


def shutdown():
    _lib.load().rimphony_b200_shutdown()


def bessel_jn(n, x):
    """``(J_n(x), J_n'(x))`` by the device Leung evaluator (leung-bessel/src/lib.rs:56-75)."""
    n = np.ascontiguousarray(np.atleast_1d(n), dtype=np.float64)
    x = np.ascontiguousarray(np.atleast_1d(x), dtype=np.float64)
    if n.shape != x.shape:
        raise ValueError("n and x must have the same shape")
    j = np.empty_like(n)
    dj = np.empty_like(n)
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)  # noqa: E731
    _lib.check(_lib.load().rimphony_b200_bessel_jn(n.size, dp(n), dp(x), dp(j), dp(dj)))
    return j, dj


def dist_eval(kind, params, gamma, cos_xi):
    """``f, df/dgamma, df/dcos_xi`` with norm = 1 (trait DistributionFunction, lib.rs:111-146)."""
    gamma = np.ascontiguousarray(np.atleast_1d(gamma), dtype=np.float64)
    cos_xi = np.ascontiguousarray(np.atleast_1d(cos_xi), dtype=np.float64)
    pv = (ctypes.c_double * len(params))(*[float(p) for p in params])
    out = np.empty((3, gamma.size))
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)  # noqa: E731
    _lib.check(_lib.load().rimphony_b200_dist_eval(kind, pv, len(params), gamma.size, dp(gamma), dp(cos_xi), dp(out)))
    return out[0], out[1], out[2]


# ---------------------------------------------------------------------------
# Polarized transfer through rays of cells (include/rimphony_b200.h, DESIGN.md section 13).


def _ray_geometry(shape):
    """(n_rays, n_cells) of a per-cell array shape: [n] is n uniform slabs, [n_rays, n_cells] rays."""
    if len(shape) <= 1:
        return (int(np.prod(shape)) if shape else 1), 1
    if len(shape) == 2:
        return int(shape[0]), int(shape[1])
    raise ValueError(f"per-cell arrays are [n] (slabs) or [n_rays, n_cells], got shape {shape}")


def _per_cell(x, shape):
    return np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=np.float64), shape)).reshape(-1)


def transfer(coeffs_cgs, psi, ds, stokes0=None, *, device=-1):
    """Emergent Stokes ``(I, Q, U, V)`` of rays of cells with constant coefficients.

    ``coeffs_cgs`` is ``[8, n]`` (n uniform slabs) or ``[8, n_rays, n_cells]``, in the order of
    ``COEFFICIENT_NAMES`` and the units of ``compute_all_cgs``; cell 0 is where a ray enters.
    ``psi`` (radian) and ``ds`` (cm) broadcast to the cell shape; ``stokes0`` (incident, ``[4]`` or
    ``[4, n_rays]``) defaults to zero.  Returns ``(stokes [4, n_rays], status [n_rays])``; a ray
    with a non-finite input, a negative length or a cell out of range (``alpha_I ds`` below -10, or
    ``alpha_I ds``, ``|alpha_pol| ds``, ``|rho| ds`` above 1e102) is NaN with ``STATUS_NAN``.
    """
    c = np.asarray(coeffs_cgs, dtype=np.float64)
    if c.ndim not in (2, 3) or c.shape[0] != 8:
        raise ValueError(f"coeffs_cgs must be [8, n] or [8, n_rays, n_cells], got shape {c.shape}")
    cell_shape = c.shape[1:]
    n_rays, n_cells = _ray_geometry(cell_shape)
    c = np.ascontiguousarray(c).reshape(8, -1)
    psi, ds = _per_cell(psi, cell_shape), _per_cell(ds, cell_shape)
    s0 = None if stokes0 is None else np.ascontiguousarray(
        np.broadcast_to(np.asarray(stokes0, dtype=np.float64).reshape(4, -1), (4, n_rays)))
    out = np.empty((4, n_rays))
    status = np.zeros(n_rays, dtype=np.int32)
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)  # noqa: E731
    L = _lib.load()
    with _lib.current_device(device):
        rc = L.rimphony_b200_transfer(n_rays, n_cells, dp(c), dp(psi), dp(ds), dp(s0) if s0 is not None else None,
                                      dp(out), status.ctypes.data_as(_lib.c_int32_p))
    _lib.check(rc)
    return out, status


def transfer_device(coeffs8, psi, ds, stokes4, stokes0=None, status=None, *, stream=None, synchronize=True):
    """Device-resident ``transfer``: CUDA ``torch.Tensor`` arguments (float64, contiguous; ``status``
    int32) on one device, nothing copied.  ``coeffs8`` holds ``8 n`` values, ``psi`` and ``ds`` ``n``,
    ``stokes4`` (and ``stokes0``) ``4 n_rays``; ``n_cells = n / n_rays``.  ``stream`` is a
    ``torch.cuda.Stream`` (default: the library's own); with ``synchronize=False`` the call returns
    once the kernel is enqueued."""
    import torch

    n_rays = stokes4.numel() // 4
    n = psi.numel()
    for t in (coeffs8, psi, ds, stokes4) + ((stokes0,) if stokes0 is not None else ()):
        if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
            raise ValueError("device path needs contiguous float64 CUDA tensors")
    if status is not None and not (status.is_cuda and status.dtype == torch.int32 and status.is_contiguous()):
        raise ValueError("status must be a contiguous int32 CUDA tensor")
    tensors = (coeffs8, psi, ds, stokes4) + tuple(t for t in (stokes0, status) if t is not None)
    if any(t.device != stokes4.device for t in tensors):
        raise ValueError("all tensors must be on the device of stokes4")
    if status is not None and status.numel() != n_rays:
        raise ValueError("status must have n_rays values")
    if stokes4.numel() != 4 * n_rays or n_rays == 0 or n % n_rays or coeffs8.numel() != 8 * n or ds.numel() != n:
        raise ValueError("need coeffs8 of 8 n, psi and ds of n and stokes4 of 4 n_rays values, n_rays dividing n")
    if stokes0 is not None and stokes0.numel() != 4 * n_rays:
        raise ValueError("stokes0 must have 4 n_rays values")
    L = _lib.load()
    with _lib.current_device(stokes4.device.index):
        rc = L.rimphony_b200_transfer_device(
            n_rays, n // n_rays, coeffs8.data_ptr(), psi.data_ptr(), ds.data_ptr(),
            stokes0.data_ptr() if stokes0 is not None else None, stokes4.data_ptr(),
            status.data_ptr() if status is not None else None,
            stream.cuda_stream if stream is not None else None, 1 if synchronize else 0)
    _lib.check(rc)


class StokesResult:
    """What ``compute_stokes_cgs`` returns: ``stokes`` ``[4, n_rays]`` (I, Q, U, V), ``status``
    ``[n_rays]`` (the OR of the cells' status words, ``STATUS_NAN`` if the ray is NaN) and ``coeffs``,
    the cells' cgs coefficients, ``[8, n_rays, n_cells]``."""

    def __init__(self, stokes, status, coeffs):
        self.stokes = stokes
        self.status = status
        self.coeffs = coeffs


def compute_stokes_cgs(kind, nu, b, n_e, theta, psi, ds, params, *, mode=MODE_FAST, device=-1, **tolerances):
    """Coefficients and transfer in one call on the device (``rimphony_b200_compute_stokes_cgs``).
    The per-cell arguments and the distribution's parameter columns broadcast together to ``[n]``
    (n uniform slabs) or ``[n_rays, n_cells]``; rays enter with no radiation.  Returns a
    ``StokesResult``."""
    shape = np.broadcast_shapes(*(np.shape(x) for x in (nu, b, n_e, theta, psi, ds)),
                                *(np.shape(p) for p in params))
    n_rays, n_cells = _ray_geometry(shape)
    cols = [_per_cell(x, shape) for x in (nu, b, n_e, theta, psi, ds)]
    pcols, bmask = [], 0
    for j, p in enumerate(params):
        if np.ndim(p) == 0:
            pcols.append(np.full(1, float(p)))
            bmask |= 1 << j
        else:
            pcols.append(_per_cell(p, shape))
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)  # noqa: E731
    ptrs = (_lib.c_double_p * max(len(pcols), 1))(*[dp(c) for c in pcols])
    opts = make_options(mode=mode, broadcast_mask=bmask, device=device, **tolerances)
    stokes = np.empty((4, n_rays))
    coeffs = np.empty((8, n_rays * n_cells))
    status = np.zeros(n_rays, dtype=np.int32)
    rc = _lib.load().rimphony_b200_compute_stokes_cgs(
        kind, n_rays, n_cells, *[dp(c) for c in cols], ptrs, len(pcols), ctypes.byref(opts), dp(stokes), dp(coeffs),
        status.ctypes.data_as(_lib.c_int32_p))
    _lib.check(rc)
    return StokesResult(stokes, status, coeffs.reshape(8, n_rays, n_cells))


# ---------------------------------------------------------------------------
# The reference's calculator trait and distribution types.


class SynchrotronCalculator:
    """trait SynchrotronCalculator (src/lib.rs:150-210)."""

    def compute_dimensionless(self, coeff, stokes, s, theta):
        raise NotImplementedError

    def compute_cgs(self, coeff, stokes, nu, b, n_e, theta):
        # lib.rs:163-173
        nu_c = ELECTRON_CHARGE * np.asarray(b, dtype=np.float64) / (TWO_PI * MASS_ELECTRON * SPEED_LIGHT)
        val = self.compute_dimensionless(coeff, stokes, nu / nu_c, theta)
        if Coefficient(coeff) == Coefficient.Emission:
            return val * n_e * nu
        return val * n_e / nu

    def compute_all_dimensionless(self, s, theta):
        # the provided method of the trait (lib.rs:178-191): [j_I, alpha_I, j_Q, alpha_Q, j_V, alpha_V, rho_Q, rho_V]
        order = [(Coefficient.Emission, Stokes.I), (Coefficient.Absorption, Stokes.I), (Coefficient.Emission, Stokes.Q),
                 (Coefficient.Absorption, Stokes.Q), (Coefficient.Emission, Stokes.V), (Coefficient.Absorption, Stokes.V),
                 (Coefficient.Faraday, Stokes.Q), (Coefficient.Faraday, Stokes.V)]
        return np.stack([np.asarray(self.compute_dimensionless(c, st, s, theta), dtype=np.float64) for c, st in order],
                        axis=-1)

    def compute_all_cgs(self, nu, b, n_e, theta):
        # lib.rs:196-209
        nu_c = ELECTRON_CHARGE * np.asarray(b, dtype=np.float64) / (TWO_PI * MASS_ELECTRON * SPEED_LIGHT)
        rv = np.array(self.compute_all_dimensionless(nu / nu_c, theta), dtype=np.float64)
        scale_j = n_e * nu
        scale_a = n_e / nu
        for c in (0, 2, 4):
            rv[..., c] = rv[..., c] * scale_j
        for c in (1, 3, 5, 6, 7):
            rv[..., c] = rv[..., c] * scale_a
        return rv


class FullSynchrotronCalculator(SynchrotronCalculator):
    """The fully detailed double-integral calculator (src/lib.rs:231-247).

    With scalar arguments the methods return what the reference returns (a float,
    or the ``[f64; 8]`` vector).  With array arguments they return one result per
    point: ``[n]`` or ``[n, 8]``.
    """

    def __init__(self, distrib, logger=None, mode=MODE_FAST, device=-1):
        self.distrib = distrib
        self.logger = logger
        self.mode = mode
        self.device = device

    def _batch(self, s, theta, coeff_mask, extras=False):
        return compute_all_dimensionless_batch(self.distrib.KIND, s, theta, self.distrib._columns(),
                                               mode=self.mode, coeff_mask=coeff_mask, device=self.device,
                                               extras=extras)

    def _is_scalar_call(self, s, theta):
        return np.ndim(s) == 0 and np.ndim(theta) == 0 and self.distrib._is_scalar()

    def compute_dimensionless(self, coeff, stokes, s, theta):
        slot = output_slot(coeff, stokes)
        scalar = self._is_scalar_call(s, theta)
        if slot < 0:  # (Faraday, I): lib.rs:239-240
            return math.nan if scalar else np.full(np.broadcast(s, theta).shape, np.nan)
        s_arr = np.atleast_1d(np.asarray(s, dtype=np.float64))
        if s_arr.shape == (1,) and not self.distrib._is_scalar():
            s_arr = np.full(self.distrib._length(), s_arr[0])
        res = self._batch(s_arr, theta, 1 << slot)
        return float(res.values[slot, 0]) if scalar else res.values[slot]

    def compute_all_dimensionless(self, s, theta):
        scalar = self._is_scalar_call(s, theta)
        s_arr = np.atleast_1d(np.asarray(s, dtype=np.float64))
        if s_arr.shape == (1,) and not self.distrib._is_scalar():
            s_arr = np.full(self.distrib._length(), s_arr[0])
        res = self._batch(s_arr, theta, 0xFF)
        return res.rows()[0] if scalar else res.rows()

    def compute_all_dimensionless_batch(self, s, theta, extras=False):
        """The additive batch entry point (SURVEY.md section 8-b): returns a ``BatchResult``."""
        return self._batch(np.atleast_1d(np.asarray(s, dtype=np.float64)), theta, 0xFF, extras=extras)

    def compute_stokes_cgs(self, nu, b, n_e, theta, psi, ds):
        """Emergent Stokes ``(I, Q, U, V)`` of uniform slabs (arguments of shape ``[n]`` or scalars) or
        of rays of cells (``[n_rays, n_cells]``, cell 0 where the ray enters) of this distribution:
        the coefficients of ``compute_all_cgs`` in every cell, then ``transfer`` through the cells of
        length ``ds`` (cm) with field angle ``psi``, in one call on the device.  Returns a
        ``StokesResult``; ``.stokes`` is ``[4, n_rays]``."""
        return compute_stokes_cgs(self.distrib.KIND, nu, b, n_e, theta, psi, ds, self.distrib._columns(),
                                  mode=self.mode, device=self.device)


    # -- diagnostics of the Symphony double integral (src/lib.rs:249-299) ----------------
    # Scalar arguments give the reference's scalar; arrays give one value per element (one
    # warp each).  The distribution must be a single one (scalar parameters).

    def _diagnostic(self, what, coeff, stokes, s, theta, a, b=None):
        if not self.distrib._is_scalar():
            raise ValueError("the Symphony diagnostics take a single distribution (scalar parameters)")
        if Coefficient(coeff) == Coefficient.Faraday:
            raise ValueError("the Symphony diagnostics are defined for emission and absorption")
        scalar = np.ndim(a) == 0 and (b is None or np.ndim(b) == 0)
        if b is None:
            a_arr = np.ascontiguousarray(np.atleast_1d(a), dtype=np.float64)
            b_arr = None
        else:
            a_b, b_b = np.broadcast_arrays(np.atleast_1d(np.asarray(a, dtype=np.float64)),
                                           np.atleast_1d(np.asarray(b, dtype=np.float64)))
            a_arr, b_arr = np.ascontiguousarray(a_b), np.ascontiguousarray(b_b)
        pv = np.array([float(np.asarray(c).reshape(-1)[0]) for c in self.distrib._columns()], dtype=np.float64)
        out = np.full(a_arr.shape, np.nan)
        L = _lib.load()
        _lib.check(L.rimphony_b200_diagnostic_symphony(
            self.distrib.KIND, pv.ctypes.data_as(_lib.c_double_p), len(pv), int(coeff), int(stokes), float(s),
            float(theta), what, a_arr.size, a_arr.ctypes.data_as(_lib.c_double_p),
            b_arr.ctypes.data_as(_lib.c_double_p) if b_arr is not None else None,
            out.ctypes.data_as(_lib.c_double_p), None))
        return float(out.reshape(-1)[0]) if scalar else out

    def diagnostic_symphony_n_integral(self, coeff, stokes, s, theta, n_lo, n_hi):
        """QAG over n of the gamma integral (lib.rs:254-260).  The reference returns a
        ``GslResult``; its ``Err`` is NaN here."""
        return self._diagnostic(DIAG_N_INTEGRAL, coeff, stokes, s, theta, n_lo, n_hi)

    def diagnostic_symphony_gamma_integral(self, coeff, stokes, s, theta, n):
        """G(n), the gamma integral at harmonic number n (lib.rs:266-272)."""
        return self._diagnostic(DIAG_GAMMA_INTEGRAL, coeff, stokes, s, theta, n)

    def diagnostic_symphony_gamma_integrand(self, coeff, stokes, s, theta, n, gamma):
        """The integrand at (n, gamma) (lib.rs:278-284)."""
        return self._diagnostic(DIAG_GAMMA_INTEGRAND, coeff, stokes, s, theta, n, gamma)

    def diagnostic_symphony_gamma_contribution(self, coeff, stokes, s, theta, gamma):
        """The double integral sliced the other way: all n at fixed gamma (lib.rs:291-297)."""
        return self._diagnostic(DIAG_GAMMA_CONTRIBUTION, coeff, stokes, s, theta, gamma)


class _PowerLawHighFrequency(SynchrotronCalculator):
    """``HighFrequencyApproximation`` of src/power_law.rs:119-170: closed-form Faraday coefficients
    (Huang & Shcherbakov 2011), a checker for the full calculation.  Host arithmetic, as in the
    reference; everything but (Faraday, Q) and (Faraday, V) is NaN."""

    def __init__(self, distrib):
        self.distrib = distrib

    def compute_dimensionless(self, coeff, stokes, s, theta):
        d = self.distrib
        s, theta = np.asarray(s, dtype=np.float64), np.asarray(theta, dtype=np.float64)
        p, gmin = np.asarray(d.p, dtype=np.float64), np.asarray(d.gamma_min, dtype=np.float64)
        if Coefficient(coeff) != Coefficient.Faraday or Stokes(stokes) == Stokes.I:
            out = np.full(np.broadcast(s, theta, p).shape, np.nan)
        elif Stokes(stokes) == Stokes.Q:  # power_law.rs:146-152
            out = (0.0085 * 2.0 / (p - 2.0) * ((s / (np.sin(theta) * gmin ** 2)) ** ((p - 2.0) / 2.0) - 1.0) *
                   (p - 1.0) / gmin ** (1.0 - p) * (np.sin(theta) / s) ** ((p + 2.0) / 2.0))
        else:  # power_law.rs:155-161
            out = 0.017 * (np.log(gmin) * (p - 1.0)) / ((p + 1.0) * gmin ** 2) / s * np.sin(theta)
        return float(out) if np.ndim(out) == 0 else out


class _ThermalHighFrequency(SynchrotronCalculator):
    """``HighFrequencyApproximation`` of src/thermal_juettner.rs:92-142 (Heyvaerts' high-frequency
    limits with K_0, K_1, K_2 of 1/T)."""

    def __init__(self, distrib):
        self.distrib = distrib

    def compute_dimensionless(self, coeff, stokes, s, theta):
        from scipy.special import kve  # exponentially scaled: the ratios below are scale-free

        s, theta = np.asarray(s, dtype=np.float64), np.asarray(theta, dtype=np.float64)
        t = np.asarray(self.distrib.t, dtype=np.float64)
        inv_t = 1.0 / t
        factor = 2.0 * ELECTRON_CHARGE * ELECTRON_CHARGE / MASS_ELECTRON
        k0, k1, k2 = kve(0, inv_t), kve(1, inv_t), kve(2, inv_t)
        if Coefficient(coeff) != Coefficient.Faraday or Stokes(stokes) == Stokes.I:
            out = np.full(np.broadcast(s, theta, t).shape, np.nan)
        elif Stokes(stokes) == Stokes.Q:  # thermal_juettner.rs:112-127
            out = factor * np.sin(theta) ** 2 * (k1 + 6.0 * t * k2) / (2.0 * SPEED_LIGHT * s ** 2 * k2)
        else:  # thermal_juettner.rs:129-141
            out = factor * np.cos(theta) * k0 / (SPEED_LIGHT * s * k2)
        return float(out) if np.ndim(out) == 0 else out


class _Distribution:
    KIND = -1

    def _columns(self):
        raise NotImplementedError

    def _is_scalar(self):
        return all(np.ndim(c) == 0 for c in self._columns())

    def _length(self):
        for c in self._columns():
            if np.ndim(c) != 0:
                return len(c)
        return 1

    def full_calculation(self, logger=None, mode=MODE_FAST, device=-1):
        """Consumes the parameters and returns the calculator.  The normalisation
        integral the reference computes here (e.g. power_law.rs:93-103) runs on the
        device at the start of every batched call, once per point."""
        return FullSynchrotronCalculator(self, logger, mode=mode, device=device)

    def calc_f(self, gamma, cos_xi):
        """trait DistributionFunction::calc_f with norm = 1 (lib.rs:141)."""
        f, _, _ = dist_eval(self.KIND, self._scalar_columns(), gamma, cos_xi)
        return f if np.ndim(gamma) else float(f[0])

    def calc_f_derivatives(self, gamma, cos_xi):
        """trait DistributionFunction::calc_f_derivatives with norm = 1 (lib.rs:145)."""
        _, a, b = dist_eval(self.KIND, self._scalar_columns(), gamma, cos_xi)
        return (a, b) if np.ndim(gamma) else (float(a[0]), float(b[0]))

    def _scalar_columns(self):
        if not self._is_scalar():
            raise ValueError("calc_f needs scalar distribution parameters")
        return [float(c) for c in self._columns()]

    def __repr__(self):
        return f"{type(self).__name__}({', '.join(repr(c) for c in self._columns())})"


class PowerLawDistribution(_Distribution):
    """src/power_law.rs:27-87: dN/dgamma ~ gamma^-p exp(-gamma/gamma_cutoff) on [gamma_min, gamma_max]."""
    KIND = POWER_LAW

    def __init__(self, p):
        self.p = p
        self.gamma_min, self.gamma_max, self._gamma_cutoff = 1.0, 1e12, 1e10

    def gamma_limits(self, gamma_min, gamma_max, gamma_cutoff):
        self.gamma_min, self.gamma_max, self._gamma_cutoff = gamma_min, gamma_max, gamma_cutoff
        return self

    def _columns(self):
        return [self.p, self.gamma_min, self.gamma_max, self._gamma_cutoff]

    def high_freq_approximation(self):
        """src/power_law.rs:112-115"""
        return _PowerLawHighFrequency(self)


class ThermalJuettnerDistribution(_Distribution):
    """src/thermal_juettner.rs:23-50: f ~ exp(-gamma/T)."""
    KIND = THERMAL_JUETTNER

    def __init__(self, t):
        self.t = t

    def _columns(self):
        return [self.t]

    def high_freq_approximation(self):
        """src/thermal_juettner.rs:74-77"""
        return _ThermalHighFrequency(self)


class PitchyPowerLawDistribution(_Distribution):
    """src/pitchy_pl.rs:22-90: the power law times sin^k(pitch angle)."""
    KIND = PITCHY_PL

    def __init__(self, p, k):
        self.p, self.k = p, k
        self.gamma_min, self.gamma_max, self._gamma_cutoff = 1.0, 1e12, 1e10

    def gamma_limits(self, gamma_min, gamma_max, gamma_cutoff):
        self.gamma_min, self.gamma_max, self._gamma_cutoff = gamma_min, gamma_max, gamma_cutoff
        return self

    def _columns(self):
        return [self.p, self.k, self.gamma_min, self.gamma_max, self._gamma_cutoff]


class PitchyBrokenPowerLawDistribution(_Distribution):
    """A broken power law times sin^k(pitch angle), built as src/pitchy_pl.rs builds its single one:
    dN/dgamma ~ gamma^-p1 below gamma_break and gamma_break^(p2 - p1) gamma^-p2 from it on (continuous
    at the break), times exp(-gamma/gamma_cutoff), on [gamma_min, gamma_max].  p1 = p2, or a break at
    or above gamma_max, is PitchyPowerLawDistribution(p1, k)."""
    KIND = PITCHY_BROKEN_PL

    def __init__(self, p1, p2, gamma_break, k):
        self.p1, self.p2, self.gamma_break, self.k = p1, p2, gamma_break, k
        self.gamma_min, self.gamma_max, self._gamma_cutoff = 1.0, 1e12, 1e10

    def gamma_limits(self, gamma_min, gamma_max, gamma_cutoff):
        self.gamma_min, self.gamma_max, self._gamma_cutoff = gamma_min, gamma_max, gamma_cutoff
        return self

    def _columns(self):
        return [self.p1, self.p2, self.gamma_break, self.k, self.gamma_min, self.gamma_max, self._gamma_cutoff]


class PitchyKappaDistribution(_Distribution):
    """src/pitchy_kappa.rs:28-85: relativistic kappa distribution times sin^k(pitch angle)."""
    KIND = PITCHY_KAPPA

    def __init__(self, kappa, width, k):
        self.kappa, self.width, self.k = kappa, width, k
        self._gamma_cutoff = 1e10

    def gamma_cutoff(self, gamma_cutoff):
        self._gamma_cutoff = gamma_cutoff
        return self

    def _columns(self):
        return [self.kappa, self.width, self.k, self._gamma_cutoff]


from .sampler import Sampler, synthetic_batch  # noqa: E402,F401
