"""Polarized radiative transfer through rays of cells: the propagator of rimphony_b200/csrc/rb_transfer.cuh
(built for the host by tests/hostemu_transfer and for the device by inst_transfer.cu), the C entry points
rimphony_b200_transfer, _transfer_device and _compute_stokes_cgs, and their Python surface.

The reference is independent of the closed form: mpmath at 50 digits exponentiates the Van Loan matrix
[[-K ds, J ds], [0, 0]], whose top rows are [P, Q J], cell after cell.  The bound is the normwise error relative
to max(|I|, |S0|) of 1e-12 (1 + |rho| ds): the second factor is the conditioning of the phase of a Faraday or
conversion rotation through |rho| ds radian."""
import ctypes
import functools
import io
import itertools
import math
import os
import re
import subprocess

import mpmath as mp
import numpy as np
import pytest

import rimphony_b200 as R
from rimphony_b200 import _lib, examples

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NEW_SYMBOLS = ("rimphony_b200_transfer", "rimphony_b200_transfer_device", "rimphony_b200_compute_stokes_cgs")
TOL = 1e-12


# ---------------------------------------------------------------------------
# the host build of rb_transfer.cuh and the mpmath reference


@functools.lru_cache(maxsize=None)
def _emu_lib():
    subprocess.run(["make", "-s", "-C", os.path.join(HERE, "hostemu_transfer")], check=True)
    return ctypes.CDLL(os.path.join(HERE, "hostemu_transfer", "_build", "libhostemu_transfer.so"))


def _rays(coeffs, psi, ds, stokes0):
    c = np.asarray(coeffs, dtype=np.float64)
    cell_shape = c.shape[1:]
    if c.ndim == 2:
        c = c[:, :, None]
    n_rays, n_cells = c.shape[1:]
    psi = np.ascontiguousarray(np.broadcast_to(np.asarray(psi, dtype=np.float64), cell_shape)).reshape(-1)
    ds = np.ascontiguousarray(np.broadcast_to(np.asarray(ds, dtype=np.float64), cell_shape)).reshape(-1)
    s0 = None if stokes0 is None else np.ascontiguousarray(
        np.broadcast_to(np.asarray(stokes0, dtype=np.float64).reshape(4, -1), (4, n_rays)))
    return np.ascontiguousarray(c).reshape(8, -1), psi, ds, s0, n_rays, n_cells


def emu_transfer(coeffs, psi, ds, stokes0=None):
    """The host build, with the arguments of R.transfer: returns (stokes [4, n_rays], status)."""
    c, psi, ds, s0, n_rays, n_cells = _rays(coeffs, psi, ds, stokes0)
    out = np.empty((4, n_rays))
    status = np.zeros(n_rays, dtype=np.int32)
    dp = lambda a: a.ctypes.data_as(_lib.c_double_p)  # noqa: E731
    _emu_lib().emu_transfer(ctypes.c_longlong(n_rays), ctypes.c_longlong(n_cells), dp(c), dp(psi), dp(ds),
                            dp(s0) if s0 is not None else None, dp(out), status.ctypes.data_as(_lib.c_int32_p))
    return out, status


def _ref_cell(k8, psi, ds, S):
    jI, aI, jQ, aQ, jV, aV, rQ, rV = [mp.mpf(float(v)) for v in k8]
    # the double values of cos 2 psi and sin 2 psi, as the propagator has them
    c, s2 = mp.mpf(float(np.cos(2.0 * psi))), mp.mpf(float(np.sin(2.0 * psi)))
    K = [[aI, aQ * c, aQ * s2, aV], [aQ * c, aI, rV, -rQ * s2], [aQ * s2, -rV, aI, rQ * c], [aV, rQ * s2, -rQ * c, aI]]
    J = [jI, jQ * c, jQ * s2, jV]
    d = mp.mpf(float(ds))
    A = mp.zeros(5, 5)
    for i in range(4):
        for j in range(4):
            A[i, j] = -K[i][j] * d
        A[i, 4] = J[i] * d
    E = mp.expm(A)
    return [mp.fsum(E[i, j] * S[j] for j in range(4)) + E[i, 4] for i in range(4)]


def ref_transfer(coeffs, psi, ds, stokes0=None, dps=50):
    """The mpmath reference, with the arguments of R.transfer: stokes [4, n_rays]."""
    c, psi, ds, s0, n_rays, n_cells = _rays(coeffs, psi, ds, stokes0)
    out = np.empty((4, n_rays))
    with mp.workdps(dps):
        for r in range(n_rays):
            S = [mp.mpf(0)] * 4 if s0 is None else [mp.mpf(float(v)) for v in s0[:, r]]
            for k in range(n_cells):
                p = r * n_cells + k
                S = _ref_cell(c[:, p], psi[p], ds[p], S)
            out[:, r] = [float(v) for v in S]
    return out


def normwise_error(got, want, stokes0=None):
    """Per ray: |got - want| / max(|I|, |S0|)."""
    scale = np.abs(want[0])
    if stokes0 is not None:
        scale = np.maximum(scale, np.linalg.norm(np.broadcast_to(np.asarray(stokes0).reshape(4, -1), want.shape), axis=0))
    return np.linalg.norm(got - want, axis=0) / scale


# ---------------------------------------------------------------------------
# the grid of the regimes: every combination of optical depth, degree of polarized absorption, Faraday depth,
# the geometry of a = (alpha_Q, alpha_V) and r = (rho_Q, rho_V), and the field angle

GRID_TAU = (0.0, 1e-12, 1e-6, 1.0, 30.0, 700.0, 1e4)
GRID_POL = (0.0, 0.5, 1.0 - 1e-12, 1.0)
GRID_RHO = (0.0, 1e-8, 1.0, 1e3, 1e6)
GRID_GEOMETRY = ("parallel", "perpendicular", "generic")
GRID_PSI = (0.0, math.pi / 4, 0.37)
STOKES0 = np.array([2.0, 0.5, -0.7, 0.3])


def _grid_cell(tau, pol, rho, geometry, ds=1.0):
    ua = np.array([0.6, 0.8])  # (Q, V)
    ur = {"parallel": ua, "perpendicular": np.array([-0.8, 0.6]),
          "generic": np.array([0.3, -0.9]) / math.hypot(0.3, 0.9)}[geometry]
    a_i = tau / ds
    a, r = pol * a_i * ua, rho / ds * ur
    return np.array([1.0, a_i, 0.3, a[0], 0.2, a[1], r[0], r[1]])


@functools.lru_cache(maxsize=None)
def grid():
    """(coeffs [8, n], psi [n], |rho| ds [n]) of the single-cell grid, and its reference with and without S0."""
    cells, psis, rhos = [], [], []
    for tau, pol, rho, geometry, psi in itertools.product(GRID_TAU, GRID_POL, GRID_RHO, GRID_GEOMETRY, GRID_PSI):
        cells.append(_grid_cell(tau, pol, rho, geometry))
        psis.append(psi)
        rhos.append(rho)
    coeffs, psi, rho = np.array(cells).T.copy(), np.array(psis), np.array(rhos)
    return coeffs, psi, rho, ref_transfer(coeffs, psi, 1.0), ref_transfer(coeffs, psi, 1.0, STOKES0)


@functools.lru_cache(maxsize=None)
def ray_cases():
    """Rays of 2 and of 64 random physical cells (alpha_I >= |a|), with their reference and sum of |rho| ds."""
    rng = np.random.default_rng(20261022)
    out = []
    for n_rays, n_cells in ((24, 2), (4, 64)):
        tau = 10.0 ** rng.uniform(-6, 1.5, (n_rays, n_cells))
        ds = 10.0 ** rng.uniform(10, 16, (n_rays, n_cells))
        a_i = tau / ds
        pol = rng.uniform(0, 1, (n_rays, n_cells))
        ang = rng.uniform(0, 2 * np.pi, (2, n_rays, n_cells))
        rho = 10.0 ** rng.uniform(-8, 3, (n_rays, n_cells)) / ds
        j_i = 10.0 ** rng.uniform(-22, -18, (n_rays, n_cells))
        jpol = rng.uniform(0, 1, (n_rays, n_cells)) * j_i
        jang = rng.uniform(0, 2 * np.pi, (n_rays, n_cells))
        coeffs = np.array([j_i, a_i, jpol * np.cos(jang), pol * a_i * np.cos(ang[0]), jpol * np.sin(jang),
                           pol * a_i * np.sin(ang[0]), rho * np.cos(ang[1]), rho * np.sin(ang[1])])
        psi = rng.uniform(-np.pi, np.pi, (n_rays, n_cells))
        s0 = np.array([1e-5, 2e-6, -3e-6, 1e-6])
        out.append((coeffs, psi, ds, s0, ref_transfer(coeffs, psi, ds, s0), (rho * ds).sum(axis=1)))
    return out


def _check_grid(transfer_fn, tol):
    coeffs, psi, rho, want0, want1 = grid()
    for s0, want in ((None, want0), (STOKES0, want1)):
        got, status = transfer_fn(coeffs, psi, 1.0, s0)
        assert (status == 0).all()
        err = normwise_error(got, want, s0)
        bound = tol * (1.0 + rho)
        worst = np.argmax(err / bound)
        assert (err <= bound).all(), (s0 is not None, coeffs[:, worst], psi[worst], got[:, worst], want[:, worst],
                                      err[worst])


def _check_rays(transfer_fn, tol):
    for coeffs, psi, ds, s0, want, rho in ray_cases():
        got, status = transfer_fn(coeffs, psi, ds, s0)
        assert (status == 0).all()
        err = normwise_error(got, want, s0)
        assert (err <= tol * (1.0 + rho)).all(), (coeffs.shape, err, rho)


# ---------------------------------------------------------------------------
# CPU: the host build


def test_host_build_matches_mpmath_on_the_grid():
    _check_grid(emu_transfer, TOL)


def test_host_build_matches_mpmath_on_rays_of_2_and_64_cells():
    _check_rays(emu_transfer, TOL)


def test_reference_is_converged():
    """50 and 80 digits agree far below the bound, on the hardest corners of the grid."""
    cells = np.array([_grid_cell(1e4, 1.0 - 1e-12, 1e6, "generic"), _grid_cell(1.0, 1.0, 1.0, "perpendicular"),
                      _grid_cell(700.0, 0.5, 1e3, "parallel"), _grid_cell(1e-12, 1.0, 1e6, "generic")]).T
    a = ref_transfer(cells, 0.37, 1.0, STOKES0, dps=50)
    b = ref_transfer(cells, 0.37, 1.0, STOKES0, dps=80)
    assert (normwise_error(a, b, STOKES0) < 1e-25).all()


def test_thin_cell_is_j_ds():
    k8 = _grid_cell(1e-9, 0.5, 1e-9, "generic")
    for ds in (1e-3, 1e-6):
        got, _ = emu_transfer((k8 / [1, ds, 1, ds, 1, ds, ds, ds])[:, None], 0.2, ds)
        j = np.array([k8[0], k8[2] * math.cos(0.4), k8[2] * math.sin(0.4), k8[4]]) * ds
        assert np.abs(got[:, 0] - j).max() <= 1e-8 * np.abs(j).max()  # the O(alpha ds) = 1e-9 correction


def test_thick_cell_is_the_source_function():
    """alpha_I ds >> 700: e^{-x} underflows; S = K^-1 J, finite."""
    for pol in (0.0, 0.5, 0.9):
        k8 = _grid_cell(1.0, pol, 0.3, "generic")
        psi = 0.3
        got, status = emu_transfer(k8[:, None], psi, 1e5)
        c, s2 = math.cos(2 * psi), math.sin(2 * psi)
        jI, aI, jQ, aQ, jV, aV, rQ, rV = k8
        K = np.array([[aI, aQ * c, aQ * s2, aV], [aQ * c, aI, rV, -rQ * s2], [aQ * s2, -rV, aI, rQ * c],
                      [aV, rQ * s2, -rQ * c, aI]])
        want = np.linalg.solve(K, [jI, jQ * c, jQ * s2, jV])
        assert status[0] == 0 and np.isfinite(got).all()
        assert np.abs(got[:, 0] - want).max() <= 1e-13 * np.abs(want).max()


def _thick_cell(tau, pol, rho):
    """A cell of alpha_I = 1e-3 / cm and length tau / alpha_I, and its K and J."""
    k8 = _grid_cell(1.0, pol, rho, "generic") * np.array([1, 1e-3, 1, 1e-3, 1, 1e-3, 1e-3, 1e-3])
    c, s2 = math.cos(0.6), math.sin(0.6)
    jI, aI, jQ, aQ, jV, aV, rQ, rV = k8
    K = np.array([[aI, aQ * c, aQ * s2, aV], [aQ * c, aI, rV, -rQ * s2], [aQ * s2, -rV, aI, rQ * c],
                  [aV, rQ * s2, -rQ * c, aI]])
    return k8, tau / 1e-3, K, np.array([jI, jQ * c, jQ * s2, jV])


@pytest.mark.parametrize("tau", [1e5, 1e10, 1e15, 1e50, 1e100])
def test_very_thick_cells_are_the_source_function(tau):
    """alpha_I ds up to 1e100: the psi_k(z) ~ z^{-k-1} of the integrated propagator are carried scaled by
    z^{k+1}, so they never underflow; with and without polarized absorption and Faraday rotation."""
    for pol, rho in itertools.product((0.0, 0.5, 0.9), (0.0, 1.0, 10.0)):
        k8, ds, K, J = _thick_cell(tau, pol, rho)
        got, status = emu_transfer(k8[:, None], 0.3, ds)
        want = np.linalg.solve(K, J)
        assert status[0] == 0 and np.abs(got[:, 0] - want).max() <= 1e-13 * np.abs(want).max(), (pol, rho, got, want)


@pytest.mark.parametrize("tau", [1e10, 1e15])
def test_very_thick_fully_polarized_cells_match_mpmath(tau):
    """|a| = alpha_I (1 - 1e-12) and |a| = alpha_I: the slowly absorbed mode decays as e^{-(alpha_I - Lambda_1) ds},
    whose exponent a relative rounding of Lambda_1 moves by eps alpha_I ds; that is the bound here."""
    for pol in (1.0 - 1e-12, 1.0):
        k8, ds, _, _ = _thick_cell(tau, pol, 0.0)
        got, status = emu_transfer(k8[:, None], 0.3, ds)
        want = ref_transfer(k8[:, None], 0.3, ds)
        assert status[0] == 0
        assert normwise_error(got, want)[0] <= 1e-12 + 4 * np.finfo(float).eps * tau, (pol, got, want)


def test_depths_beyond_the_range_are_nan_with_the_status_bit():
    """Above 1e102 the closed form's X^3 and 1 / X^3 leave FP64; below alpha_I ds = -10 (a masing cell of gain
    above e^10) its series alternate.  Both are flagged rather than wrong."""
    for tau, pol, rho in ((1e103, 0.5, 0.0), (1e50, 0.5, 1e60), (1e-3, 0.0, 1e106)):
        k8, ds, _, _ = _thick_cell(tau, pol, rho)
        got, status = emu_transfer(k8[:, None], 0.3, ds)
        assert np.isnan(got).all() and status[0] == R.STATUS_NAN, (tau, pol, rho)
    k8 = _grid_cell(-10.5, 0.5, 1.0, "generic")
    got, status = emu_transfer(k8[:, None], 0.3, 1.0, STOKES0)
    assert np.isnan(got).all() and status[0] == R.STATUS_NAN
    got, status = emu_transfer(k8[:, None], 0.3, 10.0 / 10.5, STOKES0)  # alpha_I ds = -10: in range
    assert status[0] == 0 and np.isfinite(got).all()


def test_negative_absorption_matches_mpmath():
    """Masing cells, -10 <= alpha_I ds < 0, with |a| <= |alpha_I|."""
    cells = [_grid_cell(tau, pol, rho, geometry) for tau, pol, rho, geometry in
             itertools.product((-1e-6, -0.1, -1.0, -5.0, -10.0), (0.0, 0.5, 1.0), (0.0, 1.0, 1e3),
                               ("generic", "parallel", "perpendicular"))]
    coeffs = np.array(cells).T.copy()
    got, status = emu_transfer(coeffs, 0.37, 1.0, STOKES0)
    want = ref_transfer(coeffs, 0.37, 1.0, STOKES0)
    rho = np.hypot(coeffs[6], coeffs[7])
    assert (status == 0).all() and (normwise_error(got, want, STOKES0) <= TOL * (1 + rho)).all()


def _rot(q, u, angle):
    return q * math.cos(angle) - u * math.sin(angle), q * math.sin(angle) + u * math.cos(angle)


def test_faraday_rotation_turns_q_into_u():
    """psi = 0, no absorption or emission, rho_V only: (Q, U) turns through +rho_V ds."""
    s0 = np.array([1.0, 0.6, 0.2, 0.3])
    for rv, ds in ((0.7, 1.0), (2.0, 3.0), (1e3, 1.1)):
        got, _ = emu_transfer(np.array([0, 0, 0, 0, 0, 0, 0, rv])[:, None], 0.0, ds, s0)
        q, u = _rot(s0[1], s0[2], rv * ds)
        assert np.allclose(got[:, 0], [1.0, q, u, 0.3], rtol=0, atol=1e-15 * (1 + rv * ds))


def test_conversion_turns_u_into_v():
    """psi = 0, rho_Q only: (U, V) turns through +rho_Q ds."""
    s0 = np.array([1.0, 0.6, 0.2, 0.3])
    for rq, ds in ((0.7, 1.0), (2.0, 3.0), (1e3, 1.1)):
        got, _ = emu_transfer(np.array([0, 0, 0, 0, 0, 0, rq, 0])[:, None], 0.0, ds, s0)
        u, v = _rot(s0[2], s0[3], rq * ds)
        assert np.allclose(got[:, 0], [1.0, 0.6, u, v], rtol=0, atol=1e-15 * (1 + rq * ds))


def test_changing_psi_turns_q_u_through_twice_the_angle():
    k8 = _grid_cell(1.0, 0.6, 2.0, "generic")
    s0 = np.array([1.0, 0.3, -0.2, 0.1])
    for psi, delta in ((0.0, 0.3), (0.37, -1.1), (1.2, math.pi / 4)):
        a, _ = emu_transfer(k8[:, None], psi, 0.8, s0)
        q0, u0 = _rot(s0[1], s0[2], 2 * delta)
        b, _ = emu_transfer(k8[:, None], psi + delta, 0.8, np.array([s0[0], q0, u0, s0[3]]))
        q, u = _rot(a[1, 0], a[2, 0], 2 * delta)
        assert np.allclose(b[:, 0], [a[0, 0], q, u, a[3, 0]], rtol=0, atol=1e-14)
        # and with no incident radiation
        a, _ = emu_transfer(k8[:, None], psi, 0.8)
        b, _ = emu_transfer(k8[:, None], psi + delta, 0.8)
        q, u = _rot(a[1, 0], a[2, 0], 2 * delta)
        assert np.allclose(b[:, 0], [a[0, 0], q, u, a[3, 0]], rtol=0, atol=1e-14 * abs(a[0, 0]))


def test_physical_inputs_give_physical_stokes_vectors():
    """alpha_I >= |a| and j_I >= |j_pol|: I >= sqrt(Q^2 + U^2 + V^2) within rounding."""
    rng = np.random.default_rng(7)
    n = 4000
    a_i = 10.0 ** rng.uniform(-3, 2, n)
    pol = rng.uniform(0, 1, n) * a_i
    ang = rng.uniform(0, 2 * np.pi, (3, n))
    rho = 10.0 ** rng.uniform(-3, 4, n)
    j_i = rng.uniform(0.1, 1, n)
    jpol = rng.uniform(0, 1, n) * j_i
    coeffs = np.array([j_i, a_i, jpol * np.cos(ang[2]), pol * np.cos(ang[0]), jpol * np.sin(ang[2]),
                       pol * np.sin(ang[0]), rho * np.cos(ang[1]), rho * np.sin(ang[1])])
    got, _ = emu_transfer(coeffs, rng.uniform(0, np.pi, n), 10.0 ** rng.uniform(-2, 2, n))
    assert (got[0] >= np.linalg.norm(got[1:], axis=0) * (1 - 1e-12)).all()


def test_identical_cells_equal_one_cell_of_the_total_length():
    for tau, pol, rho, geometry in ((0.3, 0.5, 2.0, "generic"), (30.0, 1.0, 10.0, "parallel"),
                                    (1e-6, 0.9, 40.0, "perpendicular")):
        k8 = _grid_cell(tau, pol, rho, geometry)
        for n in (2, 7, 64):
            ray, _ = emu_transfer(np.repeat(k8[:, None, None], n, axis=2), 0.37, 1.0 / n, STOKES0)
            one, _ = emu_transfer(k8[:, None], 0.37, 1.0, STOKES0)
            assert normwise_error(ray, one, STOKES0)[0] <= 1e-13 * (1 + rho), (tau, pol, rho, n)


def test_bad_inputs_give_nan_and_the_status_bit():
    k8 = _grid_cell(1.0, 0.5, 1.0, "generic")
    coeffs = np.repeat(k8[:, None, None], 3, axis=2).repeat(6, axis=1)
    ds = np.full((6, 3), 0.5)
    psi = np.full((6, 3), 0.1)
    s0 = np.tile(STOKES0[:, None], (1, 6))
    coeffs[1, 1, 2] = np.nan
    coeffs[7, 2, 0] = np.inf
    ds[3, 1] = -1e-300
    psi[4, 2] = -np.inf
    s0[2, 5] = np.nan
    got, status = emu_transfer(coeffs, psi, ds, s0)
    assert np.isfinite(got[:, 0]).all() and status[0] == 0
    assert np.isnan(got[:, 1:]).all() and (status[1:] == R.STATUS_NAN).all()
    # a zero length is allowed and changes nothing
    got, status = emu_transfer(k8[:, None], 0.1, 0.0, STOKES0)
    assert status[0] == 0 and np.array_equal(got[:, 0], STOKES0)


# ---------------------------------------------------------------------------
# CPU: the entry points without a device


def test_new_symbols_are_declared_everywhere():
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rimphony_b200.h")).read(), flags=re.S)
    ffi = open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read()
    L = _lib.load()
    for name in NEW_SYMBOLS:
        assert re.search(rf"\b{name}\s*\(", header) and name in _lib.EXPORTED_SYMBOLS and f"pub fn {name}(" in ffi
        assert hasattr(L, name)
    assert L.rimphony_b200_abi_version() == 2
    # the matrix is written out in the header, so the sign convention can be read off
    assert "| alpha_Q c    alpha_I      rho_V       -rho_Q s2   |" in open(os.path.join(ROOT, "include",
                                                                                   "rimphony_b200.h")).read()


def test_bad_arguments_are_infrastructure_errors():
    L = _lib.load()
    buf = (ctypes.c_double * 64)()
    st = (ctypes.c_int32 * 8)()
    assert L.rimphony_b200_transfer(-1, 1, buf, buf, buf, None, buf, st) != 0
    assert b"negative" in L.rimphony_b200_last_error()
    assert L.rimphony_b200_transfer(1, -1, buf, buf, buf, None, buf, st) != 0
    assert L.rimphony_b200_transfer(1, 1, None, buf, buf, None, buf, st) != 0
    assert b"null" in L.rimphony_b200_last_error()
    assert L.rimphony_b200_transfer(1, 1, buf, buf, buf, None, None, st) != 0
    assert L.rimphony_b200_transfer(2 ** 40, 2 ** 40, buf, buf, buf, None, buf, st) != 0
    assert b"overflows" in L.rimphony_b200_last_error()
    assert L.rimphony_b200_transfer_device(1, 1, None, None, None, None, None, None, None, 1) != 0
    assert L.rimphony_b200_transfer(0, 5, None, None, None, None, None, None) == 0  # nothing to do
    cols = (_lib.c_double_p * 1)(ctypes.cast(buf, _lib.c_double_p))
    o = R.make_options(coeff_mask=0x3F)
    args = (1, 1, buf, buf, buf, buf, buf, buf, cols, 1, None, buf, None, st)
    assert L.rimphony_b200_compute_stokes_cgs(17, *args) != 0
    assert b"kind" in L.rimphony_b200_last_error()
    a = list(args)
    a[10] = ctypes.byref(o)
    assert L.rimphony_b200_compute_stokes_cgs(R.POWER_LAW, *a) != 0
    assert b"coeff_mask" in L.rimphony_b200_last_error()
    bad_mode = R.make_options(mode=9)
    a[10] = ctypes.byref(bad_mode)
    assert L.rimphony_b200_compute_stokes_cgs(R.POWER_LAW, *a) != 0
    assert b"mode" in L.rimphony_b200_last_error()
    a[4] = None  # b
    a[10] = None
    assert L.rimphony_b200_compute_stokes_cgs(R.POWER_LAW, *a) != 0
    assert b"null" in L.rimphony_b200_last_error()
    with pytest.raises(ValueError):
        R.transfer(np.ones((7, 3)), 0.0, 1.0)


@pytest.mark.skipif(R.device_count() > 0, reason="a CUDA device is present")
def test_fails_loudly_without_a_gpu():
    with pytest.raises(R.RimphonyB200Error):
        R.transfer(np.ones((8, 3)), 0.1, 1.0)
    with pytest.raises(R.RimphonyB200Error):
        R.PitchyKappaDistribution(3.5, 10.0, 1.0).full_calculation().compute_stokes_cgs(1e10, 10.0, 1e3, 0.5, 0.2, 1e15)
    L = _lib.load()
    buf = (ctypes.c_double * 64)()
    assert L.rimphony_b200_transfer_device(1, 1, buf, buf, buf, None, buf, None, None, 1) != 0


class _FakeSlabModule:
    """The package surface stokes-slab-pitchykappa-cgs uses, with the device call replaced."""

    def __getattr__(self, name):
        return getattr(R, name)

    class PitchyKappaDistribution:
        def __init__(self, *a):
            self.args = a

        def gamma_cutoff(self, c):
            self.cutoff = c
            return self

        def full_calculation(self, mode=0):
            outer = self

            class _Calc:
                def compute_stokes_cgs(self, *a):
                    _FakeSlabModule.seen = (outer.args, outer.cutoff, a)
                    return R.StokesResult(np.array([[1.5e-3], [-2e-5], [3.25e-6], [0.0]]), np.zeros(1, np.int32), None)
            return _Calc()


def test_stokes_slab_example_layout():
    out = io.StringIO()
    argv = ["stokes-slab-pitchykappa-cgs", "1e9", "100", "1e3", "0.7", "0.2", "1e12", "3.5", "5", "1"]
    assert examples.main(argv, module=_FakeSlabModule(), out=out) == 0
    lines = out.getvalue().splitlines()
    assert [ln.split(": ")[0] for ln in lines] == ["I", "Q", "U", "V"]
    assert all(re.fullmatch(r"-?\d\.\d{18}e-?\d+", ln.split(": ")[1]) for ln in lines)
    assert float(lines[0].split(": ")[1]) == 1.5e-3 and float(lines[2].split(": ")[1]) == 3.25e-6
    assert _FakeSlabModule.seen == ((3.5, 5.0, 1.0), 100.0, (1e9, 100.0, 1e3, 0.7, 0.2, 1e12))


# ---------------------------------------------------------------------------
# GPU


def _device_transfer(coeffs, psi, ds, s0):
    return R.transfer(coeffs, psi, ds, s0)


@pytest.mark.gpu
def test_kernel_matches_mpmath_on_the_grid_and_rays():
    _check_grid(_device_transfer, TOL)
    _check_rays(_device_transfer, TOL)


@pytest.mark.gpu
def test_kernel_matches_the_host_build():
    """1e-14 of the scale, times the conditioning (1 + |a| ds + |rho| ds).  The two builds differ in FMA
    contraction (the host build has none) and in their exp and sincos, so the eigenvalues Lambda_1,2 ds, computed
    from |a| ds and |rho| ds, differ by an ulp of those: the decay exponent of the slowly absorbed mode and the
    rotation phase move by that much, and the cubic in M loses eps |M| ds in either build."""
    def bound(coeffs, ds):
        c = np.asarray(coeffs).reshape(8, np.shape(coeffs)[1], -1)
        d = np.broadcast_to(ds, c.shape[1:])
        return 1e-14 * (1 + ((np.hypot(c[3], c[5]) + np.hypot(c[6], c[7])) * d).sum(axis=1))

    coeffs, psi, rho, _, _ = grid()
    for s0 in (None, STOKES0):
        got, st = R.transfer(coeffs, psi, 1.0, s0)
        host, st_host = emu_transfer(coeffs, psi, 1.0, s0)
        assert np.array_equal(st, st_host)
        err, lim = normwise_error(got, host, s0), bound(coeffs, 1.0)
        bad = np.flatnonzero(err > lim)
        assert bad.size == 0, [(coeffs[:, i], psi[i], err[i] / lim[i]) for i in bad[:8]]
    for coeffs, psi, ds, s0, _, rho in ray_cases():
        got, _ = R.transfer(coeffs, psi, ds, s0)
        host, _ = emu_transfer(coeffs, psi, ds, s0)
        assert (normwise_error(got, host, s0) <= bound(coeffs, ds)).all()


@pytest.mark.gpu
def test_kernel_on_very_thick_masing_and_out_of_range_cells():
    for tau, pol, rho in itertools.product((1e10, 1e15, 1e100), (0.0, 0.5, 0.9), (0.0, 1.0, 10.0)):
        k8, ds, K, J = _thick_cell(tau, pol, rho)
        got, status = R.transfer(k8[:, None], 0.3, ds)
        want = np.linalg.solve(K, J)
        assert status[0] == 0 and np.abs(got[:, 0] - want).max() <= 1e-13 * np.abs(want).max(), (tau, pol, rho)
    cells = np.array([_grid_cell(tau, pol, 1.0, "generic") for tau, pol in
                      itertools.product((-0.1, -1.0, -10.0), (0.0, 0.5, 1.0))]).T.copy()
    got, status = R.transfer(cells, 0.37, 1.0, STOKES0)
    want = ref_transfer(cells, 0.37, 1.0, STOKES0)
    assert (status == 0).all() and (normwise_error(got, want, STOKES0) <= 2 * TOL).all()
    k8, ds, _, _ = _thick_cell(1e103, 0.5, 0.0)
    got, status = R.transfer(np.stack([k8, _grid_cell(-10.5, 0.5, 1.0, "generic")], axis=1), 0.3, [ds, 1.0])
    assert np.isnan(got).all() and (status == R.STATUS_NAN).all()


def _nu_c(b):
    return R.ELECTRON_CHARGE * b / (R.TWO_PI * R.MASS_ELECTRON * R.SPEED_LIGHT)


def _composition(kind, nu, b, n_e, theta, psi, ds, params, mode):
    """compute_all_dimensionless_batch -> the cgs scaling of compute_all_cgs -> transfer."""
    shape = np.shape(nu)
    flat = lambda x: np.broadcast_to(np.asarray(x, dtype=np.float64), shape).reshape(-1)  # noqa: E731
    nu_f, b_f, ne_f = flat(nu), flat(b), flat(n_e)
    s = nu_f / _nu_c(b_f)
    res = R.compute_all_dimensionless_batch(kind, s, flat(theta),
                                            [p if np.ndim(p) == 0 else flat(p) for p in params], mode=mode)
    rv = res.values.copy()
    scale_j, scale_a = ne_f * nu_f, ne_f / nu_f
    for c in (0, 2, 4):
        rv[c] = rv[c] * scale_j
    for c in (1, 3, 5, 6, 7):
        rv[c] = rv[c] * scale_a
    coeffs = rv.reshape((8,) + shape)
    stokes, status = R.transfer(coeffs, psi, ds)
    return coeffs, stokes, status, res.status


def _rays_of(config, n_rays, n_cells, seed):
    if config == "juettner":
        kind, s, theta, params = R.synthetic_batch("juettner_sweep", 0)
        idx = np.random.default_rng(seed).choice(s.size, n_rays * n_cells, replace=False)
        s, theta, params = s[idx], theta[idx], [params[0][idx]]
    else:
        kind, s, theta, params = R.synthetic_batch(config, n_rays * n_cells, seed=seed)
    rng = np.random.default_rng(seed)
    shape = (n_rays, n_cells)
    b = 10.0 ** rng.uniform(-1, 2, shape)
    nu = s.reshape(shape) * _nu_c(b)
    n_e = 10.0 ** rng.uniform(2, 6, shape)
    psi = rng.uniform(-np.pi, np.pi, shape)
    ds = 10.0 ** rng.uniform(12, 17, shape)
    params = [p if np.ndim(p) == 0 else p.reshape(shape) for p in params]
    return kind, nu, b, n_e, theta.reshape(shape), psi, ds, params


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [R.MODE_FAST, R.MODE_FAITHFUL])
@pytest.mark.parametrize("config", ["powerlaw", "juettner", "pitchy_pl", "pitchy_kappa", "pitchy_bpl"])
def test_compute_stokes_cgs_is_the_composition_to_the_bit(config, mode):
    n_rays, n_cells = (3, 4) if mode == R.MODE_FAST else (2, 2)
    kind, nu, b, n_e, theta, psi, ds, params = _rays_of(config, n_rays, n_cells, 11)
    res = R.compute_stokes_cgs(kind, nu, b, n_e, theta, psi, ds, params, mode=mode)
    coeffs, stokes, status, cell_status = _composition(kind, nu, b, n_e, theta, psi, ds, params, mode)
    np.testing.assert_array_equal(res.coeffs, coeffs)
    np.testing.assert_array_equal(res.stokes, stokes)
    want = np.bitwise_or.reduce(cell_status.reshape(n_rays, n_cells), axis=1) | status
    assert np.array_equal(res.status, want)


@pytest.mark.gpu
def test_device_variant_equals_the_host_one_on_a_caller_stream():
    import torch

    for coeffs, psi, ds, s0, _, _ in ray_cases():
        want, want_status = R.transfer(coeffs, psi, ds, s0)
        n_rays = want.shape[1]
        dev = torch.device("cuda:0")
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64).reshape(-1)).to(dev)  # noqa: E731
        c_d, psi_d, ds_d, s0_d = t(coeffs.reshape(8, -1)), t(psi), t(ds), t(np.broadcast_to(s0[:, None], (4, n_rays)))
        out = torch.full((4 * n_rays,), float("nan"), dtype=torch.float64, device=dev)
        st = torch.full((n_rays,), -1, dtype=torch.int32, device=dev)
        stream = torch.cuda.Stream(device=dev)
        stream.wait_stream(torch.cuda.current_stream(dev))
        R.transfer_device(c_d, psi_d, ds_d, out, s0_d, st, stream=stream, synchronize=False)
        stream.synchronize()
        np.testing.assert_array_equal(out.cpu().numpy().reshape(4, n_rays), want)
        np.testing.assert_array_equal(st.cpu().numpy(), want_status)
        # a status tensor of the wrong size, or a tensor on another device, is refused before the launch
        with pytest.raises(ValueError):
            R.transfer_device(c_d, psi_d, ds_d, out, s0_d, st[:-1])
        with pytest.raises(ValueError):
            R.transfer_device(c_d, psi_d.cpu(), ds_d, out, s0_d, st)


@pytest.mark.gpu
def test_nan_coefficients_and_reference_divergence_reach_the_ray_status():
    coeffs = np.repeat(_grid_cell(1.0, 0.5, 1.0, "generic")[:, None, None], 2, axis=2).repeat(2, axis=1)
    coeffs[6, 1, 1] = np.nan
    stokes, status = R.transfer(coeffs, 0.1, 1.0)
    assert np.isfinite(stokes[:, 0]).all() and status[0] == 0
    assert np.isnan(stokes[:, 1]).all() and status[1] == R.STATUS_NAN
    # a power law with gamma_min = 1 below s = 0.35: the reference's rho quadrature diverges
    nu_c = _nu_c(10.0)
    nu = np.array([[0.2 * nu_c, 50.0 * nu_c], [20.0 * nu_c, 50.0 * nu_c]])
    res = R.compute_stokes_cgs(R.POWER_LAW, nu, 10.0, 1e3, 0.8, 0.1, 1e14, [2.5, 1.0, 1e12, 1e10])
    assert res.status[0] & R.STATUS_REFERENCE_DIVERGES and res.status[0] & R.STATUS_NAN
    assert np.isnan(res.stokes[:, 0]).all() and np.isnan(res.coeffs[6:, 0, 0]).any()
    assert res.status[1] == 0 and np.isfinite(res.stokes[:, 1]).all()


@pytest.mark.gpu
def test_rays_with_broadcast_parameter_columns():
    kind, nu, b, n_e, theta, psi, ds, params = _rays_of("pitchy_pl", 5, 3, 3)
    scalar = [2.5, 1.0, 1.0, 1e12, 1e10]
    res = R.compute_stokes_cgs(kind, nu, b, n_e, theta, psi, ds, scalar)
    full = R.compute_stokes_cgs(kind, nu, b, n_e, theta, psi, ds, [np.full(nu.shape, v) for v in scalar])
    np.testing.assert_array_equal(res.stokes, full.stokes)
    np.testing.assert_array_equal(res.coeffs, full.coeffs)
    # with gamma_min = 1, rho is NaN at small s (the reference diverges there): exactly those rays are NaN
    nan_cells = np.isnan(res.coeffs).any(axis=0).any(axis=1)
    assert nan_cells.any() and not nan_cells.all()
    assert np.array_equal(np.isnan(res.stokes).any(axis=0), nan_cells)
    assert np.array_equal((res.status & R.STATUS_NAN) != 0, nan_cells)
    calc = R.PitchyPowerLawDistribution(2.5, 1.0).full_calculation()
    np.testing.assert_array_equal(calc.compute_stokes_cgs(nu, b, n_e, theta, psi, ds).stokes, res.stokes)


# demo almostuniform1 as slabs: the row's s is reproduced with B = 1 G and nu = s nu_c(1 G); the row's d, psi and
# n_e are the slab's depth, field angle and density
DEMO_B = 1.0


@pytest.mark.gpu
def test_demo_almostuniform1_slabs_match_mpmath():
    from rimphony_b200 import crank_out

    cols = crank_out.demo_almostuniform1()
    nu = cols["s"] * _nu_c(DEMO_B)
    params = [cols["p"], crank_out.GAMMA_MIN, crank_out.GAMMA_MAX, crank_out.GAMMA_CUTOFF]
    res = R.compute_stokes_cgs(R.POWER_LAW, nu, DEMO_B, cols["n_e"], cols["theta"], cols["psi"], cols["d"], params)
    coeffs = res.coeffs[:, :, 0]
    assert np.isfinite(coeffs).all() and np.isfinite(res.stokes).all()
    want = ref_transfer(coeffs, cols["psi"], cols["d"])
    live = cols["d"] > 0
    rho = np.hypot(coeffs[6], coeffs[7]) * cols["d"]
    assert (normwise_error(res.stokes[:, live], want[:, live]) <= TOL * (1 + rho[live])).all()
    assert (res.stokes[:, ~live] == 0).all()  # the first row has d = 0
