"""Parity of the CUDA path against the CPU oracle, through the C ABI (-m gpu).

Tolerances (BASELINE.json north_star: "<= 1e-3 relative, or within the reference's own
integration tolerance, with sign agreement on rho_Q/V and alpha_V"):

* FAITHFUL mode performs the reference's own sequence of Gauss-Kronrod applications per
  coefficient: it must agree with the oracle to 1e-6 relative on 99 % of the finite values
  and to 1e-5 on all (rounding differences between libm and CUDA math are amplified where
  lobes or chunks cancel), and reproduce the NaNs (the reference's failure marker) up to the
  knife-edge cases described at FAITHFUL_NAN_SLACK.
* FAST mode (the product default) integrates the same integrands over the same domains with
  the same truncation rules, but organises the quadrature differently (rb_symfast.cuh,
  rb_heyfast.cuh).  Its own quadrature error is ~1e-5 (test_fast_mode_is_converged).  The bar is
  the north-star one: <= 1e-3 (Stokes V: of |lobe+| + |lobe-|) on >= 99.9 % of the points, never a NaN
  where the reference has a number (<= 0.1 %), same signs, over the entries where the reference's own algorithm is
  defined to 1e-3 (rimphony_b200/parity.py; the excluded entries are counted and bounded).
  Exception, documented in tests/golden/heyvaerts_low_s.md: rho_Q / rho_V of the power laws at
  s < 1, where the reference's NaN verdict is a property of its tolerance; the test asserts the
  measured agreement of the reference-divergence rule there (>= 85 % of the verdicts, >= 97 % of
  the pairs that are finite on both sides within 1e-3).
* FUSED mode keeps the reference's control flow on shared nodes.  Both it and
  the reference then carry an independent integration error of up to the QAG tolerance
  (epsrel = 1e-3 per nested level, symphony.rs:266, 376), so the bar is
    - I and Q coefficients: <= 1e-3 relative on >= 99 % of points and <= 2.5e-3 on all;
    - Stokes V (two lobes integrated separately that nearly cancel, symphony.rs:97-107):
      |gpu - oracle| <= 1e-3 * (|lobe+| + |lobe-|), the reference's own integration scale;
    - rho_Q, rho_V: exact-sequence parity for s sin(theta) < 3 (the kernel switches to the
      faithful sequence there), <= 1e-3 on >= 99 % and <= 3e-3 on all points above.
"""
import math

import numpy as np
import pytest

import rimphony_b200 as R

pytestmark = pytest.mark.gpu

NAMES = R.COEFFICIENT_NAMES
FIXTURES = ["pitchy_pl", "powerlaw", "pitchy_kappa", "symphony_rows"]


def run(fx, mode, mask=0xFF, extras=True, **kw):
    return R.compute_all_dimensionless_batch(fx["kind"], fx["s"], fx["theta"], fx["params"], mode=mode,
                                             coeff_mask=mask, extras=extras, **kw)


def finite_pairs(a, b):
    return ~np.isnan(a) & ~np.isnan(b)


def nan_mismatches(a, b):
    return int((np.isnan(a) != np.isnan(b)).sum())


# NaN is the reference's failure marker.  Where it comes from a QUADPACK round-off / singularity
# verdict or from the n >= 1e15 Bessel-derivative rule it sits on a knife edge of the last bits
# of libm vs CUDA math, so even the exact rule sequence flips a few of them (observed: 3 of 400
# rho_V values, 6 of 443 Juettner rho values, 1 of 200 kappa points): the faithful tests allow 2 %.
FAITHFUL_NAN_SLACK = 0.02


# --- kernel 2: the Leung Bessel evaluator ---------------------------------------------

def test_device_bessel_matches_reference_bessel_c(oracle):
    rng = np.random.default_rng(0)
    m = 30000
    n = 10 ** rng.uniform(math.log10(30), 10, m)
    n[::3] = np.floor(n[::3])
    eps = 10 ** rng.uniform(-12, 0, m)
    x = n * (1 - eps)
    # the integer-order branch (gsl_sf_bessel_Jn in the reference, bessel.c:327-334)
    n[:4000] = np.floor(rng.uniform(0, 30, 4000))
    x[:4000] = rng.uniform(0, 1, 4000) * (n[:4000] + 1)
    # x > n: Debye / blend / Meissel-2
    x[4000:6000] = n[4000:6000] * (1 + 10 ** rng.uniform(-10, 0.3, 2000))
    j, dj = R.bessel_jn(n, x)
    rj = np.array([oracle.ref_bessel_j(a, b) for a, b in zip(n, x)])
    rdj = np.array([oracle.ref_bessel_dj(a, b) for a, b in zip(n, x)])
    assert np.array_equal(np.isnan(j), np.isnan(rj)) and np.array_equal(np.isnan(dj), np.isnan(rdj))
    for got, want in ((j, rj), (dj, rdj)):
        sig = np.abs(want) > 1e-250
        rel = np.abs(got[sig] / want[sig] - 1)
        # the exponent n (ln(..) - ..) - lgamma(n) carries ~ulp(n ln n) of rounding noise in BOTH
        # implementations (1e-6 at n = 1e10), amplified in J' by the n J_n/x - J_{n+1} difference
        assert np.median(rel) < 1e-14
        assert np.percentile(rel, 99) < 1e-6
        assert rel.max() < 2e-3
    small = slice(0, 4000)
    ok = np.abs(rj[small]) > 1e-280
    assert np.abs(j[small][ok] / rj[small][ok] - 1).max() < 1e-10


def test_device_bessel_special_arguments():
    j, dj = R.bessel_jn(np.array([0.0, 5.0, 0.0, 29.5, -1.0, 40.0, 1e15, 1.0, 0.0]),
                        np.array([0.0, 5.0, 17.0, 3.0, 2.0, 0.0, 1e14, 0.0, 0.0]))
    assert abs(j[0] - 1.0) < 1e-6 and abs(j[1] - 0.2611405) < 1e-6 and abs(j[2] + 0.1698543) < 1e-6  # lib.rs:83-85
    assert math.isnan(j[3]) and math.isnan(j[4])       # non-integer n < 30, negative n (bessel.c:323-331)
    assert j[5] == 0.0 and dj[5] == 0.0                 # x = 0, n >= 2 (bessel.c:393-395)
    assert math.isnan(dj[6])                            # n >= 1e15 (bessel.c:382-388)
    assert dj[8] == 0.0 or abs(dj[8]) < 1e-300          # J_0'(0) = -J_1(0) = 0


# --- distributions and normalisation ---------------------------------------------------

@pytest.mark.parametrize("kind,params", [(R.POWER_LAW, [2.5, 1.0, 1e12, 1e10]), (R.THERMAL_JUETTNER, [10.0]),
                                         (R.PITCHY_PL, [3.1, 1.7, 1.0, 1e12, 1e10]), (R.PITCHY_KAPPA, [2.7, 5.0, 0.8, 1e10])])
def test_distribution_functions(oracle, kind, params):
    import ctypes
    rng = np.random.default_rng(1)
    gamma = 1.0 + 10 ** rng.uniform(-3, 6, 2000)
    cx = rng.uniform(-0.99, 0.99, 2000)
    f, dg, dc = R.dist_eval(kind, params, gamma, cx)
    d = oracle.make_dist(kind, params)
    d.norm = 1.0
    a, b = ctypes.c_double(), ctypes.c_double()
    L = oracle.lib()
    for i in range(0, 2000, 7):
        want_f = L.orc_calc_f(ctypes.byref(d), gamma[i], cx[i])
        L.orc_calc_f_derivatives(ctypes.byref(d), gamma[i], cx[i], ctypes.byref(a), ctypes.byref(b))
        assert f[i] == pytest.approx(want_f, rel=1e-12, abs=1e-300)
        assert dg[i] == pytest.approx(a.value, rel=1e-11, abs=1e-300)
        assert dc[i] == pytest.approx(b.value, rel=1e-11, abs=1e-300)


def test_hard_gamma_cutoffs_are_exact_zero():
    f, dg, dc = R.dist_eval(R.POWER_LAW, [2.5, 10.0, 1e3, 1e10], np.array([9.999, 10.0, 1e3, 1000.001]), np.zeros(4))
    assert f[0] == 0.0 and f[3] == 0.0 and f[1] > 0 and f[2] > 0 and dg[0] == 0.0  # power_law.rs:38, 49


@pytest.mark.parametrize("name", ["pitchy_pl", "powerlaw", "pitchy_kappa", "juettner_sweep"])
def test_normalisation_matches_oracle(oracle, golden, name):
    fx = golden(name)
    sel = np.arange(0, len(fx["s"]), max(1, len(fx["s"]) // 40))
    sub = {"kind": fx["kind"], "s": fx["s"][sel], "theta": fx["theta"][sel], "params": [p[sel] for p in fx["params"]]}
    res = run(sub, R.MODE_FUSED, mask=0x01)
    for i in range(len(sel)):
        d = oracle.make_dist(fx["kind"], [p[i] for p in sub["params"]])
        assert res.norm[i] == pytest.approx(d.norm, rel=1e-10)


# --- the hot path: faithful mode is the reference's algorithm ------------------------------

@pytest.mark.parametrize("name", FIXTURES)
def test_faithful_mode_reproduces_the_oracle(golden, name):
    fx = golden(name)
    res = run(fx, R.MODE_FAITHFUL)
    want = fx["out"]
    for c in range(8):
        got_c, want_c = res.values[c], want[c]
        assert nan_mismatches(got_c, want_c) <= FAITHFUL_NAN_SLACK * len(want_c), f"NaN pattern differs for {NAMES[c]}"
        ok = finite_pairs(got_c, want_c)
        rel = np.abs(got_c[ok] / want_c[ok] - 1)
        # V = lobe(+) + lobe(-) nearly cancel: the lobes carry the 1e-6, their sum a little more
        assert rel.max() < 1e-5, (NAMES[c], rel.max(), np.argmax(rel))
        assert np.percentile(rel, 99) < 1e-6, (NAMES[c], np.percentile(rel, 99))
        assert np.median(rel) < 1e-9
    ok = ~np.isnan(fx["lobes"]).any(axis=0) & ~np.isnan(res.lobes).any(axis=0)
    assert np.allclose(res.lobes[:, ok], fx["lobes"][:, ok], rtol=1e-6, atol=0.0)
    assert ((res.status & R.STATUS_NAN) != 0).tolist() == np.isnan(res.values).any(axis=0).tolist()
    # the device interval lists (48 / 128 entries) are far smaller than the reference's workspaces
    # (1000-5000); they fill up only on Faraday integrals that fail anyway (s sin(theta) < 3)
    assert ((res.status & R.STATUS_CAP_HIT) != 0).mean() <= 0.03


def test_faithful_juettner_faraday_sweep(golden):
    fx = golden("juettner_sweep")
    res = run(fx, R.MODE_FAITHFUL, mask=0xC0)
    for c in (6, 7):
        assert nan_mismatches(res.values[c], fx["out"][c]) <= FAITHFUL_NAN_SLACK * len(fx["s"])
        ok = finite_pairs(res.values[c], fx["out"][c])
        assert np.abs(res.values[c][ok] / fx["out"][c][ok] - 1).max() < 1e-6
    assert np.isnan(res.values[:6]).all()  # slots that were not requested come back as NaN


# --- the hot path: fused mode (the product) --------------------------------------------------

@pytest.mark.parametrize("name", FIXTURES)
def test_fused_mode_within_the_integration_tolerance(golden, name):
    fx = golden(name)
    if fx["kind"] == R.PITCHY_KAPPA:
        # hard kappa spectra: the reference value is set by where its gamma quadrature loses the
        # J_n^2 peak (DESIGN.md section 5.4), which only its exact rule sequence reproduces; the
        # shared-node variant of that sequence is compared on the other points
        guard = run(fx, R.MODE_FAST, mask=0x3F, extras=False)
        keep = (guard.status & R.STATUS_REROUTED) == 0
        fx = {"kind": fx["kind"], "s": fx["s"][keep], "theta": fx["theta"][keep],
              "params": [p[keep] for p in fx["params"]], "out": fx["out"][:, keep], "lobes": fx["lobes"][:, keep]}
    res = run(fx, R.MODE_FUSED)
    want, lobes = fx["out"], fx["lobes"]
    sigma0 = fx["s"] * np.sin(fx["theta"])

    for c in range(4):  # j_I, alpha_I, j_Q, alpha_Q
        assert nan_mismatches(res.values[c], want[c]) <= FAITHFUL_NAN_SLACK * len(want[c]), NAMES[c]
        ok = finite_pairs(res.values[c], want[c])
        rel = np.abs(res.values[c][ok] / want[c][ok] - 1)
        assert (rel <= 1e-3).mean() >= 0.99, (NAMES[c], (rel <= 1e-3).mean())
        assert rel.max() <= 2.5e-3, (NAMES[c], rel.max())
        assert (np.sign(res.values[c][ok]) == np.sign(want[c][ok])).all()

    for c, (lp, lm) in ((4, (0, 1)), (5, (2, 3))):  # Stokes V against the lobe scale
        assert nan_mismatches(res.values[c], want[c]) <= FAITHFUL_NAN_SLACK * len(want[c]), NAMES[c]
        ok = finite_pairs(res.values[c], want[c])
        scale = np.abs(lobes[lp]) + np.abs(lobes[lm])
        err = np.abs(res.values[c] - want[c])[ok] / scale[ok]
        assert err.max() <= 1e-3, (NAMES[c], err.max())
        # sign agreement wherever the reference's V is resolved above its own integration noise
        resolved = ok & (np.abs(want[c]) > 4e-3 * scale)
        assert (np.sign(res.values[c][resolved]) == np.sign(want[c][resolved])).all()

    for c in (6, 7):  # Faraday
        low = sigma0 < 3.0
        # exact-sequence parity where the reference's answer depends on the sequence
        assert nan_mismatches(res.values[c][low], want[c][low]) <= 2 + FAITHFUL_NAN_SLACK * low.sum(), NAMES[c]
        ok = finite_pairs(res.values[c], want[c]) & low
        if ok.any():
            assert np.abs(res.values[c][ok] / want[c][ok] - 1).max() < 1e-6
        hi = ~low
        assert nan_mismatches(res.values[c][hi], want[c][hi]) <= 2 + FAITHFUL_NAN_SLACK * hi.sum(), NAMES[c]
        ok = finite_pairs(res.values[c], want[c]) & hi
        if ok.any():
            rel = np.abs(res.values[c][ok] / want[c][ok] - 1)
            assert (rel <= 1e-3).mean() >= 0.99, (NAMES[c], (rel <= 1e-3).mean())
            assert rel.max() <= 3e-3, (NAMES[c], rel.max())
            assert (np.sign(res.values[c][ok]) == np.sign(want[c][ok])).all()


# --- the hot path: fast mode (the product default) -----------------------------------------
#
# The bar is BASELINE.json's: <= 1e-3 relative (Stokes V: of the lobe scale) on >= 99.9 % of the
# points, the reference's NaN pattern on >= 99.9 %, no sign difference.  Entries where the
# reference's own algorithm is not defined to 1e-3 (its value moves by more than that, or its NaN
# flips, when its tolerance goes from 1e-3 to 3e-4 or s is nudged by 1e-9: the *_stability.npz
# companions, tests/golden/make_stability.py) are excluded and counted (rimphony_b200/parity.py).
# One documented exception: rho_Q / rho_V of the power laws at s < 1, where the reference's NaN is a
# property of its tolerance (tests/golden/heyvaerts_low_s.md); there the test asserts the measured
# agreement of the reference-divergence rule instead.

def _fast_stats(name, mask=0xFF, rows=None):
    from rimphony_b200 import parity as P
    fx = P.load_fixture(name)
    res = R.compute_all_dimensionless_batch(int(fx["kind"]), fx["s"], fx["theta"], list(fx["params"]), coeff_mask=mask,
                                            extras=True)
    sel = slice(None) if rows is None else rows
    stats = P.parity_stats(res.values[:, sel], fx["out"][:, sel], fx["lobes"][:, sel], fx["defined"][:, sel], mask=mask)
    return fx, res, stats


@pytest.mark.parametrize("name", ["pitchy_pl_4k", "pitchy_pl_10k", "powerlaw_10k", "pitchy_kappa_2k", "pitchy_kappa_10k"])
def test_fast_mode_meets_the_north_star_bar(name):
    import os
    from rimphony_b200 import parity as P
    if not os.path.exists(os.path.join(P.GOLDEN_DIR, name + ".npz")):
        pytest.skip("fixture not generated")
    fx, res, stats = _fast_stats(name)
    n = len(fx["s"])
    # without converged-reference evidence (pitchy_kappa_2k, pitchy_kappa_10k: Symphony at epsrel 1e-5 on hard kappa
    # spectra takes hours per point) the reference's own 2e-3 ... 1e-2 integration errors stay in the count: 99.8 %
    bar = 0.999 if fx["converged_entries"] else 0.998
    for nm in NAMES[:6]:   # j and alpha: everywhere
        v = stats[nm]
        assert v["frac_within"] >= bar, (nm, v)
        assert v["nan_here_only"] <= 0.001 * n, (nm, v)   # never a failure where the reference has a number
        assert v["nan_ref_only"] <= 0.003 * n, (nm, v)    # the reference's own failures (kappa, n -> 1e15): 0.2 %
        assert v["sign_mismatch"] == 0 or nm in ("j_V", "alpha_V"), (nm, v)
        assert v["undefined"] <= 0.02 * n, (nm, v)
    # Faraday: the bar holds for s >= 1 ...
    hi = np.where(fx["s"] >= 1.0)[0]
    st_hi = P.parity_stats(res.values[:, hi], fx["out"][:, hi], None, fx["defined"][:, hi], mask=0xC0)
    for nm in NAMES[6:]:
        v = st_hi[nm]
        assert v["frac_within"] >= bar, (nm, v)
        assert v["nan_here_only"] <= 0.001 * len(hi), (nm, v)   # never a failure where the reference has a number
        assert v["nan_ref_only"] <= 0.012 * len(hi), (nm, v)    # the reference's QAG gives up on 0.4-1.0 % (DESIGN 7)
        assert v["sign_mismatch"] == 0, (nm, v)
    # ... and below s = 1 (power laws only: the kappa configuration has s >= 1) the measured agreement
    lo = np.where(fx["s"] < 1.0)[0]
    if len(lo) >= 100:
        st_lo = P.parity_stats(res.values[:, lo], fx["out"][:, lo], None, fx["defined"][:, lo], mask=0xC0)
        for nm in NAMES[6:]:
            v = st_lo[nm]
            assert v["frac_within"] >= 0.97, (nm, v)      # finite on both sides: the same number
            assert v["nan_mismatch"] <= 0.20 * len(lo), (nm, v)   # the verdict: 80 % at least (measured 85-93 %)
            assert v["sign_mismatch"] == 0, (nm, v)
        diverges = (res.status & R.STATUS_REFERENCE_DIVERGES) != 0
        # rb_heyfast.cuh kHeyRefDiverges*: rho_V below a threshold on s; rho_Q below one that rises with theta
        iso = fx["kind"] == R.POWER_LAW
        s_v = 0.33 if iso else 0.38
        lo, hi, t0, t1 = (0.0, 0.30, 0.20, 1.40) if iso else (0.18, 0.37, 0.15, 0.40)
        s_q = lo + (hi - lo) * np.clip((fx["theta"] - t0) / (t1 - t0), 0.0, 1.0)
        assert np.array_equal(diverges, fx["s"] < s_v)
        assert np.isnan(res.values[7][diverges]).all() and np.isnan(res.values[6][fx["s"] < s_q * (1 - 1e-12)]).all()
    # the fidelity guard: never on the power-law batches, a quarter of the hard kappa spectra
    rerouted = (res.status & R.STATUS_REROUTED) != 0
    if fx["kind"] in (R.POWER_LAW, R.PITCHY_PL):
        assert rerouted.mean() <= 0.002


@pytest.mark.parametrize("name", ["pitchy_pl", "powerlaw", "pitchy_kappa", "symphony_rows", "pitchy_pl_high_s"])
def test_fast_mode_small_fixtures(golden, name):
    """The 64-400-point sets (no stability companions): at most one entry per coefficient beyond 1e-3 on j / alpha,
    rho for s >= 1 within 1e-3 up to two entries."""
    from rimphony_b200 import parity as P
    fx = golden(name)
    res = run(fx, R.MODE_FAST)
    stats = P.parity_stats(res.values, fx["out"], fx["lobes"], None)
    for nm in NAMES[:6]:
        v = stats[nm]
        assert v["finite"] - v["within"] <= 1 and v["nan_here_only"] == 0 and v["nan_ref_only"] <= 1, (nm, v)
        assert v["max_err"] <= 1e-2, (nm, v)
    hi = fx["s"] >= 1.0
    st_hi = P.parity_stats(res.values[:, hi], fx["out"][:, hi], None, None, mask=0xC0)
    for nm in NAMES[6:]:
        v = st_hi[nm]
        assert v["finite"] - v["within"] <= 2 and v["nan_here_only"] == 0 and v["sign_mismatch"] == 0, (nm, v)
        assert v["nan_ref_only"] <= 2 + 0.02 * v["n"], (nm, v)   # the reference's QAG gave up (theta < 0.1, k < 0.5)


def test_fast_mode_juettner_faraday_sweep(golden):
    fx = golden("juettner_sweep")
    res = run(fx, R.MODE_FAST, mask=0xC0)
    for c in (6, 7):
        ok = finite_pairs(res.values[c], fx["out"][c])
        assert ok.mean() > 0.97
        rel = np.abs(res.values[c][ok] / fx["out"][c][ok] - 1)
        assert rel.max() <= 1e-3, (NAMES[c], rel.max())
        assert (np.sign(res.values[c][ok]) == np.sign(fx["out"][c][ok])).all()
        assert np.isnan(res.values[c]).sum() == 0
    assert np.isnan(res.values[:6]).all()  # slots that were not requested come back as NaN


def test_fast_mode_is_converged(golden):
    """The product path's own quadrature error: default tolerances against 1e-6 ones.  This is
    what shows that its distance from the oracle is the reference's integration noise."""
    fx = golden("pitchy_pl")
    a = run(fx, R.MODE_FAST)
    b = run(fx, R.MODE_FAST, epsrel_gamma=1e-6, epsrel_n=1e-6, epsrel_heyvaerts_inner=1e-6,
            epsrel_heyvaerts_outer=1e-6)
    sigma0 = fx["s"] * np.sin(fx["theta"])
    for c in range(8):
        ok = finite_pairs(a.values[c], b.values[c])
        scale = np.abs(b.values[c])
        if c in (4, 5):
            scale = np.abs(b.lobes[2 * (c - 4)]) + np.abs(b.lobes[2 * (c - 4) + 1])
        if c >= 6:
            ok &= sigma0 >= 1.0
        err = (np.abs(a.values[c] - b.values[c]) / scale)[ok]
        assert np.percentile(err, 99) <= 1e-4, (NAMES[c], np.percentile(err, 99))
        assert err.max() <= 1e-3, (NAMES[c], err.max())


def test_fast_mode_against_the_symphony_golden_file(symphony_rows):
    """tests/symphony.rs: six coefficients vs Symphony itself at 1 % (cgs at nu = 1e9, n_e = 1)."""
    g = symphony_rows
    nu = 1e9
    b = R.TWO_PI * R.MASS_ELECTRON * R.SPEED_LIGHT * nu / (R.ELECTRON_CHARGE * g[:, 0])  # symphony.rs:54
    calc = R.PowerLawDistribution(g[:, 2]).gamma_limits(1.0, 1e12, 1e10).full_calculation()
    ours = calc.compute_all_cgs(nu, b, 1.0, g[:, 1])
    rel = np.abs(ours[:, :6] / g[:, 3:9] - 1)
    assert rel[:, :4].max() < 2e-3
    assert (rel[:, 4:] < 0.01).mean() > 0.99 and rel[:, 4:].max() < 0.015


def test_fused_mode_against_the_symphony_golden_file(golden, symphony_rows):
    """tests/symphony.rs: six coefficients vs Symphony itself at 1 % (cgs at nu = 1e9, n_e = 1)."""
    g = symphony_rows
    nu = 1e9
    b = R.TWO_PI * R.MASS_ELECTRON * R.SPEED_LIGHT * nu / (R.ELECTRON_CHARGE * g[:, 0])  # symphony.rs:54
    calc = R.PowerLawDistribution(g[:, 2]).gamma_limits(1.0, 1e12, 1e10).full_calculation(mode=R.MODE_FUSED)
    ours = calc.compute_all_cgs(nu, b, 1.0, g[:, 1])
    rel = np.abs(ours[:, :6] / g[:, 3:9] - 1)
    assert rel[:, :4].max() < 2e-3
    assert (rel[:, 4:] < 0.01).mean() > 0.99 and rel[:, 4:].max() < 0.015


def test_live_oracle_on_seeded_points(oracle):
    """A handful of points the fixtures do not contain, oracle run now."""
    kind, s, theta, params = R.synthetic_batch("pitchy_pl", 8, seed=987)
    want, lobes = oracle.batch(kind, s, theta, params)
    got = R.compute_all_dimensionless_batch(kind, s, theta, params, mode=R.MODE_FAITHFUL).values
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.abs(got[ok] / want[ok] - 1).max() < 1e-6


# --- diagnostics of the Symphony double integral (src/lib.rs:249-299) --------------------------

@pytest.mark.parametrize("make,okind,params", [
    (lambda: R.PitchyPowerLawDistribution(2.5, 1.0), "PITCHY_PL", [2.5, 1.0]),
    (lambda: R.PowerLawDistribution(3.0), "POWER_LAW", [3.0]),
    (lambda: R.PitchyKappaDistribution(3.5, 5.0, 1.2), "PITCHY_KAPPA", [3.5, 5.0, 1.2]),
    (lambda: R.ThermalJuettnerDistribution(10.0), "THERMAL_JUETTNER", [10.0]),
])
def test_symphony_diagnostics_match_the_oracle(oracle, make, okind, params):
    """diagnostic_symphony_{gamma_integrand, gamma_integral, n_integral, gamma_contribution}: the device
    performs the reference's sequence of rule applications, so it agrees with the oracle to rounding
    (amplified where J_n' = n J_n / z - J_{n+1} cancels)."""
    calc = make().full_calculation()
    d = oracle.make_dist(getattr(oracle, okind), params)
    rng = np.random.default_rng(5)
    bad = []
    for s, theta in ((50.0, 0.9), (3.0, 0.3), (2e6, 1.2)):
        n0 = s * math.sin(theta)
        n = n0 * 10 ** rng.uniform(0.02, 4.0, 24) + 31.0  # from the first harmonics to far up the tail
        # gamma around the peak of the integrand: the window of symphony.rs:315-323, narrowed like n^-1/3
        peak = (n / s) / math.sin(theta) ** 2
        half = abs(math.cos(theta)) * np.sqrt((n / s) ** 2 - math.sin(theta) ** 2) / math.sin(theta) ** 2
        gamma = peak + half * np.minimum(1.0, 2.6 * n ** (-1 / 3)) * rng.uniform(-1, 1, 24)
        n_hi = n * (1.0 + rng.random(24))
        g_fixed = np.array([1.5, 2.0, 7.0, 40.0, 300.0, 2e3, 3e4])
        for coeff in (R.Coefficient.Emission, R.Coefficient.Absorption):
            for stokes in (R.Stokes.I, R.Stokes.Q, R.Stokes.V):
                cases = [
                    (calc.diagnostic_symphony_gamma_integrand(coeff, stokes, s, theta, n, gamma),
                     [oracle.symphony_diagnostic(d, coeff, stokes, s, theta, oracle.DIAG_GAMMA_INTEGRAND, a, b)
                      for a, b in zip(n, gamma)], 1e-7),  # Q = (M J_n)^2 - (N J_n')^2 cancels: 1.2e-9 observed
                    (calc.diagnostic_symphony_gamma_integral(coeff, stokes, s, theta, n),
                     [oracle.symphony_diagnostic(d, coeff, stokes, s, theta, oracle.DIAG_GAMMA_INTEGRAL, a) for a in n],
                     1e-6),
                    (calc.diagnostic_symphony_n_integral(coeff, stokes, s, theta, n[:6], n_hi[:6]),
                     [oracle.symphony_diagnostic(d, coeff, stokes, s, theta, oracle.DIAG_N_INTEGRAL, a, b)
                      for a, b in zip(n[:6], n_hi[:6])], 1e-6),
                    (calc.diagnostic_symphony_gamma_contribution(coeff, stokes, s, theta, g_fixed),
                     [oracle.symphony_diagnostic(d, coeff, stokes, s, theta, oracle.DIAG_GAMMA_CONTRIBUTION, g)
                      for g in g_fixed], 1e-6),
                ]
                for which, (got, want, tol) in enumerate(cases):
                    want = np.asarray(want)
                    # J_n carries ~n ulp of rounding in both implementations (see the Bessel test above)
                    tol = tol if s < 1e3 else max(tol, 1e-5) * 10
                    where = (okind, s, int(coeff), int(stokes), which)
                    if not np.array_equal(np.isnan(got), np.isnan(want)):
                        bad.append(where + ("nan pattern", got, want))
                        continue
                    ok = ~np.isnan(want) & (want != 0)
                    zero = ~ok & ~np.isnan(want)
                    if not np.array_equal(got[zero], want[zero]):
                        bad.append(where + ("zeros",))
                    if ok.any() and not np.abs(got[ok] / want[ok] - 1).max() < tol:
                        bad.append(where + (float(np.abs(got[ok] / want[ok] - 1).max()), tol))
    assert not bad, bad
    # scalar arguments give the reference's scalar
    v = calc.diagnostic_symphony_gamma_integral(R.Coefficient.Emission, R.Stokes.I, 50.0, 0.9, 75.0)
    assert isinstance(v, float)


# --- known answers through the reference-shaped API ------------------------------------------

def test_one_powerlaw_direct():
    """examples/one-powerlaw-direct.rs."""
    ji = (R.PowerLawDistribution(2.5).gamma_limits(1.0, 1e12, 1e10).full_calculation()
          .compute_cgs(R.Coefficient.Emission, R.Stokes.I, 1e9, 1e3, 1.0, 0.9))
    assert isinstance(ji, float) and abs(ji / 2.64399749412774e-21 - 1) < 0.01


@pytest.mark.parametrize("mode", [R.MODE_FAST, R.MODE_FUSED, R.MODE_FAITHFUL])
def test_heyvaerts_known_answers(mode):
    C, S = R.Coefficient, R.Stokes
    pl = R.PowerLawDistribution(2.5).gamma_limits(10.0, 1e12, 1e10).full_calculation(mode=mode)
    assert pl.compute_dimensionless(C.Faraday, S.Q, 1e4, 0.25 * math.pi) == pytest.approx(1.89e-9, rel=0.01)   # power_law.rs:209-216
    assert pl.compute_dimensionless(C.Faraday, S.V, 1e4, 0.25 * math.pi) == pytest.approx(5.28e-8, rel=0.01)   # power_law.rs:233-240
    assert (R.ThermalJuettnerDistribution(10.0).full_calculation(mode=mode)
            .compute_dimensionless(C.Faraday, S.Q, 4e4, 0.4)) == pytest.approx(4.8081e-11, rel=0.01)           # thermal_juettner.rs:183-190
    assert (R.ThermalJuettnerDistribution(0.1).full_calculation(mode=mode)
            .compute_dimensionless(C.Faraday, S.V, 40.0, 0.5)) == pytest.approx(3.064e-4, rel=0.01)            # thermal_juettner.rs:203-210


def test_scalar_c_abi_entry_points():
    import ctypes
    from rimphony_b200 import _lib
    L = _lib.load()
    pv = (ctypes.c_double * 4)(2.5, 1.0, 1e12, 1e10)
    out = ctypes.c_double()
    _lib.check(L.rimphony_b200_compute_cgs(R.POWER_LAW, pv, 4, 0, 0, 1e9, 1e3, 1.0, 0.9, ctypes.byref(out)))
    assert abs(out.value / 2.64399749412774e-21 - 1) < 0.01
    _lib.check(L.rimphony_b200_compute_dimensionless(R.POWER_LAW, pv, 4, 2, 0, 10.0, 0.5, ctypes.byref(out)))
    assert math.isnan(out.value)  # (Faraday, I)


def test_pitchy_k_zero_equals_isotropic():
    """pitchy_pl.rs:128-201: the Latin square of (s, theta, p), all eight coefficients."""
    ss = np.array([1e0, 1e1, 1e2, 1e3, 1e4])
    thetas = np.array([0.05, 0.430, 0.810, 1.190, 1.5707])
    ps = np.array([1.5, 1.75, 2.5, 3.25, 4.0])
    choices = [1, 4, 2, 3, 1, 0, 0, 3, 1, 2, 0, 4, 4, 2, 3]
    s = ss[choices[0::3]]
    th = thetas[choices[1::3]]
    p = ps[choices[2::3]]
    iso = R.PowerLawDistribution(p).full_calculation().compute_all_dimensionless(s, th)
    pit = R.PitchyPowerLawDistribution(p, 0.0).full_calculation().compute_all_dimensionless(s, th)
    assert iso.shape == (5, 8)
    assert np.array_equal(np.isnan(iso), np.isnan(pit))
    ok = ~np.isnan(iso)
    assert np.abs(pit[ok] / iso[ok] - 1).max() < 1e-6


# --- batch semantics and size-independent properties --------------------------------------

def test_empty_single_and_ragged_batches():
    kind, s, theta, params = R.synthetic_batch("pitchy_pl", 131, seed=3)
    full = R.compute_all_dimensionless_batch(kind, s, theta, params).values
    assert R.compute_all_dimensionless_batch(kind, s[:0], theta[:0], [p[:0] if np.ndim(p) else p for p in params]).values.shape == (8, 0)
    for n in (1, 31, 33, 130):
        part = R.compute_all_dimensionless_batch(kind, s[:n], theta[:n], [p[:n] if np.ndim(p) else p for p in params]).values
        assert np.array_equal(part, full[:, :n], equal_nan=True)


def test_degenerate_arguments_end_in_nan_and_leave_their_neighbours_alone():
    """NaN, infinite, zero and negative s / theta / parameters, theta = 0, pi/2, pi: the kernels terminate
    (application budget, chunk and step limits), the affected slots are NaN with STATUS_NAN set -- numerical
    failure is never an infrastructure error (symphony.rs:115-146, heyvaerts.rs:98-177) -- and the regular
    points interleaved with them come out as in a batch of their own."""
    kind, s, theta, params = R.synthetic_batch("pitchy_pl", 24, seed=5)
    params = [np.array(np.broadcast_to(p, s.shape), dtype=np.float64) for p in params]
    clean = R.compute_all_dimensionless_batch(kind, s, theta, params).values
    bad_s = {0: np.nan, 3: np.inf, 6: 0.0, 9: -1.0}
    bad_theta = {1: np.nan, 4: 0.0, 7: math.pi / 2, 10: math.pi, 13: -0.5}
    s2, th2, par2 = s.copy(), theta.copy(), [p.copy() for p in params]
    for i, v in bad_s.items():
        s2[i] = v
    for i, v in bad_theta.items():
        th2[i] = v
    par2[0][15] = np.nan   # p
    par2[1][18] = np.inf   # k
    touched = sorted(set(bad_s) | set(bad_theta) | {15, 18})
    res = R.compute_all_dimensionless_batch(kind, s2, th2, par2)
    rest = np.setdiff1d(np.arange(len(s)), touched)
    assert np.array_equal(res.values[:, rest], clean[:, rest], equal_nan=True)
    for i in (0, 1, 3, 6, 15):   # nothing can be computed from these
        assert np.isnan(res.values[:, i]).all() and (res.status[i] & (R.STATUS_NAN | R.STATUS_NORM_FAILED))
    for i in touched:            # every slot is either a number or NaN-with-status, never garbage
        bad = np.isnan(res.values[:, i])
        assert not bad.any() or (res.status[i] & (R.STATUS_NAN | R.STATUS_NORM_FAILED))
        assert np.isfinite(res.values[:, i][~bad]).all()


def test_results_do_not_depend_on_batch_order_or_composition():
    """Points are independent: any permutation or split of the batch gives bitwise the same values,
    and so does running it twice (no races in the shared-memory interval lists)."""
    kind, s, theta, params = R.synthetic_batch("pitchy_pl", 4096, seed=11)
    a = R.compute_all_dimensionless_batch(kind, s, theta, params, extras=True)
    b = R.compute_all_dimensionless_batch(kind, s, theta, params, extras=True)
    assert np.array_equal(a.values, b.values, equal_nan=True) and np.array_equal(a.status, b.status)
    perm = np.random.default_rng(0).permutation(len(s))
    pp = [p[perm] if np.ndim(p) else p for p in params]
    c = R.compute_all_dimensionless_batch(kind, s[perm], theta[perm], pp)
    assert np.array_equal(c.values, a.values[:, perm], equal_nan=True)
    # symphony slots never fail on this envelope; Faraday NaNs only in the s sin(theta) < 3 corner
    assert not np.isnan(a.values[:6]).any()
    sigma0 = s * np.sin(theta)
    assert not np.isnan(a.values[6:, sigma0 >= 3.0]).any()
    assert ((a.status & R.STATUS_NAN) != 0).tolist() == np.isnan(a.values).any(axis=0).tolist()
    # budgets only bind where the Heyvaerts expansions are outside their range (s sin(theta) < 1)
    assert (a.status & R.STATUS_CAP_HIT)[sigma0 >= 3.0].mean() < 0.002
    # physics: |j_Q| <= j_I, |j_V| <= j_I, j_I > 0, alpha_V is the sum of its lobes
    assert (a.values[0] > 0).all() and (np.abs(a.values[2]) <= a.values[0]).all() and (np.abs(a.values[4]) <= a.values[0]).all()
    assert np.allclose(a.lobes[0] + a.lobes[1], a.values[4], rtol=1e-12, atol=0) and np.allclose(a.lobes[2] + a.lobes[3], a.values[5], rtol=1e-12, atol=0)


def test_coefficient_mask_and_broadcast_parameters():
    kind, s, theta, params = R.synthetic_batch("pitchy_pl", 64, seed=5)
    full = R.compute_all_dimensionless_batch(kind, s, theta, params).values
    only = R.compute_all_dimensionless_batch(kind, s, theta, params, coeff_mask=(1 << 2) | (1 << 7)).values
    assert np.array_equal(only[2], full[2], equal_nan=True) and np.array_equal(only[7], full[7], equal_nan=True)
    assert np.isnan(only[[0, 1, 3, 4, 5, 6]]).all()
    expanded = [np.full(len(s), p) if not np.ndim(p) else p for p in params]
    again = R.compute_all_dimensionless_batch(kind, s, theta, expanded).values
    assert np.array_equal(again, full, equal_nan=True)
    short = R.compute_all_dimensionless_batch(kind, s, theta, params[:2]).values  # trailing defaults of pitchy_pl.rs:73-82
    assert np.array_equal(short, full, equal_nan=True)


def test_device_pointer_path_and_multi_entry_agree_with_host_path():
    import torch
    kind, s, theta, params = R.synthetic_batch("powerlaw", 257, seed=2)
    host = R.compute_all_dimensionless_batch(kind, s, theta, params)
    dev = torch.device("cuda", 0)
    d_s, d_t = torch.from_numpy(s).to(dev), torch.from_numpy(theta).to(dev)
    d_p = [torch.from_numpy(np.atleast_1d(np.asarray(p, dtype=np.float64))).to(dev) for p in params]
    d_out = torch.empty(8 * len(s), dtype=torch.float64, device=dev)
    d_status = torch.zeros(len(s), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        R.compute_all_dimensionless_device(kind, d_s, d_t, d_p, d_out, d_status, stream=torch.cuda.current_stream())
    assert np.array_equal(d_out.cpu().numpy().reshape(8, -1), host.values, equal_nan=True)
    assert np.array_equal(d_status.cpu().numpy(), host.status)
    multi = R.compute_all_dimensionless_batch(kind, s, theta, params, n_devices=0)
    assert np.array_equal(multi.values, host.values, equal_nan=True) and np.array_equal(multi.status, host.status)


def test_multi_entry_shards_over_two_gpus_bitwise():
    """north_star's sharding path (one process, one host thread + stream per GPU, host gather): the
    result must be bit-identical to the single-device one, odd sizes and broadcast columns included."""
    if R.device_count() < 2:
        pytest.skip("needs two GPUs")
    kind, s, theta, params = R.synthetic_batch("pitchy_pl", 1001, seed=4)
    one = R.compute_all_dimensionless_batch(kind, s, theta, params, device=0)
    for nd in (2, 0):
        multi = R.compute_all_dimensionless_batch(kind, s, theta, params, n_devices=nd)
        assert np.array_equal(multi.values, one.values, equal_nan=True)
        assert np.array_equal(multi.status, one.status)
    # fewer points than devices
    tiny = R.compute_all_dimensionless_batch(kind, s[:1], theta[:1], [np.asarray(p)[:1] if np.ndim(p) else p for p in params],
                                             n_devices=2)
    assert np.array_equal(tiny.values[:, 0], one.values[:, 0], equal_nan=True)


def test_async_calls_on_two_streams_do_not_race():
    """The device entry with synchronize=0 on two different streams back to back: the library's
    per-device scratch is protected by an on-device wait on the previous call's completion event
    (include/rimphony_b200.h), so both results must equal the synchronous ones."""
    import torch
    dev = torch.device("cuda", 0)
    batches = [R.synthetic_batch("pitchy_pl", 3000, seed=21), R.synthetic_batch("pitchy_kappa", 1500, seed=22)]
    want = [R.compute_all_dimensionless_batch(k, s, th, p, device=0) for k, s, th, p in batches]
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    outs, keep = [], []
    for (kind, s, th, p), st in zip(batches, streams):
        d_s, d_t = torch.from_numpy(s).to(dev), torch.from_numpy(th).to(dev)
        d_p = [torch.from_numpy(np.atleast_1d(np.asarray(c, dtype=np.float64))).to(dev) for c in p]
        d_out = torch.full((8 * len(s),), float("nan"), dtype=torch.float64, device=dev)
        d_status = torch.zeros(len(s), dtype=torch.int32, device=dev)
        keep.append((d_s, d_t, d_p))
        outs.append((d_out, d_status))
    torch.cuda.synchronize()
    for (kind, s, th, p), st, (d_s, d_t, d_p), (d_out, d_status) in zip(batches, streams, keep, outs):
        R.compute_all_dimensionless_device(kind, d_s, d_t, d_p, d_out, d_status, stream=st, synchronize=False)
    torch.cuda.synchronize()
    for (d_out, d_status), w in zip(outs, want):
        assert np.array_equal(d_out.cpu().numpy().reshape(8, -1), w.values, equal_nan=True)
        assert np.array_equal(d_status.cpu().numpy(), w.status)


def test_calls_leave_the_current_device_alone():
    import torch
    if R.device_count() < 2:
        pytest.skip("needs two GPUs")
    torch.cuda.set_device(0)
    kind, s, theta, params = R.synthetic_batch("powerlaw", 8, seed=2)
    R.compute_all_dimensionless_batch(kind, s, theta, params, device=1)
    assert torch.cuda.current_device() == 0


def test_high_harmonic_corner_runs_and_is_finite():
    """BASELINE C4: s >= 1e5 (rel_width switch at s >= 1e6, symphony.rs:337-341)."""
    s = np.array([1e5, 3e5, 1e6, 3e6, 1e7])
    theta = np.array([0.8, 0.3, 1.2, 0.05, 0.8])
    calc = R.PitchyKappaDistribution(3.0, 5.0, 1.0).gamma_cutoff(1e10).full_calculation()
    res = calc.compute_all_dimensionless_batch(s, theta, extras=True)
    assert np.isfinite(res.values[:6]).all()
    assert (res.values[0] > 0).all()


def test_bench_dumps_what_the_timed_steps_computed(tmp_path):
    """bench.py --dump-outputs writes the device buffers of the last timed step: the library's own result for the
    same seeded points, bit for bit, with its NaNs moved into nan_mask so that every dumped value is finite."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n = 2048
    subprocess.check_call([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "1", "--points", str(n),
                           "--no-parity", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], timeout=600,
                          stdout=subprocess.DEVNULL)
    import bench
    kind, s, theta, params = bench.draw("pitchy_pl", n)
    want = R.compute_all_dimensionless_batch(kind, s, theta, params)
    assert np.load(tmp_path / "index.npy").tolist() == list(range(n))
    values, nan_mask = np.load(tmp_path / "coefficients.npy"), np.load(tmp_path / "nan_mask.npy")
    assert np.isfinite(values).all() and np.array_equal(nan_mask == 1.0, np.isnan(want.values))
    assert np.array_equal(np.where(nan_mask == 1.0, np.nan, values), want.values, equal_nan=True)
    assert np.array_equal(np.load(tmp_path / "status.npy"), want.status.astype(np.float64))


def test_graft_entry_smoke():
    import __graft_entry__ as g
    g.smoke()
