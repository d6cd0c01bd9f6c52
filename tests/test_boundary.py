"""The drop-in boundary and the host logic, without a GPU: the C-ABI library loads and exports
every symbol include/rimphony_b200.h declares, struct layouts agree, the facade mirrors the
reference's names and error behaviour, and the product never touches the oracle."""
import ctypes
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import rimphony_b200 as R
from rimphony_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rimphony_b200.h")
GCC = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rimphony_b200_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    L = _lib.load()
    names = declared_functions()
    assert len(names) >= 14
    for name in names:
        assert hasattr(L, name), f"{name} is declared in the header but not exported"
    assert sorted(_lib.EXPORTED_SYMBOLS) == names
    assert L.rimphony_b200_abi_version() == 2


def test_header_is_plain_c_and_struct_layout_matches(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "rimphony_b200.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu\n", sizeof(rimphony_b200_options), offsetof(rimphony_b200_options, coeff_mask),
           offsetof(rimphony_b200_options, device_plus_one), offsetof(rimphony_b200_options, epsrel_gamma),
           offsetof(rimphony_b200_options, epsrel_heyvaerts_outer), sizeof(rimphony_b200_extras));
    return 0;
}''')
    exe = tmp_path / "layout"
    subprocess.check_call([GCC, "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    O = _lib.Options
    assert got == [ctypes.sizeof(O), O.coeff_mask.offset, O.device_plus_one.offset, O.epsrel_gamma.offset,
                   O.epsrel_heyvaerts_outer.offset, ctypes.sizeof(_lib.Extras)]
    # and as C++
    cpp = tmp_path / "layout.cpp"
    cpp.write_text('#include "rimphony_b200.h"\nint main() { return rimphony_b200_abi_version() * 0; }\n')
    subprocess.check_call([GXX, "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(cpp)])


def test_no_cuda_types_in_signatures():
    text = open(HEADER).read()
    assert "cudaStream_t " not in re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    assert "#include <cuda" not in text and "torch" not in re.sub(r"/\*.*?\*/", "", text, flags=re.S)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "rimphony_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle", text, flags=re.M), f
                assert "liboracle" not in text and "oracle/_ref" not in text and "libleung_ref" not in text, f
                assert "#include \"../../oracle" not in text and "rimphony_oracle.h" not in text, f


@pytest.mark.skipif(R.device_count() > 0, reason="a CUDA device is present")
def test_fails_loudly_without_a_gpu():
    calc = R.PowerLawDistribution(2.5).full_calculation()
    with pytest.raises(R.RimphonyB200Error):
        calc.compute_all_dimensionless(1.0, 0.5)
    with pytest.raises(R.RimphonyB200Error):
        R.bessel_jn(50.0, 40.0)


def test_bad_arguments_are_infrastructure_errors():
    L = _lib.load()
    s = (ctypes.c_double * 1)(1.0)
    cols = (_lib.c_double_p * 1)(ctypes.cast(s, _lib.c_double_p))
    out = (ctypes.c_double * 8)()
    # POWER_LAW takes 1 or 4 columns, never 2
    assert L.rimphony_b200_compute_all_dimensionless(R.POWER_LAW, 1, s, s, cols, 2, None, out, None) != 0
    assert b"POWER_LAW" in L.rimphony_b200_last_error()
    assert L.rimphony_b200_compute_all_dimensionless(17, 1, s, s, cols, 1, None, out, None) != 0
    assert L.rimphony_b200_compute_all_dimensionless(R.POWER_LAW, -1, s, s, cols, 1, None, out, None) != 0
    # an empty batch is a successful no-op, with or without a device
    assert L.rimphony_b200_compute_all_dimensionless(R.POWER_LAW, 0, s, s, cols, 1, None, out, None) == 0
    # diagnostics: Faraday is not a Symphony coefficient; two-argument diagnostics need both arrays
    p = (ctypes.c_double * 1)(2.5)
    assert L.rimphony_b200_diagnostic_symphony(R.POWER_LAW, p, 1, 2, 0, 10.0, 0.5, 1, 1, s, None, out, None) != 0
    assert L.rimphony_b200_diagnostic_symphony(R.POWER_LAW, p, 1, 0, 0, 10.0, 0.5, 0, 1, s, None, out, None) != 0
    assert L.rimphony_b200_diagnostic_symphony(R.POWER_LAW, p, 1, 0, 0, 10.0, 0.5, 9, 1, s, s, out, None) != 0
    assert L.rimphony_b200_diagnostic_symphony(R.POWER_LAW, p, 1, 0, 0, 10.0, 0.5, 1, 0, s, None, out, None) == 0
    with pytest.raises(ValueError):
        R.PowerLawDistribution(2.5).full_calculation().diagnostic_symphony_gamma_integral(
            R.Coefficient.Faraday, R.Stokes.Q, 10.0, 0.5, 40.0)


def test_output_slots_follow_lib_rs():
    """src/lib.rs:176-191: [j_I, alpha_I, j_Q, alpha_Q, j_V, alpha_V, rho_Q, rho_V]."""
    C, S = R.Coefficient, R.Stokes
    order = [(C.Emission, S.I), (C.Absorption, S.I), (C.Emission, S.Q), (C.Absorption, S.Q),
             (C.Emission, S.V), (C.Absorption, S.V), (C.Faraday, S.Q), (C.Faraday, S.V)]
    assert [R.output_slot(c, s) for c, s in order] == list(range(8))
    assert R.output_slot(C.Faraday, S.I) == -1
    assert R.COEFFICIENT_NAMES == ("j_I", "alpha_I", "j_Q", "alpha_Q", "j_V", "alpha_V", "rho_Q", "rho_V")


def test_faraday_stokes_i_is_nan_without_touching_the_device():
    calc = R.PitchyPowerLawDistribution(2.5, 1.0).full_calculation()
    assert math.isnan(calc.compute_dimensionless(R.Coefficient.Faraday, R.Stokes.I, 10.0, 0.5))  # lib.rs:239-240
    got = calc.compute_dimensionless(R.Coefficient.Faraday, R.Stokes.I, np.array([1.0, 2.0]), np.array([0.5, 0.6]))
    assert got.shape == (2,) and np.isnan(got).all()


def test_constants_and_defaults_match_the_reference():
    assert R.MASS_ELECTRON == 9.1093826e-28 and R.SPEED_LIGHT == 2.99792458e10 and R.ELECTRON_CHARGE == 4.80320680e-10
    assert R.TWO_PI == 2 * math.pi
    assert R.PowerLawDistribution(2.5)._columns() == [2.5, 1.0, 1e12, 1e10]              # power_law.rs:71-79
    assert R.PitchyPowerLawDistribution(2.5, 1.0)._columns() == [2.5, 1.0, 1.0, 1e12, 1e10]  # pitchy_pl.rs:73-82
    assert R.PitchyKappaDistribution(3.0, 5.0, 1.0)._columns() == [3.0, 5.0, 1.0, 1e10]   # pitchy_kappa.rs:70-79
    assert R.PowerLawDistribution(2.5).gamma_limits(10.0, 1e12, 1e10)._columns()[1] == 10.0
    assert R.PitchyKappaDistribution(3.0, 5.0, 1.0).gamma_cutoff(1e8)._columns()[3] == 1e8


def test_compute_cgs_scaling():
    """src/lib.rs:163-173 and 196-209 against a stub calculator."""
    class Stub(R.SynchrotronCalculator):
        def compute_dimensionless(self, coeff, stokes, s, theta):
            return 2.0 * s

        def compute_all_dimensionless(self, s, theta):
            return np.full(8, 2.0 * s)

    nu, b, n_e = 1e9, 1e3, 7.0
    nu_c = R.ELECTRON_CHARGE * b / (R.TWO_PI * R.MASS_ELECTRON * R.SPEED_LIGHT)
    st = Stub()
    assert st.compute_cgs(R.Coefficient.Emission, R.Stokes.I, nu, b, n_e, 0.3) == pytest.approx(2 * nu / nu_c * n_e * nu)
    assert st.compute_cgs(R.Coefficient.Absorption, R.Stokes.Q, nu, b, n_e, 0.3) == pytest.approx(2 * nu / nu_c * n_e / nu)
    assert st.compute_cgs(R.Coefficient.Faraday, R.Stokes.V, nu, b, n_e, 0.3) == pytest.approx(2 * nu / nu_c * n_e / nu)
    allc = st.compute_all_cgs(nu, b, n_e, 0.3)
    assert allc[0] == pytest.approx(2 * nu / nu_c * n_e * nu) and allc[7] == pytest.approx(2 * nu / nu_c * n_e / nu)


def test_sampler_semantics():
    """test-support/src/lib.rs:39-63: swapped bounds, log-uniform = exp(U[ln lo, ln hi])."""
    rng = np.random.default_rng(0)
    lin = R.Sampler(False, 3.0, 1.0, rng)
    v = lin.get(10000)
    assert v.min() >= 1.0 and v.max() <= 3.0 and abs(v.mean() - 2.0) < 0.05
    lg = R.Sampler(True, 0.07, 1e4, rng)
    v = lg.get(20000)
    assert v.min() >= 0.07 and v.max() <= 1e4
    assert abs(np.log(v).mean() - 0.5 * (math.log(0.07) + math.log(1e4))) < 0.1


def test_synthetic_batches_are_reproducible_and_sharded():
    k1, s1, t1, p1 = R.synthetic_batch("pitchy_pl", 1000, seed=5, shard=0)
    k2, s2, t2, p2 = R.synthetic_batch("pitchy_pl", 1000, seed=5, shard=0)
    k3, s3, _, _ = R.synthetic_batch("pitchy_pl", 1000, seed=5, shard=1)
    assert k1 == R.PITCHY_PL and np.array_equal(s1, s2) and np.array_equal(t1, t2)
    assert all(np.array_equal(a, b) for a, b in zip(p1, p2))
    assert not np.array_equal(s1, s3)
    assert 0.07 <= s1.min() and s1.max() <= 1e4 and 0.003 <= t1.min() and t1.max() <= 1.5705
    assert 1.5 <= p1[0].min() and p1[0].max() <= 4.0 and 0.0 <= p1[1].min() and p1[1].max() <= 3.0
    assert p1[2:] == [1.0, 1e12, 1e10]
    kk, sk, tk, pk = R.synthetic_batch("pitchy_kappa", 4000, seed=5)
    assert kk == R.PITCHY_KAPPA and 0.1 < (sk >= 1e5).mean() < 0.25  # the high-harmonic corner (BASELINE C4)
    kj, sj, tj, pj = R.synthetic_batch("juettner_sweep", 0)
    assert kj == R.THERMAL_JUETTNER and len(sj) == 64 * 128 * 2 and pj[0].min() == 1.0 and pj[0].max() == pytest.approx(100.0)


def test_bench_reference_arm_line(tmp_path):
    """bench.py --impl reference prints one JSON line with the contract's keys (tiny sample)."""
    import json
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                                   "--warmup", "0", "--cpu-sample", "4", "--config", "powerlaw",
                                   "--dump-outputs", str(tmp_path / "dump")],
                                  env={**os.environ, "OMP_NUM_THREADS": "4"}, timeout=300)
    line = json.loads(out.decode().strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "coefficient-sets/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["higher_is_better"] is True and line["dtype"] == "f64"
    values = np.load(tmp_path / "dump" / "coefficients.npy")
    nan_mask = np.load(tmp_path / "dump" / "nan_mask.npy")
    assert values.shape == nan_mask.shape == (8, 4) and values.dtype == nan_mask.dtype == np.float64
    assert np.isfinite(values).all() and not nan_mask[:6].any() and (values[0] > 0).all()
    # the last (second) step computed points 4 .. 7 of the seeded batch, and the dump says so
    index = np.load(tmp_path / "dump" / "index.npy")
    assert index.tolist() == [4.0, 5.0, 6.0, 7.0]
    import bench
    from oracle import oracle as O
    kind, s, theta, params = R.synthetic_batch("powerlaw", 8, seed=bench.SEED)
    sel = index.astype(np.int64)
    want, _ = O.batch(kind, s[sel], theta[sel], [np.asarray(p)[sel] if np.ndim(p) else p for p in params])
    assert np.array_equal(np.where(nan_mask == 1.0, np.nan, values), want, equal_nan=True)


def test_bench_dump_outputs_is_bounded_and_reproducible(tmp_path):
    """--dump-outputs: a batch above 64 MB is cut to the same seeded sample of points on every run; NaN is written
    as 0 with its place in nan_mask, so that every dumped value is finite."""
    import bench
    n = 600_000   # 8 coefficients + 8 NaN flags + status + index = 144 bytes per point: 86 MB in all
    values = np.arange(8 * n, dtype=np.float64).reshape(8, n)
    values[6:, ::3] = np.nan
    status = np.arange(n, dtype=np.int32) % 7
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), values, status)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert 60 << 20 < total <= 64 << 20
    for f in ("coefficients.npy", "nan_mask.npy", "status.npy", "index.npy"):
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b) and np.isfinite(a).all()
    idx = np.load(tmp_path / "a" / "index.npy").astype(np.int64)
    assert (np.diff(idx) > 0).all()
    nan_mask = np.load(tmp_path / "a" / "nan_mask.npy")
    assert np.array_equal(nan_mask == 1.0, np.isnan(values[:, idx])) and nan_mask[6:].any()
    got = np.where(nan_mask == 1.0, np.nan, np.load(tmp_path / "a" / "coefficients.npy"))
    assert np.array_equal(got, values[:, idx], equal_nan=True)
    assert np.array_equal(np.load(tmp_path / "a" / "status.npy"), status[idx].astype(np.float64))


def test_high_frequency_approximations_known_answers():
    """power_law.rs:200-207, 224-231; thermal_juettner.rs:174-181, 194-201 (1 %)."""
    C, S = R.Coefficient, R.Stokes
    pl = R.PowerLawDistribution(2.5).gamma_limits(10.0, 1e12, 1e10).high_freq_approximation()
    assert pl.compute_dimensionless(C.Faraday, S.Q, 1e4, 0.25 * math.pi) == pytest.approx(1.81e-9, rel=0.01)
    assert pl.compute_dimensionless(C.Faraday, S.V, 1e4, 0.25 * math.pi) == pytest.approx(1.19e-8, rel=0.01)
    assert (R.ThermalJuettnerDistribution(10.0).high_freq_approximation()
            .compute_dimensionless(C.Faraday, S.Q, 4e4, 0.4)) == pytest.approx(4.8081e-11, rel=0.01)
    assert (R.ThermalJuettnerDistribution(0.1).high_freq_approximation()
            .compute_dimensionless(C.Faraday, S.V, 40.0, 0.5)) == pytest.approx(3.064e-4, rel=0.01)
    assert math.isnan(pl.compute_dimensionless(C.Emission, S.I, 1e4, 0.5))
    assert math.isnan(pl.compute_dimensionless(C.Faraday, S.I, 1e4, 0.5))
    # array arguments evaluate a batch
    q = pl.compute_dimensionless(C.Faraday, S.Q, np.array([1e3, 1e4]), 0.25 * math.pi)
    assert q.shape == (2,) and q[1] == pytest.approx(1.81e-9, rel=0.01)


def test_rust_facade_declares_the_same_abi():
    """rust/ cannot be compiled in this image (no rustc); what can be checked is that its extern "C" block
    names exactly the symbols of the header and that its Options struct has the header's fields in order."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ffi = open(os.path.join(root, "rust", "src", "ffi.rs")).read()
    declared = set(re.findall(r"pub fn (rimphony_b200_\w+)", ffi))
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    fields = re.findall(r"pub (\w+): ", ffi.split("pub struct Options")[1].split("}")[0])
    assert fields == [name for name, _ in _lib.Options._fields_]
    header = open(os.path.join(root, "include", "rimphony_b200.h")).read()
    assert "ABI_VERSION 2" in header and "ABI version 2" in ffi
