"""Random parameter generation for the crank-out workloads.

``Sampler`` mirrors ``rimphony_test_support::Sampler`` (test-support/src/lib.rs:31-64):
uniform, or log-uniform = exp(U[ln lo, ln hi]).  ``synthetic_batch`` draws the
benchmark / parity configurations of BASELINE.md with a counter-based generator
(numpy Philox), so that any shard of a batch can be regenerated independently.
"""
import math

import numpy as np

POWER_LAW, THERMAL_JUETTNER, PITCHY_PL, PITCHY_KAPPA, PITCHY_BROKEN_PL = 0, 1, 2, 3, 4


class Sampler:
    """test-support/src/lib.rs:31-64"""

    def __init__(self, is_log, low, high, rng=None):
        if low > high:
            low, high = high, low
        if is_log:
            low, high = math.log(low), math.log(high)
        self.is_log = bool(is_log)
        self.low = low
        self.range = high - low
        self.rng = rng if rng is not None else np.random.default_rng()

    def get(self, size=None):
        n = self.low + self.rng.random(size) * self.range
        return np.exp(n) if self.is_log else n


# name -> (kind, [(column, is_log, lo, hi) ...] for s, theta and the sampled parameter columns,
#          fixed trailing columns)
CONFIGS = {
    # C2: benches/powerlaw.rs shape, golden-file envelope
    "powerlaw": (POWER_LAW,
                 [("s", True, 0.07, 1e4), ("theta", False, 0.003, 1.5705), ("p", False, 1.5, 4.0)],
                 [1.0, 1e12, 1e10]),
    # C3: crank-out-pitchypl.rs / neurosynchro training-set shape
    "pitchy_pl": (PITCHY_PL,
                  [("s", True, 0.07, 1e4), ("theta", False, 0.003, 1.5705), ("p", False, 1.5, 4.0),
                   ("k", False, 0.0, 3.0)],
                  [1.0, 1e12, 1e10]),
    # C4: crank-out-pitchykappa.rs incl. the s >= 1e5 corner
    "pitchy_kappa": (PITCHY_KAPPA,
                     [("s", True, 1.0, 1e6), ("theta", False, 0.003, 1.5705), ("kappa", False, 1.5, 4.5),
                      ("width", True, math.e, math.e ** 3), ("k", False, 0.0, 3.0)],
                     [1e10]),
    # a cooled population: a power law that steepens by 0.5-1.5 above a break; the drawn column
    # `dp` is replaced by p2 = p1 + dp
    "pitchy_bpl": (PITCHY_BROKEN_PL,
                   [("s", True, 0.07, 1e4), ("theta", False, 0.003, 1.5705), ("p1", False, 1.5, 3.0),
                    ("dp", False, 0.5, 1.5), ("gamma_break", True, 10.0, 1e4), ("k", False, 0.0, 3.0)],
                   [1.0, 1e12, 1e10]),
}


def synthetic_batch(config, n, seed=20260, shard=0, sequential=False):
    """Draw ``n`` points of a named configuration.

    Returns ``(kind, s, theta, params)`` where ``params`` is the list of columns of
    the C ABI (sampled columns as arrays, fixed trailing columns as scalars).
    ``shard`` selects an independent Philox key, e.g. the rank of a GPU.  Every column
    has its own counter block of that key, so the first m points of a batch do not depend
    on n: the 10^4-point parity fixtures are prefixes of the benchmark batches (SURVEY 8d).
    ``sequential=True`` is the round-1 draw (one stream, column after column), kept so that
    tests/golden/make_golden.py still regenerates the round-1 fixtures.
    """
    if config == "juettner_sweep":
        return juettner_sweep()
    kind, cols, fixed = CONFIGS[config]
    rng = np.random.Generator(np.random.Philox(key=[int(seed), int(shard)]))
    drawn = {}
    for j, (name, is_log, lo, hi) in enumerate(cols):
        if not sequential:
            rng = np.random.Generator(np.random.Philox(key=[int(seed), int(shard)], counter=[0, 0, 0, j + 1]))
        drawn[name] = Sampler(is_log, lo, hi, rng).get(n)
    if "dp" in drawn:
        drawn["dp"] = drawn["p1"] + drawn["dp"]
    s = drawn.pop("s")
    theta = drawn.pop("theta")
    params = [drawn[name] for name, *_ in cols[2:]] + list(fixed)
    return kind, s, theta, params


def juettner_sweep():
    """C5: T on 64 log-spaced values in [1, 100] x s on 128 log-spaced values in
    [1, 1e6] x theta in {0.4, pi/4}."""
    t = np.logspace(0, 2, 64)
    s = np.logspace(0, 6, 128)
    th = np.array([0.4, 0.25 * math.pi])
    tt, ss, thth = np.meshgrid(t, s, th, indexing="ij")
    return THERMAL_JUETTNER, ss.ravel().copy(), thth.ravel().copy(), [tt.ravel().copy()]
