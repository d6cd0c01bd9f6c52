"""A/B of two builds of the library: runs the one RIMPHONY_B200_LIB names (default: the in-tree build; another
one comes from `make -C rimphony_b200/csrc OUT=... OBJDIR=...` in a second checkout) on the seeded pitchy
power-law batch and prints kernel times and a digest of the results (builds that only change scheduling or
code layout must reproduce it bit for bit).
usage: [RIMPHONY_B200_LIB=...] python tools/variant_bench.py [N=131072] [CONFIG=pitchy_pl] [REPS=2]"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rimphony_b200 as R  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 131072
cfg = sys.argv[2] if len(sys.argv) > 2 else "pitchy_pl"
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 2
kind, s, th, params = R.synthetic_batch(cfg, n, seed=1)
tag = os.path.basename(os.environ.get("RIMPHONY_B200_LIB", "default"))
for mk, name in ((0x3F, "sym"), (0xC0, "hey"), (0xFF, "all")):
    best = None
    for _ in range(reps):
        res = R.compute_all_dimensionless_batch(kind, s, th, params, coeff_mask=mk, extras=True)
        ms = res.kernel_ms
        if best is None or ms[3] < best[3]:
            best = ms
    digest = hashlib.sha256(np.ascontiguousarray(res.values).tobytes()).hexdigest()[:12]
    print(f"{tag:36s} {cfg} n={n} {name}: kernel ms norm/sym/hey/span = {[round(v, 1) for v in best]} -> "
          f"{n / best[3] * 1e3:.0f} sets/s; apps/pt sym {res.counters[0].mean():.0f} hey {res.counters[1].mean():.0f}; sha {digest}",
          flush=True)
