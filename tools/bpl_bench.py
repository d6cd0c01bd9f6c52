"""Throughput of the pitchy broken power law next to the pitchy power law, in one process on one GPU.

Both kinds run their seeded synthetic batches (sampler configs pitchy_bpl and pitchy_pl, N points each) in
FAST mode, alternated REPS times after a warm-up call each.  For each kind it prints sets/s (N over the
wall time of the synchronous call, copies included), ms per step, the device span of the kernels and the rule
applications per point in Symphony and Heyvaerts, with the card's name, power limit and SM clock read in the
same process.  Writes the JSON lines to OUTDIR/bpl_bench.jsonl when OUTDIR is given.
usage: python tools/bpl_bench.py [N=131072] [REPS=3] [OUTDIR]"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rimphony_b200 as R  # noqa: E402


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                              capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}
    return dict(zip(q.split(","), (v.strip() for v in line.split(","))))


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 131072
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    outdir = sys.argv[3] if len(sys.argv) > 3 else None
    batches = {cfg: R.synthetic_batch(cfg, n, seed=20260) for cfg in ("pitchy_pl", "pitchy_bpl")}
    for kind, s, theta, params in batches.values():   # warm-up: module load, scratch buffers
        R.compute_all_dimensionless_batch(kind, s[:4096], theta[:4096], [p[:4096] if np.ndim(p) else p for p in params])
    runs = {cfg: [] for cfg in batches}
    for _ in range(reps):
        for cfg, (kind, s, theta, params) in batches.items():
            t0 = time.perf_counter()
            res = R.compute_all_dimensionless_batch(kind, s, theta, params, extras=True)
            wall = time.perf_counter() - t0
            runs[cfg].append((wall, res))
    info = card()
    lines = []
    for cfg, rs in runs.items():
        walls = np.array([w for w, _ in rs])
        res = rs[int(np.argmin(walls))][1]
        lines.append({
            "config": cfg, "n": n, "reps": reps, "mode": "FAST",
            "sets_per_s": round(n / walls.min(), 1), "ms_per_step": round(1e3 * walls.min(), 2),
            "ms_per_step_all": [round(1e3 * w, 2) for w in walls],
            "kernel_span_ms": round(float(res.kernel_ms[3]), 2),
            "apps_per_point_symphony": round(float(res.counters[0].mean()), 1),
            "apps_per_point_heyvaerts": round(float(res.counters[1].mean()), 1),
            "nan_fraction": [round(float(v), 4) for v in np.isnan(res.values).mean(axis=1)],
            "card": info,
        })
    lines.append({"ratio_sets_per_s_bpl_over_pl": round(lines[1]["sets_per_s"] / lines[0]["sets_per_s"], 3)})
    text = "".join(json.dumps(ln) + "\n" for ln in lines)
    print(text, end="")
    if outdir:
        os.makedirs(outdir, exist_ok=True)
        with open(os.path.join(outdir, "bpl_bench.jsonl"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
