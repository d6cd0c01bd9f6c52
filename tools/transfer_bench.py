"""Throughput of the polarized transfer, alone and inside the fused coefficients-and-transfer call, in one
process on one GPU.

* Transfer only: RAYS rays of 1 and of 64 cells (random physical coefficients drawn on the device), through
  rimphony_b200_transfer_device on a torch stream; CUDA events on that stream around each call, REPS calls
  after a warm-up.  Prints rays/s and cells/s.
* Fused: N seeded C3 points (sampler config pitchy_pl) as N uniform slabs, compute_stokes_cgs next to
  compute_all_dimensionless_batch on the same points (host arrays, copies included), alternated REPS times.
  The transfer's share of the fused call is the transfer-only time of N one-cell rays over the fused time.
Every figure comes with its spread over the REPS runs and with the card's name, power limit and SM clock read in
the same process.  Writes the JSON lines to OUTDIR/transfer_bench.jsonl when OUTDIR is given.
usage: python tools/transfer_bench.py [RAYS=1000000] [N=131072] [REPS=5] [OUTDIR]"""
import json
import math
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


def spread(v):
    v = np.asarray(v, dtype=np.float64)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}


def random_rays(torch, n_rays, n_cells, dev):
    g = torch.Generator(device=dev).manual_seed(20261022)
    shape = (n_rays * n_cells,)
    u = lambda lo, hi: lo + (hi - lo) * torch.rand(shape, generator=g, device=dev, dtype=torch.float64)  # noqa: E731
    ds = 10.0 ** u(12, 16)
    a_i = 10.0 ** u(-6, 1.5) / ds
    pol, ang, rho_ang, jang = u(0, 1) * a_i, u(0, 2 * math.pi), u(0, 2 * math.pi), u(0, 2 * math.pi)
    rho = 10.0 ** u(-8, 3) / ds
    j_i = 10.0 ** u(-22, -18)
    jpol = u(0, 1) * j_i
    coeffs = torch.stack([j_i, a_i, jpol * torch.cos(jang), pol * torch.cos(ang), jpol * torch.sin(jang),
                          pol * torch.sin(ang), rho * torch.cos(rho_ang), rho * torch.sin(rho_ang)]).contiguous()
    return coeffs, u(-math.pi, math.pi), ds


def transfer_only(torch, n_rays, n_cells, reps, dev):
    coeffs, psi, ds = random_rays(torch, n_rays, n_cells, dev)
    out = torch.empty(4 * n_rays, dtype=torch.float64, device=dev)
    status = torch.empty(n_rays, dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)  # not the legacy default stream, which the library does not use
    stream.wait_stream(torch.cuda.current_stream(dev))
    R.transfer_device(coeffs, psi, ds, out, None, status, stream=stream)  # warm-up
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        R.transfer_device(coeffs, psi, ds, out, None, status, stream=stream, synchronize=False)
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    nan = float(torch.isnan(out).double().mean())
    del coeffs, psi, ds, out, status
    torch.cuda.empty_cache()
    return {"what": "transfer_only", "n_rays": n_rays, "n_cells": n_cells, "ms": spread(ms),
            "rays_per_s": n_rays / (np.median(ms) * 1e-3), "cells_per_s": n_rays * n_cells / (np.median(ms) * 1e-3),
            "nan_fraction": nan}


def fused(n, reps):
    kind, s, theta, params = R.synthetic_batch("pitchy_pl", n, seed=20260)
    rng = np.random.default_rng(5)
    b = 10.0 ** rng.uniform(-1, 2, n)
    nu = s * (R.ELECTRON_CHARGE * b / (R.TWO_PI * R.MASS_ELECTRON * R.SPEED_LIGHT))
    n_e, psi, ds = 10.0 ** rng.uniform(2, 6, n), rng.uniform(-np.pi, np.pi, n), 10.0 ** rng.uniform(12, 16, n)
    w = slice(0, 4096)
    R.compute_all_dimensionless_batch(kind, s[w], theta[w], [p[w] if np.ndim(p) else p for p in params])
    R.compute_stokes_cgs(kind, nu[w], b[w], n_e[w], theta[w], psi[w], ds[w], [p[w] if np.ndim(p) else p for p in params])
    coeff_s, stokes_s = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        R.compute_all_dimensionless_batch(kind, s, theta, params)
        coeff_s.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        res = R.compute_stokes_cgs(kind, nu, b, n_e, theta, psi, ds, params)
        stokes_s.append(time.perf_counter() - t0)
    return {"what": "fused_vs_coefficients", "config": "pitchy_pl (C3)", "n": n, "mode": "FAST",
            "compute_all_dimensionless_batch_ms": spread(1e3 * np.array(coeff_s)),
            "compute_stokes_cgs_ms": spread(1e3 * np.array(stokes_s)),
            "coefficient_sets_per_s": n / np.median(coeff_s), "stokes_slabs_per_s": n / np.median(stokes_s),
            "ray_nan_fraction": float(np.isnan(res.stokes[0]).mean())}


def main():
    import torch

    rays = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 131072
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    outdir = sys.argv[4] if len(sys.argv) > 4 else None
    if R.device_count() < 1:
        raise SystemExit("transfer_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    lines = [transfer_only(torch, rays, 1, reps, dev), transfer_only(torch, rays, 64, reps, dev),
             transfer_only(torch, n, 1, reps, dev), fused(n, reps)]
    share = lines[2]["ms"]["median"] / lines[3]["compute_stokes_cgs_ms"]["median"]
    lines.append({"transfer_share_of_fused_call": share, "card": card()})
    text = "".join(json.dumps(ln) + "\n" for ln in lines)
    print(text, end="")
    if outdir:
        os.makedirs(outdir, exist_ok=True)
        with open(os.path.join(outdir, "transfer_bench.jsonl"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
