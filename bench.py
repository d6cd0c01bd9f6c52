#!/usr/bin/env python
"""bench.py -- coefficient-sets/s of the hot path on N B200s.

    python bench.py --gpus N --steps K --warmup W            # the CUDA path
    python bench.py --impl reference --gpus N ...            # the reference's CPU algorithm

A "step" is one pass of the hot path (normalisation + Symphony + Heyvaerts, all
eight coefficients) over one batch of synthetic pitchy power-law points, the
crank-out-pitchypl workload BASELINE.json's metric is quoted on.  The batch per
GPU is fixed (weak scaling): the full 10 M-point configuration is --points
10000000.  One process per GPU; points are independent, so ranks exchange
nothing on the data path (torch.distributed only carries the barrier and the
max-over-ranks of the timing).

Printed JSON (rank 0): value = whole-job sets/s with inputs resident in HBM;
e2e = the same through the public C ABI with host buffers (H2D and D2H copies
inside the timed region); roofline = FP64 work of the dominant kernel against the
measured FP64 FMA peak; cpu_baseline = the oracle on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "8-coefficient sets/sec"
UNIT = "coefficient-sets/s"
SEED = 20260

# FP64 floating-point operations executed per Gauss-Kronrod application (one pass of the 32 lanes
# over 31 nodes, or over two 15-node panels in the Symphony gamma integral; FMA = 2) and DRAM bytes
# per point of the two product kernels.  Not hand-typed: tools/ncu_constants.py derives them from an
# ncu capture of the head build (the predicated-on thread counts of DFMA / DMUL / DADD and
# dram__bytes_{read,write}.sum of one launch of each kernel, divided by the rule applications /
# points that launch counted) and writes profiles/kernel_constants.json, next to the capture.
CONSTANTS_PATH = os.path.join(ROOT, "profiles", "kernel_constants.json")
# SURVEY 8(d): FP64 flop-equivalents the REFERENCE's algorithm spends per coefficient set on the
# C2/C3 mix (1.4e6 Symphony integrand evaluations x ~1.3 kflop + 2 x ~3e5 Heyvaerts elements x
# ~0.3 kflop): sets/s x W_REF is the reference-equivalent work rate, which may exceed the executed
# rate because the product path shares nodes between coefficients and needs fewer rule applications.
W_REF_FLOP_PER_SET = 2.0e9


def kernel_constants():
    with open(CONSTANTS_PATH) as f:
        return json.load(f)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--points", type=int, default=262144,
                    help="points per GPU per step (the full BASELINE configs[2] batch is 10000000)")
    ap.add_argument("--config", default="pitchy_pl", choices=["pitchy_pl", "powerlaw", "pitchy_kappa", "juettner_sweep"],
                    help="BASELINE configs: pitchy_pl = C3 (the metric's config), powerlaw = C2, pitchy_kappa = C4, "
                         "juettner_sweep = C5 (rho_Q, rho_V on the 64 x 128 x 2 grid; --points is ignored)")
    ap.add_argument("--single-process", action="store_true",
                    help="north_star's sharding: ONE process drives --gpus devices through "
                         "rimphony_b200_compute_all_dimensionless_multi on a FIXED batch of --points points "
                         "(strong scaling, host buffers, host gather inside the timed region)")
    ap.add_argument("--no-parity", action="store_true", help="skip the (untimed) parity leg")
    ap.add_argument("--cpu-sample", type=int, default=0, help="points of the CPU sample (0 = auto, ~20 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy "
                         "(float64; a fixed seeded sample of the points when the whole batch exceeds 64 MB; "
                         "rank 0 only; every value finite): coefficients [8, k] in the slot order j_I, alpha_I, j_Q, "
                         "alpha_Q, j_V, alpha_V, rho_Q, rho_V with 0 where the library returned NaN, nan_mask [8, k] "
                         "(1 there, 0 elsewhere), status [k] (the per-point status bits, absent for --impl reference) "
                         "and index [k] (the points' positions in the seeded batch).  --impl reference dumps the sample "
                         "of its last step, whose size follows the host's cores unless --cpu-sample is given")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES_MAX = 64 << 20


def dump_outputs(out_dir, values, status=None, positions=None):
    """--dump-outputs: values [8, n] (and status [n]) of the last timed step as float64 .npy files, with the
    positions of the dumped points in the batch.  NaN, the library's marker for a coefficient the reference's
    algorithm does not produce (or that was not requested), is written as 0 in coefficients.npy and as 1 in
    nan_mask.npy, so that every dumped value is finite and nothing is lost.  Above DUMP_BYTES_MAX the same
    seeded sample of points is kept on every run, so that two builds can be compared output for output.
    `positions` are the points' positions in the seeded batch (default: the batch itself, 0 .. n-1)."""
    values = np.asarray(values, dtype=np.float64)
    n = values.shape[1]
    per_point = 8 * (2 * values.shape[0] + 1 + (status is not None))
    budget = DUMP_BYTES_MAX - 1024   # the .npy headers
    if n * per_point > budget:
        index = np.sort(np.random.default_rng(SEED).choice(n, budget // per_point, replace=False))
    else:
        index = np.arange(n)
    os.makedirs(out_dir, exist_ok=True)
    kept = values[:, index]
    nan = np.isnan(kept)
    np.save(os.path.join(out_dir, "coefficients.npy"), np.where(nan, 0.0, kept))
    np.save(os.path.join(out_dir, "nan_mask.npy"), nan.astype(np.float64))
    if status is not None:
        np.save(os.path.join(out_dir, "status.npy"), np.asarray(status)[index].astype(np.float64))
    positions = np.arange(n) if positions is None else np.asarray(positions)
    np.save(os.path.join(out_dir, "index.npy"), positions[index].astype(np.float64))


WORKLOADS = {
    "pitchy_pl": ("BASELINE configs[2] (C3), crank-out-pitchypl shape: pitchy power-law points", 10_000_000),
    "powerlaw": ("BASELINE configs[1] (C2), benches/powerlaw.rs shape: isotropic power-law points", 1_000_000),
    "pitchy_kappa": ("BASELINE configs[3] (C4), crank-out-pitchykappa shape incl. s >= 1e5: pitchy kappa points", 10_000_000),
    "juettner_sweep": ("BASELINE configs[4] (C5), thermal Juettner Faraday sweep: T 64 x s 128 x theta 2 grid", 16384),
}
PARITY_FIXTURE = {"pitchy_pl": "pitchy_pl_10k", "powerlaw": "powerlaw_10k", "pitchy_kappa": "pitchy_kappa_10k",
                  "juettner_sweep": "juettner_sweep"}


def coeff_mask_of(config):
    return 0xC0 if config == "juettner_sweep" else 0xFF


def workload_name(config, points):
    what, full = WORKLOADS[config]
    if config == "juettner_sweep":
        return f"{what} = {full} points per step, rho_Q and rho_V only, mode=fast"
    part = "the whole batch" if points >= full else f"a seeded slice of the {full}-point batch; --points {full} runs all of it"
    return f"{what}, {points} points per GPU per step ({part}), all 8 coefficients, mode=fast"


def draw(config, n, shard=0):
    from rimphony_b200.sampler import synthetic_batch
    kind, s, theta, params = synthetic_batch(config, n, seed=SEED, shard=shard)
    return kind, s, theta, params


def parity_leg(config, device):
    """Untimed: the product path on the committed golden fixture of this configuration (the fixed
    1e4-point prefix of the seeded batch, SURVEY 8(d); the oracle's outputs are read from the
    .npz, nothing under oracle/ runs here) -> the `parity` object of the JSON line."""
    import rimphony_b200 as R
    from rimphony_b200 import parity as P

    name = PARITY_FIXTURE[config]
    path = os.path.join(P.GOLDEN_DIR, name + ".npz")
    if not os.path.exists(path):
        return {"fixture": name, "error": "fixture missing"}
    fx = P.load_fixture(name)
    mask = coeff_mask_of(config)
    res = R.compute_all_dimensionless_batch(int(fx["kind"]), fx["s"], fx["theta"], list(fx["params"]), device=device,
                                            coeff_mask=mask)
    stats = P.parity_stats(res.values, fx["out"], fx.get("lobes"), fx["defined"], mask=mask)
    out = P.summarize(stats)
    out["fixture"] = f"tests/golden/{name}.npz"
    out["bar"] = "rel err <= 1e-3 (Stokes V: of the lobe scale) vs the CPU oracle"
    out["reference_undefined_note"] = ("entries where the reference's own algorithm moves by > 1e-3 or flips NaN under "
                                       "epsrel 1e-3 -> 3e-4 or s -> s(1+1e-9) (tests/golden/make_stability.py); excluded "
                                       "from the other counts" if fx["stability_mask"] else "no stability companion: every entry counted")
    verdict = {k: v for k, v in stats.items() if k not in ("rho_Q", "rho_V")}
    if int(fx["kind"]) in (R.POWER_LAW, R.PITCHY_PL) and (mask & 0xC0):
        # rho of the power laws: the bar applies for s >= 1; below, the reference's NaN verdict is a property of
        # its tolerance (tests/golden/heyvaerts_low_s.md) and the agreement of the rule is reported as measured
        for tag, sel in (("rho_s_ge_1", fx["s"] >= 1.0), ("rho_s_lt_1", fx["s"] < 1.0)):
            idx = np.where(sel)[0]
            st = P.parity_stats(res.values[:, idx], fx["out"][:, idx], None, fx["defined"][:, idx], mask=0xC0)
            out[tag] = P.summarize(st)
            if tag == "rho_s_ge_1":
                verdict.update(st)
        out["meets_north_star_scope"] = "j, alpha on every point; rho_Q, rho_V for s >= 1 (rho_s_lt_1 is reported, not judged)"
    else:
        verdict = stats
        out["meets_north_star_scope"] = "every requested coefficient on every point"
    out["meets_north_star"] = bool(P.meets_north_star(verdict))
    out["meets_north_star_but_for_reference_failures"] = bool(P.meets_north_star(verdict, reference_failures_allowed=0.02))
    out["reference_failures_note"] = ("second flag: entries where the reference returned NaN (its QAG gave up) and this path a "
                                      "number are tolerated up to 2 % of the points; a NaN here where the reference has a number "
                                      "never is")
    return out


class ClockSampler:
    """nvidia-smi clocks and throttle reasons during the timed region."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def max_over_ranks(values, world, device):
    """Timing of a multi-GPU step = the slowest rank (one all-reduce MAX of a tiny tensor)."""
    import torch
    import torch.distributed as dist

    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def whole_job_value(points_per_rank, world, steps, ms):
    """Units all ranks processed / max-over-ranks time (weak scaling: per-GPU batch fixed)."""
    return points_per_rank * world * steps / (ms * 1e-3)


def host_threads():
    """Every host core this process may use.  torchrun exports OMP_NUM_THREADS=1 to its workers;
    the CPU arm must not inherit that, it is asked for all the host threads it can use."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def sample_positions(config, first, count):
    """Positions in the seeded batch of `config` of the CPU sample's points [first, first + count)."""
    if config == "juettner_sweep":
        n = WORKLOADS[config][1]
        return (np.arange(first, first + count) * 2731) % n  # 2731 is coprime to 16384: a permutation
    return np.arange(first, first + count)


def cpu_sample(config, first, count):
    """Points [first, first + count) of the seeded batch of `config` (rank 0's shard; the sampler is
    prefix-stable, so these are the same points whatever the batch size).  The Juettner sweep is a
    fixed grid: there the sample strides through it, so that every sample covers the whole (T, s) range."""
    if config == "juettner_sweep":
        kind, s, theta, params = draw(config, 0)
        idx = sample_positions(config, first, count)
        return kind, s[idx], theta[idx], [np.asarray(p)[idx] for p in params]
    kind, s, theta, params = draw(config, first + count)
    sl = slice(first, first + count)
    return kind, s[sl], theta[sl], [np.asarray(p)[sl] if np.ndim(p) else p for p in params]


def cpu_baseline(config, n_sample, kind_label):
    """The oracle (the reference's algorithm; its own bessel.c where at hand) on the host cores: a bounded sample
    of the same seeded batch, in four sub-batches so that the spread is visible."""
    from oracle import oracle as O

    threads = host_threads()
    if n_sample <= 0:
        n_sample = max(16, 12 * threads)  # ~1 s per point per core => ~15-25 s
    parts = 4
    per = max(1, n_sample // parts)
    rates = []
    t_all = 0.0
    for k in range(parts):
        kind, s, theta, params = cpu_sample(config, k * per, per)
        t0 = time.perf_counter()
        O.batch(kind, s, theta, params, coeff_mask=coeff_mask_of(config), n_threads=threads)
        dt = time.perf_counter() - t0
        t_all += dt
        rates.append(per / dt)
    return {"value": parts * per / t_all, "unit": UNIT, "cores": threads, "kind": kind_label,
            "spread": {"min": min(rates), "max": max(rates), "parts": parts},
            "sample": f"points 0..{parts * per - 1} of the seeded {config} batch in {parts} sub-batches, one point per "
                      f"OpenMP thread, {t_all:.1f} s wall"}, t_all


def run_reference(args):
    """--impl reference: the reference's CPU algorithm.  rimphony itself cannot be built in
    this image (no Rust toolchain, no GSL), so this is the oracle port: the restated
    symphony.rs / heyvaerts.rs control flow driving the reference's own bessel.c compiled
    in place (oracle/_ref), or its restatement oracle/leung_bessel.c where that file is not
    at hand (oracle.bessel_source()).  Rank 0 alone runs; other ranks exit 0.  Every step computes a
    DIFFERENT slice of the seeded batch (per-point cost spans more than 10x), so K steps time
    K x sample distinct points; the per-step spread is reported."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as O

    threads = host_threads()
    n_sample = args.cpu_sample if args.cpu_sample > 0 else max(8, 4 * threads)
    mask = coeff_mask_of(args.config)
    for w in range(min(args.warmup, 1)):
        kind, s, theta, params = cpu_sample(args.config, 0, max(threads, 1))
        O.batch(kind, s, theta, params, coeff_mask=mask, n_threads=threads)
    rates = []
    t_all = 0.0
    for k in range(args.steps):
        kind, s, theta, params = cpu_sample(args.config, k * n_sample, n_sample)
        t0 = time.perf_counter()
        values, _ = O.batch(kind, s, theta, params, coeff_mask=mask, n_threads=threads)
        dt = time.perf_counter() - t0
        t_all += dt
        rates.append(n_sample / dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, values, positions=sample_positions(args.config, (args.steps - 1) * n_sample, n_sample))
    value = args.steps * n_sample / t_all
    spread = {"min": min(rates), "median": float(np.median(rates)), "max": max(rates), "steps": args.steps}
    points = WORKLOADS[args.config][1] if args.config == "juettner_sweep" else args.points
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.config, points),
                   "note": "CPU reference arm: each step is a bounded, distinct sample of the workload"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "spread": spread,
                         "sample": f"{n_sample} points per step x {args.steps} steps = points 0..{args.steps * n_sample - 1} "
                                   f"of the seeded {args.config} batch (a different slice every step)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def run_single_process(args):
    """north_star's own sharding, measured: ONE process, a FIXED batch of --points points in host
    memory, rimphony_b200_compute_all_dimensionless_multi cutting it into contiguous slices for
    --gpus devices (one host thread + stream each), results gathered by the host.  Strong scaling;
    the timed region holds H2D, kernels, D2H and the gather; wall clock around synchronous calls."""
    import torch

    import rimphony_b200 as R

    n_dev = args.gpus
    if R.device_count() < n_dev:
        raise SystemExit(f"--single-process --gpus {n_dev}: only {R.device_count()} devices visible")
    n = WORKLOADS[args.config][1] if args.config == "juettner_sweep" else args.points
    mask = coeff_mask_of(args.config)
    kind, s, theta, params = draw(args.config, n)
    h_s = torch.from_numpy(s).pin_memory().numpy()
    h_theta = torch.from_numpy(theta).pin_memory().numpy()
    h_params = [torch.from_numpy(np.ascontiguousarray(p)).pin_memory().numpy() if np.ndim(p) else p for p in params]
    flush = [torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=f"cuda:{d}") for d in range(n_dev)]

    def step():
        for f in flush:
            f.fill_(1)
        return R.compute_all_dimensionless_batch(kind, h_s, h_theta, h_params, coeff_mask=mask, n_devices=n_dev)

    for _ in range(args.warmup):
        step()
    for d in range(n_dev):
        torch.cuda.synchronize(d)
    launches0 = R.kernel_launch_count()
    sampler = ClockSampler(0)
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step()
    for d in range(n_dev):
        torch.cuda.synchronize(d)
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = R.kernel_launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out.values, out.status)
    value = n * args.steps / dt
    h2d = 8 * n * (2 + sum(1 for p in params if np.ndim(p))) + 8 * n_dev * sum(1 for p in params if not np.ndim(p))
    d2h = 8 * 8 * n + 4 * n
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_dev, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.config, n) + f"; FIXED batch of {n} points sharded over {n_dev} GPUs",
                   "seed": SEED, "l2": "flushed between steps (256 MB write per device)",
                   "nan_rate": float(np.isnan(out.values).any(axis=0).mean()),
                   "sharding": f"single process, rimphony_b200_compute_all_dimensionless_multi: {n_dev} contiguous slices, "
                               "one host thread + stream per device, host gather, no collective",
                   "timing": "host wall clock around synchronous C-ABI calls (copies and gather inside)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    if not args.no_parity:
        line["parity"] = parity_leg(args.config, 0)
    print(json.dumps(line))
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.single_process:
        return run_single_process(args)

    import torch
    import torch.distributed as dist

    import rimphony_b200 as R

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    mask = coeff_mask_of(args.config)
    n = WORKLOADS[args.config][1] if args.config == "juettner_sweep" else args.points
    kind, s, theta, params = draw(args.config, n, shard=rank)

    # --- device-resident leg -------------------------------------------------
    d_s = torch.from_numpy(s).to(dev)
    d_theta = torch.from_numpy(theta).to(dev)
    d_params = [torch.from_numpy(np.atleast_1d(np.asarray(p, dtype=np.float64))).to(dev) for p in params]
    d_out = torch.empty(8 * n, dtype=torch.float64, device=dev)
    d_status = torch.zeros(n, dtype=torch.int32, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    # a real (non-default) stream: the library launches on the stream it is handed, and the
    # CUDA events below must be recorded on that same stream to see the kernels
    stream = torch.cuda.Stream(device=dev)

    def step_device():
        with torch.cuda.stream(stream):
            flush.fill_(1)
            R.compute_all_dimensionless_device(kind, d_s, d_theta, d_params, d_out, d_status, stream=stream,
                                               coeff_mask=mask, synchronize=False)

    torch.cuda.synchronize()
    for _ in range(args.warmup):
        step_device()
    barrier()
    launches0 = R.kernel_launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = R.kernel_launch_count() - launches0
    ms_dev = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        # d_out / d_status as the last timed step left them (the legs below write their own buffers)
        dump_outputs(args.dump_outputs, d_out.view(8, n).cpu().numpy(), d_status.cpu().numpy())

    # per-kernel device time and work counters of one more (untimed) step, for the roofline
    res = R.compute_all_dimensionless_batch(kind, s, theta, params, device=local_rank, coeff_mask=mask, extras=True)
    k_ms = res.kernel_ms
    apps_sym = float(res.counters[0].astype(np.float64).sum())
    apps_hey = float(res.counters[1].astype(np.float64).sum())
    nan_rate = float(np.isnan(res.values[[c for c in range(8) if (mask >> c) & 1]]).any(axis=0).mean())
    rerouted = float(((res.status & 8) != 0).mean())

    # --- end-to-end leg: host buffers through the public C ABI --------------
    h_s = torch.from_numpy(s).pin_memory().numpy()
    h_theta = torch.from_numpy(theta).pin_memory().numpy()
    h_params = [torch.from_numpy(np.ascontiguousarray(p)).pin_memory().numpy() if np.ndim(p) else p for p in params]

    def step_host():
        flush.fill_(1)
        return R.compute_all_dimensionless_batch(kind, h_s, h_theta, h_params, device=local_rank, coeff_mask=mask)

    step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step_host()
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    h2d = 8 * n * (2 + sum(1 for p in params if np.ndim(p))) + 8 * sum(1 for p in params if not np.ndim(p))
    d2h = 8 * 8 * n + 4 * n
    del out

    ms_dev, ms_e2e = max_over_ranks([ms_dev, t_e2e * 1e3], world, dev)

    if rank == 0:
        value = whole_job_value(n, world, args.steps, ms_dev)
        e2e_value = whole_job_value(n, world, args.steps, ms_e2e)
        peak = R.fp64_peak_tflops(local_rank)
        # The two product kernels run concurrently on two streams and share the SMs, so the roofline
        # is taken over both: FP64 flops executed by one step's Symphony + Heyvaerts launches (rule
        # applications counted by the kernels x flops per application from the ncu capture) over the
        # CUDA-event time of a step of the TIMED region (recorded on the launching stream; it also
        # holds the normalisation, the classification and the L2 flush, which makes the figure a
        # lower bound); `dominant` names the larger contributor.
        kc = kernel_constants()
        flops_sym = apps_sym * kc["flop_per_application"]["symphony"]
        flops_hey = apps_hey * kc["flop_per_application"]["heyvaerts"]
        dominant = "heyvaerts" if flops_hey >= flops_sym else "symphony"
        step_s = ms_dev / args.steps * 1e-3
        achieved = (flops_sym + flops_hey) / step_s * 1e-12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.config, n), "seed": SEED, "l2": "flushed between steps (256 MB write)",
                       "nan_rate": nan_rate, "rerouted_rate": rerouted,
                       "sharding": f"{world} independent shards, no data-path collective"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "fp64", "kernel": "k_symphony_fast + k_heyvaerts_fast (concurrent; larger share: " + dominant + ")",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak if peak else None,
                         "traffic": (kc["dram_bytes_per_point"]["symphony"] + kc["dram_bytes_per_point"]["heyvaerts"]) * n,
                         "traffic_note": "bytes per launch, scaled per point from the ncu --set full capture in profiles/ "
                                         "(local-memory spills; the algorithmic traffic is ~110 B per point)",
                         "constants": {"source": kc.get("source"), "flop_per_application": kc["flop_per_application"]},
                         "peak_source": "measured in this run: register-resident DFMA kernel "
                                        "(MEASURED_PEAKS.json has no FP64 figure)",
                         "kernel_ms": {"normalize": k_ms[0], "symphony": k_ms[1], "heyvaerts": k_ms[2], "span": k_ms[3],
                                       "note": "one extra untimed step, the library's own CUDA events"},
                         "gk31_applications_per_point": {"symphony": apps_sym / n, "heyvaerts": apps_hey / n},
                         "reference_equivalent_tflops": value * W_REF_FLOP_PER_SET * 1e-12,
                         "reference_equivalent_note": "sets/s x W_ref (2.0e9 flop-equivalents per set, SURVEY 8d): the rate at "
                                                      "which the reference's own work is retired; exceeds `achieved` because the "
                                                      "product path shares nodes and needs fewer rule applications"},
        }
        if not args.no_parity:
            line["parity"] = parity_leg(args.config, local_rank)
        if not args.no_cpu_baseline and world == 1:
            cb, _ = cpu_baseline(args.config, args.cpu_sample, "port")
            line["cpu_baseline"] = cb
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
