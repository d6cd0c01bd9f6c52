"""Batched crank-out tools: the training-set generators of the reference,
``examples/crank-out-pitchypl.rs`` and ``examples/crank-out-pitchykappa.rs``, on the GPU.

    python -m rimphony_b200.crank_out pitchypl   S_MIN S_MAX THETA_MIN THETA_MAX P_MIN P_MAX K_MIN K_MAX OUTFILE
    python -m rimphony_b200.crank_out pitchykappa S_MIN S_MAX THETA_MIN THETA_MAX KAPPA_MIN KAPPA_MAX \\
                                                  WIDTH_MIN WIDTH_MAX K_MIN K_MAX OUTFILE
    python -m rimphony_b200.crank_out pitchybpl   S_MIN S_MAX THETA_MIN THETA_MAX P1_MIN P1_MAX P2_MIN P2_MAX \
                                                  GAMMA_BREAK_MIN GAMMA_BREAK_MAX K_MIN K_MAX OUTFILE
    python -m rimphony_b200.crank_out demo almostuniform1          # examples/demo-powerlaw.rs, to stdout

Same positional arguments (crank-out-pitchypl.rs:17-74, crank-out-pitchykappa.rs:17-92), same
sampling (``Sampler``: s and width log-uniform, the rest uniform), same output file: opened
create + append, the tab-separated header with the ``(log)/(lin)/(meta)/(res)`` tags re-emitted
at every start (crank-out-pitchypl.rs:132-155), one row per point with every number written
as ``{:.16e}`` (:175-194).  The reference loops forever, one point at a time; this tool draws
blocks of ``--block`` points, evaluates each block with one batched call and appends its rows;
``time_ms(meta)`` is the block's wall time divided by the block size.  ``--count`` stops after
that many points (default: run until interrupted, like the reference); ``--gpus`` shards each
block over several GPUs of the box.

``pitchybpl`` has no counterpart in the reference: it is ``pitchypl`` for the pitchy broken power law
(``PitchyBrokenPowerLawDistribution``), with gamma_break drawn log-uniform and p1, p2 uniform, each
from its own range.
"""
import argparse
import sys
import time

import numpy as np

from .sampler import Sampler

PITCHYPL_HEADER = ("s(log)", "theta(lin)", "p(lin)", "k(lin)", "time_ms(meta)", "j_I(res)", "alpha_I(res)", "j_Q(res)",
                   "alpha_Q(res)", "j_V(res)", "alpha_V(res)", "rho_Q(res)", "rho_V(res)")
PITCHYKAPPA_HEADER = ("s(log)", "theta(lin)", "kappa(lin)", "width(log)", "k(lin)", "time_ms(meta)", "j_I(res)",
                      "alpha_I(res)", "j_Q(res)", "alpha_Q(res)", "j_V(res)", "alpha_V(res)", "rho_Q(res)", "rho_V(res)")

PITCHYBPL_HEADER = ("s(log)", "theta(lin)", "p1(lin)", "p2(lin)", "gamma_break(log)", "k(lin)", "time_ms(meta)",
                    "j_I(res)", "alpha_I(res)", "j_Q(res)", "alpha_Q(res)", "j_V(res)", "alpha_V(res)", "rho_Q(res)",
                    "rho_V(res)")

DEMO_HEADER = ("s(lin)", "theta(lin)", "p(lin)", "d(meta)", "psi(meta)", "n_e(meta)", "time_ms(meta)", "j_I(res)",
               "alpha_I(res)", "j_Q(res)", "alpha_Q(res)", "j_V(res)", "alpha_V(res)", "rho_Q(res)", "rho_V(res)")

GAMMA_MIN, GAMMA_MAX, GAMMA_CUTOFF = 1.0, 1e12, 1e10  # crank-out-pitchypl.rs:163-165


def demo_almostuniform1():
    """The 64-step sweep of examples/demo-powerlaw.rs:80-98 (neurosynchro's end-to-end fixture)."""
    x = np.arange(64) / 63.0
    return {"s": 100.0 - 10.0 * x, "theta": 0.5 + 0.1 * x, "p": 3.0 - 0.5 * x, "d": x * 3e10, "psi": 0.1 * x,
            "n_e": 1e5 - 3e4 * x}


def evaluate_demo(cols, n_devices=1):
    import rimphony_b200 as R

    res = R.compute_all_dimensionless_batch(R.POWER_LAW, cols["s"], cols["theta"],
                                            [cols["p"], GAMMA_MIN, GAMMA_MAX, GAMMA_CUTOFF])
    return res.values


def run_demo(name, out, evaluate_fn=evaluate_demo):
    if name != "almostuniform1":
        raise SystemExit(f"unknown demo {name!r} (the reference has: almostuniform1)")
    cols = demo_almostuniform1()
    n = len(cols["s"])
    t0 = time.perf_counter()
    vals = evaluate_fn(cols)
    ms = (time.perf_counter() - t0) * 1e3 / n
    out.write("\t".join(DEMO_HEADER) + "\n")
    out.write(format_rows([cols["s"], cols["theta"], cols["p"], cols["d"], cols["psi"], cols["n_e"], np.full(n, ms)] +
                          [vals[c] for c in range(8)]))
    return 0


def rust_sci(x):
    """Rust's ``{:.16e}``: 16 fractional digits, exponent without sign padding or leading zeros."""
    if x != x:
        return "NaN"
    if x in (float("inf"), float("-inf")):
        return "inf" if x > 0 else "-inf"
    mant, exp = f"{x:.16e}".split("e")
    return f"{mant}e{int(exp)}"


def format_rows(columns):
    """``columns``: equal-length 1-D arrays; returns the TSV text of their rows."""
    return "".join("\t".join(rust_sci(float(v)) for v in row) + "\n" for row in zip(*columns))


def parse(argv):
    ap = argparse.ArgumentParser(prog="python -m rimphony_b200.crank_out", description=__doc__,
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--block", type=int, default=65536, help="points per batched call")
    ap.add_argument("--count", type=int, default=0, help="stop after this many points (0 = never)")
    ap.add_argument("--gpus", type=int, default=1, help="GPUs of this box to shard each block over")
    ap.add_argument("--seed", type=int, default=None, help="seed of the parameter sampler (default: entropy)")
    sub = ap.add_subparsers(dest="tool", required=True)
    pl = sub.add_parser("pitchypl")
    for name in ("S_MIN", "S_MAX", "THETA_MIN", "THETA_MAX", "P_MIN", "P_MAX", "K_MIN", "K_MAX"):
        pl.add_argument(name, type=float)
    pl.add_argument("OUTFILE")
    pk = sub.add_parser("pitchykappa")
    for name in ("S_MIN", "S_MAX", "THETA_MIN", "THETA_MAX", "KAPPA_MIN", "KAPPA_MAX", "WIDTH_MIN", "WIDTH_MAX",
                 "K_MIN", "K_MAX"):
        pk.add_argument(name, type=float)
    pk.add_argument("OUTFILE")
    pb = sub.add_parser("pitchybpl")
    for name in ("S_MIN", "S_MAX", "THETA_MIN", "THETA_MAX", "P1_MIN", "P1_MAX", "P2_MIN", "P2_MAX", "GAMMA_BREAK_MIN",
                 "GAMMA_BREAK_MAX", "K_MIN", "K_MAX"):
        pb.add_argument(name, type=float)
    pb.add_argument("OUTFILE")
    dm = sub.add_parser("demo")
    dm.add_argument("DEMONAME", choices=["almostuniform1"])
    return ap.parse_args(argv)


def samplers(args, rng):
    """(header, kind name, [(column name, Sampler)]) in the order of the output columns."""
    if args.tool == "pitchypl":
        return PITCHYPL_HEADER, [("s", Sampler(True, args.S_MIN, args.S_MAX, rng)),
                                 ("theta", Sampler(False, args.THETA_MIN, args.THETA_MAX, rng)),
                                 ("p", Sampler(False, args.P_MIN, args.P_MAX, rng)),
                                 ("k", Sampler(False, args.K_MIN, args.K_MAX, rng))]
    if args.tool == "pitchybpl":
        return PITCHYBPL_HEADER, [("s", Sampler(True, args.S_MIN, args.S_MAX, rng)),
                                  ("theta", Sampler(False, args.THETA_MIN, args.THETA_MAX, rng)),
                                  ("p1", Sampler(False, args.P1_MIN, args.P1_MAX, rng)),
                                  ("p2", Sampler(False, args.P2_MIN, args.P2_MAX, rng)),
                                  ("gamma_break", Sampler(True, args.GAMMA_BREAK_MIN, args.GAMMA_BREAK_MAX, rng)),
                                  ("k", Sampler(False, args.K_MIN, args.K_MAX, rng))]
    return PITCHYKAPPA_HEADER, [("s", Sampler(True, args.S_MIN, args.S_MAX, rng)),
                                ("theta", Sampler(False, args.THETA_MIN, args.THETA_MAX, rng)),
                                ("kappa", Sampler(False, args.KAPPA_MIN, args.KAPPA_MAX, rng)),
                                ("width", Sampler(True, args.WIDTH_MIN, args.WIDTH_MAX, rng)),
                                ("k", Sampler(False, args.K_MIN, args.K_MAX, rng))]


def evaluate(tool, cols, n_devices):
    """All eight coefficients of one block: ``[8, n]``."""
    import rimphony_b200 as R

    if tool == "pitchypl":
        kind, params = R.PITCHY_PL, [cols["p"], cols["k"], GAMMA_MIN, GAMMA_MAX, GAMMA_CUTOFF]
    elif tool == "pitchybpl":
        kind, params = R.PITCHY_BROKEN_PL, [cols["p1"], cols["p2"], cols["gamma_break"], cols["k"], GAMMA_MIN, GAMMA_MAX,
                                            GAMMA_CUTOFF]
    else:
        kind, params = R.PITCHY_KAPPA, [cols["kappa"], cols["width"], cols["k"], GAMMA_CUTOFF]
    res = R.compute_all_dimensionless_batch(kind, cols["s"], cols["theta"], params,
                                            n_devices=(n_devices if n_devices > 1 else None))
    return res.values


def main(argv=None, evaluate_fn=evaluate):
    args = parse(sys.argv[1:] if argv is None else argv)
    if args.tool == "demo":
        return run_demo(args.DEMONAME, sys.stdout)
    rng = np.random.default_rng(args.seed)
    header, samp = samplers(args, rng)
    done = 0
    with open(args.OUTFILE, "a") as out:  # create + append, header at every start
        out.write("\t".join(header) + "\n")
        while args.count <= 0 or done < args.count:
            n = args.block if args.count <= 0 else min(args.block, args.count - done)
            cols = {name: np.atleast_1d(s.get(n)) for name, s in samp}
            t0 = time.perf_counter()
            vals = evaluate_fn(args.tool, cols, args.gpus)
            ms = (time.perf_counter() - t0) * 1e3 / n
            out.write(format_rows([cols[name] for name, _ in samp] + [np.full(n, ms)] + [vals[c] for c in range(8)]))
            out.flush()
            done += n
    return 0


if __name__ == "__main__":
    sys.exit(main())
