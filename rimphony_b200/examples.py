"""The reference's one-shot example programs on the GPU path.

    python -m rimphony_b200.examples all-pitchykappa-cgs NU B N_E THETA KAPPA WIDTH K
    python -m rimphony_b200.examples stokes-slab-pitchykappa-cgs NU B N_E THETA PSI DEPTH KAPPA WIDTH K
    python -m rimphony_b200.examples one-powerlaw-direct
    python -m rimphony_b200.examples one-powerlaw-normalized
    python -m rimphony_b200.examples one-pitchypl-normalized

Same positional arguments, constants and output lines as ``examples/all-pitchykappa-cgs.rs:13-133``,
``one-powerlaw-direct.rs:10-30``, ``one-powerlaw-normalized.rs:13-47`` and
``one-pitchypl-normalized.rs:11-29``.  ``stokes-slab-pitchykappa-cgs`` has no counterpart in the
reference: it prints the emergent Stokes I, Q, U, V of a uniform slab of depth DEPTH (cm) with the
coefficients ``all-pitchykappa-cgs`` prints and field angle PSI.  (The crank-out tools and ``demo-powerlaw`` are in
``rimphony_b200.crank_out``.)  ``--mode faithful`` runs the reference's own sequence of rule
applications instead of the product path.
"""
import argparse
import math
import sys

GAMMA_MIN, GAMMA_MAX, GAMMA_CUTOFF = 1.0, 1e12, 1e10


def rust_e(x, digits=None):
    """Rust's ``{:e}`` (shortest round-trip mantissa) or ``{:.Ne}``."""
    if x != x:
        return "NaN"
    if math.isinf(x):
        return "inf" if x > 0 else "-inf"
    if digits is None:
        mant, exp = repr(float(x)), 0
        if "e" in mant or "E" in mant:
            mant, e = mant.lower().split("e")
            exp = int(e)
        # normalise to d.ddd form
        sign = "-" if mant.startswith("-") else ""
        mant = mant.lstrip("-")
        whole, _, frac = mant.partition(".")
        digits_all = (whole + frac).lstrip("0")
        if not digits_all:
            return sign + "0e0"
        first_sig = len(whole + frac) - len((whole + frac).lstrip("0"))
        exp += len(whole) - 1 - first_sig
        digits_all = digits_all.rstrip("0") or "0"
        body = digits_all[0] + ("." + digits_all[1:] if len(digits_all) > 1 else "")
        return f"{sign}{body}e{exp}"
    mant, exp = f"{x:.{digits}e}".split("e")
    return f"{mant}e{int(exp)}"


def all_pitchykappa_cgs(args, R, out):
    """examples/all-pitchykappa-cgs.rs:96-133: eight cgs coefficients, gamma cutoff 100."""
    calc = (R.PitchyKappaDistribution(args.KAPPA, args.WIDTH, args.K).gamma_cutoff(100.0)
            .full_calculation(mode=args.mode))
    vals = calc.compute_all_cgs(args.NU, args.B, args.N_E, args.THETA)
    for label, v in zip(("    j_I", "alpha_I", "    j_Q", "alpha_Q", "    j_V", "alpha_V", "  rho_Q", "  rho_V"), vals):
        out.write(f"{label}: {rust_e(float(v), 18)}\n")
    return 0


def stokes_slab_pitchykappa_cgs(args, R, out):
    """Emergent (I, Q, U, V) of a uniform slab of the all-pitchykappa-cgs distribution (gamma cutoff 100)."""
    calc = (R.PitchyKappaDistribution(args.KAPPA, args.WIDTH, args.K).gamma_cutoff(100.0)
            .full_calculation(mode=args.mode))
    res = calc.compute_stokes_cgs(args.NU, args.B, args.N_E, args.THETA, args.PSI, args.DEPTH)
    for label, v in zip(("I", "Q", "U", "V"), res.stokes[:, 0]):
        out.write(f"{label}: {rust_e(float(v), 18)}\n")
    return 0


def one_powerlaw_direct(args, R, out):
    """examples/one-powerlaw-direct.rs:10-30."""
    symphony_ji = 2.64399749412774e-21
    ji = (R.PowerLawDistribution(2.5).gamma_limits(GAMMA_MIN, GAMMA_MAX, GAMMA_CUTOFF).full_calculation(mode=args.mode)
          .compute_cgs(R.Coefficient.Emission, R.Stokes.I, 1e9, 1e3, 1.0, 0.9))
    out.write(f"Symphony j_I: {rust_e(symphony_ji)}   Ours: {rust_e(ji)}\n")
    return 0


def one_powerlaw_normalized(args, R, out):
    """examples/one-powerlaw-normalized.rs:13-47 (alpha_I at one (s, theta, p), with and without units)."""
    s, theta, p = 1.0360583634e3, 7.4017422303e-1, 2.3306843452e0
    symphony_val = 0.0
    nu = 1e9
    b = R.TWO_PI * R.MASS_ELECTRON * R.SPEED_LIGHT * nu / (R.ELECTRON_CHARGE * s)
    val = (R.PowerLawDistribution(p).gamma_limits(GAMMA_MIN, GAMMA_MAX, GAMMA_CUTOFF).full_calculation(mode=args.mode)
           .compute_cgs(R.Coefficient.Absorption, R.Stokes.I, nu, b, 1.0, theta))
    remove_units = (-2.0 * R.MASS_ELECTRON * R.SPEED_LIGHT * nu * abs(math.cos(theta)) /
                    (R.TWO_PI * R.ELECTRON_CHARGE) ** 2)
    out.write(f"Inner Symphony: {rust_e(symphony_val * remove_units)}   Us: {rust_e(val * remove_units)}\n")
    out.write(f"Outer Symphony: {rust_e(symphony_val)}   Us: {rust_e(val)}\n")
    return 0


def one_pitchypl_normalized(args, R, out):
    """examples/one-pitchypl-normalized.rs:11-29 (rho_Q at one point of the pitchy power law)."""
    s, theta, p, k = 8.0973407678629616e0, 7.2687065355210786e-2, 2.7273434060193211e0, 2.7016346500930695e0
    val = (R.PitchyPowerLawDistribution(p, k).gamma_limits(GAMMA_MIN, GAMMA_MAX, GAMMA_CUTOFF)
           .full_calculation(mode=args.mode).compute_dimensionless(R.Coefficient.Faraday, R.Stokes.Q, s, theta))
    out.write(f"{rust_e(val, 18)}\n")
    return 0


TOOLS = {"all-pitchykappa-cgs": all_pitchykappa_cgs, "stokes-slab-pitchykappa-cgs": stokes_slab_pitchykappa_cgs,
         "one-powerlaw-direct": one_powerlaw_direct,
         "one-powerlaw-normalized": one_powerlaw_normalized, "one-pitchypl-normalized": one_pitchypl_normalized}


def parse(argv):
    ap = argparse.ArgumentParser(prog="python -m rimphony_b200.examples", description=__doc__,
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--mode", choices=["fast", "faithful"], default="fast")
    sub = ap.add_subparsers(dest="tool", required=True)
    cgs = sub.add_parser("all-pitchykappa-cgs")
    for name in ("NU", "B", "N_E", "THETA", "KAPPA", "WIDTH", "K"):
        cgs.add_argument(name, type=float)
    slab = sub.add_parser("stokes-slab-pitchykappa-cgs")
    for name in ("NU", "B", "N_E", "THETA", "PSI", "DEPTH", "KAPPA", "WIDTH", "K"):
        slab.add_argument(name, type=float)
    for name in ("one-powerlaw-direct", "one-powerlaw-normalized", "one-pitchypl-normalized"):
        sub.add_parser(name)
    return ap.parse_args(argv)


def main(argv=None, module=None, out=None):
    args = parse(sys.argv[1:] if argv is None else argv)
    if module is None:
        import rimphony_b200 as module
    args.mode = module.MODE_FAITHFUL if args.mode == "faithful" else module.MODE_FAST
    return TOOLS[args.tool](args, module, sys.stdout if out is None else out)


if __name__ == "__main__":
    sys.exit(main())
