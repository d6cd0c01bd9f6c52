// rb_symfast.cuh -- j_I/Q/V and alpha_I/Q/V of one point on the product
// ("fast") path: the Symphony harmonic sum + (n, gamma) double integral of
//   src/symphony.rs:66-187 (compute), :196-295 (n_integration),
//   :312-389 (gamma_integral), :398-479 (gamma_integrand)
// evaluated with the compact engine of rb_engine.cuh.
//
// Same integrand, same integration domain, same truncation rule as the
// reference; what differs is how the quadrature is organised:
//
//   * all six integrands share every gamma node (one J_n, J_{n+1}, f, df pair
//     per node) and the two Stokes-V lobes fall out of the left/right halves;
//   * the gamma integral is seeded where the integrand lives.  For large n the
//     integrand is a peak of relative half-width ~ n^(-1/3) around gamma_peak:
//     with gamma = gamma_peak + t (gamma_+ - gamma_peak), z/n = 1 - t^2/2 - ... and
//     J_n(z)^2 ~ rb_exp(-(2n/3) |t|^3).  The seeds cover [-T, T], T = kPeakSpan n^(-1/3), cut
//     where the reference's J_n switches expansion (Debye / blend / Meissel), plus the two outer
//     remainders while T is not yet small, instead of the reference's bisection cascade from the
//     full [gamma_-, gamma_+] (15-45 rule applications per gamma integral at n >= 1e3, measured);
//     they are evaluated two per application as 15-point Kronrod rules (rb_engine.cuh);
//   * the integral over continuous n keeps the reference's chunks [n_start, n_start + delta_n],
//     growth rules and stop rule |chunk| < |sum| / 1e5 (symphony.rs:196-295) -- where the loop
//     ends is part of the result -- but integrates each chunk in u = ln n (n G(n) is a smooth
//     bump in u) with the sequential 15- and 7-point rules, and probes dG/dn by a central
//     difference.
#pragma once

#include "rb_bessel.cuh"
#include "rb_dist.cuh"
#include "rb_engine.cuh"

namespace rb {

constexpr double kPeakSpan = 2.6;    // seed half-width in units of n^(-1/3): exp(-(2/3) 2.6^3) = 8e-6, tail beyond < 1e-6
constexpr double kGrade = 0.875;     // low n: the central panels are cut again at this fraction of the first cut
constexpr double kUncutSplit = 0.5;  // a side without cuts is seeded as two panels, split at this fraction of the span
constexpr double kLightChunk = 1e-3; // a chunk after one that added less than this fraction gets the 7-point rule
constexpr double kLightGammaTolerance = 100.0; // gamma integrals of a light chunk: this times epsrel_gamma (10 %:
                                              // the one 15-point panel per side is refined only if it is garbage)
constexpr double kInnerFloor = 1.0; // acceptance floor of a gamma panel, fraction of the integral so far
constexpr double kPanelWidth = 2.302585092994046; // outer panel width in u = ln n (one decade)
constexpr int kMaxChunks = 400;   // safety net of the chunk loop (the reference has none)

// Reference-fidelity guard.  Above n ~ 1e10 the J_n^2 peak (half-width n^(-1/3) of the gamma
// range) falls between the nodes of the reference's GK31 bisection from the full [gamma_-,
// gamma_+] and its gamma integral collapses to ~0 (for s < 1e6; above that the reference
// shrinks the window, symphony.rs:337-341).  A point whose chunks starting beyond
// kSensitiveN still contribute more than kSensitiveFraction of a coefficient therefore has
// a reference value that is set by that quadrature failure, not by the integral.  Such
// points (hard kappa spectra) are not computed here: they are flagged and re-run with the
// reference's exact sequence of rule applications (MODE_FAITHFUL kernel).
constexpr double kSensitiveN = 5e9;
constexpr double kSensitiveFraction = 5e-4; // per chunk; the chunks above decay at least like 1/2 per decade: < 1e-3 in all
// A flagged point does not start over: up to n ~ 1e9 the reference's quadrature is sound and
// the product path reproduces it, so the faithful sequence resumes from the chunk-loop state
// recorded at the first chunk starting beyond kHandoverN (s >= 10, where the chunk sequence
// 1e5 x 10^k is the same for every coefficient; below that the point is re-run from scratch).
constexpr double kHandoverN = 1e9;
constexpr double kNegligibleExponent = 200.0; // see sym_gamma_integral
constexpr double kTailSkipSpan = 0.25; // outer remainders of the gamma range are dropped below this span
constexpr bool kCutAtBlendEnd = true;  // also cut the central panels where the blend meets Meissel

constexpr double kNarrowPanel = 0.75; // outer panels narrower than this in u use the 7-point rule

// Layout of a hand-over record (doubles): the state of the chunk loop at the first chunk that
// starts beyond kHandoverN, for the faithful continuation (rb_symphony.cuh symphony_tail_faithful).
constexpr int kSnapNStart = 0, kSnapDeltaN = 1, kSnapIncr = 2, kSnapValid = 3, kSnapDisc = 4, kSnapTail = 12,
              kSnapContrib = 20, kSnapActive = 28, kSnapDone = 29, kSnapDoubles = 32;
// (kSnapDone: where the warps that finish the accumulators of a handed point count themselves out, k_symphony)

constexpr int kSymInnerChan = 6;
struct SymFastWS {
    EngLevelT<kSymInnerChan> inner; // the six integrands of a node (the V lobes are halves of the same panels)
    OuterLevel outer; // the n level: running sums instead of a tile (rb_engine.cuh)
    LeungOrder on, on1;
    double snap[kSnapDoubles];
    // the warp-uniform context of the point in work (SymFastCtx + the distribution): in shared memory, not
    // on the stack of the kernel, because the out-of-line quadrature functions read it through a reference
    // and the L1 left beside 214 KB of shared memory does not hold 640 stacks (DESIGN.md section 12)
    Dist dist;
    double ctx_store[10];
};

// Warp-uniform context of one point.
template <int KIND>
struct SymFastCtx {
    const Dist *d;
    SymFastWS *ws;
    double s, cos_th, sin_th;
    double inv_s, inv_sin_th;
    double epsrel_gamma;
};

// J_n(x) for the argument range of the Symphony integrand (0 <= x <= n): the
// Debye and Meissel expansions appear once each (pkgw_bessel_j, bessel.c:318-357).
RB_FN_NOINLINE double leung_j_general(const LeungOrder &o, double x) { return leung_j(o, x); }

// J_n(x) and J_{n+1}(x), n >= 30, 0 <= x <= n (pkgw_bessel_j, bessel.c:341-357, for both orders), with the
// Debye expansion evaluated once for both (leung_debye_eps_pair).
RB_FN void leung_j_pair_below(const LeungOrder &o0, const LeungOrder &o1, double x, double (&jv)[2])
{
    const double eps0 = (o0.n - x) * o0.ninv, eps1 = (o1.n - x) * o1.ninv;
    const bool deb0 = !(eps0 > o0.hi_minus), deb1 = !(eps1 > o1.hi_minus);
    const bool mei0 = !(eps0 < o0.lo_minus) && x != o0.n, mei1 = !(eps1 < o1.lo_minus);
    double dv[2] = {0.0, 0.0};
    if (deb0 || deb1)
        leung_debye_eps_pair(o0.n, o1.n, x, dv[0], dv[1]);
#pragma unroll 1
    for (int k = 0; k < 2; k++) {
        const LeungOrder &o = k ? o1 : o0;
        const double eps = k ? eps1 : eps0;
        const bool use_debye = k ? deb1 : deb0, use_meissel = k ? mei1 : mei0;
        double v = dv[k];
        if (use_meissel) {
            const double mv = leung_meissel_first(o, x);
            v = mv;
            if (use_debye) {
                const double eta = rb_log(eps) * kLog10e;
                const double pos = (eta - o.eta_lo_minus) * (1.0 / (kMinusEtaB - kMinusEtaA));
                v = dv[k] * (1.0 - pos) + mv * pos;
            }
        }
        jv[k] = v;
    }
}

// Kinematics of one (n, gamma) node: beta, cos/sin of the pitch angle xi fixed by the
// resonance condition, and the Bessel argument z with gamma sin(xi) stabilised against
// cancellation at large gamma, n (symphony.rs:406-439).
template <int KIND>
RB_FN double sym_bessel_arg(const SymFastCtx<KIND> &cx, double n, double gamma, double &beta, double &cos_xi,
                            double &sin_xi)
{
    const double s = cx.s, costh = cx.cos_th, sinth = cx.sin_th;
    const double inv_g = rb_rcp(gamma);
    beta = rb_sqrt(1.0 - inv_g * inv_g);
    cos_xi = rb_div(s * gamma - n, s * gamma * beta * costh);
    sin_xi = rb_sqrt(1.0 - cos_xi * cos_xi);
    double gamma_sin_xi;
    if (beta < 0.1) {
        gamma_sin_xi = gamma * sin_xi;
    } else {
        const double bc = beta * costh;
        const double beta2_costh2 = bc * bc;
        const double s_on_r = 2.0 * rb_div(n, s * (beta2_costh2 - 1.0));
        const double inv_b2c2 = rb_rcp(beta2_costh2);
        const double nos = n * cx.inv_s;
        gamma_sin_xi = rb_sqrt((1.0 - inv_b2c2) * (gamma * (gamma + s_on_r)) - nos * nos * inv_b2c2);
    }
    return s * beta * sinth * gamma_sin_xi;
}

// eps = (n - z)/n at gamma, for the seed placement: one out-of-line copy (it is called from
// five places of the warp-uniform seeding code).
template <int KIND>
RB_FN_NOINLINE double sym_eps_at(const SymFastCtx<KIND> &cx, double n, double gamma)
{
    double b_, c_, s_;
    return rb_div(n - sym_bessel_arg<KIND>(cx, n, gamma, b_, c_, s_), n);
}

// The six gamma integrands at one node (symphony.rs:398-479); one call site.
template <int KIND>
RB_FN void sym_node(const SymFastCtx<KIND> &cx, double n, double gamma, double (&out)[6])
{
    const double costh = cx.cos_th;
    double beta, cos_xi, sin_xi;
    const double z = sym_bessel_arg<KIND>(cx, n, gamma, beta, cos_xi, sin_xi);
    const double m = (costh - beta * cos_xi) * cx.inv_sin_th;
    const double big_n = beta * sin_xi;

    // J_n(z), J_{n+1}(z): one copy of the evaluator, two trips
    double jv[2];
    if (cx.ws->on1.kind == kOrderInteger && cx.ws->on.kind == kOrderInteger && z > 0.0 && z < n + 1.0) {
        bessel_jn_pair_small_int(cx.ws->on.nint, z, jv[0], jv[1]); // a discrete harmonic below order 29
    } else if (cx.ws->on.kind == kOrderLeung && cx.ws->on1.kind == kOrderLeung && z <= n) {
        leung_j_pair_below(cx.ws->on, cx.ws->on1, z, jv);
    } else { // order 29 with 30, the first harmonics of s sin(theta) < 1: out of line
#pragma unroll 1
        for (int k = 0; k < 2; k++)
            jv[k] = leung_j_general(k ? cx.ws->on1 : cx.ws->on, z);
    }
    const double jn = jv[0];
    double djn;
    if (n >= 1e15)
        djn = NAN; // bessel.c:382-388
    else if (z == 0.0)
        djn = (n >= 2.0) ? 0.0 : ((n == 0.0) ? -jv[1] : n * jn / DBL_MIN - jv[1]);
    else
        djn = rb_div(n * jn, z) - jv[1];

    const double mj = m * jn;
    const double njp = big_n * djn;

    double f, dfdg, dfdcx;
    dist_eval<KIND>(*cx.d, gamma, cos_xi, f, dfdg, dfdcx, NAN, gamma * beta); // sqrt(gamma^2 - 1) = gamma beta
    const double dfdcx_factor = rb_div(beta * costh - cos_xi, gamma - rb_rcp(gamma));
    const double f_abs = dfdg + dfdcx_factor * dfdcx;

    const double g2 = gamma * gamma;
    const double pol_i = g2 * (mj * mj + njp * njp);
    const double pol_q = g2 * (mj * mj - njp * njp);
    const double pol_v = g2 * (2.0 * mj * njp);
    out[0] = pol_i * f;
    out[1] = pol_i * f_abs;
    out[2] = pol_q * f;
    out[3] = pol_q * f_abs;
    out[4] = pol_v * f;
    out[5] = pol_v * f_abs;
}

// G(n): the gamma integral at harmonic number n for all eight accumulators,
//   0 j_I, 1 a_I, 2 j_Q, 3 a_Q, 4 j_V(+), 5 a_V(+), 6 j_V(-), 7 a_V(-)
// ((+) = gamma > gamma_peak, symphony.rs:356-363), multiplied by wa / wb and
// parked in column `col` of the outer tile (A rows / B rows).
template <int KIND>
RB_FN_NOINLINE void sym_gamma_integral(Warp &w, const SymFastCtx<KIND> &cx, double n, int col, double wa, double wb,
                                       bool light = false)
{
    SymFastWS &ws = *cx.ws;
    const double s = cx.s, costh = cx.cos_th, sinth = cx.sin_th;
    const double nos = n * cx.inv_s;
    const double root = sqrt(nos * nos - sinth * sinth);
    const double inv_sin2 = cx.inv_sin_th * cx.inv_sin_th;
    const double gamma_minus = (nos - fabs(costh) * root) * inv_sin2;
    const double gamma_plus = (nos + fabs(costh) * root) * inv_sin2;
    const double gamma_peak = 0.5 * (gamma_plus + gamma_minus);
    const double rel_width = (s < 1e6) ? 1.0 : rb_exp(-0.27 * rb_log(n) - 0.1);
    // gamma = gamma_peak + t half, t in [-1, 1]
    const double half = (gamma_plus - gamma_peak) * rel_width;

    // Far below the critical harmonic J_n(z)^2 ~ rb_exp(-2n(alpha - tanh alpha)), sech(alpha) = z/n,
    // is beyond any power-law factor (the first harmonics of a large-s point: exponent ~ s sin(theta)).
    // With the exponent at the peak of the gamma range above kNegligibleExponent the whole gamma
    // integral is < e^-200 of the harmonics that make up the coefficient: it is not evaluated.
    const double eps_peak = (n >= kNJn) ? sym_eps_at<KIND>(cx, n, gamma_peak) : 0.0;
    if (n >= kNJn) {
        const double x0 = 1.0 - eps_peak;
        if (x0 > 0.0 && x0 < 1.0) {
            const double th = sqrt((1.0 - x0) * (1.0 + x0));
            const double exponent = 2.0 * n * (rb_log(rb_div(1.0 + th, x0)) - th);
            if (exponent > kNegligibleExponent) {
                return; // adds nothing to the sums of the outer rule
            }
        }
    }

    warp_fence();
#ifdef RB_DEVICE_BUILD
    if (w.lane < 2) // orders n and n + 1 side by side
        leung_prepare(n + (double)w.lane, w.lane ? ws.on1 : ws.on);
#else
    leung_prepare(n, ws.on);
    leung_prepare(n + 1.0, ws.on1);
#endif

    // Seeds.  Central panels [0, +-T] first (they are popped last-in first-out), outer
    // remainders after them.  The reference's J_n switches from the Debye expansion to a
    // blend to Meissel's expansion where eps = (n - z)/n crosses lo_minus and hi_minus
    // (bessel.c:341-357); the integrand has slope breaks there, so the central panels are
    // cut at those two values of t (found by a secant solve on the exact eps(t)): every
    // seed is then smooth and is usually accepted at its first application.
    PanelStack stk;
    stk.reset(&ws.inner);
    const double w_peak = rb_exp(-(1.0 / 3.0) * rb_log(n));
    const double inv_rel_width = rb_rcp(rel_width);
    double span = kPeakSpan * w_peak * inv_rel_width;
    const bool full = !(span < 0.5);
    if (full)
        span = 1.0;
    // Beyond |t| = T the Bessel factor is below exp(-(2/3) kPeakSpan^3) of its peak while f grows
    // at most like (1 - |t|)^-(p+2); the remainders [+-T, +-1] are integrated only while T is not
    // yet small (n <~ 1000), as a guard for the mildly relativistic regime.
    const bool keep_remainders = !full && !(span < kTailSkipSpan);
    double cut[2][2]; // [side][which]: 0 < |cut0| <= |cut1| <= span, or == span when absent
    // A chunk far up the tail (`light`: the previous one added less than kLightChunk of the sum) needs
    // its gamma integrals to a few per cent: one 15-point panel per side of the peak, no cuts at the
    // expansion boundaries, a hundred times the tolerance.  A few per cent of < 1e-3 of the coefficient is
    // inside its tolerance and the stop rule |chunk| < |sum| / 1e5 does not notice it.
    if (light) {
        cut[0][0] = cut[0][1] = cut[1][0] = cut[1][1] = span;
    } else {
        const bool leung = n >= kNJn;
        warp_fence(); // orders prepared by lane 0
        const double lo = ws.on.lo_minus, hi = ws.on.hi_minus;
        const double eps0 = eps_peak;

        // The four cuts at once: lane group g = 2 side + which samples eps(t) at eight points around
        // the quadratic guess t0 = sqrt(2 (target - eps0)) (one evaluation per lane instead of
        // ~20 warp-uniform ones), a ballot finds the bracketing pair and a linear interpolation
        // between them places the cut to ~1e-3 of its panel.  A cut that is not bracketed falls
        // back to the secant iteration below.
        double found[2][2];
        {
#ifdef RB_DEVICE_BUILD
            const int grp = w.lane >> 3, j = w.lane & 7;
            const double tgt = (grp & 1) ? hi : lo;
            const double sg = (grp & 2) ? 1.0 : -1.0;
            const double t0g = sqrt(2.0 * (tgt - eps0)) * inv_rel_width; // NaN when there is no crossing
            const double tj = t0g * (0.7 + (0.6 / 7.0) * j);
            const bool valid = leung && (eps0 < tgt) && (1.3 * t0g < span);
            double fj = 0.0;
            if (valid)
                fj = sym_eps_at<KIND>(cx, n, gamma_peak + half * sg * tj) - tgt;
            const unsigned below = __ballot_sync(0xffffffffu, valid && fj < 0.0);
            const unsigned bits = (below >> (8 * grp)) & 0xffu;
            const int cnt = __popc(bits);
            const bool ok = valid && cnt >= 1 && cnt <= 7 && bits == ((1u << cnt) - 1u);
            const int src = 8 * grp + (ok ? cnt - 1 : 0);
            const double fa = __shfl_sync(0xffffffffu, fj, src), ta = __shfl_sync(0xffffffffu, tj, src);
            const double fb = __shfl_sync(0xffffffffu, fj, src + 1), tb = __shfl_sync(0xffffffffu, tj, src + 1);
            const double tcross = ok ? ta - fa * rb_div(tb - ta, fb - fa) : NAN;
#pragma unroll
            for (int g = 0; g < 4; g++)
                found[g >> 1][g & 1] = __shfl_sync(0xffffffffu, tcross, 8 * g);
#else
            for (int g = 0; g < 4; g++) {
                const double tgt = (g & 1) ? hi : lo;
                const double sg = (g & 2) ? 1.0 : -1.0;
                const double t0g = sqrt(2.0 * (tgt - eps0)) * inv_rel_width;
                const bool valid = leung && (eps0 < tgt) && (1.3 * t0g < span);
                double tcross = NAN;
                if (valid) {
                    double fj[8], tj[8];
                    int cnt = 0;
                    bool mono = true;
                    for (int j = 0; j < 8; j++) {
                        tj[j] = t0g * (0.7 + (0.6 / 7.0) * j);
                        fj[j] = sym_eps_at<KIND>(cx, n, gamma_peak + half * sg * tj[j]) - tgt;
                        if (fj[j] < 0.0) {
                            if (cnt != j)
                                mono = false;
                            cnt++;
                        }
                    }
                    if (mono && cnt >= 1 && cnt <= 7)
                        tcross = tj[cnt - 1] - fj[cnt - 1] * (tj[cnt] - tj[cnt - 1]) / (fj[cnt] - fj[cnt - 1]);
                }
                found[g >> 1][g & 1] = tcross;
            }
#endif
        }
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            const double sgn = side ? 1.0 : -1.0;
#pragma unroll 1
            for (int k = 0; k < 2; k++) {
                const double target = k ? hi : lo;
                double tcut = span;
                if (found[side][k] > 0.0 && found[side][k] < span && (k == 0 || kCutAtBlendEnd)) {
                    tcut = found[side][k];
                } else
                if (leung && eps0 < target && (k == 0 || kCutAtBlendEnd)) {
                    // eps(t) ~ eps0 + (t rel_width)^2 / 2; refine on the exact function
                    double t0 = sqrt(2.0 * (target - eps0)) / rel_width;
                    if (t0 < span) {
                        double t1 = 1.05 * t0;
                        double f0 = sym_eps_at<KIND>(cx, n, gamma_peak + half * sgn * t0) - target;
#pragma unroll 1
                        for (int it = 0; it < 4; it++) {
                            if (!(t1 < 1.0))
                                t1 = 0.5 * (t0 + 1.0);
                            const double f1 = sym_eps_at<KIND>(cx, n, gamma_peak + half * sgn * t1) - target;
                            const double den = f1 - f0;
                            if (den == 0.0 || !(den == den))
                                break;
                            const double t2 = t1 - f1 * (t1 - t0) / den;
                            t0 = t1;
                            f0 = f1;
                            t1 = t2;
                            if (!(t1 > 0.0)) {
                                t1 = t0;
                                break;
                            }
                            if (fabs(t1 - t0) <= 1e-5 * t1) // a panel boundary needs no more than this
                                break;
                        }
                        if (t1 > 0.0 && t1 < span)
                            tcut = t1;
                    }
                }
                cut[side][k] = tcut;
            }
            if (cut[side][0] > cut[side][1])
                cut[side][0] = cut[side][1];
        }
    }

    // est: integral of |f| over the accepted panels; big: the largest |panel value| seen so far,
    // accepted or not (the central seeds are evaluated first, so it knows the scale at once)
    PerChan<double> sum_l, sum_r, est, big;
    RB_FOR_CHAN(c, kEngChan)
    {
        sum_l[c] = 0.0;
        sum_r[c] = 0.0;
        est[c] = 0.0;
        big[c] = 0.0;
    }

    // Seeds, pushed so that they are popped in like pairs: the two central panels first (they fix
    // the scale `big`), then the two blend panels, the two tails, the two remainders.  Both panels
    // of such a pair run the same Bessel branch (Debye / both / Meissel, bessel.c:346-357), so a
    // paired application costs what one of them would alone.
    if (keep_remainders) {
        stk.push(w, -1.0, -span, 0);
        stk.push(w, span, 1.0, 1);
    }
    const bool graded = (full || keep_remainders) && !light;
    if (graded) {
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            const double c0 = cut[side][0];
            if (c0 < span)
                stk.push(w, side ? kGrade * c0 : -c0, side ? c0 : -kGrade * c0, side);
        }
    }
#pragma unroll 1
    for (int which = 0; which < 3; which++) {
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            // panels [c1, span], [c0, c1], [0, c0]; empty ones are skipped
            const double c0 = cut[side][0], c1 = cut[side][1];
            double lo = (which == 0) ? c1 : ((which == 1) ? c0 : 0.0);
            double hi = (which == 0) ? span : ((which == 1) ? c1 : c0);
            if (!(c0 < span)) { // no cut on this side: two halves instead of one wide panel
                lo = (which == 0) ? span : ((which == 1) ? kUncutSplit * span : 0.0);
                hi = (which == 0) ? span : ((which == 1) ? span : kUncutSplit * span);
                if (light) { // ... or the whole side as one
                    lo = (which == 2) ? 0.0 : span;
                    hi = span;
                }
            }
            if (graded && which == 2 && c0 < span)
                hi = kGrade * c0;
            if (hi > lo)
                stk.push(w, side ? lo : -hi, side ? hi : -lo, side);
        }
    }
    // A broken power law's df/dgamma jumps at the break, and f has a kink there: no panel straddles it.
    if (KIND == kDistPitchyBrokenPL)
        stk.cut_at(w, (bpl_gamma_break(*cx.d) - gamma_peak) / half, true);
    stk.seal();

    // Every application carries TWO panels as 15-point Kronrod rules, one per half warp (lanes
    // 0-14 and 16-30; lanes 15 and 31 have weight zero): the two topmost panels of the stack, or
    // the two halves of the last one.  The seeds are smooth by construction, so the 15-point
    // rule meets the tolerance on most of them at once and the number of applications per gamma
    // integral halves; a panel that misses its tolerance is bisected and its halves form the
    // next pair.
    while (stk.sp > 0) {
        double ta0, tb0, ta1, tb1;
        int side0, side1;
        stk.pop(ta0, tb0, side0);
        if (stk.sp > 0) {
            stk.pop(ta1, tb1, side1);
        } else {
            const double mid = 0.5 * (ta0 + tb0);
            ta1 = mid, tb1 = tb0, side1 = side0;
            tb0 = mid;
        }
        warp_fence(); // the previous reduce has finished reading the tile

#ifdef RB_DEVICE_BUILD
        {
            const bool second = (w.lane & 16) != 0;
            const double pa = second ? ta1 : ta0, pb = second ? tb1 : tb0;
            const double x = L15_X[w.lane], wk = L15_WK[w.lane], wd = L15_WD[w.lane];
            double vals[6];
            sym_node<KIND>(cx, n, gamma_peak + half * (0.5 * (pa + pb) + 0.5 * (pb - pa) * x), vals);
            tile_store_weighted<6, kSymInnerChan>(ws.inner.tile, w.lane, wk, wd, vals);
        }
#else
        for (int l = 0; l < 32; l++) {
            const bool second = (l & 16) != 0;
            const double pa = second ? ta1 : ta0, pb = second ? tb1 : tb0;
            double vals[6];
            sym_node<KIND>(cx, n, gamma_peak + half * (0.5 * (pa + pb) + 0.5 * (pb - pa) * L15_X[l]), vals);
            tile_store_weighted<6, kSymInnerChan>(ws.inner.tile, l, L15_WK[l], L15_WD[l], vals);
        }
#endif
        w.n_apply_lanes++;
        warp_fence();

        PerChan<double> r0, e0, r1, e1;
        tile_reduce_pair<kSymInnerChan>(ws.inner.tile, 6, 0.5 * (tb0 - ta0) * half, 0.5 * (tb1 - ta1) * half, r0, e0, r1, e1);

#pragma unroll
        for (int p = 0; p < 2; p++) {
            const PerChan<double> &r = p ? r1 : r0;
            const PerChan<double> &e = p ? e1 : e0;
            const double ta = p ? ta1 : ta0, tb = p ? tb1 : tb0;
            const int side = p ? side1 : side0;
            PerChan<bool> ok;
            RB_FOR_CHAN(c, kEngChan) { ok[c] = true; }
            RB_FOR_CHAN(c, 6)
            {
                big[c] = fmax(big[c], fabs(r[c]));
                ok[c] = panel_ok(r[c], e[c], light ? kLightGammaTolerance * cx.epsrel_gamma : cx.epsrel_gamma,
                                 kInnerFloor * fmax(est[c] + fabs(r[c]), big[c]));
            }
            const bool accept = chan_all(ok, 6);
            if (accept || !stk.room(2) || panel_too_small(ta, tb) || w.n_apply_lanes > kAppBudget) {
                if (!accept && w.n_apply_lanes > kAppBudget)
                    w.status |= kStatusCapHit; // (a panel at the bisection floor is an integrable end-point singularity)
                RB_FOR_CHAN(c, 6)
                {
                    est[c] += fabs(r[c]);
                    if (side)
                        sum_r[c] += r[c];
                    else
                        sum_l[c] += r[c];
                }
            } else {
                const double tc = 0.5 * (ta + tb);
                stk.push(w, ta, tc, side);
                stk.push(w, tc, tb, side);
            }
        }
        stk.seal();
    }

    // add the eight accumulators to the sums of the outer rule
    (void)col;
    warp_fence();
#ifdef RB_DEVICE_BUILD
    if ((w.lane & 3) == 0)
#endif
    {
        RB_FOR_CHAN(c, 6)
        {
            if (c < 4) {
                acc_add(ws.outer.acc, c, wa, wb, sum_l[c] + sum_r[c]);
            } else {
                acc_add(ws.outer.acc, c, wa, wb, sum_r[c]);
                acc_add(ws.outer.acc, c + 2, wa, wb, sum_l[c]);
            }
        }
    }
    warp_fence();
}

// Where G(n) is not smooth in n.  At the peak of the gamma window eps = (n - z)/n falls like
// n0^2 / (2 n^2) (n0 = s sin(theta)) while the thresholds at which pkgw_bessel_j switches
// Meissel -> blend -> Debye fall like n^(-2/3) (bessel.c:341-357): at n_a ~ (n0^2 / (2 10^B))^(3/4)
// the peak enters the blend zone, 23 % further up the Debye zone, and J_{n+1} does the same 1 %
// apart from J_n.  G(n) has a (n - n_a)^(3/2) onset at each of the four places, and between the
// two of a pair J_n' = n J_n / z - J_{n+1} mixes two expansions: a bump of ~1e-3 in G that the
// outer rule otherwise chases down to panels of 3 % width.  The four places are found here (one
// root each of eps_peak(n) - threshold(n + d), eight lanes per root, two passes) and the outer
// panels are cut at them.  kink[] is ascending; entries that do not exist are +inf.
template <int KIND>
RB_FN void sym_find_kinks(Warp &w, const SymFastCtx<KIND> &cx, double (&kink)[4])
{
    const double n0 = cx.s * fabs(cx.sin_th);
    const double sin2 = cx.sin_th * cx.sin_th;
    double found[4];
#ifdef RB_DEVICE_BUILD
    const int grp = w.lane >> 3, j = w.lane & 7;
#else
    for (int grp = 0; grp < 4; grp++) {
#endif
        const double shift = (double)(grp & 1);                      // order n or n + 1
        const double thr = (grp & 2) ? kTenMinusA : kTenMinusB;      // blend -> Debye, Meissel -> blend
        const double est = rb_exp(0.75 * rb_log(n0 * n0 / (2.0 * thr)));
        double lo = est * 0.7, hi = est * 1.4;
        double root = INFINITY;
        bool ok = est > 1.02 * n0 && est == est;
#pragma unroll 1
        for (int pass = 0; pass < 2; pass++) {
            const double ratio = rb_log(hi / lo) / 7.0;
#ifdef RB_DEVICE_BUILD
            const double nj = lo * rb_exp(ratio * j);
            double fj = NAN;
            if (ok && nj > n0 * (1.0 + 1e-9) && nj >= kNJn) {
                const double e = sym_eps_at<KIND>(cx, nj, (nj / cx.s) / sin2);
                fj = (shift + nj * e) / (nj + shift) - thr * rb_exp(kEtaSlope * rb_log(nj + shift));
            }
            const unsigned pos = (__ballot_sync(0xffffffffu, fj > 0.0) >> (8 * grp)) & 0xffu;
            const unsigned neg = (__ballot_sync(0xffffffffu, fj < 0.0) >> (8 * grp)) & 0xffu;
            const int cnt = __popc(pos);
            ok = ok && cnt >= 1 && cnt <= 7 && pos == ((1u << cnt) - 1u) && neg == (0xffu & ~pos);
            const int src = 8 * grp + (ok ? cnt - 1 : 0);
            const double fa = __shfl_sync(0xffffffffu, fj, src), na = __shfl_sync(0xffffffffu, nj, src);
            const double fb = __shfl_sync(0xffffffffu, fj, src + 1), nb = __shfl_sync(0xffffffffu, nj, src + 1);
#else
            double fv[8], nv[8];
            int cnt = 0;
            bool mono = true;
            for (int j = 0; j < 8; j++) {
                nv[j] = lo * rb_exp(ratio * j);
                fv[j] = NAN;
                if (ok && nv[j] > n0 * (1.0 + 1e-9) && nv[j] >= kNJn) {
                    const double e = sym_eps_at<KIND>(cx, nv[j], (nv[j] / cx.s) / sin2);
                    fv[j] = (shift + nv[j] * e) / (nv[j] + shift) - thr * rb_exp(kEtaSlope * rb_log(nv[j] + shift));
                }
                if (fv[j] > 0.0) {
                    if (cnt != j)
                        mono = false;
                    cnt++;
                } else if (!(fv[j] < 0.0))
                    mono = false;
            }
            ok = ok && mono && cnt >= 1 && cnt <= 7;
            const double fa = fv[ok ? cnt - 1 : 0], na = nv[ok ? cnt - 1 : 0];
            const double fb = fv[ok ? cnt : 1], nb = nv[ok ? cnt : 1];
#endif
            if (ok) {
                lo = na;
                hi = nb;
                // linear interpolation in ln n
                root = na * rb_exp(rb_log(nb / na) * (fa / (fa - fb)));
            }
        }
#ifdef RB_DEVICE_BUILD
    const double mine = ok ? root : INFINITY;
#pragma unroll
    for (int g = 0; g < 4; g++)
        found[g] = __shfl_sync(0xffffffffu, mine, 8 * g);
#else
        found[grp] = ok ? root : INFINITY;
    }
#endif
    // ascending (four values: a fixed network)
#define RB_SWAP_IF(a, b) do { if (found[a] > found[b]) { const double t_ = found[a]; found[a] = found[b]; found[b] = t_; } } while (0)
    RB_SWAP_IF(0, 1);
    RB_SWAP_IF(2, 3);
    RB_SWAP_IF(0, 2);
    RB_SWAP_IF(1, 3);
    RB_SWAP_IF(1, 2);
#undef RB_SWAP_IF
#pragma unroll
    for (int g = 0; g < 4; g++)
        kink[g] = found[g];
}

// All six j/alpha coefficients of one point, dimensionless (lib.rs:178-191);
// out6 = j_I, a_I, j_Q, a_Q, j_V, a_V; lobes4 = j_V(+), j_V(-), a_V(+), a_V(-).
template <int KIND>
RB_FN void symphony_point_fast(Warp &w, const Dist &dist, double s, double theta, double epsrel_gamma,
                               double epsrel_n, SymFastWS &ws, double (&out6)[6], double (&lobes4)[4])
{
    constexpr double kNMax = 30.0, kTolerance = 1e5;

    static_assert(sizeof(SymFastCtx<KIND>) <= sizeof(ws.ctx_store), "context store too small");
    warp_fence();
    SymFastCtx<KIND> &cx = *reinterpret_cast<SymFastCtx<KIND> *>(ws.ctx_store);
    ws.dist = dist; // every lane stores the same values
    cx.d = &ws.dist;
    cx.ws = &ws;
    cx.s = s;
    cx.cos_th = cos(theta);
    cx.sin_th = sin(theta);
    cx.inv_s = 1.0 / s;
    cx.inv_sin_th = 1.0 / cx.sin_th;
    cx.epsrel_gamma = epsrel_gamma;
    warp_fence();

    const double n_minus = s * fabs(cx.sin_th);
    const long long n_lo = (long long)(n_minus + 1.0);
    const long long n_hi = (long long)(n_minus + 1.0 + kNMax);
    const double n_start = floor(n_minus + 1.0 + kNMax);

    // the first 30 harmonics, discretely (symphony.rs:96-108): a tile with unit weights
    warp_fence();
    acc_clear(w, ws.outer.acc);
    warp_fence();
    {
        int col = 0;
        for (long long n = n_lo; n < n_hi; n++, col++)
            sym_gamma_integral<KIND>(w, cx, (double)n, tile_col(col), 1.0, 0.0);
    }
    warp_fence();
    PerChan<double> disc, unused;
    acc_reduce(ws.outer.acc, 1.0, disc, unused);

    // The rest, treating n as continuous (symphony.rs:124-140).  The chunks [n_start,
    // n_start + delta_n] and the rules that grow delta_n and end the loop are the
    // reference's (symphony.rs:196-295), because where the loop ends decides how much of a
    // slowly decaying tail (hard kappa spectra) is included: the result is a truncated
    // integral and parity means truncating it at the same place.  Each chunk is integrated
    // in u = ln n with the outer rule; the derivative probe is a central difference.
    PerChan<double> tail, contrib;
    PerChan<bool> active, handed; // handed: left to the faithful continuation by the fidelity guard
    RB_FOR_CHAN(c, kEngChan)
    {
        tail[c] = 0.0;
        contrib[c] = 0.0;
        active[c] = (disc[c] - disc[c] == 0.0); // finite so far
        handed[c] = false;
    }
    double n_lo_chunk = n_start;
    double delta_n = 1e5, incr_step_factor = 10.0;
    if (s < 10.0) { // "At low harmonic numbers, step conservatively since every n counts."
        delta_n = 1.0;
        incr_step_factor = 2.0;
    }
    constexpr double kDerivTol = 1e-5, kDerivStep = 1e-3;
    PanelStack stk;
    double kink[4];
    sym_find_kinks<KIND>(w, cx, kink);

    bool have_snap = false;
#ifdef RB_DEVICE_BUILD
    if (w.lane == 0)
#endif
    {
        ws.snap[kSnapValid] = 0.0;
        ws.snap[kSnapDone] = 0.0;
    }

    for (int chunk_no = 0; chunk_no < kMaxChunks; chunk_no++) {
        if (!have_snap && n_lo_chunk >= kHandoverN && s >= 10.0 && s < 1e6) {
            have_snap = true;
            warp_fence();
#ifdef RB_DEVICE_BUILD
            if (w.lane == 0)
#endif
            {
                ws.snap[kSnapNStart] = n_lo_chunk;
                ws.snap[kSnapDeltaN] = delta_n;
                ws.snap[kSnapIncr] = incr_step_factor;
                ws.snap[kSnapValid] = 1.0;
                ws.snap[kSnapActive] = 0.0;
                ws.snap[kSnapDone] = 0.0;
            }
            warp_fence();
#ifdef RB_DEVICE_BUILD
            if ((w.lane & 3) == 0)
#endif
            {
                RB_FOR_CHAN(c, kEngChan)
                {
                    ws.snap[kSnapDisc + c] = disc[c];
                    ws.snap[kSnapTail + c] = tail[c];
                    ws.snap[kSnapContrib + c] = contrib[c];
                }
            }
            // active mask, assembled by lane 0 from a vote
            unsigned mask = 0;
#ifdef RB_DEVICE_BUILD
            mask = __ballot_sync(0xffffffffu, active.v && (w.lane & 3) == 0);
            unsigned packed = 0;
            for (int c = 0; c < kEngChan; c++)
                packed |= ((mask >> (4 * c)) & 1u) << c;
            if (w.lane == 0)
                ws.snap[kSnapActive] = (double)packed;
#else
            for (int c = 0; c < kEngChan; c++)
                mask |= (active.v[c] ? 1u : 0u) << c;
            ws.snap[kSnapActive] = (double)mask;
#endif
            warp_fence();
        }

        // d G / d n at the start of the chunk
        warp_fence();
        acc_clear(w, ws.outer.acc);
        warp_fence();
        {
            const double dn = kDerivStep * n_lo_chunk;
            // Kronrod sum: the central difference; the second sum: the mean of the two probes, G at the start
            sym_gamma_integral<KIND>(w, cx, n_lo_chunk - dn, tile_col(0), -0.5 / dn, 0.5);
            sym_gamma_integral<KIND>(w, cx, n_lo_chunk + dn, tile_col(1), 0.5 / dn, 0.5);
        }
        warp_fence();
        PerChan<double> deriv, unused2;
        acc_reduce(ws.outer.acc, 1.0, deriv, unused2);
        // G at the start of the chunk, from the same two probes
        PerChan<double> g_start;
        RB_FOR_CHAN(c, kEngChan) { g_start[c] = ws.outer.acc.d[c]; }
        PerChan<bool> grow_c;
        RB_FOR_CHAN(c, kEngChan)
        {
            grow_c[c] = !active[c] || deriv[c] == 0.0 || (contrib[c] != 0.0 && fabs(deriv[c] / contrib[c]) < kDerivTol);
        }
#ifdef RB_TRACE_VOTE
        RB_TRACE_VOTE(chunk_no, n_lo_chunk, delta_n, active, grow_c);
#endif
        if (chan_all(grow_c, kEngChan))
            delta_n *= incr_step_factor;
        if (delta_n < n_lo_chunk / incr_step_factor)
            delta_n *= incr_step_factor;

        // the chunk, cut into panels of at most kPanelWidth in u; the rightmost is popped first
        const double u_lo = rb_log(n_lo_chunk), u_hi = rb_log(n_lo_chunk + delta_n);
        stk.reset(&ws.outer);
        {
            // segments between the kinks of G(n) that fall inside the chunk (sym_find_kinks)
            double seg_lo = u_lo;
#pragma unroll 1
            for (int g = 0; g <= 4; g++) {
                double seg_hi = u_hi;
                if (g < 4) {
                    const double nk = kink[g];
                    if (!(nk > n_lo_chunk * (1.0 + 1e-6) && nk < (n_lo_chunk + delta_n) * (1.0 - 1e-6)))
                        continue;
                    seg_hi = rb_log(nk);
                }
                if (seg_hi > seg_lo) {
                    int n_seed = (int)ceil((seg_hi - seg_lo) / kPanelWidth);
                    n_seed = n_seed < 1 ? 1 : (n_seed > 6 ? 6 : n_seed);
                    for (int k = 0; k < n_seed && stk.room(3); k++)
                        stk.push(w, seg_lo + (seg_hi - seg_lo) * k / n_seed,
                                 (k + 1 == n_seed) ? seg_hi : seg_lo + (seg_hi - seg_lo) * (k + 1) / n_seed, 0);
                    seg_lo = seg_hi;
                }
            }
            if (stk.sp == 0) // degenerate bounds (NaN, infinite): one panel, whose value is NaN
                stk.push(w, u_lo, u_hi, 0);
        }
        stk.seal();

        PerChan<double> chunk;
        RB_FOR_CHAN(c, kEngChan) { chunk[c] = 0.0; }
        // far up the tail, where the previous chunk added less than kLightChunk of the sum, the
        // 7-point rule is plenty for a decade of a power law (and 1e-3 of such a chunk is
        // far inside the tolerance)
        // ... or, without waiting for a chunk to say so: past the maximum |G| falls, so |G(n_start)| delta_n bounds
        // the chunk from above; when that bound is below kLightChunk of the sum the chunk is minor already
        PerChan<bool> minor;
        RB_FOR_CHAN(c, kEngChan)
        {
            const double sum_c = fabs(disc[c] + tail[c]);
            const bool falling = g_start[c] * deriv[c] < 0.0;
            // a power-law tail G ~ n^-a (a = -d ln G / d ln n from the probe) integrates to G n / (a - 1); twice
            // that, or the cruder |G| delta_n, whichever is smaller
            const double a_slope = -deriv[c] * n_lo_chunk / g_start[c];
            double bound = fabs(g_start[c]) * delta_n;
            if (a_slope > 1.25)
                bound = fmin(bound, 2.0 * fabs(g_start[c]) * n_lo_chunk / (a_slope - 1.0));
            minor[c] = !active[c] || (contrib[c] != 0.0 && fabs(contrib[c]) < kLightChunk * sum_c) ||
                       (falling && bound < kLightChunk * sum_c);
        }
        const bool light = chunk_no > 0 && chan_all(minor, kEngChan);
        warp_fence();
        while (stk.sp > 0) {
            double ua, ub;
            int tag;
            stk.pop(ua, ub, tag);
            const double uc = 0.5 * (ua + ub), uhl = 0.5 * (ub - ua);
            warp_fence();
            // outer rule by panel width: K15 for wide panels, K7 for narrow ones
            const bool narrow = light || (ub - ua) < kNarrowPanel;
            const int n_nodes = narrow ? 7 : 15;
            const double *rx = narrow ? GK7_X : GK15_X;
            const double *rwk = narrow ? GK7_WK : GK15_WK;
            const double *rwd = narrow ? GK7_WD : GK15_WD;
            acc_clear(w, ws.outer.acc);
            warp_fence();
#pragma unroll 1
            for (int j = 0; j < n_nodes; j++) {
                const double n = rb_exp(uc + uhl * rx[j]);
                sym_gamma_integral<KIND>(w, cx, n, tile_col(j), rwk[j] * n, rwd[j] * n, light);
            }
            warp_fence();
            PerChan<double> r, e;
            acc_reduce(ws.outer.acc, uhl, r, e);

            PerChan<bool> ok;
            RB_FOR_CHAN(c, kEngChan)
            {
                ok[c] = !active[c] || panel_ok(r[c], e[c], epsrel_n, fabs(disc[c] + tail[c] + chunk[c]));
            }
            const bool accept = chan_all(ok, kEngChan);
            if (accept || !stk.room(2) || panel_too_small(ua, ub) || w.n_apply_lanes > kAppBudget) {
                if (!accept)
                    w.status |= kStatusCapHit;
                RB_FOR_CHAN(c, kEngChan) { chunk[c] += r[c]; }
            } else {
                stk.push(w, ua, uc, 0);
                stk.push(w, uc, ub, 0);
                stk.seal();
            }
        }

        if (n_lo_chunk >= kSensitiveN && s < 1e6) {
            // Fidelity guard, per accumulator: one whose chunks up here still matter leaves this
            // path (it is the emission coefficients of hard spectra, as a rule; absorption and
            // Stokes V decay faster) and is finished by the faithful sequence from the recorded
            // state; the others carry on here and keep their values.  Without a recorded state
            // (s < 10) the whole point is handed over.
            PerChan<bool> calm;
            RB_FOR_CHAN(c, kEngChan)
            {
                calm[c] = !active[c] || !(fabs(chunk[c]) > kSensitiveFraction * fabs(disc[c] + tail[c] + chunk[c]));
                if (!calm[c]) {
                    handed[c] = true;
                    active[c] = false;
                }
            }
            if (!chan_all(calm, kEngChan)) {
                w.status |= kStatusRerouted;
                if (!have_snap)
                    break;
            }
        }

        PerChan<bool> done;
        RB_FOR_CHAN(c, kEngChan)
        {
            if (active[c]) {
                contrib[c] = chunk[c];
                tail[c] += chunk[c];
                // loop condition of the reference (symphony.rs:225); a NaN contribution also ends it
                if (!(fabs(contrib[c]) >= fabs(tail[c] / kTolerance)))
                    active[c] = false;
            }
            done[c] = !active[c];
        }
        if (chan_all(done, kEngChan))
            break;
        n_lo_chunk += delta_n;
        if (n_lo_chunk > 1e13)
            incr_step_factor = 1.0;
        if (chunk_no == kMaxChunks - 1)
            w.status |= kStatusCapHit;
    }

    if ((w.status & kStatusRerouted) && have_snap) {
        // partial handover: the recorded state keeps (tail, contrib) of the accumulators that are
        // handed over; the others get their final sums and are marked finished, which is how
        // symphony_tail_faithful treats an accumulator that had converged before the record
        warp_fence();
#ifdef RB_DEVICE_BUILD
        if ((w.lane & 3) == 0)
#endif
        {
            RB_FOR_CHAN(c, kEngChan)
            {
                if (!handed[c])
                    ws.snap[kSnapTail + c] = tail[c];
            }
        }
        unsigned packed = 0;
#ifdef RB_DEVICE_BUILD
        const unsigned mask = __ballot_sync(0xffffffffu, handed.v && (w.lane & 3) == 0);
        for (int c = 0; c < kEngChan; c++)
            packed |= ((mask >> (4 * c)) & 1u) << c;
        if (w.lane == 0)
            ws.snap[kSnapActive] = (double)packed;
#else
        for (int c = 0; c < kEngChan; c++)
            packed |= (handed.v[c] ? 1u : 0u) << c;
        ws.snap[kSnapActive] = (double)packed;
#endif
        warp_fence();
    }

    PerChan<double> ans;
    RB_FOR_CHAN(c, kEngChan) { ans[c] = disc[c] + tail[c]; }

    // dimensional constants outside the integrals (symphony.rs:173-183)
    const double two_pi_e = kTwoPi * kElectronCharge;
    const double pre_j = two_pi_e * two_pi_e / (kSpeedLight * fabs(cx.cos_th));
    const double pre_a = -1.0 * two_pi_e * two_pi_e / (2.0 * kMassElectron * kSpeedLight * fabs(cx.cos_th));

    double total[kEngChan];
#pragma unroll
    for (int c = 0; c < kEngChan; c++)
        total[c] = chan_get(ans, c);

    out6[0] = total[0] * pre_j;
    out6[1] = total[1] * pre_a;
    out6[2] = total[2] * pre_j;
    out6[3] = total[3] * pre_a;
    lobes4[0] = total[4] * pre_j;
    lobes4[1] = total[6] * pre_j;
    lobes4[2] = total[5] * pre_a;
    lobes4[3] = total[7] * pre_a;
    out6[4] = lobes4[0] + lobes4[1];
    out6[5] = lobes4[2] + lobes4[3];
}

} // namespace rb
