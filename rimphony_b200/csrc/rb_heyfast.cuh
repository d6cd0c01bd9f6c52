// rb_heyfast.cuh -- rho_Q (Heyvaerts' "h") and rho_V ("f") of one point on the
// product ("fast") path: the non-resonant (NR) + quasi-resonant (QR) double
// integrals of src/heyvaerts.rs:60-191 evaluated with the compact engine of
// rb_engine.cuh.
//
// Same integrands (rb_heyvaerts.cuh HeyNRIntegrand / HeyQRIntegrand restate
// heyvaerts.rs:302-468), same domains, same outward-stepping sequence and
// termination rule as the reference (heyvaerts.rs:85-185): the result is a
// truncated integral, so the steps [edge, edge + delta], the rule that grows
// delta (x5 when |1 / (F'(edge) delta)| > 5) and the stop test |contrib / total|
// <= 1e-5 are kept.  What differs is the quadrature inside a step:
//
//   * h and f share every node (coordinates, df/dsigma, the four I_{+-1/3},
//     I_{+-2/3} or the J/Y pair) and are converged together;
//   * the NR inner integral over sigma in [sigma_min, sigma_min^1.5/sqrt(3)] and
//     every outward step are integrated in the logarithm of the variable (the
//     integrands are algebraic times a power-law-like df/dsigma: smooth in the
//     log, a bisection cascade towards the lower end in the variable itself);
//   * the central NR integral over pomega in [-3 sigma0, 3 sigma0] is cut at 0 and,
//     for sigma0 < 3, at the edges of the hole |pomega| < sqrt(9 - sigma0^2) where
//     the NR domain is empty (the integrand has slope breaks there);
//   * the derivative probe of the step rule is a central difference.
#pragma once

#include "rb_engine.cuh"
#include "rb_heyvaerts.cuh"

namespace rb {

constexpr int kHeyChan = 2; // channel rows of the tiles: rho_Q and rho_V
constexpr double kHeyInnerFloor = 1.0;
constexpr double kHeyInnerWidth = 4.0; // widest NR inner seed panel in t = arccosh(sigma / sigma_min)
constexpr double kHeyPanelWidth = 2.0; // widest outer panel in the log of the variable
constexpr double kHeyLightStep = 1e-3; // a step after one that added less than this fraction gets the 7-point rule
constexpr double kHeyDerivStep = 1e-4; // relative step of the derivative probe
constexpr int kHeyOuterMaxDepth = 13;  // bisections below a seed after which an outer panel is accepted as it is

// Where the reference's own quadrature gives up.  A distribution with 1/(gamma^2 beta) in it (the
// power laws with gamma_min = 1) makes df/dsigma diverge like (gamma - 1)^-3/2 where gamma -> 1.  In
// the QR domain that is the single point sigma = s, pomega = s cos(theta) (the line gamma = 1 touches
// the edge x = 0 of the domain there; for s > 3 the point lies outside pomega_max).  The QR
// elements vanish at that point (pi^2 x^2 J'Y' - pi^2 pomega^2 JY + t3 -> 0), the next order is
// J_sigma(x)^2 ~ x^(2 sigma): along sigma = s the inner integrand goes like delta^(s - 3/2) in the
// distance delta to the end of the pomega range and the outer integrand like |sigma - s|^(2 s - 1),
// an integrable singularity for s < 1/2 (a cusp above).  The reference's QAG (epsrel 1e-3, no
// extrapolation) bisects towards sigma = s; the inner integrals next to it chase their own
// end-point singularity down to the last ulps of the pomega range, where the rounded cos(xi)
// reaches 1 and sin^k(xi), 1 / sin^2(xi) turn into NaN (heyvaerts.rs:194-201, pitchy_pl.rs:44-61):
// QAG error -> NaN coefficient (heyvaerts.rs:175-177).  Whether the outer QAG converges before it
// samples such a sigma is decided by the exponent: measured on 14 096 oracle points
// (tests/golden/heyvaerts_low_s.md) the reference returns NaN for 97 % of the points with
// s < 0.3 and a finite value for 97 % of those with s > 0.5 (rho_Q; rho_V the same 0.04 higher),
// and the set moves with the reference's tolerance (1e-4: +15 % NaN, 1e-5: +40 %) while its
// finite values do not.  The product path integrates the same integrand with cos(xi) -> +-1
// handled exactly (HeyNode::fill), so it would return the finite value of the integral there;
// to stay a drop-in it reports what the reference reports: NaN + STATUS_REFERENCE_DIVERGES below
// the thresholds that follow, without spending the 10-50 k rule applications such a point costs.
// A point that has used this many rule applications is not going to converge (the ones that do
// need 0.5-10 k): it is chasing the x^(k-2) end-point behaviour of d f / d cos(xi) at small k or
// theta -> 0, where the reference fails as well (tests/golden/heyvaerts_low_s.md).  NaN + CAP_HIT,
// and the tail of the persistent kernel stays short.
constexpr unsigned kHeyAppBudget = 20000;
// rho_V: a sharp boundary in s.  rho_Q: the strength of the singular term goes like sin^2(theta), so the
// boundary rises with theta (fitted on the oracle's verdicts for 14 096 pitchy and 10 000 isotropic points,
// tests/golden/study_heyvaerts_low_s.py map): s_c = lo + (hi - lo) clamp((theta - t0) / (t1 - t0), 0, 1).
constexpr double kHeyRefDivergesV = 0.38;    // pitchy power law
constexpr double kHeyRefDivergesIsoV = 0.33; // isotropic power law (k = 0: no pitch-angle factor)
constexpr double kHeyDivQLo = 0.18, kHeyDivQHi = 0.37, kHeyDivQT0 = 0.15, kHeyDivQT1 = 0.40;       // pitchy
constexpr double kHeyDivIsoQLo = 0.0, kHeyDivIsoQHi = 0.30, kHeyDivIsoQT0 = 0.20, kHeyDivIsoQT1 = 1.40; // isotropic
constexpr double kHeyRefDivergesMax = 0.38; // no point with s at or above this is touched by the rule

RB_HD double hey_ref_diverges_q(bool isotropic, double sin_th, double cos_th)
{
    const double lo = isotropic ? kHeyDivIsoQLo : kHeyDivQLo, hi = isotropic ? kHeyDivIsoQHi : kHeyDivQHi;
    const double t0 = isotropic ? kHeyDivIsoQT0 : kHeyDivQT0, t1 = isotropic ? kHeyDivIsoQT1 : kHeyDivQT1;
    const double theta = atan2(fabs(sin_th), fabs(cos_th)); // folded into [0, pi/2]
    double x = (theta - t0) / (t1 - t0);
    x = x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x);
    return lo + (hi - lo) * x;
}

struct HeyFastWS {
    EngLevelT<kHeyChan> inner, outer;
    // the warp-uniform context of the point in work, in shared memory rather than on the kernel's stack
    // (see SymFastWS)
    Dist dist;
    double ctx_store[10];
    JYOrder jy; // J/Y orders of the quasi-resonant inner integral in work (rb_special.cuh)
};

template <int KIND>
struct HeyFastCtx {
    const Dist *d;
    HeyFastWS *ws;
    HeyGeometry g;
    double epsrel_inner, epsrel_outer;
};

enum { kHeyNR = 0, kHeyQR = 1 };
// how the outer variable is mapped: v = t, v = rb_exp(t), v = -rb_exp(t), v = v_lo + t^2
enum { kMapLinear = 0, kMapLog = 1, kMapNegLog = 2, kMapSqrt = 3 };

// Note on NaN: at the isolated points of the (sigma, pomega) plane where gamma = 1 a power law's
// f and its derivatives are infinite and df/dsigma evaluates to inf - inf.  For s sin(theta) < 1
// deep bisection towards such a point can land a node on it; the NaN then propagates to the
// coefficient (status NAN), which is also what the reference's QAG does when it happens to it.
// (Dropping the sample instead makes these points integrate a non-integrable singularity to
// the application budget: 10x the cost for values nobody can use.)

// One inner integral (both channels) at the outer node `v` (pomega for NR, sigma for
// QR), multiplied by wa / wb and parked in column `col` of the outer tile.
// Returns true when the integral is NaN in both channels (a NaN node value: the integrand is
// inf - inf where gamma = 1, see the note above); the caller's result is NaN then, whatever
// the other nodes hold.
template <int KIND>
RB_FN_NOINLINE bool hey_inner_integral(Warp &w, const HeyFastCtx<KIND> &cx, int which, double v, int col, double wa,
                                       double wb)
{
    HeyFastWS &ws = *cx.ws;
    const HeyGeometry &g = cx.g;
    PanelStack stk;
    stk.reset(&ws.inner);

    bool empty = false;
    // QR with pomega_max = sqrt(sigma^2 - sigma0^2): x -> 0 at both ends of the pomega range and the
    // elements behave like powers of x = sqrt(pomega_max^2 - pomega^2) there; pomega = pomega_max sin(phi)
    // makes x = pomega_max cos(phi) and the integrand analytic in phi.
    bool sine_map = false;
    double sine_amp = 0.0;
    double nr_sigma_min = 0.0;
    if (which == kHeyNR) {
        // heyvaerts.rs:213-250: sigma in [sigma_min, sigma_min^1.5 / sqrt(3)], in t = ln sigma
        const double sigma_min = rb_sqrt(v * v + g.sigma0_sq);
        const double sigma_max = kInverseSqrt3 * sigma_min * rb_sqrt(sigma_min);
        if (!(sigma_max > sigma_min)) {
            empty = true;
        } else {
            // sigma = sigma_min cosh(t): x = sigma_min sinh(t) exactly, d sigma = x dt.  Near the
            // lower end (x -> 0, where the integrand has algebraic end-point behaviour, strongest
            // around the cusp pomega*) t is linear in x; far out it is ln sigma.
            nr_sigma_min = sigma_min;
            const double ratio = kInverseSqrt3 * rb_sqrt(sigma_min);
            const double t_lo = 0.0, t_hi = rb_log(ratio + rb_sqrt((ratio - 1.0) * (ratio + 1.0)));
            int n_seed = (int)ceil((t_hi - t_lo) / kHeyInnerWidth);
            n_seed = n_seed < 1 ? 1 : (n_seed > 8 ? 8 : n_seed);
            for (int k = n_seed - 1; k >= 0; k--) // the lowest panel (largest values) is popped first
                stk.push(w, t_lo + (t_hi - t_lo) * k / n_seed, (k + 1 == n_seed) ? t_hi : t_lo + (t_hi - t_lo) * (k + 1) / n_seed, 0);
            if (KIND == kDistPitchyBrokenPL) {
                // df/dsigma jumps where the line gamma = gamma_break, sigma = gamma_break sigma0 sin(theta) +
                // pomega cos(theta), crosses the range: cut at its t
                const double r = (bpl_gamma_break(*cx.d) * g.sigma0 * g.sin_th + v * g.cos_th) / sigma_min;
                stk.cut_at(w, (r > 1.0) ? rb_log(r + rb_sqrt((r - 1.0) * (r + 1.0))) : NAN, false);
            }
        }
    } else {
        // heyvaerts.rs:262-296: pomega in [-pomega_max, pomega_max]
        const double pomega_max_phys = rb_sqrt(kThreeTwoThirds * rb_cbrt(v) * v - g.sigma0_sq);
        const double pomega_max_qr = rb_sqrt(v * v - g.sigma0_sq);
        const double pomega_max = fmin(pomega_max_phys, pomega_max_qr);
        if (!(pomega_max > 0.0) && pomega_max == pomega_max)
            empty = true;
        else {
            // The QR elements switch from the I_{+-1/3}, I_{+-2/3} form to the J/Y form where
            // g = sqrt(8)/3 (sigma - x)^1.5 / sqrt(x) reaches 10 (heyvaerts.rs:33, 330, 358,
            // 434): the integrand jumps there.  Find x_g with g(x_g) = 10 (g decreases in x;
            // safeguarded Newton) and cut the pomega range at +-sqrt(sigma^2 - sigma0^2 - x_g^2).
            double cut = pomega_max;
            // g grows towards the ends of the range (x shrinks): no cut when it stays below 10 there
            const double x_end_sq = v * v - g.sigma0_sq - pomega_max * pomega_max;
            bool g_reaches_cutoff = true;
            if (x_end_sq > 0.0) {
                const double x_end = rb_sqrt(x_end_sq);
                const double d_end = v - x_end;
                // g < 10  <=>  (sigma - x)^3 < (10 / (sqrt(8)/3))^2 x
                g_reaches_cutoff = !(d_end * d_end * d_end < (kGApproximationCutoff / kSqrt8Over3) * (kGApproximationCutoff / kSqrt8Over3) * x_end);
            }
            if (g_reaches_cutoff) {
                // (v - x)^1.5 = K sqrt(x), K = 10 / (sqrt(8)/3): with u = x / v the cubic (1 - u)^3 v^2 - K^2 u = 0,
                // convex and falling on [0, 1]: Newton from u = 0 approaches the root from the left, no square roots
                constexpr double big_k2 = (kGApproximationCutoff / kSqrt8Over3) * (kGApproximationCutoff / kSqrt8Over3);
                const double v2 = v * v;
                double u = 0.0;
#pragma unroll 1
                for (int it = 0; it < 60; it++) {
                    const double w1 = 1.0 - u;
                    const double w2 = w1 * w1 * v2;
                    const double un = u + rb_div(w1 * w2 - big_k2 * u, 3.0 * w2 + big_k2);
                    const bool done = fabs(un - u) <= 1e-10; // (a panel boundary)
                    u = un;
                    if (done)
                        break;
                }
                const double x = u * v;
                const double p2 = v * v - g.sigma0_sq - x * x;
                if (p2 > 0.0) {
                    const double pg = rb_sqrt(p2);
                    if (pg < pomega_max)
                        cut = pg;
                } else
                    cut = 0.0; // g >= 10 on the whole range
            }
            double end = pomega_max;
            if (pomega_max_qr <= pomega_max_phys) {
                sine_map = true;
                sine_amp = pomega_max;
                end = 0.5 * kPi;
                if (cut > 0.0 && cut < pomega_max)
                    cut = asin(cut / pomega_max);
                else if (cut >= pomega_max)
                    cut = end;
            }
            // the ends of the range beyond the cut (all of it when cut = 0) are in the J/Y form: its orders
            // sigma, sigma - 1 are the same for every node of this integral and are prepared once
            warp_fence();
            if (cut < end)
                jy_prepare(v, ws.jy); // every lane writes the same values
            else
                ws.jy.sigma = NAN;
            warp_fence();
            if (cut > 0.0 && cut < end) {
                stk.push(w, -end, -cut, 0);
                stk.push(w, cut, end, 0);
                stk.push(w, -cut, cut, 0);
            } else
                stk.push(w, -end, end, 0);
            if (KIND == kDistPitchyBrokenPL) {
                // df/dsigma jumps on the line gamma = gamma_break, pomega = (sigma - gamma_break sigma0 sin(theta)) /
                // cos(theta): cut at its pomega, or its phi under the sine map (NaN outside the range: no cut)
                const double pomega_b = (v - bpl_gamma_break(*cx.d) * g.sigma0 * g.sin_th) / g.cos_th;
                stk.cut_at(w, sine_map ? asin(pomega_b / sine_amp) : pomega_b, false);
            }
        }
    }
    stk.seal();

    PerChan<double> sum, est, big;
    RB_FOR_CHAN(c, kEngChan)
    {
        sum[c] = 0.0;
        est[c] = 0.0;
        big[c] = 0.0;
    }

    bool all_nan = false;
    while (!empty && stk.sp > 0) {
        double ta, tb;
        int tag;
        stk.pop(ta, tb, tag);
        const double tc = 0.5 * (ta + tb), thl = 0.5 * (tb - ta);
        warp_fence();
#ifdef RB_DEVICE_BUILD
        {
            double vals[2];
            const double t = tc + thl * w.xk;
            if (which == kHeyNR) {
                const double et = rb_exp(t), eti = rb_rcp(et);
                const double sigma = nr_sigma_min * 0.5 * (et + eti);
                const double x = nr_sigma_min * 0.5 * (et - eti);
                HeyNRIntegrand<KIND, 2> f{cx.d, &g, v, 0};
                f.eval(sigma, vals, x);
                vals[0] *= x;
                vals[1] *= x;
            } else {
                HeyQRIntegrand<KIND, 2> f{cx.d, &g, v, 0, &ws.jy};
                if (sine_map) {
                    double sin_t, cos_t;
                    sincos(t, &sin_t, &cos_t);
                    const double jac = sine_amp * cos_t; // = x, exactly
                    f.eval(sine_amp * sin_t, vals, jac);
                    vals[0] *= jac;
                    vals[1] *= jac;
                } else
                    f.eval(t, vals);
            }
            tile_store<2, kHeyChan>(ws.inner.tile, w, w.lane, vals);
        }
#else
        for (int l = 0; l < 32; l++) {
            double vals[2];
            const double t = tc + thl * LANE_X[l];
            if (which == kHeyNR) {
                const double et = rb_exp(t), eti = rb_rcp(et);
                const double sigma = nr_sigma_min * 0.5 * (et + eti);
                const double x = nr_sigma_min * 0.5 * (et - eti);
                HeyNRIntegrand<KIND, 2> f{cx.d, &g, v, 0};
                f.eval(sigma, vals, x);
                vals[0] *= x;
                vals[1] *= x;
            } else {
                HeyQRIntegrand<KIND, 2> f{cx.d, &g, v, 0, &ws.jy};
                if (sine_map) {
                    double sin_t, cos_t;
                    sincos(t, &sin_t, &cos_t);
                    const double jac = sine_amp * cos_t; // = x, exactly
                    f.eval(sine_amp * sin_t, vals, jac);
                    vals[0] *= jac;
                    vals[1] *= jac;
                } else
                    f.eval(t, vals);
            }
            tile_store<2, kHeyChan>(ws.inner.tile, w, l, vals);
        }
#endif
        w.n_apply_lanes++;
        warp_fence();

        PerChan<double> r, e;
        tile_reduce<kHeyChan>(ws.inner.tile, 2, thl, r, e);

        PerChan<bool> ok;
        RB_FOR_CHAN(c, kEngChan) { ok[c] = true; }
        RB_FOR_CHAN(c, 2)
        {
            big[c] = fmax(big[c], fabs(r[c]));
            ok[c] = panel_ok(r[c], e[c], cx.epsrel_inner, kHeyInnerFloor * fmax(est[c] + fabs(r[c]), big[c]));
        }
        const bool accept = chan_all(ok, 2);
        if (accept || !stk.room(2) || panel_too_small(ta, tb) || w.n_apply_lanes > kAppBudget) {
            if (!accept && w.n_apply_lanes > kAppBudget)
                w.status |= kStatusCapHit; // (a panel at the bisection floor is an integrable end-point singularity)
            RB_FOR_CHAN(c, 2)
            {
                est[c] += fabs(r[c]);
                sum[c] += r[c];
            }
            // an accepted NaN panel makes the sum NaN: nothing is left to integrate once that
            // holds for both channels
            PerChan<bool> gone;
            RB_FOR_CHAN(c, kEngChan) { gone[c] = true; }
            RB_FOR_CHAN(c, 2) { gone[c] = !(sum[c] == sum[c]); }
            if (chan_all(gone, 2)) {
                all_nan = true;
                break;
            }
        } else {
            stk.push(w, tc, tb, 0);
            stk.push(w, ta, tc, 0);
            stk.seal();
        }
    }

    double *ot = ws.outer.tile;
#ifdef RB_DEVICE_BUILD
    if ((w.lane & 3) == 0)
#endif
    {
        RB_FOR_CHAN(c, 2)
        {
            ot[c * kEngRow + col] = wa * sum[c];
            ot[(kHeyChan + c) * kEngRow + col] = wb * sum[c];
        }
    }
    return all_nan;
}

// The outer integral of one step: both channels over v in [v_lo, v_hi] (same sign, or any
// interval for the linear map), adaptive in the mapped variable with the sequential K15 / K7
// rules.  `scale` is the magnitude of the running total, the floor of the acceptance test.
template <int KIND>
RB_FN_NOINLINE void hey_outer_integral(Warp &w, const HeyFastCtx<KIND> &cx, int which, int map, double v_lo, double v_hi,
                                       const PerChan<double> &scale, PerChan<double> &result, bool light = false)
{
    HeyFastWS &ws = *cx.ws;
    PanelStack stk;
    stk.reset(&ws.outer);

    // mapped range [t_lo, t_hi]; `offset` is the start of the sqrt map v = offset + t^2
    double t_lo, t_hi;
    if (map == kMapLinear) {
        t_lo = v_lo;
        t_hi = v_hi;
    } else if (map == kMapSqrt) {
        t_lo = 0.0;
        t_hi = sqrt(v_hi - v_lo);
    } else {
        // v = +-rb_exp(t); for the negative branch t runs from ln|v_hi| to ln|v_lo|
        t_lo = (map == kMapLog) ? rb_log(v_lo) : rb_log(-v_hi);
        t_hi = (map == kMapLog) ? rb_log(v_hi) : rb_log(-v_lo);
    }
    const double offset = v_lo;
    {
        // Break point: the NR integrand has a cusp at pomega* = sigma0 cot(theta), where the
        // lower end of the inner sigma range touches gamma = 1 (there a power law's
        // 1/(gamma^2 beta) is singular); panels are cut there.
        double t_star = t_hi;
        if (which == kHeyNR) {
            const double p_star = cx.g.sigma0 * cx.g.cos_th / cx.g.sin_th;
            if (p_star > v_lo && p_star < v_hi)
                t_star = (map == kMapLinear) ? p_star : rb_log(p_star); // p_star > 0: linear or log map
        }
        const double max_w = (map == kMapLog || map == kMapNegLog) ? kHeyPanelWidth : INFINITY;
        // upper segment [t_star, t_hi] first so that the lower one is popped first
#pragma unroll 1
        for (int seg = 1; seg >= 0; seg--) {
            const double a = seg ? t_star : t_lo, b = seg ? t_hi : t_star;
            if (!(b > a))
                continue;
            int n_seed = (max_w < INFINITY) ? (int)ceil((b - a) / max_w) : 1;
            n_seed = n_seed < 1 ? 1 : (n_seed > 8 ? 8 : n_seed);
            for (int k = n_seed - 1; k >= 0; k--)
                stk.push(w, a + (b - a) * k / n_seed, (k + 1 == n_seed) ? b : a + (b - a) * (k + 1) / n_seed, 0);
        }
    }
    stk.seal();

    PerChan<double> big; // largest |panel value| seen in this step, accepted or not
    RB_FOR_CHAN(c, kEngChan)
    {
        result[c] = 0.0;
        big[c] = 0.0;
    }
    warp_fence();
    tile_clear<kHeyChan>(w, ws.outer.tile);
    int filled = 0;

    while (stk.sp > 0) {
        if (w.n_apply_lanes > kHeyAppBudget) {
            RB_FOR_CHAN(c, 2) { result[c] = NAN; }
            w.status |= kStatusCapHit;
            return;
        }
        double ta, tb;
        int tag;
        stk.pop(ta, tb, tag);
        const double tc = 0.5 * (ta + tb), thl = 0.5 * (tb - ta);
        warp_fence();
        // 7-point rule: narrow panels, and the steps far out whose contribution is already below
        // 1e-3 of the total (`light`): 1e-3 of that is far inside the tolerance
        const bool narrow = light || ((map == kMapLog || map == kMapNegLog) && (tb - ta) < 0.75);
        const int n_nodes = narrow ? 7 : 15;
        const double *rx = narrow ? GK7_X : GK15_X;
        const double *rwk = narrow ? GK7_WK : GK15_WK;
        const double *rwd = narrow ? GK7_WD : GK15_WD;
        if (n_nodes < filled) {
            tile_clear<kHeyChan>(w, ws.outer.tile);
            warp_fence();
        }
        filled = n_nodes;
#pragma unroll 1
        for (int j = 0; j < n_nodes; j++) {
            const double t = tc + thl * rx[j];
            double v = t, jac = 1.0;
            if (map == kMapSqrt) {
                v = offset + t * t;
                jac = 2.0 * t;
            } else if (map != kMapLinear) {
                jac = rb_exp(t);
                v = (map == kMapLog) ? jac : -jac;
            }
            if (hey_inner_integral<KIND>(w, cx, which, v, tile_col(j), rwk[j] * jac, rwd[j] * jac)) {
                // both channels NaN at this node: so is the panel, and with it the whole integral
                RB_FOR_CHAN(c, 2) { result[c] = NAN; }
                return;
            }
        }
        warp_fence();
        PerChan<double> r, e;
        tile_reduce<kHeyChan>(ws.outer.tile, 2, thl, r, e);

        PerChan<bool> ok;
        RB_FOR_CHAN(c, kEngChan) { ok[c] = true; }
        RB_FOR_CHAN(c, 2)
        {
            big[c] = fmax(big[c], fabs(r[c]));
            ok[c] = panel_ok(r[c], e[c], cx.epsrel_outer, fmax(fabs(scale[c]) + fabs(result[c]), big[c]));
        }
        bool accept = chan_all(ok, 2);
        // An outer panel that still fails kHeyOuterMaxDepth bisections below its seed sits next to
        // sigma = s, where the outer integrand behaves like |sigma - s|^(2 s - 1) (see kHeyRefDivergesV).
        // It is accepted as it is, with STATUS_CAP_HIT: the singularity is integrable and what is left
        // beyond 2^-13 of the seed is below the tolerance wherever the reference itself converges (round 1
        // declared such a panel divergent -> NaN; measured against the oracle that produced 290 NaNs on
        // 10 000 isotropic power-law points where the reference has a converged number).
        if (!accept && tag >= kHeyOuterMaxDepth) {
            w.status |= kStatusCapHit;
            accept = true;
        }
        if (accept || !stk.room(2) || panel_too_small(ta, tb) || w.n_apply_lanes > kAppBudget) {
            if (!accept && w.n_apply_lanes > kAppBudget)
                w.status |= kStatusCapHit; // (a panel at the bisection floor is an integrable end-point singularity)
            RB_FOR_CHAN(c, 2) { result[c] += r[c]; }
            // nothing left to integrate for once both coefficients are NaN
            PerChan<bool> dead;
            RB_FOR_CHAN(c, kEngChan) { dead[c] = true; }
            RB_FOR_CHAN(c, 2) { dead[c] = !(result[c] == result[c]); }
            if (chan_all(dead, 2))
                return;
        } else {
            stk.push(w, tc, tb, tag + 1);
            stk.push(w, ta, tc, tag + 1);
            stk.seal();
        }
    }
}

// d F / d v of the outer integrand at `v` (both channels), by a central difference.
template <int KIND>
RB_FN void hey_outer_derivative(Warp &w, const HeyFastCtx<KIND> &cx, int which, double v, PerChan<double> &deriv)
{
    HeyFastWS &ws = *cx.ws;
    warp_fence();
    tile_clear<kHeyChan>(w, ws.outer.tile);
    warp_fence();
    const double dv = kHeyDerivStep * fabs(v);
    hey_inner_integral<KIND>(w, cx, which, v - dv, tile_col(0), -0.5 / dv, 0.0);
    hey_inner_integral<KIND>(w, cx, which, v + dv, tile_col(1), 0.5 / dv, 0.0);
    warp_fence();
    PerChan<double> unused;
    tile_reduce<kHeyChan>(ws.outer.tile, 2, 1.0, deriv, unused);
}

// One outward-stepping stage of heyvaerts.rs:102-185 (cf. hey_step_outward<> in
// rb_heyvaerts.cuh, whose bookkeeping this follows with per-lane channel state).
template <int KIND>
RB_FN_NOINLINE void hey_march(Warp &w, const HeyFastCtx<KIND> &cx, int which, double edge, double delta, int dir,
                              bool skip_while_zero, double delta_cap, PerChan<double> &val, PerChan<bool> &alive)
{
    constexpr double kTol = 1e-5, kDeltaScale = 5.0;
    PerChan<bool> keep;
    PerChan<double> last; // the previous step's contribution
    RB_FOR_CHAN(c, kEngChan)
    {
        keep[c] = false;
        last[c] = INFINITY;
    }
    RB_FOR_CHAN(c, 2) { keep[c] = alive[c]; }

    for (int steps = 0;; steps++) {
        PerChan<bool> idle;
        RB_FOR_CHAN(c, kEngChan) { idle[c] = !keep[c]; }
        if (chan_all(idle, kEngChan))
            break;
        if (steps >= kHeyMaxSteps) {
            w.status |= kStatusCapHit;
            break;
        }

        // the step-size rule is voted by the channels that take part in it
        PerChan<bool> voter, none;
        RB_FOR_CHAN(c, kEngChan)
        {
            voter[c] = keep[c] && !(skip_while_zero && val[c] == 0.0);
            none[c] = !voter[c];
        }
        if (!chan_all(none, kEngChan)) {
            PerChan<double> deriv;
            hey_outer_derivative<KIND>(w, cx, which, edge, deriv);
            PerChan<bool> grow;
            RB_FOR_CHAN(c, kEngChan)
            {
                grow[c] = !voter[c] || deriv[c] == 0.0 || (fabs(1.0 / (deriv[c] * delta)) > kDeltaScale);
            }
            if (chan_all(grow, kEngChan) && delta < delta_cap)
                delta *= kDeltaScale;
        }

        const double lo = dir > 0 ? edge : edge - delta, hi = dir > 0 ? edge + delta : edge;
        // the QR outer integrand starts like sqrt(sigma - sigma_low) (pomega_max = 0 there):
        // the first QR step is integrated in t = sqrt(sigma - sigma_low)
        const int map = (which == kHeyQR && steps == 0) ? kMapSqrt
                                                       : ((lo > 0.0) ? kMapLog : ((hi < 0.0) ? kMapNegLog : kMapLinear));
        PerChan<bool> minor;
        RB_FOR_CHAN(c, kEngChan) { minor[c] = !keep[c] || fabs(last[c]) < kHeyLightStep * fabs(val[c]); }
        PerChan<double> contrib;
        hey_outer_integral<KIND>(w, cx, which, map, lo, hi, val, contrib, chan_all(minor, kEngChan));
        RB_FOR_CHAN(c, 2) { last[c] = contrib[c]; }

        RB_FOR_CHAN(c, 2)
        {
            if (keep[c]) {
                if (!(contrib[c] == contrib[c])) { // NaN: the reference returns NaN
                    val[c] = NAN;
                    alive[c] = false;
                    keep[c] = false;
                } else {
                    if (!(skip_while_zero && val[c] == 0.0)) {
                        if (!(fabs(contrib[c] / val[c]) > kTol))
                            keep[c] = false;
                    }
                    val[c] += contrib[c];
                }
            }
        }
        edge += dir * delta;
    }
}

// rho_Q and rho_V of one point, dimensionless (heyvaerts.rs:60-191).
template <int KIND>
RB_FN void heyvaerts_point_fast(Warp &w, const Dist &dist, double s, double theta, double epsrel_inner,
                                double epsrel_outer, HeyFastWS &ws, double (&out2)[2])
{
    static_assert(sizeof(HeyFastCtx<KIND>) <= sizeof(ws.ctx_store), "context store too small");
    warp_fence();
    HeyFastCtx<KIND> &cx = *reinterpret_cast<HeyFastCtx<KIND> *>(ws.ctx_store);
    ws.dist = dist; // every lane stores the same values
    cx.d = &ws.dist;
    cx.ws = &ws;
    cx.g.cos_th = cos(theta);
    cx.g.sin_th = sin(theta);
    cx.g.sigma0 = s * cx.g.sin_th;
    cx.g.sigma0_sq = cx.g.sigma0 * cx.g.sigma0;
    cx.epsrel_inner = epsrel_inner;
    cx.epsrel_outer = epsrel_outer;
    warp_fence();
    const double sigma0 = cx.g.sigma0;

    PerChan<bool> alive;
    PerChan<double> nr_val, qr_val;
    RB_FOR_CHAN(c, kEngChan)
    {
        alive[c] = false;
        nr_val[c] = 0.0;
        qr_val[c] = 0.0;
    }
    RB_FOR_CHAN(c, 2) { alive[c] = true; }
    const double div_q = hey_ref_diverges_q(KIND == kDistPowerLaw, cx.g.sin_th, cx.g.cos_th);
    const double div_v = (KIND == kDistPowerLaw) ? kHeyRefDivergesIsoV : kHeyRefDivergesV;
    // (the broken power law is PITCHY_PL with p = p1 near gamma = 1: the same rule, the same thresholds)
    if ((KIND == kDistPowerLaw || KIND == kDistPitchyPL || KIND == kDistPitchyBrokenPL) && dist.gamma_min == 1.0 &&
        s < div_v) {
        // the reference's NaN region (see kHeyRefDivergesQ)
        w.status |= kStatusRefDiverges;
        RB_FOR_CHAN(c, 2) { alive[c] = (c == 0) && !(s < div_q); }
        if (s < div_q) {
            out2[0] = NAN;
            out2[1] = NAN;
            return;
        }
    }

    // The QR part first (heyvaerts.rs:156-185; the two parts are independent sums): where the
    // calculation fails it is almost always here (the QR domain of a point with s <= 3 touches
    // gamma = 1), and a channel that is NaN needs no NR part.
    const double s15 = kInverseSqrt3 * sigma0 * sqrt(sigma0);
    const double sigma_low = sigma0 > s15 ? sigma0 : s15;
    hey_march<KIND>(w, cx, kHeyQR, sigma_low, sigma0, +1, true, 1e6 * sigma0, qr_val, alive);
    PerChan<bool> dead;
    RB_FOR_CHAN(c, kEngChan) { dead[c] = !alive[c]; }
    const bool skip_nr = chan_all(dead, kEngChan);

    // the central NR integral over [-3 sigma0, 3 sigma0] (heyvaerts.rs:97), cut at 0 and at
    // the edges of the empty region sigma_min <= 3
    if (!skip_nr) {
        const double p3 = 3.0 * sigma0;
        const double hole = (sigma0 < 3.0) ? sqrt(9.0 - cx.g.sigma0_sq) : 0.0;
        if (p3 > hole) {
            PerChan<double> part;
            hey_outer_integral<KIND>(w, cx, kHeyNR, kMapLinear, hole, p3, nr_val, part);
            RB_FOR_CHAN(c, 2) { nr_val[c] += part[c]; }
            hey_outer_integral<KIND>(w, cx, kHeyNR, kMapLinear, -p3, -hole, nr_val, part);
            RB_FOR_CHAN(c, 2) { nr_val[c] += part[c]; }
        }
        RB_FOR_CHAN(c, 2)
        {
            if (!(nr_val[c] == nr_val[c]))
                alive[c] = false;
        }
    }

    const double p3 = 3.0 * sigma0;
    hey_march<KIND>(w, cx, kHeyNR, p3, p3, +1, true, INFINITY, nr_val, alive);
    hey_march<KIND>(w, cx, kHeyNR, -p3, p3, -1, false, INFINITY, nr_val, alive);

    const double scale = 2.0 * kElectronCharge * kElectronCharge / (kMassElectron * (s * cx.g.sin_th) * (s * cx.g.sin_th));
    PerChan<double> total;
    RB_FOR_CHAN(c, kEngChan) { total[c] = NAN; }
    RB_FOR_CHAN(c, 2)
    {
        // a node that lands exactly on gamma = 1 makes the sum infinite: a failure like any other
        const double v = scale * (nr_val[c] + qr_val[c]);
        total[c] = (alive[c] && v - v == 0.0) ? v : NAN;
    }
    out2[0] = chan_get(total, 0);
    out2[1] = chan_get(total, 1);
}

} // namespace rb
