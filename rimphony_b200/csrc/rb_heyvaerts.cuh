// rb_heyvaerts.cuh -- Faraday conversion (rho_Q, Heyvaerts' "h") and rotation
// (rho_V, "f") coefficients by the Heyvaerts et al. (2013) non-resonant (NR) +
// quasi-resonant (QR) double integrals in (sigma, pomega).
//
// Replaces (reference file:line):
//   src/heyvaerts.rs:60-191    compute_dimensionless / CalculationState::compute
//   src/heyvaerts.rs:194-201   fill_coord_vars
//   src/heyvaerts.rs:204-296   nr/qr outer integrals and integrands
//   src/heyvaerts.rs:302-468   h_qr, h_nr, f_qr, f_nr elements
//   src/heyvaerts.rs:472-493   dfdsigma
//
// FUSED: h and f share every node (coordinates, df/dsigma, the four I_{+-1/3},
// I_{+-2/3} or the J/Y pair) and are converged together.  !FUSED: one
// coefficient per pass with the reference's exact sequence of rule applications.
#pragma once

#include "rb_core.cuh"
#include "rb_dist.cuh"
#include "rb_special.cuh"

namespace rb {

constexpr double kFourOverSqrt27 = 0.769800358919501;
constexpr double kInverseC = 1.0 / kSpeedLight;
constexpr double kInverseSqrt3 = 0.5773502691896257;
constexpr double kSqrt8Over3 = 0.9428090415820635;
constexpr double kThreeTwoThirds = 2.080083823051904;
constexpr double kGApproximationCutoff = 10.0;
constexpr int kHeyMaxSteps = 400; // safety net for the outward stepping loops

struct HeyGeometry {
    double cos_th, sin_th;
    double sigma0, sigma0_sq;
};

// Heyvaerts coordinates of one node (heyvaerts.rs:194-201) and df/dsigma
// (heyvaerts.rs:472-493).
template <int KIND>
struct HeyNode {
    double sigma, pomega, x, dfds;

    // x_exact: the value of x when the caller knows it without cancellation (the product
    // path's pomega = pomega_max sin(phi) substitution); NaN = compute it as the reference does.
    RB_MFN_NOINLINE void fill(const Dist &d, const HeyGeometry &g, double sigma_, double pomega_, double x_exact = NAN)
    {
        sigma = sigma_;
        pomega = pomega_;
        x = (x_exact == x_exact) ? x_exact : rb_sqrt(sigma * sigma - pomega * pomega - g.sigma0_sq);
        const double t = g.sigma0 * g.sin_th;
        const double inv_t = rb_rcp(t);
        const double gamma = (sigma - pomega * g.cos_th) * inv_t;
        const double sq = rb_sqrt(gamma * gamma - 1.0); // gamma beta: also what dist_eval and d cos(xi) / d sigma need
        double mu = rb_div(sigma * g.cos_th - pomega, t * sq);

        // sin^2(xi) = 1 - mu^2 = x^2 sin^2(theta) / ((sigma - pomega cos(theta))^2 - t^2) identically.
        // Where the caller knows x without cancellation (the product path's substitutions) this
        // form is used: at the ends of the inner range, where mu -> +-1, the rounded mu reaches
        // exactly 1 (or beyond) a few 1e-6 of the range before the end, and the pitch-angle factor
        // sin^k(xi), d f / d cos(xi) ~ 1 / sin^2(xi) turn into 0/0 there.
        double sin2 = NAN;
        if (x_exact == x_exact) {
            const double q = sigma - pomega * g.cos_th;
            const double xs = x * g.sin_th;
            sin2 = rb_div(xs * xs, (q - t) * (q + t));
            if (sin2 <= 1.0) {
                const double mag = rb_sqrt(1.0 - sin2);
                if (fabs(mu) > mag || !(mu == mu))
                    mu = (sigma * g.cos_th - pomega < 0.0) ? -mag : mag;
            } else
                sin2 = NAN;
        }

        double f, dfdg, dfdcxi;
        dist_eval<KIND>(d, gamma, mu, f, dfdg, dfdcxi, sin2, sq);
        const double g_term = dfdg * inv_t;
        double mu_term = 0.0;
        if (dfdcxi != 0.0) {
            const double q = sigma - pomega * g.cos_th;
            const double r = pomega - sigma * g.cos_th;
            const double u = q * q - t * t;
            // sqrt(u) = sigma0 sin(theta) sqrt(gamma^2 - 1)
            const double dcxi_dsigma = rb_div(q * u * g.cos_th + u * r + r * t * t, u * (t * sq) * q);
            mu_term = dcxi_dsigma * dfdcxi;
        }
        dfds = g_term + mu_term;
    }
};

// NR elements (heyvaerts.rs:379-394 and 453-468); inner variable sigma.
template <int KIND, int NV>
struct HeyNRIntegrand {
    const Dist *d;
    const HeyGeometry *g;
    double pomega;
    int sel; // 0 = h (rho_Q), 1 = f (rho_V) when NV == 1

    RB_FN void eval(double sigma, double (&out)[NV], double x_exact = NAN) const
    {
        HeyNode<KIND> nd;
        nd.fill(*d, *g, sigma, pomega, x_exact);
        const double s_sq = sigma * sigma;
        const double x_sq = nd.x * nd.x;
        const double v = s_sq - x_sq;
        const double sv = rb_sqrt(v);
        // powers of 1 / rb_sqrt(v) from one reciprocal (the reference divides seven times, heyvaerts.rs:379-394)
        const double isv = rb_rcp(sv);
        const double iv = isv * isv, iv15 = iv * isv, iv2 = iv * iv, iv25 = iv2 * isv;
        const double ratio = s_sq * iv;
        const double a1 = 1.0 / 8.0 - 5.0 / 24.0 * ratio;
        const double a2 = 3.0 / 128.0 - 77.0 / 576.0 * ratio + 385.0 / 3456.0 * (ratio * ratio);
        const double xa1p = -5.0 / 12.0 * s_sq * x_sq * iv2;

        const double t1 = (6.0 * a2 - a1 * a1 + xa1p) * isv + a1 * x_sq * iv15 - x_sq * x_sq * iv25 * 0.125;
        const double t2 = (6.0 * a2 - a1 * a1) * iv15;
        const double u1 = 2.0 * t1 - g->sigma0_sq * t2;
        const double h = kPi * kInverseC * u1 * nd.dfds;

        const double z = 0.5 * x_sq * iv15 + (6.0 * a2 + xa1p - a1 * a1) * iv + 1.5 * a1 * x_sq * iv2;
        const double f = -2.0 * kPi * kInverseC * z * pomega * nd.dfds;

        if constexpr (NV == 2) {
            out[0] = h;
            out[1] = f;
        } else {
            out[0] = sel ? f : h;
        }
    }
};

// QR elements (heyvaerts.rs:302-373 and 400-447); inner variable pomega.
template <int KIND, int NV>
struct HeyQRIntegrand {
    const Dist *d;
    const HeyGeometry *g;
    double sigma;
    int sel;
    const JYOrder *jy = nullptr; // the J/Y orders of this sigma, prepared by the caller (product path), or none

    RB_FN void eval(double pomega, double (&out)[NV], double x_exact = NAN) const
    {
        HeyNode<KIND> nd;
        nd.fill(*d, *g, sigma, pomega, x_exact);
        const double x = nd.x;
        const double po_sq = pomega * pomega;
        const double smx = sigma - x;
        const double inv_x = rb_rcp(x);
        const double smxox = smx * inv_x;
        const double gg = kSqrt8Over3 * smx * rb_sqrt(smx * inv_x);

        double y_h1, y_h2, y_f;
        if (gg < kGApproximationCutoff) {
            double ip13, im13, ip23, im23;
            bessel_i_thirds(gg, ip13, im13, ip23, im23);
            y_h1 = kFourOverSqrt27 * smxox * smxox * (im23 - ip23) * (im23 + ip23);
            y_h2 = 0.5 * kFourOverSqrt27 * smxox * (im13 - ip13) * (im13 + ip13);
            y_f = kInverseSqrt3 * gg * (im23 - ip23) * (im13 + ip13);
        } else {
            double js, jsm1, ys, ysm1;
            if (jy != nullptr && jy->sigma == sigma)
                bessel_jy_pair_prepared(*jy, x, js, jsm1, ys, ysm1);
            else
                bessel_jy_pair(sigma, x, js, jsm1, ys, ysm1);
            const double jvp = jsm1 - sigma * js * inv_x;
            const double yvp = ysm1 - sigma * ys * inv_x;
            y_h1 = jvp * yvp;
            y_h2 = -js * ys;
            y_f = -x * jvp * ys;
        }

        const double t1 = kPi * kPi * x * x * y_h1;
        const double t2 = kPi * kPi * po_sq * y_h2;
        const double t3 = -kPi * rb_div(2.0 * po_sq + g->sigma0_sq, rb_sqrt(po_sq + g->sigma0_sq));
        const double h = kInverseC * (t1 + t2 + t3) * nd.dfds;
        const double f = -kTwoPi * kInverseC * pomega * (kPi * y_f - 1.0) * nd.dfds;

        if constexpr (NV == 2) {
            out[0] = h;
            out[1] = f;
        } else {
            out[0] = sel ? f : h;
        }
    }
};

// Outer integrands: an inner adaptive integral per outer node.
template <int KIND, int NV>
struct HeyNROuter {
    const Dist *d;
    const HeyGeometry *g;
    IntervalList<NV> *ilist;
    unsigned want;
    int sel;
    double epsrel;

    // heyvaerts.rs:213-250
    RB_MFN_NOINLINE void eval_collective(Warp &w, double pomega, double (&out)[NV])
    {
        const double sigma_min = sqrt(pomega * pomega + g->sigma0_sq);
        const double sigma_max = kInverseSqrt3 * sigma_min * sqrt(sigma_min);
        if (sigma_max <= sigma_min) {
#pragma unroll
            for (int c = 0; c < NV; c++)
                out[c] = 0.0;
            return;
        }
        HeyNRIntegrand<KIND, NV> f{d, g, pomega, sel};
        ApplyLanes<NV, HeyNRIntegrand<KIND, NV>> ap{f};
        const double bounds[2] = {sigma_min, sigma_max};
        qag_joint<PolicyPlain<NV>>(w, ap, 1, bounds, epsrel, *ilist, want, out);
    }
};

template <int KIND, int NV>
struct HeyQROuter {
    const Dist *d;
    const HeyGeometry *g;
    IntervalList<NV> *ilist;
    unsigned want;
    int sel;
    double epsrel;

    // heyvaerts.rs:262-296
    RB_MFN_NOINLINE void eval_collective(Warp &w, double sigma, double (&out)[NV])
    {
        const double pomega_max_phys = sqrt(kThreeTwoThirds * cbrt(sigma) * sigma - g->sigma0_sq);
        const double pomega_max_qr = sqrt(sigma * sigma - g->sigma0_sq);
        const double pomega_max = fmin(pomega_max_phys, pomega_max_qr);
        HeyQRIntegrand<KIND, NV> f{d, g, sigma, sel};
        ApplyLanes<NV, HeyQRIntegrand<KIND, NV>> ap{f};
        const double bounds[2] = {-pomega_max, pomega_max};
        qag_joint<PolicyPlain<NV>>(w, ap, 1, bounds, epsrel, *ilist, want, out);
    }
};

template <bool FUSED, int INNER_CAP, int OUTER_CAP>
struct HeyWorkspace {
    static constexpr int NV = FUSED ? 2 : 1;
    double inner_store[INNER_CAP * IntervalList<NV>::doubles_per_interval];
    double outer_store[OUTER_CAP * IntervalList<NV>::doubles_per_interval];
};

// One outward-stepping stage of heyvaerts.rs:102-185.
//   dir = +1: integrate [edge, edge + delta], dir = -1: [edge - delta, edge].
//   first_needs_value: the derivative probe and the relative-contribution test
//   are skipped while the running value is exactly zero (NR right side, QR).
template <int NV, bool REFINE, class Outer>
RB_FN_NOINLINE void hey_step_outward(Warp &w, Outer &F, IntervalList<NV> &olist, double epsrel_outer, double edge,
                            double delta, int dir, bool skip_while_zero, double delta_cap, double (&val)[NV],
                            unsigned &alive)
{
    constexpr double kTol = 1e-5, kDeltaScale = 5.0;
    ApplySeq<NV, Outer> ap{F};
    unsigned keep = alive;
    int steps = 0;

    while (keep) {
        if (++steps > kHeyMaxSteps) {
            w.status |= kStatusCapHit;
            break;
        }
        F.want = keep;

        unsigned voters = 0;
#pragma unroll
        for (int c = 0; c < NV; c++)
            if (((keep >> c) & 1u) && !(skip_while_zero && val[c] == 0.0))
                voters |= 1u << c;

        if (voters) {
            double rel_deriv[NV];
            deriv_central_joint<NV, REFINE>(w, F, edge, 1e-6, rel_deriv);
            bool grow = true;
#pragma unroll
            for (int c = 0; c < NV; c++) {
                if (!((voters >> c) & 1u))
                    continue;
                const bool g_c = (rel_deriv[c] == 0.0) || (fabs(1.0 / (rel_deriv[c] * delta)) > kDeltaScale);
                grow = grow && g_c;
            }
            if (grow && delta < delta_cap)
                delta *= kDeltaScale;
        }

        const double bounds[2] = {dir > 0 ? edge : edge - delta, dir > 0 ? edge + delta : edge};
        double contrib[NV];
        qag_joint<PolicyPlain<NV>>(w, ap, 1, bounds, epsrel_outer, olist, keep, contrib);

#pragma unroll
        for (int c = 0; c < NV; c++) {
            if (!((keep >> c) & 1u))
                continue;
            if (!(contrib[c] == contrib[c])) { // NaN: the reference returns NaN
                val[c] = NAN;
                alive &= ~(1u << c);
                keep &= ~(1u << c);
                continue;
            }
            if (!(skip_while_zero && val[c] == 0.0)) {
                if (!(fabs(contrib[c] / val[c]) > kTol))
                    keep &= ~(1u << c);
            }
            val[c] += contrib[c];
        }
        edge += dir * delta;
    }
}

// rho_Q and rho_V of one point, dimensionless (heyvaerts.rs:60-191).
template <int KIND, bool FUSED, int INNER_CAP, int OUTER_CAP>
RB_FN void heyvaerts_point(Warp &w, const Dist &dist, double s, double theta, double epsrel_inner,
                           double epsrel_outer, HeyWorkspace<FUSED, INNER_CAP, OUTER_CAP> &ws, double (&out2)[2])
{
    constexpr int NV = FUSED ? 2 : 1;
    HeyGeometry geom;
    geom.cos_th = cos(theta);
    geom.sin_th = sin(theta);
    geom.sigma0 = s * geom.sin_th;
    geom.sigma0_sq = geom.sigma0 * geom.sigma0;

    IntervalList<NV> ilist, olist;
    ilist.bind(ws.inner_store, INNER_CAP);
    olist.bind(ws.outer_store, OUTER_CAP);

    const unsigned all = FUSED ? 3u : 1u;
    const double scale = 2.0 * kElectronCharge * kElectronCharge /
                         (kMassElectron * (s * geom.sin_th) * (s * geom.sin_th));

    constexpr int n_pass = FUSED ? 1 : 2;
    for (int pass = 0; pass < n_pass; pass++) {
        HeyNROuter<KIND, NV> nr{&dist, &geom, &ilist, all, pass, epsrel_inner};
        HeyQROuter<KIND, NV> qr{&dist, &geom, &ilist, all, pass, epsrel_inner};
        unsigned alive = all;

        // initial NR integral over [-3 sigma0, 3 sigma0]
        double nr_val[NV];
        {
            ApplySeq<NV, HeyNROuter<KIND, NV>> ap{nr};
            const double bounds[2] = {-3.0 * geom.sigma0, 3.0 * geom.sigma0};
            qag_joint<PolicyPlain<NV>>(w, ap, 1, bounds, epsrel_outer, olist, all, nr_val);
#pragma unroll
            for (int c = 0; c < NV; c++)
                if (!(nr_val[c] == nr_val[c]))
                    alive &= ~(1u << c);
        }

        const double p3 = 3.0 * geom.sigma0;
        hey_step_outward<NV, !FUSED>(w, nr, olist, epsrel_outer, p3, p3, +1, true, INFINITY, nr_val, alive);
        hey_step_outward<NV, !FUSED>(w, nr, olist, epsrel_outer, -p3, p3, -1, false, INFINITY, nr_val, alive);

        double qr_val[NV];
#pragma unroll
        for (int c = 0; c < NV; c++)
            qr_val[c] = 0.0;
        const double s15 = kInverseSqrt3 * geom.sigma0 * sqrt(geom.sigma0);
        const double sigma_low = geom.sigma0 > s15 ? geom.sigma0 : s15;
        hey_step_outward<NV, !FUSED>(w, qr, olist, epsrel_outer, sigma_low, geom.sigma0, +1, true,
                                     1e6 * geom.sigma0, qr_val, alive);

#pragma unroll
        for (int c = 0; c < NV; c++) {
            const double v = ((alive >> c) & 1u) ? scale * (nr_val[c] + qr_val[c]) : NAN;
            out2[FUSED ? c : pass] = v;
        }
    }
}

} // namespace rb
