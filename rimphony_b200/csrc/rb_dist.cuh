// rb_dist.cuh -- the electron distribution functions and their normalisation
// ("full_calculation") as device code.
//
// Replaces (reference file:line):
//   src/power_law.rs:36-62, 93-103         PowerLawDistribution
//   src/thermal_juettner.rs:29-39, 56-64   ThermalJuettnerDistribution
//   src/pitchy_pl.rs:32-64, 95-115         PitchyPowerLawDistribution
//   src/pitchy_kappa.rs:38-62, 90-125      PitchyKappaDistribution
// and a pitchy broken power law built the way src/pitchy_pl.rs builds its single one.
//
// f, df/dgamma and df/dcos(xi) are produced together: they share one rb_exp() and
// one or two rb_log() per call (gamma^-p rb_exp(-gamma/gc) sin^k(xi) is evaluated as a
// single exponential), instead of the reference's separate powf/exp per term.
#pragma once

#include "rb_core.cuh"

namespace rb {

// numbering shared with include/rimphony_b200.h
enum { kDistPowerLaw = 0, kDistThermalJuettner = 1, kDistPitchyPL = 2, kDistPitchyKappa = 3, kDistPitchyBrokenPL = 4 };

struct Dist {
    double p, k; // p: the index below the break for PITCHY_BROKEN_PL
    double gamma_min, gamma_max, inv_gamma_cutoff;
    double kappa, width, inv_kappa_width;
    double neg_inverse_t;
    double norm;
};

// PITCHY_BROKEN_PL keeps p2, gamma_break and (p2 - p1) ln(gamma_break) in the kappa fields, which it does not
// use.  (Named fields in a union there would change how the other kinds' kernels compile.)
RB_HD double bpl_p2(const Dist &d) { return d.kappa; }
RB_HD double bpl_gamma_break(const Dist &d) { return d.width; }
RB_HD double bpl_log_offset(const Dist &d) { return d.inv_kappa_width; }

// Fill `d` from the C-ABI parameter vector of one point (see the header for
// the order); `norm` is left NaN until dist_normalize<>() has run.
template <int KIND>
RB_HD bool dist_from_params(const double *pv, int n_params, Dist &d)
{
    d.p = d.k = d.kappa = d.width = d.inv_kappa_width = d.neg_inverse_t = 0.0;
    d.gamma_min = 1.0;
    d.gamma_max = 1e12;
    d.inv_gamma_cutoff = 1e-10;
    d.norm = NAN;
    if (KIND == kDistPowerLaw) {
        if (n_params != 1 && n_params != 4)
            return false;
        d.p = pv[0];
        if (n_params == 4) {
            d.gamma_min = pv[1];
            d.gamma_max = pv[2];
            d.inv_gamma_cutoff = 1.0 / pv[3];
        }
    } else if (KIND == kDistThermalJuettner) {
        if (n_params != 1)
            return false;
        d.neg_inverse_t = -1.0 / pv[0];
    } else if (KIND == kDistPitchyPL) {
        if (n_params != 2 && n_params != 5)
            return false;
        d.p = pv[0];
        d.k = pv[1];
        if (n_params == 5) {
            d.gamma_min = pv[2];
            d.gamma_max = pv[3];
            d.inv_gamma_cutoff = 1.0 / pv[4];
        }
    } else if (KIND == kDistPitchyBrokenPL) {
        if (n_params != 4 && n_params != 7)
            return false;
        d.p = pv[0];
        d.kappa = pv[1];                          // bpl_p2
        d.width = pv[2];                          // bpl_gamma_break
        d.inv_kappa_width = (pv[1] - pv[0]) * log(pv[2]); // bpl_log_offset
        d.k = pv[3];
        if (n_params == 7) {
            d.gamma_min = pv[4];
            d.gamma_max = pv[5];
            d.inv_gamma_cutoff = 1.0 / pv[6];
        }
    } else {
        if (n_params != 3 && n_params != 4)
            return false;
        d.kappa = pv[0];
        d.width = pv[1];
        d.inv_kappa_width = 1.0 / (pv[0] * pv[1]);
        d.k = pv[2];
        if (n_params == 4)
            d.inv_gamma_cutoff = 1.0 / pv[3];
    }
    return true;
}

// sin^k(xi) given sin^2(xi); pow(x, 0) = 1 for every x including NaN.
RB_FN double log_pitch_term(double k, double sin2)
{
    return (k == 0.0) ? 0.0 : 0.5 * k * rb_log(sin2);
}

// calc_f and calc_f_derivatives in one go.  `sin2_exact`: sin^2(xi) when the caller knows it
// without the cancellation of 1 - cos^2 (the Heyvaerts product path, where |cos xi| -> 1 at the
// ends of the inner range and the rounded 1 - cos^2 turns into 0 or a negative number); NaN =
// compute it from cos_xi as the reference does.  `sqrt_g2m1`: sqrt(gamma^2 - 1) when the caller has it already.
template <int KIND>
RB_FN void dist_eval(const Dist &d, double gamma, double cos_xi, double &f, double &dfdg, double &dfdcx,
                     double sin2_exact = NAN, double sqrt_g2m1 = NAN)
{
    if (KIND == kDistPowerLaw) {
        if (gamma < d.gamma_min || gamma > d.gamma_max) {
            f = dfdg = dfdcx = 0.0;
            return;
        }
        const double g2m1 = gamma * gamma - 1.0;
        // norm gamma^-p rb_exp(-gamma/gc) / (gamma^2 beta),  gamma^2 beta = gamma rb_sqrt(gamma^2 - 1)
        const double sq = (sqrt_g2m1 == sqrt_g2m1) ? sqrt_g2m1 : rb_sqrt(g2m1);
        const double inv = rb_rcp(gamma * sq); // 1 / (gamma^2 beta); 1 / gamma = inv sq, 1 / (gamma^2 - 1) = (inv gamma)^2
        const double ig = inv * gamma;
        f = d.norm * rb_exp(-d.p * rb_log(gamma) - gamma * d.inv_gamma_cutoff) * inv;
        dfdg = -f * ((d.p + 1.0) * (inv * sq) + gamma * (ig * ig) + d.inv_gamma_cutoff);
        dfdcx = 0.0;
    } else if (KIND == kDistThermalJuettner) {
        f = d.norm * rb_exp(d.neg_inverse_t * gamma);
        dfdg = f * d.neg_inverse_t;
        dfdcx = 0.0;
    } else if (KIND == kDistPitchyPL) {
        if (gamma < d.gamma_min || gamma > d.gamma_max) {
            f = dfdg = dfdcx = 0.0;
            return;
        }
        const double sin2 = (sin2_exact == sin2_exact) ? sin2_exact : 1.0 - cos_xi * cos_xi;
        const double g2m1 = gamma * gamma - 1.0;
        const double sq = (sqrt_g2m1 == sqrt_g2m1) ? sqrt_g2m1 : rb_sqrt(g2m1);
        const double inv = rb_rcp(gamma * sq); // 1 / (gamma^2 beta); 1 / gamma = inv sq, 1 / (gamma^2 - 1) = (inv gamma)^2
        const double ig = inv * gamma;
        f = d.norm * rb_exp(log_pitch_term(d.k, sin2) - d.p * rb_log(gamma) - gamma * d.inv_gamma_cutoff) * inv;
        dfdg = -f * ((d.p + 1.0) * (inv * sq) + gamma * (ig * ig) + d.inv_gamma_cutoff);
        dfdcx = -f * d.k * rb_div(cos_xi, sin2);
    } else if (KIND == kDistPitchyBrokenPL) {
        if (gamma < d.gamma_min || gamma > d.gamma_max) {
            f = dfdg = dfdcx = 0.0;
            return;
        }
        // PITCHY_PL with gamma^-p1 below the break and gamma_break^(p2 - p1) gamma^-p2 from it on
        const bool upper = !(gamma < bpl_gamma_break(d));
        const double p = upper ? bpl_p2(d) : d.p;
        const double sin2 = (sin2_exact == sin2_exact) ? sin2_exact : 1.0 - cos_xi * cos_xi;
        const double g2m1 = gamma * gamma - 1.0;
        const double sq = (sqrt_g2m1 == sqrt_g2m1) ? sqrt_g2m1 : rb_sqrt(g2m1);
        const double inv = rb_rcp(gamma * sq);
        const double ig = inv * gamma;
        f = d.norm *
            rb_exp(log_pitch_term(d.k, sin2) + (upper ? bpl_log_offset(d) : 0.0) - p * rb_log(gamma) -
                   gamma * d.inv_gamma_cutoff) *
            inv;
        dfdg = -f * ((p + 1.0) * (inv * sq) + gamma * (ig * ig) + d.inv_gamma_cutoff);
        dfdcx = -f * d.k * rb_div(cos_xi, sin2);
    } else {
        const double sin2 = (sin2_exact == sin2_exact) ? sin2_exact : 1.0 - cos_xi * cos_xi;
        f = d.norm * rb_exp(log_pitch_term(d.k, sin2) -
                         (d.kappa + 1.0) * rb_log(1.0 + (gamma - 1.0) * d.inv_kappa_width) -
                         gamma * d.inv_gamma_cutoff);
        dfdg = -f * (rb_div(d.kappa + 1.0, d.kappa * d.width + gamma - 1.0) + d.inv_gamma_cutoff);
        dfdcx = -f * d.k * rb_div(cos_xi, sin2);
    }
}

// --- normalisation ---------------------------------------------------------

struct PLNormIntegrand {
    double p, inv_gamma_cutoff;
    RB_FN void eval(double g, double (&out)[1]) const { out[0] = rb_exp(-p * rb_log(g) - g * inv_gamma_cutoff); }
};

struct BrokenPLNormIntegrand {
    double p1, p2, gamma_break, log_offset, inv_gamma_cutoff;
    RB_FN void eval(double g, double (&out)[1]) const
    {
        const bool upper = !(g < gamma_break);
        out[0] = rb_exp((upper ? log_offset : 0.0) - (upper ? p2 : p1) * rb_log(g) - g * inv_gamma_cutoff);
    }
};

struct KappaNormIntegrand {
    double kappa, inv_kappa_width, inv_gamma_cutoff;
    RB_FN void eval(double g, double (&out)[1]) const
    {
        out[0] = g * sqrt(g * g - 1.0) *
                 rb_exp(-(kappa + 1.0) * rb_log(1.0 + (g - 1.0) * inv_kappa_width) - g * inv_gamma_cutoff);
    }
};

// 2F1(1/2, -k/2; 3/2; 1) = (sqrt(pi)/2) Gamma(1 + k/2) / Gamma(3/2 + k/2)
// (what gsl_sf_hyperg_2F1 returns at x = 1; pitchy_pl.rs:98, pitchy_kappa.rs:93).
RB_FN double pitch_angle_integral(double k)
{
    return 0.886226925452758013649083741670573 * rb_exp(lgamma(1.0 + 0.5 * k) - lgamma(1.5 + 0.5 * k));
}

// int_1^inf g sqrt(g^2-1) rb_exp(-g/T) dg = T K_2(1/T), with K_2 from the
// trapezoid rule on int_0^inf rb_exp(-z cosh t) cosh 2t dt (lanes split the
// abscissae).  The reference uses QAGIU with epsrel 1e-5
// (thermal_juettner.rs:56-64); the closed form is what that converges to.
RB_FN double juettner_gamma_integral(const Warp &w, double t)
{
    const double z = 1.0 / t;
    const double h = 0.0625;
    double sum = 0.0;
#ifdef RB_DEVICE_BUILD
    for (int i = w.lane; i < 4000; i += 32) {
        const double tt = i * h;
        const double arg = z * cosh(tt);
        const bool live = arg <= 745.0;
        if (live)
            sum += ((i == 0) ? 0.5 : 1.0) * rb_exp(-arg) * cosh(2.0 * tt);
        if (__all_sync(0xffffffffu, !live))
            break;
    }
    sum = warp_sum(sum);
#else
    (void)w;
    for (int i = 0; i < 4000; i++) {
        const double tt = i * h;
        const double arg = z * cosh(tt);
        if (arg > 745.0)
            break;
        sum += ((i == 0) ? 0.5 : 1.0) * rb_exp(-arg) * cosh(2.0 * tt);
    }
#endif
    return t * sum * h;
}

// full_calculation(): computes d.norm.  `list` is scratch for one
// single-integrand interval list.  Returns false if the integral failed (the
// reference `unwrap()`s, i.e. panics; we report status and leave norm NaN).
template <int KIND>
RB_FN bool dist_normalize(Warp &w, Dist &d, double t_juettner, IntervalList<1> &list)
{
    double integral[1];
    if (KIND == kDistThermalJuettner) {
        integral[0] = juettner_gamma_integral(w, t_juettner);
        d.norm = 1.0 / (2.0 * kTwoPi * integral[0]);
        return integral[0] == integral[0];
    }
    double pa = 1.0;
    if (KIND == kDistPowerLaw || KIND == kDistPitchyPL) {
        PLNormIntegrand f{d.p, d.inv_gamma_cutoff};
        ApplyLanes<1, PLNormIntegrand> ap{f};
        const double bounds[2] = {d.gamma_min, d.gamma_max};
        qag_joint<PolicyPlain<1>>(w, ap, 1, bounds, 1e-8, list, 1u, integral);
        if (KIND == kDistPitchyPL)
            pa = pitch_angle_integral(d.k);
    } else if (KIND == kDistPitchyBrokenPL) {
        // one QAG over the whole range, no split at the break: what the reference's
        // full_calculation (pitchy_pl.rs:95-112) does with this gamma term
        BrokenPLNormIntegrand f{d.p, bpl_p2(d), bpl_gamma_break(d), bpl_log_offset(d), d.inv_gamma_cutoff};
        ApplyLanes<1, BrokenPLNormIntegrand> ap{f};
        const double bounds[2] = {d.gamma_min, d.gamma_max};
        qag_joint<PolicyPlain<1>>(w, ap, 1, bounds, 1e-8, list, 1u, integral);
        pa = pitch_angle_integral(d.k);
    } else {
        KappaNormIntegrand f{d.kappa, d.inv_kappa_width, d.inv_gamma_cutoff};
        ApplyLanes<1, KappaNormIntegrand> ap{f};
        const double bounds[2] = {1.0, 1e3 * (1.0 / d.inv_gamma_cutoff)};
        qag_joint<PolicyPlain<1>>(w, ap, 1, bounds, 1e-8, list, 1u, integral);
        pa = pitch_angle_integral(d.k);
    }
    d.norm = 1.0 / (2.0 * kTwoPi * pa * integral[0]);
    return integral[0] == integral[0];
}

} // namespace rb
