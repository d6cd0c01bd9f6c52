// rb_symphony.cuh -- emission and absorption coefficients (j_I/Q/V,
// alpha_I/Q/V) by the Symphony harmonic sum + (n, gamma) double integral.
//
// Replaces (reference file:line):
//   src/symphony.rs:66-187    CalculationState::compute
//   src/symphony.rs:196-295   n_integration
//   src/symphony.rs:312-389   gamma_integral
//   src/symphony.rs:398-479   gamma_integrand
//
// Two modes share all of the code below:
//   FUSED  (product default): one pass per point.  Every gamma node evaluates
//          J_n, J_{n+1}, f, df once and yields all six integrands; the gamma
//          range is split at gamma_peak so that the two Stokes-V lobes fall out
//          of the same nodes; the n integration carries eight accumulators.
//   !FUSED ("faithful"): eight passes, one integrand each, performing the same
//          sequence of rule applications as the reference does.  ~6-8x the work.
#pragma once

#include "rb_bessel.cuh"
#include "rb_core.cuh"
#include "rb_dist.cuh"

namespace rb {

// accumulator numbering: 0 j_I, 1 a_I, 2 j_Q, 3 a_Q, 4 j_V(+), 5 a_V(+), 6 j_V(-), 7 a_V(-)
constexpr int kSymNA = 8;

struct SymGeometry {
    double s;
    double cos_th, sin_th;
};

// Warp-uniform data of the current gamma integral; lives in shared memory so
// that it does not occupy registers across the node evaluation.
struct SymOrders {
    LeungOrder on, on1;
};

// All six gamma integrands at one node (symphony.rs:398-479), or one of them.
template <int KIND, int NV>
struct SymGammaIntegrand {
    const Dist *d;
    const SymGeometry *g;
    const SymOrders *ord;
    double n;
    int sel; // node value to produce when NV == 1

    RB_FN void eval(double gamma, double (&out)[NV]) const
    {
        const double s = g->s, costh = g->cos_th, sinth = g->sin_th;
        const double beta = sqrt(1.0 - 1.0 / (gamma * gamma));
        const double cos_xi = (s * gamma - n) / (s * gamma * beta * costh);
        const double sin_xi = sqrt(1.0 - cos_xi * cos_xi);
        const double m = (costh - beta * cos_xi) / sinth;
        const double big_n = beta * sin_xi;

        // gamma sin(xi), stabilised against cancellation at large gamma, n
        // (symphony.rs:430-437)
        double gamma_sin_xi;
        if (beta < 0.1) {
            gamma_sin_xi = gamma * sin_xi;
        } else {
            const double bc = beta * costh;
            const double beta2_costh2 = bc * bc;
            const double s_on_r = 2.0 * n / (s * (beta2_costh2 - 1.0));
            const double r = 1.0 - 1.0 / beta2_costh2;
            gamma_sin_xi = sqrt(r * (gamma * (gamma + s_on_r)) - (n * n / (s * s * beta2_costh2)));
        }

        const double z = s * beta * sinth * gamma_sin_xi;

        double jn, djn;
        leung_j_and_dj(ord->on, ord->on1, z, jn, djn);
        const double mj = m * jn;
        const double njp = big_n * djn;

        double f, dfdg, dfdcx;
        dist_eval<KIND>(*d, gamma, cos_xi, f, dfdg, dfdcx);
        const double dfdcx_factor = (beta * costh - cos_xi) / (gamma - 1.0 / gamma);
        const double f_abs = dfdg + dfdcx_factor * dfdcx;

        const double g2 = gamma * gamma;
        const double pol_i = mj * mj + njp * njp;
        const double pol_q = mj * mj - njp * njp;
        const double pol_v = 2.0 * mj * njp;

        if constexpr (NV == 6) {
            out[0] = g2 * pol_i * f;
            out[1] = g2 * pol_i * f_abs;
            out[2] = g2 * pol_q * f;
            out[3] = g2 * pol_q * f_abs;
            out[4] = g2 * pol_v * f;
            out[5] = g2 * pol_v * f_abs;
        } else {
            const double pol = (sel < 2) ? pol_i : (sel < 4 ? pol_q : pol_v);
            out[0] = g2 * pol * ((sel & 1) ? f_abs : f);
        }
    }
};

// G(n): the gamma integral at harmonic number n (symphony.rs:312-389) for all
// accumulators (FUSED) or for accumulator `sel` (faithful).
template <int KIND, bool FUSED>
struct SymGammaIntegral {
    static constexpr int NV = FUSED ? 6 : 1;
    static constexpr int NA = FUSED ? kSymNA : 1;

    const Dist *d;
    const SymGeometry *g;
    SymOrders *ord;
    IntervalList<NV> *list;
    unsigned want; // accumulators that must converge (FUSED)
    int sel;       // accumulator to compute (faithful)
    double epsrel; // relative tolerance of the gamma integral (reference: 1e-3)

    RB_MFN_NOINLINE void eval_collective(Warp &w, double n, double (&out)[NA])
    {
        const double s = g->s, costh = g->cos_th, sinth = g->sin_th;
        const double nos = n / s;
        const double root = sqrt(nos * nos - sinth * sinth);
        const double sin2 = sinth * sinth;
        const double gamma_minus = (nos - fabs(costh) * root) / sin2;
        const double gamma_plus = (nos + fabs(costh) * root) / sin2;
        const double gamma_peak = 0.5 * (gamma_plus + gamma_minus);
        const double rel_width = (s < 1e6) ? 1.0 : exp(-0.27 * log(n) - 0.1);
        const double gamma_minus_high = gamma_peak - (gamma_peak - gamma_minus) * rel_width;
        const double gamma_plus_high = gamma_peak - (gamma_peak - gamma_plus) * rel_width;

        warp_fence();
#ifdef RB_DEVICE_BUILD
        if (w.lane == 0)
#endif
        {
            leung_prepare(n, ord->on);
            leung_prepare(n + 1.0, ord->on1);
        }
        warp_fence();

        SymGammaIntegrand<KIND, NV> f{d, g, ord, n, 0};
        ApplyLanes<NV, SymGammaIntegrand<KIND, NV>> ap{f};

        if constexpr (FUSED) {
            const double bounds[3] = {gamma_minus_high, gamma_peak, gamma_plus_high};
            qag_joint<PolicySymphonySplit>(w, ap, 2, bounds, epsrel, *list, want, out);
        } else {
            f.sel = PolicySymphonySplit::val(sel);
            double bounds[2];
            if (sel < 4) {
                bounds[0] = gamma_minus_high;
                bounds[1] = gamma_plus_high;
            } else if (sel < 6) { // positive lobe
                bounds[0] = gamma_peak;
                bounds[1] = gamma_plus_high;
            } else {
                bounds[0] = gamma_minus_high;
                bounds[1] = gamma_peak;
            }
            qag_joint<PolicyPlain<1>>(w, ap, 1, bounds, epsrel, *list, 1u, out);
        }
    }
};

// The chunked adaptive integration over continuous n (symphony.rs:196-295).
// State of the chunk loop of symphony.rs:196-295 between two chunks: what the product path
// hands to the faithful sequence when its fidelity guard fires (rb_symfast.cuh).
struct SymChunkState {
    double n_start, delta_n, incr_step_factor;
    double ans, contrib;
};

template <int KIND, bool FUSED>
RB_FN void sym_n_integration(Warp &w, SymGammaIntegral<KIND, FUSED> &G, double n_start, unsigned want,
                             double epsrel_n, IntervalList<FUSED ? kSymNA : 1> &nlist,
                             double (&ans)[FUSED ? kSymNA : 1], const SymChunkState *resume = nullptr)
{
    constexpr int NA = FUSED ? kSymNA : 1;
    constexpr double kDerivTol = 1e-5, kTolerance = 1e5;
    double contrib[NA];
    double delta_n = 1e5, incr_step_factor = 10.0;
    unsigned active = want;

#pragma unroll
    for (int c = 0; c < NA; c++) {
        ans[c] = 0.0;
        contrib[c] = 0.0;
    }

    // "At low harmonic numbers, step conservatively since every n counts."
    if (G.g->s < 10.0) {
        delta_n = 1.0;
        incr_step_factor = 2.0;
    }
    if (resume) { // single-integrand (faithful) continuation
        n_start = resume->n_start;
        delta_n = resume->delta_n;
        incr_step_factor = resume->incr_step_factor;
        ans[0] = resume->ans;
        contrib[0] = resume->contrib;
    }

    ApplySeq<NA, SymGammaIntegral<KIND, FUSED>> ap{G};

    while (active) {
        G.want = active;

        double deriv[NA];
        deriv_central_joint<NA, !FUSED>(w, G, n_start, 1e-10 * n_start, deriv);

        // grow the step when every integral still being converged says so
        bool grow = true;
#pragma unroll
        for (int c = 0; c < NA; c++) {
            if (!((active >> c) & 1u))
                continue;
            const bool g_c = (deriv[c] == 0.0) || (contrib[c] != 0.0 && fabs(deriv[c] / contrib[c]) < kDerivTol);
            grow = grow && g_c;
        }
        if (grow)
            delta_n *= incr_step_factor;
        if (delta_n < n_start / incr_step_factor)
            delta_n *= incr_step_factor;

        const double bounds[2] = {n_start, n_start + delta_n};
        double chunk[NA];
        qag_joint<PolicyPlain<NA>>(w, ap, 1, bounds, epsrel_n, nlist, active, chunk);

#pragma unroll
        for (int c = 0; c < NA; c++) {
            if (!((active >> c) & 1u))
                continue;
            contrib[c] = chunk[c];
            ans[c] += chunk[c];
        }

        n_start += delta_n;
        if (n_start > 1e13)
            incr_step_factor = 1.0;

#pragma unroll
        for (int c = 0; c < NA; c++) {
            if (!((active >> c) & 1u))
                continue;
            // loop condition of the reference; a NaN contribution also ends it
            if (!(fabs(contrib[c]) >= fabs(ans[c] / kTolerance)))
                active &= ~(1u << c);
        }
    }
}

// Shared-memory working set of one warp for the Symphony kernel.
template <bool FUSED, int GAMMA_CAP, int N_CAP>
struct SymWorkspace {
    static constexpr int NVG = FUSED ? 6 : 1;
    static constexpr int NVN = FUSED ? kSymNA : 1;
    double gamma_store[GAMMA_CAP * IntervalList<NVG>::doubles_per_interval];
    double n_store[N_CAP * IntervalList<NVN>::doubles_per_interval];
    SymOrders orders;
};

// All six j/alpha coefficients of one point, dimensionless (the `s`-scaled
// form of compute_dimensionless, lib.rs:178-191).  out6 = j_I, a_I, j_Q, a_Q,
// j_V, a_V; lobes4 = j_V(+), j_V(-), a_V(+), a_V(-) with the prefactor applied.
template <int KIND, bool FUSED, int GAMMA_CAP, int N_CAP>
RB_FN void symphony_point(Warp &w, const Dist &dist, double s, double theta, double epsrel_gamma,
                          double epsrel_n, SymWorkspace<FUSED, GAMMA_CAP, N_CAP> &ws, double (&out6)[6],
                          double (&lobes4)[4])
{
    constexpr int NVG = FUSED ? 6 : 1;
    constexpr int NA = FUSED ? kSymNA : 1;
    constexpr double kNMax = 30.0;

    SymGeometry geom;
    geom.s = s;
    geom.cos_th = cos(theta);
    geom.sin_th = sin(theta);

    IntervalList<NVG> glist;
    glist.bind(ws.gamma_store, GAMMA_CAP);
    IntervalList<NA> nlist;
    nlist.bind(ws.n_store, N_CAP);

    SymGammaIntegral<KIND, FUSED> G{&dist, &geom, &ws.orders, &glist, FUSED ? 0xFFu : 1u, 0, epsrel_gamma};

    const double n_minus = s * fabs(geom.sin_th);
    const long long n_lo = (long long)(n_minus + 1.0);
    const long long n_hi = (long long)(n_minus + 1.0 + kNMax);
    const double n_start = floor(n_minus + 1.0 + kNMax);

    double total[kSymNA];

    constexpr int n_pass = FUSED ? 1 : kSymNA;
    for (int pass = 0; pass < n_pass; pass++) {
        double acc[NA];
#pragma unroll
        for (int c = 0; c < NA; c++)
            acc[c] = 0.0;
        G.sel = pass;
        G.want = FUSED ? 0xFFu : 1u;

        // the first 30 harmonics, discretely (symphony.rs:96-108)
        for (long long n = n_lo; n < n_hi; n++) {
            double gn[NA];
            G.eval_collective(w, (double)n, gn);
#pragma unroll
            for (int c = 0; c < NA; c++)
                acc[c] += gn[c];
        }

        // the rest, treating n as continuous (symphony.rs:124-140)
        unsigned want = 0;
#pragma unroll
        for (int c = 0; c < NA; c++)
            if (acc[c] - acc[c] == 0.0) // finite
                want |= 1u << c;

        double tail[NA];
        sym_n_integration<KIND, FUSED>(w, G, n_start, want, epsrel_n, nlist, tail);

#pragma unroll
        for (int c = 0; c < NA; c++) {
            const double v = ((want >> c) & 1u) ? acc[c] + tail[c] : NAN;
            total[FUSED ? c : pass] = (v - v == 0.0) ? v : NAN;
        }
    }

    // dimensional constants outside the integrals (symphony.rs:173-183)
    const double two_pi_e = kTwoPi * kElectronCharge;
    const double pre_j = two_pi_e * two_pi_e / (kSpeedLight * fabs(geom.cos_th));
    const double pre_a = -1.0 * two_pi_e * two_pi_e / (2.0 * kMassElectron * kSpeedLight * fabs(geom.cos_th));

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

// The faithful continuation of a point the product path handed over (rb_symfast.cuh, fidelity
// guard): `snap` is the chunk-loop state at the first chunk beyond n ~ 1e9 (layout kSnap* of
// rb_symfast.cuh: n_start, delta_n, incr, -, disc[8], tail[8], contrib[8], active mask).  Each
// accumulator that was still being integrated resumes the reference's own loop
// (symphony.rs:225-292) from there, on its own, with the reference's rule sequence.
template <int KIND, int GAMMA_CAP, int N_CAP>
RB_FN double symphony_tail_faithful_one(Warp &w, const Dist &dist, double s, double theta, double epsrel_gamma,
                                        double epsrel_n, SymWorkspace<false, GAMMA_CAP, N_CAP> &ws, const double *snap,
                                        int c)
{
    SymGeometry geom;
    geom.s = s;
    geom.cos_th = cos(theta);
    geom.sin_th = sin(theta);

    IntervalList<1> glist;
    glist.bind(ws.gamma_store, GAMMA_CAP);
    IntervalList<1> nlist;
    nlist.bind(ws.n_store, N_CAP);
    SymGammaIntegral<KIND, false> G{&dist, &geom, &ws.orders, &glist, 1u, 0, epsrel_gamma};

    const double disc = snap[4 + c];
    SymChunkState st{snap[0], snap[1], snap[2], snap[12 + c], snap[20 + c]};
    G.sel = c;
    G.want = 1u;
    double ans[1];
    sym_n_integration<KIND, false>(w, G, st.n_start, 1u, epsrel_n, nlist, ans, &st);
    const double v = disc + ans[0];
    return (v - v == 0.0) ? v : NAN;
}

// The eight accumulator totals -> the six coefficients and the four Stokes V lobes (symphony.rs:173-183)
RB_FN void symphony_tail_combine(double theta, const double (&total)[kSymNA], double (&out6)[6], double (&lobes4)[4])
{
    const double cos_th = cos(theta);
    const double two_pi_e = kTwoPi * kElectronCharge;
    const double pre_j = two_pi_e * two_pi_e / (kSpeedLight * fabs(cos_th));
    const double pre_a = -1.0 * two_pi_e * two_pi_e / (2.0 * kMassElectron * kSpeedLight * fabs(cos_th));
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

// All accumulators of a handed point one after the other (the host harness; the kernel gives each accumulator
// its own warp, k_symphony in rb_kernels.cuh).
template <int KIND, int GAMMA_CAP, int N_CAP>
RB_FN void symphony_tail_faithful(Warp &w, const Dist &dist, double s, double theta, double epsrel_gamma,
                                  double epsrel_n, SymWorkspace<false, GAMMA_CAP, N_CAP> &ws, const double *snap,
                                  double (&out6)[6], double (&lobes4)[4])
{
    const unsigned active = (unsigned)snap[28];
    double total[kSymNA];
    for (int c = 0; c < kSymNA; c++) {
        if ((active >> c) & 1u)
            total[c] = symphony_tail_faithful_one<KIND, GAMMA_CAP, N_CAP>(w, dist, s, theta, epsrel_gamma, epsrel_n, ws,
                                                                          snap, c);
        else
            total[c] = snap[4 + c] + snap[12 + c];
    }
    symphony_tail_combine(theta, total, out6, lobes4);
}

// ---------------------------------------------------------------------------
// The reference's diagnostics of the Symphony double integral (lib.rs:254-298), one value
// each: the integrand at (n, gamma), G(n), the QAG of G over [n_lo, n_hi], and the
// "other slicing", the sum over n at fixed gamma (symphony.rs:481-569).  Reference
// sequence of rule applications throughout (these exist to look inside the calculation).
enum { kDiagGammaIntegrand = 0, kDiagGammaIntegral = 1, kDiagNIntegral = 2, kDiagGammaContribution = 3 };

// gamma_integrand(gamma, n) as a function of n: the closure of symphony.rs:518, 536.
template <int KIND>
struct SymIntegrandOfN {
    const Dist *d;
    const SymGeometry *g;
    double gamma;
    int sel;

    RB_FN void eval(double n, double (&out)[1]) const
    {
        SymOrders ord;
        leung_prepare(n, ord.on);
        leung_prepare(n + 1.0, ord.on1);
        SymGammaIntegrand<KIND, 1> f{d, g, &ord, n, sel};
        f.eval(gamma, out);
    }
};

template <int KIND, int GAMMA_CAP, int N_CAP>
RB_FN double symphony_diagnostic(Warp &w, const Dist &dist, int coeff, int stokes, double s, double theta, int what,
                                 double a, double b, double epsrel_gamma, double epsrel_n,
                                 SymWorkspace<false, GAMMA_CAP, N_CAP> &ws)
{
    SymGeometry geom;
    geom.s = s;
    geom.cos_th = cos(theta);
    geom.sin_th = sin(theta);

    // CalculationState::new leaves the Stokes V switch on the negative lobe (symphony.rs:62),
    // and the diagnostics never move it: G(n) of Stokes V is the integral below gamma_peak.
    const int acc = (stokes == 2) ? 6 + coeff : 2 * stokes + coeff;
    const int sel = PolicySymphonySplit::val(acc);

    IntervalList<1> glist;
    glist.bind(ws.gamma_store, GAMMA_CAP);
    IntervalList<1> nlist;
    nlist.bind(ws.n_store, N_CAP);
    double out[1];

    if (what == kDiagGammaIntegrand) { // a = n, b = gamma (symphony.rs:585-590)
        SymIntegrandOfN<KIND> f{&dist, &geom, b, sel};
        f.eval(a, out);
        return out[0];
    }

    SymGammaIntegral<KIND, false> G{&dist, &geom, &ws.orders, &glist, 1u, acc, epsrel_gamma};
    if (what == kDiagGammaIntegral) { // a = n (symphony.rs:391-395)
        G.eval_collective(w, a, out);
        return out[0];
    }
    if (what == kDiagNIntegral) { // [a, b] = [n_lo, n_hi] (symphony.rs:297-307); Err -> NaN here
        ApplySeq<1, SymGammaIntegral<KIND, false>> ap{G};
        const double bounds[2] = {a, b};
        qag_joint<PolicyPlain<1>>(w, ap, 1, bounds, epsrel_n, nlist, 1u, out);
        return out[0];
    }

    // a = gamma (symphony.rs:491-569)
    const double gamma = a;
    const double delta = fabs(geom.cos_th) * sqrt(gamma * gamma - 1.0);
    const long long n_minus = (long long)(s * (gamma - delta) + 1.0);
    const long long n_plus = (long long)(s * (gamma + delta));
    constexpr long long kFullyDiscrete = 1000, kNDiscrete = 30;
    SymIntegrandOfN<KIND> f{&dist, &geom, gamma, sel};
    double ans = 0.0;
    if (n_plus - n_minus < kFullyDiscrete) {
        for (long long n = n_minus; n < n_plus + 1; n++) {
            f.eval((double)n, out);
            ans += out[0];
        }
    } else {
        for (long long n = n_minus; n < n_minus + kNDiscrete + 1; n++) {
            f.eval((double)n, out);
            ans += out[0];
        }
        ApplyLanes<1, SymIntegrandOfN<KIND>> ap{f};
        const double bounds[2] = {(double)(n_minus + kNDiscrete + 1), (double)n_plus};
        qag_joint<PolicyPlain<1>>(w, ap, 1, bounds, epsrel_n, glist, 1u, out);
        ans += out[0];
    }
    if (!(ans - ans == 0.0))
        return NAN;
    const double two_pi_e = kTwoPi * kElectronCharge;
    const double pre = (coeff == 0) ? two_pi_e * two_pi_e / (kSpeedLight * fabs(geom.cos_th))
                                    : -1.0 * two_pi_e * two_pi_e / (2.0 * kMassElectron * kSpeedLight * fabs(geom.cos_th));
    return ans * pre;
}

} // namespace rb
