/* oracle/rimphony_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement of rimphony's hot path: all eight polarized synchrotron
 * transfer coefficients for one (s, theta, distribution) point, with exactly
 * the control flow of the reference:
 *
 *   src/lib.rs:163-191, 236-247      dispatch, output order, cgs scaling
 *   src/symphony.rs:66-187           harmonic sum + n integration + prefactor
 *   src/symphony.rs:196-295          n_integration (chunked adaptive)
 *   src/symphony.rs:312-389          gamma_integral
 *   src/symphony.rs:398-479          gamma_integrand
 *   src/heyvaerts.rs:81-191          NR + QR outer stepping
 *   src/heyvaerts.rs:194-296         coordinates, nested integrals
 *   src/heyvaerts.rs:302-493         elements + df/dsigma
 *   src/power_law.rs:36-62, 93-103   src/pitchy_pl.rs:32-64, 95-115
 *   src/pitchy_kappa.rs:38-62, 90-125  src/thermal_juettner.rs:29-39, 56-64
 *
 * The Bessel functions J_n, J_n' are NOT restated here: they are the
 * reference's own leung-bessel/src/bessel.c, compiled in place into
 * oracle/_ref/ by oracle/Makefile (pkgw_bessel_j, pkgw_bessel_dj), or, where
 * that file is not at hand, its restatement leung_bessel.c.  GSL QAG /
 * deriv_central are restated in gsl_restated.h, Cephes-backed special
 * functions in special.h.
 *
 * This file is the checker (tests/, smoke(), bench.py cpu_baseline and
 * --impl reference).  The product (rimphony_b200/) never links or loads it.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifdef _OPENMP
#include <omp.h>
#endif

#include "gsl_restated.h"
#include "special.h"
#include "rimphony_oracle.h"

/* The reference's native component (leung-bessel/src/bessel.c:318-405). */
extern double pkgw_bessel_j(double n, double x);
extern double pkgw_bessel_dj(double n, double x);

/* src/lib.rs:55-67 */
#define ORC_PI 3.14159265358979323846264338327950288
#define ORC_TWO_PI (2. * ORC_PI)
#define ORC_MASS_ELECTRON 9.1093826e-28
#define ORC_SPEED_LIGHT 2.99792458e10
#define ORC_ELECTRON_CHARGE 4.80320680e-10

#define ORC_MAXV(a, b) ((a) > (b) ? (a) : (b))

/* The reference passes epsrel = 1e-3 to every QAG call of this path (src/gsl.rs:169-180 through
 * symphony.rs:327,251 and heyvaerts.rs:98,225,278).  These two are that constant.  They can be
 * changed ONLY for the stability study of tests/golden/make_stability.py, which asks how far the
 * reference's own output moves when its own tolerance is tightened (where it moves by more than
 * 1e-3 the reference value is not defined to 1e-3).  Set before a batch, never during one. */
static double g_sym_epsrel = 1e-3;
static double g_hey_epsrel = 1e-3;

static int g_trace_hey_outer = 0;
void orc_set_trace(int heyvaerts_outer) { g_trace_hey_outer = heyvaerts_outer; }

void orc_set_epsrel(double symphony_epsrel, double heyvaerts_epsrel)
{
    g_sym_epsrel = symphony_epsrel > 0. ? symphony_epsrel : 1e-3;
    g_hey_epsrel = heyvaerts_epsrel > 0. ? heyvaerts_epsrel : 1e-3;
}

/* ------------------------------------------------------------------------- */
/* Distribution functions                                                     */

static double pl_gamma_norm_integrand(double g, void *ctx)
{
    const orc_dist *d = (const orc_dist *)ctx;
    return pow(g, -d->p) * exp(-g * d->inv_gamma_cutoff);
}

static double kappa_gamma_norm_integrand(double g, void *ctx)
{
    const orc_dist *d = (const orc_dist *)ctx;
    return g * sqrt(g * g - 1.) * pow(1. + (g - 1.) * d->inv_kappa_width, -(d->kappa + 1.)) *
           exp(-g * d->inv_gamma_cutoff);
}

int orc_dist_init(orc_dist *d, int kind, const double *params, int n_params)
{
    orc_workspace *ws;
    double integral = NAN, abserr;
    int status = 0;

    memset(d, 0, sizeof(*d));
    d->kind = kind;
    d->norm = NAN;
    d->gamma_min = 1.;
    d->gamma_max = 1e12;
    d->inv_gamma_cutoff = 1e-10;

    ws = (orc_workspace *)malloc(sizeof(orc_workspace));
    orc_workspace_init(ws, 1000);

    switch (kind) {
    case ORC_DIST_POWER_LAW:
        /* params: p [, gamma_min, gamma_max, gamma_cutoff] (power_law.rs:71-87) */
        if (n_params != 1 && n_params != 4) {
            status = -1;
            break;
        }
        d->p = params[0];
        if (n_params == 4) {
            d->gamma_min = params[1];
            d->gamma_max = params[2];
            d->inv_gamma_cutoff = 1. / params[3];
        }
        /* power_law.rs:93-103 */
        status = orc_qag31(pl_gamma_norm_integrand, d, d->gamma_min, d->gamma_max, 0., 1e-8, ws,
                           &integral, &abserr);
        d->norm = 1. / (2. * ORC_TWO_PI * integral);
        break;

    case ORC_DIST_THERMAL_JUETTNER:
        /* params: T (thermal_juettner.rs:45-50) */
        if (n_params != 1) {
            status = -1;
            break;
        }
        d->neg_inverse_t = -1. / params[0];
        /* thermal_juettner.rs:56-64: int_1^inf g sqrt(g^2-1) exp(-g/T) dg,
         * by QAGIU(epsrel 1e-5) in the reference; = T K_2(1/T) exactly. */
        integral = params[0] * orc_bessel_k2(1. / params[0]);
        d->norm = 1. / (2. * ORC_TWO_PI * integral);
        break;

    case ORC_DIST_PITCHY_PL:
        /* params: p, k [, gamma_min, gamma_max, gamma_cutoff] (pitchy_pl.rs:73-90) */
        if (n_params != 2 && n_params != 5) {
            status = -1;
            break;
        }
        d->p = params[0];
        d->k = params[1];
        if (n_params == 5) {
            d->gamma_min = params[2];
            d->gamma_max = params[3];
            d->inv_gamma_cutoff = 1. / params[4];
        }
        /* pitchy_pl.rs:95-112 */
        status = orc_qag31(pl_gamma_norm_integrand, d, d->gamma_min, d->gamma_max, 0., 1e-8, ws,
                           &integral, &abserr);
        d->norm = 1. / (2. * ORC_TWO_PI * orc_pitch_angle_integral(d->k) * integral);
        break;

    case ORC_DIST_PITCHY_KAPPA:
        /* params: kappa, width, k [, gamma_cutoff] (pitchy_kappa.rs:70-85) */
        if (n_params != 3 && n_params != 4) {
            status = -1;
            break;
        }
        d->kappa = params[0];
        d->width = params[1];
        d->inv_kappa_width = 1. / (params[0] * params[1]);
        d->k = params[2];
        if (n_params == 4)
            d->inv_gamma_cutoff = 1. / params[3];
        /* pitchy_kappa.rs:90-121 */
        status = orc_qag31(kappa_gamma_norm_integrand, d, 1., 1e3 * (1. / d->inv_gamma_cutoff), 0.,
                           1e-8, ws, &integral, &abserr);
        d->norm = 1. / (2. * ORC_TWO_PI * orc_pitch_angle_integral(d->k) * integral);
        break;

    default:
        status = -1;
    }

    free(ws);
    /* the reference `unwrap()`s the normalisation integral, i.e. panics; the
     * oracle reports a nonzero status and a NaN norm instead. */
    if (status != 0)
        d->norm = NAN;
    return status;
}

double orc_calc_f(const orc_dist *d, double gamma, double cos_xi)
{
    switch (d->kind) {
    case ORC_DIST_POWER_LAW: {
        /* power_law.rs:37-46 */
        double beta;
        if (gamma < d->gamma_min || gamma > d->gamma_max)
            return 0.;
        beta = sqrt(1. - 1. / (gamma * gamma));
        return d->norm * pow(gamma, -d->p) * exp(-gamma * d->inv_gamma_cutoff) /
               (gamma * gamma * beta);
    }
    case ORC_DIST_THERMAL_JUETTNER:
        /* thermal_juettner.rs:30-32 */
        return d->norm * exp(d->neg_inverse_t * gamma);
    case ORC_DIST_PITCHY_PL: {
        /* pitchy_pl.rs:33-45 */
        double sin_xi, pa_term, beta, gamma_term;
        if (gamma < d->gamma_min || gamma > d->gamma_max)
            return 0.;
        sin_xi = sqrt(1. - cos_xi * cos_xi);
        pa_term = pow(sin_xi, d->k);
        beta = sqrt(1. - 1. / (gamma * gamma));
        gamma_term = pow(gamma, -d->p) * exp(-gamma * d->inv_gamma_cutoff);
        return d->norm * pa_term * gamma_term / (gamma * gamma * beta);
    }
    case ORC_DIST_PITCHY_KAPPA: {
        /* pitchy_kappa.rs:39-47 */
        double sin_xi = sqrt(1. - cos_xi * cos_xi);
        double pa_term = pow(sin_xi, d->k);
        double gamma_term = pow(1. + (gamma - 1.) * d->inv_kappa_width, -(d->kappa + 1.)) *
                            exp(-gamma * d->inv_gamma_cutoff);
        return d->norm * pa_term * gamma_term;
    }
    }
    return NAN;
}

void orc_calc_f_derivatives(const orc_dist *d, double gamma, double cos_xi, double *dfdg,
                            double *dfdcx)
{
    switch (d->kind) {
    case ORC_DIST_POWER_LAW: {
        /* power_law.rs:48-61 */
        double p_plus_1, g2_minus_1;
        if (gamma < d->gamma_min || gamma > d->gamma_max) {
            *dfdg = 0.;
            *dfdcx = 0.;
            return;
        }
        p_plus_1 = d->p + 1.;
        g2_minus_1 = gamma * gamma - 1.;
        *dfdg = -d->norm * pow(gamma, -p_plus_1) / sqrt(g2_minus_1) *
                exp(-gamma * d->inv_gamma_cutoff) *
                (p_plus_1 / gamma + gamma / g2_minus_1 + d->inv_gamma_cutoff);
        *dfdcx = 0.;
        return;
    }
    case ORC_DIST_THERMAL_JUETTNER:
        /* thermal_juettner.rs:34-38 */
        *dfdg = d->norm * exp(d->neg_inverse_t * gamma) * d->neg_inverse_t;
        *dfdcx = 0.;
        return;
    case ORC_DIST_PITCHY_PL: {
        /* pitchy_pl.rs:47-63 */
        double sin_xi, pa_term, beta, gamma_term, f;
        if (gamma < d->gamma_min || gamma > d->gamma_max) {
            *dfdg = 0.;
            *dfdcx = 0.;
            return;
        }
        sin_xi = sqrt(1. - cos_xi * cos_xi);
        pa_term = pow(sin_xi, d->k);
        beta = sqrt(1. - 1. / (gamma * gamma));
        gamma_term = pow(gamma, -d->p) * exp(-gamma * d->inv_gamma_cutoff);
        f = d->norm * pa_term * gamma_term / (gamma * gamma * beta);
        *dfdg = -f * ((d->p + 1.) / gamma + gamma / (gamma * gamma - 1.) + d->inv_gamma_cutoff);
        *dfdcx = -f * d->k * cos_xi / (sin_xi * sin_xi);
        return;
    }
    case ORC_DIST_PITCHY_KAPPA: {
        /* pitchy_kappa.rs:49-61 */
        double sin_xi = sqrt(1. - cos_xi * cos_xi);
        double pa_term = pow(sin_xi, d->k);
        double gamma_term = pow(1. + (gamma - 1.) * d->inv_kappa_width, -(d->kappa + 1.)) *
                            exp(-gamma * d->inv_gamma_cutoff);
        double f = d->norm * pa_term * gamma_term;
        *dfdg = -f * ((d->kappa + 1.) / (d->kappa * d->width + gamma - 1.) + d->inv_gamma_cutoff);
        *dfdcx = -f * d->k * cos_xi / (sin_xi * sin_xi);
        return;
    }
    }
    *dfdg = NAN;
    *dfdcx = NAN;
}

/* ------------------------------------------------------------------------- */
/* Symphony: emission and absorption (src/symphony.rs)                        */

enum { LOBE_POSITIVE = 0, LOBE_NEGATIVE = 1 };

typedef struct {
    const orc_dist *d;
    int coeff;
    int stokes;
    double s;
    double cos_observer_angle;
    double sin_observer_angle;
    int stokes_v_switch;
    orc_workspace *gamma_ws;
    orc_stats *stats;
    double cur_n; /* closure variable for the gamma integrand */
    double cur_gamma; /* closure variable of the gamma-contribution diagnostic */
} sym_state;

/* src/symphony.rs:398-479 */
static double sym_gamma_integrand(double gamma, void *ctx)
{
    sym_state *st = (sym_state *)ctx;
    const double n = st->cur_n;
    const double s = st->s;
    const double costh = st->cos_observer_angle;
    const double sinth = st->sin_observer_angle;

    const double beta = sqrt(1. - 1. / (gamma * gamma));
    const double cos_xi = (s * gamma - n) / (s * gamma * beta * costh);
    const double sin_xi = sqrt(1. - cos_xi * cos_xi);
    const double m = (costh - beta * cos_xi) / sinth;
    const double big_n = beta * sin_xi;
    double gamma_sin_xi, z, mj, njp, pol_term, f_term;

    if (st->stats)
        st->stats->n_symphony_integrand++;

    if (beta < 0.1) {
        gamma_sin_xi = gamma * sin_xi;
    } else {
        const double bc = beta * costh;
        const double beta2_costh2 = bc * bc;
        const double s_on_r = 2. * n / (s * (beta2_costh2 - 1.));
        const double r = 1. - 1. / beta2_costh2;
        gamma_sin_xi = sqrt(r * (gamma * (gamma + s_on_r)) - (n * n / (s * s * beta2_costh2)));
    }

    z = s * beta * sinth * gamma_sin_xi;

    mj = m * pkgw_bessel_j(n, z);
    njp = big_n * pkgw_bessel_dj(n, z);

    switch (st->stokes) {
    case ORC_STOKES_I:
        pol_term = mj * mj + njp * njp;
        break;
    case ORC_STOKES_Q:
        pol_term = mj * mj - njp * njp;
        break;
    default:
        pol_term = 2. * mj * njp;
    }

    if (st->coeff == ORC_COEFF_EMISSION) {
        f_term = orc_calc_f(st->d, gamma, cos_xi);
    } else {
        double dfdg, dfdcx, dfdcx_factor;
        orc_calc_f_derivatives(st->d, gamma, cos_xi, &dfdg, &dfdcx);
        dfdcx_factor = (beta * costh - cos_xi) / (gamma - 1. / gamma);
        f_term = dfdg + dfdcx_factor * dfdcx;
    }

    return gamma * gamma * pol_term * f_term;
}

/* src/symphony.rs:312-389 */
static double sym_gamma_integral(double n, void *ctx)
{
    sym_state *st = (sym_state *)ctx;
    const double s = st->s;
    const double costh = st->cos_observer_angle;
    const double sinth = st->sin_observer_angle;
    const double nos = n / s;
    const double root = sqrt(nos * nos - sinth * sinth);
    const double gamma_minus = (nos - fabs(costh) * root) / (sinth * sinth);
    const double gamma_plus = (nos + fabs(costh) * root) / (sinth * sinth);
    const double gamma_peak = 0.5 * (gamma_plus + gamma_minus);
    const double rel_width = (s < 1e6) ? 1. : exp(-0.27 * log(n) - 0.1);
    const double gamma_minus_high = gamma_peak - (gamma_peak - gamma_minus) * rel_width;
    const double gamma_plus_high = gamma_peak - (gamma_peak - gamma_plus) * rel_width;
    double gamma0, gamma1, contrib, abserr;
    int status;

    if (st->stokes == ORC_STOKES_V) {
        if (st->stokes_v_switch == LOBE_POSITIVE) {
            gamma0 = gamma_peak;
            gamma1 = gamma_plus_high;
        } else {
            gamma0 = gamma_minus_high;
            gamma1 = gamma_peak;
        }
    } else {
        gamma0 = gamma_minus_high;
        gamma1 = gamma_plus_high;
    }

    st->cur_n = n;
    status = orc_qag31(sym_gamma_integrand, st, gamma0, gamma1, 0., g_sym_epsrel, st->gamma_ws, &contrib,
                       &abserr);
    if (st->stats) {
        st->stats->n_gamma_qag++;
        if (st->gamma_ws->size > st->stats->max_gamma_intervals)
            st->stats->max_gamma_intervals = st->gamma_ws->size;
        if (status != ORC_SUCCESS)
            st->stats->n_gamma_qag_failed++;
    }
    if (status != ORC_SUCCESS)
        return NAN;
    return contrib;
}

/* src/symphony.rs:196-295; returns nonzero when the reference's `?` would
 * have propagated an Err (the caller maps that to NaN). */
static int sym_n_integration(sym_state *st, double n_start, double *out)
{
    double ans = 0., contrib = 0., delta_n = 1e5, incr_step_factor = 10.;
    const double DERIV_TOL = 1e-5, TOLERANCE = 1e5;
    orc_workspace *n_ws = (orc_workspace *)malloc(sizeof(orc_workspace));
    int rc = 0;

    orc_workspace_init(n_ws, 1000);

    if (st->s < 10.) {
        delta_n = 1.;
        incr_step_factor = 2.;
    }

    while (fabs(contrib) >= fabs(ans / TOLERANCE)) {
        double deriv, deriv_err, abserr;
        int status;

        orc_deriv_central(sym_gamma_integral, st, n_start, 1e-10 * n_start, &deriv, &deriv_err);

        if (deriv == 0. || (contrib != 0. && fabs(deriv / contrib) < DERIV_TOL))
            delta_n *= incr_step_factor;

        if (delta_n < n_start / incr_step_factor)
            delta_n *= incr_step_factor;

        status = orc_qag31(sym_gamma_integral, st, n_start, n_start + delta_n, 0., g_sym_epsrel, n_ws,
                           &contrib, &abserr);
        if (st->stats) {
            st->stats->n_chunks++;
            if (n_ws->size > st->stats->max_n_intervals)
                st->stats->max_n_intervals = n_ws->size;
        }
        if (status != ORC_SUCCESS) {
            rc = status;
            break;
        }

        ans += contrib;
        n_start += delta_n;

        if (n_start > 1e13)
            incr_step_factor = 1.;
    }

    free(n_ws);
    *out = ans;
    return rc;
}

double orc_symphony_lobes(const orc_dist *d, int coeff, int stokes, double s, double theta,
                          orc_stats *stats, double lobes[2])
{
    const double N_MAX = 30.;
    sym_state st;
    double ans = 0., n_minus, n_start, contrib, prefactor;
    double lobe_sum[2] = {0., 0.};
    int64_t n, n_lo, n_hi;
    int rc;

    st.d = d;
    st.coeff = coeff;
    st.stokes = stokes;
    st.s = s;
    st.cos_observer_angle = cos(theta);
    st.sin_observer_angle = sin(theta);
    st.stokes_v_switch = LOBE_NEGATIVE;
    st.stats = stats;
    st.cur_n = NAN;
    st.gamma_ws = (orc_workspace *)malloc(sizeof(orc_workspace));
    orc_workspace_init(st.gamma_ws, 5000);

    if (coeff == ORC_COEFF_EMISSION)
        prefactor = (ORC_TWO_PI * ORC_ELECTRON_CHARGE) * (ORC_TWO_PI * ORC_ELECTRON_CHARGE) /
                    (ORC_SPEED_LIGHT * fabs(st.cos_observer_angle));
    else
        prefactor = -1. * (ORC_TWO_PI * ORC_ELECTRON_CHARGE) * (ORC_TWO_PI * ORC_ELECTRON_CHARGE) /
                    (2. * ORC_MASS_ELECTRON * ORC_SPEED_LIGHT * fabs(st.cos_observer_angle));

    n_minus = s * fabs(st.sin_observer_angle);
    n_lo = (int64_t)(n_minus + 1.);
    n_hi = (int64_t)(n_minus + 1. + N_MAX);

    for (n = n_lo; n < n_hi; n++) {
        st.stokes_v_switch = LOBE_POSITIVE;
        contrib = sym_gamma_integral((double)n, &st);
        ans += contrib;
        lobe_sum[0] += contrib;

        if (stokes == ORC_STOKES_V) {
            st.stokes_v_switch = LOBE_NEGATIVE;
            contrib = sym_gamma_integral((double)n, &st);
            ans += contrib;
            lobe_sum[1] += contrib;
        }
    }

    if (!isfinite(ans))
        goto fail;

    n_start = floor(n_minus + 1. + N_MAX);

    st.stokes_v_switch = LOBE_POSITIVE;
    rc = sym_n_integration(&st, n_start, &contrib);
    if (rc != 0)
        contrib = NAN;
    ans += contrib;
    lobe_sum[0] += contrib;

    if (!isfinite(ans))
        goto fail;

    if (stokes == ORC_STOKES_V) {
        st.stokes_v_switch = LOBE_NEGATIVE;
        rc = sym_n_integration(&st, n_start, &contrib);
        if (rc != 0)
            contrib = NAN;
        ans += contrib;
        lobe_sum[1] += contrib;
    }

    if (!isfinite(ans))
        goto fail;

    free(st.gamma_ws);
    if (lobes) {
        lobes[0] = lobe_sum[0] * prefactor;
        lobes[1] = lobe_sum[1] * prefactor;
    }
    return ans * prefactor;

fail:
    free(st.gamma_ws);
    if (lobes) {
        lobes[0] = NAN;
        lobes[1] = NAN;
    }
    return NAN;
}

double orc_symphony(const orc_dist *d, int coeff, int stokes, double s, double theta,
                    orc_stats *stats)
{
    return orc_symphony_lobes(d, coeff, stokes, s, theta, stats, NULL);
}

/* The reference's diagnostics of the Symphony double integral (src/lib.rs:254-298):
 * what = 0 gamma_integrand(gamma = b, n = a)            (symphony.rs:585-590)
 *        1 gamma_integral(n = a)                        (symphony.rs:391-395, 576-580)
 *        2 the QAG of gamma_integral over [a, b]; NaN for the reference's Err (symphony.rs:297-307)
 *        3 gamma_contribution(gamma = a)                (symphony.rs:491-569)
 * CalculationState::new leaves the Stokes V switch on the negative lobe (symphony.rs:62). */
static double sym_integrand_of_n(double n, void *ctx)
{
    sym_state *st = (sym_state *)ctx;
    const double gamma = st->cur_gamma;
    st->cur_n = n;
    return sym_gamma_integrand(gamma, st);
}

double orc_symphony_diagnostic(const orc_dist *d, int coeff, int stokes, double s, double theta,
                               int what, double a, double b)
{
    sym_state st;
    double result = NAN, abserr;

    st.d = d;
    st.coeff = coeff;
    st.stokes = stokes;
    st.s = s;
    st.cos_observer_angle = cos(theta);
    st.sin_observer_angle = sin(theta);
    st.stokes_v_switch = LOBE_NEGATIVE;
    st.stats = NULL;
    st.cur_n = NAN;
    st.cur_gamma = NAN;
    st.gamma_ws = (orc_workspace *)malloc(sizeof(orc_workspace));
    orc_workspace_init(st.gamma_ws, 5000);

    if (what == 0) {
        st.cur_n = a;
        result = sym_gamma_integrand(b, &st);
    } else if (what == 1) {
        result = sym_gamma_integral(a, &st);
    } else if (what == 2) {
        orc_workspace *n_ws = (orc_workspace *)malloc(sizeof(orc_workspace));
        orc_workspace_init(n_ws, 1000);
        if (orc_qag31(sym_gamma_integral, &st, a, b, 0., 1e-3, n_ws, &result, &abserr) != ORC_SUCCESS)
            result = NAN;
        free(n_ws);
    } else {
        const double gamma = a;
        const double delta = fabs(st.cos_observer_angle) * sqrt(gamma * gamma - 1.);
        const int64_t n_minus = (int64_t)(s * (gamma - delta) + 1.);
        const int64_t n_plus = (int64_t)(s * (gamma + delta));
        const int64_t FULLY_DISCRETE_THRESHOLD = 1000, N_DISCRETE = 30;
        double ans = 0., contrib;
        int64_t n;

        st.cur_gamma = gamma;
        if (n_plus - n_minus < FULLY_DISCRETE_THRESHOLD) {
            for (n = n_minus; n < n_plus + 1; n++)
                ans += sym_integrand_of_n((double)n, &st);
        } else {
            for (n = n_minus; n < n_minus + N_DISCRETE + 1; n++)
                ans += sym_integrand_of_n((double)n, &st);
            if (orc_qag31(sym_integrand_of_n, &st, (double)(n_minus + N_DISCRETE + 1), (double)n_plus,
                          0., 1e-3, st.gamma_ws, &contrib, &abserr) != ORC_SUCCESS)
                contrib = NAN;
            ans += contrib;
        }
        if (!isfinite(ans))
            result = NAN;
        else if (coeff == ORC_COEFF_EMISSION)
            result = ans * ((ORC_TWO_PI * ORC_ELECTRON_CHARGE) * (ORC_TWO_PI * ORC_ELECTRON_CHARGE) /
                            (ORC_SPEED_LIGHT * fabs(st.cos_observer_angle)));
        else
            result = ans * (-1. * (ORC_TWO_PI * ORC_ELECTRON_CHARGE) * (ORC_TWO_PI * ORC_ELECTRON_CHARGE) /
                            (2. * ORC_MASS_ELECTRON * ORC_SPEED_LIGHT * fabs(st.cos_observer_angle)));
    }

    free(st.gamma_ws);
    return result;
}

/* ------------------------------------------------------------------------- */
/* Heyvaerts: Faraday conversion (Q, "h") and rotation (V, "f")               */

#define FOUR_OVER_SQRT_27 0.769800358919501
#define INVERSE_C (1. / ORC_SPEED_LIGHT)
#define INVERSE_SQRT_3 0.5773502691896257
#define SQRT_8_OVER_3 0.9428090415820635
#define THREE_TWO_THIRDS 2.080083823051904
#define G_APPROXIMATION_CUTOFF 10.

typedef struct {
    const orc_dist *d;
    int stokes;
    double s;
    double cos_observer_angle;
    double sin_observer_angle;
    double sigma0;
    double sigma0_sq;
    double sigma, pomega, x, gamma, mu;
    double outer_var; /* closure variable of the inner integrands */
    orc_workspace *iws;
    orc_stats *stats;
    int stage; /* diagnostics: which part of orc_heyvaerts is running */
} hey_state;

/* src/heyvaerts.rs:194-201 */
static void hey_fill_coord_vars(hey_state *st, double sigma, double pomega)
{
    st->sigma = sigma;
    st->pomega = pomega;
    st->x = sqrt(sigma * sigma - pomega * pomega - st->sigma0_sq);
    st->gamma = (sigma - pomega * st->cos_observer_angle) / (st->sigma0 * st->sin_observer_angle);
    st->mu = (sigma * st->cos_observer_angle - pomega) /
             (st->sigma0 * st->sin_observer_angle * sqrt(st->gamma * st->gamma - 1.));
}

/* src/heyvaerts.rs:472-493 */
static double hey_dfdsigma(const hey_state *st)
{
    double dfdg, dfdcxi, g_term, mu_term;
    orc_calc_f_derivatives(st->d, st->gamma, st->mu, &dfdg, &dfdcxi);
    g_term = dfdg / (st->sigma0 * st->sin_observer_angle);

    if (dfdcxi == 0.) {
        mu_term = 0.;
    } else {
        const double q = st->sigma - st->pomega * st->cos_observer_angle;
        const double r = st->pomega - st->sigma * st->cos_observer_angle;
        const double t = st->sigma0 * st->sin_observer_angle;
        const double u = q * q - t * t;
        const double dcxi_dsigma =
            (q * u * st->cos_observer_angle + u * r + r * t * t) / (pow(u, 1.5) * q);
        mu_term = dcxi_dsigma * dfdcxi;
    }

    return g_term + mu_term;
}

static double hey_jv(double order, double x)
{
    double j, y;
    orc_bessel_jy(order, x, &j, &y);
    return j;
}

static double hey_yv(double order, double x)
{
    double j, y;
    orc_bessel_jy(order, x, &j, &y);
    return y;
}

/* src/heyvaerts.rs:302-373 */
static double hey_h_qr_element(hey_state *st)
{
    const double po_sq = st->pomega * st->pomega;
    const double smxox = (st->sigma - st->x) / st->x;
    const double g = SQRT_8_OVER_3 * pow(st->sigma - st->x, 1.5) / sqrt(st->x);
    double y, t1, t2, t3;

    if (g < G_APPROXIMATION_CUTOFF) {
        const double plus = orc_bessel_i_series(2. / 3., g);
        const double minus = orc_bessel_i_series(-2. / 3., g);
        y = FOUR_OVER_SQRT_27 * smxox * smxox * (minus - plus) * (minus + plus);
    } else {
        const double jvp = hey_jv(st->sigma - 1., st->x) - st->sigma * hey_jv(st->sigma, st->x) / st->x;
        const double yvp = hey_yv(st->sigma - 1., st->x) - st->sigma * hey_yv(st->sigma, st->x) / st->x;
        if (st->stats)
            st->stats->n_heyvaerts_jy++;
        y = jvp * yvp;
    }

    t1 = ORC_PI * ORC_PI * st->x * st->x * y;

    if (g < G_APPROXIMATION_CUTOFF) {
        const double plus = orc_bessel_i_series(1. / 3., g);
        const double minus = orc_bessel_i_series(-1. / 3., g);
        y = 0.5 * FOUR_OVER_SQRT_27 * smxox * (minus - plus) * (minus + plus);
    } else {
        y = -hey_jv(st->sigma, st->x) * hey_yv(st->sigma, st->x);
    }

    t2 = ORC_PI * ORC_PI * st->pomega * st->pomega * y;
    t3 = -ORC_PI * (2. * po_sq + st->sigma0_sq) / sqrt(po_sq + st->sigma0_sq);

    return INVERSE_C * (t1 + t2 + t3) * hey_dfdsigma(st);
}

/* src/heyvaerts.rs:379-394 */
static double hey_h_nr_element(hey_state *st)
{
    const double s_sq = st->sigma * st->sigma;
    const double x_sq = st->x * st->x;
    const double ssqmxsq = s_sq - x_sq;
    const double ratio = s_sq / ssqmxsq;
    const double a1 = 1. / 8. - 5. / 24. * s_sq / ssqmxsq;
    const double a2 = 3. / 128. - 77. / 576. * s_sq / ssqmxsq + 385. / 3456. * (ratio * ratio);
    const double xa1p = -5. / 12. * s_sq * x_sq / (ssqmxsq * ssqmxsq);
    const double t1 = (6. * a2 - a1 * a1 + xa1p) / sqrt(ssqmxsq) + a1 * x_sq / pow(ssqmxsq, 1.5) -
                      x_sq * x_sq / pow(ssqmxsq, 2.5) / 8.;
    const double t2 = (6. * a2 - a1 * a1) / pow(ssqmxsq, 1.5);
    const double u1 = 2. * t1 - st->sigma0_sq * t2;

    return ORC_PI * INVERSE_C * u1 * hey_dfdsigma(st);
}

/* src/heyvaerts.rs:400-447 */
static double hey_f_qr_element(hey_state *st)
{
    const double g = SQRT_8_OVER_3 * pow(st->sigma - st->x, 1.5) / sqrt(st->x);
    double y;

    if (g < G_APPROXIMATION_CUTOFF) {
        y = INVERSE_SQRT_3 * g *
            (orc_bessel_i_series(-2. / 3., g) - orc_bessel_i_series(2. / 3., g)) *
            (orc_bessel_i_series(-1. / 3., g) + orc_bessel_i_series(1. / 3., g));
    } else {
        const double jvp = hey_jv(st->sigma - 1., st->x) - st->sigma * hey_jv(st->sigma, st->x) / st->x;
        if (st->stats)
            st->stats->n_heyvaerts_jy++;
        y = -st->x * jvp * hey_yv(st->sigma, st->x);
    }

    return -ORC_TWO_PI * INVERSE_C * st->pomega * (ORC_PI * y - 1.) * hey_dfdsigma(st);
}

/* src/heyvaerts.rs:453-468 */
static double hey_f_nr_element(hey_state *st)
{
    const double s_sq = st->sigma * st->sigma;
    const double x_sq = st->x * st->x;
    const double ssqmxsq = s_sq - x_sq;
    const double ratio = s_sq / ssqmxsq;
    const double a1 = 1. / 8. - 5. / 24. * s_sq / ssqmxsq;
    const double a2 = 3. / 128. - 77. / 576. * s_sq / ssqmxsq + 385. / 3456. * (ratio * ratio);
    const double xa1p = -5. / 12. * s_sq * x_sq / (ssqmxsq * ssqmxsq);
    const double z = 0.5 * x_sq / pow(ssqmxsq, 1.5) + (6. * a2 + xa1p - a1 * a1) / ssqmxsq +
                     1.5 * a1 * x_sq / (ssqmxsq * ssqmxsq);

    return -2. * ORC_PI * INVERSE_C * z * st->pomega * hey_dfdsigma(st);
}

static void hey_note_nonfinite(hey_state *st, int kind, double v)
{
    if (st->stats && !isfinite(v) && st->stats->hey_nan_kind == 0) {
        st->stats->hey_nan_kind = 1 + kind;
        st->stats->hey_nan_sigma = st->sigma;
        st->stats->hey_nan_pomega = st->pomega;
        st->stats->hey_nan_x = st->x;
        st->stats->hey_nan_gamma = st->gamma;
        st->stats->hey_nan_mu = st->mu;
        st->stats->hey_nan_value = v;
    }
}

static double hey_nr_inner(double sigma, void *ctx)
{
    hey_state *st = (hey_state *)ctx;
    if (st->stats)
        st->stats->n_heyvaerts_element++;
    hey_fill_coord_vars(st, sigma, st->outer_var);
    {
        const double v = st->stokes == ORC_STOKES_Q ? hey_h_nr_element(st) : hey_f_nr_element(st);
        hey_note_nonfinite(st, 0, v);
        return v;
    }
}

static double hey_qr_inner(double pomega, void *ctx)
{
    hey_state *st = (hey_state *)ctx;
    if (st->stats)
        st->stats->n_heyvaerts_element++;
    hey_fill_coord_vars(st, st->outer_var, pomega);
    {
        const double v = st->stokes == ORC_STOKES_Q ? hey_h_qr_element(st) : hey_f_qr_element(st);
        hey_note_nonfinite(st, 1, v);
        return v;
    }
}

/* src/heyvaerts.rs:213-250 */
static double hey_nr_outer_integrand(double pomega, void *ctx)
{
    hey_state *st = (hey_state *)ctx;
    const double sigma_min = sqrt(pomega * pomega + st->sigma0_sq);
    const double sigma_max = INVERSE_SQRT_3 * pow(sigma_min, 1.5);
    double result, abserr;
    int status;

    if (sigma_max <= sigma_min)
        return 0.;

    st->outer_var = pomega;
    status = orc_qag31(hey_nr_inner, st, sigma_min, sigma_max, 0., g_hey_epsrel, st->iws, &result, &abserr);
    if (st->stats) {
        st->stats->n_heyvaerts_qag++;
        if (status != ORC_SUCCESS && !st->stats->hey_fail_inner_status) {
            st->stats->hey_fail_inner_status = status;
            st->stats->hey_fail_inner_kind = 0;
            st->stats->hey_fail_inner_var = pomega;
        }
    }
    return status == ORC_SUCCESS ? result : NAN;
}

/* src/heyvaerts.rs:262-296 */
static double hey_qr_outer_integrand(double sigma, void *ctx)
{
    hey_state *st = (hey_state *)ctx;
    const double pomega_max_phys = sqrt(THREE_TWO_THIRDS * pow(sigma, 4. / 3.) - st->sigma0_sq);
    const double pomega_max_qr = sqrt(sigma * sigma - st->sigma0_sq);
    /* Rust f64::min: if one operand is NaN the other is returned */
    const double pomega_max = fmin(pomega_max_phys, pomega_max_qr);
    double result, abserr;
    int status;

    st->outer_var = sigma;
    status = orc_qag31(hey_qr_inner, st, -pomega_max, pomega_max, 0., g_hey_epsrel, st->iws, &result, &abserr);
    if (st->stats) {
        st->stats->n_heyvaerts_qag++;
        if (status != ORC_SUCCESS && !st->stats->hey_fail_inner_status) {
            st->stats->hey_fail_inner_status = status;
            st->stats->hey_fail_inner_kind = 1;
            st->stats->hey_fail_inner_var = sigma;
        }
    }
    return status == ORC_SUCCESS ? result : NAN;
}

static double hey_outer_integral(hey_state *st, orc_workspace *ows, orc_fn f, double a, double b)
{
    double result, abserr;
    int status = orc_qag31(f, st, a, b, 0., g_hey_epsrel, ows, &result, &abserr);
    if (st->stats) {
        st->stats->n_heyvaerts_qag++;
        if (status != ORC_SUCCESS && !st->stats->hey_fail_outer_status) {
            st->stats->hey_fail_outer_status = status;
            st->stats->hey_fail_stage = st->stage;
            st->stats->hey_fail_lo = a;
            st->stats->hey_fail_hi = b;
        }
    }
    return status == ORC_SUCCESS ? result : NAN;
}

/* src/heyvaerts.rs:60-191 */
double orc_heyvaerts(const orc_dist *d, int stokes, double s, double theta, orc_stats *stats)
{
    hey_state st;
    orc_workspace *ows, *iws;
    double pomega_left, pomega_right, delta_left, delta_right, nr_val, qr_val, sigma_low, delta_sigma;
    double result = NAN;
    int keep_going = 1;
    const double TOL = 1e-5, DELTA_SCALE_FACTOR = 5.;

    memset(&st, 0, sizeof(st));
    st.d = d;
    st.stokes = stokes;
    st.s = s;
    st.cos_observer_angle = cos(theta);
    st.sin_observer_angle = sin(theta);
    st.sigma0 = s * sin(theta);
    st.sigma0_sq = st.sigma0 * st.sigma0;
    st.sigma = st.pomega = st.x = st.gamma = st.mu = NAN;
    st.stats = stats;

    ows = (orc_workspace *)malloc(sizeof(orc_workspace));
    iws = (orc_workspace *)malloc(sizeof(orc_workspace));
    orc_workspace_init(ows, 4096);
    orc_workspace_init(iws, 4096);
    ows->trace = g_trace_hey_outer;
    st.iws = iws;

    pomega_left = -3. * st.sigma0;
    pomega_right = 3. * st.sigma0;
    delta_left = pomega_right;
    delta_right = pomega_right;

    st.stage = 1;
    nr_val = hey_outer_integral(&st, ows, hey_nr_outer_integrand, pomega_left, pomega_right);
    if (isnan(nr_val))
        goto done;

    st.stage = 2;
    while (keep_going) {
        double contrib;

        if (nr_val != 0.) {
            double rel_deriv, err;
            orc_deriv_central(hey_nr_outer_integrand, &st, pomega_right, 1e-6, &rel_deriv, &err);
            if (rel_deriv == 0. || fabs(1. / (rel_deriv * delta_right)) > DELTA_SCALE_FACTOR)
                delta_right *= DELTA_SCALE_FACTOR;
        }

        contrib = hey_outer_integral(&st, ows, hey_nr_outer_integrand, pomega_right,
                                     pomega_right + delta_right);
        if (isnan(contrib))
            goto done;

        if (nr_val != 0.)
            keep_going = fabs(contrib / nr_val) > TOL;

        nr_val += contrib;
        pomega_right += delta_right;
    }

    keep_going = 1;
    st.stage = 3;

    while (keep_going) {
        double contrib, rel_deriv, err;

        orc_deriv_central(hey_nr_outer_integrand, &st, pomega_left, 1e-6, &rel_deriv, &err);
        if (rel_deriv == 0. || fabs(1. / (rel_deriv * delta_left)) > DELTA_SCALE_FACTOR)
            delta_left *= DELTA_SCALE_FACTOR;

        contrib = hey_outer_integral(&st, ows, hey_nr_outer_integrand, pomega_left - delta_left,
                                     pomega_left);
        if (isnan(contrib))
            goto done;

        keep_going = fabs(contrib / nr_val) > TOL;
        nr_val += contrib;
        pomega_left -= delta_left;
    }

    qr_val = 0.;
    sigma_low = ORC_MAXV(st.sigma0, INVERSE_SQRT_3 * pow(st.sigma0, 1.5));
    delta_sigma = st.sigma0;
    keep_going = 1;
    st.stage = 4;

    while (keep_going) {
        double contrib;

        if (qr_val != 0.) {
            double rel_deriv, err;
            orc_deriv_central(hey_qr_outer_integrand, &st, sigma_low, 1e-6, &rel_deriv, &err);
            if (rel_deriv == 0. || fabs(1. / (rel_deriv * delta_sigma)) > DELTA_SCALE_FACTOR) {
                if (delta_sigma < 1e6 * st.sigma0)
                    delta_sigma *= DELTA_SCALE_FACTOR;
            }
        }

        contrib = hey_outer_integral(&st, ows, hey_qr_outer_integrand, sigma_low,
                                     sigma_low + delta_sigma);
        if (isnan(contrib))
            goto done;

        if (qr_val != 0.)
            keep_going = fabs(contrib / qr_val) > TOL;

        qr_val += contrib;
        sigma_low += delta_sigma;
    }

    if (stats) {
        stats->hey_nr_val = nr_val;
        stats->hey_qr_val = qr_val;
    }

    result = 2. * ORC_ELECTRON_CHARGE * ORC_ELECTRON_CHARGE * (nr_val + qr_val) /
             (ORC_MASS_ELECTRON * (s * st.sin_observer_angle) * (s * st.sin_observer_angle));

done:
    free(ows);
    free(iws);
    return result;
}

/* Parity-study hook: the outer integrands of orc_heyvaerts at one value of the outer variable
 * (which = 0: NR at pomega, 1: QR at sigma); NaN when the inner QAG fails, as in the flow above. */
double orc_test_hey_outer_integrand(const orc_dist *d, int stokes, double s, double theta, int which,
                                    double outer_var, orc_stats *stats)
{
    hey_state st;
    orc_workspace *iws = (orc_workspace *)malloc(sizeof(orc_workspace));
    double v;
    memset(&st, 0, sizeof(st));
    st.d = d;
    st.stokes = stokes;
    st.s = s;
    st.cos_observer_angle = cos(theta);
    st.sin_observer_angle = sin(theta);
    st.sigma0 = s * sin(theta);
    st.sigma0_sq = st.sigma0 * st.sigma0;
    st.stats = stats;
    orc_workspace_init(iws, 4096);
    st.iws = iws;
    v = which ? hey_qr_outer_integrand(outer_var, &st) : hey_nr_outer_integrand(outer_var, &st);
    if (stats)
        stats->max_gamma_intervals = iws->max_size_seen; /* reused: live intervals of the inner QAG */
    free(iws);
    return v;
}

/* ------------------------------------------------------------------------- */
/* Public calculator surface (src/lib.rs:150-247)                             */

double orc_compute_dimensionless(const orc_dist *d, int coeff, int stokes, double s, double theta,
                                 orc_stats *stats)
{
    if (coeff == ORC_COEFF_FARADAY) {
        if (stokes == ORC_STOKES_I)
            return NAN;
        return orc_heyvaerts(d, stokes, s, theta, stats);
    }
    return orc_symphony(d, coeff, stokes, s, theta, stats);
}

double orc_compute_cgs(const orc_dist *d, int coeff, int stokes, double nu, double b, double n_e,
                       double theta, orc_stats *stats)
{
    const double nu_c = ORC_ELECTRON_CHARGE * b / (ORC_TWO_PI * ORC_MASS_ELECTRON * ORC_SPEED_LIGHT);
    const double val = orc_compute_dimensionless(d, coeff, stokes, nu / nu_c, theta, stats);
    if (coeff == ORC_COEFF_EMISSION)
        return val * n_e * nu;
    return val * n_e / nu;
}

void orc_compute_all_dimensionless(const orc_dist *d, double s, double theta, double out[8],
                                   double lobes[4], orc_stats *stats)
{
    double lb[2];
    out[0] = orc_symphony(d, ORC_COEFF_EMISSION, ORC_STOKES_I, s, theta, stats);
    out[1] = orc_symphony(d, ORC_COEFF_ABSORPTION, ORC_STOKES_I, s, theta, stats);
    out[2] = orc_symphony(d, ORC_COEFF_EMISSION, ORC_STOKES_Q, s, theta, stats);
    out[3] = orc_symphony(d, ORC_COEFF_ABSORPTION, ORC_STOKES_Q, s, theta, stats);
    out[4] = orc_symphony_lobes(d, ORC_COEFF_EMISSION, ORC_STOKES_V, s, theta, stats, lb);
    if (lobes) {
        lobes[0] = lb[0];
        lobes[1] = lb[1];
    }
    out[5] = orc_symphony_lobes(d, ORC_COEFF_ABSORPTION, ORC_STOKES_V, s, theta, stats, lb);
    if (lobes) {
        lobes[2] = lb[0];
        lobes[3] = lb[1];
    }
    out[6] = orc_heyvaerts(d, ORC_STOKES_Q, s, theta, stats);
    out[7] = orc_heyvaerts(d, ORC_STOKES_V, s, theta, stats);
}

/* Batch driver, one point per OpenMP thread; same argument convention as the
 * product's C ABI (include/rimphony_b200.h): SoA inputs, out8 is [8][n]. */
int orc_batch_compute_all_dimensionless(int kind, int64_t n_points, const double *s,
                                        const double *theta, const double *const *params,
                                        int n_params, unsigned coeff_mask, double *out8,
                                        double *lobes4, int n_threads)
{
    int64_t i;
    int bad = 0;
#ifdef _OPENMP
    if (n_threads > 0)
        omp_set_num_threads(n_threads);
#else
    (void)n_threads;
#endif

#pragma omp parallel for schedule(dynamic, 1) reduction(| : bad)
    for (i = 0; i < n_points; i++) {
        orc_dist d;
        double pv[8];
        double o[8], lb[4] = {NAN, NAN, NAN, NAN}, l2[2];
        int j, c;
        for (j = 0; j < n_params && j < 8; j++)
            pv[j] = params[j][i];
        if (orc_dist_init(&d, kind, pv, n_params) != 0)
            bad |= 1;
        for (c = 0; c < 8; c++)
            o[c] = NAN;
        if (coeff_mask & 1u)
            o[0] = orc_symphony(&d, ORC_COEFF_EMISSION, ORC_STOKES_I, s[i], theta[i], NULL);
        if (coeff_mask & 2u)
            o[1] = orc_symphony(&d, ORC_COEFF_ABSORPTION, ORC_STOKES_I, s[i], theta[i], NULL);
        if (coeff_mask & 4u)
            o[2] = orc_symphony(&d, ORC_COEFF_EMISSION, ORC_STOKES_Q, s[i], theta[i], NULL);
        if (coeff_mask & 8u)
            o[3] = orc_symphony(&d, ORC_COEFF_ABSORPTION, ORC_STOKES_Q, s[i], theta[i], NULL);
        if (coeff_mask & 16u) {
            o[4] = orc_symphony_lobes(&d, ORC_COEFF_EMISSION, ORC_STOKES_V, s[i], theta[i], NULL, l2);
            lb[0] = l2[0];
            lb[1] = l2[1];
        }
        if (coeff_mask & 32u) {
            o[5] = orc_symphony_lobes(&d, ORC_COEFF_ABSORPTION, ORC_STOKES_V, s[i], theta[i], NULL, l2);
            lb[2] = l2[0];
            lb[3] = l2[1];
        }
        if (coeff_mask & 64u)
            o[6] = orc_heyvaerts(&d, ORC_STOKES_Q, s[i], theta[i], NULL);
        if (coeff_mask & 128u)
            o[7] = orc_heyvaerts(&d, ORC_STOKES_V, s[i], theta[i], NULL);
        for (c = 0; c < 8; c++)
            out8[(int64_t)c * n_points + i] = o[c];
        if (lobes4)
            for (c = 0; c < 4; c++)
                lobes4[(int64_t)c * n_points + i] = lb[c];
    }
    return bad;
}

int orc_num_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* Thin wrappers so tests can pin the building blocks individually. */
double orc_ref_bessel_j(double n, double x) { return pkgw_bessel_j(n, x); }
double orc_ref_bessel_dj(double n, double x) { return pkgw_bessel_dj(n, x); }
double orc_test_bessel_i(double nu, double x) { return orc_bessel_i_series(nu, x); }
void orc_test_bessel_jy(double nu, double x, double *j, double *y) { orc_bessel_jy(nu, x, j, y); }
double orc_test_bessel_k2(double z) { return orc_bessel_k2(z); }
double orc_test_pitch_angle_integral(double k) { return orc_pitch_angle_integral(k); }

typedef struct {
    int which;
    double a;
} test_fn_ctx;

static double test_fn(double x, void *ctx)
{
    const test_fn_ctx *c = (const test_fn_ctx *)ctx;
    switch (c->which) {
    case 0:
        return exp(-c->a * x) * sin(x) + 1.0; /* smooth */
    case 1:
        return pow(x, -c->a); /* endpoint-peaked */
    case 2:
        return 1.0 / (1e-4 + (x - c->a) * (x - c->a)); /* narrow peak */
    default:
        return NAN;
    }
}

int orc_test_qag(int which, double a_param, double lo, double hi, double epsrel, double *result,
                 double *abserr, int *n_intervals)
{
    orc_workspace *ws = (orc_workspace *)malloc(sizeof(orc_workspace));
    test_fn_ctx c;
    int status;
    c.which = which;
    c.a = a_param;
    orc_workspace_init(ws, 1000);
    status = orc_qag31(test_fn, &c, lo, hi, 0., epsrel, ws, result, abserr);
    *n_intervals = (int)ws->size;
    free(ws);
    return status;
}

double orc_test_deriv(int which, double a_param, double x, double h)
{
    test_fn_ctx c;
    double r, e;
    c.which = which;
    c.a = a_param;
    orc_deriv_central(test_fn, &c, x, h, &r, &e);
    return r;
}

void orc_gk31_tables(double xgk[16], double wgk[16], double wg[8])
{
    memcpy(xgk, orc_xgk31, sizeof(orc_xgk31));
    memcpy(wgk, orc_wgk31, sizeof(orc_wgk31));
    memcpy(wg, orc_wg15, sizeof(orc_wg15));
}
