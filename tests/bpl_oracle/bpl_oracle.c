/* tests/bpl_oracle/bpl_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * The pitchy broken power law (kind 4 of include/rimphony_b200.h) for the CPU oracle.  The reference is
 * generic over DistributionFunction (src/lib.rs:111-146, 231-247); this is the `impl` a user would write,
 * built as src/pitchy_pl.rs builds its single power law:
 *
 *   f(gamma, cos xi) = norm B(gamma) exp(-gamma/gamma_c) sin^k xi / (gamma^2 beta)  on [gamma_min, gamma_max]
 *   B(gamma) = gamma^-p1 below gamma_break, gamma_break^(p2 - p1) gamma^-p2 from it on
 *
 * The derivatives are pointwise (pitchy_pl.rs:47-63) with the index of the side gamma lies on, and the
 * normalisation is pitchy_pl.rs:95-112 unchanged: one QAG (GK31, epsrel 1e-8) over [gamma_min, gamma_max],
 * without a split at the break.  The other kinds go to the oracle's own functions (bpl_oracle_base.c).
 *
 * orc_dist has no fields for p2 and gamma_break; like the device's Dist (rimphony_b200/csrc/rb_dist.cuh) the
 * kind keeps them in fields only PITCHY_KAPPA uses: p = p1, kappa = p2, width = gamma_break. */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "gsl_restated.h"
#include "special.h"
#include "rimphony_oracle.h"

enum { ORC_DIST_PITCHY_BROKEN_PL = 4 };

int orc_dist_init_base(orc_dist *d, int kind, const double *params, int n_params);
double orc_calc_f_base(const orc_dist *d, double gamma, double cos_xi);
void orc_calc_f_derivatives_base(const orc_dist *d, double gamma, double cos_xi, double *dfdg, double *dfdcx);

static double bpl_index(const orc_dist *d, double gamma) { return gamma < d->width ? d->p : d->kappa; }

static double bpl_gamma_term(const orc_dist *d, double gamma)
{
    if (gamma < d->width)
        return pow(gamma, -d->p);
    return pow(d->width, d->kappa - d->p) * pow(gamma, -d->kappa);
}

static double bpl_gamma_norm_integrand(double g, void *ctx)
{
    const orc_dist *d = (const orc_dist *)ctx;
    return bpl_gamma_term(d, g) * exp(-g * d->inv_gamma_cutoff);
}

int orc_dist_init(orc_dist *d, int kind, const double *params, int n_params)
{
    orc_workspace *ws;
    double integral = NAN, abserr;
    int status;

    if (kind != ORC_DIST_PITCHY_BROKEN_PL)
        return orc_dist_init_base(d, kind, params, n_params);
    memset(d, 0, sizeof(*d));
    d->kind = kind;
    d->norm = NAN;
    d->gamma_min = 1.;
    d->gamma_max = 1e12;
    d->inv_gamma_cutoff = 1e-10;
    /* params: p1, p2, gamma_break, k [, gamma_min, gamma_max, gamma_cutoff] */
    if (n_params != 4 && n_params != 7)
        return -1;
    d->p = params[0];
    d->kappa = params[1];
    d->width = params[2];
    d->k = params[3];
    if (n_params == 7) {
        d->gamma_min = params[4];
        d->gamma_max = params[5];
        d->inv_gamma_cutoff = 1. / params[6];
    }
    ws = (orc_workspace *)malloc(sizeof(orc_workspace));
    orc_workspace_init(ws, 1000);
    status = orc_qag31(bpl_gamma_norm_integrand, d, d->gamma_min, d->gamma_max, 0., 1e-8, ws, &integral, &abserr);
    free(ws);
    d->norm = (status == 0) ? 1. / (2. * (2. * M_PI) * orc_pitch_angle_integral(d->k) * integral) : NAN;
    return status;
}

double orc_calc_f(const orc_dist *d, double gamma, double cos_xi)
{
    double sin_xi, pa_term, beta, gamma_term;
    if (d->kind != ORC_DIST_PITCHY_BROKEN_PL)
        return orc_calc_f_base(d, gamma, cos_xi);
    if (gamma < d->gamma_min || gamma > d->gamma_max)
        return 0.;
    sin_xi = sqrt(1. - cos_xi * cos_xi);
    pa_term = pow(sin_xi, d->k);
    beta = sqrt(1. - 1. / (gamma * gamma));
    gamma_term = bpl_gamma_term(d, gamma) * exp(-gamma * d->inv_gamma_cutoff);
    return d->norm * pa_term * gamma_term / (gamma * gamma * beta);
}

void orc_calc_f_derivatives(const orc_dist *d, double gamma, double cos_xi, double *dfdg, double *dfdcx)
{
    double sin_xi, f;
    if (d->kind != ORC_DIST_PITCHY_BROKEN_PL) {
        orc_calc_f_derivatives_base(d, gamma, cos_xi, dfdg, dfdcx);
        return;
    }
    if (gamma < d->gamma_min || gamma > d->gamma_max) {
        *dfdg = 0.;
        *dfdcx = 0.;
        return;
    }
    sin_xi = sqrt(1. - cos_xi * cos_xi);
    f = orc_calc_f(d, gamma, cos_xi);
    *dfdg = -f * ((bpl_index(d, gamma) + 1.) / gamma + gamma / (gamma * gamma - 1.) + d->inv_gamma_cutoff);
    *dfdcx = -f * d->k * cos_xi / (sin_xi * sin_xi);
}
