/* oracle/leung_bessel.c -- TEST INFRASTRUCTURE ONLY.
 *
 * C restatement of the reference's one native component, leung-bessel/src/bessel.c:
 * the Leung, Gammie & Noble (2011, Appendix B) fast evaluator of J_n(x), J_n'(x)
 * for real order n (pkgw_bessel_j :318-376, pkgw_bessel_dj :379-405,
 * BesselJ_Meissel_First :94-149, BesselJ_Meissel_Second :57-88,
 * BesselJ_Debye_Eps_Exp :159-213, exp_factor :22-51).  It reproduces the
 * reference's approximations, including the (n+1)*Gamma(n) substitution of
 * bessel.c:123-124; it is NOT a general-purpose accurate Bessel function.
 *
 * oracle/Makefile links it only where the reference's own file is not at hand
 * (neither oracle/_ref/libleung_ref.so nor $(REFERENCE)/leung-bessel/src/bessel.c).
 *
 * Provenance: the polynomial coefficients and their grouping are those of the IEEE
 * path of the device port, rimphony_b200/csrc/rb_bessel.cuh, with the reference's
 * own forms put back where the port documents a departure: lgamma() from libm,
 * region thresholds on eta = log10(eps), acosl/cosl in Meissel's second expansion,
 * and libm's jn() for integer orders below 30 (the reference calls
 * gsl_sf_bessel_Jn, the same function to double precision).  It is therefore NOT
 * an independent check of the port's transcription; what checks both is the
 * golden fixtures, which the reference's own bessel.c produced:
 * tests/test_oracle.py::test_oracle_reproduces_the_fixtures_made_with_the_reference
 * holds this file to them (x < n, the range of the Symphony integrand).
 */
#ifndef _DEFAULT_SOURCE
#define _DEFAULT_SOURCE 1 /* jn() */
#endif
#include <float.h>
#include <math.h>

#define LB_PI 3.14159265358979323846264338327950288

/* bessel.c:313-316 */
#define MINUS_ETA_A 0.174857
#define MINUS_ETA_B 0.295966
#define PLUS_ETA_A 0.151550
#define PLUS_ETA_B 0.438914
#define ETA_SLOPE (-0.6666666)
#define N_JN 30.0

/* bessel.c:171-174: At[m] = sin(pi (m+1)/3) 6^((m+1)/3) Gamma((m+1)/3), in double */
static const double At0 = 4.215772156113926;
static const double At1 = 3.8721718521798665;
static const double At3 = -8.431544312227844;
static const double At4 = -15.488687408719468;
static const double At6 = 67.45235449782282;
static const double At7 = 154.88687408719463;
static const double At9 = -944.3329629695189;
static const double At10 = -2478.189985395116;
static const double At12 = 18886.65925939032;
static const double At13 = 54520.17967869256;
static const double At15 = -491053.1407441488;

/* bessel.c:22-51: f_factor * exp(f_exp) without overflow where the product is representable */
static double exp_factor(double f_factor, double f_exp)
{
    if (f_factor == 0.0)
        return 0.0;
    if (fabs(f_exp) < 1e-3) {
        const double x = f_exp;
        return f_factor * (1.0 + ((40320.0 + (20160.0 + (6720.0 + (1680.0 + (336.0 + (56.0 + (8.0 + x) * x) * x) * x) *
                                  x) * x) * x) * x / 40320.0));
    }
    if (fabs(f_exp) > 690.0) {
        const double log_f = log(fabs(f_factor));
        if (log_f * f_exp < 0.0)
            return ((f_factor < 0.0) ? -1.0 : 1.0) * exp(log_f + f_exp);
    }
    return f_factor * exp(f_exp);
}

/* Meissel's second expansion, x > n (bessel.c:57-88) */
static double meissel_second(double n, double x)
{
    const double z = x / n;
    const double eps = (x - n) / n;
    const double Z = sqrt(eps * (1.0 + z));
    const double U = 1.0 / (n * Z * Z * Z);
    const double t1 = z * z;
    const double t2 = U * U;

    const double exp_val =
        (t1 * t2 * (-3072.0 - 768.0 * t1 + (3072.0 + (27648.0 + (22272.0 + 1248.0 * t1) * t1) * t1 +
        (-3072.0 + (-165120.0 + (-952576.0 + (-1119552.0 + (-271488.0 - 6592.0 * t1) * t1) * t1) * t1) * t1 +
        (3072.0 + (744960.0 + (15287808.0 + (72179904.0 + (102842688.0 + (45756144.0 + (5297808.0 +
        71391.0 * t1) * t1) * t1) * t1) * t1) * t1) * t1) * t2) * t2) * t2)) / 0.12288e5;

    const long double Qt = (long double)n * ((long double)Z - acosl(n / x));   /* n / x rounded in double, as there */

    const double Qsum =
        -(U * (860160.0 + 1290240.0 * t1 + (28672.0 + (-2709504.0 + (-6547968.0 - 672000.0 * t1) * t1) * t1 +
        (8192.0 + (2519040.0 + (60518400.0 + (151828480.0 + (61254720.0 + 2163168.0 * t1) * t1) * t1) * t1) * t1 +
        (-6144.0 + (2644992.0 + (299351808.0 + (3405435264.0 + (8653594320.0 + (5897669400.0 +
        (954875250.0 + 16907985.0 * t1) * t1) * t1) * t1) * t1) * t1) * t1) * t2) * t2) * t2)) / 0.10321920e8;

    const double factor = sqrt(2.0 / (LB_PI * n * Z)) * (double)cosl((long double)Qsum + Qt - 0.25L * (long double)LB_PI);
    return exp_factor(factor, exp_val);
}

/* Meissel's first expansion, x < n (bessel.c:94-149) */
static double meissel_first(double n, double x)
{
    const double z = x / n;
    const double eps = (n - x) / n;
    const double Z = sqrt(eps * (1.0 + z));
    const double U = 1.0 / (n * Z * Z * Z);
    const double t1 = z * z;
    const double D = 1.0 / 10321920.0;

    /* V_n sum: a polynomial in U whose coefficients are polynomials in z^2 */
    const double p0 = (860160.0 + 1290240.0 * t1) * D;
    const double p1 = ((-2580480.0 - 645120.0 * t1) * t1) * D;
    const double p2 = (-28672.0 + (2709504.0 + (6547968.0 + 672000.0 * t1) * t1) * t1) * D;
    const double p3 = ((-2580480.0 + (-23224320.0 + (-18708480.0 - 1048320.0 * t1) * t1) * t1) * t1) * D;
    const double p4 = (-8192.0 + (-2519040.0 + (-60518400.0 + (-151828480.0 + (-61254720.0 - 2163168.0 * t1) * t1) * t1) *
                       t1) * t1) * D;
    const double p5 = ((2580480.0 + (138700800.0 + (800163840.0 + (940423680.0 + (228049920.0 + 5537280.0 * t1) * t1) *
                        t1) * t1) * t1) * t1) * D;
    const double p6 = (6144.0 + (-2644992.0 + (-299351808.0 + (-3405435264.0 + (-8653594320.0 + (-5897669400.0 +
                       (-954875250.0 - 16907985.0 * t1) * t1) * t1) * t1) * t1) * t1) * t1) * D;
    const double p7 = ((2580480.0 + (625766400.0 + (12841758720.0 + (60631119360.0 + (86387857920.0 + (38435160960.0 +
                        (4450158720.0 + 59968440.0 * t1) * t1) * t1) * t1) * t1) * t1) * t1) * t1) * D;
    const double ninv = 1.0 / n;
    const double vsum1 = U * (p0 + U * (p1 + U * (p2 + U * (p3 + U * (p4 + U * (p5 + U * (p6 + U * p7)))))));
    const double ni2 = ninv * ninv;
    const double vsum2 = -(ninv * (420.0 + (-14.0 + (-4.0 + 3.0 * ni2) * ni2) * ni2)) / 5040.0;

    /* "I substitute Gamma(n+1) with (n+1)*Gamma(n) in the denominator" (bessel.c:123) */
    const double factor = 1.0 / ((n + 1.0) * sqrt(Z));

    double exp_val;
    if (eps < 1e-4 && n > 1e3) {
        /* Stirling's series for ln Gamma(n) and the expansion of n (ln(z / (1 + Z)) + Z) about eps = 0 (bessel.c:127-135) */
        const double ni4 = ni2 * ni2;
        const double loggamma_exp = (ninv * (-420.0 + 14.0 * ni2 - 4.0 * ni4 + 3.0 * ni4 * ni2)) / 5040.0;
        const double exp2 = -n * sqrt(2.0 * eps) * eps *
                            (0.984023040e9 + (0.442810368e9 + (0.303114240e9 + (0.233192960e9 + (0.190139040e9 +
                             (0.160692840e9 + 0.139204065e9 * eps) * eps) * eps) * eps) * eps) * eps) / 0.1476034560e10;
        exp_val = 0.5 * (log(n) - 1.837877066409345483560659472811235) + loggamma_exp - vsum2 + exp2 - vsum1;
    } else {
        double inv_zp1;
        if (Z < 1e-3)
            inv_zp1 = 1.0 + (-1.0 + (1.0 + (-1.0 + (1.0 + (-1.0 + (1.0 - Z) * Z) * Z) * Z) * Z) * Z) * Z;
        else
            inv_zp1 = 1.0 / (1.0 + Z);
        exp_val = n * (log(x * inv_zp1) - (1.0 - Z)) - vsum1 + (-vsum2 - lgamma(n));   /* bessel.c:145 */
    }
    return exp_factor(factor, exp_val);
}

/* The Debye "epsilon" expansion about x = n (bessel.c:159-213): a degree-14 polynomial
 * in ez = x - n whose coefficients are polynomials in x^(1/3). */
static double debye_eps(double n, double x)
{
    if (x > 1.0e55)
        return NAN;

    const double ez = x - n;
    const double z = cbrt(x);
    const double t3 = z * z;
    const double t4 = x * z;
    const double t10 = t4 * t4;
    const double t38 = 810485676000000.0 * At4 * t3;
    const double t70 = At7 * t3;
    const double t93 = At10 * t3;
    const double t107 = At13 * t3;
    const double t114 = ez * ez;
    const double t146 = t10 * t10;

    const double lead = (-5403237840000.0 * At6 + (69470200800000.0 * At4 + 19451656224000000.0 * At0 * t4) * t3) * t10 * z;

    const double e0 = -401283384.0 * At15 + (4707059994.0 * At13 + (3012121710.0 * At12 + (-36011689560.0 * At10 +
                      (8027667648000.0 * At9 + (-8027667648000.0 * At7 + (-1296777081600000.0 * At3 +
                      19451656224000000.0 * At1 * t3) * t4) * t3) * z) * t3) * z) * t3;
    const double e1 = (-41423013450.0 * At12 + (484040056500.0 * At10 + (67540473000000.0 * At6 - t38) * t4) * t3) * x;
    const double e2 = 1748257220.0 * At15 + (-19964735910.0 * At13 + (-2594411820000.0 * At9 +
                      (29331862560000.0 * At7 + 3241942704000000.0 * At3 * t4) * t3) * t4) * t3;
    const double e3 = (78248884350.0 * At12 + (-860873013000.0 * At10 + (-94556662200000.0 * At6 + t38) * t4) * t3) * x;
    const double e4 = -1938419560.0 * At15 + (20997160275.0 * At13 + (2283511230000.0 * At9 - 21612951360000.0 * t70) * t4) * t3;
    const double e5 = (-47153256150.0 * At12 + (459918459000.0 * At10 + 27016189200000.0 * At6 * t4) * t3) * x;
    const double e6 = 849093050.0 * At15 + (-8397889500.0 * At13 + (-643242600000.0 * At9 + 3859455600000.0 * t70) * t4) * t3;
    const double e7 = (11448186750.0 * At12 - 88445857500.0 * t93) * x;
    const double e8 = -173573400.0 * At15 + (1474097625.0 * At13 + 53603550000.0 * At9 * t4) * t3;
    const double e9 = (-1161410250.0 * At12 + 5360355000.0 * t93) * x;
    const double e10 = -113704500.0 * t107 + 17481100.0 * At15;
    const double e11 = 40608750.0 * At12 * x;
    const double e12 = -833000.0 * At15 + 3123750.0 * t107 + 14875.0 * At15 * t114;

    const double poly = (e0 + (e1 + (e2 + (e3 + (e4 + (e5 + (e6 + (e7 + (e8 + (e9 + (e10 + (e11 + e12 * ez) * ez) * ez) * ez) *
                        ez) * ez) * ez) * ez) * ez) * ez) * ez) * ez) * ez;

    return (lead + poly) / (LB_PI * t146 * 0.58354968672000000e17);
}

/* bessel.c:318-376 */
double pkgw_bessel_j(double n, double x)
{
    if (!(n >= 0.0) || !(x >= 0.0))
        return NAN;
    if (n < N_JN) {
        const int ni = (int)n;
        if ((double)ni != n)
            return NAN;
        return jn(ni, x);
    }
    if (x == n)
        return debye_eps(n, x);

    const double logn = log10(n);
    if (x < n) {
        const double eta = log10((n - x) / n);
        const double lo = ETA_SLOPE * logn + MINUS_ETA_A, hi = ETA_SLOPE * logn + MINUS_ETA_B;
        if (eta < lo)
            return debye_eps(n, x);
        if (eta > hi)
            return meissel_first(n, x);
        const double pos = (eta - lo) / (hi - lo);
        return debye_eps(n, x) * (1.0 - pos) + meissel_first(n, x) * pos;
    } else {
        const double eta = log10((x - n) / x);
        const double lo = ETA_SLOPE * logn + PLUS_ETA_A, hi = ETA_SLOPE * logn + PLUS_ETA_B;
        if (eta < lo)
            return debye_eps(n, x);
        if (eta > hi)
            return meissel_second(n, x);
        const double pos = (eta - lo) / (hi - lo);
        return debye_eps(n, x) * (1.0 - pos) + meissel_second(n, x) * pos;
    }
}

/* J_n'(x) = n J_n(x) / x - J_{n+1}(x) (bessel.c:379-405) */
double pkgw_bessel_dj(double n, double x)
{
    const double jn_ = pkgw_bessel_j(n, x);
    if (n >= 1e15)
        return NAN;
    const double jnp1 = pkgw_bessel_j(n + 1.0, x);
    if (x == 0.0) {
        if (n >= 2.0)
            return 0.0;
        if (n == 0.0)
            return -jnp1;
        return n * jn_ / DBL_MIN - jnp1;
    }
    return n * jn_ / x - jnp1;
}
