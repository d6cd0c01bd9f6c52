// rb_transfer.cuh -- polarized radiative transfer through cells of constant coefficients, in FP64.
//
// Convention (include/rimphony_b200.h states the same matrix).  In each cell the eight coefficients of
// compute_all_cgs, [j_I, alpha_I, j_Q, alpha_Q, j_V, alpha_V, rho_Q, rho_V], are constant, and along the path s
//
//     dS/ds = J - K S,   S = (I, Q, U, V),   J = (j_I, j_Q c, j_Q s2, j_V)
//
//     K = | alpha_I      alpha_Q c    alpha_Q s2   alpha_V    |
//         | alpha_Q c    alpha_I      rho_V       -rho_Q s2   |
//         | alpha_Q s2  -rho_V        alpha_I      rho_Q c    |
//         | alpha_V      rho_Q s2    -rho_Q c      alpha_I    |
//
// with c = cos 2 psi, s2 = sin 2 psi.  A cell of length ds maps S to P S + Q J, P = exp(-K ds),
// Q = int_0^ds exp(-K t) dt.
//
// The closed form (DESIGN.md section 13).  Write K ds = z + M, z = alpha_I ds, M the polarized part times ds.
// M has the eigenvalues +-X1, +-i X2 (X1,2 = Lambda_1,2 ds), so any f(z + M) is the cubic
//     f = c0 + c1 M + c2 M^2 + c3 M^3,
//     c2 = w1 g[X1^2] + w2 g[-X2^2],      c3 = -(w1 h[X1^2] + w2 h[-X2^2]),
//     c0 = g0(-X2^2) + X2^2 c2,           c1 = -h0(-X2^2) + X2^2 c3,        w1,2 = X1,2^2 / (X1^2 + X2^2),
// where, for P (u = 1) and for Q / ds (integrated over u in [0, 1]),
//     g0(y) = e^{-zu} cosh(sqrt(y) u),  h0(y) = e^{-zu} sinh(sqrt(y) u) / sqrt(y),
//     g[y]  = e^{-zu} (cosh(sqrt(y) u) - 1) / y,   h[y] = e^{-zu} (sinh(sqrt(y) u) - sqrt(y) u) / y^{3/2},
// (y = -X2^2 turns cosh, sinh into cos, sin).  Each of these eight is positive or bounded by e^{-zu} cosh(X1 u),
// so nothing cancels beyond the factor (1 + |M|) that the monomial basis costs.  Each is evaluated
//   * by its power series in y when |X| is small: sum_m y^m u^{2m+j} / (2m+j)!, and for Q the same with
//     psi_k(z) = int_0^1 e^{-zu} u^k / k! du in place of u^k / k!, computed by a downward recurrence that only
//     adds positive terms;
//   * in closed form otherwise, from e^{-(z -+ X1)}, expm1 and (1 - e^{-w}) / w, where the differences left
//     are at most a factor 20 below their terms.
#pragma once

#include "rb_core.cuh"

namespace rb {

constexpr int kTransferK = 31; // top order of the psi_k and 1/k! chains (terms below 1e-17 of the sum)

constexpr double rb_inv_factorial(int n)
{
    double f = 1.0;
    for (int k = 2; k <= n; k++)
        f *= k;
    return 1.0 / f;
}

// (1 - e^{-w}) / w, with its limit 1 at w = 0
RB_HD double transfer_phi1(double w) { return (w == 0.0) ? 1.0 : -expm1(-w) / w; }

// The eight scalar pieces of one eigenvalue pair: [0..3] = g0, h0, g, h for P; [4..7] the same for Q / ds, each
// times sig^{j+1} (j = 0..3, sig = the scale of the integrated pieces, see transfer_cell).  `hyper`: y = X^2
// (cosh, sinh) or y = -X^2 (cos, sin).  chi0, chi1: sig psi_0(z), sig^2 psi_1(z); ser_p, ser_q: the series
// values [g0, h0, g, h] (valid when X is small), ser_q already scaled.
RB_HD void transfer_pieces(bool hyper, double z, double x, double sig, double chi0, double chi1, const double ser_p[4],
                           const double ser_q[4], double out[8])
{
    const double e0 = exp(-z);
    const double tq = fmax(1.0, 0.25 * z); // series threshold of the integrated pieces
    const double x2 = x * x;
    if (x <= 1.0) {
        for (int j = 0; j < 4; j++)
            out[j] = e0 * ser_p[j];
    } else if (hyper) {
        const double ep = exp(x - z), em = exp(-z - x);
        out[0] = 0.5 * (ep + em);
        out[1] = 0.5 * (ep - em) / x;
        out[2] = (out[0] - e0) / x2;
        out[3] = (out[1] - e0) / x2;
    } else {
        double sn, cs, sh, ch;
        sincos(x, &sn, &cs);
        sincos(0.5 * x, &sh, &ch);
        out[0] = e0 * cs;
        out[1] = e0 * sn / x;
        out[2] = e0 * (2.0 * sh * sh) / x2;
        out[3] = e0 * ((x - sn) / x) / x2;
    }
    if (x <= tq) {
        for (int j = 0; j < 4; j++)
            out[4 + j] = ser_q[j];
        return;
    }
    const double r = sig / x; // <= 4 when sig = z, since x > z / 4
    double sa, s2b;           // sig A and sig^2 B of the closed forms
    if (hyper) {
        const double fm = transfer_phi1(z - x), fp = transfer_phi1(z + x);
        sa = sig * (0.5 * (fm + fp));
        s2b = sig * r * (0.5 * (fm - fp));
    } else {
        // (1 - e^{-z - ix}) / (z + ix), numerator 1 - e^{-z} cos x + i e^{-z} sin x without cancellation
        double sn, cs, sh, ch;
        sincos(x, &sn, &cs);
        sincos(0.5 * x, &sh, &ch);
        const double nr = -expm1(-z) + 2.0 * e0 * sh * sh, ni = e0 * sn;
        double re, im;
        if (fabs(z) >= x) { // Smith's division
            const double q = x / z, d = z + x * q;
            re = (nr + ni * q) / d;
            im = (ni - nr * q) / d;
        } else {
            const double q = z / x, d = x + z * q;
            re = (nr * q + ni) / d;
            im = (ni * q - nr) / d;
        }
        sa = sig * re;
        s2b = -sig * r * im;
    }
    out[4] = sa;
    out[5] = s2b;
    out[6] = (hyper ? sa - chi0 : chi0 - sa) * (r * r);
    out[7] = (hyper ? s2b - chi1 : chi1 - s2b) * (r * r);
}

// out = sum_k c_k M^k v, by Horner: three products with M, whose entries are
// mq, mu, mv (absorption Q, U, V) and nq, nu, nv (Faraday Q, U, V).
RB_HD void transfer_horner(const double c[4], const double v[4], const double m[6], double out[4])
{
    double w[4];
    for (int i = 0; i < 4; i++)
        w[i] = c[3] * v[i];
    for (int k = 2; k >= 0; k--) {
        const double m0 = m[0] * w[1] + m[1] * w[2] + m[2] * w[3];
        const double m1 = m[0] * w[0] + m[5] * w[2] - m[4] * w[3];
        const double m2 = m[1] * w[0] - m[5] * w[1] + m[3] * w[3];
        const double m3 = m[2] * w[0] + m[4] * w[1] - m[3] * w[2];
        w[0] = c[k] * v[0] + m0;
        w[1] = c[k] * v[1] + m1;
        w[2] = c[k] * v[2] + m2;
        w[3] = c[k] * v[3] + m3;
    }
    for (int i = 0; i < 4; i++)
        out[i] = w[i];
}

// Cells whose alpha_I ds, |a| ds or |rho| ds exceeds this are outside the range of the closed form in FP64 (its
// cubic needs X^3 and 1 / X^3): transfer_ray makes such a ray NaN with kStatusNaN.
constexpr double kTransferMaxDepth = 1e102;
// Negative absorption (alpha_I < 0, a masing cell) is evaluated by the same formulas, whose power series then
// alternate and whose psi_k recurrence subtracts; they hold 3e-14 of the bound down to alpha_I ds = -12.  A cell
// with alpha_I ds below this is NaN with kStatusNaN: split it into cells of gain e^10 or less.
constexpr double kTransferMinDepth = -10.0;

// One cell: S <- P S + Q J.  k8 = [j_I, alpha_I, j_Q, alpha_Q, j_V, alpha_V, rho_Q, rho_V] (cgs), the field
// angle psi and the length ds (cm).  Inputs are assumed finite, ds >= 0 and alpha_I ds in [kTransferMinDepth,
// kTransferMaxDepth], |a| ds and |rho| ds below kTransferMaxDepth (transfer_ray checks).
RB_HD void transfer_cell(const double k8[8], double psi, double ds, double S[4])
{
    double s2, c;
    sincos(2.0 * psi, &s2, &c);
    const double z = k8[1] * ds;
    // the invariants of the polarized part, from the unrotated (Q, V) components: a rotation about V changes
    // neither |a|, |r| nor a.r
    const double aq = k8[3] * ds, av = k8[5] * ds, rq = k8[6] * ds, rv = k8[7] * ds;
    const double half_d = 0.5 * ((aq * aq + av * av) - (rq * rq + rv * rv));
    const double ar = fabs(aq * rq + av * rv);
    const double root = hypot(half_d, ar);
    double x1, x2;
    if (half_d >= 0.0) {
        x1 = sqrt(root + half_d);
        x2 = (x1 > 0.0) ? ar / x1 : 0.0;
    } else {
        x2 = sqrt(root - half_d);
        x1 = ar / x2;
    }
    const double y1 = x1 * x1, y2 = -(x2 * x2);

    // The integrated pieces are carried scaled: chi_k = sig^{k+1} psi_k(z) with sig = z when z > K + 1 (else 1),
    // so that they stay of order 1 where psi_k ~ z^{-k-1} would underflow (alpha_I ds ~ 1e10 and beyond), and
    // Q J = (ds / sig) sum_k chat_k (M / sig)^k J.  The recurrences, in the scaled variables:
    //   down  chi_k = (z / sig) chi_{k+1} + T_{k+1},   up (sig = z)  chi_k = chi_{k-1} - T_k,
    //   T_k = e^{-z} sig^k / k!.
    const bool big = z > kTransferK + 1.0;
    const double sig = big ? z : 1.0, mu = big ? 1.0 : z;
    double chi, tk; // chi_K and T_K
    if (!big) {     // psi_K(z) by its positive series
        double t = rb_inv_factorial(kTransferK + 1), sum = 0.0;
        for (int n = 0; n < 400; n++) {
            sum += t;
            t *= z / (kTransferK + 2 + n);
            if (fabs(t) <= 1e-18 * fabs(sum))
                break;
        }
        chi = exp(-z) * sum;
        tk = exp(-z) * rb_inv_factorial(kTransferK);
    } else { // upward from chi_0 = z phi1(z) = 1 - e^{-z}, stable for z > k
        chi = -expm1(-z);
        tk = exp(-z);
        for (int k = 1; k <= kTransferK; k++) {
            tk *= z / k;
            chi -= tk;
        }
    }
    // Downward over k, and Horner in y of G_j = psi_j + y G_{j+2} (Q, in the scaled variables: y / sig^2) and
    // c_j = 1/j! + y c_{j+2} (P), for y1 and y2 at once.
    const double yq1 = y1 / sig / sig, yq2 = y2 / sig / sig;
    double inv = rb_inv_factorial(kTransferK);
    double q1o = chi, q2o = chi, p1o = inv, p2o = inv; // odd chains start at k = K
    double q1e = 0.0, q2e = 0.0, p1e = 0.0, p2e = 0.0;
    double ser_q1[4], ser_q2[4], ser_p1[4], ser_p2[4];
    double chi0 = 0.0, chi1 = 0.0;
    for (int k = kTransferK - 1; k >= 0; k--) {
        chi = mu * chi + tk;  // chi_k
        tk *= (k + 1) / sig;  // T_k
        inv *= (k + 1);       // 1/k!
        if (k & 1) {
            q1o = chi + yq1 * q1o;
            q2o = chi + yq2 * q2o;
            p1o = inv + (y1 <= 1.0 ? y1 : 0.0) * p1o;
            p2o = inv + (-y2 <= 1.0 ? y2 : 0.0) * p2o;
        } else {
            q1e = chi + yq1 * q1e;
            q2e = chi + yq2 * q2e;
            p1e = inv + (y1 <= 1.0 ? y1 : 0.0) * p1e;
            p2e = inv + (-y2 <= 1.0 ? y2 : 0.0) * p2e;
        }
        if (k == 3 || k == 2) {
            ser_q1[k] = (k & 1) ? q1o : q1e;
            ser_q2[k] = (k & 1) ? q2o : q2e;
            ser_p1[k] = (k & 1) ? p1o : p1e;
            ser_p2[k] = (k & 1) ? p2o : p2e;
        }
        if (k == 1)
            chi1 = chi;
        if (k == 0)
            chi0 = chi;
    }
    ser_q1[0] = q1e;
    ser_q1[1] = q1o;
    ser_q2[0] = q2e;
    ser_q2[1] = q2o;
    ser_p1[0] = p1e;
    ser_p1[1] = p1o;
    ser_p2[0] = p2e;
    ser_p2[1] = p2o;

    double hyp[8], trig[8];
    transfer_pieces(true, z, x1, sig, chi0, chi1, ser_p1, ser_q1, hyp);
    transfer_pieces(false, z, x2, sig, chi0, chi1, ser_p2, ser_q2, trig);
    const double ysum = y1 - y2;
    const double w1 = (ysum > 0.0) ? y1 / ysum : 0.5, w2 = (ysum > 0.0) ? -y2 / ysum : 0.5;
    double cp[4], cq[4];
    for (int o = 0; o < 8; o += 4) {
        double *cc = o ? cq : cp;
        const double yy = o ? yq2 : y2;
        cc[2] = w1 * hyp[o + 2] + w2 * trig[o + 2];
        cc[3] = -(w1 * hyp[o + 3] + w2 * trig[o + 3]);
        cc[0] = trig[o + 0] - yy * cc[2];
        cc[1] = -trig[o + 1] - yy * cc[3];
    }

    // S <- sum_k cp_k M^k S + (ds / sig) sum_k cq_k (M / sig)^k J
    const double m[6] = {k8[3] * c * ds, k8[3] * s2 * ds, av, k8[6] * c * ds, k8[6] * s2 * ds, rv};
    double ms[6];
    for (int i = 0; i < 6; i++)
        ms[i] = m[i] / sig;
    const double l = ds / sig;
    const double J[4] = {k8[0] * l, k8[2] * c * l, k8[2] * s2 * l, k8[4] * l};
    double ps[4], qj[4];
    transfer_horner(cp, S, m, ps);
    transfer_horner(cq, J, ms, qj);
    for (int i = 0; i < 4; i++)
        S[i] = ps[i] + qj[i];
}

// One ray: cells ray * n_cells .. ray * n_cells + n_cells - 1 of the [8][n_points] coefficient array, entering
// with stokes0 (column `ray` of [4][n_rays], or zero if null).  Writes column `ray` of stokes4 and returns
// kStatusNaN if the result is NaN: a non-finite input, ds < 0 or a depth outside [kTransferMinDepth,
// kTransferMaxDepth] makes all four NaN, as does a non-finite result.
RB_HD unsigned transfer_ray(long long ray, long long n_rays, long long n_cells, const double *coeffs8,
                            const double *psi, const double *ds, const double *stokes0, double *stokes4)
{
    const long long n_points = n_rays * n_cells;
    double S[4];
    bool bad = false;
    for (int i = 0; i < 4; i++) {
        S[i] = stokes0 ? stokes0[i * n_rays + ray] : 0.0;
        bad |= !isfinite(S[i]);
    }
    for (long long cell = 0; cell < n_cells; cell++) {
        const long long p = ray * n_cells + cell;
        double k8[8];
        for (int c = 0; c < 8; c++) {
            k8[c] = coeffs8[c * n_points + p];
            bad |= !isfinite(k8[c]);
        }
        const double a = psi[p], l = ds[p];
        bad |= !isfinite(a) || !isfinite(l) || !(l >= 0.0);
        const double z = k8[1] * l;
        bad |= !(z >= kTransferMinDepth && z <= kTransferMaxDepth) ||
               fmax(fabs(k8[3]), fabs(k8[5])) * l > kTransferMaxDepth ||
               fmax(fabs(k8[6]), fabs(k8[7])) * l > kTransferMaxDepth;
        if (bad)
            break;
        transfer_cell(k8, a, l, S);
    }
    for (int i = 0; i < 4; i++)
        bad |= !isfinite(S[i]);
    for (int i = 0; i < 4; i++)
        stokes4[i * n_rays + ray] = bad ? NAN : S[i];
    return bad ? kStatusNaN : 0u;
}

} // namespace rb

#ifdef __CUDACC__
#include <cuda_runtime.h>

// Launchers of the transfer stage (inst_transfer.cu), called by the C ABI in rimphony_b200.cu.  Each returns the
// launch's error code.
namespace rbhost {
// One thread per ray.  status[ray] (nullable) = the ray's kStatusNaN, ORed with the status words of its cells
// when cell_status is given.
cudaError_t launch_transfer(long long n_rays, long long n_cells, const double *coeffs8, const double *psi,
                            const double *ds, const double *stokes0, const int *cell_status, double *stokes4,
                            int *status, cudaStream_t st);
// s[i] = nu[i] / nu_c(b[i]), the operations of compute_cgs (src/lib.rs:163-173)
cudaError_t launch_cgs_s(long long n, const double *nu, const double *b, double *s, cudaStream_t st);
// out8 in place: j * (n_e nu), alpha and rho * (n_e / nu), as compute_all_cgs (src/lib.rs:196-209)
cudaError_t launch_cgs_scale(long long n, const double *nu, const double *n_e, double *out8, cudaStream_t st);
} // namespace rbhost
#endif
