/* rimphony_b200.h -- C ABI of the B200-native implementation of rimphony's
 * data-parallel hot path: all eight polarized synchrotron transfer
 * coefficients for a batch of independent (s, theta, distribution) points.
 *
 * This is the drop-in boundary: the entry points below are what a Rust `extern
 * "C"` block (built from build.rs with nvcc, see INTEGRATION.md and rust/)
 * binds in place of the reference's per-point scalar path.  Plain pointers and
 * sizes only; no CUDA, torch or C++ types appear in any signature.
 *
 * Reference interface replaced (file:line in pkgw/rimphony):
 *   src/lib.rs:150-210   trait SynchrotronCalculator { compute_dimensionless,
 *                        compute_cgs, compute_all_dimensionless, compute_all_cgs }
 *   src/lib.rs:231-247   FullSynchrotronCalculator<D> dispatch
 *   src/power_law.rs:71-111, src/thermal_juettner.rs:45-72,
 *   src/pitchy_pl.rs:73-115, src/pitchy_kappa.rs:70-125
 *                        XDistribution::new(..)[.gamma_limits(..)].full_calculation(..)
 *   leung-bessel/src/lib.rs:56-75   Jn, Jn_prime   (rimphony_b200_bessel_jn)
 *
 * Error model (SURVEY.md section 8-b): a NUMERICAL failure is not an error.  It
 * yields NaN in the affected output slot, exactly as the reference does
 * (symphony.rs:115-146, heyvaerts.rs:98-177, lib.rs:239-240), plus a nonzero
 * per-point status word.  The return code is nonzero only for infrastructure
 * errors (bad arguments, no CUDA device, CUDA failure); rimphony_b200_last_error()
 * then describes it.  There is no CPU fallback of any kind.
 */
#ifndef RIMPHONY_B200_H
#define RIMPHONY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RIMPHONY_B200_ABI_VERSION 2

/* Distribution kinds and the order of their parameter columns.
 *   POWER_LAW         p [, gamma_min, gamma_max, gamma_cutoff]        1 or 4 columns
 *   THERMAL_JUETTNER  T                                                1 column
 *   PITCHY_PL         p, k [, gamma_min, gamma_max, gamma_cutoff]     2 or 5 columns
 *   PITCHY_KAPPA      kappa, width, k [, gamma_cutoff]                 3 or 4 columns
 *   PITCHY_BROKEN_PL  p1, p2, gamma_break, k                           4 or 7 columns
 *                     [, gamma_min, gamma_max, gamma_cutoff]
 *                     gamma^-p1 below gamma_break, gamma_break^(p2 - p1) gamma^-p2 from it on,
 *                     times sin^k(xi) as in PITCHY_PL
 * Omitted trailing columns take the reference's defaults: gamma_min = 1,
 * gamma_max = 1e12, gamma_cutoff = 1e10. */
enum rimphony_b200_dist_kind {
    RIMPHONY_B200_POWER_LAW = 0,
    RIMPHONY_B200_THERMAL_JUETTNER = 1,
    RIMPHONY_B200_PITCHY_PL = 2,
    RIMPHONY_B200_PITCHY_KAPPA = 3,
    RIMPHONY_B200_PITCHY_BROKEN_PL = 4
};

/* src/lib.rs:92-107 and :75-87 */
enum rimphony_b200_coefficient { RIMPHONY_B200_EMISSION = 0, RIMPHONY_B200_ABSORPTION = 1, RIMPHONY_B200_FARADAY = 2 };
enum rimphony_b200_stokes { RIMPHONY_B200_STOKES_I = 0, RIMPHONY_B200_STOKES_Q = 1, RIMPHONY_B200_STOKES_V = 2 };

/* Output slots, the order of compute_all_dimensionless (src/lib.rs:176-177). */
enum {
    RIMPHONY_B200_J_I = 0,
    RIMPHONY_B200_ALPHA_I = 1,
    RIMPHONY_B200_J_Q = 2,
    RIMPHONY_B200_ALPHA_Q = 3,
    RIMPHONY_B200_J_V = 4,
    RIMPHONY_B200_ALPHA_V = 5,
    RIMPHONY_B200_RHO_Q = 6,
    RIMPHONY_B200_RHO_V = 7
};

/* Evaluation modes.
 *   FAST      product default.  Same integrands, domains and truncation rules as the
 *             reference, evaluated by the compact warp engine: the six j/alpha
 *             integrands share every node, the gamma integral is seeded on the
 *             J_n^2 peak and cut at the reference Bessel evaluator's region
 *             boundaries, the harmonic integral marches in ln n.  Agrees with the
 *             reference's algorithm within its own integration tolerance (1e-3).
 *   FAITHFUL  every coefficient is integrated on its own with the same sequence
 *             of Gauss-Kronrod applications as the reference performs; agrees with
 *             the reference's algorithm to rounding.  The parity anchor; slow.
 *   FUSED     the reference's control flow (QUADPACK bisection, chunked n
 *             integration with derivative probes) with the six j/alpha integrands,
 *             and rho_Q / rho_V, converged together on shared nodes; points with
 *             s sin(theta) < 3 take the faithful Faraday sequence.
 *   FUSED_ALL FUSED without the s sin(theta) < 3 exception (experiments). */
enum rimphony_b200_mode {
    RIMPHONY_B200_MODE_FAST = 0,
    RIMPHONY_B200_MODE_FAITHFUL = 1,
    RIMPHONY_B200_MODE_FUSED_ALL = 2,
    RIMPHONY_B200_MODE_FUSED = 3
};

/* Per-point status bits. */
#define RIMPHONY_B200_STATUS_NAN 1u         /* at least one requested coefficient is NaN */
#define RIMPHONY_B200_STATUS_CAP_HIT 2u     /* an interval list or step budget filled up */
#define RIMPHONY_B200_STATUS_NORM_FAILED 4u /* the normalisation integral failed */
#define RIMPHONY_B200_STATUS_REROUTED 8u    /* FAST mode handed the point to the FAITHFUL sequence: its reference
                                               value is set by where the reference's quadrature loses the J_n^2
                                               peak (n > 1e10, hard spectra), see DESIGN.md */
#define RIMPHONY_B200_STATUS_REFERENCE_DIVERGES 16u /* FAST mode, rho_Q / rho_V of a power law with gamma_min = 1 at
                                               s < 0.38 (rho_V) / 0.35 (rho_Q): the reference's adaptive quadrature
                                               cannot converge on the |sigma - s|^(2s-1) singularity of the
                                               quasi-resonant integrand and returns NaN (heyvaerts.rs:175-177); so
                                               does this path, without integrating (DESIGN.md section 6) */

typedef struct rimphony_b200_options {
    uint32_t struct_size;          /* sizeof(rimphony_b200_options); 0-initialise the rest for defaults */
    int32_t mode;                  /* enum rimphony_b200_mode */
    uint32_t coeff_mask;           /* bit i: compute output slot i; 0 means all eight */
    uint32_t param_broadcast_mask; /* bit j: params[j] points to ONE value used for every point */
    int32_t device_plus_one;       /* CUDA ordinal + 1; 0 = the calling thread's current device */
    int32_t reserved0;
    double epsrel_gamma;           /* Symphony gamma integral, 0 = reference value 1e-3 (symphony.rs:376) */
    double epsrel_n;               /* Symphony n integral,     0 = 1e-3 (symphony.rs:266) */
    double epsrel_heyvaerts_inner; /* 0 = 1e-3 (heyvaerts.rs:228, 274) */
    double epsrel_heyvaerts_outer; /* 0 = 1e-3 (heyvaerts.rs:206, 255) */
} rimphony_b200_options;

/* Optional extra outputs (any pointer may be NULL). */
typedef struct rimphony_b200_extras {
    double *lobes4;     /* [4][n]: j_V(+), j_V(-), alpha_V(+), alpha_V(-): the two Stokes-V lobes
                           the reference integrates separately (symphony.rs:97-107, 126-140) */
    uint32_t *counters; /* [2][n]: Gauss-Kronrod applications spent in Symphony / in Heyvaerts */
    double *norm;       /* [n]: the distribution's normalisation constant */
} rimphony_b200_extras;

/* The batched hot path (replaces the loop body of examples/crank-out-pitchypl.rs:157-172).
 *
 *   s, theta   [n_points] host arrays
 *   params     n_params host column pointers, each [n_points] (or 1 value, see
 *              param_broadcast_mask)
 *   out8       [8][n_points] host array, slot-major (SoA), order of lib.rs:176-177
 *   status     [n_points] or NULL
 *
 * Host -> device copies, the kernels and the device -> host copies all run inside
 * the call.  Returns 0 on success. */
int rimphony_b200_compute_all_dimensionless(int kind, int64_t n_points, const double *s, const double *theta,
                                            const double *const *params, int n_params,
                                            const rimphony_b200_options *opts, double *out8, int32_t *status);

int rimphony_b200_compute_all_dimensionless_ex(int kind, int64_t n_points, const double *s, const double *theta,
                                               const double *const *params, int n_params,
                                               const rimphony_b200_options *opts, double *out8, int32_t *status,
                                               const rimphony_b200_extras *extras);

/* Same, but every array pointer (s, theta, params[j], out8, status, extras->*) is a
 * DEVICE pointer on the selected device and `stream` is a cudaStream_t passed as void*
 * (NULL = the library's own stream for that device).  Nothing is copied; the
 * call returns after the kernels have been enqueued and, if `synchronize` is
 * nonzero, completed.  Output slots that coeff_mask does not request are left
 * untouched (the host entry points fill them with NaN).
 *
 * Asynchronous use (synchronize = 0): the library keeps one set of scratch buffers per
 * device, so batched calls on one device are serialised ON THE DEVICE: a call enqueued
 * while an earlier one is still running (on the same or on another stream) first waits
 * for that call's completion event.  The host never blocks for this, results are ordered
 * after `stream` as usual, and rimphony_b200_last_kernel_ms() is meaningful only after a
 * synchronize = 1 call. */
int rimphony_b200_compute_all_dimensionless_device(int kind, int64_t n_points, const double *s, const double *theta,
                                                   const double *const *params, int n_params,
                                                   const rimphony_b200_options *opts, double *out8,
                                                   int32_t *status, const rimphony_b200_extras *extras,
                                                   void *stream, int synchronize);

/* Shard the batch evenly over the first `n_devices` GPUs of this box (0 = all visible;
 * opts->device_plus_one is ignored): one host thread and stream per device, contiguous
 * slices, no inter-GPU communication.  Each shard's eight result rows are copied straight
 * into their slices of the caller's [8][n_points] array, so the host gathers by
 * construction.  Host arrays. */
int rimphony_b200_compute_all_dimensionless_multi(int kind, int64_t n_points, const double *s, const double *theta,
                                                  const double *const *params, int n_params,
                                                  const rimphony_b200_options *opts, double *out8,
                                                  int32_t *status, int n_devices);

/* Scalar conveniences behind the per-point trait methods (src/lib.rs:154-173).
 * `params` holds one value per column.  (Faraday, I) yields NaN as in lib.rs:239-240. */
int rimphony_b200_compute_dimensionless(int kind, const double *params, int n_params, int coeff, int stokes,
                                        double s, double theta, double *out);
int rimphony_b200_compute_cgs(int kind, const double *params, int n_params, int coeff, int stokes, double nu,
                              double b, double n_e, double theta, double *out);

/* The reference's diagnostics of the Symphony double integral at ONE point
 * (FullSynchrotronCalculator::diagnostic_symphony_*, src/lib.rs:254-298), evaluated for `count`
 * arguments at once, one warp each, with the reference's own sequence of rule applications:
 *   GAMMA_INTEGRAND     out[i] = gamma_integrand(gamma = b[i], n = a[i])   (symphony.rs:398-479, 585-590)
 *   GAMMA_INTEGRAL      out[i] = G(n = a[i])                               (symphony.rs:312-395, 576-580)
 *   N_INTEGRAL          out[i] = QAG of G over [a[i], b[i]]; the reference's Err is NaN here
 *                                                                          (symphony.rs:297-307, 571-574)
 *   GAMMA_CONTRIBUTION  out[i] = sum over n at gamma = a[i], dimensional constants applied
 *                                                                          (symphony.rs:481-569, 592-598)
 * coeff is EMISSION or ABSORPTION.  For Stokes V the gamma integral covers the lobe below
 * gamma_peak, as in the reference (CalculationState::new, symphony.rs:62).  b may be null for
 * the one-argument diagnostics; status (nullable) receives RIMPHONY_B200_STATUS_* bits.  Host arrays. */
enum rimphony_b200_diagnostic {
    RIMPHONY_B200_DIAG_GAMMA_INTEGRAND = 0,
    RIMPHONY_B200_DIAG_GAMMA_INTEGRAL = 1,
    RIMPHONY_B200_DIAG_N_INTEGRAL = 2,
    RIMPHONY_B200_DIAG_GAMMA_CONTRIBUTION = 3
};
int rimphony_b200_diagnostic_symphony(int kind, const double *params, int n_params, int coeff, int stokes, double s,
                                      double theta, int what, int64_t count, const double *a, const double *b,
                                      double *out, int32_t *status);

/* The Leung fast Bessel evaluator on the device: j[i] = J_n(x) as pkgw_bessel_j,
 * dj[i] = J_n'(x) as pkgw_bessel_dj (leung-bessel/src/bessel.c:318-405).  Host arrays. */
int rimphony_b200_bessel_jn(int64_t count, const double *n, const double *x, double *j, double *dj);

/* The distribution function and its partial derivatives on the device
 * (trait DistributionFunction, src/lib.rs:111-146), with norm = 1:
 * out3 = [3][count]: f, df/dgamma, df/dcos(xi).  Host arrays. */
int rimphony_b200_dist_eval(int kind, const double *params, int n_params, int64_t count, const double *gamma,
                            const double *cos_xi, double *out3);

/* Polarized radiative transfer through rays of cells (DESIGN.md section 13).
 *
 * In each cell the eight coefficients are constant, in the units of compute_all_cgs (j in
 * erg s^-1 cm^-3 Hz^-1 sr^-1, alpha and rho in cm^-1), and along the path s
 *
 *     dS/ds = J - K S,   S = (I, Q, U, V),   J = (j_I, j_Q c, j_Q s2, j_V)
 *
 *     K = | alpha_I      alpha_Q c    alpha_Q s2   alpha_V    |
 *         | alpha_Q c    alpha_I      rho_V       -rho_Q s2   |
 *         | alpha_Q s2  -rho_V        alpha_I      rho_Q c    |
 *         | alpha_V      rho_Q s2    -rho_Q c      alpha_I    |
 *
 * with c = cos 2 psi and s2 = sin 2 psi: psi rotates the coefficients' frame, in which the U
 * components are zero, into the observer's Stokes basis.  So with psi = 0, rho_V alone turns
 * (Q, U) through +rho_V ds (Q -> U), and rho_Q alone turns (U, V) through +rho_Q ds (U -> V).
 * Another convention maps onto this one by negating inputs: the sign of V (negate j_V, alpha_V and
 * rho_V), the sense of the Faraday rotation (rho_V) or of psi.
 *
 * A ray has n_cells cells; cell 0 is where it enters, with the incident Stokes vector stokes0
 * (zero if NULL), and cell n_cells - 1 is on the observer's side.  Each cell of length ds applies
 *     S <- P S + Q J,   P = exp(-K ds),   Q = int_0^ds exp(-K t) dt,
 * evaluated in closed form in FP64 (accurate for optically thin and thick cells up to alpha_I ds =
 * 1e100, fully polarized absorption and Faraday depths |rho| ds up to 1e6).  A uniform slab is
 * n_cells = 1.  Negative absorption (a masing cell) is supported down to alpha_I ds = -10; a cell
 * with alpha_I ds below -10, or with alpha_I ds, |alpha_pol| ds or |rho| ds above 1e102, makes its
 * ray NaN (split such a cell into shorter ones).
 *
 *   coeffs8   [8][n_rays * n_cells], slot-major in the order of out8; point index ray * n_cells + cell
 *   psi, ds   [n_rays * n_cells] (radian, cm)
 *   stokes0   [4][n_rays] or NULL
 *   stokes4   [4][n_rays], the emergent (I, Q, U, V)
 *   status    [n_rays] or NULL: RIMPHONY_B200_STATUS_NAN if the ray's Stokes vector is NaN, which it
 *             is when an input of the ray is not finite, a ds is negative or a cell is out of range
 * Host arrays.  Runs on the calling thread's current device. */
int rimphony_b200_transfer(int64_t n_rays, int64_t n_cells, const double *coeffs8, const double *psi, const double *ds,
                           const double *stokes0, double *stokes4, int32_t *status);

/* Same, with every array a DEVICE pointer on the calling thread's current device and `stream` a
 * cudaStream_t passed as void* (NULL = the library's own stream), as in
 * rimphony_b200_compute_all_dimensionless_device.  Uses no scratch memory of the library. */
int rimphony_b200_transfer_device(int64_t n_rays, int64_t n_cells, const double *coeffs8, const double *psi,
                                  const double *ds, const double *stokes0, double *stokes4, int32_t *status,
                                  void *stream, int synchronize);

/* The whole chain for rays of cells, in one call on the device: s = nu / nu_c(b) per cell, the
 * eight coefficients (opts as in the batched call; coeff_mask must be 0 or 0xFF), the cgs scaling of
 * compute_all_cgs (src/lib.rs:196-209, the same operations in the same order, so both agree to the
 * bit), then the transfer above with no incident radiation.
 *   nu, b, n_e, theta, psi, ds   [n_rays * n_cells] (Hz, G, cm^-3, radian, radian, cm)
 *   params       as in the batched call, [n_rays * n_cells] columns (or broadcast)
 *   stokes4      [4][n_rays]
 *   coeffs8_cgs  [8][n_rays * n_cells] or NULL: the cells' cgs coefficients
 *   status       [n_rays] or NULL: the OR of the status words of the ray's cells, with
 *                RIMPHONY_B200_STATUS_NAN set if the ray's Stokes vector is NaN
 * Host arrays. */
int rimphony_b200_compute_stokes_cgs(int kind, int64_t n_rays, int64_t n_cells, const double *nu, const double *b,
                                     const double *n_e, const double *theta, const double *psi, const double *ds,
                                     const double *const *params, int n_params, const rimphony_b200_options *opts,
                                     double *stokes4, double *coeffs8_cgs, int32_t *status);

/* Device time (ms, CUDA events on the launching stream) of the kernels of the most
 * recent batched call made by this thread's device: [0] normalisation,
 * [1] Symphony, [2] Heyvaerts, [3] whole enqueue-to-completion span. */
int rimphony_b200_last_kernel_ms(int device, float out_ms[4]);

/* Measured FP64 FMA throughput of the device (TFLOP/s, best of 5 runs of a
 * register-resident DFMA kernel): the roofline denominator for these kernels,
 * which are bound by the FP64 pipe of the CUDA cores. */
int rimphony_b200_fp64_peak_tflops(int device, double *out_tflops);

/* Number of kernels this library has launched since it was loaded. */
uint64_t rimphony_b200_kernel_launch_count(void);

int rimphony_b200_device_count(void);
int rimphony_b200_abi_version(void);
const char *rimphony_b200_last_error(void);

/* Free every device buffer, stream and event the library holds. */
void rimphony_b200_shutdown(void);

#ifdef __cplusplus
}
#endif
#endif
