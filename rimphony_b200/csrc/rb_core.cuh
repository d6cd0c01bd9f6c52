// rb_core.cuh -- warp-cooperative Gauss-Kronrod quadrature for sm_100a.
//
// One warp owns one parameter point.  A 31-point Gauss-Kronrod application
// puts one node on each of lanes 0..30 (lane 31 carries weight zero) and
// reduces with __shfl_xor_sync; the adaptive bisection logic above it is
// warp-uniform scalar code whose interval list lives in shared memory.
//
// Replaces (reference file:line):
//   src/gsl.rs:169-180   gsl_integration_qag(key = 3)  -> qag_joint<>
//   src/gsl.rs:246       gsl_deriv_central             -> deriv_central_joint<>
// The numerical semantics (error rescaling, round-off detection, termination)
// follow QUADPACK's QAG as restated in SURVEY.md Appendix A; what is new is
// that several integrands ("node values") share one set of nodes and are
// converged together ("accumulators"), see DESIGN.md section 4.
//
// The same header compiles under plain g++ with -DRB_HOST_EMU: the lane
// dimension then becomes an explicit loop.  That build exists only for the
// development harness under tests/hostemu/ and is never part of the product.
#pragma once

#include <float.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define RB_FN __device__ __forceinline__
#define RB_HD __host__ __device__ __forceinline__
#define RB_FN_NOINLINE static __device__ __noinline__
#define RB_MFN_NOINLINE __device__ __noinline__
#define RB_TABLE static __constant__ // not const: a const table is folded into literals, and every FP64 literal costs two UMOVs
#define RB_DEVICE_BUILD 1
#else
#ifndef RB_HOST_EMU
#error "rb_core.cuh needs nvcc (product) or -DRB_HOST_EMU (development harness)"
#endif
#define RB_FN inline
#define RB_HD inline
#define RB_FN_NOINLINE inline __attribute__((noinline))
#define RB_MFN_NOINLINE inline __attribute__((noinline))
#define RB_TABLE static const
#endif

namespace rb {

// Out-of-line double-precision transcendentals.  The product kernels are bound by instruction
// fetch (profiles/): every inlined log/exp/cbrt costs 40-80 SASS instructions per call site, and
// the hot loop has a dozen of them.  One shared copy each keeps the loop in the instruction cache.
//
// RB_LEAN_MATH (defined by the Symphony translation units inst_k*_symfast.cu / inst_k*_sym.cu, by the product
// Heyvaerts units inst_k*_heyfast.cu and by the host harness; only inst_k*_hey.cu, with the faithful Heyvaerts,
// normalisation and dist_eval kernels, keep the CUDA library's functions): the kernels issue
// 0.7-1.2 instructions per cycle and SM, every instruction counts the same, and ncu's source page says a
// quarter of them is spent on IEEE-correct division (16 instructions each, 26-36 per node), on libdevice's
// log/exp (87 / 64 instructions, two of every three of them moves of literal constants into uniform
// registers) and on square roots.  The lean versions: division = a * rcp(b) with rcp from MUFU.RCP64H and one
// cubic Newton step (6 instructions, <= 1.5 ulp; b = 0, |b| < 2^-1022, |b| = inf give NaN, |b| > 2^1022 gives
// 0: no node of a quadrature rule depends on those), exp and log with their coefficients read from the
// constant bank as instruction operands (32 / 38 instructions, <= 2 ulp).
// the two words of a double
RB_FN int rb_hi32(double x)
{
#ifdef RB_DEVICE_BUILD
    return __double2hiint(x);
#else
    int64_t u;
    memcpy(&u, &x, 8);
    return (int)(u >> 32);
#endif
}
RB_FN int rb_lo32(double x)
{
#ifdef RB_DEVICE_BUILD
    return __double2loint(x);
#else
    int64_t u;
    memcpy(&u, &x, 8);
    return (int)(u & 0xffffffff);
#endif
}
RB_FN double rb_from_hilo(int hi, int lo)
{
#ifdef RB_DEVICE_BUILD
    return __hiloint2double(hi, lo);
#else
    const uint64_t u = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo;
    double x;
    memcpy(&x, &u, 8);
    return x;
#endif
}

#if defined(RB_LEAN_MATH)
#ifdef RB_DEVICE_BUILD
RB_FN double rb_rcp_seed(double b)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
    return r;
}
#else
// what MUFU.RCP64H returns, to 2^-23: subnormal arguments and results are flushed to zero
inline double rb_rcp_seed(double b)
{
    if (b != b)
        return b;
    const double ab = fabs(b);
    if (ab < DBL_MIN)
        return copysign(INFINITY, b);
    if (ab > 0x1p1022)
        return copysign(0.0, b);
    return (1.0 / b) * (1.0 + 0x1p-24);
}
#endif
RB_FN double rb_rcp(double b)
{
    const double r = rb_rcp_seed(b);
    double e = fma(-b, r, 1.0);
    e = fma(e, e, e);
    return fma(r, e, r);
}
RB_FN double rb_div(double a, double b) { return a * rb_rcp(b); }

// Square root from MUFU.RSQ64H (2^-22) and two coupled Newton steps on (sqrt x, 1 / (2 sqrt x)): 11 instructions
// where the IEEE-correct sequence with its range check takes 19; <= 1 ulp.  +-0 and subnormal arguments give 0,
// negative ones NaN; +inf gives NaN (no caller can tell: an infinite node value ends in NaN either way).
#ifdef RB_DEVICE_BUILD
RB_FN double rb_rsqrt_seed(double x)
{
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
}
#else
inline double rb_rsqrt_seed(double x)
{
    if (x != x || x < 0.0)
        return NAN;
    if (x < DBL_MIN)
        return INFINITY;
    if (x == INFINITY)
        return 0.0;
    return (1.0 / sqrt(x)) * (1.0 + 0x1p-23);
}
#endif
RB_FN double rb_sqrt(double x)
{
    const double y = rb_rsqrt_seed(x);
    double g = x * y, h = 0.5 * y;
    const double r = fma(-h, g, 0.5);
    g = fma(g, r, g);
    h = fma(h, r, h);
    const double d = fma(-g, g, x);
    g = fma(d, h, g);
    return (fabs(x) < DBL_MIN) ? 0.0 : g;
}

// exp(r) on |r| <= ln(2)/2: Taylor to r^13 (remainder 4e-18), highest power first
RB_TABLE double EXP_POLY[14] = {1.0 / 6227020800.0, 1.0 / 479001600.0, 1.0 / 39916800.0, 1.0 / 3628800.0, 1.0 / 362880.0,
                                1.0 / 40320.0,      1.0 / 5040.0,      1.0 / 720.0,      1.0 / 120.0,     1.0 / 24.0,
                                1.0 / 6.0,          0.5,               1.0,              1.0};
// log2(e), -ln(2) in two parts: read from the table like the coefficients (a literal costs two UMOVs)
RB_TABLE double LN2_CONST[3] = {1.4426950408889634074, -6.93147180559945286227e-01, -2.31904681384629955842e-17};
// log(m) = 2 atanh(f), f = (m - 1) / (m + 1), |f| <= 0.1716: 2 f + f^3 (2/3 + 2/5 f^2 + ... + 2/23 f^20)
RB_TABLE double LOG_POLY[11] = {2.0 / 23.0, 2.0 / 21.0, 2.0 / 19.0, 2.0 / 17.0, 2.0 / 15.0, 2.0 / 13.0,
                                2.0 / 11.0, 2.0 / 9.0,  2.0 / 7.0,  2.0 / 5.0,  2.0 / 3.0};

#ifdef RB_DEVICE_BUILD
static __device__ __noinline__
#else
inline
#endif
double rb_exp(double x)
{
    // beyond +-1400 the result is 0 or inf whatever the argument (the comparisons let NaN through)
    x = (x > 1400.0) ? 1400.0 : x;
    x = (x < -1400.0) ? -1400.0 : x;
    const double magic = 6755399441055744.0; // 1.5 * 2^52: the integer lands in the low word
    double t = fma(x, LN2_CONST[0], magic);
    const int k = rb_lo32(t);
    t -= magic;
    double r = fma(t, LN2_CONST[1], x);
    r = fma(t, LN2_CONST[2], r);
    double p = EXP_POLY[0];
#pragma unroll
    for (int i = 1; i < 14; i++)
        p = fma(p, r, EXP_POLY[i]);
    // 2^k in two factors (|k| <= 2020), so that results down to the subnormals and overflow come out right
    const int k1 = k >> 1, k2 = k - k1;
    p *= rb_from_hilo((k1 + 1023) << 20, 0);
    return p * rb_from_hilo((k2 + 1023) << 20, 0);
}

#ifdef RB_DEVICE_BUILD
static __device__ __noinline__
#else
inline
#endif
double rb_log(double x)
{
    int hi = rb_hi32(x);
    // zero, negative, subnormal, infinite and NaN arguments: the library function
    if ((unsigned)(hi - 0x00100000) >= 0x7fe00000u)
        return log(x);
    int e = (hi >> 20) - 1023;
    hi = (hi & 0x000fffff) | 0x3ff00000;
    if (hi >= 0x3ff6a09f) { // m in [sqrt(1/2), sqrt(2))
        hi -= 0x00100000;
        e += 1;
    }
    const double m = rb_from_hilo(hi, rb_lo32(x));
    const double f = (m - 1.0) * rb_rcp(m + 1.0);
    const double f2 = f * f;
    double p = LOG_POLY[0];
#pragma unroll
    for (int i = 1; i < 11; i++)
        p = fma(p, f2, LOG_POLY[i]);
    const double ke = (double)e;
    const double lm = fma(f * f2, p, f + f);
    return fma(-ke, LN2_CONST[1], fma(-ke, LN2_CONST[2], lm));
}
#ifdef RB_DEVICE_BUILD
static __device__ __noinline__ double rb_cbrt(double x) { return cbrt(x); }
#else
inline double rb_cbrt(double x) { return cbrt(x); }
#endif
#else // !RB_LEAN_MATH
RB_FN double rb_rcp(double b) { return 1.0 / b; }
RB_FN double rb_div(double a, double b) { return a / b; }
RB_FN double rb_sqrt(double x) { return sqrt(x); }
#ifdef RB_DEVICE_BUILD // measured: +9 % sets/s over inlining
static __device__ __noinline__ double rb_log(double x) { return log(x); }
static __device__ __noinline__ double rb_exp(double x) { return exp(x); }
static __device__ __noinline__ double rb_cbrt(double x) { return cbrt(x); }
#else
RB_FN double rb_log(double x) { return log(x); }
RB_FN double rb_exp(double x) { return exp(x); }
RB_FN double rb_cbrt(double x) { return cbrt(x); }
#endif
#endif

constexpr double kPi = 3.14159265358979323846264338327950288;
constexpr double kTwoPi = 2.0 * kPi;
// src/lib.rs:58-67
constexpr double kMassElectron = 9.1093826e-28;
constexpr double kSpeedLight = 2.99792458e10;
constexpr double kElectronCharge = 4.80320680e-10;

// per-point status bits (include/rimphony_b200.h RIMPHONY_B200_STATUS_*)
constexpr unsigned kStatusNaN = 1u;        // at least one coefficient is NaN
constexpr unsigned kStatusCapHit = 2u;     // an interval list filled up
constexpr unsigned kStatusNormFailed = 4u; // normalisation integral failed
constexpr unsigned kStatusRerouted = 8u;   // computed with the reference's exact rule sequence (fidelity guard)
constexpr unsigned kStatusRefDiverges = 16u; // rho: NaN because the reference's quadrature fails here (rb_heyfast.cuh)

// ---------------------------------------------------------------------------
// Gauss-Kronrod (15, 31) tables laid out by lane: lane l < 31 holds the node
// x = LANE_X[l] in [-1, 1]; lanes 0..14 are the negative abscissae, lane 15 the
// centre, lanes 16..30 the positive ones.  LANE_WG is the weight of the
// embedded 15-point Gauss rule (zero on the Kronrod-only nodes).
RB_TABLE double LANE_X[32] = {
    -0.998002298693397060285172840152271, -0.987992518020485428489565718586613,
    -0.967739075679139134257347978784337, -0.937273392400705904307758947710209,
    -0.897264532344081900882509656454496, -0.848206583410427216200648320774217,
    -0.790418501442465932967649294817947, -0.724417731360170047416186054613938,
    -0.650996741297416970533735895313275, -0.570972172608538847537226737253911,
    -0.485081863640239680693655740232351, -0.394151347077563369897207370981045,
    -0.299180007153168812166780024266389, -0.201194093997434522300628303394596,
    -0.101142066918717499027074231447392, 0.0,
    0.101142066918717499027074231447392,  0.201194093997434522300628303394596,
    0.299180007153168812166780024266389,  0.394151347077563369897207370981045,
    0.485081863640239680693655740232351,  0.570972172608538847537226737253911,
    0.650996741297416970533735895313275,  0.724417731360170047416186054613938,
    0.790418501442465932967649294817947,  0.848206583410427216200648320774217,
    0.897264532344081900882509656454496,  0.937273392400705904307758947710209,
    0.967739075679139134257347978784337,  0.987992518020485428489565718586613,
    0.998002298693397060285172840152271,  0.0};

RB_TABLE double LANE_WK[32] = {
    0.005377479872923348987792051430128, 0.015007947329316122538374763075807,
    0.025460847326715320186874001019653, 0.035346360791375846222037948478360,
    0.044589751324764876608227299373280, 0.053481524690928087265343147239430,
    0.062009567800670640285139230960803, 0.069854121318728258709520077099147,
    0.076849680757720378894432777482659, 0.083080502823133021038289247286104,
    0.088564443056211770647275443693774, 0.093126598170825321225486872747346,
    0.096642726983623678505179907627589, 0.099173598721791959332393173484603,
    0.100769845523875595044946662617570, 0.101330007014791549017374792767493,
    0.100769845523875595044946662617570, 0.099173598721791959332393173484603,
    0.096642726983623678505179907627589, 0.093126598170825321225486872747346,
    0.088564443056211770647275443693774, 0.083080502823133021038289247286104,
    0.076849680757720378894432777482659, 0.069854121318728258709520077099147,
    0.062009567800670640285139230960803, 0.053481524690928087265343147239430,
    0.044589751324764876608227299373280, 0.035346360791375846222037948478360,
    0.025460847326715320186874001019653, 0.015007947329316122538374763075807,
    0.005377479872923348987792051430128, 0.0};

RB_TABLE double LANE_WG[32] = {
    0.0, 0.030753241996117268354628393577204,
    0.0, 0.070366047488108124709267416450667,
    0.0, 0.107159220467171935011869546685869,
    0.0, 0.139570677926154314447804794511028,
    0.0, 0.166269205816993933553200860481209,
    0.0, 0.186161000015562211026800561866423,
    0.0, 0.198431485327111576456118326443839,
    0.0, 0.202578241925561272880620199967519,
    0.0, 0.198431485327111576456118326443839,
    0.0, 0.186161000015562211026800561866423,
    0.0, 0.166269205816993933553200860481209,
    0.0, 0.139570677926154314447804794511028,
    0.0, 0.107159220467171935011869546685869,
    0.0, 0.070366047488108124709267416450667,
    0.0, 0.030753241996117268354628393577204,
    0.0, 0.0};

// ---------------------------------------------------------------------------
// Warp context: the lane's own node and weights, plus work counters.
struct Warp {
#ifdef RB_DEVICE_BUILD
    int lane;
    double xk, wk, wg;
#endif
    unsigned n_apply_lanes; // GK31 applications with nodes across lanes
    unsigned status;
    int max_list; // largest interval list seen (diagnostics)

    RB_FN void init()
    {
#ifdef RB_DEVICE_BUILD
        lane = threadIdx.x & 31;
        xk = LANE_X[lane];
        wk = LANE_WK[lane];
        wg = LANE_WG[lane];
#endif
        n_apply_lanes = 0;
        status = 0;
        max_list = 0;
    }
};

#ifdef RB_DEVICE_BUILD
RB_FN double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
RB_FN void warp_fence() { __syncwarp(); }
#else
RB_FN void warp_fence() {}
#endif

// The values of NV integrands at the 31 nodes of one rule application.
template <int NV>
struct LaneVals {
#ifdef RB_DEVICE_BUILD
    double v[NV];
    RB_FN void set(const Warp &w, int node, const double (&vals)[NV])
    {
        if (w.lane == node) {
#pragma unroll
            for (int c = 0; c < NV; c++)
                v[c] = vals[c];
        }
    }
    RB_FN void clear()
    {
#pragma unroll
        for (int c = 0; c < NV; c++)
            v[c] = 0.0;
    }
#else
    double v[32][NV];
    RB_FN void set(const Warp &, int node, const double (&vals)[NV])
    {
        for (int c = 0; c < NV; c++)
            v[node][c] = vals[c];
    }
    RB_FN void clear()
    {
        for (int l = 0; l < 32; l++)
            for (int c = 0; c < NV; c++)
                v[l][c] = 0.0;
    }
#endif
};

template <int NV>
struct GKOut {
    double r[NV];    // Kronrod estimate of the integral
    double e[NV];    // rescaled error estimate
    double rabs[NV]; // integral of |f|
    double rasc[NV]; // integral of |f - mean|
};

// QUADPACK's error heuristic (SURVEY.md Appendix A).
RB_FN double rescale_error(double err, double result_abs, double result_asc)
{
    err = fabs(err);
    if (result_asc != 0.0 && err != 0.0) {
        const double q = 200.0 * err / result_asc;
        const double scale = q * sqrt(q); // q^1.5
        err = (scale < 1.0) ? result_asc * scale : result_asc;
    }
    if (result_abs > DBL_MIN / (50.0 * DBL_EPSILON)) {
        const double min_err = 50.0 * DBL_EPSILON * result_abs;
        if (min_err > err)
            err = min_err;
    }
    return err;
}

template <int NV>
RB_FN void gk31_reduce(const Warp &w, const LaneVals<NV> &lv, double half_length, GKOut<NV> &o)
{
    const double abs_half = fabs(half_length);
#pragma unroll
    for (int c = 0; c < NV; c++) {
#ifdef RB_DEVICE_BUILD
        const double f = lv.v[c];
        const double k = warp_sum(w.wk * f);
        const double g = warp_sum(w.wg * f);
        const double a = warp_sum(w.wk * fabs(f));
        const double mean = 0.5 * k;
        const double asc = warp_sum(w.wk * fabs(f - mean));
#else
        double k = 0, g = 0, a = 0, asc = 0;
        for (int l = 0; l < 31; l++) {
            k += LANE_WK[l] * lv.v[l][c];
            g += LANE_WG[l] * lv.v[l][c];
            a += LANE_WK[l] * fabs(lv.v[l][c]);
        }
        const double mean = 0.5 * k;
        for (int l = 0; l < 31; l++)
            asc += LANE_WK[l] * fabs(lv.v[l][c] - mean);
#endif
        const double err = (k - g) * half_length;
        o.r[c] = k * half_length;
        o.rabs[c] = a * abs_half;
        o.rasc[c] = asc * abs_half;
        o.e[c] = rescale_error(err, o.rabs[c], o.rasc[c]);
    }
}

// One GK31 application with the nodes spread across lanes.  F::eval(x, out[NV])
// is ordinary per-lane scalar code.
template <int NV, class F>
RB_FN void gk31_lanes(Warp &w, F &f, double a, double b, GKOut<NV> &o)
{
    const double center = 0.5 * (a + b);
    const double half_length = 0.5 * (b - a);
    LaneVals<NV> lv;
#ifdef RB_DEVICE_BUILD
    f.eval(center + half_length * w.xk, lv.v);
    if (w.lane == 31) {
#pragma unroll
        for (int c = 0; c < NV; c++)
            lv.v[c] = 0.0;
    }
#else
    for (int l = 0; l < 31; l++)
        f.eval(center + half_length * LANE_X[l], lv.v[l]);
    for (int c = 0; c < NV; c++)
        lv.v[31][c] = 0.0;
#endif
    w.n_apply_lanes++;
    gk31_reduce<NV>(w, lv, half_length, o);
}

// One GK31 application whose 31 node values are themselves warp-collective
// computations (an inner adaptive integral): nodes are visited one after the
// other, the (warp-uniform) result of node j is parked on lane j, and the same
// lane-parallel reduction finishes the rule.
template <int NV, class F>
RB_FN void gk31_seq(Warp &w, F &f, double a, double b, GKOut<NV> &o)
{
    const double center = 0.5 * (a + b);
    const double half_length = 0.5 * (b - a);
    LaneVals<NV> lv;
    lv.clear();
#pragma unroll 1
    for (int j = 0; j < 31; j++) {
        double tmp[NV];
        f.eval_collective(w, center + half_length * LANE_X[j], tmp);
        lv.set(w, j, tmp);
    }
    gk31_reduce<NV>(w, lv, half_length, o);
}

// Adapters so that qag_joint<> can be written once.
template <int NV, class F>
struct ApplyLanes {
    F &f;
    RB_FN void operator()(Warp &w, double a, double b, GKOut<NV> &o) { gk31_lanes<NV, F>(w, f, a, b, o); }
};
template <int NV, class F>
struct ApplySeq {
    F &f;
    RB_FN void operator()(Warp &w, double a, double b, GKOut<NV> &o) { gk31_seq<NV, F>(w, f, a, b, o); }
};

// ---------------------------------------------------------------------------
// Interval list of one adaptive integration (shared memory on the device).
template <int NV>
struct IntervalList {
    double *a;  // [cap]
    double *b;  // [cap]
    double *r;  // [NV][cap]
    double *e;  // [NV][cap]
    int cap;
    int size;
    int max_size; // high-water mark, for diagnostics

    static constexpr int doubles_per_interval = 2 + 2 * NV;

    RB_FN void bind(double *storage, int capacity)
    {
        a = storage;
        b = storage + capacity;
        r = storage + 2 * capacity;
        e = storage + (2 + NV) * capacity;
        cap = capacity;
        size = 0;
        max_size = 0;
    }

    RB_FN void store(const Warp &w, int i, double lo, double hi, const GKOut<NV> &o)
    {
#ifdef RB_DEVICE_BUILD
        if (w.lane == 0)
#endif
        {
            a[i] = lo;
            b[i] = hi;
#pragma unroll
            for (int c = 0; c < NV; c++) {
                r[c * cap + i] = o.r[c];
                e[c * cap + i] = o.e[c];
            }
        }
    }
};

// Accumulator policies: which node value feeds accumulator c, and over which
// part of the integration range.
constexpr int kSideBoth = -1, kSideLeft = 0, kSideRight = 1;

template <int NV>
struct PolicyPlain {
    static constexpr int kNV = NV;
    static constexpr int kNA = NV;
    RB_FN static int val(int c) { return c; }
    RB_FN static int side(int) { return kSideBoth; }
};

// Symphony gamma integral, all six j/alpha integrands on shared nodes.  Node
// values: 0 j_I, 1 a_I, 2 j_Q, 3 a_Q, 4 j_V, 5 a_V.  The range is split at
// gamma_peak (symphony.rs:356-363): I and Q accumulate over both halves, the
// Stokes V integrands give one accumulator per lobe.
// Accumulators: 0..3 as above, 4 j_V(+), 5 a_V(+), 6 j_V(-), 7 a_V(-).
struct PolicySymphonySplit {
    static constexpr int kNV = 6;
    static constexpr int kNA = 8;
    RB_FN static int val(int c) { return c < 6 ? c : c - 2; }
    RB_FN static int side(int c) { return c < 4 ? kSideBoth : (c < 6 ? kSideRight : kSideLeft); }
};

constexpr int kChanActive = 0, kChanDone = 1, kChanFailed = 2, kChanIgnored = 3;

// Select the interval with the largest error estimate of node value `v`,
// restricted to one side of `split` when side >= 0.  Returns -1 if none.
template <int NV>
RB_FN int list_argmax(const Warp &w, const IntervalList<NV> &L, int v, int side, double split)
{
#ifdef RB_DEVICE_BUILD
    double best_e = -1.0;
    int best_i = 0x7fffffff;
    for (int i = w.lane; i < L.size; i += 32) {
        const double ei = L.e[v * L.cap + i];
        const bool ok = (side < 0) || ((L.a[i] >= split) == (side == kSideRight));
        if (ok && ei > best_e) {
            best_e = ei;
            best_i = i;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oe = __shfl_xor_sync(0xffffffffu, best_e, o);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        if (oe > best_e || (oe == best_e && oi < best_i)) {
            best_e = oe;
            best_i = oi;
        }
    }
    return best_e >= 0.0 ? best_i : -1;
#else
    double best_e = -1.0;
    int best_i = -1;
    for (int i = 0; i < L.size; i++) {
        const double ei = L.e[v * L.cap + i];
        const bool ok = (side < 0) || ((L.a[i] >= split) == (side == kSideRight));
        if (ok && ei > best_e) {
            best_e = ei;
            best_i = i;
        }
    }
    return best_i;
#endif
}

RB_FN bool subinterval_too_small(double a1, double a2, double b2)
{
    const double tmp = (1.0 + 100.0 * DBL_EPSILON) * (fabs(a2) + 1000.0 * DBL_MIN);
    return fabs(a1) <= tmp && fabs(b2) <= tmp;
}

// Adaptive GK31 integration of Policy::kNV integrands on shared nodes, with
// QUADPACK QAG semantics per accumulator (epsabs = 0):
//   * n_init = 1: plain QAG on [bounds[0], bounds[1]];
//   * n_init = 2: the list starts with [bounds[0], bounds[1]] and
//     [bounds[1], bounds[2]]; bounds[1] is the side split of the policy.
// `want` is the set of accumulators that must converge; the others are carried
// along.  result[c] is NaN for an accumulator whose integration failed (the
// reference maps every GSL error to NaN: symphony.rs:375-380, heyvaerts.rs:205-210).
// With a single accumulator this performs the same sequence of rule
// applications as gsl_integration_qag.
template <class Policy, class Apply>
RB_FN void qag_joint(Warp &w, Apply &apply, int n_init, const double *bounds, double epsrel,
                     IntervalList<Policy::kNV> &L, unsigned want, double (&result)[Policy::kNA])
{
    constexpr int NV = Policy::kNV;
    constexpr int NA = Policy::kNA;
    const double split = bounds[1];

    double area[NA], errsum[NA];
    double rabs0[NA], rasc0[NA];
    int state[NA];
    int rnd1[NA], rnd2[NA];

#pragma unroll
    for (int c = 0; c < NA; c++) {
        area[c] = 0.0;
        errsum[c] = 0.0;
        rabs0[c] = 0.0;
        rasc0[c] = 0.0;
        rnd1[c] = 0;
        rnd2[c] = 0;
        state[c] = ((want >> c) & 1u) ? kChanActive : kChanIgnored;
    }

    warp_fence(); // previous users of the list storage are done
    L.size = 0;
#pragma unroll 1
    for (int k = 0; k < n_init; k++) {
        GKOut<NV> o;
        apply(w, bounds[k], bounds[k + 1], o);
        L.store(w, k, bounds[k], bounds[k + 1], o);
        const int sd = (n_init == 2) ? k : 0;
#pragma unroll
        for (int c = 0; c < NA; c++) {
            const int ps = Policy::side(c);
            if (ps == kSideBoth || ps == sd) {
                const int v = Policy::val(c);
                area[c] += o.r[v];
                errsum[c] += o.e[v];
                rabs0[c] += o.rabs[v];
                rasc0[c] += o.rasc[v];
            }
        }
    }
    L.size = n_init;
    warp_fence();

    int n_active = 0;
#pragma unroll
    for (int c = 0; c < NA; c++) {
        if (state[c] != kChanActive)
            continue;
        const double tol = epsrel * fabs(area[c]);
        const double round_off = 50.0 * DBL_EPSILON * rabs0[c];
        if (errsum[c] <= round_off && errsum[c] > tol)
            state[c] = kChanFailed; // GSL_EROUND on the first application
        else if ((errsum[c] <= tol && errsum[c] != rasc0[c]) || errsum[c] == 0.0)
            state[c] = kChanDone;
        else if (!(errsum[c] == errsum[c]) || !(area[c] == area[c]))
            state[c] = kChanFailed; // NaN integrand: GSL ends in EFAILED
        else
            n_active++;
    }

    int iteration = 1;
    while (n_active > 0) {
        if (L.size >= L.cap) {
            // The reference's workspaces (1000..5000 intervals) are never a
            // binding limit; ours is small.  Keep the current estimate and flag it.
            w.status |= kStatusCapHit;
            break;
        }

        // the accumulator that is furthest from its tolerance drives the bisection
        int cw = -1;
        double worst = -1.0;
#pragma unroll
        for (int c = 0; c < NA; c++) {
            if (state[c] != kChanActive)
                continue;
            const double tol = epsrel * fabs(area[c]);
            const double ratio = (tol > 0.0) ? errsum[c] / tol : DBL_MAX;
            if (ratio > worst) {
                worst = ratio;
                cw = c;
            }
        }

        const int vw = Policy::val(cw);
        const int i_max = list_argmax<NV>(w, L, vw, Policy::side(cw), split);
        if (i_max < 0) {
            state[cw] = kChanFailed;
            n_active--;
            continue;
        }

        const double a_i = L.a[i_max], b_i = L.b[i_max];
        const double a1 = a_i, b1 = 0.5 * (a_i + b_i), a2 = b1, b2 = b_i;
        const int sd = (n_init == 2 && a_i >= split) ? kSideRight : kSideLeft;

        double r_i[NV], e_i[NV];
#pragma unroll
        for (int v = 0; v < NV; v++) {
            r_i[v] = L.r[v * L.cap + i_max];
            e_i[v] = L.e[v * L.cap + i_max];
        }
        warp_fence();

        GKOut<NV> o12[2];
#pragma unroll 1
        for (int h = 0; h < 2; h++)
            apply(w, h ? a2 : a1, h ? b2 : b1, o12[h]);
        const GKOut<NV> &o1 = o12[0];
        const GKOut<NV> &o2 = o12[1];

        const bool too_small = subinterval_too_small(a1, a2, b2);

#pragma unroll
        for (int c = 0; c < NA; c++) {
            const int ps = Policy::side(c);
            if (!(ps == kSideBoth || ps == sd || n_init == 1))
                continue;
            const int v = Policy::val(c);
            const double area12 = o1.r[v] + o2.r[v];
            const double error12 = o1.e[v] + o2.e[v];
            errsum[c] += (error12 - e_i[v]);
            area[c] += area12 - r_i[v];

            if (state[c] != kChanActive)
                continue;

            // QUADPACK's round-off heuristics judge whether bisecting the
            // integrand's OWN worst interval still helps; they only make sense
            // for the accumulator that chose this interval.
            if (c == cw && o1.rasc[v] != o1.e[v] && o2.rasc[v] != o2.e[v]) {
                const double delta = r_i[v] - area12;
                if (fabs(delta) <= 1.0e-5 * fabs(area12) && error12 >= 0.99 * e_i[v])
                    rnd1[c]++;
                if (iteration >= 10 && error12 > e_i[v])
                    rnd2[c]++;
            }

            const double tol = epsrel * fabs(area[c]);
            if (errsum[c] <= tol) {
                state[c] = kChanDone;
                n_active--;
            } else if (!(errsum[c] > tol)) {
                state[c] = kChanFailed; // NaN
                n_active--;
            } else if (c == cw && (rnd1[c] >= 6 || rnd2[c] >= 20 || too_small)) {
                state[c] = kChanFailed; // GSL_EROUND / GSL_ESING
                n_active--;
            }
        }

        // replace the bisected interval by its halves, larger error first
        if (o2.e[vw] > o1.e[vw]) {
            L.store(w, i_max, a2, b2, o2);
            L.store(w, L.size, a1, b1, o1);
        } else {
            L.store(w, i_max, a1, b1, o1);
            L.store(w, L.size, a2, b2, o2);
        }
        L.size++;
        if (L.size > L.max_size)
            L.max_size = L.size;
        warp_fence();
        iteration++;
    }

    if (L.size > w.max_list)
        w.max_list = L.size;
#pragma unroll
    for (int c = 0; c < NA; c++)
        result[c] = (state[c] == kChanFailed) ? NAN : area[c];
}

// gsl_deriv_central restated for NV functions evaluated together.  With
// REFINE (single-function, faithful mode) the optimal-step retry of GSL is
// performed; without it only the first 5-point estimate is used (the joint
// mode cannot pick a different h per function).
// Four-point evaluation of gsl's central_deriv: f at x-h, x+h, x-h/2, x+h/2.
template <int NV, class F>
RB_FN void deriv_probe(Warp &w, F &f, double x, double h, double (&fv)[4][NV])
{
#pragma unroll 1
    for (int k = 0; k < 4; k++) {
        const double off = (k == 0) ? -h : (k == 1) ? h : (k == 2) ? -h / 2 : h / 2;
        f.eval_collective(w, x + off, fv[k]);
    }
}

template <int NV, bool REFINE, class F>
RB_FN void deriv_central_joint(Warp &w, F &f, double x, double h, double (&result)[NV])
{
    double fv[4][NV]; // fm1, fp1, fmh, fph
    deriv_probe<NV, F>(w, f, x, h, fv);

    double round0 = 0, trunc0 = 0;
#pragma unroll
    for (int c = 0; c < NV; c++) {
        const double r3 = 0.5 * (fv[1][c] - fv[0][c]);
        const double r5 = (4.0 / 3.0) * (fv[3][c] - fv[2][c]) - (1.0 / 3.0) * r3;
        result[c] = r5 / h;
        if (REFINE && c == 0) {
            const double e3 = (fabs(fv[1][c]) + fabs(fv[0][c])) * DBL_EPSILON;
            const double e5 = 2.0 * (fabs(fv[3][c]) + fabs(fv[2][c])) * DBL_EPSILON + e3;
            const double q3 = fabs(r3 / h), q5 = fabs(r5 / h);
            const double dy = (q3 > q5 ? q3 : q5) * (fabs(x) / h) * DBL_EPSILON;
            trunc0 = fabs((r5 - r3) / h);
            round0 = fabs(e5 / h) + dy;
        }
    }

    if (REFINE) {
        const double error = round0 + trunc0;
        if (round0 < trunc0 && (round0 > 0 && trunc0 > 0)) {
            const double h_opt = h * cbrt(round0 / (2.0 * trunc0));
            deriv_probe<NV, F>(w, f, x, h_opt, fv);
            const double r3 = 0.5 * (fv[1][0] - fv[0][0]);
            const double r5 = (4.0 / 3.0) * (fv[3][0] - fv[2][0]) - (1.0 / 3.0) * r3;
            const double e3 = (fabs(fv[1][0]) + fabs(fv[0][0])) * DBL_EPSILON;
            const double e5 = 2.0 * (fabs(fv[3][0]) + fabs(fv[2][0])) * DBL_EPSILON + e3;
            const double q3 = fabs(r3 / h_opt), q5 = fabs(r5 / h_opt);
            const double dy = (q3 > q5 ? q3 : q5) * (fabs(x) / h_opt) * DBL_EPSILON;
            const double error_opt = fabs((r5 - r3) / h_opt) + fabs(e5 / h_opt) + dy;
            const double r_opt = r5 / h_opt;
            if (error_opt < error && fabs(r_opt - result[0]) < 4.0 * error)
                result[0] = r_opt;
        }
    }
}

} // namespace rb
