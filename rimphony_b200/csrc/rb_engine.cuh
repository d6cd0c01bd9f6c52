// rb_engine.cuh -- the compact warp-cooperative quadrature engine of the
// product ("fast") path.
//
// One warp owns one parameter point.  The building block is one 31-point
// Gauss-Kronrod application of up to eight integrands ("channels") that share
// their nodes:
//
//   * lanes-as-nodes: lane j evaluates every channel at node j and stores the
//     pre-weighted values  A = wk_j f_j  and  B = (wk_j - wg_j) f_j  into a
//     [channel][node] tile of the warp's shared memory;
//   * lanes-as-channels: lane L = 4 c + q then sums a quarter of channel c's row
//     (8 conflict-free LDS.64 per tile), two xor-shuffles finish the sums, and the
//     Kronrod estimate, the |K - G| error estimate and the acceptance test of
//     channel c are ordinary per-lane scalar code on lanes 4c..4c+3.
//
// So nothing on the bookkeeping side is unrolled over channels: eight integrals
// are converged by eight lane groups in SIMD, and a warp vote decides whether
// the panel is accepted or bisected.  The adaptive driver is "local" (a stack of
// pending panels in shared memory, each accepted on its own error estimate),
// which needs no interval list, no arg-max and no stored partial results.  The
// same driver runs both quadrature levels: at the outer level the 31 node values
// are themselves inner integrals, computed one after the other and parked in
// the outer tile.
//
// This replaces the reference's use of GSL QAG (src/gsl.rs:169-180) on the
// product path; the QUADPACK-faithful list-based driver (rb_core.cuh
// qag_joint<>) remains the parity anchor of MODE_FAITHFUL.  Design notes:
// DESIGN.md section 4.
//
// Like rb_core.cuh this header also compiles under g++ with -DRB_HOST_EMU
// (development harness only): lanes and channels become explicit loops.
#pragma once

#include "rb_core.cuh"

namespace rb {

constexpr int kEngChan = 8;         // channels per tile
constexpr int kEngRow = 36;         // padded row length: node j sits at column j + (j >> 3), so that the
                                    // four quarter rows of four channels hit 16 distinct 8-byte banks
constexpr int kEngStack = 24;       // pending panels per level
constexpr int kEngTile = 2 * kEngChan * kEngRow; // doubles per tile (A rows then B rows)
constexpr unsigned kAppBudget = 150000; // rule applications per point after which every panel is accepted as is
                                        // (status CAP_HIT): bounds the cost of a point whose integral does not converge

// per-warp shared-memory working set of one quadrature level; CH = channel rows of the tile (the Heyvaerts
// kernel has two integrands: a quarter of the shared memory, which is what bounds its CTAs per SM)
template <int CH>
struct EngLevelT {
    double tile[2 * CH * kEngRow];
    double stk_a[kEngStack];
    double stk_b[kEngStack];
    int stk_tag[kEngStack];
};
using EngLevel = EngLevelT<kEngChan>;

// Per-channel state: one register on the device (the lane's own channel), an
// array in the host emulation.
template <class T>
struct PerChan {
#ifdef RB_DEVICE_BUILD
    T v;
    RB_FN T &operator[](int) { return v; }
    RB_FN const T &operator[](int) const { return v; }
#else
    T v[kEngChan];
    RB_FN T &operator[](int c) { return v[c]; }
    RB_FN const T &operator[](int c) const { return v[c]; }
#endif
};

#ifdef RB_DEVICE_BUILD
// the body runs once, for the lane's own channel
#define RB_FOR_CHAN(c, nv) for (int c = (threadIdx.x & 31) >> 2, rb_once_ = 1; rb_once_ && c < (nv); rb_once_ = 0)
#else
#define RB_FOR_CHAN(c, nv) for (int c = 0; c < (nv); c++)
#endif

// Value of channel `c` made warp-uniform (read from the first lane of its group).
RB_FN double chan_get(const PerChan<double> &x, int c)
{
#ifdef RB_DEVICE_BUILD
    return __shfl_sync(0xffffffffu, x.v, 4 * c);
#else
    return x.v[c];
#endif
}

// Kronrod - Gauss weight difference per lane (B rows of the tile).
RB_TABLE double LANE_WD[32] = {
    0.005377479872923348987792051430128,  0.015007947329316122538374763075807 - 0.030753241996117268354628393577204,
    0.025460847326715320186874001019653,  0.035346360791375846222037948478360 - 0.070366047488108124709267416450667,
    0.044589751324764876608227299373280,  0.053481524690928087265343147239430 - 0.107159220467171935011869546685869,
    0.062009567800670640285139230960803,  0.069854121318728258709520077099147 - 0.139570677926154314447804794511028,
    0.076849680757720378894432777482659,  0.083080502823133021038289247286104 - 0.166269205816993933553200860481209,
    0.088564443056211770647275443693774,  0.093126598170825321225486872747346 - 0.186161000015562211026800561866423,
    0.096642726983623678505179907627589,  0.099173598721791959332393173484603 - 0.198431485327111576456118326443839,
    0.100769845523875595044946662617570,  0.101330007014791549017374792767493 - 0.202578241925561272880620199967519,
    0.100769845523875595044946662617570,  0.099173598721791959332393173484603 - 0.198431485327111576456118326443839,
    0.096642726983623678505179907627589,  0.093126598170825321225486872747346 - 0.186161000015562211026800561866423,
    0.088564443056211770647275443693774,  0.083080502823133021038289247286104 - 0.166269205816993933553200860481209,
    0.076849680757720378894432777482659,  0.069854121318728258709520077099147 - 0.139570677926154314447804794511028,
    0.062009567800670640285139230960803,  0.053481524690928087265343147239430 - 0.107159220467171935011869546685869,
    0.044589751324764876608227299373280,  0.035346360791375846222037948478360 - 0.070366047488108124709267416450667,
    0.025460847326715320186874001019653,  0.015007947329316122538374763075807 - 0.030753241996117268354628393577204,
    0.005377479872923348987792051430128,  0.0};

// The 15-point Kronrod extension of the 7-point Gauss rule (QUADPACK qk15), for the
// outer quadrature level, whose nodes are visited one after the other: node, Kronrod
// weight and Kronrod-minus-Gauss weight.
RB_TABLE double GK15_X[15] = {
    -0.991455371120812639206854697526329, -0.949107912342758524526189684047851,
    -0.864864423359769072789712788640926, -0.741531185599394439863864773280788,
    -0.586087235467691130294144838258730, -0.405845151377397166906606412076961,
    -0.207784955007898467600689403773245, 0.0,
    0.207784955007898467600689403773245,  0.405845151377397166906606412076961,
    0.586087235467691130294144838258730,  0.741531185599394439863864773280788,
    0.864864423359769072789712788640926,  0.949107912342758524526189684047851,
    0.991455371120812639206854697526329};
RB_TABLE double GK15_WK[15] = {
    0.022935322010529224963732008058970, 0.063092092629978553290700663189204,
    0.104790010322250183839876322541518, 0.140653259715525918745189590510238,
    0.169004726639267902826583426598550, 0.190350578064785409913256402421014,
    0.204432940075298892414161999234649, 0.209482141084727828012999174891714,
    0.204432940075298892414161999234649, 0.190350578064785409913256402421014,
    0.169004726639267902826583426598550, 0.140653259715525918745189590510238,
    0.104790010322250183839876322541518, 0.063092092629978553290700663189204,
    0.022935322010529224963732008058970};
RB_TABLE double GK15_WD[15] = {
    0.022935322010529224963732008058970, 0.063092092629978553290700663189204 - 0.129484966168869693270611432679082,
    0.104790010322250183839876322541518, 0.140653259715525918745189590510238 - 0.279705391489276667901467771423780,
    0.169004726639267902826583426598550, 0.190350578064785409913256402421014 - 0.381830050505118944950369775488975,
    0.204432940075298892414161999234649, 0.209482141084727828012999174891714 - 0.417959183673469387755102040816327,
    0.204432940075298892414161999234649, 0.190350578064785409913256402421014 - 0.381830050505118944950369775488975,
    0.169004726639267902826583426598550, 0.140653259715525918745189590510238 - 0.279705391489276667901467771423780,
    0.104790010322250183839876322541518, 0.063092092629978553290700663189204 - 0.129484966168869693270611432679082,
    0.022935322010529224963732008058970};

// The 7-point Kronrod extension of the 3-point Gauss rule, for narrow outer panels.
RB_TABLE double GK7_X[7] = {-0.9604912687080202834235071, -0.7745966692414833770358531, -0.4342437493468025580020715, 0.0,
                            0.4342437493468025580020715,  0.7745966692414833770358531,  0.9604912687080202834235071};
RB_TABLE double GK7_WK[7] = {0.1046562260264672651938239, 0.2684880898683334407285693, 0.4013974147759622229050518,
                             0.4509165386584741423451101, 0.4013974147759622229050518, 0.2684880898683334407285693,
                             0.1046562260264672651938239};
RB_TABLE double GK7_WD[7] = {0.1046562260264672651938239, 0.2684880898683334407285693 - 0.5555555555555555555555556,
                             0.4013974147759622229050518, 0.4509165386584741423451101 - 0.8888888888888888888888889,
                             0.4013974147759622229050518, 0.2684880898683334407285693 - 0.5555555555555555555555556,
                             0.1046562260264672651938239};

RB_FN int tile_col(int node) { return node + (node >> 3); }

// Store the node values of one lane (node = lane) into a tile, pre-weighted.
template <int NV, int CH = kEngChan>
RB_FN void tile_store(double *tile, const Warp &w, int node, const double (&vals)[NV])
{
#ifdef RB_DEVICE_BUILD
    const double wk = w.wk; // the lane's own weights live in registers
    const double wd = w.wk - w.wg;
#else
    (void)w;
    const double wk = LANE_WK[node];
    const double wd = LANE_WD[node];
#endif
    const int col = tile_col(node);
#pragma unroll
    for (int c = 0; c < NV; c++) {
        const double f = (node < 31) ? vals[c] : 0.0;
        tile[c * kEngRow + col] = wk * f;
        tile[(CH + c) * kEngRow + col] = wd * f;
    }
}

// --- two panels in one application --------------------------------------------------------
// The 32 lanes of one application can also carry two 15-point Kronrod panels (lanes 0-14 and
// 16-30; lanes 15 and 31 have weight 0).  The tile and the quarter-row sums of the reduction do
// not care which rule a lane belongs to: a lane stores its pre-weighted values, a pair of
// quarters is one panel.  Per-lane abscissa and weights of that layout; read with the lane as
// index, so they live in global memory (L1-cached) rather than in the constant bank, which
// serialises divergent indices.
#ifdef RB_DEVICE_BUILD
#define RB_LANE_TABLE static __device__ const
#else
#define RB_LANE_TABLE static const
#endif

#define RB_K15_ROW(T) T(0), T(1), T(2), T(3), T(4), T(5), T(6), T(7), T(8), T(9), T(10), T(11), T(12), T(13), T(14), 0.0

// the literal values (the RB_TABLE copies above are __constant__ and cannot initialise these)
#define RB_K15X(i) ((i) == 7 ? 0.0 : ((i) < 7 ? -1.0 : 1.0) * \
    ((i) == 0 || (i) == 14 ? 0.991455371120812639206854697526329 : (i) == 1 || (i) == 13 ? 0.949107912342758524526189684047851 : \
     (i) == 2 || (i) == 12 ? 0.864864423359769072789712788640926 : (i) == 3 || (i) == 11 ? 0.741531185599394439863864773280788 : \
     (i) == 4 || (i) == 10 ? 0.586087235467691130294144838258730 : (i) == 5 || (i) == 9 ? 0.405845151377397166906606412076961 : \
     0.207784955007898467600689403773245))
#define RB_K15WK(i) ((i) == 7 ? 0.209482141084727828012999174891714 : \
    ((i) == 0 || (i) == 14 ? 0.022935322010529224963732008058970 : (i) == 1 || (i) == 13 ? 0.063092092629978553290700663189204 : \
     (i) == 2 || (i) == 12 ? 0.104790010322250183839876322541518 : (i) == 3 || (i) == 11 ? 0.140653259715525918745189590510238 : \
     (i) == 4 || (i) == 10 ? 0.169004726639267902826583426598550 : (i) == 5 || (i) == 9 ? 0.190350578064785409913256402421014 : \
     0.204432940075298892414161999234649))
#define RB_K15WG(i) ((i) == 7 ? 0.417959183673469387755102040816327 : \
    ((i) == 1 || (i) == 13 ? 0.129484966168869693270611432679082 : (i) == 3 || (i) == 11 ? 0.279705391489276667901467771423780 : \
     (i) == 5 || (i) == 9 ? 0.381830050505118944950369775488975 : 0.0))
#define RB_K15WD(i) (RB_K15WK(i) - RB_K15WG(i))

RB_LANE_TABLE double L15_X[32] = {RB_K15_ROW(RB_K15X), RB_K15_ROW(RB_K15X)};
RB_LANE_TABLE double L15_WK[32] = {RB_K15_ROW(RB_K15WK), RB_K15_ROW(RB_K15WK)};
RB_LANE_TABLE double L15_WD[32] = {RB_K15_ROW(RB_K15WD), RB_K15_ROW(RB_K15WD)};

// Store the node values of lane `lane` with explicit weights (multi-panel layouts).
template <int NV, int CH = kEngChan>
RB_FN void tile_store_weighted(double *tile, int lane, double wk, double wd, const double (&vals)[NV])
{
    const int col = tile_col(lane);
#pragma unroll
    for (int c = 0; c < NV; c++) {
        const double f = (wk != 0.0) ? vals[c] : 0.0;
        tile[c * kEngRow + col] = wk * f;
        tile[(CH + c) * kEngRow + col] = wd * f;
    }
}

RB_FN double quad_error(double d, double a, double hl)
{
    const double rabs = a * fabs(hl);
    double err = fabs(d * hl);
    if (rabs != 0.0 && err != 0.0) {
        const double qq = 200.0 * rb_div(err, rabs);
        const double scale = qq * rb_sqrt(qq);
        err = (scale < 1.0) ? rabs * scale : rabs;
    }
    const double min_err = 50.0 * DBL_EPSILON * rabs;
    return (min_err > err) ? min_err : err;
}

// Reduce a tile that holds two 15-point panels (columns of quarters 0-1 and 2-3) of half-lengths
// hl0, hl1: per channel the estimates (r0, e0) and (r1, e1) of the two panels.
template <int CH = kEngChan>
RB_FN_NOINLINE void tile_reduce_pair(const double *tile, int nv, double hl0, double hl1, PerChan<double> &r0,
                                     PerChan<double> &e0, PerChan<double> &r1, PerChan<double> &e1)
{
#ifdef RB_DEVICE_BUILD
    const int lane = threadIdx.x & 31;
    const int c = lane >> 2, q = lane & 3;
    double k = 0.0, d = 0.0, a = 0.0;
    if (c < nv) {
        const double *ra = tile + c * kEngRow + 9 * q;
        const double *rb = ra + CH * kEngRow;
#pragma unroll
        for (int t = 0; t < 8; t++) {
            const double va = ra[t];
            k += va;
            a += fabs(va);
            d += rb[t];
        }
    }
    k += __shfl_xor_sync(0xffffffffu, k, 1);
    d += __shfl_xor_sync(0xffffffffu, d, 1);
    a += __shfl_xor_sync(0xffffffffu, a, 1);
    const bool second = (q & 2) != 0;
    const double my_hl = second ? hl1 : hl0;
    const double my_r = k * my_hl;
    const double my_e = quad_error(d, a, my_hl);
    const double ot_r = __shfl_xor_sync(0xffffffffu, my_r, 2);
    const double ot_e = __shfl_xor_sync(0xffffffffu, my_e, 2);
    r0.v = second ? ot_r : my_r;
    e0.v = second ? ot_e : my_e;
    r1.v = second ? my_r : ot_r;
    e1.v = second ? my_e : ot_e;
#else
    for (int c = 0; c < nv; c++) {
        for (int p = 0; p < 2; p++) {
            double k = 0.0, d = 0.0, a = 0.0;
            for (int q = 2 * p; q < 2 * p + 2; q++) {
                double kq = 0.0, dq = 0.0, aq = 0.0;
                for (int t = 0; t < 8; t++) {
                    const double va = tile[c * kEngRow + 9 * q + t];
                    kq += va;
                    aq += fabs(va);
                    dq += tile[(CH + c) * kEngRow + 9 * q + t];
                }
                k += kq;
                d += dq;
                a += aq;
            }
            const double hl = p ? hl1 : hl0;
            (p ? r1 : r0).v[c] = k * hl;
            (p ? e1 : e0).v[c] = quad_error(d, a, hl);
        }
    }
#endif
}

template <int CH = kEngChan>
RB_FN void tile_clear(const Warp &w, double *tile)
{
#ifdef RB_DEVICE_BUILD
    for (int i = w.lane; i < 2 * CH * kEngRow; i += 32)
        tile[i] = 0.0;
#else
    (void)w;
    for (int i = 0; i < 2 * CH * kEngRow; i++)
        tile[i] = 0.0;
#endif
}

// Reduce a tile: per channel the Kronrod estimate r of the integral over a panel
// of half-length `hl` and an error estimate e.  The estimate is QUADPACK's
// (200 |K - G| / scale)^1.5 heuristic with the integral of |f| as the scale (the
// reference's second pass for the integral of |f - mean| is not needed at the
// tolerances of this path), floored at 50 ulp of the integral of |f|.
template <int CH = kEngChan>
RB_FN_NOINLINE void tile_reduce(const double *tile, int nv, double hl, PerChan<double> &r, PerChan<double> &e)
{
#ifdef RB_DEVICE_BUILD
    const int lane = threadIdx.x & 31;
    const int c = lane >> 2, q = lane & 3;
    double k = 0.0, d = 0.0, a = 0.0;
    if (c < nv) {
        const double *ra = tile + c * kEngRow + 9 * q;
        const double *rb = ra + CH * kEngRow;
#pragma unroll
        for (int t = 0; t < 8; t++) {
            const double va = ra[t];
            k += va;
            a += fabs(va);
            d += rb[t];
        }
    }
    k += __shfl_xor_sync(0xffffffffu, k, 1);
    d += __shfl_xor_sync(0xffffffffu, d, 1);
    a += __shfl_xor_sync(0xffffffffu, a, 1);
    k += __shfl_xor_sync(0xffffffffu, k, 2);
    d += __shfl_xor_sync(0xffffffffu, d, 2);
    a += __shfl_xor_sync(0xffffffffu, a, 2);
    {
#else
    for (int c = 0; c < nv; c++) {
        double k = 0.0, d = 0.0, a = 0.0;
        for (int q = 0; q < 4; q++) {
            double kq = 0.0, dq = 0.0, aq = 0.0;
            for (int t = 0; t < 8; t++) {
                const double va = tile[c * kEngRow + 9 * q + t];
                kq += va;
                aq += fabs(va);
                dq += tile[(CH + c) * kEngRow + 9 * q + t];
            }
            k += kq;
            d += dq;
            a += aq;
        }
#endif
        const double ahl = fabs(hl);
        const double rabs = a * ahl;
        double err = fabs(d * hl);
        if (rabs != 0.0 && err != 0.0) {
            const double qq = 200.0 * rb_div(err, rabs);
            const double scale = qq * rb_sqrt(qq);
            err = (scale < 1.0) ? rabs * scale : rabs;
        }
        const double min_err = 50.0 * DBL_EPSILON * rabs;
        if (min_err > err)
            err = min_err;
        r[c] = k * hl;
        e[c] = err;
    }
}

// The outer level without a tile: its node values (inner integrals) arrive one after the other, and what the
// rule needs of them are three sums per channel -- sum wk G (Kronrod), sum (wk - wg) G (Kronrod - Gauss) and
// sum |wk G| -- so they are accumulated as they arrive instead of being parked and reduced (4.6 KB of shared
// memory per warp less: the Symphony kernel's CTAs per SM were bound by it).
struct OuterAcc {
    double k[kEngChan], d[kEngChan], a[kEngChan];
};
struct OuterLevel {
    OuterAcc acc;
    double stk_a[kEngStack];
    double stk_b[kEngStack];
    int stk_tag[kEngStack];
};
RB_FN void acc_clear(const Warp &w, OuterAcc &acc)
{
#ifdef RB_DEVICE_BUILD
    if (w.lane < kEngChan)
        acc.k[w.lane] = 0.0;
    else if (w.lane < 2 * kEngChan)
        acc.d[w.lane - kEngChan] = 0.0;
    else if (w.lane < 3 * kEngChan)
        acc.a[w.lane - 2 * kEngChan] = 0.0;
#else
    (void)w;
    for (int i = 0; i < kEngChan; i++)
        acc.k[i] = acc.d[i] = acc.a[i] = 0.0;
#endif
}
// one node value of channel c (called by one lane per channel)
RB_FN void acc_add(OuterAcc &acc, int c, double wa, double wb, double v)
{
    const double t = wa * v;
    acc.k[c] += t;
    acc.d[c] += wb * v;
    acc.a[c] += fabs(t);
}
RB_FN void acc_reduce(const OuterAcc &acc, double hl, PerChan<double> &r, PerChan<double> &e)
{
    RB_FOR_CHAN(c, kEngChan)
    {
        r[c] = acc.k[c] * hl;
        e[c] = quad_error(acc.d[c], acc.a[c], hl);
    }
}

// Warp vote over the channels 0..nv-1.
RB_FN bool chan_all(const PerChan<bool> &ok, int nv)
{
#ifdef RB_DEVICE_BUILD
    const int c = (threadIdx.x & 31) >> 2;
    return __all_sync(0xffffffffu, ok.v || c >= nv);
#else
    bool all = true;
    for (int c = 0; c < nv; c++)
        all = all && ok.v[c];
    return all;
#endif
}

// A pending-panel stack (warp-uniform; lane 0 writes, everybody reads).
struct PanelStack {
    struct Arrays {
        double *stk_a, *stk_b;
        int *stk_tag;
    } store;
    int sp;

    template <class Level>
    RB_FN void reset(Level *level)
    {
        store.stk_a = level->stk_a;
        store.stk_b = level->stk_b;
        store.stk_tag = level->stk_tag;
        sp = 0;
        warp_fence();
    }
    RB_FN bool room(int k) const { return sp + k <= kEngStack; }
    RB_FN void push(const Warp &w, double a, double b, int tag)
    {
#ifdef RB_DEVICE_BUILD
        if (w.lane == 0)
#endif
        {
            store.stk_a[sp] = a;
            store.stk_b[sp] = b;
            store.stk_tag[sp] = tag;
        }
        sp++;
    }
    RB_FN void seal() const { warp_fence(); } // make pushes visible before the next pop
    // reverse the order of the pending panels (the first one pushed is then popped first)
    RB_FN void reverse(const Warp &w)
    {
        warp_fence();
#ifdef RB_DEVICE_BUILD
        if (w.lane == 0)
#endif
        {
            for (int i = 0, j = sp - 1; i < j; i++, j--) {
                const double a = store.stk_a[i], b = store.stk_b[i];
                const int g = store.stk_tag[i];
                store.stk_a[i] = store.stk_a[j];
                store.stk_b[i] = store.stk_b[j];
                store.stk_tag[i] = store.stk_tag[j];
                store.stk_a[j] = a;
                store.stk_b[j] = b;
                store.stk_tag[j] = g;
            }
        }
        warp_fence();
    }
    RB_FN void pop(double &a, double &b, int &tag)
    {
        sp--;
        a = store.stk_a[sp];
        b = store.stk_b[sp];
        tag = store.stk_tag[sp];
    }

    // Cut the pending panel that straddles t at t, in its place in the stack (the pending panels are
    // disjoint): where the integrand jumps at t, no rule is then applied across the jump.  `paired`:
    // the panels are popped two at a time, so the pop partner is cut at the same fraction of its width
    // and each pop pair holds one part of both: a pair then still lies inside the pair it was cut from
    // (for the gamma integral: inside one Bessel branch).  A NaN t, or no room, cuts nothing.  Call
    // between the pushes and seal().
    RB_FN void cut_at(const Warp &w, double t, bool paired)
    {
        warp_fence(); // lane 0's pushes
        int i = -1;
        for (int j = 0; j < sp; j++) {
            if (store.stk_a[j] < t && t < store.stk_b[j])
                i = j;
        }
        // pop pairs run from the top, (sp - 1, sp - 2), ...; a bottom panel left over is popped alone
        const bool pair = paired && !(i == 0 && (sp & 1));
        const int lo = pair ? i - ((sp - 1 - i) & 1 ? 0 : 1) : i; // first entry of the pair
        const int grow = pair ? 2 : 1;
        if (i < 0 || !room(grow))
            return;
        warp_fence(); // every lane has read the stack
#ifdef RB_DEVICE_BUILD
        if (w.lane == 0)
#endif
        {
            for (int j = sp - 1; j > i; j--) { // the entries above make room
                store.stk_a[j + grow] = store.stk_a[j];
                store.stk_b[j + grow] = store.stk_b[j];
                store.stk_tag[j + grow] = store.stk_tag[j];
            }
            if (pair) { // [a0, c0], [a1, c1] below [c0, b0], [c1, b1]
                const double frac = (t - store.stk_a[i]) / (store.stk_b[i] - store.stk_a[i]);
                for (int k = 1; k >= 0; k--) {
                    const double a = store.stk_a[lo + k], b = store.stk_b[lo + k];
                    const int tag = store.stk_tag[lo + k];
                    const double c = (lo + k == i) ? t : a + frac * (b - a);
                    store.stk_a[lo + k] = a;
                    store.stk_b[lo + k] = c;
                    store.stk_a[lo + 2 + k] = c;
                    store.stk_b[lo + 2 + k] = b;
                    store.stk_tag[lo + 2 + k] = tag;
                }
            } else { // [t, b] below [a, t]: the lower part is popped first
                store.stk_a[i + 1] = store.stk_a[i];
                store.stk_b[i + 1] = t;
                store.stk_tag[i + 1] = store.stk_tag[i];
                store.stk_a[i] = t;
            }
        }
        sp += grow;
    }
};

// The acceptance rule of a panel for one channel: the error estimate is within
// `epsrel` of the larger of the panel's own value and `floor` (a fraction of the
// magnitude of the whole integral as known so far).  NaN compares as accepted so
// that it propagates into the sum, which is how the reference reports failure.
RB_FN bool panel_ok(double r, double e, double epsrel, double floor)
{
    const double m = fmax(fabs(r), floor);
    return !(e > epsrel * m);
}

RB_FN bool panel_too_small(double a, double b)
{
    const double m = fmax(fabs(a), fabs(b));
    return !(fabs(b - a) > 64.0 * DBL_EPSILON * m);
}

} // namespace rb
