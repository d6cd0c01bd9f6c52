// rb_launch.cuh -- launch geometry, kernel arguments and the per-stage launcher
// declarations shared by the translation units of the product library.  The
// kernels and launchers are in rb_kernels.cuh, instantiated per distribution kind
// in inst_*.cu so that they compile in parallel.
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <mutex>
#include <string>

#include "rb_heyvaerts.cuh"
#include "rb_heyfast.cuh"
#include "rb_symfast.cuh"
#include "rb_symphony.cuh"

namespace rbhost {

using namespace rb;

// ---------------------------------------------------------------------------
// launch geometry

constexpr int kWarpsPerBlock = 4;
constexpr int kThreadsPerBlock = kWarpsPerBlock * 32;

constexpr int kSymGammaCap = 48; // observed high-water mark 36 (DESIGN.md section 6)
constexpr int kSymNCap = 48;
constexpr int kHeyInnerCap = 128; // observed 112 in the s sin(theta) < 3 corner
constexpr int kHeyOuterCap = 64;
constexpr int kNormCap = 128; // QAG to 1e-8 on [1, 1e12] needs ~40 live intervals

constexpr int kMaxParams = 8;

struct BatchArgs {
    long long n;
    const double *s;
    const double *theta;
    const double *params[kMaxParams];
    int n_params;
    unsigned bcast;
    double *norm;
    double *out8;
    double *lobes4;
    int *status;
    unsigned *counters;
    unsigned long long *next;
    unsigned coeff_mask;
    double eps_gamma, eps_n, eps_hey_inner, eps_hey_outer;
    double sigma0_lo, sigma0_hi; // Heyvaerts: only points with sigma0 in [lo, hi)
    // Symphony fidelity guard: the product kernel appends the points it will not compute to
    // `reroute_list` (length in reroute_count[0]); the faithful kernel launched after it
    // takes its points from that list instead of from 0..n-1.
    int *reroute_list;
    unsigned long long *reroute_count;
    double *handover; // [slot][kSnapDoubles]: chunk-loop state for the faithful continuation
    int from_reroute_list;
    // Cost-ordered scheduling of the product kernels: k_classify sorts the points into three cost
    // classes per kernel (expensive first); ticket t of the atomic counter maps to
    // order[class][t - (points in the classes before)].  The per-point cost spans 10x and a
    // warp works on one point at a time, so handing out the long points first is what keeps the
    // tail of the persistent kernel short.
    double hey_free_below;            // scheduling hint: Heyvaerts points with s below this cost nothing (0 = none)
    int *order;                       // [2 kernels][kCostClasses][n]
    unsigned long long *class_counts; // [2 kernels][kCostClasses]
};

constexpr int kCostClasses = 4;

// One diagnostic of the Symphony double integral at `count` arguments of ONE point (the
// point is element 0 of the BatchArgs arrays): lib.rs:254-298.
struct DiagArgs {
    int coeff, stokes, what; // what: kDiag* of rb_symphony.cuh
    long long count;
    const double *a, *b;     // n / n_lo / gamma, and gamma / n_hi (b may be null)
    double *out;
    int *status;             // kStatus* bits per element (nullable)
};

// ticket -> point index for kernel `which` (0 = Symphony, 1 = Heyvaerts)
__device__ __forceinline__ long long ordered_point(const BatchArgs &a, int which, long long ticket)
{
    const unsigned long long *cnt = a.class_counts + which * kCostClasses;
    const int *ord = a.order + (size_t)which * kCostClasses * a.n;
    long long t = ticket;
#pragma unroll
    for (int k = 0; k < kCostClasses; k++) {
        const long long c = (long long)cnt[k];
        if (t < c)
            return ord[(size_t)k * a.n + t];
        t -= c;
    }
    return a.n; // not reached: the classes hold n points in total
}

__device__ __forceinline__ long long next_point(unsigned long long *counter, int lane)
{
    unsigned long long i = 0;
    if (lane == 0)
        i = atomicAdd(counter, 1ULL);
    return (long long)__shfl_sync(0xffffffffu, i, 0);
}

template <int KIND>
__device__ __forceinline__ bool load_dist(const BatchArgs &a, long long i, Dist &d, double &first_param)
{
    double pv[kMaxParams];
#pragma unroll
    for (int j = 0; j < kMaxParams; j++)
        pv[j] = (j < a.n_params) ? a.params[j][((a.bcast >> j) & 1u) ? 0 : i] : 0.0;
    first_param = pv[0];
    return dist_from_params<KIND>(pv, a.n_params, d);
}


// ---------------------------------------------------------------------------
// host-side state shared between translation units (defined in rimphony_b200.cu)

int fail(const char *fmt, ...);
extern std::atomic<uint64_t> g_launches;

#define RB_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return ::rbhost::fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Per-stage launchers, explicitly instantiated in inst_*.cu.
template <int KIND>
int stage_normalize(const BatchArgs &a, int sm_count, cudaStream_t st);
template <int KIND, bool FUSED>
int stage_symphony(const BatchArgs &a, int sm_count, cudaStream_t st);
int stage_classify(const BatchArgs &a, cudaStream_t st);
template <int KIND>
int stage_symphony_fast(const BatchArgs &a, int sm_count, cudaStream_t st);
template <int KIND>
int stage_symphony_diag(const BatchArgs &a, const DiagArgs &g, int sm_count, cudaStream_t st);
template <int KIND, bool FUSED>
int stage_heyvaerts(const BatchArgs &a, int sm_count, cudaStream_t st);
template <int KIND>
int stage_heyvaerts_fast(const BatchArgs &a, int sm_count, cudaStream_t st);
template <int KIND>
int stage_dist_eval(const double *params, int n_params, long long count, const double *gamma, const double *cos_xi,
                    double *out3, cudaStream_t st);

} // namespace rbhost
