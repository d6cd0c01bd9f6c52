// rimphony_b200.cu -- the C ABI (include/rimphony_b200.h) and its host side.
//
// A batch runs these kernels (rb_kernels.cuh, instantiated per distribution kind in inst_*.cu):
//   k_normalize        full_calculation(): the normalisation constant of each point
//   k_classify         the cost-ordered schedule of the two product kernels (this file)
//   k_symphony_fast    j_I, alpha_I, j_Q, alpha_Q, j_V, alpha_V       (rb_symfast.cuh)
//   k_heyvaerts_fast   rho_Q, rho_V                                    (rb_heyfast.cuh)
// That is MODE_FAST, the default.  k_symphony (rb_symphony.cuh) computes the points k_symphony_fast
// hands over to the reference's exact rule sequence; it and k_heyvaerts (rb_heyvaerts.cuh) replace
// the product kernels in the other modes.  Points are independent, their cost varies by more than
// 10x, so each warp of the persistent kernels pulls the next point from a global atomic counter.
// All arithmetic is FP64 on the CUDA cores; there is no dense contraction for the tensor cores to do.
//
// rimphony_b200_transfer* and rimphony_b200_compute_stokes_cgs add the polarized transfer through rays of cells
// (rb_transfer.cuh, kernels in inst_transfer.cu): one thread per ray.
//
// There is deliberately no host implementation behind these entry points: with
// no usable CUDA device every call fails with a nonzero return code.
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/rimphony_b200.h"
#include "rb_launch.cuh"
#include "rb_transfer.cuh"

namespace {

using namespace rb;

// FP64 FMA throughput probe: the denominator of the roofline (the pool's
// MEASURED_PEAKS.json has no FP64 figure).  16 independent DFMA chains per thread.
__global__ void __launch_bounds__(256) k_dfma_peak(double *sink, int iters, double a, double b)
{
    double v[16];
#pragma unroll
    for (int k = 0; k < 16; k++)
        v[k] = a + k + threadIdx.x;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int k = 0; k < 16; k++)
            v[k] = fma(v[k], b, a);
    }
    double t = 0;
#pragma unroll
    for (int k = 0; k < 16; k++)
        t += v[k];
    if (t == 12345.678)
        sink[0] = t;
}

// Cost classes of the product kernels (rb_launch.cuh BatchArgs::order).  Symphony: rule
// applications grow with s (500 at s < 1 to 3000 at s ~ 1e4).  Heyvaerts: 0.38 <= s < 1 costs
// 3.7-5.3 k applications (the quasi-resonant integrand is singular at sigma = s), s sin(theta) < 3
// about 2.3 k, the rest 0.5 k; the power-law points below s = 0.38 cost nothing (the reference's
// NaN region, rb_heyfast.cuh) and go last.
__global__ void k_classify(rbhost::BatchArgs a)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n)
        return;
    const double s = a.s[i];
    const double sigma0 = s * sin(a.theta[i]);
    const int cs = (s >= 300.0) ? 0 : ((s >= 10.0) ? 1 : 2);
    int ch = (s < 1.0) ? 1 : ((sigma0 < 3.0) ? 2 : 3); // NaN lands in the last class
    // The points that can run into the application budget (20 k applications, 15 x the mean; measured on 65 536
    // points: all but a handful of those above 15 k have s sin(theta) < 0.1 and s < 10) start first: a launch is at
    // least as long as its longest point, and one of these picked up late is the tail of a 1e5-point launch
    // (simulated on the measured costs: 1.29 -> 1.05 x the ideal makespan at 131 072 points).
    if (sigma0 < 0.1 && s < 10.0)
        ch = 0;
    if (a.hey_free_below > 0.0 && s < a.hey_free_below)
        ch = 3;
    const unsigned long long ks = atomicAdd(&a.class_counts[cs], 1ULL);
    a.order[(size_t)cs * a.n + ks] = (int)i;
    const unsigned long long kh = atomicAdd(&a.class_counts[rbhost::kCostClasses + ch], 1ULL);
    a.order[(size_t)(rbhost::kCostClasses + ch) * a.n + kh] = (int)i;
}

// test entry point: the device Bessel evaluator
__global__ void k_bessel(long long count, const double *n, const double *x, double *j, double *dj)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count)
        return;
    LeungOrder o, o1;
    leung_prepare(n[i], o);
    leung_prepare(n[i] + 1.0, o1);
    double jn, djn;
    leung_j_and_dj(o, o1, x[i], jn, djn);
    j[i] = jn;
    dj[i] = djn;
}


// ---------------------------------------------------------------------------
// host side

thread_local std::string g_error;

} // namespace
namespace rbhost {
int stage_classify(const BatchArgs &a, cudaStream_t st)
{
    RB_CUDA(cudaMemsetAsync(a.class_counts, 0, 2 * kCostClasses * sizeof(unsigned long long), st));
    k_classify<<<(unsigned)((a.n + 255) / 256), 256, 0, st>>>(a);
    g_launches++;
    RB_CUDA(cudaGetLastError());
    return 0;
}
std::atomic<uint64_t> g_launches{0};
int fail(const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return 1;
}
} // namespace rbhost
namespace {
using namespace rbhost;

struct DeviceBuffer {
    void *ptr = nullptr;
    size_t bytes = 0;
    int reserve(size_t want)
    {
        if (want <= bytes)
            return 0;
        if (ptr)
            cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
        cudaError_t e = cudaMalloc(&ptr, want);
        if (e != cudaSuccess)
            return fail("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        bytes = want;
        return 0;
    }
    void release()
    {
        if (ptr)
            cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
    }
};

// Restores the calling thread's current CUDA device on scope exit: the entry points select the
// device they run on and must not leave that as a side effect (callers such as torch keep their
// own notion of the current device).
struct DeviceGuard {
    int saved = -1;
    DeviceGuard() { if (cudaGetDevice(&saved) != cudaSuccess) saved = -1; }
    ~DeviceGuard() { if (saved >= 0) cudaSetDevice(saved); }
};

struct DeviceContext {
    bool ready = false;
    int device = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;       // Symphony + copies
    cudaStream_t stream_hey = nullptr;   // Heyvaerts, overlaps the Symphony tail
    cudaEvent_t ev[8] = {};
    cudaEvent_t ev_done = nullptr;       // completion of the most recent batched call on this device
    bool have_done = false;
    DeviceBuffer in, out, scratch, counters, reroute, handover, order;
    float last_ms[4] = {0, 0, 0, 0};
    std::mutex lock;
};

constexpr int kMaxDevices = 16;
DeviceContext g_ctx[kMaxDevices];
std::mutex g_ctx_lock;

int get_context(int device, DeviceContext **out)
{
    if (device < 0)
        RB_CUDA(cudaGetDevice(&device));
    if (device >= kMaxDevices)
        return fail("device ordinal %d out of range", device);
    DeviceContext &c = g_ctx[device];
    std::lock_guard<std::mutex> g(g_ctx_lock);
    if (!c.ready) {
        int count = 0;
        RB_CUDA(cudaGetDeviceCount(&count));
        if (device >= count)
            return fail("CUDA device %d not present (%d visible)", device, count);
        RB_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        RB_CUDA(cudaGetDeviceProperties(&prop, device));
        c.sm_count = prop.multiProcessorCount;
        RB_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        RB_CUDA(cudaStreamCreateWithFlags(&c.stream_hey, cudaStreamNonBlocking));
        for (auto &e : c.ev)
            RB_CUDA(cudaEventCreate(&e));
        RB_CUDA(cudaEventCreateWithFlags(&c.ev_done, cudaEventDisableTiming));
        c.device = device;
        c.ready = true;
    }
    *out = &c;
    return 0;
}

struct ResolvedOptions {
    int mode;
    unsigned coeff_mask;
    unsigned bcast;
    int device;
    double eps_gamma, eps_n, eps_hi, eps_ho;
};

ResolvedOptions resolve(const rimphony_b200_options *o)
{
    ResolvedOptions r{RIMPHONY_B200_MODE_FAST, 0xFFu, 0u, -1, 1e-3, 1e-3, 1e-3, 1e-3};
    if (!o)
        return r;
    rimphony_b200_options tmp;
    memset(&tmp, 0, sizeof tmp);
    const size_t sz = o->struct_size ? (o->struct_size < sizeof tmp ? o->struct_size : sizeof tmp) : sizeof tmp;
    memcpy(&tmp, o, sz);
    r.mode = tmp.mode;
    r.coeff_mask = tmp.coeff_mask ? (tmp.coeff_mask & 0xFFu) : 0xFFu;
    r.bcast = tmp.param_broadcast_mask;
    // ordinal + 1, so that a zero-initialised (or older, shorter) struct means "the calling
    // thread's current device"
    r.device = (tmp.device_plus_one > 0) ? tmp.device_plus_one - 1 : -1;
    if (tmp.epsrel_gamma > 0)
        r.eps_gamma = tmp.epsrel_gamma;
    if (tmp.epsrel_n > 0)
        r.eps_n = tmp.epsrel_n;
    if (tmp.epsrel_heyvaerts_inner > 0)
        r.eps_hi = tmp.epsrel_heyvaerts_inner;
    if (tmp.epsrel_heyvaerts_outer > 0)
        r.eps_ho = tmp.epsrel_heyvaerts_outer;
    return r;
}

int check_params(int kind, int n_params)
{
    switch (kind) {
    case RIMPHONY_B200_POWER_LAW:
        return (n_params == 1 || n_params == 4) ? 0 : fail("POWER_LAW takes 1 or 4 parameter columns, got %d", n_params);
    case RIMPHONY_B200_THERMAL_JUETTNER:
        return n_params == 1 ? 0 : fail("THERMAL_JUETTNER takes 1 parameter column, got %d", n_params);
    case RIMPHONY_B200_PITCHY_PL:
        return (n_params == 2 || n_params == 5) ? 0 : fail("PITCHY_PL takes 2 or 5 parameter columns, got %d", n_params);
    case RIMPHONY_B200_PITCHY_KAPPA:
        return (n_params == 3 || n_params == 4) ? 0 : fail("PITCHY_KAPPA takes 3 or 4 parameter columns, got %d", n_params);
    case RIMPHONY_B200_PITCHY_BROKEN_PL:
        return (n_params == 4 || n_params == 7) ? 0
                                                : fail("PITCHY_BROKEN_PL takes 4 or 7 parameter columns, got %d", n_params);
    }
    return fail("unknown distribution kind %d", kind);
}

// The argument checks of the batched entry points; nonzero means a bad argument (the message is
// set).  With n == 0 there is nothing to compute and nothing more to check; otherwise *o is resolved.
int check_batch(int kind, int64_t n, const double *s, const double *theta, const double *const *params, int n_params,
                const double *out8, const rimphony_b200_options *opts, ResolvedOptions *o)
{
    if (n < 0)
        return fail("n_points is negative");
    if (check_params(kind, n_params))
        return 1;
    if (n == 0)
        return 0;
    if (!s || !theta || !params || !out8)
        return fail("null array pointer");
    *o = resolve(opts);
    if (o->mode < 0 || o->mode > 3)
        return fail("unknown mode %d", o->mode);
    return 0;
}

template <int KIND>
int launch_kind(DeviceContext &c, BatchArgs a, const ResolvedOptions &o, cudaStream_t user_stream)
{
    cudaStream_t st = user_stream ? user_stream : c.stream;
    // Heyvaerts always runs on the library's second stream, forked from and joined back
    // into `st` with events, so a caller-supplied stream keeps its ordering semantics.
    const cudaStream_t st_hey = c.stream_hey;
    unsigned long long *counters = static_cast<unsigned long long *>(c.counters.ptr);
    const bool faithful = (o.mode == RIMPHONY_B200_MODE_FAITHFUL);
    const bool want_sym = (o.coeff_mask & 0x3Fu) != 0;
    const bool want_hey = (o.coeff_mask & 0xC0u) != 0;

    RB_CUDA(cudaMemsetAsync(counters, 0, 4 * sizeof(unsigned long long), st));
    RB_CUDA(cudaEventRecord(c.ev[0], st));
    // the broken power law is PITCHY_PL with p = p1 near gamma = 1, where the reference diverges
    a.hey_free_below =
        (KIND == kDistPitchyPL || KIND == kDistPitchyBrokenPL) ? kHeyDivQLo : ((KIND == kDistPowerLaw) ? 0.05 : 0.0);

    // 1. normalisation (+ the cost-ordered schedule of the product kernels)
    if (stage_normalize<KIND>(a, c.sm_count, st))
        return 1;
    if (o.mode == RIMPHONY_B200_MODE_FAST && stage_classify(a, st))
        return 1;
    RB_CUDA(cudaEventRecord(c.ev[1], st));
    RB_CUDA(cudaStreamWaitEvent(st_hey, c.ev[1], 0));

    // 2. Symphony
    if (want_sym) {
        a.next = counters + 0;
        if (o.mode == RIMPHONY_B200_MODE_FAST) {
            a.reroute_count = counters + 3;
            if (stage_symphony_fast<KIND>(a, c.sm_count, st))
                return 1;
            // fidelity guard: the points the product kernel handed over, if any
            BatchArgs b = a;
            b.next = counters + 0; // reused: reset between the two kernels
            RB_CUDA(cudaMemsetAsync(counters + 0, 0, sizeof(unsigned long long), st));
            b.from_reroute_list = 1;
            if (stage_symphony<KIND, false>(b, c.sm_count, st))
                return 1;
        } else if (faithful ? stage_symphony<KIND, false>(a, c.sm_count, st)
                            : stage_symphony<KIND, true>(a, c.sm_count, st))
            return 1;
    }
    RB_CUDA(cudaEventRecord(c.ev[2], st));

    // 3. Heyvaerts (second stream: fills the SMs that the Symphony tail leaves idle)
    RB_CUDA(cudaEventRecord(c.ev[3], st_hey));
    if (want_hey && o.mode == RIMPHONY_B200_MODE_FAST) {
        BatchArgs b = a;
        b.next = counters + 1;
        if (stage_heyvaerts_fast<KIND>(b, c.sm_count, st_hey))
            return 1;
    } else if (want_hey) {
        const bool split_mode = (o.mode == RIMPHONY_B200_MODE_FUSED);
        const double split = split_mode ? 3.0 : (faithful ? INFINITY : -INFINITY);
        if (split > -INFINITY) { // the reference's exact sequence for sigma0 < split
            BatchArgs b = a;
            b.next = counters + 1;
            b.sigma0_lo = -INFINITY;
            b.sigma0_hi = split;
            if (stage_heyvaerts<KIND, false>(b, c.sm_count, st_hey))
                return 1;
        }
        if (split < INFINITY) { // h and f on shared nodes for sigma0 >= split
            BatchArgs b = a;
            b.next = counters + 2;
            b.sigma0_lo = split;
            b.sigma0_hi = INFINITY;
            if (stage_heyvaerts<KIND, true>(b, c.sm_count, st_hey))
                return 1;
        }
    }
    RB_CUDA(cudaEventRecord(c.ev[4], st_hey));
    RB_CUDA(cudaStreamWaitEvent(st, c.ev[4], 0));
    RB_CUDA(cudaEventRecord(c.ev[5], st));
    return 0;
}

// Runs f(std::integral_constant<int, KIND>) for the distribution kind of the C ABI.
template <class F>
int dispatch_kind(int kind, F &&f)
{
    switch (kind) {
    case RIMPHONY_B200_POWER_LAW:
        return f(std::integral_constant<int, kDistPowerLaw>{});
    case RIMPHONY_B200_THERMAL_JUETTNER:
        return f(std::integral_constant<int, kDistThermalJuettner>{});
    case RIMPHONY_B200_PITCHY_PL:
        return f(std::integral_constant<int, kDistPitchyPL>{});
    case RIMPHONY_B200_PITCHY_KAPPA:
        return f(std::integral_constant<int, kDistPitchyKappa>{});
    case RIMPHONY_B200_PITCHY_BROKEN_PL:
        return f(std::integral_constant<int, kDistPitchyBrokenPL>{});
    }
    return fail("unknown distribution kind %d", kind);
}

int collect_times(DeviceContext &c)
{
    float t;
    RB_CUDA(cudaEventElapsedTime(&t, c.ev[0], c.ev[1]));
    c.last_ms[0] = t;
    RB_CUDA(cudaEventElapsedTime(&t, c.ev[1], c.ev[2]));
    c.last_ms[1] = t;
    RB_CUDA(cudaEventElapsedTime(&t, c.ev[3], c.ev[4]));
    c.last_ms[2] = t;
    RB_CUDA(cudaEventElapsedTime(&t, c.ev[0], c.ev[5]));
    c.last_ms[3] = t;
    return 0;
}

// Device-pointer path shared by every public entry point.
int run_device(int kind, int64_t n, const double *s, const double *theta, const double *const *params, int n_params,
               const ResolvedOptions &o, double *out8, int32_t *status, const rimphony_b200_extras *extras,
               void *stream, int synchronize, DeviceContext &c)
{
    RB_CUDA(cudaSetDevice(c.device));
    const size_t norm_bytes = (size_t)n * sizeof(double);
    double *norm = extras ? extras->norm : nullptr;
    if (!norm) {
        if (c.scratch.reserve(norm_bytes))
            return 1;
        norm = static_cast<double *>(c.scratch.ptr);
    }
    if (c.counters.reserve(4 * sizeof(unsigned long long)))
        return 1;
    if (c.reroute.reserve((size_t)n * sizeof(int)))
        return 1;
    if (c.order.reserve((size_t)n * 2 * kCostClasses * sizeof(int) + 2 * kCostClasses * sizeof(unsigned long long)))
        return 1;
    if (o.mode == RIMPHONY_B200_MODE_FAST && (o.coeff_mask & 0x3Fu) &&
        c.handover.reserve((size_t)n * kSnapDoubles * sizeof(double)))
        return 1;

    BatchArgs a;
    memset(&a, 0, sizeof a);
    a.reroute_list = static_cast<int *>(c.reroute.ptr);
    a.handover = static_cast<double *>(c.handover.ptr);
    a.class_counts = static_cast<unsigned long long *>(c.order.ptr);
    a.order = reinterpret_cast<int *>(a.class_counts + 2 * kCostClasses);
    a.n = n;
    a.s = s;
    a.theta = theta;
    for (int j = 0; j < n_params; j++)
        a.params[j] = params[j];
    a.n_params = n_params;
    a.bcast = o.bcast;
    a.norm = norm;
    a.out8 = out8;
    a.lobes4 = extras ? extras->lobes4 : nullptr;
    a.status = status;
    a.counters = extras ? extras->counters : nullptr;
    a.coeff_mask = o.coeff_mask;
    a.eps_gamma = o.eps_gamma;
    a.eps_n = o.eps_n;
    a.eps_hey_inner = o.eps_hi;
    a.eps_hey_outer = o.eps_ho;
    a.sigma0_lo = -INFINITY;
    a.sigma0_hi = INFINITY;

    cudaStream_t user = static_cast<cudaStream_t>(stream);
    cudaStream_t st = user ? user : c.stream;
    // The work counters, the reroute list, the hand-over records and the cost-ordered schedule
    // are per-device scratch: a call enqueued while an earlier asynchronous one (possibly on
    // another stream) is still running must not touch them.  It waits, on the device, for that
    // call's completion event; the host does not block.
    if (c.have_done)
        RB_CUDA(cudaStreamWaitEvent(st, c.ev_done, 0));
    if (status)
        RB_CUDA(cudaMemsetAsync(status, 0, (size_t)n * sizeof(int32_t), st));
    if (dispatch_kind(kind, [&](auto k) { return launch_kind<decltype(k)::value>(c, a, o, user); }))
        return 1;
    RB_CUDA(cudaEventRecord(c.ev_done, st));
    c.have_done = true;
    if (synchronize) {
        RB_CUDA(cudaStreamSynchronize(st));
        if (collect_times(c))
            return 1;
    }
    return 0;
}

// `out_stride`: distance in doubles between two slots of the caller's out8 (n for a whole batch;
// the batch size of the caller when this call computes one shard of it, see _multi).
int run_host(int kind, int64_t n, const double *s, const double *theta, const double *const *params, int n_params,
             const rimphony_b200_options *opts, double *out8, int32_t *status, const rimphony_b200_extras *extras,
             int device_override, int64_t out_stride = 0)
{
    DeviceGuard restore_device;
    ResolvedOptions o;
    if (check_batch(kind, n, s, theta, params, n_params, out8, opts, &o))
        return 1;
    if (n == 0)
        return 0;
    if (device_override >= 0)
        o.device = device_override;

    DeviceContext *cp = nullptr;
    if (get_context(o.device, &cp))
        return 1;
    DeviceContext &c = *cp;
    std::lock_guard<std::mutex> guard(c.lock);
    RB_CUDA(cudaSetDevice(c.device));

    // device staging: [s | theta | param columns] in, [out8 | status | lobes | counters | norm] out
    size_t in_doubles = 2 * (size_t)n;
    for (int j = 0; j < n_params; j++)
        in_doubles += ((o.bcast >> j) & 1u) ? 1 : (size_t)n;
    if (c.in.reserve(in_doubles * sizeof(double)))
        return 1;
    const bool want_lobes = extras && extras->lobes4;
    const bool want_counters = extras && extras->counters;
    const bool want_norm = extras && extras->norm;
    size_t out_bytes = 8 * (size_t)n * sizeof(double) + (size_t)n * sizeof(int32_t) + 64;
    out_bytes += want_lobes ? 4 * (size_t)n * sizeof(double) : 0;
    out_bytes += want_counters ? 2 * (size_t)n * sizeof(uint32_t) + 64 : 0;
    out_bytes += (size_t)n * sizeof(double);
    if (c.out.reserve(out_bytes))
        return 1;

    double *d_in = static_cast<double *>(c.in.ptr);
    double *d_s = d_in;
    double *d_theta = d_in + n;
    const double *d_params[kMaxParams] = {};
    {
        double *cur = d_in + 2 * n;
        RB_CUDA(cudaMemcpyAsync(d_s, s, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, c.stream));
        RB_CUDA(cudaMemcpyAsync(d_theta, theta, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, c.stream));
        for (int j = 0; j < n_params; j++) {
            if (!params[j])
                return fail("params[%d] is null", j);
            const size_t cnt = ((o.bcast >> j) & 1u) ? 1 : (size_t)n;
            RB_CUDA(cudaMemcpyAsync(cur, params[j], cnt * sizeof(double), cudaMemcpyHostToDevice, c.stream));
            d_params[j] = cur;
            cur += cnt;
        }
    }

    char *d_out = static_cast<char *>(c.out.ptr);
    double *d_out8 = reinterpret_cast<double *>(d_out);
    d_out += 8 * (size_t)n * sizeof(double);
    double *d_norm = reinterpret_cast<double *>(d_out);
    d_out += (size_t)n * sizeof(double);
    double *d_lobes = nullptr;
    if (want_lobes) {
        d_lobes = reinterpret_cast<double *>(d_out);
        d_out += 4 * (size_t)n * sizeof(double);
    }
    int32_t *d_status = reinterpret_cast<int32_t *>(d_out);
    d_out += ((size_t)n * sizeof(int32_t) + 63) / 64 * 64;
    uint32_t *d_counters = nullptr;
    if (want_counters) {
        d_counters = reinterpret_cast<uint32_t *>(d_out);
        RB_CUDA(cudaMemsetAsync(d_counters, 0, 2 * (size_t)n * sizeof(uint32_t), c.stream));
    }

    // slots that are not requested come back as NaN
    RB_CUDA(cudaMemsetAsync(d_out8, 0xFF, 8 * (size_t)n * sizeof(double), c.stream));

    rimphony_b200_extras dev_extras;
    dev_extras.lobes4 = d_lobes;
    dev_extras.counters = d_counters;
    dev_extras.norm = d_norm;
    if (run_device(kind, n, d_s, d_theta, d_params, n_params, o, d_out8, d_status, &dev_extras, nullptr, 0, c))
        return 1;

    if (out_stride > n) // a shard: each slot row lands in its slice of the caller's [8][out_stride] array
        RB_CUDA(cudaMemcpy2DAsync(out8, (size_t)out_stride * sizeof(double), d_out8, (size_t)n * sizeof(double),
                                  (size_t)n * sizeof(double), 8, cudaMemcpyDeviceToHost, c.stream));
    else
        RB_CUDA(cudaMemcpyAsync(out8, d_out8, 8 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    if (status)
        RB_CUDA(cudaMemcpyAsync(status, d_status, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    if (want_lobes)
        RB_CUDA(cudaMemcpyAsync(extras->lobes4, d_lobes, 4 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    if (want_counters)
        RB_CUDA(cudaMemcpyAsync(extras->counters, d_counters, 2 * (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                c.stream));
    if (want_norm)
        RB_CUDA(cudaMemcpyAsync(extras->norm, d_norm, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    RB_CUDA(cudaStreamSynchronize(c.stream));
    return collect_times(c);
}

// The argument checks of the transfer entry points; *n_points = n_rays * n_cells.
int check_rays(int64_t n_rays, int64_t n_cells, int64_t *n_points)
{
    if (n_rays < 0 || n_cells < 0)
        return fail("n_rays and n_cells must not be negative");
    if (n_cells > 0 && n_rays > INT64_MAX / n_cells)
        return fail("n_rays * n_cells overflows");
    *n_points = n_rays * n_cells;
    return 0;
}

int check_transfer(int64_t n_rays, int64_t n_cells, const double *coeffs8, const double *psi, const double *ds,
                   const double *stokes4, int64_t *n_points)
{
    if (check_rays(n_rays, n_cells, n_points))
        return 1;
    if (n_rays > 0 && (!stokes4 || (*n_points > 0 && (!coeffs8 || !psi || !ds))))
        return fail("null array pointer");
    return 0;
}

} // namespace

// ---------------------------------------------------------------------------
// C ABI

extern "C" {

int rimphony_b200_compute_all_dimensionless(int kind, int64_t n_points, const double *s, const double *theta,
                                            const double *const *params, int n_params,
                                            const rimphony_b200_options *opts, double *out8, int32_t *status)
{
    return run_host(kind, n_points, s, theta, params, n_params, opts, out8, status, nullptr, -1);
}

int rimphony_b200_compute_all_dimensionless_ex(int kind, int64_t n_points, const double *s, const double *theta,
                                               const double *const *params, int n_params,
                                               const rimphony_b200_options *opts, double *out8, int32_t *status,
                                               const rimphony_b200_extras *extras)
{
    return run_host(kind, n_points, s, theta, params, n_params, opts, out8, status, extras, -1);
}

int rimphony_b200_compute_all_dimensionless_device(int kind, int64_t n_points, const double *s, const double *theta,
                                                   const double *const *params, int n_params,
                                                   const rimphony_b200_options *opts, double *out8, int32_t *status,
                                                   const rimphony_b200_extras *extras, void *stream, int synchronize)
{
    ResolvedOptions o;
    if (check_batch(kind, n_points, s, theta, params, n_params, out8, opts, &o))
        return 1;
    if (n_points == 0)
        return 0;
    DeviceGuard restore_device;
    DeviceContext *cp = nullptr;
    if (get_context(o.device, &cp))
        return 1;
    std::lock_guard<std::mutex> guard(cp->lock);
    return run_device(kind, n_points, s, theta, params, n_params, o, out8, status, extras, stream, synchronize, *cp);
}

int rimphony_b200_compute_all_dimensionless_multi(int kind, int64_t n_points, const double *s, const double *theta,
                                                  const double *const *params, int n_params,
                                                  const rimphony_b200_options *opts, double *out8, int32_t *status,
                                                  int n_devices)
{
    ResolvedOptions o;
    if (check_batch(kind, n_points, s, theta, params, n_params, out8, opts, &o))
        return 1;
    if (n_points == 0)
        return 0;
    for (int j = 0; j < n_params; j++)
        if (!params[j])
            return fail("params[%d] is null", j);
    int visible = 0;
    RB_CUDA(cudaGetDeviceCount(&visible));
    if (visible < 1)
        return fail("no CUDA device visible");
    if (visible > kMaxDevices)
        visible = kMaxDevices;
    if (n_devices <= 0 || n_devices > visible)
        n_devices = visible;
    if ((int64_t)n_devices > n_points)
        n_devices = (int)n_points;

    // Contiguous slices, devices 0 .. n_devices-1 (opts->device_plus_one does not apply here).  out8
    // is slot-major over the WHOLE batch: every shard copies its eight rows straight into their
    // slices of it (one strided device-to-host copy), the host gathers by construction.
    std::vector<std::thread> workers;
    std::vector<int> rc(n_devices, 0);
    std::vector<std::string> msg(n_devices);
    try {
        for (int d = 0; d < n_devices; d++) {
            const int64_t lo = n_points * d / n_devices, hi = n_points * (d + 1) / n_devices;
            workers.emplace_back([&, d, lo, hi]() {
                try {
                    const int64_t m = hi - lo;
                    if (m == 0)
                        return;
                    const double *cols[kMaxParams] = {};
                    for (int j = 0; j < n_params; j++)
                        cols[j] = ((o.bcast >> j) & 1u) ? params[j] : params[j] + lo;
                    rc[d] = run_host(kind, m, s + lo, theta + lo, cols, n_params, opts, out8 + lo,
                                     status ? status + lo : nullptr, nullptr, d, n_points);
                    if (rc[d])
                        msg[d] = g_error; // thread-local: carry it to the caller's thread
                } catch (const std::exception &e) {
                    rc[d] = 1;
                    msg[d] = e.what();
                } catch (...) {
                    rc[d] = 1;
                    msg[d] = "unknown exception";
                }
            });
        }
    } catch (const std::exception &e) { // thread creation failed: join what was started
        for (auto &t : workers)
            t.join();
        return fail("could not start the per-device worker threads: %s", e.what());
    }
    for (auto &t : workers)
        t.join();
    for (int d = 0; d < n_devices; d++)
        if (rc[d])
            return fail("device %d: %s", d, msg[d].c_str());
    return 0;
}

int rimphony_b200_compute_dimensionless(int kind, const double *params, int n_params, int coeff, int stokes, double s,
                                        double theta, double *out)
{
    if (!out || !params)
        return fail("null pointer");
    if (coeff < 0 || coeff > 2 || stokes < 0 || stokes > 2)
        return fail("bad coefficient/stokes selector");
    if (check_params(kind, n_params))
        return 1;
    if (coeff == RIMPHONY_B200_FARADAY && stokes == RIMPHONY_B200_STOKES_I) {
        *out = NAN; // src/lib.rs:239-240
        return 0;
    }
    const int slot = (coeff == RIMPHONY_B200_FARADAY) ? (stokes == RIMPHONY_B200_STOKES_Q ? 6 : 7) : (2 * stokes + coeff);
    rimphony_b200_options o;
    memset(&o, 0, sizeof o);
    o.struct_size = sizeof o;
    o.coeff_mask = 1u << slot;
    o.device_plus_one = 0; // the current device
    const double *cols[kMaxParams];
    for (int j = 0; j < n_params; j++)
        cols[j] = params + j;
    double out8[8];
    if (run_host(kind, 1, &s, &theta, cols, n_params, &o, out8, nullptr, nullptr, -1))
        return 1;
    *out = out8[slot];
    return 0;
}

int rimphony_b200_compute_cgs(int kind, const double *params, int n_params, int coeff, int stokes, double nu, double b,
                              double n_e, double theta, double *out)
{
    // src/lib.rs:163-173
    const double nu_c = kElectronCharge * b / (kTwoPi * kMassElectron * kSpeedLight);
    double val;
    if (rimphony_b200_compute_dimensionless(kind, params, n_params, coeff, stokes, nu / nu_c, theta, &val))
        return 1;
    *out = (coeff == RIMPHONY_B200_EMISSION) ? val * n_e * nu : val * n_e / nu;
    return 0;
}

int rimphony_b200_diagnostic_symphony(int kind, const double *params, int n_params, int coeff, int stokes, double s,
                                      double theta, int what, int64_t count, const double *a, const double *b,
                                      double *out, int32_t *status)
{
    if (count < 0 || !params || !a || !out)
        return fail("bad arguments");
    if (coeff < 0 || coeff > 1 || stokes < 0 || stokes > 2)
        return fail("bad coefficient/stokes selector (the Symphony diagnostics take emission or absorption)");
    if (what < 0 || what > 3)
        return fail("unknown diagnostic %d", what);
    if ((what == RIMPHONY_B200_DIAG_GAMMA_INTEGRAND || what == RIMPHONY_B200_DIAG_N_INTEGRAL) && !b)
        return fail("this diagnostic takes two argument arrays");
    if (check_params(kind, n_params))
        return 1;
    if (count == 0)
        return 0;
    DeviceContext *cp = nullptr;
    if (get_context(-1, &cp))
        return 1;
    DeviceContext &c = *cp;
    std::lock_guard<std::mutex> guard(c.lock);
    RB_CUDA(cudaSetDevice(c.device));

    // device staging: [s | theta | params | norm | a | b] in, [out | status] out
    const size_t head = 2 + (size_t)n_params + 1;
    if (c.in.reserve((head + 2 * (size_t)count) * sizeof(double)) ||
        c.out.reserve((size_t)count * (sizeof(double) + sizeof(int32_t))))
        return 1;
    double host_head[2 + kMaxParams];
    host_head[0] = s;
    host_head[1] = theta;
    for (int j = 0; j < n_params; j++)
        host_head[2 + j] = params[j];
    double *d_in = static_cast<double *>(c.in.ptr);
    RB_CUDA(cudaMemcpyAsync(d_in, host_head, (2 + (size_t)n_params) * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    double *d_a = d_in + head, *d_b = d_a + count;
    RB_CUDA(cudaMemcpyAsync(d_a, a, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    if (b)
        RB_CUDA(cudaMemcpyAsync(d_b, b, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    double *d_out = static_cast<double *>(c.out.ptr);
    int32_t *d_status = reinterpret_cast<int32_t *>(d_out + count);

    BatchArgs ba;
    memset(&ba, 0, sizeof ba);
    ba.n = 1;
    ba.s = d_in;
    ba.theta = d_in + 1;
    for (int j = 0; j < n_params; j++)
        ba.params[j] = d_in + 2 + j;
    ba.n_params = n_params;
    ba.norm = d_in + 2 + n_params;
    ba.eps_gamma = ba.eps_n = 1e-3;
    DiagArgs g{coeff, stokes, what, (long long)count, d_a, b ? d_b : nullptr, d_out, d_status};

    if (dispatch_kind(kind, [&](auto k) {
            constexpr int KIND = decltype(k)::value;
            return stage_normalize<KIND>(ba, c.sm_count, c.stream) ||
                   stage_symphony_diag<KIND>(ba, g, c.sm_count, c.stream);
        }))
        return 1;
    RB_CUDA(cudaMemcpyAsync(out, d_out, (size_t)count * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    if (status)
        RB_CUDA(cudaMemcpyAsync(status, d_status, (size_t)count * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    RB_CUDA(cudaStreamSynchronize(c.stream));
    return 0;
}

int rimphony_b200_bessel_jn(int64_t count, const double *n, const double *x, double *j, double *dj)
{
    if (count < 0 || !n || !x || !j || !dj)
        return fail("bad arguments");
    if (count == 0)
        return 0;
    DeviceContext *cp = nullptr;
    if (get_context(-1, &cp))
        return 1;
    DeviceContext &c = *cp;
    std::lock_guard<std::mutex> guard(c.lock);
    RB_CUDA(cudaSetDevice(c.device));
    const size_t bytes = (size_t)count * sizeof(double);
    if (c.in.reserve(2 * bytes) || c.out.reserve(2 * bytes))
        return 1;
    double *d_n = static_cast<double *>(c.in.ptr), *d_x = d_n + count;
    double *d_j = static_cast<double *>(c.out.ptr), *d_dj = d_j + count;
    RB_CUDA(cudaMemcpyAsync(d_n, n, bytes, cudaMemcpyHostToDevice, c.stream));
    RB_CUDA(cudaMemcpyAsync(d_x, x, bytes, cudaMemcpyHostToDevice, c.stream));
    k_bessel<<<(unsigned)((count + 127) / 128), 128, 0, c.stream>>>(count, d_n, d_x, d_j, d_dj);
    g_launches++;
    RB_CUDA(cudaGetLastError());
    RB_CUDA(cudaMemcpyAsync(j, d_j, bytes, cudaMemcpyDeviceToHost, c.stream));
    RB_CUDA(cudaMemcpyAsync(dj, d_dj, bytes, cudaMemcpyDeviceToHost, c.stream));
    RB_CUDA(cudaStreamSynchronize(c.stream));
    return 0;
}

int rimphony_b200_dist_eval(int kind, const double *params, int n_params, int64_t count, const double *gamma,
                            const double *cos_xi, double *out3)
{
    if (count < 0 || !params || !gamma || !cos_xi || !out3)
        return fail("bad arguments");
    if (check_params(kind, n_params))
        return 1;
    if (count == 0)
        return 0;
    DeviceContext *cp = nullptr;
    if (get_context(-1, &cp))
        return 1;
    DeviceContext &c = *cp;
    std::lock_guard<std::mutex> guard(c.lock);
    RB_CUDA(cudaSetDevice(c.device));
    const size_t bytes = (size_t)count * sizeof(double);
    if (c.in.reserve(2 * bytes) || c.out.reserve(3 * bytes))
        return 1;
    double *d_g = static_cast<double *>(c.in.ptr), *d_c = d_g + count;
    double *d_o = static_cast<double *>(c.out.ptr);
    RB_CUDA(cudaMemcpyAsync(d_g, gamma, bytes, cudaMemcpyHostToDevice, c.stream));
    RB_CUDA(cudaMemcpyAsync(d_c, cos_xi, bytes, cudaMemcpyHostToDevice, c.stream));
    if (dispatch_kind(kind, [&](auto k) {
            return stage_dist_eval<decltype(k)::value>(params, n_params, count, d_g, d_c, d_o, c.stream);
        }))
        return 1;
    RB_CUDA(cudaMemcpyAsync(out3, d_o, 3 * bytes, cudaMemcpyDeviceToHost, c.stream));
    RB_CUDA(cudaStreamSynchronize(c.stream));
    return 0;
}

int rimphony_b200_last_kernel_ms(int device, float out_ms[4])
{
    if (!out_ms)
        return fail("null pointer");
    DeviceGuard restore_device;
    DeviceContext *cp = nullptr;
    if (get_context(device, &cp))
        return 1;
    memcpy(out_ms, cp->last_ms, sizeof cp->last_ms);
    return 0;
}

int rimphony_b200_fp64_peak_tflops(int device, double *out_tflops)
{
    if (!out_tflops)
        return fail("null pointer");
    DeviceGuard restore_device;
    DeviceContext *cp = nullptr;
    if (get_context(device, &cp))
        return 1;
    DeviceContext &c = *cp;
    std::lock_guard<std::mutex> guard(c.lock);
    RB_CUDA(cudaSetDevice(c.device));
    if (c.counters.reserve(4 * sizeof(unsigned long long)))
        return 1;
    const int blocks = c.sm_count * 8, threads = 256, iters = 1 << 15;
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        RB_CUDA(cudaEventRecord(c.ev[6], c.stream));
        k_dfma_peak<<<blocks, threads, 0, c.stream>>>(static_cast<double *>(c.counters.ptr), iters, 1.0000001, 0.9999999);
        g_launches++;
        RB_CUDA(cudaGetLastError());
        RB_CUDA(cudaEventRecord(c.ev[7], c.stream));
        RB_CUDA(cudaEventSynchronize(c.ev[7]));
        float ms = 0;
        RB_CUDA(cudaEventElapsedTime(&ms, c.ev[6], c.ev[7]));
        const double flops = 2.0 * 16.0 * (double)iters * (double)blocks * (double)threads;
        const double tf = flops / (ms * 1e-3) * 1e-12;
        if (rep > 0 && tf > best)
            best = tf;
    }
    *out_tflops = best;
    return 0;
}

int rimphony_b200_transfer(int64_t n_rays, int64_t n_cells, const double *coeffs8, const double *psi, const double *ds,
                           const double *stokes0, double *stokes4, int32_t *status)
{
    int64_t n;
    if (check_transfer(n_rays, n_cells, coeffs8, psi, ds, stokes4, &n))
        return 1;
    if (n_rays == 0)
        return 0;
    DeviceGuard restore_device;
    DeviceContext *cp = nullptr;
    if (get_context(-1, &cp))
        return 1;
    DeviceContext &c = *cp;
    std::lock_guard<std::mutex> guard(c.lock);
    RB_CUDA(cudaSetDevice(c.device));

    // device staging: [coeffs8 | psi | ds | stokes0] in, [stokes4 | status] out
    const size_t nb = (size_t)n * sizeof(double), rb4 = 4 * (size_t)n_rays * sizeof(double);
    if (c.in.reserve(10 * nb + rb4) || c.out.reserve(rb4 + (size_t)n_rays * sizeof(int32_t)))
        return 1;
    double *d_coeffs = static_cast<double *>(c.in.ptr), *d_psi = d_coeffs + 8 * n, *d_ds = d_psi + n;
    double *d_s0 = stokes0 ? d_ds + n : nullptr;
    double *d_stokes = static_cast<double *>(c.out.ptr);
    int32_t *d_status = reinterpret_cast<int32_t *>(d_stokes + 4 * n_rays);
    if (n > 0) {
        RB_CUDA(cudaMemcpyAsync(d_coeffs, coeffs8, 8 * nb, cudaMemcpyHostToDevice, c.stream));
        RB_CUDA(cudaMemcpyAsync(d_psi, psi, nb, cudaMemcpyHostToDevice, c.stream));
        RB_CUDA(cudaMemcpyAsync(d_ds, ds, nb, cudaMemcpyHostToDevice, c.stream));
    }
    if (stokes0)
        RB_CUDA(cudaMemcpyAsync(d_s0, stokes0, rb4, cudaMemcpyHostToDevice, c.stream));
    RB_CUDA(launch_transfer(n_rays, n_cells, d_coeffs, d_psi, d_ds, d_s0, nullptr, d_stokes, d_status, c.stream));
    g_launches++;
    RB_CUDA(cudaMemcpyAsync(stokes4, d_stokes, rb4, cudaMemcpyDeviceToHost, c.stream));
    if (status)
        RB_CUDA(cudaMemcpyAsync(status, d_status, (size_t)n_rays * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    RB_CUDA(cudaStreamSynchronize(c.stream));
    return 0;
}

int rimphony_b200_transfer_device(int64_t n_rays, int64_t n_cells, const double *coeffs8, const double *psi,
                                  const double *ds, const double *stokes0, double *stokes4, int32_t *status,
                                  void *stream, int synchronize)
{
    int64_t n;
    if (check_transfer(n_rays, n_cells, coeffs8, psi, ds, stokes4, &n))
        return 1;
    if (n_rays == 0)
        return 0;
    DeviceGuard restore_device;
    DeviceContext *cp = nullptr;
    if (get_context(-1, &cp))
        return 1;
    DeviceContext &c = *cp;
    std::lock_guard<std::mutex> guard(c.lock);
    RB_CUDA(cudaSetDevice(c.device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : c.stream;
    RB_CUDA(launch_transfer(n_rays, n_cells, coeffs8, psi, ds, stokes0, nullptr, stokes4, status, st));
    g_launches++;
    if (synchronize)
        RB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int rimphony_b200_compute_stokes_cgs(int kind, int64_t n_rays, int64_t n_cells, const double *nu, const double *b,
                                     const double *n_e, const double *theta, const double *psi, const double *ds,
                                     const double *const *params, int n_params, const rimphony_b200_options *opts,
                                     double *stokes4, double *coeffs8_cgs, int32_t *status)
{
    int64_t n;
    if (check_rays(n_rays, n_cells, &n))
        return 1;
    ResolvedOptions o;
    if (check_batch(kind, n, nu, theta, params, n_params, stokes4, opts, &o))
        return 1;
    if (n_rays == 0)
        return 0;
    if (!stokes4)
        return fail("null array pointer");
    if (n == 0) { // rays without cells: nothing enters, nothing is emitted
        for (int64_t i = 0; i < 4 * n_rays; i++)
            stokes4[i] = 0.0;
        if (status)
            memset(status, 0, (size_t)n_rays * sizeof(int32_t));
        return 0;
    }
    if (!b || !n_e || !psi || !ds)
        return fail("null array pointer");
    if (o.coeff_mask != 0xFFu)
        return fail("compute_stokes_cgs needs all eight coefficients: coeff_mask must be 0 or 0xFF, got 0x%x",
                    o.coeff_mask);
    for (int j = 0; j < n_params; j++)
        if (!params[j])
            return fail("params[%d] is null", j);
    DeviceGuard restore_device;
    DeviceContext *cp = nullptr;
    if (get_context(o.device, &cp))
        return 1;
    DeviceContext &c = *cp;
    std::lock_guard<std::mutex> guard(c.lock);
    RB_CUDA(cudaSetDevice(c.device));

    // device staging: [nu | b | n_e | theta | psi | ds | s | param columns] in,
    // [out8 | norm | stokes4 | cell status | ray status] out
    const size_t nb = (size_t)n * sizeof(double);
    size_t in_doubles = 7 * (size_t)n;
    for (int j = 0; j < n_params; j++)
        in_doubles += ((o.bcast >> j) & 1u) ? 1 : (size_t)n;
    const size_t out_bytes = 9 * nb + 4 * (size_t)n_rays * sizeof(double) + (size_t)(n + n_rays) * sizeof(int32_t);
    if (c.in.reserve(in_doubles * sizeof(double)) || c.out.reserve(out_bytes))
        return 1;
    double *d_nu = static_cast<double *>(c.in.ptr), *d_b = d_nu + n, *d_ne = d_b + n, *d_theta = d_ne + n;
    double *d_psi = d_theta + n, *d_ds = d_psi + n, *d_s = d_ds + n;
    const double *host_cols[6] = {nu, b, n_e, theta, psi, ds};
    for (int k = 0; k < 6; k++)
        RB_CUDA(cudaMemcpyAsync(d_nu + k * n, host_cols[k], nb, cudaMemcpyHostToDevice, c.stream));
    const double *d_params[kMaxParams] = {};
    double *cur = d_s + n;
    for (int j = 0; j < n_params; j++) {
        const size_t cnt = ((o.bcast >> j) & 1u) ? 1 : (size_t)n;
        RB_CUDA(cudaMemcpyAsync(cur, params[j], cnt * sizeof(double), cudaMemcpyHostToDevice, c.stream));
        d_params[j] = cur;
        cur += cnt;
    }
    double *d_out8 = static_cast<double *>(c.out.ptr), *d_norm = d_out8 + 8 * n, *d_stokes = d_norm + n;
    int32_t *d_cell_status = reinterpret_cast<int32_t *>(d_stokes + 4 * n_rays), *d_status = d_cell_status + n;

    RB_CUDA(launch_cgs_s(n, d_nu, d_b, d_s, c.stream));
    g_launches++;
    rimphony_b200_extras dev_extras;
    dev_extras.lobes4 = nullptr;
    dev_extras.counters = nullptr;
    dev_extras.norm = d_norm;
    if (run_device(kind, n, d_s, d_theta, d_params, n_params, o, d_out8, d_cell_status, &dev_extras, nullptr, 0, c))
        return 1;
    RB_CUDA(launch_cgs_scale(n, d_nu, d_ne, d_out8, c.stream));
    g_launches++;
    RB_CUDA(launch_transfer(n_rays, n_cells, d_out8, d_psi, d_ds, nullptr, d_cell_status, d_stokes, d_status, c.stream));
    g_launches++;

    RB_CUDA(cudaMemcpyAsync(stokes4, d_stokes, 4 * (size_t)n_rays * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    if (coeffs8_cgs)
        RB_CUDA(cudaMemcpyAsync(coeffs8_cgs, d_out8, 8 * nb, cudaMemcpyDeviceToHost, c.stream));
    if (status)
        RB_CUDA(cudaMemcpyAsync(status, d_status, (size_t)n_rays * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    RB_CUDA(cudaStreamSynchronize(c.stream));
    return collect_times(c);
}

uint64_t rimphony_b200_kernel_launch_count(void) { return g_launches.load(); }

int rimphony_b200_device_count(void)
{
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess)
        return 0;
    return count;
}

int rimphony_b200_abi_version(void) { return RIMPHONY_B200_ABI_VERSION; }

const char *rimphony_b200_last_error(void) { return g_error.c_str(); }

void rimphony_b200_shutdown(void)
{
    std::lock_guard<std::mutex> g(g_ctx_lock);
    for (auto &c : g_ctx) {
        if (!c.ready)
            continue;
        cudaSetDevice(c.device);
        c.in.release();
        c.out.release();
        c.scratch.release();
        c.counters.release();
        c.reroute.release();
        c.handover.release();
        c.order.release();
        for (auto &e : c.ev)
            cudaEventDestroy(e);
        cudaEventDestroy(c.ev_done);
        c.have_done = false;
        cudaStreamDestroy(c.stream);
        cudaStreamDestroy(c.stream_hey);
        c.ready = false;
    }
}

} // extern "C"
