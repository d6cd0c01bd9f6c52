// rb_kernels.cuh -- the sm_100a kernels and their launch code.  Included by the
// inst_*.cu translation units only.
#pragma once

#include "rb_launch.cuh"

namespace rbhost {

// ---------------------------------------------------------------------------
// kernels

template <int KIND>
__global__ void __launch_bounds__(kThreadsPerBlock) k_normalize(BatchArgs a)
{
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5;
    double *store = smem + (size_t)warp * kNormCap * IntervalList<1>::doubles_per_interval;
    Warp w;
    w.init();
    const long long stride = (long long)gridDim.x * kWarpsPerBlock;
    for (long long i = (long long)blockIdx.x * kWarpsPerBlock + warp; i < a.n; i += stride) {
        w.status = 0;
        Dist d;
        double p0;
        bool ok = load_dist<KIND>(a, i, d, p0);
        if (ok) {
            IntervalList<1> list;
            list.bind(store, kNormCap);
            ok = dist_normalize<KIND>(w, d, p0, list);
        }
        if (w.lane == 0) {
            a.norm[i] = ok ? d.norm : NAN;
            if (a.status && (!ok || w.status))
                atomicOr(&a.status[i], (int)(w.status | (ok ? 0u : kStatusNormFailed)));
        }
    }
}

// Lane 0's write-back of one point: the requested coefficient slots FIRST.. of out8, the lobes
// (Symphony only: `lobes4` is null for Heyvaerts), the work-counter row of the kernel and the
// status bits, in that order (writing the lobes first changes the register allocation of k_symphony_fast).
// CONTINUATION: the kernel may run as the faithful continuation of the product kernel
// (a.from_reroute_list), whose rule applications go on top of what the product kernel counted.
template <int FIRST, bool CONTINUATION = false, int NC>
__device__ __forceinline__ void write_point(const BatchArgs &a, const Warp &w, long long i, const double (&out)[NC],
                                            const double *lobes4)
{
    bool any_nan = false;
#pragma unroll
    for (int c = 0; c < NC; c++) {
        if ((a.coeff_mask >> (FIRST + c)) & 1u) {
            a.out8[(long long)(FIRST + c) * a.n + i] = out[c];
            any_nan |= !(out[c] == out[c]);
        }
    }
    if (lobes4 && a.lobes4) {
#pragma unroll
        for (int c = 0; c < 4; c++)
            a.lobes4[(long long)c * a.n + i] = lobes4[c];
    }
    if (a.counters) {
        unsigned *row = a.counters + (FIRST ? a.n : 0);
        if (CONTINUATION && a.from_reroute_list)
            atomicAdd(&row[i], w.n_apply_lanes);
        else
            row[i] = w.n_apply_lanes;
    }
    const unsigned st = w.status | (any_nan ? kStatusNaN : 0u);
    if (a.status && st)
        atomicOr(&a.status[i], (int)st);
}

template <int KIND, bool FUSED>
__global__ void __launch_bounds__(kThreadsPerBlock, FUSED ? 3 : 4) k_symphony(BatchArgs a)
{
    using WS = SymWorkspace<FUSED, kSymGammaCap, kSymNCap>;
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5;
    WS &ws = reinterpret_cast<WS *>(smem)[warp];
    Warp w;
    w.init();

    for (;;) {
        long long i = next_point(a.next, w.lane);
        long long slot = i;
        int acc = -1; // >= 0: this warp finishes ONE accumulator of a handed point
        if (a.from_reroute_list) {
            // The faithful continuation (fidelity guard of rb_symfast.cuh).  A ticket is (handed point, accumulator):
            // the 2-4 accumulators of a point that are still being integrated replay the reference's sequence
            // independently of each other (100-250 k rule applications each), so each gets its own warp; the warp
            // that finishes last puts the point together.  With fewer handed points than warps (any batch below
            // ~1e5 points) the launch is as long as its longest chain, which this cuts by the number of chains.
            slot = i >> 3;
            acc = (int)(i & 7);
            if (slot >= (long long)*a.reroute_count)
                break;
            i = a.reroute_list[slot];
        } else if (i >= a.n)
            break;
        w.status = 0;
        w.n_apply_lanes = 0;

        Dist d;
        double p0;
        load_dist<KIND>(a, i, d, p0);
        d.norm = a.norm[i];

        double out6[6], lobes4[4];
        bool resumed = false;
        if constexpr (!FUSED) {
            if (a.from_reroute_list) {
                double *snap = a.handover + (size_t)slot * kSnapDoubles;
                if (snap[kSnapValid] == 1.0) { // resume the chunk loop where the product path stopped
                    const unsigned active = (unsigned)snap[kSnapActive];
                    if (active != 0u) {
                        if (!((active >> acc) & 1u))
                            continue; // nothing to integrate for this accumulator: its total is already in the record
                        const double total = symphony_tail_faithful_one<KIND, kSymGammaCap, kSymNCap>(
                            w, d, a.s[i], a.theta[i], a.eps_gamma, a.eps_n, ws, snap, acc);
                        // hand the total in (the slot of this accumulator's last chunk: nobody else reads it), count out
                        double done = 0.0;
                        if (w.lane == 0) {
                            snap[kSnapContrib + acc] = total;
                            if (a.counters)
                                atomicAdd(&a.counters[i], w.n_apply_lanes);
                            if (a.status && w.status)
                                atomicOr(&a.status[i], (int)w.status);
                            __threadfence();
                            done = atomicAdd(&snap[kSnapDone], 1.0) + 1.0;
                        }
                        done = __shfl_sync(0xffffffffu, done, 0);
                        if (done != (double)__popc(active))
                            continue; // another warp of this point is still at work
                        __threadfence();
                    } else if (acc != 0)
                        continue; // (a record without a chain left: the first ticket writes the point out)
                    double totals[kSymNA];
#pragma unroll
                    for (int c = 0; c < kSymNA; c++) {
                        const volatile double *vs = snap;
                        totals[c] = ((active >> c) & 1u) ? vs[kSnapContrib + c] : vs[kSnapDisc + c] + vs[kSnapTail + c];
                    }
                    symphony_tail_combine(a.theta[i], totals, out6, lobes4);
                    w.n_apply_lanes = 0; // counted above
                    w.status = 0;
                    resumed = true;
                } else if (acc != 0)
                    continue; // a point that starts over (s < 10) is one chain: the first ticket takes all of it
            }
        }
        if (!resumed)
            symphony_point<KIND, FUSED, kSymGammaCap, kSymNCap>(w, d, a.s[i], a.theta[i], a.eps_gamma, a.eps_n, ws,
                                                                out6, lobes4);

        if (w.lane == 0)
            write_point<0, true>(a, w, i, out6, lobes4);
    }
}

// diagnostic_symphony_* (lib.rs:254-298): one warp per argument, reference rule sequence.
template <int KIND>
__global__ void __launch_bounds__(kThreadsPerBlock, 4) k_symphony_diag(BatchArgs a, DiagArgs g)
{
    using WS = SymWorkspace<false, kSymGammaCap, kSymNCap>;
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5;
    WS &ws = reinterpret_cast<WS *>(smem)[warp];
    Warp w;
    w.init();

    Dist d;
    double p0;
    load_dist<KIND>(a, 0, d, p0);
    d.norm = a.norm[0];
    const double s = a.s[0], theta = a.theta[0];

    const long long stride = (long long)gridDim.x * kWarpsPerBlock;
    for (long long i = (long long)blockIdx.x * kWarpsPerBlock + warp; i < g.count; i += stride) {
        w.status = 0;
        w.n_apply_lanes = 0;
        const double v = symphony_diagnostic<KIND, kSymGammaCap, kSymNCap>(w, d, g.coeff, g.stokes, s, theta, g.what,
                                                                           g.a[i], g.b ? g.b[i] : 0.0, a.eps_gamma,
                                                                           a.eps_n, ws);
        if (w.lane == 0) {
            g.out[i] = v;
            if (g.status)
                g.status[i] = (int)(w.status | ((v == v) ? 0u : kStatusNaN));
        }
    }
}

constexpr int kFastBlocks = 5; // resident CTAs per SM the product kernels are compiled for (96 registers; +5 % over 4)
constexpr int kHeyBlocks = 8;  // the Heyvaerts kernel (64 registers; its tiles have two channel rows, 14 KB per CTA).  5 -> 8 CTAs per SM: -13 % kernel time; 10 (48 registers) is as fast but its 768 B of stack per thread x 1280 threads x 148 SMs no longer fit the L2 and 0.7 MB per point go to DRAM (0.1 MB at 8)
constexpr int kFastWarps = 4;  // warps per CTA of the product kernels
constexpr int kFastThreads = kFastWarps * 32;

// The product path: compact engine (rb_engine.cuh, rb_symfast.cuh).
template <int KIND>
__global__ void __launch_bounds__(kFastThreads, kFastBlocks) k_symphony_fast(BatchArgs a)
{
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5;
    SymFastWS &ws = reinterpret_cast<SymFastWS *>(smem)[warp];
    Warp w;
    w.init();

    for (;;) {
        const long long ticket = next_point(a.next, w.lane);
        if (ticket >= a.n)
            break;
        const long long i = ordered_point(a, 0, ticket);
        w.status = 0;
        w.n_apply_lanes = 0;

        Dist d;
        double p0;
        load_dist<KIND>(a, i, d, p0);
        d.norm = a.norm[i];

        double out6[6], lobes4[4];
        symphony_point_fast<KIND>(w, d, a.s[i], a.theta[i], a.eps_gamma, a.eps_n, ws, out6, lobes4);

        if (w.status & kStatusRerouted) {
            // fidelity guard (rb_symfast.cuh): the faithful kernel computes this point, resuming
            // from the recorded chunk-loop state when there is one
            unsigned long long slot = 0;
            if (w.lane == 0) {
                slot = atomicAdd(a.reroute_count, 1ULL);
                a.reroute_list[slot] = (int)i;
                if (a.counters)
                    a.counters[i] = w.n_apply_lanes;
                if (a.status)
                    atomicOr(&a.status[i], (int)kStatusRerouted);
            }
            slot = __shfl_sync(0xffffffffu, slot, 0);
            __syncwarp();
            a.handover[slot * kSnapDoubles + w.lane] = ws.snap[w.lane];
            continue;
        }

        if (w.lane == 0)
            write_point<0>(a, w, i, out6, lobes4);
    }
}

template <int KIND, bool FUSED>
__global__ void __launch_bounds__(kThreadsPerBlock, 4) k_heyvaerts(BatchArgs a)
{
    using WS = HeyWorkspace<FUSED, kHeyInnerCap, kHeyOuterCap>;
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5;
    WS &ws = reinterpret_cast<WS *>(smem)[warp];
    Warp w;
    w.init();

    for (;;) {
        const long long i = next_point(a.next, w.lane);
        if (i >= a.n)
            break;
        const double s = a.s[i], theta = a.theta[i];
        const double sigma0 = s * sin(theta);
        if (!(sigma0 >= a.sigma0_lo && sigma0 < a.sigma0_hi) && !(a.sigma0_lo < 0.0 && !(sigma0 == sigma0)))
            continue; // another launch owns this point (NaN sigma0 goes with the lowest band)
        w.status = 0;
        w.n_apply_lanes = 0;

        Dist d;
        double p0;
        load_dist<KIND>(a, i, d, p0);
        d.norm = a.norm[i];

        double out2[2];
        heyvaerts_point<KIND, FUSED, kHeyInnerCap, kHeyOuterCap>(w, d, s, theta, a.eps_hey_inner, a.eps_hey_outer, ws,
                                                                 out2);

        if (w.lane == 0)
            write_point<6>(a, w, i, out2, nullptr);
    }
}

// The product path for rho_Q, rho_V: compact engine (rb_engine.cuh, rb_heyfast.cuh).
template <int KIND>
__global__ void __launch_bounds__(kFastThreads, kHeyBlocks) k_heyvaerts_fast(BatchArgs a)
{
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5;
    HeyFastWS &ws = reinterpret_cast<HeyFastWS *>(smem)[warp];
    Warp w;
    w.init();

    for (;;) {
        const long long ticket = next_point(a.next, w.lane);
        if (ticket >= a.n)
            break;
        const long long i = ordered_point(a, 1, ticket);
        w.status = 0;
        w.n_apply_lanes = 0;

        Dist d;
        double p0;
        load_dist<KIND>(a, i, d, p0);
        d.norm = a.norm[i];

        double out2[2];
        heyvaerts_point_fast<KIND>(w, d, a.s[i], a.theta[i], a.eps_hey_inner, a.eps_hey_outer, ws, out2);

        if (w.lane == 0)
            write_point<6>(a, w, i, out2, nullptr);
    }
}

template <int KIND>
__global__ void k_dist_eval(Dist d, long long count, const double *gamma, const double *cos_xi, double *out3)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count)
        return;
    double f, a, b;
    dist_eval<KIND>(d, gamma[i], cos_xi[i], f, a, b);
    out3[i] = f;
    out3[count + i] = a;
    out3[2 * count + i] = b;
}


// ---------------------------------------------------------------------------
// stage launchers

// One persistent launch: every CTA slot the device holds at once (`threads` per CTA, `smem` bytes of
// dynamic shared memory each), but no more CTAs than `max_ctas` when that is positive.
template <class... P, class... A>
int launch_persistent(void (*kernel)(P...), size_t smem, int threads, long long max_ctas, int sm_count, cudaStream_t st,
                      const A &...args)
{
    RB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    RB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1)
        return fail("kernel does not fit on an SM (smem %zu)", smem);
    int grid = per_sm * sm_count; // a multiple of the SM count
    if (max_ctas > 0 && max_ctas < grid)
        grid = (int)max_ctas;
    kernel<<<grid, threads, smem, st>>>(args...);
    g_launches++;
    RB_CUDA(cudaGetLastError());
    return 0;
}

template <int KIND>
int stage_normalize(const BatchArgs &a, int sm_count, cudaStream_t st)
{
    const size_t smem = (size_t)kWarpsPerBlock * kNormCap * IntervalList<1>::doubles_per_interval * sizeof(double);
    return launch_persistent(k_normalize<KIND>, smem, kThreadsPerBlock, (a.n + kWarpsPerBlock - 1) / kWarpsPerBlock,
                             sm_count, st, a);
}

template <int KIND, bool FUSED>
int stage_symphony(const BatchArgs &a, int sm_count, cudaStream_t st)
{
    const size_t smem = kWarpsPerBlock * sizeof(SymWorkspace<FUSED, kSymGammaCap, kSymNCap>);
    return launch_persistent(k_symphony<KIND, FUSED>, smem, kThreadsPerBlock, 0, sm_count, st, a);
}

template <int KIND>
int stage_symphony_diag(const BatchArgs &a, const DiagArgs &g, int sm_count, cudaStream_t st)
{
    const size_t smem = kWarpsPerBlock * sizeof(SymWorkspace<false, kSymGammaCap, kSymNCap>);
    return launch_persistent(k_symphony_diag<KIND>, smem, kThreadsPerBlock, (g.count + kWarpsPerBlock - 1) / kWarpsPerBlock,
                             sm_count, st, a, g);
}

template <int KIND>
int stage_symphony_fast(const BatchArgs &a, int sm_count, cudaStream_t st)
{
    return launch_persistent(k_symphony_fast<KIND>, kFastWarps * sizeof(SymFastWS), kFastThreads, 0, sm_count, st, a);
}

template <int KIND, bool FUSED>
int stage_heyvaerts(const BatchArgs &a, int sm_count, cudaStream_t st)
{
    const size_t smem = kWarpsPerBlock * sizeof(HeyWorkspace<FUSED, kHeyInnerCap, kHeyOuterCap>);
    return launch_persistent(k_heyvaerts<KIND, FUSED>, smem, kThreadsPerBlock, 0, sm_count, st, a);
}

template <int KIND>
int stage_heyvaerts_fast(const BatchArgs &a, int sm_count, cudaStream_t st)
{
    return launch_persistent(k_heyvaerts_fast<KIND>, kFastWarps * sizeof(HeyFastWS), kFastThreads, 0, sm_count, st, a);
}

template <int KIND>
int stage_dist_eval(const double *params, int n_params, long long count, const double *gamma, const double *cos_xi,
                    double *out3, cudaStream_t st)
{
    Dist d;
    dist_from_params<KIND>(params, n_params, d);
    d.norm = 1.0;
    k_dist_eval<KIND><<<(unsigned)((count + 127) / 128), 128, 0, st>>>(d, count, gamma, cos_xi, out3);
    g_launches++;
    RB_CUDA(cudaGetLastError());
    return 0;
}

} // namespace rbhost
