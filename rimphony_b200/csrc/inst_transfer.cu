// inst_transfer.cu -- the polarized transfer stage (rb_transfer.cuh) and the two cgs helpers of
// rimphony_b200_compute_stokes_cgs.  A translation unit of its own, so that adding it leaves every other
// object of the library as it was.
#include "rb_transfer.cuh"

namespace {

using namespace rb;

constexpr int kTransferThreads = 128;

__global__ void __launch_bounds__(kTransferThreads)
k_transfer(long long n_rays, long long n_cells, const double *coeffs8, const double *psi, const double *ds,
           const double *stokes0, const int *cell_status, double *stokes4, int *status)
{
    const long long ray = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (ray >= n_rays)
        return;
    unsigned st = transfer_ray(ray, n_rays, n_cells, coeffs8, psi, ds, stokes0, stokes4);
    if (!status)
        return;
    if (cell_status)
        for (long long c = 0; c < n_cells; c++)
            st |= (unsigned)cell_status[ray * n_cells + c];
    status[ray] = (int)st;
}

// The same operations, in the same order, as SynchrotronCalculator.compute_all_cgs; __dmul_rn / __ddiv_rn keep
// the compiler from contracting any of them.
__global__ void k_cgs_s(long long n, const double *nu, const double *b, double *s)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const double nu_c = __ddiv_rn(__dmul_rn(kElectronCharge, b[i]), kTwoPi * kMassElectron * kSpeedLight);
    s[i] = __ddiv_rn(nu[i], nu_c);
}

__global__ void k_cgs_scale(long long n, const double *nu, const double *n_e, double *out8)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const double scale_j = __dmul_rn(n_e[i], nu[i]), scale_a = __ddiv_rn(n_e[i], nu[i]);
#pragma unroll
    for (int c = 0; c < 8; c++) {
        double &v = out8[(size_t)c * n + i];
        v = __dmul_rn(v, (c == 0 || c == 2 || c == 4) ? scale_j : scale_a);
    }
}

unsigned blocks_for(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

} // namespace

namespace rbhost {

cudaError_t launch_transfer(long long n_rays, long long n_cells, const double *coeffs8, const double *psi,
                            const double *ds, const double *stokes0, const int *cell_status, double *stokes4,
                            int *status, cudaStream_t st)
{
    k_transfer<<<blocks_for(n_rays, kTransferThreads), kTransferThreads, 0, st>>>(n_rays, n_cells, coeffs8, psi, ds,
                                                                                 stokes0, cell_status, stokes4, status);
    return cudaGetLastError();
}

cudaError_t launch_cgs_s(long long n, const double *nu, const double *b, double *s, cudaStream_t st)
{
    k_cgs_s<<<blocks_for(n, 256), 256, 0, st>>>(n, nu, b, s);
    return cudaGetLastError();
}

cudaError_t launch_cgs_scale(long long n, const double *nu, const double *n_e, double *out8, cudaStream_t st)
{
    k_cgs_scale<<<blocks_for(n, 256), 256, 0, st>>>(n, nu, n_e, out8);
    return cudaGetLastError();
}

} // namespace rbhost
