// tests/hostemu_transfer/hostemu_transfer.cpp -- DEVELOPMENT HARNESS, not part of the product.
// The host build of rimphony_b200/csrc/rb_transfer.cuh: emu_transfer is rimphony_b200_transfer with the same
// propagator source run on the CPU, one ray after the other.
#include "../../rimphony_b200/csrc/rb_transfer.cuh"

extern "C" void emu_transfer(long long n_rays, long long n_cells, const double *coeffs8, const double *psi,
                             const double *ds, const double *stokes0, double *stokes4, int *status)
{
    for (long long r = 0; r < n_rays; r++) {
        const unsigned st = rb::transfer_ray(r, n_rays, n_cells, coeffs8, psi, ds, stokes0, stokes4);
        if (status)
            status[r] = (int)st;
    }
}
