// tests/hostemu_bpl/hostemu_bpl.cpp -- DEVELOPMENT HARNESS (see tests/hostemu/hostemu.cpp), not part of the product.
// The host build of the device headers with the pitchy broken power law (kind 4) added: emu_point_bpl is
// emu_point for that kind.  Everything else is tests/hostemu/hostemu.cpp as it stands.
#include "../hostemu/hostemu.cpp"

extern "C" int emu_point_bpl(const double *params, int n_params, int fused, int which, double s, double theta,
                             const double *eps, double *out8, double *lobes4, unsigned *info)
{
    return point_kind<kDistPitchyBrokenPL>(params, n_params, fused, which, s, theta, eps, out8, lobes4, info);
}
