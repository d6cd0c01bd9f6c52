/* tests/bpl_oracle/bpl_oracle_base.c -- TEST INFRASTRUCTURE ONLY.
 *
 * The CPU oracle (oracle/rimphony_oracle.c), compiled unchanged, with its three distribution entry points
 * made weak.  bpl_oracle.c defines them again with PITCHY_BROKEN_PL added; the library is linked with
 * -Bsymbolic, so every call the Symphony and Heyvaerts restatements make to them lands there, and the
 * reference's algorithm runs on the new distribution function.  The originals stay reachable under the
 * names orc_*_base for the other kinds. */
#pragma weak orc_dist_init
#pragma weak orc_calc_f
#pragma weak orc_calc_f_derivatives

#include "rimphony_oracle.c"

extern int orc_dist_init_base(orc_dist *d, int kind, const double *params, int n_params)
    __attribute__((alias("orc_dist_init")));
extern double orc_calc_f_base(const orc_dist *d, double gamma, double cos_xi) __attribute__((alias("orc_calc_f")));
extern void orc_calc_f_derivatives_base(const orc_dist *d, double gamma, double cos_xi, double *dfdg, double *dfdcx)
    __attribute__((alias("orc_calc_f_derivatives")));
