// explicit instantiation: normalisation, Heyvaerts and dist_eval kernels, distribution kind 0
#include "rb_kernels.cuh"
namespace rbhost {
template int stage_normalize<rb::kDistPowerLaw>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistPowerLaw, false>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistPowerLaw, true>(const BatchArgs &, int, cudaStream_t);
template int stage_dist_eval<rb::kDistPowerLaw>(const double *, int, long long, const double *, const double *, double *,
                                       cudaStream_t);
}
