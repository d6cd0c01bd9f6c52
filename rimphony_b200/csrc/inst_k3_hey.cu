// explicit instantiation: normalisation, Heyvaerts and dist_eval kernels, distribution kind 3
#include "rb_kernels.cuh"
namespace rbhost {
template int stage_normalize<rb::kDistPitchyKappa>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistPitchyKappa, false>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistPitchyKappa, true>(const BatchArgs &, int, cudaStream_t);
template int stage_dist_eval<rb::kDistPitchyKappa>(const double *, int, long long, const double *, const double *, double *,
                                       cudaStream_t);
}
