// explicit instantiation: normalisation, Heyvaerts and dist_eval kernels, distribution kind 2
#include "rb_kernels.cuh"
namespace rbhost {
template int stage_normalize<rb::kDistPitchyPL>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistPitchyPL, false>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistPitchyPL, true>(const BatchArgs &, int, cudaStream_t);
template int stage_dist_eval<rb::kDistPitchyPL>(const double *, int, long long, const double *, const double *, double *,
                                       cudaStream_t);
}
