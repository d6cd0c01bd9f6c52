// explicit instantiation: normalisation, Heyvaerts and dist_eval kernels, distribution kind 4
#include "rb_kernels.cuh"
namespace rbhost {
template int stage_normalize<rb::kDistPitchyBrokenPL>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistPitchyBrokenPL, false>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistPitchyBrokenPL, true>(const BatchArgs &, int, cudaStream_t);
template int stage_dist_eval<rb::kDistPitchyBrokenPL>(const double *, int, long long, const double *, const double *, double *,
                                              cudaStream_t);
}
