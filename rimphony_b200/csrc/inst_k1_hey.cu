// explicit instantiation: normalisation, Heyvaerts and dist_eval kernels, distribution kind 1
#include "rb_kernels.cuh"
namespace rbhost {
template int stage_normalize<rb::kDistThermalJuettner>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistThermalJuettner, false>(const BatchArgs &, int, cudaStream_t);
template int stage_heyvaerts<rb::kDistThermalJuettner, true>(const BatchArgs &, int, cudaStream_t);
template int stage_dist_eval<rb::kDistThermalJuettner>(const double *, int, long long, const double *, const double *, double *,
                                       cudaStream_t);
}
