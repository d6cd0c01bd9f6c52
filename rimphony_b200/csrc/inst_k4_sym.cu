// explicit instantiation: Symphony kernels, distribution kind 4
#define RB_LEAN_MATH 1 // lean division, exp, log and square root (rb_core.cuh): same rule sequence, -13 % time, GPU parity tests unchanged
#include "rb_kernels.cuh"
namespace rbhost {
template int stage_symphony<rb::kDistPitchyBrokenPL, false>(const BatchArgs &, int, cudaStream_t);
template int stage_symphony<rb::kDistPitchyBrokenPL, true>(const BatchArgs &, int, cudaStream_t);
template int stage_symphony_diag<rb::kDistPitchyBrokenPL>(const BatchArgs &, const DiagArgs &, int, cudaStream_t);
}
