// explicit instantiation: product-path (fast) Heyvaerts kernel, distribution kind 4
#define RB_LEAN_MATH 1 // lean division, exp and log (rb_core.cuh)
#include "rb_kernels.cuh"
namespace rbhost {
template int stage_heyvaerts_fast<rb::kDistPitchyBrokenPL>(const BatchArgs &, int, cudaStream_t);
}
