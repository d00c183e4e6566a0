#include "lec_score_fast_impl.cuh"
namespace lec {
int score_fast_lorentz(FastArgs& a, cudaStream_t st) { return fast_launch_geom<LEC_GEOM_LORENTZ>(a, st); }
}  // namespace lec
