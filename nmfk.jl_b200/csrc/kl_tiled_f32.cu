// Float32 instantiation of the tiled KL engine (see kl_tiled.cuh).
#include "kl_tiled.cuh"

namespace nmfk {
cudaError_t solve_tiled_f32(const SolveArgs& a, cudaStream_t s, int64_t* launches, bool div) {
    return solve_tiled_t<float, float>(a, s, launches, div);
}
}  // namespace nmfk
