// Float64 instantiation of the tiled KL engine (see kl_tiled.cuh).
#include "kl_tiled.cuh"

namespace nmfk {
cudaError_t solve_tiled_f64(const SolveArgs& a, cudaStream_t s, int64_t* launches, bool div) {
    return solve_tiled_t<double, double>(a, s, launches, div);
}
}  // namespace nmfk
