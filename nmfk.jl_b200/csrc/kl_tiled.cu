// Tiled KL engine: dtype dispatch (kernels and host driver live in kl_tiled.cuh).
#include "nmfk_internal.h"

namespace nmfk {

cudaError_t solve_tiled_f64(const SolveArgs& a, cudaStream_t s, int64_t* launches);
cudaError_t solve_tiled_f32(const SolveArgs& a, cudaStream_t s, int64_t* launches);

bool tiled_supported(int k) { return k >= 1 && k <= kTiledMaxK; }

cudaError_t solve_tiled(const SolveArgs& a, int dtype, cudaStream_t s, int64_t* launches) {
    return dtype == 1 ? solve_tiled_f64(a, s, launches) : solve_tiled_f32(a, s, launches);
}

}  // namespace nmfk
