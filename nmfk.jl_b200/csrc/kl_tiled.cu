// Tiled KL engine: dtype dispatch (kernels and host driver live in kl_tiled.cuh).
#include "nmfk_internal.h"

namespace nmfk {

cudaError_t solve_tiled_f64(const SolveArgs& a, cudaStream_t s, int64_t* launches, bool div);
cudaError_t solve_tiled_f32(const SolveArgs& a, cudaStream_t s, int64_t* launches, bool div);

bool tiled_supported(int k) { return k >= 1 && k <= kTiledMaxK; }

// div: Variant KL_DIV (NMF.jl's MultUpdate(obj=:div)) on the same engine
cudaError_t solve_tiled(const SolveArgs& a, int dtype, cudaStream_t s, int64_t* launches, bool div) {
    return dtype == 1 ? solve_tiled_f64(a, s, launches, div) : solve_tiled_f32(a, s, launches, div);
}

}  // namespace nmfk
