// Arguments of one half-update launch of the tiled KL engine (kl_tiled.cuh, kl_tiled_tc.cu).
#pragma once
#include "nmfk_internal.h"

namespace nmfk {

struct TiledPassArgs {
    const void* D;      // data in "own-contiguous" layout: element (o,t) at D[o + t*nown]
    void* U;            // own factor stack
    const void* V;      // broadcast factor stack
    const void* den;    // R x kTiledMaxK : sum_t V[t,a]
    void* partial;      // slices x R x nown x K partial numerators (S > 1) or nullptr
    const UnitState* st;
    const void* ximp;   // R x n x m (X layout) or nullptr
    long long u_rstride, v_rstride;  // elements between restarts
    long long su_o, su_a, sv_t, sv_a;
    int nown, nred, k, R, S, nblocks;
    int transposed;     // 1: D is X^T (H-update) -> imputation index = t + o*ldimp
    int ldimp;
    int has_nan, first_iter;
    double lambda;
    // objective mode (tc_objective): sum over non-NaN entries of (x - U V^T)^2 per restart and block of 128 own indices
    double* obj_partials;  // [(r * nblocks + block) * 2 + {0: weighted, 1: plain}]
    double obj_weight;
    int obj_restore;       // 1: substituted zeros (x == lambda) count as 0 (final objective on the restored X)
    int obj_sel;           // 0: running restarts (stop == 0); 1: restarts that stopped and are not finished (done == 0)
    int wait_hint_ns;      // nanosleep between barrier polls: low 16 bits X producer, high 16 bits V stagers
    int qwait_ns;          // nanosleep between the quotient warps' polls of p_full (0 = spin)
    long long* trace;   // debug: clock64 stamps of CTA 0 ([role][unit < 64][8]); nullptr in production
    int ktmpl;          // column stride of `partial` (the template K of the combine kernel)
    const void* Dstep;  // the same data STEP-contiguous: element (o,t) at Dstep[t + o*nred] (tc2 pass: X tiles)
    void* vimg;         // tc2 pass: scratch for the V operand images, tc2_image_bytes(k, R, nred) bytes
};

// Float32 half-update on the 5th-generation tensor cores (kl_tiled_tc.cu): tcgen05.mma kind::tf32 with the
// 3-term split, accumulators / quotient tiles in tensor memory.  nblocks = ceil(nown / 128), grid =
// S x nblocks x ceil(R / tc_pass_group(k)).
bool tc_pass_supported(const TiledPassArgs& a);
int tc_pass_group(int k);  // restarts that share one X tile inside a CTA
int tc_pass_ctas_per_sm(int k);
int tc_pass_chunk(int k);  // steps per chunk (slices hold whole chunks)
// div: the quotient flavour of Variant KL_DIV, x / (p + kKlDivDelta) (a.den must already hold the sums + kKlDivDelta)
cudaError_t launch_tc_pass(const TiledPassArgs& a, int* d_errflag, cudaStream_t s, bool div = false);
// second generation for k <= 16 (kl_tiled_tc2.cu): U in shared memory, separate P and Q tiles; same grid and arguments
bool tc2_pass_enabled(int k);
cudaError_t launch_tc2_pass(const TiledPassArgs& a, int* d_errflag, cudaStream_t s, bool div = false);
// scratch of the tc2 pass (a.vimg): the V operand images of R restarts over a reduction range of nred steps (0: the pass does
// not serve k).  A launch first builds the images of its running restarts there, then the pass copies them into shared memory.
size_t tc2_image_bytes(int k, int R, int nred);
// one-time host-side set-up (driver entry point of the tensor-map encoder, kernel attributes): called when a context is
// created so that it never falls inside a timed solve
void tc2_pass_prepare();
// Float32 objective sums on the same machinery (MMA#1 only): a = the W-update arguments (D = X, U = W, V = H), S = 1
cudaError_t launch_tc_objective(const TiledPassArgs& a, int* d_errflag, cudaStream_t s);

// Float64 half-update on the FP64 tensor pipe (kl_tiled_dmma.cu): DMMA fragment formulation of the resident engine with
// the other factor streamed through shared memory.  a.D = STEP-contiguous data (H-update: X, W-update: X^T),
// nblocks = ceil(nown / tiled_dmma_own()), 4 <= k <= 64, no NaN.
int tiled_dmma_own();
int tiled_dmma_chunk();
cudaError_t launch_tiled_dmma_pass(const TiledPassArgs& a, cudaStream_t s, bool div = false);
cudaError_t launch_tiled_dmma_objective(const TiledPassArgs& a, cudaStream_t s);

// NMF.jl stop_condition after an iteration (fro_solve.cu's fro_converge_kernel): restarts whose every column of W and row of H
// moved by less than tol relative stop with reason 2.  convW / convH: per-tile sums, [((r * tiles + tile) * k + a) * 2 + {0,1}]
cudaError_t launch_fro_converge(UnitState* st, int R, int k, const double* convW, int tilesW, const double* convH, int tilesH,
                                int wactive, int hactive, double tol, int it, cudaStream_t s);

}  // namespace nmfk
