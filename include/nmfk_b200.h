/*
 * nmfk_b200.h - C ABI of the B200-native NMFk factorization hot path.
 *
 * The reference (SmartTensors/NMFk.jl 1.4.21) is pure Julia and has NO FFI / plugin interface
 * for this path: its boundary is a set of Julia method signatures.  Each entry point below
 * therefore replaces a Julia function (file:line relative to /root/reference) and is what a
 * Julia `ccall` (or Python `ctypes`) binds; INTEGRATION.md shows the reference-side stubs.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no exceptions cross the boundary.
 *   - every function returns int32 status: 0 ok; <0 argument / domain error (mirrors the
 *     reference's exceptions, see NMFK_E_*); >0 CUDA error code (cudaError_t).
 *     nmfk_last_error(ctx) gives the message (ctx may be NULL for creation failures).
 *   - all matrices are COLUMN-MAJOR, contiguous (Julia `Array` memory): W is n x k, H is k x m,
 *     stacks are restart-major (W stack = n x k x R, H stack = k x m x R).
 *   - the caller owns host buffers; the library owns device memory inside nmfk_ctx.
 *   - one ctx = one CUDA device; calls on one ctx must be serialised by the caller.
 *   - dtype: NMFK_F32 / NMFK_F64 is the element type T of X and of the factor buffers.
 *   - there is NO CPU fallback: without a CUDA device nmfk_ctx_create fails.
 */
#ifndef NMFK_B200_H
#define NMFK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NMFK_ABI_VERSION 2

enum nmfk_dtype { NMFK_F32 = 0, NMFK_F64 = 1 };

/* status codes (<0): the reference's exceptions for this path */
enum nmfk_status {
    NMFK_OK = 0,
    NMFK_E_INVALID = -1,      /* bad pointer / size / enum */
    NMFK_E_NEGATIVE = -2,     /* ErrorException("All matrix entries must be nonnegative!") NMFkMultiplicative.jl:4-7 */
    NMFK_E_NAN_INIT = -3,     /* error("Initial values for the W/H matrix entries include NaNs!") :42-44,52-54 */
    NMFK_E_SHAPE = -4,        /* AssertionError size(Winit)==(n,k) :40,50 ; normalizevector length :30 */
    NMFK_E_NO_X = -5,         /* nmfk_set_X has not been called */
    NMFK_E_UNSUPPORTED = -6,  /* k or shape outside what the engines cover */
    NMFK_E_EMPTY = -7,        /* error("Input array has a zero dimension!") NMFkExecute.jl:242-244 */
    NMFK_E_NO_DEVICE = -8     /* no CUDA device / library built without one: fail loudly, never fall back */
};

/* why a restart stopped (NMFkMultiplicative.jl:64,75,112) */
enum nmfk_stop_reason {
    NMFK_STOP_PAUSED = 0,       /* iter_limit reached (trace / resumable runs) */
    NMFK_STOP_MAXITER = 1,      /* iters >= maxiter */
    NMFK_STOP_TOL = 2,          /* objvalue < tol */
    NMFK_STOP_REATTEMPTS = 3,   /* reattempts >= maxreattempts */
    NMFK_STOP_CONSISTENCY = 4,  /* inc > stopconv */
    NMFK_STOP_BADITERS = 5      /* baditers >= maxbaditers (unreachable with the reference's reset, kept for the guard) */
};

/* AUTO: resident when the factors fit in one SM's shared memory, else tiled.  RESIDENT uses the
 * tensor-pipe (DMMA m8n8k4) formulation for Float64 and the scalar-FMA one for Float32;
 * RESIDENT_SCALAR forces the scalar-FMA formulation (kept for A/B measurements and parity).
 * TILED: Float32 data without NaN (row and column counts multiples of 4) run both half-updates on the
 * 5th-generation tensor cores (tcgen05.mma kind::tf32, 3-term split, tensor-memory accumulators);
 * Float64, NaN-imputing and odd-sized problems use the scalar-FMA pass kernel. */
enum nmfk_engine {
    NMFK_ENGINE_AUTO = 0,
    NMFK_ENGINE_RESIDENT = 1,
    NMFK_ENGINE_TILED = 2,
    NMFK_ENGINE_RESIDENT_SCALAR = 3,
    NMFK_ENGINE_TILED_SCALAR = 4 /* tiled engine with the scalar-FMA pass kernel also for Float32 (A/B, parity) */
};

/* Keyword arguments of NMFmultiplicative (NMFkMultiplicative.jl:24) and of
 * execute_singlerun_compute (NMFkExecute.jl:729), one field per keyword. */
typedef struct nmfk_params {
    double tol;             /* tol=1e-19 (as reached from execute, NMFkExecute.jl:729) */
    double tolOF;           /* tolOF=1e-3 */
    double eps_clamp;       /* eps() == eps(Float64) = 2.220446049250313e-16, NMFkMultiplicative.jl:99-100 */
    double weight;          /* scalar weight=1; vector / matrix weights are set on the ctx with nmfk_set_weight and multiply this */
    int32_t maxiter;        /* maxiter=10000 from execute (NMFkExecute.jl:729); 1000000 when called directly */
    int32_t maxbaditers;    /* 10 */
    int32_t maxreattempts;  /* 2 */
    int32_t stopconv;       /* 1000 */
    int32_t check_every;    /* 10, the mod(iters, 10) of :73 */
    int32_t Wfixed;         /* Wfixed=false */
    int32_t Hfixed;         /* Hfixed=false */
    int32_t normalize;      /* execute_singlerun_compute's modifymatrices && mixture==:null: 1 = rows of H sum to one
                               (NMFkExecute.jl:800-804); 2 = its own clusterWmatrix=true branch (:796-799), reached only by a
                               direct call: execute_run never forwards clusterWmatrix to the restarts (:516-540); 0 = raw W,H */
    int32_t iter_limit;     /* >0: pause every restart once iters reaches this value (resumable); 0 = none */
    int32_t engine;         /* nmfk_engine */
    int32_t clusterWmatrix; /* execute_run's own keyword (NMFkExecute.jl:483, 620-637): cluster the columns of W instead of the
                               rows of H.  Used by nmfk_execute_run / nmfk_execute only; independent of `normalize` */
    int32_t stop_rule;      /* 0 = NMFmultiplicative(::AbstractMatrix) (NMFkMultiplicative.jl:64-118);
                               1 = NMFmultiplicative(::DArray) (:129-197): no tolOF/baditers/reattempts logic, no weight,
                                   no NaN imputation; stops on objvalue < tol, inc > stopconv (default 10000) or maxiter */
    int32_t variant;        /* nmfk_variant: 0 = KL (method=:simple), 1 = FRO (method=:nmf, algorithm=:multdiv),
                               2 = SPARSITY (method=:sparsity), 3 = KL_DIV (method=:nmf, algorithm=:multmse) */
    int32_t reserved[1];
} nmfk_params;

/* Which multiplicative update the solve runs.
 * NMFK_VARIANT_KL  : NMFmultiplicative (NMFkMultiplicative.jl:67,70) - the reference's method=:simple, the default.
 * NMFK_VARIANT_FRO : H <- H .* (W'X) ./ (W'W*H + d), W <- W .* (X*H') ./ (W*H*H' + d), d = sqrt(eps(T)): the update
 *   execute_singlerun_compute reaches with method=:nmf, algorithm=:multdiv (NMFkExecute.jl:763-766:
 *   NMF.MultUpdate(obj=:mse), third-party NMF.jl, restated in oracle/nmfk_oracle.py).  All R restarts of a batch are
 *   STACKED: W'X is one (R*k x n)(n x m) GEMM and X*H' one (n x m)(m x R*k) GEMM on the tensor cores (tcgen05 kind::tf32
 *   with the 3-term split for Float32, DMMA for Float64).  Stops when every column of W and row of H moved by less than
 *   `tol` relative (NMF.jl stop_condition) or at maxiter.
 * NMFK_VARIANT_SPARSITY : NMFsparsity (NMFkSparsity.jl:1-113; method=:sparsity, NMFkExecute.jl:757-758): beta-divergence updates
 *   with an L1 penalty on H and unit-norm columns of W; its own options come from nmfk_set_sparsity_options.
 * NMFK_VARIANT_KL_DIV : Q = X ./ (W*H .+ d), H .*= (W'Q) ./ (colsum(W)' .+ d), then the same with the new H for
 *   W .*= (Q*H') ./ (rowsum(H)' .+ d), d = sqrt(eps(T)): the update execute_singlerun_compute reaches with method=:nmf,
 *   algorithm=:multmse (NMFkExecute.jl:765-768: NMF.MultUpdate(obj=:div), third-party NMF.jl, restated in
 *   tests/test_oracle_multmse_cpu.py).  The KL update of method=:simple with d added, on the tiled engine's passes for every size and
 *   engine choice (tcgen05 for Float32, DMMA for Float64 with k >= 4, scalar FMA otherwise; k <= 64); no lambda imputation,
 *   clamp or objective checks.  Stops when every column of W and row of H moved by less than `tol` relative (NMF.jl
 *   stop_condition, checked after every iteration) or at maxiter.  Not available with NaN in X, a row-sharded ctx,
 *   normalizevector, array weights, stop_rule 1 or the resident engines. */
enum nmfk_variant { NMFK_VARIANT_KL = 0, NMFK_VARIANT_FRO = 1, NMFK_VARIANT_SPARSITY = 2, NMFK_VARIANT_KL_DIV = 3 };

/* Solution filtering of execute_run (NMFkExecute.jl:551-596): which of the R sorted restarts reach clustersolutions /
 * finalize.  Defaults acceptratio=1, acceptfactor=Inf, nanaction=:zeroed keep all of them. */
enum nmfk_nanaction { NMFK_NAN_ZEROED = 0, NMFK_NAN_REMOVED = 1 };

/* facts about X found by the preprocessing kernel (NMFpreprocessing!, NMFkMultiplicative.jl:3-22) */
typedef struct nmfk_xinfo {
    int64_t n, m;
    int64_t nnan;        /* count(isnan, X) */
    int64_t nzero;       /* count(X .<= 0) */
    int32_t zero_row;    /* some row sums to 0 -> the reference warns (:9-11) */
    int32_t zero_col;    /* some column sums to 0 (:12-14) */
    double xmin;         /* minimum(X) over non-NaN entries */
    int32_t dtype;
    int32_t reserved;
} nmfk_xinfo;

typedef struct nmfk_ctx nmfk_ctx;     /* one device, one X */
typedef struct nmfk_batch nmfk_batch; /* R restarts at one k: device-resident W/H stacks + per-restart state */

int32_t nmfk_abi_version(void);
const char* nmfk_last_error(const nmfk_ctx* ctx);
void nmfk_default_params(nmfk_params* p); /* the defaults reached from NMFk.execute(...; method=:simple) */

/* ---- context ---------------------------------------------------------------------------- */
int32_t nmfk_ctx_create(int32_t device, nmfk_ctx** out);
int32_t nmfk_ctx_destroy(nmfk_ctx* ctx);
int32_t nmfk_ctx_sync(nmfk_ctx* ctx); /* cudaStreamSynchronize on every stream of the ctx */

/* ---- X: replaces NMFpreprocessing! (NMFkMultiplicative.jl:3-22) ---------------------------
 * Uploads X (host pointer, or device pointer when on_device != 0), validates it (negative ->
 * NMFK_E_NEGATIVE unless X also holds NaN, exactly like `minimum(X) < 0`), builds the device
 * copies the solver streams (X with zeros -> lambda, and its transpose), and leaves the caller's
 * X untouched - the reference mutates and then restores it (:123-124).
 * normalizevector (length n, may be NULL) is the keyword of the same name (:27-31). */
int32_t nmfk_set_X(nmfk_ctx* ctx, const void* X, int64_t n, int64_t m, int32_t dtype, double lambda,
                   const void* normalizevector, int32_t on_device);
int32_t nmfk_get_xinfo(const nmfk_ctx* ctx, nmfk_xinfo* out);
/* Options of NMFsparsity (NMFkSparsity.jl:1): beta_divergence (2 = cost_function :ed, the default; 1 = :kl; 0 = :is; any other
 * value = fractional beta), sparsity (L1 weight on H, default 1) and its lambda (floor of X_est and of the denominators, default
 * 1e-9).  Used by nmfk_solve / nmfk_execute_run / nmfk_execute when params.variant == NMFK_VARIANT_SPARSITY. */
int32_t nmfk_set_sparsity_options(nmfk_ctx* ctx, double beta_divergence, double sparsity, double lambda);
/* The `weight` keyword when it is not a scalar (execute_run's assertion NMFkExecute.jl:484; used in the objective
 * sum((((X - W*H) .* weight)[.!inan]).^2) of NMFkMultiplicative.jl:74,125).  rows x cols must be (n,1): one weight per
 * row (a Julia Vector of length n), (1,m): one per column, or (n,m): one per entry; column-major, dtype of X, host
 * memory.  The effective weight is params.weight times this array.  w == NULL clears it.  Call after nmfk_set_X. */
int32_t nmfk_set_weight(nmfk_ctx* ctx, const void* w, int64_t rows, int64_t cols);

/* ---- batches of restarts: replace the restart loop of execute_run (NMFkExecute.jl:510-544) - */
int32_t nmfk_batch_create(nmfk_ctx* ctx, int32_t k, int32_t R, nmfk_batch** out);
int32_t nmfk_batch_destroy(nmfk_batch* b);
/* Winit: n x k x R, Hinit: k x m x R (dtype of X).  NaN -> NMFK_E_NAN_INIT.  Resets the state. */
int32_t nmfk_batch_set_init(nmfk_batch* b, const void* Winit, const void* Hinit);
/* U(0,1) initialisation generated on the device: restart r (0-based) uses the stream
 * numpy.random.Generator(Philox(key=seed0 + r + 1)).random(), W (column-major) then H - the draw
 * order of NMFkMultiplicative.jl:38,48 and the `seed=kwseed+i` of NMFkExecute.jl:536. */
int32_t nmfk_batch_init_random(nmfk_batch* b, uint64_t seed0);
/* Winit and Hinit independently, as the reference treats them (NMFkMultiplicative.jl:37-55): a NULL factor is drawn on the
 * device from restart r's Philox stream (key seed0 + r + 1) - after Random.seed!(seed) the reference draws W = rand(n,k)
 * only if Winit is empty and then H = rand(k,m) only if Hinit is empty, so a lone missing factor takes the FIRST numbers of
 * the stream.  This is the caller pattern of NMFkProgressive.jl:19,47,72,96 (Hinit + Hfixed) and NMFkMapping.jl:54
 * (Winit + Wfixed).  Both NULL == nmfk_batch_init_random; both given == nmfk_batch_set_init. */
int32_t nmfk_batch_set_init_partial(nmfk_batch* b, const void* Winit, const void* Hinit, uint64_t seed0);
/* Run NMFmultiplicative (+ the post-run objective and normalisation of execute_singlerun_compute,
 * NMFkExecute.jl:791-804) for every restart of every batch; batches run concurrently. */
int32_t nmfk_solve(nmfk_ctx* ctx, nmfk_batch* const* batches, int32_t nbatches, const nmfk_params* p);
/* Copy results to the host; any pointer may be NULL.  obj_ssq: NMFkMultiplicative.jl:125;
 * obj_norm: NMFkExecute.jl:792. */
int32_t nmfk_batch_get(nmfk_batch* b, void* W_out, void* H_out, double* obj_ssq, double* obj_norm,
                       int32_t* iters, int32_t* stop_reason);
/* Sum of squares sum(((X - W*H)*weight)[!inan]^2) of the current (unnormalised) W,H against the
 * lambda-substituted X, i.e. the quantity of NMFkMultiplicative.jl:74, for every restart. */
int32_t nmfk_batch_objective(nmfk_batch* b, double weight, double* obj_ssq);

/* ---- building blocks of the restart-sharded sweep (nmfk_sweep below composes them over the library's own NCCL
 * communicator; they stay exported for hosts that bring their own transport) ------------------------------------------- */
int32_t nmfk_batch_create_hstack(nmfk_ctx* ctx, int32_t k, int32_t R, nmfk_batch** out); /* no W stack */
/* device pointers of the factor stacks (W may come back NULL for an H-only batch) */
int32_t nmfk_batch_device_ptrs(nmfk_batch* b, void** W, void** H);
/* load finished solutions: H (k x m x R) and optionally W from host or device memory, plus the
 * objective (NMFkExecute.jl:792) and iteration count of every restart; marks them done */
int32_t nmfk_batch_import(nmfk_batch* b, const void* W, const void* H, const double* obj_norm,
                          const int32_t* iters, int32_t on_device);
/* phi = normnan(X - W*H) with NaN residuals dropped (NMFkExecute.jl:664-668) for host factors */
int32_t nmfk_fit(nmfk_ctx* ctx, int32_t k, const void* W, const void* H, double* phi);

/* ---- row-sharded X (BASELINE config C5; NMFmultiplicative(::DArray), NMFkMultiplicative.jl:129-197) ------
 * One process per GPU.  After nmfk_ctx_comm_init the ctx holds a BLOCK OF ROWS: nmfk_set_X receives the
 * local rows [row0, row0 + n_local) of the n_global x m matrix, W stacks are n_local x k x R, H stacks are
 * replicated (k x m x R, identical on every rank).  nmfk_solve then runs the tiled engine and, per
 * iteration, sum-all-reduces (NCCL, on the ctx stream) the stacked R x (k x m) numerators W'(X./(WH)) together
 * with the R x k column sums of W - the exchange the reference does with collect/distribute at :160-167 -
 * and, at every check, the 2R objective sums.  The W-update needs no exchange.  Objectives, iteration
 * counts and stop reasons are identical on all ranks; nmfk_batch_get returns the local rows of W.
 * nmfk_batch_init_random draws the streams of the GLOBAL matrices and keeps this rank's rows.
 * id128: 128-byte NCCL unique id made by nmfk_comm_unique_id on one rank and sent to the others by the
 * caller (any side channel).  nranks == 1 with id128 == NULL runs the same code path without NCCL. */
int32_t nmfk_comm_unique_id(void* id128);
int32_t nmfk_ctx_comm_init(nmfk_ctx* ctx, int32_t nranks, int32_t rank, const void* id128, int64_t row0, int64_t n_global);
int32_t nmfk_ctx_comm_destroy(nmfk_ctx* ctx);

/* ---- robustness: replaces sortperm + clustersolutions + finalize (NMFkExecute.jl:545-638,
 *      NMFkCluster.jl:425-517, NMFkFinalize.jl:36-79) on the device-resident H stack ----------
 * order        R      0-based restart indices sorted by objective (stable), order[0] = best
 * labels       k x R  1-based cluster of row a of the t-th sorted solution (column-major)
 * sil          k x R  silhouette of every row (NaN -> 0)
 * clustersil   k      mean silhouette per cluster; *robustness = min (1 when k == 1)
 * centroids    k x m  (k x (m+1) when the zero-column fix of NMFkCluster.jl:437-450 fired;
 *                      *centroid_cols tells which)                                              */
int32_t nmfk_batch_cluster(nmfk_batch* b, int32_t clusterWmatrix, int32_t* order, int32_t* labels, double* sil,
                           double* clustersil, double* robustness, void* centroids, int32_t* centroid_cols);
/* Solution filtering of execute_run before clustering (NMFkExecute.jl:551-596): acceptratio < 1 keeps the first
 * ceil(R * acceptratio) sorted solutions, acceptfactor < Inf keeps those with objvalue < acceptfactor * best, nanaction
 * NMFK_NAN_REMOVED drops solutions that hold NaN instead of zeroing them.  Like the reference, the three masks are ANDed
 * position by position although idxnan is indexed by restart number and the other two by sorted position (:560-596).
 * The selection is stored in the batch: nmfk_batch_cluster / nmfk_batch_cluster_means then work on the *nkept kept
 * solutions (their `order` / `labels` / `sil` outputs have nkept columns).  order_kept (R entries, first *nkept valid).
 * Defaults (1, Inf, NMFK_NAN_ZEROED) select everything, which is also the state of a fresh batch. */
int32_t nmfk_batch_select(nmfk_batch* b, double acceptratio, double acceptfactor, int32_t nanaction, int32_t* order_kept,
                          int32_t* nkept);

/* Wmean, Hmean, Wvar, Hvar of finalize(Wa, Ha, idx) (NMFkFinalize.jl:68-74): per cluster, the mean and the corrected
 * variance over the nNMF trials of the column of W / row of H that clustersolutions assigned to it - what execute_run returns
 * with best=false (NMFkExecute.jl:655-658) and what the "-all" result file stores (:650-654).  order (R) and labels (k x R,
 * 1-based, column-major) are the outputs of nmfk_batch_cluster; W outputs are n x k, H outputs k x m (column-major, the
 * batch's dtype); any output may be NULL. */
int32_t nmfk_batch_cluster_means(nmfk_batch* b, const int32_t* order, const int32_t* labels, void* Wmean, void* Hmean,
                                 void* Wvar, void* Hvar);

/* ---- one-call forms --------------------------------------------------------------------- */

/* NMFmultiplicative for R stacked restarts at one k, host buffers in and out
 * (NMFkMultiplicative.jl:24-127 + NMFkExecute.jl:791-804 when p->normalize != 0). */
int32_t nmfk_run_batch(nmfk_ctx* ctx, int32_t k, int32_t R, const void* Winit, const void* Hinit,
                       const nmfk_params* p, void* W_out, void* H_out, double* obj_ssq, double* obj_norm,
                       int32_t* iters, int32_t* stop_reason);
/* Fixed iteration count with per-iteration dumps, for parity: W_t is n x k x niter, H_t is
 * k x m x niter, obj_t[niter] is the :74 objective after every iteration (state machine, checks
 * and clamps run exactly as in a normal solve). */
int32_t nmfk_trace(nmfk_ctx* ctx, int32_t k, const void* Winit, const void* Hinit, const nmfk_params* p,
                   int32_t niter, void* W_t, void* H_t, double* obj_t);
/* execute_run(X, nk, nNMF) with defaults acceptratio=1, acceptfactor=Inf, nanaction=:zeroed,
 * best=true (NMFkExecute.jl:483-711): returns the best restart (n x k, k x m), phi = norm of the
 * residual (:664-668), robustness = min cluster silhouette (:638), aic (:708).
 * Winit/Hinit may be NULL -> device Philox streams seeded seed0 + i. */
int32_t nmfk_execute_run(nmfk_ctx* ctx, int32_t k, int32_t R, const void* Winit, const void* Hinit, uint64_t seed0,
                         const nmfk_params* p, void* W_best, void* H_best, double* phi, double* robustness,
                         double* aic, int64_t* total_iters);
/* execute(X, nkrange, nNMF; cutoff) (NMFkExecute.jl:178-233) without the JLD cache: all k of the
 * range are solved concurrently.  W_out[i] / H_out[i] (may be NULL) receive the signal-ordered
 * factors of ks[i] (signalorder, NMFkPostprocess.jl:148-158).  *kopt: k, 0 ("no successful
 * runs"), or -1 (`nothing`).  Winit[i]/Hinit[i] are per-k stacks or NULL (device Philox). */
int32_t nmfk_execute(nmfk_ctx* ctx, const int32_t* ks, int32_t nks, int32_t R, const void* const* Winit,
                     const void* const* Hinit, uint64_t seed0, const nmfk_params* p, double cutoff,
                     void* const* W_out, void* const* H_out, double* fitquality, double* robustness, double* aic,
                     int32_t* kopt, int64_t* total_iters);

/* ---- restart-sharded sweep over the GPUs of one box (the reference's `pmap` over restarts, NMFkExecute.jl:511-526) -----
 * One process per GPU, each with its own ctx that holds the whole X (nmfk_set_X on every rank).
 * nmfk_ctx_sweep_comm_init creates the library's own NCCL communicator (id128 from nmfk_comm_unique_id on one rank, sent
 * to the others by the caller - e.g. Julia's remotecall); nranks == 1 needs no id and makes nmfk_sweep == nmfk_execute.
 * nmfk_sweep = execute(X, ks, nNMF = nranks * R_local): rank q solves restarts q*R_local+1 .. (q+1)*R_local of every k
 * (device Philox keys seed0 + global restart number, or this rank's slices Winit[i] / Hinit[i] of R_local matrices); there
 * is no collective inside the iteration loop.  Per k, one all-gather of the H stacks and of the restart states and one
 * broadcast of the best restart's W cross NVLink; the clustering + silhouettes of the nranks*R_local solutions of the i-th
 * k run on rank i mod nranks.  EVERY rank must make the same call and EVERY rank receives all outputs (as nmfk_execute);
 * *total_iters is the global count, *total_iters_local this rank's share.  clusterWmatrix is not available across ranks. */
int32_t nmfk_ctx_sweep_comm_init(nmfk_ctx* ctx, int32_t nranks, int32_t rank, const void* id128);
int32_t nmfk_sweep(nmfk_ctx* ctx, const int32_t* ks, int32_t nks, int32_t R_local, const void* const* Winit,
                   const void* const* Hinit, uint64_t seed0, const nmfk_params* p, double cutoff, void* const* W_out,
                   void* const* H_out, double* fitquality, double* robustness, double* aic, int32_t* kopt, int64_t* total_iters,
                   int64_t* total_iters_local);

/* ---- robustkmeans(X, k, repeats; maxiter=1000, tol=1e-32, distance=CosineDist(), compute_silhouettes_flag)
 *      (NMFkCluster.jl:172-246; the k-means + silhouette step postprocess runs on W[kopt], H[kopt]) ------------------------------
 * X: d x N column-major Float64, the POINTS ARE THE COLUMNS (Clustering.kmeans convention).  `repeats` runs of Lloyd k-means with
 * cosine distance execute concurrently on the device (Clustering.jl `kmeans` restated; see csrc/kmeans.cu); the first run with
 * the smallest total cost is kept (:219-225), its silhouettes are Clustering.silhouettes on pairwise(CosineDist(),
 * zerostoepsilon(X)) (:195-218), and the result is relabelled by sortclustering (:264-289: clusters ranked by size).
 * seeds: k x repeats 0-based point indices - the k-means++ seeding draws from Julia's RNG in the reference and is the caller's
 * job here (the host mirrors implement it).  Outputs (any may be NULL): assignments N (1-based, sorted labels), centers d x k,
 * costs N, counts k, totalcost, iterations, converged of the best run; best_silhouettes N; *best_repeat (0-based);
 * *empty_cluster_repeats = runs in which a cluster lost all its points (the package re-draws such a centre at random; here it
 * keeps its position). */
int32_t nmfk_robustkmeans(nmfk_ctx* ctx, const double* X, int32_t d, int32_t N, int32_t k, int32_t repeats, const int32_t* seeds,
                          int32_t maxiter, double tol, int32_t compute_silhouettes, int32_t* assignments, double* centers, double* costs,
                          int32_t* counts, double* totalcost, int32_t* iterations, int32_t* converged, double* best_silhouettes,
                          int32_t* best_repeat, int32_t* empty_cluster_repeats);

/* getk (NMFkPostprocess.jl:7-41): returns k, 0 (all NaN) or -1 (nothing). */
int32_t nmfk_getk(const int32_t* ks, const double* robustness, int32_t nks, double cutoff, int32_t strict);
/* signalorder (NMFkPostprocess.jl:148-158) on host buffers; order is 0-based. */
int32_t nmfk_signalorder(const void* W, const void* H, int64_t n, int32_t k, int64_t m, int32_t dtype,
                         int32_t* order);

/* ---- measurement helpers (bench only) --------------------------------------------------- */
/* kernel launches issued by this ctx since creation (for bench.py's gpu_launches) */
int64_t nmfk_launch_count(const nmfk_ctx* ctx);
/* Per-launch device time of the dominant kernels of the tiled engine (the two half-update pass kernels: tc_pass_kernel for
 * Float32, tiled_dmma_pass_kernel / tiled_pass_kernel for Float64), measured with CUDA events on the launching stream while
 * nmfk_solve runs: enable (resets the counters), solve, then read the summed duration and the number of launches. */
int32_t nmfk_profile_enable(nmfk_ctx* ctx, int32_t on);
int32_t nmfk_profile_get(const nmfk_ctx* ctx, double* pass_ms, int64_t* pass_launches);
/* device time (ms, CUDA events on the ctx streams) of the last nmfk_solve */
double nmfk_last_solve_ms(const nmfk_ctx* ctx);
/* micro-benchmarks that give the roofline denominators MEASURED_PEAKS.json does not hold:
 * which: 0 = FP64 DFMA TFLOP/s, 1 = FP64 DMMA (mma.sync m8n8k4) TFLOP/s, 2 = FP32 FFMA TFLOP/s,
 *        3 = device-to-device copy GB/s (read+write bytes), 13 = dense tcgen05.mma kind::tf32 TFLOP/s (M = 128, N = 256,
 *        K = 8 from shared memory on every SM; the 3-term split of the Float32 kernels runs at a third of it) */
int32_t nmfk_measure_peak(nmfk_ctx* ctx, int32_t which, double* value);
/* The stacked-restart GEMM of Variant FRO on its own (test / measurement hook; no reference counterpart beyond BLAS gemm):
 * C[M x N] = A[M x K] * B[N x K]^T, all row-major host buffers.  Float32: tcgen05.mma kind::tf32 with the 3-term split, operands
 * staged by TMA tensor maps (N and K multiples of 4); Float64: DMMA.  *ms: average device time of `reps` launches. */
int32_t nmfk_gemm_nt(nmfk_ctx* ctx, int32_t dtype, const void* A, const void* B, int32_t M, int32_t N, int32_t K, void* C,
                     int32_t reps, double* ms);
/* Device self-test of the tcgen05 / tensor-memory building blocks of the Float32 tiled engine (no reference
 * counterpart): U 128x16, V 64x16 row-major; mode bits: 1 P=UV' (A,B shared), 2 P (A tensor memory),
 * 4 / 8 ACC = 0.5 P V with the 2-term TF32 split of the A operand (B K-major copy / B MN-major alias). */
/* cycle counts of the same building blocks (tools/umma_selftest.py --timing documents the 8 slots) and the
 * accumulator of reps*8 chained K-steps (round-toward-zero accumulation test) */
int32_t nmfk_umma_timing(nmfk_ctx* ctx, const float* U, const float* V, int32_t reps, int64_t* cycles8, float* acc);
int32_t nmfk_umma_selftest(nmfk_ctx* ctx, const float* U, const float* V, int32_t mode, float* Pss, float* Pts, float* ACCa,
                           float* ACCb, int32_t* err);

/* first `count` doubles of numpy.random.Generator(Philox(key=seed)).random(), computed on the HOST with the
 * same code the device initialiser uses (test hook: bit-compatibility of the init streams without a GPU) */
int32_t nmfk_philox_host(uint64_t seed, int64_t count, double* out);

#ifdef __cplusplus
}
#endif
#endif /* NMFK_B200_H */
