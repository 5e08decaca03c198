// Internal (host+device) declarations shared by the kernels and the C ABI layer.
// Nothing here is exported; the public surface is include/nmfk_b200.h.
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include <cuda_runtime.h>

namespace nmfk {

// Per-restart solver state, device resident, so that a solve can be paused and resumed
// (trace mode, host-driven tiled engine).  Scalars of NMFkMultiplicative.jl:56-63.
struct UnitState {
    int32_t it;        // iters
    int32_t bad;       // baditers
    int32_t re;        // reattempts
    int32_t inc;       // consecutive unchanged co-clusterings
    int32_t stop;      // nmfk_stop_reason, 0 while running / paused
    int32_t has_cons;  // consold holds a real partition (it starts as falses(m,m))
    int32_t done;      // post-run objective + normalisation applied
    int32_t pad;
    double best;       // objvalue_best
    double obj_chk;    // objective of the last check (NMFkMultiplicative.jl:74)
    double obj_ssq;    // final sum of squares (:125)
    double obj_norm;   // normnan(X - W*H) (NMFkExecute.jl:792)
};

// Row-sharded X (BASELINE config C5; reference analogue NMFmultiplicative(::DArray),
// NMFkMultiplicative.jl:129-197): this rank holds a block of rows of X and of W, H is replicated.
// sum-all-reduce of `count` elements (dtype 0 = f32, 1 = f64) in place, stream ordered.
struct ShardComm {
    void* comm;  // ncclComm_t
    int nranks, rank;
    cudaError_t (*allreduce)(void* comm, void* buf, size_t count, int dtype, cudaStream_t s);
};

// Non-scalar `weight` keyword (NMFkExecute.jl:484, NMFkMultiplicative.jl:74,125): the residual of entry (i,j) is
// multiplied by scalar * wrow[i] * wcol[j] * wmat[i + j*n]; a null array counts as 1.  Element type of X.
struct WeightRef {
    const void* wrow;
    const void* wcol;
    const void* wmat;
    __host__ __device__ bool any() const { return wrow != nullptr || wcol != nullptr || wmat != nullptr; }
};
template <typename T>
__device__ __forceinline__ double weight_at(const WeightRef& w, double scalar, long long i, long long j, long long n) {
    double v = scalar;
    if (w.wrow != nullptr) v *= (double)static_cast<const T*>(w.wrow)[i];
    if (w.wcol != nullptr) v *= (double)static_cast<const T*>(w.wcol)[j];
    if (w.wmat != nullptr) v *= (double)static_cast<const T*>(w.wmat)[i + j * n];
    return v;
}

// Device time of the dominant kernels of the tiled engine (the two half-update passes), measured with CUDA events on the
// launching stream while a solve runs (bench.py's roofline.achieved): begin/end bracket one launch, harvest() is called after
// a stream synchronisation.
struct PassProfile {
    bool enabled = false;
    double ms = 0.0;
    long long launches = 0;
    std::vector<cudaEvent_t> idle, pending;  // pending holds (start, stop) pairs
    cudaEvent_t get() {
        if (!idle.empty()) {
            cudaEvent_t e = idle.back();
            idle.pop_back();
            return e;
        }
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        return e;
    }
    void begin(cudaStream_t s) {
        if (!enabled) return;
        cudaEvent_t e = get();
        cudaEventRecord(e, s);
        pending.push_back(e);
    }
    void end(cudaStream_t s) { begin(s); }
    void harvest() {
        for (size_t i = 0; i + 1 < pending.size(); i += 2) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, pending[i], pending[i + 1]) == cudaSuccess) {
                ms += t;
                ++launches;
            }
            idle.push_back(pending[i]);
            idle.push_back(pending[i + 1]);
        }
        pending.clear();
    }
    void reset() {
        ms = 0.0;
        launches = 0;
    }
    void destroy() {
        for (auto e : idle) cudaEventDestroy(e);
        for (auto e : pending) cudaEventDestroy(e);
        idle.clear();
        pending.clear();
    }
};

// A bounded barrier wait of a tcgen05 kernel (tc_ptx.cuh) that timed out during a solve.  The wait writes its site to an
// error flag in mapped pinned host memory, which stays readable after the kernel traps.  The solver then stops, fills this
// in and fails; the entry point turns it into an error message naming the kernel and the site.
struct KernelTimeout {
    const char* kernel = nullptr;  // nullptr: no time-out
    const char* where = nullptr;   // which launch of the solve
    int site = 0;                  // the `where` code of the wait that timed out
};

// Arguments of one batched KL solve (R restarts at one k).
struct SolveArgs {
    const void* X;    // n x m column-major, zeros -> lambda, NaN kept
    const void* Xt;   // m x n column-major (the transpose), same substitutions
    void* W;          // n x k x R
    void* H;          // k x m x R
    UnitState* st;    // R
    int32_t* canon;   // R x m : canonical co-clustering of the previous check
    void* ximp;       // R x n x m imputed values (only when has_nan), X layout
    int32_t n, m, k, R;
    int32_t has_nan;
    int32_t SH, SW;   // DMMA resident engine: slices of the reduction range per half-update (host heuristic)
    int32_t maxiter, maxbad, maxre, stopconv, check_every, Wfixed, Hfixed, normalize, iter_limit;
    double lambda, tol, tolOF, eps_clamp, weight;
    WeightRef wref;          // non-scalar weight (tiled engine with the scalar objective kernel only)
    int32_t tiled_tc;        // tiled engine, Float32 without NaN: 1 = tcgen05 kernel (kl_tiled_tc.cu), 0 = scalar-FMA kernel
    const ShardComm* shard;  // non-null: n is the LOCAL row count, the tiled engine all-reduces the k x m partials
    PassProfile* prof;       // non-null: time the pass-kernel launches of the tiled engine
    KernelTimeout* timeout;  // non-null: where the tiled / FRO solver reports a barrier time-out
};

// records a barrier time-out reported through a kernel's error flag; the solver returns the value of this call (the CUDA
// error of the trap that follows the time-out, when the solver has already met it)
inline cudaError_t solve_timeout(const SolveArgs& a, cudaError_t err, const char* kernel, const char* where, int site) {
    if (a.timeout != nullptr) *a.timeout = KernelTimeout{kernel, where, site};
    return err != cudaSuccess ? err : cudaErrorLaunchTimeout;
}

// threads per restart-CTA of the resident engine: 512 (<=128 registers) while u/acc fit, 256 beyond
__host__ __device__ constexpr int resident_threads(int Ktemplate) { return Ktemplate <= 12 ? 512 : 256; }
// largest k of the resident engines (factors in shared memory) and of the tiled engine (factors streamed)
constexpr int kResidentMaxK = 32;
constexpr int kTiledMaxK = 64;

// delta of Variant KL_DIV (NMF.jl's MultUpdate(obj=:div)): Q = X ./ (W*H .+ delta), U .*= (numerators) ./ (sums .+ delta) with
// delta = sqrt(eps(T)), the same (unpinned) reading of NMF.jl as Variant FRO's.  The only place the device takes it from.
template <typename T>
constexpr T kKlDivDelta = T(0);
template <>
constexpr float kKlDivDelta<float> = 3.4526698e-4f;  // sqrt(eps(Float32)) = 2^-11.5, rounded to Float32
template <>
constexpr double kKlDivDelta<double> = 1.4901161193847656e-8;  // sqrt(eps(Float64)) = 2^-26

// template K actually instantiated for a requested k (exact up to 12, then padded)
inline int resident_template_k(int k) {
    if (k <= 12) return k;
    if (k <= 16) return 16;
    if (k <= 20) return 20;
    if (k <= 24) return 24;
    if (k <= 32) return 32;
    return -1;
}
// the same for the tiled engine: identical up to 32, then padded to a multiple of 8
inline int tiled_template_k(int k) {
    if (k <= kResidentMaxK) return resident_template_k(k);
    if (k <= kTiledMaxK) return (k + 7) / 8 * 8;
    return -1;
}

// dynamic shared memory the resident kernel needs (bytes); mirrors the carve-up in kl_resident.cuh
size_t resident_smem_bytes(int n, int m, int Ktemplate, size_t sizeofTC);

// launchers (one translation unit per dtype), return cudaError_t
cudaError_t launch_kl_resident_f64(const SolveArgs& a, cudaStream_t s);
cudaError_t launch_kl_resident_f32(const SolveArgs& a, cudaStream_t s);
// Float64 tensor-pipe (DMMA) formulation of the resident engine (kl_dmma.cuh)
cudaError_t launch_kl_resident_dmma(const SolveArgs& a, cudaStream_t s);
bool resident_dmma_fits(int n, int m, int k);
// can the resident engine take this shape?  (smem budget of one CTA)
bool resident_fits(int n, int m, int k, size_t sizeofTC);

// generic residual sums of one (W,H): partials[2*b] = weighted ssq, partials[2*b+1] = plain ssq of CTA b
int residual_blocks(int n, int m);
cudaError_t launch_residual(const void* X, int dtype, int n, int m, int k, const void* W, const void* H, double lambda,
                            int restore, double weight, const WeightRef& wref, double* d_partials, cudaStream_t s);

// preprocessing (K1): raw X -> Xp, Xpt + statistics
struct PreStats {
    unsigned long long nnan, nzero, nneg;
    unsigned long long zero_rows, zero_cols;
};
cudaError_t launch_preprocess(const void* Xraw, void* Xp, void* Xpt, int64_t n, int64_t m, int dtype, double lambda,
                              PreStats* d_stats, unsigned char* d_rowflag, unsigned char* d_colflag, double* d_blockmin,
                              int nblockmin, cudaStream_t s);

// device Philox4x64-10 U(0,1) streams identical to numpy.random.Generator(Philox(key=seed)).random()
// (row-sharded X: n = global rows, this rank keeps rows [row0, row0 + nloc); otherwise row0 = 0, nloc = n)
cudaError_t launch_philox_init(void* W, void* H, int64_t n, int64_t row0, int64_t nloc, int k, int64_t m, int R,
                               uint64_t seed0, int dtype, cudaStream_t s);

// clustering / silhouettes (K10-K12)
struct ClusterArgs {
    const void* F;        // factor stack in solver layout (H: k x m x R; W: n x k x R)
    int32_t len;          // vector length (m for H rows, n for W columns)
    int32_t k, R;
    int32_t use_W;        // clusterWmatrix
    const int32_t* order; // R sorted restart indices (device)
    int32_t* labels;      // k x R (device), 1-based
    double* cent;         // k x (len+1) running-sum centroids (device scratch / output)
    double* sil;          // k x R
    double* clustersil;   // k
    int32_t* bias;        // out: 1 if the zero-column fix fired
    double* V;            // (R*k) x (len+1) gathered + floored vectors, row-major, sorted order
    double* vnorm;        // R*k
    double* Dm;           // (R*k) x (R*k) cosine distance matrix
    void* alias_best;     // clusterWmatrix: W of the best solution (n x k, factor type), overwritten with the centroids like
                          // the reference's aliased newClusterCenters (NMFkCluster.jl:453-455); nullptr otherwise
};
cudaError_t launch_cluster(const ClusterArgs& a, int dtype, cudaStream_t s);
int cluster_walk_launches(int k, int len, int R);
cudaError_t launch_zero_nan(void* p, long long len, int dtype, cudaStream_t s);
// per-cluster means / corrected variances over the trials (NMFkFinalize.jl:68-74); outputs are device buffers of the factor type
cudaError_t launch_cluster_means(const void* F, int len, int k, int R, int use_W, const int32_t* d_order, const int32_t* d_amap,
                                 void* mean_out, void* var_out, int dtype, cudaStream_t s);

cudaError_t launch_point_silhouettes(double* V, int len, int ld, int N, int k, const int* labels, double floorv, double* vnorm, double* Dm,
                                     double* sil, cudaStream_t s);
// robustkmeans: `repeats` Lloyd runs with cosine distance, one CTA each (kmeans.cu)
cudaError_t launch_kmeans(const double* X, double* xnorm, int d, int N, int k, int repeats, const int* seeds, int maxiter, double tol,
                          int* assign, double* costs, int* counts, double* centers, double* totalcost, int* iters, int* flags,
                          cudaStream_t s);

// micro-benchmarks
cudaError_t measure_peak(int which, double* value, cudaStream_t s);
// dense tcgen05.mma kind::tf32 throughput, TFLOP/s (tc_selftest.cu)
cudaError_t umma_peak(double* tflops, cudaStream_t s);
// tcgen05 building-block self-test (tc_selftest.cu)
cudaError_t umma_timing(const float* U, const float* V, int reps, long long* out8, float* bias, cudaStream_t s);
cudaError_t umma_selftest(const float* U, const float* V, int mode, float* Pss, float* Pts, float* ACCa, float* ACCb, int* err,
                          cudaStream_t s);

// Pinned host words for the device -> host flags of a solve, allocated once per host thread: cudaMallocHost / cudaFreeHost
// synchronise the device and take up to hundreds of milliseconds, which showed up as sporadic 0.3 - 0.6 s stalls inside timed
// solves.  Solves are synchronous (they return after their last stream synchronisation), so one buffer per thread is enough.
inline int* pinned_flags() {
    static thread_local int* p = nullptr;
    if (!p && cudaMallocHost(&p, 64) != cudaSuccess) p = nullptr;
    return p;
}
// Device buffers of the entry points (X images, factor stacks, temporaries): pooled like the scratch of the solves, but with
// the semantics of cudaMalloc / cudaFree - usable from any stream once dev_malloc returns (host-synchronised allocation), and
// freed only after everything on the device has finished.  cudaMalloc / cudaFree of the 0.4 GB X images and of the factor stacks
// cost 50 - 300 ms per nmfk_execute_run call (map / unmap in the driver); the pool keeps the blocks.
inline cudaError_t dev_malloc(void** p, size_t bytes) {
    cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 16, cudaStreamPerThread);
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamPerThread);
    return e;
}
template <typename T>
inline cudaError_t dev_malloc(T** p, size_t bytes) {
    return dev_malloc(reinterpret_cast<void**>(p), bytes);
}
inline void dev_free(void* p) {
    if (!p) return;
    cudaDeviceSynchronize();
    cudaFreeAsync(p, cudaStreamPerThread);
}
// Device scratch of a solve comes from the stream-ordered pool (release threshold raised when the context is created): no
// device-wide synchronisation and, in the steady state, no driver call at all.
inline cudaError_t scratch_alloc(void** p, size_t bytes, cudaStream_t s) { return cudaMallocAsync(p, bytes ? bytes : 16, s); }
template <typename T>
inline cudaError_t scratch_alloc(T** p, size_t bytes, cudaStream_t s) {
    return scratch_alloc(reinterpret_cast<void**>(p), bytes, s);
}
inline void scratch_free(void* p, cudaStream_t s) {
    if (p) cudaFreeAsync(p, s);
}

}  // namespace nmfk
