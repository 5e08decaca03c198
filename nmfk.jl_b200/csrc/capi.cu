// C ABI of the B200-native NMFk hot path (include/nmfk_b200.h): context, X upload, batches of
// restarts, solve, robustness, and the one-call forms that mirror the reference's
// execute_run / execute (/root/reference/src/NMFkExecute.jl:178-233, 483-711).
// Host-side logic only; every numeric step runs in the CUDA kernels of this directory.
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/nmfk_b200.h"
#include "fro.h"
#include "kl_tiled_args.h"
#include "nmfk_internal.h"
#include "philox.h"

using namespace nmfk;

// NCCL is bound at run time (dlopen, see ShardNccl): only the handful of types / prototypes used here are declared, with the
// values of nccl.h (2.x ABI), so the library builds on hosts without the NCCL headers.
extern "C" {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef enum { ncclSuccess = 0 } ncclResult_t;
typedef enum { ncclUint8 = 1, ncclInt32 = 2, ncclInt64 = 4, ncclFloat = 7, ncclDouble = 8 } ncclDataType_t;
typedef enum { ncclSum = 0 } ncclRedOp_t;
ncclResult_t ncclGetUniqueId(ncclUniqueId* uniqueId);
ncclResult_t ncclCommInitRank(ncclComm_t* comm, int nranks, ncclUniqueId commId, int rank);
ncclResult_t ncclCommDestroy(ncclComm_t comm);
const char* ncclGetErrorString(ncclResult_t result);
ncclResult_t ncclAllReduce(const void* sendbuff, void* recvbuff, size_t count, ncclDataType_t datatype, ncclRedOp_t op,
                           ncclComm_t comm, cudaStream_t stream);
ncclResult_t ncclAllGather(const void* sendbuff, void* recvbuff, size_t sendcount, ncclDataType_t datatype, ncclComm_t comm,
                           cudaStream_t stream);
ncclResult_t ncclBroadcast(const void* sendbuff, void* recvbuff, size_t count, ncclDataType_t datatype, int root,
                           ncclComm_t comm, cudaStream_t stream);
}

struct nmfk_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::vector<cudaStream_t> pool;
    std::vector<cudaEvent_t> pool_ev;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    void* Xp = nullptr;
    void* Xpt = nullptr;
    // nmfk_set_X keeps the two images and the H2D staging buffer when the next X has the same size (a sweep over data sets, the
    // end-to-end bench): three 0.4 GB allocations per call otherwise
    void* Xstage = nullptr;
    size_t Xbytes = 0;
    // normalizevector (NMFkMultiplicative.jl:27-31): the solver streams Xn = Xp ./ nv (and its transpose); Xp stays the
    // caller's matrix for the final objective (:119-125)
    void* Xn = nullptr;
    void* Xnt = nullptr;
    void* nv = nullptr;
    // non-scalar `weight` (nmfk_set_weight): per row, per column, or per entry; element type of X
    void* wrow = nullptr;
    void* wcol = nullptr;
    void* wmat = nullptr;
    // Variant FRO, Float32: lo images (x - tf32(x)) of Xp / Xpt for the 3-term split, built at the first FRO solve
    void* Xlo = nullptr;
    void* Xtlo = nullptr;
    // NMFsparsity options (nmfk_set_sparsity_options): beta_divergence, sparsity, lambda
    double sp_beta = 2.0, sp_sparsity = 1.0, sp_lambda = 1e-9;
    // persistent device scratch of the clustering phase (grown on demand, never shrunk)
    void* scratch = nullptr;
    size_t scratch_cap = 0;
    int64_t n = 0, m = 0;
    int dtype = NMFK_F64;
    double lambda = 1e-32;
    bool has_X = false;
    nmfk_xinfo info{};
    std::string err;
    int64_t launches = 0;
    double last_solve_ms = 0.0;
    double* d_partials = nullptr;  // residual partial sums
    size_t partials_cap = 0;
    // row-sharded X (nmfk_ctx_comm_init): this ctx holds rows [row0, row0 + n) of an n_global x m matrix
    ShardComm shard{nullptr, 1, 0, nullptr};
    bool sharded = false;
    int64_t row0 = 0, n_global = 0;
    // restart-sharded sweep (nmfk_ctx_sweep_comm_init): the library's own communicator over the ranks that share the restarts
    PassProfile prof;            // nmfk_profile_enable: device time of the tiled engine's pass kernels
    void* sweep_comm = nullptr;  // ncclComm_t
    int sweep_nranks = 1, sweep_rank = 0;
};

struct nmfk_batch {
    nmfk_ctx* ctx = nullptr;
    int k = 0, R = 0;
    void* W = nullptr;
    void* H = nullptr;
    UnitState* st = nullptr;
    int32_t* canon = nullptr;
    void* ximp = nullptr;
    bool inited = false;
    // nmfk_batch_select: sorted restart indices that reach clustersolutions / finalize (empty = all R)
    bool has_sel = false;
    std::vector<int32_t> sel;
    int32_t nanaction = NMFK_NAN_ZEROED;
};

static thread_local std::string g_err;
static int32_t residual(nmfk_ctx* c, int k, const void* W, const void* H, int restore, double weight, double out[2]);

static size_t esize(int dtype) { return dtype == NMFK_F64 ? 8 : 4; }

static int32_t fail(nmfk_ctx* c, int32_t code, const std::string& msg) {
    g_err = msg;
    if (c) c->err = msg;
    return code;
}

#define CU(ctx, call)                                                                                   \
    do {                                                                                                \
        cudaError_t e__ = (call);                                                                       \
        if (e__ != cudaSuccess)                                                                         \
            return fail((ctx), (int32_t)e__, std::string(#call) + ": " + cudaGetErrorString(e__));      \
    } while (0)

namespace {
// device allocation freed on scope exit (error paths of the entry points below must not leak GBs)
struct DevBuf {
    void* p = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() {
        if (p) dev_free(p);
    }
    cudaError_t alloc(size_t bytes) { return dev_malloc(&p, bytes ? bytes : 1); }
    void* release() {
        void* q = p;
        p = nullptr;
        return q;
    }
    template <typename T>
    T* as() const {
        return static_cast<T*>(p);
    }
};

void free_X(nmfk_ctx* c) {
    for (void** q : {&c->Xp, &c->Xpt, &c->Xn, &c->Xnt, &c->nv, &c->wrow, &c->wcol, &c->wmat, &c->Xlo, &c->Xtlo}) {
        if (*q) dev_free(*q);
        *q = nullptr;
    }
    c->has_X = false;
}

// persistent scratch of the ctx (clustering phase): at least `bytes`, contents undefined
cudaError_t ctx_scratch(nmfk_ctx* c, size_t bytes, void** out) {
    if (c->scratch_cap < bytes) {
        if (c->scratch) dev_free(c->scratch);
        c->scratch = nullptr;
        c->scratch_cap = 0;
        cudaError_t e = dev_malloc(&c->scratch, bytes);
        if (e != cudaSuccess) return e;
        c->scratch_cap = bytes;
    }
    *out = c->scratch;
    return cudaSuccess;
}
}  // namespace

namespace nmfk {
cudaError_t launch_rownormalize(const void* Xp, void* Xn, void* Xnt, int64_t n, int64_t m, const void* nv, int dtype,
                                cudaStream_t s);
cudaError_t launch_scale_rows(void* W, int64_t n, int k, const void* nv, int dtype, cudaStream_t s);
cudaError_t launch_renormalize(void* W, void* H, int64_t n, int64_t m, int k, int normalize, int dtype, cudaStream_t s);
cudaError_t launch_count_nan(const void* W, const void* H, int64_t wlen, int64_t hlen, int R, int dtype, int32_t* d_flags,
                             cudaStream_t s);
}  // namespace nmfk

// NCCL is bound with dlopen at the first nmfk_comm_* call: in a process that already loaded a
// libnccl.so.2 (torch ships its own) that copy is reused, otherwise the system library is loaded;
// libnmfk_b200.so itself has no link-time dependency on NCCL.
namespace {
struct ShardNccl {
    void* lib = nullptr;
    decltype(&ncclGetUniqueId) getUniqueId = nullptr;
    decltype(&ncclCommInitRank) commInitRank = nullptr;
    decltype(&ncclAllReduce) allReduce = nullptr;
    decltype(&ncclCommDestroy) commDestroy = nullptr;
    decltype(&ncclGetErrorString) getErrorString = nullptr;
    decltype(&ncclAllGather) allGather = nullptr;
    decltype(&ncclBroadcast) broadcast = nullptr;
    std::string err;
    bool load() {
        if (lib) return true;
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (lib) break;
        }
        if (!lib) {
            err = std::string("cannot load NCCL: ") + dlerror();
            return false;
        }
        getUniqueId = reinterpret_cast<decltype(getUniqueId)>(dlsym(lib, "ncclGetUniqueId"));
        commInitRank = reinterpret_cast<decltype(commInitRank)>(dlsym(lib, "ncclCommInitRank"));
        allReduce = reinterpret_cast<decltype(allReduce)>(dlsym(lib, "ncclAllReduce"));
        commDestroy = reinterpret_cast<decltype(commDestroy)>(dlsym(lib, "ncclCommDestroy"));
        getErrorString = reinterpret_cast<decltype(getErrorString)>(dlsym(lib, "ncclGetErrorString"));
        allGather = reinterpret_cast<decltype(allGather)>(dlsym(lib, "ncclAllGather"));
        broadcast = reinterpret_cast<decltype(broadcast)>(dlsym(lib, "ncclBroadcast"));
        if (!getUniqueId || !commInitRank || !allReduce || !commDestroy || !getErrorString || !allGather || !broadcast) {
            err = "NCCL library lacks a required symbol";
            lib = nullptr;
            return false;
        }
        return true;
    }
};
ShardNccl g_nccl;

cudaError_t nccl_allreduce(void* comm, void* buf, size_t count, int dtype, cudaStream_t s) {
    const ncclResult_t r = g_nccl.allReduce(buf, buf, count, dtype == 1 ? ncclDouble : ncclFloat, ncclSum,
                                            static_cast<ncclComm_t>(comm), s);
    return r == ncclSuccess ? cudaSuccess : cudaErrorUnknown;
}
// single-rank stand-in (nranks == 1): the sum over one rank is the buffer itself
cudaError_t identity_allreduce(void*, void*, size_t, int, cudaStream_t) { return cudaSuccess; }
}  // namespace

// Definitions below inherit C linkage from their declarations in include/nmfk_b200.h.

int32_t nmfk_comm_unique_id(void* id128) {
    if (!id128) return fail(nullptr, NMFK_E_INVALID, "nmfk_comm_unique_id: NULL buffer");
    if (!g_nccl.load()) return fail(nullptr, NMFK_E_UNSUPPORTED, g_nccl.err);
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    const ncclResult_t r = g_nccl.getUniqueId(&id);
    if (r != ncclSuccess) return fail(nullptr, NMFK_E_UNSUPPORTED, std::string("ncclGetUniqueId: ") + g_nccl.getErrorString(r));
    std::memcpy(id128, &id, 128);
    return NMFK_OK;
}

int32_t nmfk_ctx_comm_init(nmfk_ctx* c, int32_t nranks, int32_t rank, const void* id128, int64_t row0, int64_t n_global) {
    if (!c || nranks < 1 || rank < 0 || rank >= nranks || row0 < 0 || n_global < 1)
        return fail(c, NMFK_E_INVALID, "nmfk_ctx_comm_init: bad arguments");
    if (c->sharded) return fail(c, NMFK_E_INVALID, "nmfk_ctx_comm_init: ctx already has a communicator");
    CU(c, cudaSetDevice(c->device));
    if (nranks == 1 && !id128) {
        c->shard = ShardComm{nullptr, 1, 0, identity_allreduce};
    } else {
        if (!id128) return fail(c, NMFK_E_INVALID, "nmfk_ctx_comm_init: NULL unique id");
        if (!g_nccl.load()) return fail(c, NMFK_E_UNSUPPORTED, g_nccl.err);
        ncclUniqueId id;
        std::memcpy(&id, id128, 128);
        ncclComm_t comm = nullptr;
        const ncclResult_t r = g_nccl.commInitRank(&comm, nranks, id, rank);
        if (r != ncclSuccess)
            return fail(c, NMFK_E_UNSUPPORTED, std::string("ncclCommInitRank: ") + g_nccl.getErrorString(r));
        c->shard = ShardComm{comm, nranks, rank, nccl_allreduce};
        // NCCL connects its channels lazily at the first collective (hundreds of ms with 8 ranks): do it here, not inside
        // the first timed iteration of a solve
        DevBuf warm;
        CU(c, warm.alloc(256 * sizeof(float)));
        CU(c, cudaMemsetAsync(warm.p, 0, 256 * sizeof(float), c->stream));
        CU(c, nccl_allreduce(comm, warm.p, 256, 0, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    c->sharded = true;
    c->row0 = row0;
    c->n_global = n_global;
    return NMFK_OK;
}

int32_t nmfk_ctx_comm_destroy(nmfk_ctx* c) {
    if (!c) return fail(nullptr, NMFK_E_INVALID, "ctx is NULL");
    if (c->sharded && c->shard.comm) g_nccl.commDestroy(static_cast<ncclComm_t>(c->shard.comm));
    c->shard = ShardComm{nullptr, 1, 0, nullptr};
    c->sharded = false;
    if (c->sweep_comm) g_nccl.commDestroy(static_cast<ncclComm_t>(c->sweep_comm));
    c->sweep_comm = nullptr;
    c->sweep_nranks = 1;
    c->sweep_rank = 0;
    return NMFK_OK;
}

int32_t nmfk_ctx_sweep_comm_init(nmfk_ctx* c, int32_t nranks, int32_t rank, const void* id128) {
    if (!c || nranks < 1 || rank < 0 || rank >= nranks) return fail(c, NMFK_E_INVALID, "nmfk_ctx_sweep_comm_init: bad arguments");
    if (c->sweep_comm) return fail(c, NMFK_E_INVALID, "nmfk_ctx_sweep_comm_init: ctx already has a sweep communicator");
    CU(c, cudaSetDevice(c->device));
    if (nranks > 1) {
        if (!id128) return fail(c, NMFK_E_INVALID, "nmfk_ctx_sweep_comm_init: NULL unique id");
        if (!g_nccl.load()) return fail(c, NMFK_E_UNSUPPORTED, g_nccl.err);
        ncclUniqueId id;
        std::memcpy(&id, id128, 128);
        ncclComm_t comm = nullptr;
        const ncclResult_t r = g_nccl.commInitRank(&comm, nranks, id, rank);
        if (r != ncclSuccess) return fail(c, NMFK_E_UNSUPPORTED, std::string("ncclCommInitRank: ") + g_nccl.getErrorString(r));
        c->sweep_comm = comm;
        DevBuf warm;  // first collective = NCCL's lazy channel set-up: pay it here
        CU(c, warm.alloc(256 * sizeof(float)));
        CU(c, cudaMemsetAsync(warm.p, 0, 256 * sizeof(float), c->stream));
        CU(c, nccl_allreduce(comm, warm.p, 256, 0, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    c->sweep_nranks = nranks;
    c->sweep_rank = rank;
    return NMFK_OK;
}

int32_t nmfk_abi_version(void) { return NMFK_ABI_VERSION; }

const char* nmfk_last_error(const nmfk_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

void nmfk_default_params(nmfk_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->tol = 1e-19;
    p->tolOF = 1e-3;
    p->eps_clamp = 2.220446049250313e-16;
    p->weight = 1.0;
    p->maxiter = 10000;
    p->maxbaditers = 10;
    p->maxreattempts = 2;
    p->stopconv = 1000;
    p->check_every = 10;
    p->Wfixed = 0;
    p->Hfixed = 0;
    p->normalize = 1;
    p->iter_limit = 0;
    p->engine = NMFK_ENGINE_AUTO;
}

int32_t nmfk_ctx_create(int32_t device, nmfk_ctx** out) {
    if (!out) return fail(nullptr, NMFK_E_INVALID, "nmfk_ctx_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, NMFK_E_NO_DEVICE,
                    std::string("no CUDA device available (") + cudaGetErrorString(e) +
                        "); nmfk_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, NMFK_E_INVALID, "nmfk_ctx_create: bad device index");
    nmfk_ctx* c = new nmfk_ctx();
    c->device = device;
    e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    if (e != cudaSuccess) {
        const std::string msg = std::string("nmfk_ctx_create: ") + cudaGetErrorString(e);
        if (c->ev0) cudaEventDestroy(c->ev0);
        if (c->ev1) cudaEventDestroy(c->ev1);
        if (c->stream) cudaStreamDestroy(c->stream);
        delete c;
        return fail(nullptr, (int32_t)e, msg);
    }
    {  // scratch of the solves comes from the stream-ordered pool: keep freed blocks instead of returning them to the driver
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    (void)pinned_flags();
    tc2_pass_prepare();
    *out = c;
    return NMFK_OK;
}

int32_t nmfk_ctx_destroy(nmfk_ctx* c) {
    if (!c) return NMFK_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    nmfk_ctx_comm_destroy(c);
    free_X(c);
    c->prof.destroy();
    if (c->scratch) dev_free(c->scratch);
    if (c->Xstage) dev_free(c->Xstage);
    if (c->d_partials) dev_free(c->d_partials);
    for (auto s : c->pool) cudaStreamDestroy(s);
    for (auto e : c->pool_ev) cudaEventDestroy(e);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->stream) cudaStreamDestroy(c->stream);
    {  // hand the pooled blocks of this context back to the driver
        cudaMemPool_t pool = nullptr;
        cudaStreamSynchronize(cudaStreamPerThread);
        if (cudaDeviceGetDefaultMemPool(&pool, c->device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
    }
    delete c;
    return NMFK_OK;
}

int32_t nmfk_ctx_sync(nmfk_ctx* c) {
    if (!c) return fail(nullptr, NMFK_E_INVALID, "ctx is NULL");
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->stream));
    for (auto s : c->pool) CU(c, cudaStreamSynchronize(s));
    return NMFK_OK;
}

int32_t nmfk_set_X(nmfk_ctx* c, const void* X, int64_t n, int64_t m, int32_t dtype, double lambda,
                   const void* normalizevector, int32_t on_device) {
    if (!c) return fail(nullptr, NMFK_E_INVALID, "ctx is NULL");
    if (!X) return fail(c, NMFK_E_INVALID, "nmfk_set_X: X is NULL");
    if (dtype != NMFK_F32 && dtype != NMFK_F64) return fail(c, NMFK_E_INVALID, "nmfk_set_X: bad dtype");
    if (n <= 0 || m <= 0) return fail(c, NMFK_E_EMPTY, "Input array has a zero dimension!");
    if (n > INT32_MAX || m > INT32_MAX) return fail(c, NMFK_E_UNSUPPORTED, "nmfk_set_X: dimension exceeds int32");
    CU(c, cudaSetDevice(c->device));
    const size_t es = esize(dtype);
    const size_t bytes = (size_t)n * m * es;
    DevBuf Xp, Xpt, raw, stats, rf, cf, bm, Xn, Xnt, nv;
    if (c->Xp && c->Xpt && c->Xbytes == bytes) {  // same size as the previous X: reuse its images
        Xp.p = c->Xp;
        Xpt.p = c->Xpt;
        c->Xp = c->Xpt = nullptr;
    }
    raw.p = c->Xstage;
    c->Xstage = nullptr;
    if (c->Xbytes != bytes && raw.p) {
        dev_free(raw.p);
        raw.p = nullptr;
    }
    free_X(c);
    c->Xbytes = bytes;
    if (!Xp.p) CU(c, Xp.alloc(bytes));
    if (!Xpt.p) CU(c, Xpt.alloc(bytes));
    const void* src = X;
    if (!on_device) {
        if (!raw.p) CU(c, raw.alloc(bytes));
        CU(c, cudaMemcpyAsync(raw.p, X, bytes, cudaMemcpyHostToDevice, c->stream));
        src = raw.p;
    }
    const long long nb = ((n + 31) / 32) * ((m + 31) / 32);
    CU(c, stats.alloc(sizeof(PreStats)));
    CU(c, rf.alloc((size_t)n));
    CU(c, cf.alloc((size_t)m));
    CU(c, bm.alloc((size_t)nb * sizeof(double)));
    CU(c, launch_preprocess(src, Xp.p, Xpt.p, n, m, dtype, lambda, stats.as<PreStats>(), rf.as<unsigned char>(),
                            cf.as<unsigned char>(), bm.as<double>(), (int)nb, c->stream));
    c->launches += 3;
    if (normalizevector) {  // X ./= normalizevector after the lambda substitution (NMFkMultiplicative.jl:25-28)
        CU(c, Xn.alloc(bytes));
        CU(c, Xnt.alloc(bytes));
        CU(c, nv.alloc((size_t)n * es));
        CU(c, cudaMemcpyAsync(nv.p, normalizevector, (size_t)n * es, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                              c->stream));
        CU(c, launch_rownormalize(Xp.p, Xn.p, Xnt.p, n, m, nv.p, dtype, c->stream));
        c->launches += 2;
    }
    PreStats hs{};
    std::vector<double> bmh((size_t)nb);
    CU(c, cudaMemcpyAsync(&hs, stats.p, sizeof(hs), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(bmh.data(), bm.p, (size_t)nb * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    double xmin = std::numeric_limits<double>::infinity();
    for (double v : bmh) xmin = std::min(xmin, v);
    c->n = n;
    c->m = m;
    c->dtype = dtype;
    c->lambda = lambda;
    c->info = nmfk_xinfo{};
    c->info.n = n;
    c->info.m = m;
    c->info.nnan = (int64_t)hs.nnan;
    c->info.nzero = (int64_t)hs.nzero;
    c->info.zero_row = hs.zero_rows > 0;
    c->info.zero_col = hs.zero_cols > 0;
    c->info.xmin = xmin;
    c->info.dtype = dtype;
    // `minimum(X) < 0` is false when X holds a NaN (minimum propagates it): NMFkMultiplicative.jl:4
    if (hs.nneg > 0 && hs.nnan == 0) return fail(c, NMFK_E_NEGATIVE, "All matrix entries must be nonnegative!");
    c->Xp = Xp.release();
    c->Xpt = Xpt.release();
    if (bytes <= ((size_t)2 << 30)) c->Xstage = raw.release();  // larger staging copies are not worth keeping
    c->Xn = Xn.release();
    c->Xnt = Xnt.release();
    c->nv = nv.release();
    c->has_X = true;
    return NMFK_OK;
}

int32_t nmfk_set_weight(nmfk_ctx* c, const void* w, int64_t rows, int64_t cols) {
    if (!c) return fail(nullptr, NMFK_E_INVALID, "ctx is NULL");
    if (!c->has_X) return fail(c, NMFK_E_NO_X, "nmfk_set_X has not been called");
    CU(c, cudaSetDevice(c->device));
    for (void** q : {&c->wrow, &c->wcol, &c->wmat}) {
        if (*q) dev_free(*q);
        *q = nullptr;
    }
    if (!w) return NMFK_OK;
    // @assert typeof(weight) <: Number || length(weight) == size(X, 1) || size(weight, 2) == size(X, 2) || size(weight) == size(X)
    void** dst = nullptr;
    if (rows == c->n && cols == c->m)
        dst = &c->wmat;
    else if (rows == c->n && cols == 1)
        dst = &c->wrow;
    else if (rows == 1 && cols == c->m)
        dst = &c->wcol;
    else
        return fail(c, NMFK_E_SHAPE, "nmfk_set_weight: weight must be n x 1, 1 x m or n x m");
    const size_t bytes = (size_t)rows * cols * esize(c->dtype);
    CU(c, dev_malloc(dst, bytes));
    CU(c, cudaMemcpyAsync(*dst, w, bytes, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return NMFK_OK;
}

int32_t nmfk_get_xinfo(const nmfk_ctx* c, nmfk_xinfo* out) {
    if (!c || !out) return fail(nullptr, NMFK_E_INVALID, "nmfk_get_xinfo: NULL argument");
    if (!c->has_X) return fail(const_cast<nmfk_ctx*>(c), NMFK_E_NO_X, "nmfk_set_X has not been called");
    *out = c->info;
    return NMFK_OK;
}

int32_t nmfk_batch_create(nmfk_ctx* c, int32_t k, int32_t R, nmfk_batch** out) {
    if (!c || !out) return fail(c, NMFK_E_INVALID, "nmfk_batch_create: NULL argument");
    *out = nullptr;
    if (!c->has_X) return fail(c, NMFK_E_NO_X, "nmfk_set_X has not been called");
    if (k < 1 || R < 1) return fail(c, NMFK_E_INVALID, "nmfk_batch_create: k and R must be >= 1");
    CU(c, cudaSetDevice(c->device));
    nmfk_batch* b = new nmfk_batch();
    b->ctx = c;
    b->k = k;
    b->R = R;
    const size_t es = esize(c->dtype);
    cudaError_t e = dev_malloc(&b->W, (size_t)c->n * k * R * es);
    if (e == cudaSuccess) e = dev_malloc(&b->H, (size_t)k * c->m * R * es);
    if (e == cudaSuccess) e = dev_malloc(&b->st, (size_t)R * sizeof(UnitState));
    if (e == cudaSuccess) e = dev_malloc(&b->canon, (size_t)R * c->m * sizeof(int32_t));
    if (e == cudaSuccess && c->info.nnan > 0) e = dev_malloc(&b->ximp, (size_t)R * c->n * c->m * es);
    if (e != cudaSuccess) {
        nmfk_batch_destroy(b);
        CU(c, e);
    }
    *out = b;
    return NMFK_OK;
}

int32_t nmfk_batch_create_hstack(nmfk_ctx* c, int32_t k, int32_t R, nmfk_batch** out) {
    if (!c || !out) return fail(c, NMFK_E_INVALID, "nmfk_batch_create_hstack: NULL argument");
    *out = nullptr;
    if (!c->has_X) return fail(c, NMFK_E_NO_X, "nmfk_set_X has not been called");
    if (k < 1 || R < 1) return fail(c, NMFK_E_INVALID, "nmfk_batch_create_hstack: k and R must be >= 1");
    CU(c, cudaSetDevice(c->device));
    nmfk_batch* b = new nmfk_batch();
    b->ctx = c;
    b->k = k;
    b->R = R;
    cudaError_t e = dev_malloc(&b->H, (size_t)k * c->m * R * esize(c->dtype));
    if (e == cudaSuccess) e = dev_malloc(&b->st, (size_t)R * sizeof(UnitState));
    if (e != cudaSuccess) {
        nmfk_batch_destroy(b);
        CU(c, e);
    }
    *out = b;
    return NMFK_OK;
}

int32_t nmfk_batch_device_ptrs(nmfk_batch* b, void** W, void** H) {
    if (!b) return fail(nullptr, NMFK_E_INVALID, "nmfk_batch_device_ptrs: NULL batch");
    if (W) *W = b->W;
    if (H) *H = b->H;
    return NMFK_OK;
}

int32_t nmfk_batch_import(nmfk_batch* b, const void* W, const void* H, const double* obj_norm, const int32_t* iters,
                          int32_t on_device) {
    if (!b || !H || !obj_norm) return fail(b ? b->ctx : nullptr, NMFK_E_INVALID, "nmfk_batch_import: NULL argument");
    nmfk_ctx* c = b->ctx;
    CU(c, cudaSetDevice(c->device));
    const size_t es = esize(c->dtype);
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (W) {
        if (!b->W) return fail(c, NMFK_E_INVALID, "nmfk_batch_import: this batch has no W stack");
        CU(c, cudaMemcpyAsync(b->W, W, (size_t)c->n * b->k * b->R * es, kind, c->stream));
    }
    CU(c, cudaMemcpyAsync(b->H, H, (size_t)b->k * c->m * b->R * es, kind, c->stream));
    std::vector<UnitState> st((size_t)b->R);
    for (int r = 0; r < b->R; ++r) {
        std::memset(&st[r], 0, sizeof(UnitState));
        st[r].it = iters ? iters[r] : 0;
        st[r].stop = NMFK_STOP_MAXITER;
        st[r].done = 1;
        st[r].best = st[r].obj_chk = st[r].obj_ssq = std::numeric_limits<double>::quiet_NaN();
        st[r].obj_norm = obj_norm[r];
    }
    CU(c, cudaMemcpyAsync(b->st, st.data(), st.size() * sizeof(UnitState), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    b->inited = true;
    return NMFK_OK;
}

int32_t nmfk_batch_destroy(nmfk_batch* b) {
    if (!b) return NMFK_OK;
    if (b->ctx) cudaSetDevice(b->ctx->device);
    if (b->W) dev_free(b->W);
    if (b->H) dev_free(b->H);
    if (b->st) dev_free(b->st);
    if (b->canon) dev_free(b->canon);
    if (b->ximp) dev_free(b->ximp);
    delete b;
    return NMFK_OK;
}

static int32_t reset_state(nmfk_batch* b) {
    nmfk_ctx* c = b->ctx;
    std::vector<UnitState> st((size_t)b->R);
    for (auto& s : st) {
        std::memset(&s, 0, sizeof(s));
        s.best = std::numeric_limits<double>::infinity();
        s.obj_chk = std::numeric_limits<double>::quiet_NaN();
        s.obj_ssq = std::numeric_limits<double>::quiet_NaN();
        s.obj_norm = std::numeric_limits<double>::quiet_NaN();
    }
    CU(c, cudaMemcpyAsync(b->st, st.data(), st.size() * sizeof(UnitState), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemsetAsync(b->canon, 0xff, (size_t)b->R * c->m * sizeof(int32_t), c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    b->inited = true;
    return NMFK_OK;
}

static void reset_selection(nmfk_batch* b) {
    b->has_sel = false;
    b->sel.clear();
    b->nanaction = NMFK_NAN_ZEROED;
}

int32_t nmfk_batch_set_init_partial(nmfk_batch* b, const void* Winit, const void* Hinit, uint64_t seed0) {
    if (!b) return fail(nullptr, NMFK_E_INVALID, "nmfk_batch_set_init_partial: NULL batch");
    nmfk_ctx* c = b->ctx;
    CU(c, cudaSetDevice(c->device));
    if (!b->W) return fail(c, NMFK_E_INVALID, "nmfk_batch_set_init: H-only batch");
    const size_t wl = (size_t)c->n * b->k * b->R, hl = (size_t)b->k * c->m * b->R;
    if (c->sharded && (c->row0 + c->n > c->n_global))
        return fail(c, NMFK_E_SHAPE, "row-sharded ctx: row0 + local rows exceeds n_global");
    if (Winit) CU(c, cudaMemcpyAsync(b->W, Winit, wl * esize(c->dtype), cudaMemcpyHostToDevice, c->stream));
    if (Hinit) CU(c, cudaMemcpyAsync(b->H, Hinit, hl * esize(c->dtype), cudaMemcpyHostToDevice, c->stream));
    if (Winit || Hinit) {
        // "Initial values for the W / H matrix entries include NaNs!" (NMFkMultiplicative.jl:41, 52): checked on the device
        // copies (a single host thread scanning 82 MB of C3 initial factors cost 10 ms per call)
        DevBuf flags;
        const int R = b->R;
        CU(c, flags.alloc((size_t)2 * R * sizeof(int32_t)));
        int32_t* f = flags.as<int32_t>();
        if (Winit) CU(c, launch_count_nan(nullptr, b->W, 0, (int64_t)c->n * b->k, R, c->dtype, f, c->stream));
        if (Hinit) CU(c, launch_count_nan(nullptr, b->H, 0, (int64_t)b->k * c->m, R, c->dtype, f + R, c->stream));
        c->launches += (Winit ? 1 : 0) + (Hinit ? 1 : 0);
        std::vector<int32_t> hf((size_t)2 * R, 0);
        if (Winit) CU(c, cudaMemcpyAsync(hf.data(), f, (size_t)R * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        if (Hinit) CU(c, cudaMemcpyAsync(hf.data() + R, f + R, (size_t)R * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        bool wn = false, hn = false;
        for (int r = 0; r < R; ++r) {
            wn = wn || hf[r] != 0;
            hn = hn || hf[(size_t)R + r] != 0;
        }
        if (wn || hn) b->inited = false;
        if (wn) return fail(c, NMFK_E_NAN_INIT, "Initial values for the W matrix entries include NaNs!");
        if (hn) return fail(c, NMFK_E_NAN_INIT, "Initial values for the H matrix entries include NaNs!");
    }
    if (!Winit || !Hinit) {
        // the missing factor(s) from restart r's Philox stream: W = rand(n,k) only if Winit is empty, THEN H = rand(k,m) only
        // if Hinit is empty (NMFkMultiplicative.jl:37-55), so a lone missing factor takes the first numbers of the stream
        CU(c, launch_philox_init(Winit ? nullptr : b->W, Hinit ? nullptr : b->H, c->sharded ? c->n_global : c->n,
                                 c->sharded ? c->row0 : 0, c->n, b->k, c->m, b->R, seed0, c->dtype, c->stream));
        c->launches += 1;
    }
    reset_selection(b);
    return reset_state(b);
}

int32_t nmfk_batch_set_init(nmfk_batch* b, const void* Winit, const void* Hinit) {
    if (!b || !Winit || !Hinit) return fail(b ? b->ctx : nullptr, NMFK_E_INVALID, "nmfk_batch_set_init: NULL argument");
    return nmfk_batch_set_init_partial(b, Winit, Hinit, 0);
}

int32_t nmfk_batch_init_random(nmfk_batch* b, uint64_t seed0) {
    if (!b) return fail(nullptr, NMFK_E_INVALID, "nmfk_batch_init_random: NULL batch");
    return nmfk_batch_set_init_partial(b, nullptr, nullptr, seed0);
}

static int32_t check_params(nmfk_ctx* c, const nmfk_params* p) {
    if (!p) return fail(c, NMFK_E_INVALID, "params is NULL");
    if (p->check_every < 1 || p->maxiter < 0 || p->maxbaditers < 1 || p->maxreattempts < 1)
        return fail(c, NMFK_E_INVALID, "params: check_every, maxbaditers, maxreattempts must be >= 1, maxiter >= 0");
    if (p->normalize < 0 || p->normalize > 2) return fail(c, NMFK_E_INVALID, "params: normalize must be 0, 1 or 2");
    if (p->stop_rule < 0 || p->stop_rule > 1) return fail(c, NMFK_E_INVALID, "params: stop_rule must be 0 or 1");
    if (p->variant < NMFK_VARIANT_KL || p->variant > NMFK_VARIANT_KL_DIV) return fail(c, NMFK_E_INVALID, "params: unknown variant");
    if (p->stop_rule == 1 && c && c->info.nnan > 0)
        return fail(c, NMFK_E_UNSUPPORTED, "stop_rule 1 (the DArray method) with NaN entries in X is not supported: the reference "
                                           "itself returns objvalue = NaN there (NMFkMultiplicative.jl:193-195)");
    return NMFK_OK;
}

static void fill_args(const nmfk_batch* b, const nmfk_params* p, SolveArgs& a) {
    const nmfk_ctx* c = b->ctx;
    a.X = c->Xn ? c->Xn : c->Xp;  // normalizevector: the solver works on X ./ normalizevector
    a.Xt = c->Xn ? c->Xnt : c->Xpt;
    a.W = b->W;
    a.H = b->H;
    a.st = b->st;
    a.canon = b->canon;
    a.ximp = b->ximp;
    a.n = (int)c->n;
    a.m = (int)c->m;
    a.k = b->k;
    a.R = b->R;
    a.has_nan = c->info.nnan > 0;
    a.SH = a.SW = 1;
    a.maxiter = p->maxiter;
    a.maxbad = p->maxbaditers;
    a.maxre = p->maxreattempts;
    a.stopconv = p->stopconv;
    a.check_every = p->check_every;
    a.Wfixed = p->Wfixed;
    a.Hfixed = p->Hfixed;
    a.normalize = p->normalize;
    a.iter_limit = p->iter_limit;
    a.lambda = c->lambda;
    a.tol = p->tol;
    a.tolOF = p->tolOF;
    a.eps_clamp = p->eps_clamp;
    a.weight = p->weight;
    a.wref = WeightRef{c->wrow, c->wcol, c->wmat};
    if (p->stop_rule == 1) {
        // NMFmultiplicative(::DArray) (NMFkMultiplicative.jl:129-197): no tolOF / baditers / reattempts logic and no weight;
        // the loop ends on objvalue < tol, inc > stopconv or maxiter
        a.maxbad = INT32_MAX;
        a.maxre = INT32_MAX;
        a.weight = 1.0;
        a.wref = WeightRef{nullptr, nullptr, nullptr};
    }
    if (c->Xn) a.normalize = 0;  // the normalizevector epilogue (finish_normalizevector) rescales W first, then normalises
    a.tiled_tc = p->engine != NMFK_ENGINE_TILED_SCALAR;
    a.shard = c->sharded ? &c->shard : nullptr;
    a.prof = c->prof.enabled ? const_cast<PassProfile*>(&c->prof) : nullptr;
    a.timeout = nullptr;
}

// tiled engine (kl_tiled.cu): host-driven, for factors that do not fit in shared memory
namespace nmfk {
cudaError_t solve_tiled(const SolveArgs& a, int dtype, cudaStream_t s, int64_t* launches, bool div = false);
bool tiled_supported(int k);
}  // namespace nmfk

// a solver's return value; a barrier time-out it reported becomes an error naming the kernel and the site, like nmfk_gemm_nt's
// (status: the CUDA error of the trap that ends the time-out when the solver met it, NMFK_E_INVALID otherwise)
static int32_t solve_status(nmfk_ctx* c, const char* solver, cudaError_t e, const KernelTimeout& to) {
    if (to.kernel != nullptr)
        return fail(c, e == cudaErrorLaunchTimeout ? NMFK_E_INVALID : (int32_t)e,
                    std::string(solver) + ": barrier time-out inside " + to.kernel + " (" + to.where + ", site " + std::to_string(to.site) +
                        "): " + cudaGetErrorString(e));
    CU(c, e);
    return NMFK_OK;
}

// Epilogue of NMFmultiplicative with a normalizevector (NMFkMultiplicative.jl:119-125) followed by the objective / normalisation
// of execute_singlerun_compute (NMFkExecute.jl:791-804), for the restarts an engine has just finished (done == 1) on the
// normalised matrix: W .*= normalizevector; objvalue against the caller's X; then the H-row (or W-column) normalisation.
static int32_t finish_normalizevector(nmfk_batch* b, const nmfk_params* p) {
    nmfk_ctx* c = b->ctx;
    std::vector<UnitState> st((size_t)b->R);
    CU(c, cudaMemcpy(st.data(), b->st, st.size() * sizeof(UnitState), cudaMemcpyDeviceToHost));
    const size_t es = esize(c->dtype);
    bool touched = false;
    for (int r = 0; r < b->R; ++r) {
        if (st[r].stop == 0 || st[r].done != 1) continue;
        char* W = (char*)b->W + (size_t)r * c->n * b->k * es;
        char* H = (char*)b->H + (size_t)r * b->k * c->m * es;
        CU(c, launch_scale_rows(W, c->n, b->k, c->nv, c->dtype, c->stream));
        double o[2];
        int32_t rc = residual(c, b->k, W, H, 1, p->weight, o);  // against the caller's X (c->Xp), zeros restored
        if (rc) return rc;
        st[r].obj_ssq = o[0];
        st[r].obj_norm = std::sqrt(o[1]);
        CU(c, launch_renormalize(W, H, c->n, c->m, b->k, p->normalize, c->dtype, c->stream));
        c->launches += 1 + (p->normalize != 0);
        st[r].done = 2;
        touched = true;
    }
    if (touched) {
        CU(c, cudaMemcpyAsync(b->st, st.data(), st.size() * sizeof(UnitState), cudaMemcpyHostToDevice, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    return NMFK_OK;
}

// Variant FRO (method=:nmf, algorithm=:multdiv; NMFkExecute.jl:763-766): stacked-restart GEMMs, one batch after the other
static int32_t solve_fro_batches(nmfk_ctx* c, nmfk_batch* const* batches, int32_t nb, const nmfk_params* p) {
    if (c->info.nnan > 0) return fail(c, NMFK_E_UNSUPPORTED, "variant FRO: X holds NaN (NMF.jl's MultUpdate has no missing-data handling)");
    if (c->sharded || c->Xn || c->wrow || c->wcol || c->wmat)
        return fail(c, NMFK_E_UNSUPPORTED, "variant FRO: row-sharded X, normalizevector and array weights are not available");
    if (p->stop_rule != 0) return fail(c, NMFK_E_UNSUPPORTED, "variant FRO has its own stop rule (NMF.jl stop_condition)");
    if (c->dtype == NMFK_F32) {
        if (!fro_gemm_supported(c->m, c->n) || !fro_gemm_supported(c->n, c->m))
            return fail(c, NMFK_E_UNSUPPORTED, "variant FRO (Float32): row and column counts must be multiples of 4 (TMA strides) and "
                                               "the driver must provide cuTensorMapEncodeTiled");
        if (!c->Xlo) {
            const size_t bytes = (size_t)c->n * c->m * sizeof(float);
            CU(c, dev_malloc(&c->Xlo, bytes));
            CU(c, dev_malloc(&c->Xtlo, bytes));
            CU(c, launch_split_lo((const float*)c->Xp, (float*)c->Xlo, (long long)c->n * c->m, c->stream));
            CU(c, launch_split_lo((const float*)c->Xpt, (float*)c->Xtlo, (long long)c->n * c->m, c->stream));
            c->launches += 2;
        }
    }
    CU(c, cudaEventRecord(c->ev0, c->stream));
    for (int i = 0; i < nb; ++i) {
        if (batches[i]->k > 32) return fail(c, NMFK_E_UNSUPPORTED, "variant FRO: k > 32 is not supported");
        SolveArgs a;
        fill_args(batches[i], p, a);
        KernelTimeout to;
        a.timeout = &to;
        const int32_t rc = solve_status(c, "variant FRO", solve_fro(a, c->dtype, c->Xlo, c->Xtlo, c->stream, &c->launches), to);
        if (rc) return rc;
    }
    CU(c, cudaEventRecord(c->ev1, c->stream));
    CU(c, cudaEventSynchronize(c->ev1));
    float ms = 0.f;
    CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->last_solve_ms = ms;
    return NMFK_OK;
}

// NMFsparsity (method=:sparsity; NMFkExecute.jl:757-758, NMFkSparsity.jl:1-113), one batch after the other
static int32_t solve_sparsity_batches(nmfk_ctx* c, nmfk_batch* const* batches, int32_t nb, const nmfk_params* p) {
    if (c->info.nnan > 0) return fail(c, NMFK_E_UNSUPPORTED, "NMFsparsity: X holds NaN (the reference's preprocessing call is commented out)");
    if (c->sharded || c->Xn || c->wrow || c->wcol || c->wmat)
        return fail(c, NMFK_E_UNSUPPORTED, "NMFsparsity: row-sharded X, normalizevector and array weights are not available");
    CU(c, cudaEventRecord(c->ev0, c->stream));
    for (int i = 0; i < nb; ++i) {
        if (batches[i]->k > 32) return fail(c, NMFK_E_UNSUPPORTED, "NMFsparsity: k > 32 is not supported");
        SolveArgs a;
        fill_args(batches[i], p, a);
        CU(c, solve_sparsity(a, c->dtype, c->sp_beta, c->sp_sparsity, c->sp_lambda, c->stream, &c->launches));
    }
    CU(c, cudaEventRecord(c->ev1, c->stream));
    CU(c, cudaEventSynchronize(c->ev1));
    float ms = 0.f;
    CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->last_solve_ms = ms;
    return NMFK_OK;
}

// Variant KL_DIV (method=:nmf, algorithm=:multmse; NMFkExecute.jl:765-768): the tiled engine's passes in their delta flavour,
// one batch after the other.  Every size runs on the tiled engine (there is no resident flavour).
static int32_t solve_kl_div_batches(nmfk_ctx* c, nmfk_batch* const* batches, int32_t nb, const nmfk_params* p) {
    if (c->info.nnan > 0) return fail(c, NMFK_E_UNSUPPORTED, "variant KL_DIV: X holds NaN (NMF.jl's MultUpdate has no missing-data handling)");
    if (c->sharded) return fail(c, NMFK_E_UNSUPPORTED, "variant KL_DIV: row-sharded X is not available");
    if (c->Xn) return fail(c, NMFK_E_UNSUPPORTED, "variant KL_DIV: normalizevector is not available");
    if (c->wrow || c->wcol || c->wmat) return fail(c, NMFK_E_UNSUPPORTED, "variant KL_DIV: array weights are not available");
    if (p->stop_rule != 0) return fail(c, NMFK_E_UNSUPPORTED, "variant KL_DIV has its own stop rule (NMF.jl stop_condition)");
    if (p->engine == NMFK_ENGINE_RESIDENT || p->engine == NMFK_ENGINE_RESIDENT_SCALAR)
        return fail(c, NMFK_E_UNSUPPORTED, "variant KL_DIV: only the tiled engine is available");
    for (int i = 0; i < nb; ++i)
        if (!tiled_supported(batches[i]->k)) return fail(c, NMFK_E_UNSUPPORTED, "variant KL_DIV: k > 64 is not supported");
    CU(c, cudaEventRecord(c->ev0, c->stream));
    for (int i = 0; i < nb; ++i) {
        SolveArgs a;
        fill_args(batches[i], p, a);
        KernelTimeout to;
        a.timeout = &to;
        const int32_t rc = solve_status(c, "variant KL_DIV", solve_tiled(a, c->dtype, c->stream, &c->launches, true), to);
        if (rc) return rc;
    }
    CU(c, cudaEventRecord(c->ev1, c->stream));
    CU(c, cudaEventSynchronize(c->ev1));
    float ms = 0.f;
    CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->last_solve_ms = ms;
    return NMFK_OK;
}

int32_t nmfk_set_sparsity_options(nmfk_ctx* c, double beta_divergence, double sparsity, double lambda) {
    if (!c) return fail(nullptr, NMFK_E_INVALID, "ctx is NULL");
    if (!(lambda > 0)) return fail(c, NMFK_E_INVALID, "nmfk_set_sparsity_options: lambda must be positive");
    c->sp_beta = beta_divergence;
    c->sp_sparsity = sparsity;
    c->sp_lambda = lambda;
    return NMFK_OK;
}

int32_t nmfk_solve(nmfk_ctx* c, nmfk_batch* const* batches, int32_t nb, const nmfk_params* p) {
    if (!c || !batches || nb < 1) return fail(c, NMFK_E_INVALID, "nmfk_solve: bad arguments");
    int32_t rc = check_params(c, p);
    if (rc) return rc;
    CU(c, cudaSetDevice(c->device));
    for (int i = 0; i < nb; ++i) {
        if (!batches[i] || batches[i]->ctx != c) return fail(c, NMFK_E_INVALID, "nmfk_solve: batch of another ctx");
        if (!batches[i]->inited) return fail(c, NMFK_E_INVALID, "nmfk_solve: batch has no initialisation");
        if (!batches[i]->W || !batches[i]->canon) return fail(c, NMFK_E_INVALID, "nmfk_solve: H-only batch");
    }
    if (p->variant == NMFK_VARIANT_FRO) return solve_fro_batches(c, batches, nb, p);
    if (p->variant == NMFK_VARIANT_SPARSITY) return solve_sparsity_batches(c, batches, nb, p);
    if (p->variant == NMFK_VARIANT_KL_DIV) return solve_kl_div_batches(c, batches, nb, p);
    while ((int)c->pool.size() < nb) {
        cudaStream_t s;
        cudaEvent_t ev;
        CU(c, cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        CU(c, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        c->pool.push_back(s);
        c->pool_ev.push_back(ev);
    }
    // largest k first: its restarts are the longest units (LPT order for the block scheduler)
    std::vector<int> ord(nb);
    std::iota(ord.begin(), ord.end(), 0);
    std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return batches[x]->k > batches[y]->k; });
    const size_t es = esize(c->dtype);
    CU(c, cudaEventRecord(c->ev0, c->stream));
    // Resident engine: one CTA runs one restart to its stop, and restarts of one sweep stop anywhere
    // between a few hundred and maxiter iterations.  To keep the tail of the sweep short, a solve is
    // enqueued as a sequence of launches that each advance every unfinished restart by at most
    // kResidentChunk iterations (the state is resumable; finished restarts exit at once): SMs freed by
    // short restarts are refilled at chunk granularity and the last wave is at most one chunk long.
    constexpr int kResidentChunk = 500;
    const int user_limit = p->iter_limit > 0 ? std::min(p->iter_limit, p->maxiter) : p->maxiter;
    std::vector<int> mode(nb, 0);  // 1 dmma, 2 scalar resident, 3 tiled
    std::vector<SolveArgs> args(nb);
    for (int q = 0; q < nb; ++q) {
        nmfk_batch* b = batches[ord[q]];
        SolveArgs& a = args[q];
        fill_args(b, p, a);
        CU(c, cudaStreamWaitEvent(c->pool[q], c->ev0, 0));
        const bool want_scalar = (p->engine == NMFK_ENGINE_RESIDENT_SCALAR) || c->dtype != NMFK_F64;
        const bool fits_dmma = !want_scalar && resident_dmma_fits(a.n, a.m, a.k);
        const bool fits_scalar = resident_fits(a.n, a.m, a.k, es);
        bool resident = fits_dmma || fits_scalar;
        if (p->engine == NMFK_ENGINE_TILED || p->engine == NMFK_ENGINE_TILED_SCALAR) resident = false;
        if (a.wref.any()) {  // per-row / per-column / per-entry weights live in the tiled engine's scalar objective kernel
            if (p->engine == NMFK_ENGINE_RESIDENT || p->engine == NMFK_ENGINE_RESIDENT_SCALAR)
                return fail(c, NMFK_E_UNSUPPORTED, "vector / matrix weights: only the tiled engine is available");
            resident = false;
        }
        if (c->sharded) {  // rows of X / W live on several GPUs: only the tiled engine exchanges partials
            if (p->engine == NMFK_ENGINE_RESIDENT || p->engine == NMFK_ENGINE_RESIDENT_SCALAR)
                return fail(c, NMFK_E_UNSUPPORTED, "row-sharded ctx: only the tiled engine is available");
            if (p->normalize == 2) return fail(c, NMFK_E_UNSUPPORTED, "row-sharded ctx: clusterWmatrix normalisation is not available");
            if (c->Xn || a.wref.any())
                return fail(c, NMFK_E_UNSUPPORTED, "row-sharded ctx: normalizevector / non-scalar weights are not available");
            resident = false;
        }
        if ((p->engine == NMFK_ENGINE_RESIDENT || p->engine == NMFK_ENGINE_RESIDENT_SCALAR) && !resident)
            return fail(c, NMFK_E_UNSUPPORTED, "resident engine: factors do not fit in shared memory (or k > 32)");
        if (!resident && !tiled_supported(a.k)) return fail(c, NMFK_E_UNSUPPORTED, "tiled engine: k > 64 is not supported");
        mode[q] = resident ? (fits_dmma ? 1 : 2) : 3;
    }
    for (int lim = std::min(kResidentChunk, user_limit);; lim = std::min(lim + kResidentChunk, user_limit)) {
        for (int q = 0; q < nb; ++q) {
            if (mode[q] == 3) continue;
            SolveArgs a = args[q];
            a.iter_limit = lim < p->maxiter ? lim : p->iter_limit;  // the last launch runs to the real stop
            if (mode[q] == 1)
                CU(c, launch_kl_resident_dmma(a, c->pool[q]));
            else
                CU(c, c->dtype == NMFK_F64 ? launch_kl_resident_f64(a, c->pool[q]) : launch_kl_resident_f32(a, c->pool[q]));
            c->launches += 1;
        }
        if (lim >= user_limit) break;
    }
    for (int q = 0; q < nb; ++q) {
        if (mode[q] == 3) {
            KernelTimeout to;
            args[q].timeout = &to;
            rc = solve_status(c, "tiled engine", solve_tiled(args[q], c->dtype, c->pool[q], &c->launches), to);
            if (rc) return rc;
        }
        CU(c, cudaEventRecord(c->pool_ev[q], c->pool[q]));
        CU(c, cudaStreamWaitEvent(c->stream, c->pool_ev[q], 0));
    }
    CU(c, cudaEventRecord(c->ev1, c->stream));
    CU(c, cudaEventSynchronize(c->ev1));
    float ms = 0.f;
    CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->last_solve_ms = ms;
    if (c->Xn)
        for (int i = 0; i < nb; ++i) {
            rc = finish_normalizevector(batches[i], p);
            if (rc) return rc;
        }
    return NMFK_OK;
}

static int32_t fetch_state(nmfk_batch* b, std::vector<UnitState>& st) {
    nmfk_ctx* c = b->ctx;
    st.resize((size_t)b->R);
    CU(c, cudaMemcpy(st.data(), b->st, st.size() * sizeof(UnitState), cudaMemcpyDeviceToHost));
    return NMFK_OK;
}

int32_t nmfk_batch_get(nmfk_batch* b, void* W_out, void* H_out, double* obj_ssq, double* obj_norm, int32_t* iters,
                       int32_t* stop_reason) {
    if (!b) return fail(nullptr, NMFK_E_INVALID, "nmfk_batch_get: NULL batch");
    nmfk_ctx* c = b->ctx;
    CU(c, cudaSetDevice(c->device));
    const size_t es = esize(c->dtype);
    if (W_out) CU(c, cudaMemcpy(W_out, b->W, (size_t)c->n * b->k * b->R * es, cudaMemcpyDeviceToHost));
    if (H_out) CU(c, cudaMemcpy(H_out, b->H, (size_t)b->k * c->m * b->R * es, cudaMemcpyDeviceToHost));
    if (obj_ssq || obj_norm || iters || stop_reason) {
        std::vector<UnitState> st;
        int32_t rc = fetch_state(b, st);
        if (rc) return rc;
        for (int r = 0; r < b->R; ++r) {
            if (obj_ssq) obj_ssq[r] = st[r].obj_ssq;
            if (obj_norm) obj_norm[r] = st[r].obj_norm;
            if (iters) iters[r] = st[r].it;
            if (stop_reason) stop_reason[r] = st[r].stop;
        }
    }
    return NMFK_OK;
}

// residual sums of one (W,H) device pair; out[0] = weighted ssq, out[1] = plain ssq
static int32_t residual(nmfk_ctx* c, int k, const void* W, const void* H, int restore, double weight, double out[2]) {
    const int nb = residual_blocks((int)c->n, (int)c->m);
    if (c->partials_cap < (size_t)nb * 2) {
        if (c->d_partials) dev_free(c->d_partials);
        c->d_partials = nullptr;
        CU(c, dev_malloc(&c->d_partials, (size_t)nb * 2 * sizeof(double)));
        c->partials_cap = (size_t)nb * 2;
    }
    CU(c, launch_residual(c->Xp, c->dtype, (int)c->n, (int)c->m, k, W, H, c->lambda, restore, weight,
                          WeightRef{c->wrow, c->wcol, c->wmat}, c->d_partials, c->stream));
    c->launches += 1;
    std::vector<double> h((size_t)nb * 2);
    CU(c, cudaMemcpyAsync(h.data(), c->d_partials, h.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    out[0] = out[1] = 0.0;
    for (int i = 0; i < nb; ++i) {
        out[0] += h[2 * i];
        out[1] += h[2 * i + 1];
    }
    return NMFK_OK;
}

int32_t nmfk_batch_objective(nmfk_batch* b, double weight, double* obj_ssq) {
    if (!b || !obj_ssq) return fail(b ? b->ctx : nullptr, NMFK_E_INVALID, "nmfk_batch_objective: NULL argument");
    nmfk_ctx* c = b->ctx;
    CU(c, cudaSetDevice(c->device));
    const size_t es = esize(c->dtype);
    for (int r = 0; r < b->R; ++r) {
        double o[2];
        int32_t rc = residual(c, b->k, (const char*)b->W + (size_t)r * c->n * b->k * es,
                              (const char*)b->H + (size_t)r * b->k * c->m * es, 0, weight, o);
        if (rc) return rc;
        obj_ssq[r] = o[0];
    }
    return NMFK_OK;
}

// idxsort = sortperm(objvalue) (NMFkExecute.jl:545): stable, ascending, NaN last; objvalue is a Vector{T}
static void sorted_order(const nmfk_ctx* c, const std::vector<UnitState>& st, std::vector<double>& obj, std::vector<int32_t>& order) {
    const int R = (int)st.size();
    obj.resize((size_t)R);
    for (int r = 0; r < R; ++r) obj[r] = c->dtype == NMFK_F32 ? (double)(float)st[r].obj_norm : st[r].obj_norm;
    order.resize((size_t)R);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
        const double a = obj[x], d = obj[y];
        if (a != a) return false;  // NaN is never less
        if (d != d) return true;
        return a < d;
    });
}

int32_t nmfk_batch_select(nmfk_batch* b, double acceptratio, double acceptfactor, int32_t nanaction, int32_t* order_kept,
                          int32_t* nkept) {
    if (!b) return fail(nullptr, NMFK_E_INVALID, "nmfk_batch_select: NULL batch");
    nmfk_ctx* c = b->ctx;
    if (nanaction != NMFK_NAN_ZEROED && nanaction != NMFK_NAN_REMOVED)
        return fail(c, NMFK_E_INVALID, "nmfk_batch_select: nanaction must be :zeroed or :removed");
    CU(c, cudaSetDevice(c->device));
    const int R = b->R;
    std::vector<UnitState> st;
    int32_t rc = fetch_state(b, st);
    if (rc) return rc;
    std::vector<double> obj;
    std::vector<int32_t> order;
    sorted_order(c, st, obj, order);
    std::vector<char> keep((size_t)R, 1);
    if (acceptratio < 1) {  // idxrat = [trues(ccc); falses(nNMF - ccc)] (:552-555)
        const int ccc = (int)std::ceil((double)R * acceptratio);
        for (int t = 0; t < R; ++t) keep[t] = keep[t] && (t < ccc);
    }
    if (acceptfactor < std::numeric_limits<double>::infinity()) {  // idxcut = objvalue[idxsort] .< cutoff (:559-562)
        const double cutoff = obj[order[0]] * acceptfactor;
        for (int t = 0; t < R; ++t) keep[t] = keep[t] && (obj[order[t]] < cutoff);
    }
    if (nanaction == NMFK_NAN_REMOVED) {  // idxnan[i] = false for restart NUMBER i (:581-596), ANDed by position like the reference
        DevBuf flags;
        CU(c, flags.alloc((size_t)R * sizeof(int32_t)));
        CU(c, launch_count_nan(b->W, b->H, (int64_t)c->n * b->k, (int64_t)b->k * c->m, R, c->dtype, flags.as<int32_t>(), c->stream));
        c->launches += 1;
        std::vector<int32_t> hf((size_t)R);
        CU(c, cudaMemcpyAsync(hf.data(), flags.p, (size_t)R * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        for (int t = 0; t < R; ++t) keep[t] = keep[t] && !hf[t];
    }
    b->sel.clear();
    for (int t = 0; t < R; ++t)
        if (keep[t]) b->sel.push_back(order[t]);
    b->has_sel = true;
    b->nanaction = nanaction;
    if (order_kept) std::copy(b->sel.begin(), b->sel.end(), order_kept);
    if (nkept) *nkept = (int32_t)b->sel.size();
    return NMFK_OK;
}

int32_t nmfk_batch_cluster(nmfk_batch* b, int32_t clusterWmatrix, int32_t* order_out, int32_t* labels_out,
                           double* sil_out, double* clustersil_out, double* robustness_out, void* centroids_out,
                           int32_t* centroid_cols) {
    if (!b) return fail(nullptr, NMFK_E_INVALID, "nmfk_batch_cluster: NULL batch");
    nmfk_ctx* c = b->ctx;
    CU(c, cudaSetDevice(c->device));
    const int k = b->k;
    std::vector<int32_t> order;
    if (b->has_sel) {
        order = b->sel;
    } else {
        std::vector<UnitState> st;
        int32_t rc = fetch_state(b, st);
        if (rc) return rc;
        std::vector<double> obj;
        sorted_order(c, st, obj, order);
    }
    const int R = (int)order.size();  // solutions that reach clustersolutions / finalize
    if (R < 1) return fail(c, NMFK_E_INVALID, "nmfk_batch_cluster: no solutions remain after the acceptance filters");
    if (order_out) std::copy(order.begin(), order.end(), order_out);
    if (k == 1) {  // minsilhouette = 1 when nk == 1 (NMFkExecute.jl:618); Wbest / Hbest were copied before the NaN pass (:549-550)
        if (labels_out) std::fill(labels_out, labels_out + R, 1);
        if (sil_out) std::fill(sil_out, sil_out + R, 1.0);
        if (clustersil_out) clustersil_out[0] = 1.0;
        if (robustness_out) *robustness_out = 1.0;
        if (centroid_cols) *centroid_cols = 0;
        return NMFK_OK;
    }
    // nanaction = :zeroed (:566-580) touches every stored solution, kept or not
    if (b->nanaction == NMFK_NAN_ZEROED) {
        if (b->W) CU(c, launch_zero_nan(b->W, (long long)c->n * k * b->R, c->dtype, c->stream));
        CU(c, launch_zero_nan(b->H, (long long)k * c->m * b->R, c->dtype, c->stream));
        c->launches += 2;
    }
    const int len = clusterWmatrix ? (int)c->n : (int)c->m;
    const int N = R * k, ld = len + 1;
    if (clusterWmatrix && !b->W) return fail(c, NMFK_E_INVALID, "nmfk_batch_cluster: clusterWmatrix on an H-only batch");
    // one persistent scratch arena instead of nine cudaMalloc / cudaFree per call (the N x N distance matrix is 537 MB at
    // BASELINE C4 k = 32)
    auto up = [](size_t v) { return (v + 255) / 256 * 256; };
    const size_t o_order = 0, o_labels = o_order + up((size_t)R * 4), o_cent = o_labels + up((size_t)N * 4),
                 o_sil = o_cent + up((size_t)k * ld * 8), o_csil = o_sil + up((size_t)N * 8), o_bias = o_csil + up((size_t)k * 8),
                 o_vnorm = o_bias + 256, o_V = o_vnorm + up((size_t)N * 8), o_D = o_V + up((size_t)N * ld * 8),
                 total = o_D + up((size_t)N * N * 8);
    char* base = nullptr;
    CU(c, ctx_scratch(c, total, reinterpret_cast<void**>(&base)));
    ClusterArgs a{};
    int32_t* d_order = reinterpret_cast<int32_t*>(base + o_order);
    a.labels = reinterpret_cast<int32_t*>(base + o_labels);
    a.cent = reinterpret_cast<double*>(base + o_cent);
    a.sil = reinterpret_cast<double*>(base + o_sil);
    a.clustersil = reinterpret_cast<double*>(base + o_csil);
    a.bias = reinterpret_cast<int32_t*>(base + o_bias);
    a.vnorm = reinterpret_cast<double*>(base + o_vnorm);
    a.V = reinterpret_cast<double*>(base + o_V);
    a.Dm = reinterpret_cast<double*>(base + o_D);
    std::vector<int32_t> labels((size_t)N);
    std::vector<double> sil((size_t)N), csil((size_t)k), cent((size_t)k * ld);
    int32_t bias = 0;
    CU(c, cudaMemcpyAsync(d_order, order.data(), (size_t)R * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    a.F = clusterWmatrix ? b->W : b->H;
    a.len = len;
    a.k = k;
    a.R = R;
    a.use_W = clusterWmatrix;
    a.order = d_order;
    // clusterWmatrix = true: the reference's `newClusterCenters = factors[1]` IS WBig[bestIdx] (no copy is made on this
    // branch, NMFkCluster.jl:426-428, 453-455), so clustersolutions leaves the centroids (running sums ./ numTrials, :484,
    // :512) in the best solution's W before finalize / Wbest read it (NMFkExecute.jl:631-637).  Not when the zero-column fix
    // fired: vcat (:449) made fresh matrices.
    a.alias_best = clusterWmatrix ? ((char*)b->W + (size_t)order[0] * c->n * k * esize(c->dtype)) : nullptr;
    CU(c, launch_cluster(a, c->dtype, c->stream));
    c->launches += 5 + cluster_walk_launches(k, len, R) + (clusterWmatrix ? 1 : 0);
    CU(c, cudaMemcpyAsync(labels.data(), a.labels, labels.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(sil.data(), a.sil, sil.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(csil.data(), a.clustersil, csil.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(cent.data(), a.cent, cent.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(&bias, a.bias, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (labels_out) std::copy(labels.begin(), labels.end(), labels_out);
    if (sil_out) std::copy(sil.begin(), sil.end(), sil_out);
    if (clustersil_out) std::copy(csil.begin(), csil.end(), clustersil_out);
    if (robustness_out) {  // minimum(clustersilhouettes) (:638); Julia's minimum propagates NaN
        double mn = std::numeric_limits<double>::infinity();
        bool anynan = false;
        for (double v : csil) {
            if (v != v) anynan = true;
            mn = std::min(mn, v);
        }
        *robustness_out = anynan ? std::numeric_limits<double>::quiet_NaN() : mn;
        if (c->dtype == NMFK_F32) *robustness_out = (double)(float)*robustness_out;
    }
    const int cols = bias ? ld : len;
    if (centroid_cols) *centroid_cols = cols;
    if (centroids_out) {  // permutedims(newClusterCenters): k x cols, column-major, element type T
        for (int cc = 0; cc < k; ++cc)
            for (int j = 0; j < cols; ++j) {
                const double v = cent[(size_t)cc * ld + j];
                if (c->dtype == NMFK_F64)
                    ((double*)centroids_out)[(size_t)cc + (size_t)j * k] = v;
                else
                    ((float*)centroids_out)[(size_t)cc + (size_t)j * k] = (float)v;
            }
    }
    return NMFK_OK;
}

int32_t nmfk_fit(nmfk_ctx* c, int32_t k, const void* W, const void* H, double* phi) {
    if (!c || !W || !H || !phi || k < 1) return fail(c, NMFK_E_INVALID, "nmfk_fit: bad arguments");
    if (!c->has_X) return fail(c, NMFK_E_NO_X, "nmfk_set_X has not been called");
    CU(c, cudaSetDevice(c->device));
    const size_t es = esize(c->dtype);
    const size_t wb = (size_t)c->n * k * es, hb = (size_t)k * c->m * es;
    DevBuf dW, dH;
    CU(c, dW.alloc(wb));
    CU(c, dH.alloc(hb));
    CU(c, cudaMemcpyAsync(dW.p, W, wb, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(dH.p, H, hb, cudaMemcpyHostToDevice, c->stream));
    double o[2] = {0, 0};
    int32_t rc = residual(c, k, dW.p, dH.p, 1, 1.0, o);
    if (rc) return rc;
    *phi = std::sqrt(o[1]);
    if (c->dtype == NMFK_F32) *phi = (double)(float)*phi;
    return NMFK_OK;
}

// Wmean, Hmean, Wvar, Hvar of finalize (NMFkFinalize.jl:68-74): what execute_run returns with best=false (:655-658) and what
// the "-all" result file stores (:650-654).  order / labels as returned by nmfk_batch_cluster (labels k x R, 1-based, column t =
// trial t in sorted order).  Any output may be NULL.
int32_t nmfk_batch_cluster_means(nmfk_batch* b, const int32_t* order, const int32_t* labels, void* Wmean, void* Hmean,
                                 void* Wvar, void* Hvar) {
    if (!b || !order || !labels) return fail(b ? b->ctx : nullptr, NMFK_E_INVALID, "nmfk_batch_cluster_means: NULL argument");
    nmfk_ctx* c = b->ctx;
    CU(c, cudaSetDevice(c->device));
    const int k = b->k, R = b->has_sel ? (int)b->sel.size() : b->R;  // the solutions that reached finalize
    const long long n = c->n, m = c->m;
    if (R < 1) return fail(c, NMFK_E_INVALID, "nmfk_batch_cluster_means: no solutions selected");
    if ((Wmean || Wvar) && !b->W) return fail(c, NMFK_E_INVALID, "nmfk_batch_cluster_means: W statistics on an H-only batch");
    std::vector<int32_t> amap((size_t)k * R, -1);
    for (int t = 0; t < R; ++t) {
        if (order[t] < 0 || order[t] >= b->R) return fail(c, NMFK_E_INVALID, "nmfk_batch_cluster_means: order out of range");
        for (int a = 0; a < k; ++a) {
            const int lab = labels[(size_t)t * k + a];
            if (lab >= 1 && lab <= k && amap[(size_t)(lab - 1) * R + t] < 0) amap[(size_t)(lab - 1) * R + t] = a;
        }
    }
    const size_t es = esize(c->dtype);
    DevBuf b_order, b_amap, b_out;
    const size_t wbytes = (size_t)n * k * es, hbytes = (size_t)k * m * es;
    cudaError_t e = b_order.alloc((size_t)R * sizeof(int32_t));
    if (e == cudaSuccess) e = b_amap.alloc(amap.size() * sizeof(int32_t));
    if (e == cudaSuccess) e = b_out.alloc(2 * (wbytes + hbytes));
    CU(c, e);
    int32_t *d_order = b_order.as<int32_t>(), *d_amap = b_amap.as<int32_t>();
    unsigned char* d_out = b_out.as<unsigned char>();
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_order, order, (size_t)R * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_amap, amap.data(), amap.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
    unsigned char *dWm = d_out, *dWv = d_out + wbytes, *dHm = d_out + 2 * wbytes, *dHv = dHm + hbytes;
    if (e == cudaSuccess && (Wmean || Wvar)) {
        e = launch_cluster_means(b->W, (int)n, k, R, 1, d_order, d_amap, dWm, dWv, c->dtype, c->stream);
        c->launches += 1;
    }
    if (e == cudaSuccess && (Hmean || Hvar)) {
        e = launch_cluster_means(b->H, (int)m, k, R, 0, d_order, d_amap, dHm, dHv, c->dtype, c->stream);
        c->launches += 1;
    }
    if (e == cudaSuccess && Wmean) e = cudaMemcpyAsync(Wmean, dWm, wbytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && Wvar) e = cudaMemcpyAsync(Wvar, dWv, wbytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && Hmean) e = cudaMemcpyAsync(Hmean, dHm, hbytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess && Hvar) e = cudaMemcpyAsync(Hvar, dHv, hbytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    CU(c, e);
    return NMFK_OK;
}

int32_t nmfk_run_batch(nmfk_ctx* c, int32_t k, int32_t R, const void* Winit, const void* Hinit, const nmfk_params* p,
                       void* W_out, void* H_out, double* obj_ssq, double* obj_norm, int32_t* iters,
                       int32_t* stop_reason) {
    nmfk_batch* b = nullptr;
    int32_t rc = nmfk_batch_create(c, k, R, &b);
    if (rc) return rc;
    rc = nmfk_batch_set_init(b, Winit, Hinit);
    if (!rc) rc = nmfk_solve(c, &b, 1, p);
    if (!rc) rc = nmfk_batch_get(b, W_out, H_out, obj_ssq, obj_norm, iters, stop_reason);
    nmfk_batch_destroy(b);
    return rc;
}

int32_t nmfk_trace(nmfk_ctx* c, int32_t k, const void* Winit, const void* Hinit, const nmfk_params* p, int32_t niter,
                   void* W_t, void* H_t, double* obj_t) {
    if (!c || !p || niter < 1) return fail(c, NMFK_E_INVALID, "nmfk_trace: bad arguments");
    nmfk_batch* b = nullptr;
    int32_t rc = nmfk_batch_create(c, k, 1, &b);
    if (rc) return rc;
    rc = nmfk_batch_set_init(b, Winit, Hinit);
    const size_t es = esize(c->dtype);
    const size_t wb = (size_t)c->n * k * es, hb = (size_t)k * c->m * es;
    nmfk_params q = *p;
    for (int t = 1; t <= niter && !rc; ++t) {
        q.iter_limit = t;
        rc = nmfk_solve(c, &b, 1, &q);
        if (rc) break;
        rc = nmfk_batch_get(b, W_t ? (char*)W_t + (size_t)(t - 1) * wb : nullptr,
                            H_t ? (char*)H_t + (size_t)(t - 1) * hb : nullptr, nullptr, nullptr, nullptr, nullptr);
        if (!rc && obj_t) rc = nmfk_batch_objective(b, p->weight, obj_t + (t - 1));
    }
    nmfk_batch_destroy(b);
    return rc;
}

// host copy of one restart's factors
static int32_t fetch_factors(nmfk_batch* b, int r, std::vector<char>& W, std::vector<char>& H) {
    nmfk_ctx* c = b->ctx;
    const size_t es = esize(c->dtype);
    const size_t wb = (size_t)c->n * b->k * es, hb = (size_t)b->k * c->m * es;
    W.resize(wb);
    H.resize(hb);
    CU(c, cudaMemcpy(W.data(), (const char*)b->W + (size_t)r * wb, wb, cudaMemcpyDeviceToHost));
    CU(c, cudaMemcpy(H.data(), (const char*)b->H + (size_t)r * hb, hb, cudaMemcpyDeviceToHost));
    return NMFK_OK;
}

template <typename T>
static void signal_sums(const T* W, const T* H, int64_t n, int k, int64_t m, std::vector<double>& s) {
    // sum(W[:,i:i] * H[i:i,:]) == sum(W[:,i]) * sum(H[i,:]) up to rounding (NMFkPostprocess.jl:151-153)
    s.assign((size_t)k, 0.0);
    for (int a = 0; a < k; ++a) {
        double sw = 0.0, sh = 0.0;
        for (int64_t i = 0; i < n; ++i) sw += (double)W[i + (int64_t)a * n];
        for (int64_t j = 0; j < m; ++j) sh += (double)H[a + j * k];
        s[a] = sw * sh;
    }
}

int32_t nmfk_signalorder(const void* W, const void* H, int64_t n, int32_t k, int64_t m, int32_t dtype,
                         int32_t* order) {
    if (!W || !H || !order || k < 1) return fail(nullptr, NMFK_E_INVALID, "nmfk_signalorder: bad arguments");
    std::vector<double> s;
    if (dtype == NMFK_F64)
        signal_sums((const double*)W, (const double*)H, n, k, m, s);
    else
        signal_sums((const float*)W, (const float*)H, n, k, m, s);
    std::iota(order, order + k, 0);
    // sortperm(signal_sum; rev=true): stable, descending
    std::stable_sort(order, order + k, [&](int x, int y) {
        const double a = s[x], d = s[y];
        if (a != a) return d == d;  // rev=true puts NaN first (isless ordering reversed)
        if (d != d) return false;
        return a > d;
    });
    return NMFK_OK;
}

int32_t nmfk_getk(const int32_t* ks, const double* rob, int32_t nks, double cutoff, int32_t strict) {
    if (!ks || !rob || nks < 1) return -1;
    bool allnan = true;
    for (int i = 0; i < nks; ++i)
        if (rob[i] == rob[i]) allnan = false;
    if (allnan) return 0;  // NMFkPostprocess.jl:11-13
    if (nks == 1) {        // :14-23
        if (strict) return rob[0] > cutoff ? ks[0] : -1;
        return ks[0];
    }
    int kn = -1;
    for (int i = 0; i < nks; ++i)
        if (rob[i] > cutoff) kn = i;  // findlast (:25)
    if (kn >= 0) return ks[kn];
    if (strict) return -1;
    int best = -1;  // findmax with NaN -> -Inf (:30-34): first maximum
    double bv = -std::numeric_limits<double>::infinity();
    for (int i = 0; i < nks; ++i) {
        const double v = (rob[i] != rob[i]) ? -std::numeric_limits<double>::infinity() : rob[i];
        if (best < 0 || v > bv) {
            best = i;
            bv = v;
        }
    }
    return ks[best];
}

// phi_final = normnan(X - Wa*Ha) with NaN residuals zeroed (NMFkExecute.jl:664-668) and aic (:697-708) of host factors
static int32_t phi_aic(nmfk_ctx* c, int k, const std::vector<char>& Wb, const std::vector<char>& Hb, double* phi, double* aic) {
    DevBuf dW, dH;
    CU(c, dW.alloc(Wb.size()));
    CU(c, dH.alloc(Hb.size()));
    CU(c, cudaMemcpyAsync(dW.p, Wb.data(), Wb.size(), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(dH.p, Hb.data(), Hb.size(), cudaMemcpyHostToDevice, c->stream));
    double o[2] = {0, 0};
    int32_t rc = residual(c, k, dW.p, dH.p, 1, 1.0, o);
    if (rc) return rc;
    double ph = std::sqrt(o[1]);
    if (c->dtype == NMFK_F32) ph = (double)(float)ph;
    const double nobs = (double)(c->n * c->m - c->info.nnan);     // sum(.!isnan.(X)) (:697)
    const double nparam = (double)(c->n * k) + (double)(k * c->m);  // (:698)
    if (phi) *phi = ph;
    if (aic) *aic = 2.0 * nparam + nobs * std::log(ph / nobs);  // (:708)
    return NMFK_OK;
}

// post-solve part of execute_run for one batch (NMFkExecute.jl:545-711 with the default keywords)
static int32_t finish_run(nmfk_batch* b, int32_t clusterW, std::vector<char>& Wb, std::vector<char>& Hb, double* phi,
                          double* robustness, double* aic, int64_t* total_iters) {
    nmfk_ctx* c = b->ctx;
    const int k = b->k, R = b->R;
    std::vector<int32_t> order((size_t)R), labels((size_t)k * R);
    double rob = 1.0;
    int32_t rc = nmfk_batch_cluster(b, clusterW, order.data(), labels.data(), nullptr, nullptr, &rob, nullptr, nullptr);
    if (rc) return rc;
    const int best = order[0];
    std::vector<char> W0, H0;
    rc = fetch_factors(b, best, W0, H0);
    if (rc) return rc;
    const size_t es = esize(c->dtype);
    Wb = W0;
    Hb = H0;
    if (k > 1) {  // Wbest[:, i] = WBig[bestIdx][:, ci[i]]; Hbest[i, :] = HBig[bestIdx][ci[i], :] (:631-635)
        for (int i = 0; i < k; ++i) {
            const int ci = labels[(size_t)i] - 1;
            std::memcpy(Wb.data() + (size_t)i * c->n * es, W0.data() + (size_t)ci * c->n * es, (size_t)c->n * es);
            for (int64_t j = 0; j < c->m; ++j)
                std::memcpy(Hb.data() + ((size_t)i + (size_t)j * k) * es, H0.data() + ((size_t)ci + (size_t)j * k) * es, es);
        }
    }
    rc = phi_aic(c, k, Wb, Hb, phi, aic);
    if (rc) return rc;
    if (robustness) *robustness = rob;
    if (total_iters) {
        std::vector<UnitState> st;
        rc = fetch_state(b, st);
        if (rc) return rc;
        int64_t s = 0;
        for (auto& u : st) s += u.it;
        *total_iters = s;
    }
    return NMFK_OK;
}

int32_t nmfk_execute_run(nmfk_ctx* c, int32_t k, int32_t R, const void* Winit, const void* Hinit, uint64_t seed0,
                         const nmfk_params* p, void* W_best, void* H_best, double* phi, double* robustness, double* aic,
                         int64_t* total_iters) {
    if (!c || !p) return fail(c, NMFK_E_INVALID, "nmfk_execute_run: NULL argument");
    const bool timing = getenv("NMFK_TILED_TIMING") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    auto ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
    nmfk_batch* b = nullptr;
    int32_t rc = nmfk_batch_create(c, k, R, &b);
    if (rc) return rc;
    const double t_create = ms();
    rc = nmfk_batch_set_init_partial(b, Winit, Hinit, seed0);  // either may be NULL (NMFkMultiplicative.jl:37-55)
    const double t_init = ms();
    if (!rc) rc = nmfk_solve(c, &b, 1, p);
    const double t_solve = ms();
    std::vector<char> Wb, Hb;
    if (!rc) rc = finish_run(b, p->clusterWmatrix != 0, Wb, Hb, phi, robustness, aic, total_iters);
    const double t_finish = ms();
    if (!rc) {
        if (W_best) std::memcpy(W_best, Wb.data(), Wb.size());
        if (H_best) std::memcpy(H_best, Hb.data(), Hb.size());
    }
    nmfk_batch_destroy(b);
    if (timing)
        fprintf(stderr, "[nmfk timing] execute_run host wall clock: create %.1f, init %.1f, solve %.1f, cluster + select + scores %.1f, destroy %.1f ms\n",
                t_create, t_init - t_create, t_solve - t_init, t_finish - t_solve, ms() - t_finish);
    return rc;
}

// signal ordering of execute(X, nk) (NMFkExecute.jl:311-318; skipped with Wfixed / Hfixed, :305-307) + copy to the caller
static void order_and_store(nmfk_ctx* c, int k, const nmfk_params* p, const std::vector<char>& Wb, const std::vector<char>& Hb,
                            void* W_out, void* H_out) {
    const size_t es = esize(c->dtype);
    std::vector<int32_t> so((size_t)k);
    std::iota(so.begin(), so.end(), 0);
    if (!p->Wfixed && !p->Hfixed) nmfk_signalorder(Wb.data(), Hb.data(), c->n, k, c->m, c->dtype, so.data());
    if (W_out)
        for (int a = 0; a < k; ++a)
            std::memcpy((char*)W_out + (size_t)a * c->n * es, Wb.data() + (size_t)so[a] * c->n * es, (size_t)c->n * es);
    if (H_out)
        for (int a = 0; a < k; ++a)
            for (int64_t j = 0; j < c->m; ++j)
                std::memcpy((char*)H_out + ((size_t)a + (size_t)j * k) * es, Hb.data() + ((size_t)so[a] + (size_t)j * k) * es, es);
}

// consecutive groups of the sweep's k values whose factor stacks stay within a fixed budget (a constant, so that every
// rank of a sharded sweep forms the same groups): BASELINE C4 on one GPU would otherwise hold 108 GB of W stacks at once
static std::vector<std::pair<int, int>> k_groups(const nmfk_ctx* c, const int32_t* ks, int nks, int R) {
    const double budget = 48.0 * 1073741824.0;
    const double es = (double)esize(c->dtype);
    std::vector<std::pair<int, int>> groups;
    int begin = 0;
    double used = 0.0;
    for (int i = 0; i < nks; ++i) {
        const double bytes = ((double)c->n * ks[i] + (double)ks[i] * c->m) * R * es +
                             (c->info.nnan > 0 ? (double)R * c->n * c->m * es : 0.0);
        if (i > begin && used + bytes > budget) {
            groups.emplace_back(begin, i);
            begin = i;
            used = 0.0;
        }
        used += bytes;
    }
    groups.emplace_back(begin, nks);
    return groups;
}

static int32_t kopt_of(const int32_t* ks, int nks, const std::vector<double>& fit, const std::vector<double>& rob, double cutoff) {
    bool allinf = true;
    for (double f : fit)
        if (!std::isinf(f)) allinf = false;
    return allinf ? 0 : nmfk_getk(ks, rob.data(), nks, cutoff, 1);  // (:206-208, :225)
}

int32_t nmfk_execute(nmfk_ctx* c, const int32_t* ks, int32_t nks, int32_t R, const void* const* Winit,
                     const void* const* Hinit, uint64_t seed0, const nmfk_params* p, double cutoff, void* const* W_out,
                     void* const* H_out, double* fitquality, double* robustness, double* aic, int32_t* kopt,
                     int64_t* total_iters) {
    if (!c || !ks || !p || nks < 1 || R < 1) return fail(c, NMFK_E_INVALID, "nmfk_execute: bad arguments");
    if (!c->has_X) return fail(c, NMFK_E_NO_X, "nmfk_set_X has not been called");
    int32_t rc = NMFK_OK;
    int64_t tot = 0;
    double solve_ms = 0.0;
    std::vector<double> rob((size_t)nks, 0.0), fit((size_t)nks, 0.0);
    for (const auto& g : k_groups(c, ks, nks, R)) {
        const int gn = g.second - g.first;
        std::vector<nmfk_batch*> bs((size_t)gn, nullptr);
        for (int q = 0; q < gn && !rc; ++q) {
            const int i = g.first + q;
            rc = nmfk_batch_create(c, ks[i], R, &bs[q]);
            if (!rc) rc = nmfk_batch_set_init_partial(bs[q], Winit ? Winit[i] : nullptr, Hinit ? Hinit[i] : nullptr, seed0);
        }
        if (!rc) rc = nmfk_solve(c, bs.data(), gn, p);
        solve_ms += c->last_solve_ms;
        for (int q = 0; q < gn && !rc; ++q) {
            const int i = g.first + q;
            std::vector<char> Wb, Hb;
            double ph = 0, rb = 0, ai = 0;
            int64_t it = 0;
            rc = finish_run(bs[q], p->clusterWmatrix != 0, Wb, Hb, &ph, &rb, &ai, &it);
            if (rc) break;
            tot += it;
            order_and_store(c, ks[i], p, Wb, Hb, W_out ? W_out[i] : nullptr, H_out ? H_out[i] : nullptr);
            rob[i] = rb;
            fit[i] = ph;  // execute re-derives fit = normnan(X - W*H) from the returned factors (:212-222)
            if (fitquality) fitquality[i] = ph;
            if (robustness) robustness[i] = rb;
            if (aic) aic[i] = ai;
        }
        for (auto b : bs) nmfk_batch_destroy(b);
        if (rc) return rc;
    }
    c->last_solve_ms = solve_ms;
    if (kopt) *kopt = kopt_of(ks, nks, fit, rob, cutoff);
    if (total_iters) *total_iters = tot;
    return NMFK_OK;
}

#define NC(ctx, call)                                                                                           \
    do {                                                                                                        \
        ncclResult_t r__ = (call);                                                                              \
        if (r__ != ncclSuccess) return fail((ctx), NMFK_E_UNSUPPORTED, std::string(#call) + ": " + g_nccl.getErrorString(r__)); \
    } while (0)

// execute(X, nkrange, nNMF = nranks * R_local) with the restarts sharded over the ranks of the sweep communicator: the
// reference's `pmap` over restarts (NMFkExecute.jl:511-526).  No collective inside the iteration loop; per k one
// all-gather of the H stacks (k x m per restart) and of the 64-byte restart states, one broadcast of the best restart's W
// (n x k) from the rank that solved it; the clustering + silhouettes of the nranks * R_local solutions of a given k run on
// rank (k index mod nranks) and the robustness values are summed into place at the end.  Every rank returns everything.
int32_t nmfk_sweep(nmfk_ctx* c, const int32_t* ks, int32_t nks, int32_t R_local, const void* const* Winit,
                   const void* const* Hinit, uint64_t seed0, const nmfk_params* p, double cutoff, void* const* W_out,
                   void* const* H_out, double* fitquality, double* robustness, double* aic, int32_t* kopt, int64_t* total_iters,
                   int64_t* total_iters_local) {
    if (!c || !ks || !p || nks < 1 || R_local < 1) return fail(c, NMFK_E_INVALID, "nmfk_sweep: bad arguments");
    if (!c->has_X) return fail(c, NMFK_E_NO_X, "nmfk_set_X has not been called");
    const int world = c->sweep_nranks, rank = c->sweep_rank;
    if (world == 1) {
        int32_t rc = nmfk_execute(c, ks, nks, R_local, Winit, Hinit, seed0, p, cutoff, W_out, H_out, fitquality, robustness, aic,
                                  kopt, total_iters);
        if (!rc && total_iters_local && total_iters) *total_iters_local = *total_iters;
        return rc;
    }
    if (c->sharded) return fail(c, NMFK_E_UNSUPPORTED, "nmfk_sweep: the ctx is row-sharded");
    if (p->clusterWmatrix)
        return fail(c, NMFK_E_UNSUPPORTED, "nmfk_sweep: clusterWmatrix would gather the W stacks (n x k per restart) - not available "
                                           "across ranks");
    CU(c, cudaSetDevice(c->device));
    ncclComm_t comm = static_cast<ncclComm_t>(c->sweep_comm);
    const int R_total = world * R_local;
    const size_t es = esize(c->dtype);
    const ncclDataType_t nt = c->dtype == NMFK_F64 ? ncclDouble : ncclFloat;
    int32_t rc = NMFK_OK;
    int64_t tot_local = 0, tot_global = 0;
    double solve_ms = 0.0;
    std::vector<double> rob((size_t)nks, 0.0), fit((size_t)nks, 0.0);
    struct Guard {  // batches of the current group, destroyed on every exit path
        std::vector<nmfk_batch*> v;
        ~Guard() {
            for (auto b : v) nmfk_batch_destroy(b);
        }
    };
    for (const auto& g : k_groups(c, ks, nks, R_total)) {
        const int gn = g.second - g.first;
        Guard bs, hs;
        bs.v.assign((size_t)gn, nullptr);
        hs.v.assign((size_t)gn, nullptr);
        for (int q = 0; q < gn; ++q) {
            const int i = g.first + q;
            rc = nmfk_batch_create(c, ks[i], R_local, &bs.v[q]);
            if (!rc) rc = nmfk_batch_set_init_partial(bs.v[q], Winit ? Winit[i] : nullptr, Hinit ? Hinit[i] : nullptr,
                                                      seed0 + (uint64_t)rank * (uint64_t)R_local);
            if (!rc) rc = nmfk_batch_create_hstack(c, ks[i], R_total, &hs.v[q]);
            if (rc) return rc;
        }
        rc = nmfk_solve(c, bs.v.data(), gn, p);
        if (rc) return rc;
        solve_ms += c->last_solve_ms;
        // phase 1: everything the robustness analysis needs crosses NVLink once per k
        for (int q = 0; q < gn; ++q) {
            nmfk_batch *b = bs.v[q], *h = hs.v[q];
            const int k = b->k;
            NC(c, g_nccl.allGather(b->H, h->H, (size_t)k * c->m * R_local, nt, comm, c->stream));
            NC(c, g_nccl.allGather(b->st, h->st, (size_t)R_local * sizeof(UnitState), ncclUint8, comm, c->stream));
            h->inited = true;
        }
        CU(c, cudaStreamSynchronize(c->stream));
        // phase 2: best restart of every k (every rank sorts the same gathered objectives), its W from the rank that solved it
        DevBuf wtmp;
        for (int q = 0; q < gn; ++q) {
            const int i = g.first + q;
            nmfk_batch *b = bs.v[q], *h = hs.v[q];
            const int k = b->k;
            std::vector<UnitState> st;
            rc = fetch_state(h, st);
            if (rc) return rc;
            for (int r = 0; r < R_total; ++r) {
                tot_global += st[r].it;
                if (r / R_local == rank) tot_local += st[r].it;
            }
            std::vector<double> obj;
            std::vector<int32_t> order;
            sorted_order(c, st, obj, order);
            const int gbest = order[0], br = gbest / R_local, bl = gbest % R_local;
            const size_t wb = (size_t)c->n * k * es, hb = (size_t)k * c->m * es;
            if (wtmp.p) {
                dev_free(wtmp.p);
                wtmp.p = nullptr;
            }
            CU(c, wtmp.alloc(wb));
            char* wsrc = (char*)b->W + (size_t)bl * wb;
            if (k > 1) {  // nanaction = :zeroed before Wbest / Hbest are re-read (:566-580, :631-635)
                if (rank == br) CU(c, launch_zero_nan(wsrc, (long long)c->n * k, c->dtype, c->stream));
                CU(c, launch_zero_nan(h->H, (long long)k * c->m * R_total, c->dtype, c->stream));
                c->launches += 1 + (rank == br);
            }
            NC(c, g_nccl.broadcast(rank == br ? (const void*)wsrc : (const void*)wtmp.p, wtmp.p, (size_t)c->n * k, nt, br, comm,
                                   c->stream));
            std::vector<char> Wb(wb), Hb(hb);
            CU(c, cudaMemcpyAsync(Wb.data(), wtmp.p, wb, cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaMemcpyAsync(Hb.data(), (const char*)h->H + (size_t)gbest * hb, hb, cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
            // labels[:, 1] = 1:k by construction (NMFkCluster.jl:461), so the reordering of :631-635 is the identity
            double ph = 0, ai = 0;
            rc = phi_aic(c, k, Wb, Hb, &ph, &ai);
            if (rc) return rc;
            order_and_store(c, k, p, Wb, Hb, W_out ? W_out[i] : nullptr, H_out ? H_out[i] : nullptr);
            fit[i] = ph;
            if (fitquality) fitquality[i] = ph;
            if (aic) aic[i] = ai;
        }
        // phase 3: clustering + silhouettes of the R_total solutions, one owner per k, no communication
        for (int q = 0; q < gn; ++q) {
            const int i = g.first + q;
            if (i % world != rank) continue;
            double rb = 1.0;
            rc = nmfk_batch_cluster(hs.v[q], 0, nullptr, nullptr, nullptr, nullptr, &rb, nullptr, nullptr);
            if (rc) return rc;
            rob[i] = rb;
        }
    }
    {  // robustness of every k to every rank: the owners hold the values, the others zero
        DevBuf d;
        CU(c, d.alloc((size_t)nks * sizeof(double)));
        CU(c, cudaMemcpyAsync(d.p, rob.data(), (size_t)nks * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        NC(c, g_nccl.allReduce(d.p, d.p, (size_t)nks, ncclDouble, ncclSum, comm, c->stream));
        CU(c, cudaMemcpyAsync(rob.data(), d.p, (size_t)nks * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    c->last_solve_ms = solve_ms;
    if (robustness) std::copy(rob.begin(), rob.end(), robustness);
    if (kopt) *kopt = kopt_of(ks, nks, fit, rob, cutoff);
    if (total_iters) *total_iters = tot_global;
    if (total_iters_local) *total_iters_local = tot_local;
    return NMFK_OK;
}

int64_t nmfk_launch_count(const nmfk_ctx* c) { return c ? c->launches : 0; }

int32_t nmfk_profile_enable(nmfk_ctx* c, int32_t on) {
    if (!c) return fail(nullptr, NMFK_E_INVALID, "ctx is NULL");
    c->prof.enabled = on != 0;
    c->prof.reset();
    return NMFK_OK;
}

int32_t nmfk_profile_get(const nmfk_ctx* c, double* pass_ms, int64_t* pass_launches) {
    if (!c) return fail(nullptr, NMFK_E_INVALID, "ctx is NULL");
    if (pass_ms) *pass_ms = c->prof.ms;
    if (pass_launches) *pass_launches = c->prof.launches;
    return NMFK_OK;
}

double nmfk_last_solve_ms(const nmfk_ctx* c) { return c ? c->last_solve_ms : 0.0; }

int32_t nmfk_measure_peak(nmfk_ctx* c, int32_t which, double* value) {
    if (!c || !value) return fail(c, NMFK_E_INVALID, "nmfk_measure_peak: NULL argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, measure_peak(which, value, c->stream));
    return NMFK_OK;
}

// robustkmeans(X, k, repeats; ...) (NMFkCluster.jl:172-246): the repeats run concurrently on the device, the host keeps the
// first repeat with the smallest total cost (:219-225), computes its silhouettes and applies sortclustering (:264-289).
int32_t nmfk_robustkmeans(nmfk_ctx* c, const double* X, int32_t d, int32_t N, int32_t k, int32_t repeats, const int32_t* seeds,
                          int32_t maxiter, double tol, int32_t compute_silhouettes, int32_t* assignments, double* centers, double* costs,
                          int32_t* counts, double* totalcost, int32_t* iterations, int32_t* converged, double* best_silhouettes,
                          int32_t* best_repeat, int32_t* empty_cluster_repeats) {
    if (!c || !X || !seeds || d < 1 || N < 1 || k < 1 || repeats < 1 || maxiter < 0)
        return fail(c, NMFK_E_INVALID, "nmfk_robustkmeans: bad arguments");
    if (k >= N) return fail(c, NMFK_E_INVALID, "nmfk_robustkmeans: k must be smaller than the number of points (NMFkCluster.jl:139-142)");
    for (long long e = 0; e < (long long)k * repeats; ++e)
        if (seeds[e] < 0 || seeds[e] >= N) return fail(c, NMFK_E_INVALID, "nmfk_robustkmeans: seed index out of range");
    CU(c, cudaSetDevice(c->device));
    DevBuf dX, dxn, dseeds, dassign, dcosts, dcounts, dcent, dtc, dit, dfl;
    CU(c, dX.alloc((size_t)d * N * 8));
    CU(c, dxn.alloc((size_t)N * 8));
    CU(c, dseeds.alloc((size_t)k * repeats * 4));
    CU(c, dassign.alloc((size_t)repeats * N * 4));
    CU(c, dcosts.alloc((size_t)repeats * N * 8));
    CU(c, dcounts.alloc((size_t)repeats * k * 4));
    CU(c, dcent.alloc((size_t)repeats * d * k * 8));
    CU(c, dtc.alloc((size_t)repeats * 8));
    CU(c, dit.alloc((size_t)repeats * 4));
    CU(c, dfl.alloc((size_t)repeats * 4));
    CU(c, cudaMemcpyAsync(dX.p, X, (size_t)d * N * 8, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(dseeds.p, seeds, (size_t)k * repeats * 4, cudaMemcpyHostToDevice, c->stream));
    CU(c, launch_kmeans(dX.as<double>(), dxn.as<double>(), d, N, k, repeats, dseeds.as<int>(), maxiter, tol, dassign.as<int>(),
                        dcosts.as<double>(), dcounts.as<int>(), dcent.as<double>(), dtc.as<double>(), dit.as<int>(), dfl.as<int>(),
                        c->stream));
    c->launches += 2;
    std::vector<double> tc((size_t)repeats);
    std::vector<int32_t> its((size_t)repeats), fl((size_t)repeats);
    CU(c, cudaMemcpyAsync(tc.data(), dtc.p, (size_t)repeats * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(its.data(), dit.p, (size_t)repeats * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(fl.data(), dfl.p, (size_t)repeats * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    int best = 0, nempty = 0;
    for (int i = 0; i < repeats; ++i) {  // `if i == 1 || c_new.totalcost < best_totalcost` (:219)
        if (i > 0 && tc[i] < tc[best]) best = i;
        nempty += (fl[i] >> 1) & 1;
    }
    std::vector<int32_t> as((size_t)N), cnt((size_t)k);
    std::vector<double> cst((size_t)N), cen((size_t)d * k), sil((size_t)N, 0.0);
    CU(c, cudaMemcpyAsync(as.data(), dassign.as<int>() + (size_t)best * N, (size_t)N * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(cst.data(), dcosts.as<double>() + (size_t)best * N, (size_t)N * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(cnt.data(), dcounts.as<int>() + (size_t)best * k, (size_t)k * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(cen.data(), dcent.as<double>() + (size_t)best * d * k, (size_t)d * k * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (compute_silhouettes && best_silhouettes) {
        int maxa = 0;
        for (int v : as) maxa = std::max(maxa, v);
        if (maxa > 1) {  // `if maximum(c_new.assignments) > 1` (:208-214); otherwise the silhouettes stay zero
            // Xn = zerostoepsilon(X); Xd = pairwise(CosineDist(), Xn; dims=2); silhouettes(c_new, Xd)
            const int ld = d + 1;
            DevBuf dV, dvn, dD, dsil;
            CU(c, dV.alloc((size_t)N * ld * 8));
            CU(c, dvn.alloc((size_t)N * 8));
            CU(c, dD.alloc((size_t)N * N * 8));
            CU(c, dsil.alloc((size_t)N * 8));
            CU(c, cudaMemcpy2DAsync(dV.p, (size_t)ld * 8, dX.p, (size_t)d * 8, (size_t)d * 8, (size_t)N, cudaMemcpyDeviceToDevice, c->stream));
            const double eps = 2.220446049250313e-16;
            CU(c, launch_point_silhouettes(dV.as<double>(), d, ld, N, k, dassign.as<int>() + (size_t)best * N, eps * eps, dvn.as<double>(),
                                           dD.as<double>(), dsil.as<double>(), c->stream));
            c->launches += 3;
            CU(c, cudaMemcpyAsync(sil.data(), dsil.p, (size_t)N * 8, cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
        }
        std::copy(sil.begin(), sil.end(), best_silhouettes);
    }
    // sortclustering(c::KmeansResult) (:264-289): clusters relabelled by first appearance, then ranked by size (stable, descending)
    std::vector<int> first;  // j = unique(c.assignments)
    std::vector<int> pos((size_t)k + 1, -1);
    for (int v : as)
        if (pos[v] < 0) {
            pos[v] = (int)first.size();
            first.push_back(v);
        }
    std::vector<int> rank(first.size());
    std::iota(rank.begin(), rank.end(), 0);
    std::stable_sort(rank.begin(), rank.end(), [&](int x, int y) { return cnt[first[x] - 1] > cnt[first[y] - 1]; });
    std::vector<int> newlabel(first.size());
    for (size_t q = 0; q < rank.size(); ++q) newlabel[rank[q]] = (int)q + 1;
    if (assignments)
        for (int j = 0; j < N; ++j) assignments[j] = newlabel[pos[as[j]]];
    // centers[:, r], counts[r] with r = j[i]: only the clusters that appear (the reference drops empty ones here)
    if (counts) std::fill(counts, counts + k, 0);
    if (centers) std::fill(centers, centers + (size_t)d * k, 0.0);
    for (size_t q = 0; q < rank.size(); ++q) {
        const int old = first[rank[q]] - 1;
        if (counts) counts[q] = cnt[old];
        if (centers) std::copy(cen.begin() + (size_t)old * d, cen.begin() + (size_t)(old + 1) * d, centers + q * d);
    }
    if (costs) std::copy(cst.begin(), cst.end(), costs);
    if (totalcost) *totalcost = tc[best];
    if (iterations) *iterations = its[best];
    if (converged) *converged = fl[best] & 1;
    if (best_repeat) *best_repeat = best;
    if (empty_cluster_repeats) *empty_cluster_repeats = nempty;
    return NMFK_OK;
}

// The stacked-restart GEMM of Variant FRO on its own (test / measurement hook): C[M x N] = A[M x K] B[N x K]^T, row-major host
// buffers; Float32 = tcgen05 kind::tf32 with the 3-term split (TMA tensor maps), Float64 = DMMA.  *ms = average device time of
// `reps` launches (CUDA events on the ctx stream).
int32_t nmfk_gemm_nt(nmfk_ctx* c, int32_t dtype, const void* A, const void* B, int32_t M, int32_t N, int32_t K, void* Cout,
                     int32_t reps, double* ms) {
    if (!c || !A || !B || !Cout || M < 1 || N < 1 || K < 1 || reps < 1) return fail(c, NMFK_E_INVALID, "nmfk_gemm_nt: bad arguments");
    if (dtype != NMFK_F32 && dtype != NMFK_F64) return fail(c, NMFK_E_INVALID, "nmfk_gemm_nt: bad dtype");
    if (dtype == NMFK_F32 && !fro_gemm_supported(N, K)) return fail(c, NMFK_E_UNSUPPORTED, "nmfk_gemm_nt (Float32): N and K must be multiples of 4");
    CU(c, cudaSetDevice(c->device));
    const size_t es = esize(dtype);
    DevBuf dA, dB, dC, dAlo, dBlo, derr;
    CU(c, dA.alloc((size_t)M * K * es));
    CU(c, dB.alloc((size_t)N * K * es));
    const int S = dtype == NMFK_F32 ? fro_gemm_slices(M, N, K) : 1;  // split-K partial products side by side, summed in order
    CU(c, dC.alloc((size_t)S * M * N * es));
    CU(c, derr.alloc(sizeof(int)));
    CU(c, cudaMemsetAsync(derr.p, 0, sizeof(int), c->stream));
    CU(c, cudaMemcpyAsync(dA.p, A, (size_t)M * K * es, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaMemcpyAsync(dB.p, B, (size_t)N * K * es, cudaMemcpyHostToDevice, c->stream));
    if (dtype == NMFK_F32) {
        CU(c, dAlo.alloc((size_t)M * K * es));
        CU(c, dBlo.alloc((size_t)N * K * es));
        CU(c, launch_split_lo(dA.as<float>(), dAlo.as<float>(), (long long)M * K, c->stream));
        CU(c, launch_split_lo(dB.as<float>(), dBlo.as<float>(), (long long)N * K, c->stream));
    }
    auto launch = [&]() -> cudaError_t {
        if (dtype == NMFK_F32) {
            cudaError_t e = launch_fro_gemm(dA.as<float>(), dAlo.as<float>(), K, dB.as<float>(), dBlo.as<float>(), K, dC.as<float>(), N, M, N,
                                            K, S, (long long)M * N, derr.as<int>(), c->stream);
            return e != cudaSuccess ? e : launch_sum_slices(dC.as<float>(), S, (long long)M * N, (long long)M * N, c->stream);
        }
        return launch_fro_gemm_f64(dA.as<double>(), K, dB.as<double>(), K, dC.as<double>(), N, M, N, K, c->stream);
    };
    CU(c, launch());  // warm-up (and the launch whose result is returned when reps == 1)
    CU(c, cudaEventRecord(c->ev0, c->stream));
    for (int i = 0; i < reps; ++i) CU(c, launch());
    CU(c, cudaEventRecord(c->ev1, c->stream));
    CU(c, cudaEventSynchronize(c->ev1));
    float t = 0.f;
    CU(c, cudaEventElapsedTime(&t, c->ev0, c->ev1));
    c->launches += reps + 1;
    if (ms) *ms = (double)t / reps;
    int herr = 0;
    CU(c, cudaMemcpy(&herr, derr.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (herr) return fail(c, NMFK_E_INVALID, "nmfk_gemm_nt: barrier time-out inside fro_gemm_kernel (site " + std::to_string(herr) + ")");
    CU(c, cudaMemcpy(Cout, dC.p, (size_t)M * N * es, cudaMemcpyDeviceToHost));
    return NMFK_OK;
}

// tcgen05 / tensor-memory building blocks of the Float32 tiled engine, checked on the device (tc_selftest.cu)
int32_t nmfk_umma_selftest(nmfk_ctx* c, const float* U, const float* V, int32_t mode, float* Pss, float* Pts, float* ACCa,
                           float* ACCb, int32_t* err) {
    if (!c || !U || !V || !Pss || !Pts || !ACCa || !ACCb || !err) return fail(c, NMFK_E_INVALID, "nmfk_umma_selftest: NULL argument");
    CU(c, cudaSetDevice(c->device));
    int e = 0;
    CU(c, umma_selftest(U, V, mode, Pss, Pts, ACCa, ACCb, &e, c->stream));
    *err = e;
    return NMFK_OK;
}

int32_t nmfk_umma_timing(nmfk_ctx* c, const float* U, const float* V, int32_t reps, int64_t* cycles8, float* acc) {
    if (!c || !U || !V || !cycles8 || !acc) return fail(c, NMFK_E_INVALID, "nmfk_umma_timing: NULL argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, umma_timing(U, V, reps, reinterpret_cast<long long*>(cycles8), acc, c->stream));
    return NMFK_OK;
}

// host-side Philox stream (tests: bit-compatibility with numpy without a GPU)
int32_t nmfk_philox_host(uint64_t seed, int64_t count, double* out) {
    if (!out || count < 0) return NMFK_E_INVALID;
    for (int64_t b = 0; b * 4 < count; ++b) {
        uint64_t o[4];
        philox4x64_10((uint64_t)b + 1, seed, o);
        for (int q = 0; q < 4 && b * 4 + q < count; ++q) out[b * 4 + q] = philox_to_double(o[q]);
    }
    return NMFK_OK;
}

