// K1: preprocessing of X, replaces NMFpreprocessing! (/root/reference/src/NMFkMultiplicative.jl:3-22)
// plus the device-side U(0,1) initialisation streams (rand(n,k), rand(k,m) of :38,:48).
//
// One pass over the raw X (HBM-bound, coalesced 32x32 tiles through shared memory) produces
//   Xp  (n x m, column-major): entries <= 0 replaced by lambda, NaN kept (the solver substitutes
//        lambda / the imputed value itself, so the caller's X never has to be mutated+restored),
//   Xpt (m x n, column-major): its transpose, so that BOTH half-updates read X with consecutive
//        lanes on consecutive addresses,
// and the statistics the reference derives from X: count of NaN, of entries <= 0, of negative
// entries (-> the "must be nonnegative" error), all-zero rows / columns (-> its warnings).
#include <algorithm>

#include "nmfk_internal.h"
#include "philox.h"

namespace nmfk {

template <typename T>
__global__ void preprocess_kernel(const T* __restrict__ X, T* __restrict__ Xp, T* __restrict__ Xpt, long long n,
                                  long long m, T lambda, PreStats* stats, unsigned char* rowflag,
                                  unsigned char* colflag, double* blockmin) {
    __shared__ T tile[32][33];
    __shared__ unsigned int cnt[3];
    __shared__ double wmin[8];
    if (threadIdx.y == 0 && threadIdx.x < 3) cnt[threadIdx.x] = 0;
    __syncthreads();
    const long long i0 = (long long)blockIdx.x * 32, j0 = (long long)blockIdx.y * 32;
    unsigned int cn = 0, cz = 0, cneg = 0;
    double mn = INFINITY;
    // read 32x32 tile: lanes along rows i (contiguous in column-major X)
    for (int jj = threadIdx.y; jj < 32; jj += blockDim.y) {
        const long long i = i0 + threadIdx.x, j = j0 + jj;
        if (i < n && j < m) {
            T x = X[i + j * n];
            const bool isn = (x != x);
            if (isn) {
                ++cn;
                rowflag[i] = 1;  // a NaN makes the row/column sum NaN != 0
                colflag[j] = 1;
            } else {
                if ((double)x < mn) mn = (double)x;
                if (x < (T)0) ++cneg;
                if (x <= (T)0) {
                    ++cz;
                    if (x < (T)0) {  // only all-ZERO rows sum to zero; a negative entry never reaches the solver
                        rowflag[i] = 1;
                        colflag[j] = 1;
                    }
                    x = lambda;  // X[izero] .= lambda (:18-19)
                } else {
                    rowflag[i] = 1;
                    colflag[j] = 1;
                }
            }
            Xp[i + j * n] = x;
            tile[jj][threadIdx.x] = x;
        }
    }
    __syncthreads();
    // write the transposed tile: lanes along j (contiguous in Xpt, which is m x n column-major)
    for (int ii = threadIdx.y; ii < 32; ii += blockDim.y) {
        const long long i = i0 + ii, j = j0 + threadIdx.x;
        if (i < n && j < m) Xpt[j + i * m] = tile[threadIdx.x][ii];
    }
    // statistics
    for (int o = 16; o > 0; o >>= 1) {
        cn += __shfl_xor_sync(0xffffffffu, cn, o);
        cz += __shfl_xor_sync(0xffffffffu, cz, o);
        cneg += __shfl_xor_sync(0xffffffffu, cneg, o);
        const double other = __shfl_xor_sync(0xffffffffu, mn, o);
        mn = other < mn ? other : mn;
    }
    if (threadIdx.x == 0) {
        atomicAdd(&cnt[0], cn);
        atomicAdd(&cnt[1], cz);
        atomicAdd(&cnt[2], cneg);
        wmin[threadIdx.y] = mn;
    }
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        if (cnt[0]) atomicAdd(&stats->nnan, (unsigned long long)cnt[0]);
        if (cnt[1]) atomicAdd(&stats->nzero, (unsigned long long)cnt[1]);
        if (cnt[2]) atomicAdd(&stats->nneg, (unsigned long long)cnt[2]);
        double b = wmin[0];
        for (int w = 1; w < (int)blockDim.y; ++w) b = wmin[w] < b ? wmin[w] : b;
        blockmin[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = b;
    }
}

__global__ void count_unset_kernel(const unsigned char* flags, long long len, unsigned long long* out) {
    unsigned long long c = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < len; i += (long long)gridDim.x * blockDim.x)
        c += flags[i] ? 0 : 1;
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

cudaError_t launch_preprocess(const void* Xraw, void* Xp, void* Xpt, int64_t n, int64_t m, int dtype, double lambda,
                              PreStats* d_stats, unsigned char* d_rowflag, unsigned char* d_colflag, double* d_blockmin,
                              int nblockmin, cudaStream_t s) {
    cudaError_t e;
    if ((e = cudaMemsetAsync(d_stats, 0, sizeof(PreStats), s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_rowflag, 0, (size_t)n, s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_colflag, 0, (size_t)m, s)) != cudaSuccess) return e;
    dim3 grid((unsigned)((n + 31) / 32), (unsigned)((m + 31) / 32)), block(32, 8);
    if ((long long)grid.x * grid.y > nblockmin) return cudaErrorInvalidValue;
    if (dtype == 1)
        preprocess_kernel<double><<<grid, block, 0, s>>>((const double*)Xraw, (double*)Xp, (double*)Xpt, n, m, lambda,
                                                         d_stats, d_rowflag, d_colflag, d_blockmin);
    else
        preprocess_kernel<float><<<grid, block, 0, s>>>((const float*)Xraw, (float*)Xp, (float*)Xpt, n, m,
                                                        (float)lambda, d_stats, d_rowflag, d_colflag, d_blockmin);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    count_unset_kernel<<<148, 256, 0, s>>>(d_rowflag, n, &d_stats->zero_rows);
    count_unset_kernel<<<148, 256, 0, s>>>(d_colflag, m, &d_stats->zero_cols);
    return cudaGetLastError();
}

// ---- Philox4x64-10 U(0,1) initialisation ------------------------------------------------------
// stream element e of restart r = numpy.random.Generator(Philox(key=seed0+r+1)).random(...)[e];
// the first n*k elements fill W (column-major), the next k*m fill H: W is drawn before H.
// Row-sharded X: the stream is that of the GLOBAL n x k matrix; this rank keeps rows [row0, row0 + nloc).
// W == nullptr or H == nullptr: only the other factor is drawn, from the START of the stream (the reference draws W only when
// Winit is empty and then H only when Hinit is empty, NMFkMultiplicative.jl:37-55).
template <typename T>
__global__ void philox_init_kernel(T* __restrict__ W, T* __restrict__ H, long long n, long long row0, long long nloc,
                                   int k, long long km, int R, unsigned long long seed0) {
    const long long nk = W != nullptr ? n * k : 0;
    const long long per = nk + (H != nullptr ? km : 0);
    const long long blocks4 = (per + 3) / 4;
    const long long total = blocks4 * R;
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total;
         g += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(g / blocks4);
        const long long b = g - (long long)r * blocks4;
        uint64_t out[4];
        philox4x64_10(b + 1, seed0 + (unsigned long long)r + 1ull, out);  // numpy bumps the counter before generating
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const long long e = b * 4 + q;
            if (e >= per) break;
            const double u = philox_to_double(out[q]);
            if (e < nk) {
                const long long i = e % n - row0, c = e / n;
                if (i >= 0 && i < nloc) W[(long long)r * nloc * k + i + c * nloc] = (T)u;
            } else
                H[(long long)r * km + (e - nk)] = (T)u;
        }
    }
}

cudaError_t launch_philox_init(void* W, void* H, int64_t n, int64_t row0, int64_t nloc, int k, int64_t m, int R,
                               uint64_t seed0, int dtype, cudaStream_t s) {
    if (W == nullptr && H == nullptr) return cudaSuccess;
    const long long nk = W != nullptr ? n * k : 0, km = (long long)k * m;
    const long long total = ((nk + (H != nullptr ? km : 0) + 3) / 4) * R;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    if (dtype == 1)
        philox_init_kernel<double><<<blocks, 256, 0, s>>>((double*)W, (double*)H, n, row0, nloc, k, km, R, seed0);
    else
        philox_init_kernel<float><<<blocks, 256, 0, s>>>((float*)W, (float*)H, n, row0, nloc, k, km, R, seed0);
    return cudaGetLastError();
}

// ---- normalizevector (NMFkMultiplicative.jl:27-31): Xn = Xp ./ nv (rows), and its transpose -----------------------
template <typename T>
__global__ void rownormalize_kernel(const T* __restrict__ Xp, T* __restrict__ Xn, T* __restrict__ Xnt, long long n,
                                    long long m, const T* __restrict__ nv) {
    __shared__ T tile[32][33];
    const long long i0 = (long long)blockIdx.x * 32, j0 = (long long)blockIdx.y * 32;
    for (int jj = threadIdx.y; jj < 32; jj += blockDim.y) {
        const long long i = i0 + threadIdx.x, j = j0 + jj;
        if (i < n && j < m) {
            const T x = Xp[i + j * n] / nv[i];
            Xn[i + j * n] = x;
            tile[jj][threadIdx.x] = x;
        }
    }
    __syncthreads();
    for (int ii = threadIdx.y; ii < 32; ii += blockDim.y) {
        const long long i = i0 + ii, j = j0 + threadIdx.x;
        if (i < n && j < m) Xnt[j + i * m] = tile[threadIdx.x][ii];
    }
}

cudaError_t launch_rownormalize(const void* Xp, void* Xn, void* Xnt, int64_t n, int64_t m, const void* nv, int dtype,
                                cudaStream_t s) {
    dim3 grid((unsigned)((n + 31) / 32), (unsigned)((m + 31) / 32)), block(32, 8);
    if (dtype == 1)
        rownormalize_kernel<double><<<grid, block, 0, s>>>((const double*)Xp, (double*)Xn, (double*)Xnt, n, m, (const double*)nv);
    else
        rownormalize_kernel<float><<<grid, block, 0, s>>>((const float*)Xp, (float*)Xn, (float*)Xnt, n, m, (const float*)nv);
    return cudaGetLastError();
}

// W .*= normalizevector (NMFkMultiplicative.jl:121) for one restart's n x k factor
template <typename T>
__global__ void scale_rows_kernel(T* __restrict__ W, long long n, int k, const T* __restrict__ nv) {
    const long long total = n * k;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x)
        W[e] = W[e] * nv[e % n];
}

cudaError_t launch_scale_rows(void* W, int64_t n, int k, const void* nv, int dtype, cudaStream_t s) {
    int blocks = (int)std::min<long long>((n * k + 255) / 256, 148 * 8);
    if (blocks < 1) blocks = 1;
    if (dtype == 1)
        scale_rows_kernel<double><<<blocks, 256, 0, s>>>((double*)W, n, k, (const double*)nv);
    else
        scale_rows_kernel<float><<<blocks, 256, 0, s>>>((float*)W, n, k, (const float*)nv);
    return cudaGetLastError();
}

// The normalisation of execute_singlerun_compute (NMFkExecute.jl:795-805) for ONE restart, outside the engines (used after
// the normalizevector epilogue): normalize 1: total = sum(H; dims=2); W .*= total'; H ./= total; 2: total = sum(W; dims=1);
// W ./= total; H .*= total'.  One CTA; fixed-order sums in Float64 rounded to T like the engines' finish kernels.
template <typename T>
__global__ void __launch_bounds__(256) renormalize_kernel(T* __restrict__ W, T* __restrict__ H, long long n, long long m, int k,
                                                          int normalize) {
    __shared__ double red[8];
    __shared__ double tot[kTiledMaxK];
    const int tid = threadIdx.x, NT = blockDim.x;
    for (int c = 0; c < k; ++c) {
        double s = 0.0;
        if (normalize == 1)
            for (long long j = tid; j < m; j += NT) s += (double)H[j * k + c];
        else
            for (long long i = tid; i < n; i += NT) s += (double)W[i + (long long)c * n];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if ((tid & 31) == 0) red[tid >> 5] = s;
        __syncthreads();
        if (tid == 0) {
            double a = 0.0;
            for (int w = 0; w < NT / 32; ++w) a += red[w];
            tot[c] = (double)(T)a;
        }
        __syncthreads();
    }
    if (normalize == 1) {
        for (long long e = tid; e < n * k; e += NT) W[e] = W[e] * (T)tot[e / n];
        for (long long e = tid; e < (long long)k * m; e += NT) H[e] = H[e] / (T)tot[e % k];
    } else {
        for (long long e = tid; e < n * k; e += NT) W[e] = W[e] / (T)tot[e / n];
        for (long long e = tid; e < (long long)k * m; e += NT) H[e] = H[e] * (T)tot[e % k];
    }
}

cudaError_t launch_renormalize(void* W, void* H, int64_t n, int64_t m, int k, int normalize, int dtype, cudaStream_t s) {
    if (normalize != 1 && normalize != 2) return cudaSuccess;
    if (dtype == 1)
        renormalize_kernel<double><<<1, 256, 0, s>>>((double*)W, (double*)H, n, m, k, normalize);
    else
        renormalize_kernel<float><<<1, 256, 0, s>>>((float*)W, (float*)H, n, m, k, normalize);
    return cudaGetLastError();
}

// flags[r] = 1 when restart r's W or H holds a NaN (nanaction == :removed, NMFkExecute.jl:581-596)
template <typename T>
__global__ void count_nan_kernel(const T* __restrict__ W, const T* __restrict__ H, long long wlen, long long hlen,
                                 int32_t* __restrict__ flags) {
    const int r = blockIdx.y;
    int found = 0;
    if (W != nullptr) {
        const T* w = W + (long long)r * wlen;
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < wlen; e += (long long)gridDim.x * blockDim.x)
            found |= (w[e] != w[e]);
    }
    const T* h = H + (long long)r * hlen;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < hlen; e += (long long)gridDim.x * blockDim.x)
        found |= (h[e] != h[e]);
    if (__syncthreads_or(found) && threadIdx.x == 0) atomicOr(&flags[r], 1);
}

cudaError_t launch_count_nan(const void* W, const void* H, int64_t wlen, int64_t hlen, int R, int dtype, int32_t* d_flags,
                             cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(d_flags, 0, (size_t)R * sizeof(int32_t), s);
    if (e != cudaSuccess) return e;
    dim3 g((unsigned)std::min<long long>((std::max(wlen, hlen) + 255) / 256, 64), R);
    if (dtype == 1)
        count_nan_kernel<double><<<g, 256, 0, s>>>((const double*)W, (const double*)H, wlen, hlen, d_flags);
    else
        count_nan_kernel<float><<<g, 256, 0, s>>>((const float*)W, (const float*)H, wlen, hlen, d_flags);
    return cudaGetLastError();
}

}  // namespace nmfk
