// K10-K12: robustness of the restart solutions at one k, entirely on the device.
//   clustersolutions  /root/reference/src/NMFkCluster.jl:425-517  (greedy constrained cosine matching)
//   finalize          /root/reference/src/NMFkFinalize.jl:36-79   (pairwise cosine distances + silhouettes)
// Third-party semantics restated: Distances.cosine_dist / pairwise(CosineDist()), Clustering.silhouettes
// (neither package is vendored in the reference tree; see oracle/nmfk_oracle.py for the same restatement).
// Everything is Float64 and deterministic: fixed-order reductions, no floating-point atomics.
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>

#include "fro.h"
#include "nmfk_internal.h"

namespace nmfk {

namespace {

__device__ __forceinline__ double wsum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// nanaction == :zeroed (NMFkExecute.jl:566-580): NaN -> 0 in every stored solution
template <typename T>
__global__ void zero_nan_kernel(T* p, long long len) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < len; i += (long long)gridDim.x * blockDim.x) {
        const T v = p[i];
        if (v != v) p[i] = (T)0;
    }
}

// V[(t*k + a)][:] = vector a of the t-th best solution (row of H, or column of W), as doubles.
// One warp per vector.  Sets *bias when a vector sums to exactly zero (NMFkCluster.jl:437-444).
template <typename T>
__global__ void gather_kernel(const T* __restrict__ F, int len, int k, int R, int use_W, const int* __restrict__ order,
                              double* __restrict__ V, int ld, int* bias) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= R * k) return;
    const int t = warp / k, a = warp - t * k, r = order[t];
    const T* src;
    long long stride;
    if (use_W) {  // W_r[:, a], n x k column-major
        src = F + ((long long)r * k + a) * len;
        stride = 1;
    } else {  // H_r[a, :], k x m column-major
        src = F + (long long)r * k * len + a;
        stride = k;
    }
    double* dst = V + (long long)warp * ld;
    double s = 0.0;
    for (int j = lane; j < len; j += 32) {
        const double v = (double)src[(long long)j * stride];
        dst[j] = v;
        s += v;
    }
    s = wsum(s);
    if (lane == 0 && s == 0.0) atomicOr(bias, 1);
}

// clustersolutions: one CTA walks the R solutions in order (the running-sum centroids make the
// trials inherently sequential).  V has ld = len + 1; column `len` is the bias row of the zero fix.
__global__ void __launch_bounds__(1024) cluster_kernel(double* __restrict__ V, int len, int ld, int k, int R,
                                                       const int* __restrict__ bias, double* __restrict__ cent,
                                                       int* __restrict__ labels) {
    extern __shared__ double sm[];
    double* D = sm;                                       // k*k, column-major D[f + c*k]
    int* assign = reinterpret_cast<int*>(D + (size_t)k * k);  // k : factor column taken by centroid c
    const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = NT >> 5;
    const double b = (*bias) ? 1.0 : 0.0;
    const int L = (*bias) ? len + 1 : len;  // effective vector length
    for (int row = tid; row < R * k; row += NT) V[(long long)row * ld + len] = b;
    __syncthreads();
    // centSeeds = newClusterCenters = factors[1] (:453-455); labels[:,1] = 1:k (:461)
    for (int e = tid; e < k * ld; e += NT) cent[e] = V[e];
    for (int e = tid; e < k; e += NT) labels[e] = e + 1;
    for (int e = k + tid; e < k * R; e += NT) labels[e] = 0;
    __syncthreads();
    for (int t = 1; t < R; ++t) {
        const double* Vt = V + (long long)t * k * ld;
        // D[f,c] = cosine_dist(F_t[:,f], cent[:,c]) (:467-472), NaN -> 0 (:473)
        for (int pair = warp; pair < k * k; pair += nw) {
            const int f = pair % k, c = pair / k;
            const double* x = Vt + (long long)f * ld;
            const double* y = cent + (long long)c * ld;
            double ab = 0.0, a2 = 0.0, b2 = 0.0;
            for (int j = lane; j < L; j += 32) {
                const double xv = x[j], yv = y[j];
                ab = fma(xv, yv, ab);
                a2 = fma(xv, xv, a2);
                b2 = fma(yv, yv, b2);
            }
            ab = wsum(ab);
            a2 = wsum(a2);
            b2 = wsum(b2);
            if (lane == 0) {
                double d = 1.0 - ab / (sqrt(a2) * sqrt(b2));
                d = (d != d) ? 0.0 : (d < 0.0 ? 0.0 : d);
                D[pair] = d;
            }
        }
        __syncthreads();
        // greedy matching (:474-485): repeatedly take the first (column-major) global minimum
        if (warp == 0) {
            for (int c = lane; c < k; c += 32) assign[c] = -1;
            __syncwarp();
            for (int round = 0; round < k; ++round) {
                double bv = INFINITY;
                int bi = INT_MAX;
                for (int e = lane; e < k * k; e += 32) {
                    const double v = D[e];
                    if (v < bv) {
                        bv = v;
                        bi = e;
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    if (ov < bv || (ov == bv && oi < bi)) {
                        bv = ov;
                        bi = oi;
                    }
                }
                if (!(bv < INFINITY)) break;  // while minimum(clusterDistances) < Inf
                const int f = bi % k, c = bi / k;
                if (lane == 0) {
                    labels[f + (long long)t * k] = c + 1;
                    assign[c] = f;
                }
                for (int e = lane; e < k; e += 32) {
                    D[f + e * k] = INFINITY;  // clusterDistances[f, :] .+= Inf
                    D[e + c * k] = INFINITY;  // clusterDistances[:, c] .+= Inf
                }
                __syncwarp();
            }
        }
        __syncthreads();
        // newClusterCenters[:, c] .+= W[:, f]
        for (int e = tid; e < k * L; e += NT) {
            const int c = e / L, j = e - c * L;
            const int f = assign[c];
            if (f >= 0) cent[(long long)c * ld + j] += Vt[(long long)f * ld + j];
        }
        __syncthreads();
    }
    // repair of unassigned labels (:487-496)
    for (int t = tid; t < R; t += NT) {
        int* col = labels + (long long)t * k;
        int s = 0;
        bool anyzero = false;
        for (int a = 0; a < k; ++a) {
            s += col[a];
            anyzero |= (col[a] == 0);
        }
        if (anyzero) {
            if (s == 0)
                for (int a = 0; a < k; ++a) col[a] = a + 1;
            else
                for (int a = 0; a < k; ++a)
                    if (col[a] == 0) col[a] = a + 1;
        }
    }
    __syncthreads();
    // newClusterCenters ./= numTrials (:512)
    for (int e = tid; e < k * ld; e += NT) cent[e] = cent[e] / (double)R;
}

// The same walk as cluster_kernel spread over the whole GPU: the trials stay sequential, but the k x k distances of a trial are
// independent (one warp each, the SAME fixed-order reduction as in cluster_kernel, so results are bit-identical) and so are
// the elements of the centroid update.  Three small launches per trial; used when a trial has enough work to pay for them
// (C3: 256 dot products of length 10000 per trial took one SM 0.3 ms, 20 ms per call).
__global__ void cluster_prep_kernel(double* __restrict__ V, int len, int ld, int k, int R, const int* __restrict__ bias,
                                    int* __restrict__ labels) {
    const double b = (*bias) ? 1.0 : 0.0;
    const int gid = blockIdx.x * blockDim.x + threadIdx.x, gn = gridDim.x * blockDim.x;
    for (int row = gid; row < R * k; row += gn) V[(long long)row * ld + len] = b;
    for (int e = gid; e < k * R; e += gn) labels[e] = e < k ? e + 1 : 0;  // labels[:,1] = 1:k (:461)
}
__global__ void cluster_seed_kernel(const double* __restrict__ V, int ld, int k, double* __restrict__ cent) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x, gn = gridDim.x * blockDim.x;
    for (int e = gid; e < k * ld; e += gn) cent[e] = V[e];  // centSeeds = newClusterCenters = factors[1] (:453-455)
}
__global__ void __launch_bounds__(64) cluster_dist_kernel(const double* __restrict__ Vt, const double* __restrict__ cent, int len,
                                                           int ld, int k, const int* __restrict__ bias, double* __restrict__ D) {
    const int pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (pair >= k * k) return;
    const int L = (*bias) ? len + 1 : len;
    const int f = pair % k, c = pair / k;
    const double* x = Vt + (long long)f * ld;
    const double* y = cent + (long long)c * ld;
    double ab = 0.0, a2 = 0.0, b2 = 0.0;
    int j = lane;
    for (; j + 7 * 32 < L; j += 8 * 32) {  // eight loads of each vector in flight; the sums keep the order of the plain loop
        double xv[8], yv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            xv[u] = x[j + u * 32];
            yv[u] = y[j + u * 32];
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            ab = fma(xv[u], yv[u], ab);
            a2 = fma(xv[u], xv[u], a2);
            b2 = fma(yv[u], yv[u], b2);
        }
    }
    for (; j < L; j += 32) {
        const double xv = x[j], yv = y[j];
        ab = fma(xv, yv, ab);
        a2 = fma(xv, xv, a2);
        b2 = fma(yv, yv, b2);
    }
    ab = wsum(ab);
    a2 = wsum(a2);
    b2 = wsum(b2);
    if (lane == 0) {
        double d = 1.0 - ab / (sqrt(a2) * sqrt(b2));
        d = (d != d) ? 0.0 : (d < 0.0 ? 0.0 : d);
        D[pair] = d;
    }
}
// greedy matching of one trial (:474-485): one warp, first (column-major) global minimum each round
__global__ void cluster_assign_kernel(double* __restrict__ D, int k, int t, int* __restrict__ labels, int* __restrict__ assign) {
    const int lane = threadIdx.x;
    for (int c = lane; c < k; c += 32) assign[c] = -1;
    __syncwarp();
    for (int round = 0; round < k; ++round) {
        double bv = INFINITY;
        int bi = INT_MAX;
        for (int e = lane; e < k * k; e += 32) {
            const double v = D[e];
            if (v < bv) {
                bv = v;
                bi = e;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov < bv || (ov == bv && oi < bi)) {
                bv = ov;
                bi = oi;
            }
        }
        if (!(bv < INFINITY)) break;
        const int f = bi % k, c = bi / k;
        if (lane == 0) {
            labels[f + (long long)t * k] = c + 1;
            assign[c] = f;
        }
        for (int e = lane; e < k; e += 32) {
            D[f + e * k] = INFINITY;
            D[e + c * k] = INFINITY;
        }
        __syncwarp();
    }
}
__global__ void cluster_update_kernel(const double* __restrict__ Vt, double* __restrict__ cent, int len, int ld, int k,
                                      const int* __restrict__ bias, const int* __restrict__ assign) {
    const int L = (*bias) ? len + 1 : len;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < (long long)k * L; e += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(e / L), j = (int)(e - (long long)c * L);
        const int f = assign[c];
        if (f >= 0) cent[(long long)c * ld + j] += Vt[(long long)f * ld + j];  // newClusterCenters[:, c] .+= W[:, f]
    }
}
__global__ void cluster_finish_kernel(double* __restrict__ cent, int ld, int k, int R, int* __restrict__ labels) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x, gn = gridDim.x * blockDim.x;
    for (int t = gid; t < R; t += gn) {  // repair of unassigned labels (:487-496)
        int* col = labels + (long long)t * k;
        int s = 0;
        bool anyzero = false;
        for (int a = 0; a < k; ++a) {
            s += col[a];
            anyzero |= (col[a] == 0);
        }
        if (anyzero) {
            if (s == 0)
                for (int a = 0; a < k; ++a) col[a] = a + 1;
            else
                for (int a = 0; a < k; ++a)
                    if (col[a] == 0) col[a] = a + 1;
        }
    }
    for (int e = gid; e < k * ld; e += gn) cent[e] = cent[e] / (double)R;  // newClusterCenters ./= numTrials (:512)
}

// clusterWmatrix = true without the zero-column fix: `centSeeds` / `newClusterCenters` of the reference ARE the best solution's
// W (NMFkCluster.jl:426-428, 453-455: no copy on this branch), so after clustersolutions that matrix holds the centroids
// (:484, :512) and finalize / Wbest (NMFkExecute.jl:631-637) read them.  Mirror it: centroids -> the best W (factor type) and
// -> the gathered copy the silhouettes are computed from.
template <typename T>
__global__ void cent_writeback_kernel(const double* __restrict__ cent, int len, int ld, int k, const int* __restrict__ bias,
                                      T* __restrict__ Wbest, double* __restrict__ V) {
    if (*bias) return;  // vcat(factors[i], biasRow) made fresh matrices (:449): nothing is aliased
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < (long long)k * len;
         e += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(e / len), j = (int)(e - (long long)c * len);
        const T v = (T)cent[(long long)c * ld + j];
        Wbest[e] = v;
        V[(long long)c * ld + j] = (double)v;
    }
}

// zerostoepsilon(vcat(Ha...)) (NMFkFinalize.jl:52, NMFkHelpers.jl:529-543) + row norms
__global__ void floor_norm_kernel(double* __restrict__ V, int len, int ld, int N, double floorv,
                                  double* __restrict__ vnorm) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= N) return;
    double* row = V + (long long)warp * ld;
    double s = 0.0;
    for (int j = lane; j < len; j += 32) {
        double v = row[j];
        if (v < floorv) v = floorv;
        row[j] = v;
        s = fma(v, v, s);
    }
    s = wsum(s);
    if (lane == 0) vnorm[warp] = sqrt(s);
}

// Dm[i + j*N] = max(1 - <v_i,v_j>/(|v_i||v_j|), 0), diagonal 0, NaN -> 0
// (Distances.pairwise(CosineDist()), NMFkFinalize.jl:52-54).  64x64 tile per CTA, 4x4 per thread.
__global__ void __launch_bounds__(256) cosine_gram_kernel(const double* __restrict__ V, int len, int ld, int N,
                                                          const double* __restrict__ vnorm, double* __restrict__ Dm) {
    __shared__ double As[16][64 + 1];
    __shared__ double Bs[16][64 + 1];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int i0 = blockIdx.x * 64, j0 = blockIdx.y * 64;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
    for (int l0 = 0; l0 < len; l0 += 16) {
        // 64 rows x 16 columns of each operand; lanes along the contiguous vector dimension
        for (int e = threadIdx.x; e < 64 * 16; e += 256) {
            const int rr = e >> 4, cc = e & 15;
            const int l = l0 + cc;
            const int gi = i0 + rr, gj = j0 + rr;
            As[cc][rr] = (gi < N && l < len) ? V[(long long)gi * ld + l] : 0.0;
            Bs[cc][rr] = (gj < N && l < len) ? V[(long long)gj * ld + l] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int cc = 0; cc < 16; ++cc) {
            double av[4], bv[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) av[a] = As[cc][tx + 16 * a];
#pragma unroll
            for (int b = 0; b < 4; ++b) bv[b] = Bs[cc][ty + 16 * b];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int i = i0 + tx + 16 * a, j = j0 + ty + 16 * b;
            if (i < N && j < N) {
                double d = 1.0 - acc[a][b] / (vnorm[i] * vnorm[j]);
                d = (d != d) ? 0.0 : (d < 0.0 ? 0.0 : d);
                if (i == j) d = 0.0;
                Dm[(long long)i + (long long)j * N] = d;
            }
        }
}

// Dm holds the Gram matrix G = V V^T (DMMA GEMM, fro_gemm_f64.cu): G -> cosine distances in place, same formula as above
__global__ void cosine_from_gram_kernel(double* __restrict__ Dm, int N, const double* __restrict__ vnorm) {
    const long long total = (long long)N * N;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e % N), j = (int)(e / N);
        double d = 1.0 - Dm[e] / (vnorm[i] * vnorm[j]);
        d = (d != d) ? 0.0 : (d < 0.0 ? 0.0 : d);
        if (i == j) d = 0.0;
        Dm[e] = d;
    }
}

// pairwise cosine distances of the N rows of V: on the FP64 tensor pipe (DMMA GEMM V V^T, then the distance formula) once the
// matrix is big enough to fill the GPU, the 64 x 64 DFMA tiles otherwise
cudaError_t pairwise_cosine(const double* V, int len, int ld, int N, const double* vnorm, double* Dm, cudaStream_t s) {
    if (N >= 512) {
        cudaError_t e = launch_fro_gemm_f64(V, ld, V, ld, Dm, N, N, N, len, s);
        if (e != cudaSuccess) return e;
        cosine_from_gram_kernel<<<148 * 8, 256, 0, s>>>(Dm, N, vnorm);
        return cudaGetLastError();
    }
    dim3 grid((N + 63) / 64, (N + 63) / 64);
    cosine_gram_kernel<<<grid, 256, 0, s>>>(V, len, ld, N, vnorm, Dm);
    return cudaGetLastError();
}

// Clustering.silhouettes(assignments, dists): thread per point j, sequential over i (the order the
// package uses), k per-cluster sums kept in shared memory.
__global__ void silhouette_kernel(const double* __restrict__ Dm, int N, int k, const int* __restrict__ labels,
                                  double* __restrict__ sil) {
    extern __shared__ double sm[];
    double* rs = sm;                                                 // k x blockDim
    int* counts = reinterpret_cast<int*>(rs + (size_t)k * blockDim.x);  // k
    const int tid = threadIdx.x, NT = blockDim.x;
    for (int c = tid; c < k; c += NT) counts[c] = 0;
    __syncthreads();
    for (int i = tid; i < N; i += NT) atomicAdd(&counts[labels[i] - 1], 1);
    for (int c = 0; c < k; ++c) rs[c * NT + tid] = 0.0;
    __syncthreads();
    const int j = blockIdx.x * NT + tid;
    if (j >= N) return;
    for (int i = 0; i < N; ++i) {
        if (i == j) continue;
        const int c = labels[i] - 1;
        rs[c * NT + tid] += Dm[(long long)j + (long long)i * N];  // symmetric: D[i,j] == D[j,i], coalesced over j
    }
    const int l = labels[j] - 1;
    double a = 0.0, b = INFINITY;  // b: typemax start, strict '<' scan over the other clusters
    for (int c = 0; c < k; ++c) {
        const int cnt = counts[c] - (c == l ? 1 : 0);
        double r = rs[c * NT + tid];
        r = (cnt == 0) ? 0.0 : r / (double)cnt;
        if (c == l)
            a = r;
        else if (r < b)
            b = r;
    }
    double s;
    if (counts[l] == 1)
        s = 0.0;
    else
        s = (a < b) ? (1.0 - a / b) : ((a > b) ? (b / a - 1.0) : 0.0);
    if (s != s) s = 0.0;  // silhouettes[isnan.(silhouettes)] .= 0 (NMFkFinalize.jl:58)
    sil[j] = s;
}

// clustersilhouettes[c] = mean(silhouettes[idx .== c]) in column-major order (NMFkFinalize.jl:64-66)
__global__ void cluster_mean_kernel(const double* __restrict__ sil, const int* __restrict__ labels, int N, int k,
                                    double* __restrict__ clustersil) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= k) return;
    double s = 0.0;
    int cnt = 0;
    for (int i = 0; i < N; ++i)
        if (labels[i] == c + 1) {
            s += sil[i];
            ++cnt;
        }
    clustersil[c] = s / (double)cnt;  // mean of an empty set is NaN, like Statistics.mean
}

}  // namespace

cudaError_t launch_zero_nan(void* p, long long len, int dtype, cudaStream_t s) {
    int blocks = (int)((len + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks < 1) blocks = 1;
    if (dtype == 1)
        zero_nan_kernel<double><<<blocks, 256, 0, s>>>((double*)p, len);
    else
        zero_nan_kernel<float><<<blocks, 256, 0, s>>>((float*)p, len);
    return cudaGetLastError();
}

// Wmean / Wvar (or Hmean / Hvar) of NMFkFinalize.jl:68-74: for cluster c and trial t (sorted order) take the column of W_t
// (row of H_t) that clustersolutions assigned to c, then mean and corrected variance over the R trials.
// amap[c * R + t] = 0-based row / column index of trial t's member of cluster c (-1: none), order[t] = restart of trial t.
// Two passes in Float64 (mean, then squared deviations) like Statistics.mean / Statistics.var.
template <typename T>
__global__ void __launch_bounds__(256) cluster_means_kernel(const T* __restrict__ F, int len, int k, int R, int use_W,
                                                            const int32_t* __restrict__ order, const int32_t* __restrict__ amap,
                                                            T* __restrict__ mean_out, T* __restrict__ var_out) {
    const int c = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= len) return;
    const long long rstride = (long long)len * k;
    auto at = [&](int t) -> double {
        const int a = amap[c * R + t];
        const T* Fr = F + (long long)order[t] * rstride;
        return (double)(use_W ? Fr[(long long)e + (long long)a * len] : Fr[(long long)a + (long long)e * k]);
    };
    double sum = 0.0;
    int cnt = 0;
    for (int t = 0; t < R; ++t)
        if (amap[c * R + t] >= 0) {
            sum += at(t);
            ++cnt;
        }
    const double mean = cnt > 0 ? sum / cnt : nan("");
    double ss = 0.0;
    for (int t = 0; t < R; ++t)
        if (amap[c * R + t] >= 0) {
            const double d = at(t) - mean;
            ss = fma(d, d, ss);
        }
    const double var = cnt > 1 ? ss / (cnt - 1) : nan("");
    const long long o = use_W ? ((long long)e + (long long)c * len) : ((long long)c + (long long)e * k);
    mean_out[o] = (T)mean;
    var_out[o] = (T)var;
}

cudaError_t launch_cluster_means(const void* F, int len, int k, int R, int use_W, const int32_t* d_order, const int32_t* d_amap,
                                 void* mean_out, void* var_out, int dtype, cudaStream_t s) {
    dim3 g((len + 255) / 256, k);
    if (dtype == 1)
        cluster_means_kernel<double><<<g, 256, 0, s>>>((const double*)F, len, k, R, use_W, d_order, d_amap, (double*)mean_out,
                                                       (double*)var_out);
    else
        cluster_means_kernel<float><<<g, 256, 0, s>>>((const float*)F, len, k, R, use_W, d_order, d_amap, (float*)mean_out,
                                                      (float*)var_out);
    return cudaGetLastError();
}

// silhouettes of N labelled points (robustkmeans, NMFkCluster.jl:195-218): V = the points as rows (N x ld doubles, floored in
// place like zerostoepsilon), Dm = pairwise cosine distances, sil = Clustering.silhouettes(labels, Dm)
cudaError_t launch_point_silhouettes(double* V, int len, int ld, int N, int k, const int* labels, double floorv, double* vnorm, double* Dm,
                                     double* sil, cudaStream_t s) {
    cudaError_t e;
    floor_norm_kernel<<<(N + 7) / 8, 256, 0, s>>>(V, len, ld, N, floorv, vnorm);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if ((e = pairwise_cosine(V, len, ld, N, vnorm, Dm, s)) != cudaSuccess) return e;
    const int NT = 128;
    const size_t smem = (size_t)k * NT * sizeof(double) + (size_t)k * sizeof(int);
    if (smem > 48 * 1024 && (e = cudaFuncSetAttribute(silhouette_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
        return e;
    silhouette_kernel<<<(N + NT - 1) / NT, NT, smem, s>>>(Dm, N, k, labels, sil);
    return cudaGetLastError();
}

// kernels the clustersolutions walk launches (the wide walk is three launches per trial)
int cluster_walk_launches(int k, int len, int R) { return ((long long)k * k * len >= 200000 && R >= 2) ? 3 * (R - 1) + 3 : 1; }

cudaError_t launch_cluster(const ClusterArgs& a, int dtype, cudaStream_t s) {
    const int N = a.R * a.k, ld = a.len + 1;
    cudaError_t e;
    if ((e = cudaMemsetAsync(a.bias, 0, sizeof(int), s)) != cudaSuccess) return e;
    {
        const int warps_per_block = 8;
        const int blocks = (N + warps_per_block - 1) / warps_per_block;
        if (dtype == 1)
            gather_kernel<double><<<blocks, 256, 0, s>>>((const double*)a.F, a.len, a.k, a.R, a.use_W, a.order, a.V, ld,
                                                         a.bias);
        else
            gather_kernel<float><<<blocks, 256, 0, s>>>((const float*)a.F, a.len, a.k, a.R, a.use_W, a.order, a.V, ld,
                                                        a.bias);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    {
        if (cluster_walk_launches(a.k, a.len, a.R) > 1) {
            // wide walk: the k x k distances and the assignment flags of a trial live at the start of the (still unused) N x N matrix
            double* D = a.Dm;
            int* assign = reinterpret_cast<int*>(a.Dm + (size_t)a.k * a.k);
            const int pb = (a.k * a.k + 1) / 2;  // two warps (pairs) per CTA: k^2 / 2 CTAs
            const int ub = (int)std::min<long long>(((long long)a.k * ld + 255) / 256, 148 * 8);
            cluster_prep_kernel<<<std::min((N + 255) / 256, 148), 256, 0, s>>>(a.V, a.len, ld, a.k, a.R, a.bias, a.labels);
            cluster_seed_kernel<<<ub, 256, 0, s>>>(a.V, ld, a.k, a.cent);
            for (int t = 1; t < a.R; ++t) {
                const double* Vt = a.V + (long long)t * a.k * ld;
                cluster_dist_kernel<<<pb, 64, 0, s>>>(Vt, a.cent, a.len, ld, a.k, a.bias, D);
                cluster_assign_kernel<<<1, 32, 0, s>>>(D, a.k, t, a.labels, assign);
                cluster_update_kernel<<<ub, 256, 0, s>>>(Vt, a.cent, a.len, ld, a.k, a.bias, assign);
            }
            cluster_finish_kernel<<<ub, 256, 0, s>>>(a.cent, ld, a.k, a.R, a.labels);
        } else {
            const size_t smem = (size_t)a.k * a.k * sizeof(double) + (size_t)a.k * sizeof(int);
            cluster_kernel<<<1, 1024, smem, s>>>(a.V, a.len, ld, a.k, a.R, a.bias, a.cent, a.labels);
        }
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    if (a.alias_best != nullptr) {
        const int blocks = (int)std::min<long long>(((long long)a.k * a.len + 255) / 256, 148 * 4);
        if (dtype == 1)
            cent_writeback_kernel<double><<<blocks, 256, 0, s>>>(a.cent, a.len, ld, a.k, a.bias, (double*)a.alias_best, a.V);
        else
            cent_writeback_kernel<float><<<blocks, 256, 0, s>>>(a.cent, a.len, ld, a.k, a.bias, (float*)a.alias_best, a.V);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    {
        // eps(T)^2 of the factor element type (NMFkHelpers.jl:536-537)
        const double eps = dtype == 1 ? 2.220446049250313e-16 : (double)1.1920929e-07f;
        const double floorv = dtype == 1 ? eps * eps : (double)((float)eps * (float)eps);
        floor_norm_kernel<<<(N + 7) / 8, 256, 0, s>>>(a.V, a.len, ld, N, floorv, a.vnorm);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if ((e = pairwise_cosine(a.V, a.len, ld, N, a.vnorm, a.Dm, s)) != cudaSuccess) return e;
        const int NT = 128;
        const size_t smem = (size_t)a.k * NT * sizeof(double) + (size_t)a.k * sizeof(int);
        if (smem > 48 * 1024 &&  // k >= 48
            (e = cudaFuncSetAttribute(silhouette_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
            return e;
        silhouette_kernel<<<(N + NT - 1) / NT, NT, smem, s>>>(a.Dm, N, a.k, a.labels, a.sil);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        cluster_mean_kernel<<<1, 64, 0, s>>>(a.sil, a.labels, N, a.k, a.clustersil);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace nmfk
