// Generic residual reductions for one (W, H) pair of any size (not on the hot loop):
//   sum over non-NaN entries of ((X - W*H) * weight)^2   and of (X - W*H)^2
// used for the :74 objective in trace mode, for phi_final (/root/reference/src/NMFkExecute.jl:664-668)
// and for the per-k fit re-derivation of execute (:212-222).  Deterministic: one partial per
// CTA (128 rows x one slice of the columns), summed in CTA order on the host.
#include "nmfk_internal.h"

namespace nmfk {

namespace {

constexpr int kRows = 128;  // rows of X per CTA

template <typename T>
__global__ void __launch_bounds__(kRows) residual_kernel(const T* __restrict__ X, int n, int m, int k,
                                                         const T* __restrict__ W, const T* __restrict__ H, T lambda,
                                                         int restore, double weight, const WeightRef wref,
                                                         int slices, double* __restrict__ partials) {
    extern __shared__ unsigned char smraw[];
    T* Ws = reinterpret_cast<T*>(smraw);  // [k][kRows]
    __shared__ double red[2][kRows / 32];
    const int i0 = blockIdx.x * kRows, tid = threadIdx.x, i = i0 + tid;
    // columns of this CTA: slice blockIdx.y of `slices` (a tall-and-wide X would otherwise run on n / 128 CTAs only)
    const int j_begin = (int)(((long long)m * blockIdx.y) / slices), j_end = (int)(((long long)m * (blockIdx.y + 1)) / slices);
    for (int a = 0; a < k; ++a) Ws[a * kRows + tid] = (i < n) ? W[(size_t)i + (size_t)a * n] : (T)0;
    __syncthreads();
    double sw = 0.0, s1 = 0.0;
    const bool wany = wref.any();
    if (i < n) {
        for (int j = j_begin; j < j_end; ++j) {
            const T xr = X[(size_t)i + (size_t)j * n];
            if (xr != xr) continue;
            T x = xr;
            if (restore && x == lambda) x = (T)0;
            const T* h = H + (size_t)j * k;
            T p = (T)0;
            for (int a = 0; a < k; ++a) p = fma(Ws[a * kRows + tid], __ldg(h + a), p);
            const double e = (double)(x - p);
            s1 = fma(e, e, s1);
            const double ew = e * (wany ? weight_at<T>(wref, weight, i, j, n) : weight);
            sw = fma(ew, ew, sw);
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        sw += __shfl_xor_sync(0xffffffffu, sw, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    }
    if ((tid & 31) == 0) {
        red[0][tid >> 5] = sw;
        red[1][tid >> 5] = s1;
    }
    __syncthreads();
    if (tid == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < kRows / 32; ++w) {
            a += red[0][w];
            b += red[1][w];
        }
        const size_t slot = (size_t)blockIdx.x * slices + blockIdx.y;
        partials[2 * slot] = a;
        partials[2 * slot + 1] = b;
    }
}

}  // namespace

// column slices: enough CTAs for ~4 per SM, at least 64 columns each
static int residual_slices(int n, int m) {
    const int rb = (n + kRows - 1) / kRows;
    int sl = (148 * 4 + rb - 1) / rb;
    sl = sl < 1 ? 1 : sl;
    const int cap = m / 64 > 0 ? m / 64 : 1;
    return sl < cap ? sl : cap;
}
int residual_blocks(int n, int m) { return ((n + kRows - 1) / kRows) * residual_slices(n, m); }

cudaError_t launch_residual(const void* X, int dtype, int n, int m, int k, const void* W, const void* H, double lambda,
                            int restore, double weight, const WeightRef& wref, double* d_partials, cudaStream_t s) {
    const int slices = residual_slices(n, m);
    const dim3 grid((n + kRows - 1) / kRows, slices);
    const size_t smem = (size_t)k * kRows * (dtype == 1 ? 8 : 4);
    if (smem + sizeof(double) * 2 * (kRows / 32) > 48 * 1024) {  // the rows of W of a block, with the static sums (k >= 48 in Float64)
        const cudaError_t e = dtype == 1 ? cudaFuncSetAttribute(residual_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                                         : cudaFuncSetAttribute(residual_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    if (dtype == 1)
        residual_kernel<double><<<grid, kRows, smem, s>>>((const double*)X, n, m, k, (const double*)W, (const double*)H, lambda,
                                                          restore, weight, wref, slices, d_partials);
    else
        residual_kernel<float><<<grid, kRows, smem, s>>>((const float*)X, n, m, k, (const float*)W, (const float*)H,
                                                         (float)lambda, restore, weight, wref, slices, d_partials);
    return cudaGetLastError();
}

}  // namespace nmfk
