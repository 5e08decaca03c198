// NMFsparsity (/root/reference/src/NMFkSparsity.jl:1-113; method=:sparsity, NMFkExecute.jl:757-758) for a batch of restarts:
// beta-divergence multiplicative updates (beta = 2 Euclidean - the default cost_function=:ed -, 1 Kullback-Leibler, 0
// Itakura-Saito, or any other value) with an L1 penalty `sparsity` on H and unit-norm columns of W.
//
// Unlike Variant FRO the model X_est = max.(W*H, lambda) is clamped (:48, :71, :87), so W' * X_est is a per-restart product
// and nothing stacks: one CTA row of the grid per restart, scalar-FMA kernels in the shape of the tiled KL fallback pass -
// correctness first, not tuned (this solver sits next to the hot path, SURVEY.md 8(f4)).  With
//     e = max(<U[o,:], V[t,:]>, lambda),   est(e) = e^(beta-1),   xt(x, e) = x e^(beta-2)
// one half-update needs  A_est[o,a] = sum_t est V[t,a]  and  A_x[o,a] = sum_t xt V[t,a]  (sp_pass_kernel), then
//     H <- H .* A_x ./ max(A_est + sparsity, lambda)                                                     (:59-70)
//     W <- W .* (A_x + colsum(A_est .* W) .* W) ./ max(A_est + colsum(A_x .* W) .* W, lambda); W ./= colnorm(W)   (:73-86)
// (for beta = 1 est == 1 and A_est is the column / row sum the reference writes explicitly).  The objective
// divergence + sparsity * sum(H) is evaluated after every iteration (:89-99); the run stops when its relative change drops
// below tol (:101-106) or at maxiter.  The post-run objective / normalisation of execute_singlerun_compute are the tiled
// engine's kernels, like for the other variants.
#include <climits>
#include <cmath>
#include <vector>

#include "fro.h"
#include "kl_tiled.cuh"

namespace nmfk {
namespace {

constexpr int SP_T = 128;   // own indices per CTA
constexpr int SP_TT = 32;   // reduction steps per staged tile

template <typename T>
__device__ __forceinline__ void sp_terms(T x, T e, double beta, int bmode, T& est, T& xt) {
    if (bmode == 2) {
        est = e;
        xt = x;
    } else if (bmode == 1) {
        est = (T)1;
        xt = x / e;
    } else if (bmode == 0) {
        est = (T)1 / e;
        xt = x / (e * e);
    } else {
        est = (T)pow((double)e, beta - 1.0);
        xt = (T)((double)x * pow((double)e, beta - 2.0));
    }
}

// A_est / A_x of one half-update.  D: data with the own index contiguous (element (o,t) at D[o + t*nown]); U: own factor
// (element (o,b) at U[o*su_o + b*su_a]); V: other factor ((t,b) at V[t*sv_t + b*sv_a]); outputs [R][nown][KMAX].
// D is the preprocessed image of X, whose zeros nmfk_set_X replaced by xsub; NMFsparsity never substitutes them (its
// NMFpreprocessing! call is commented out), so x == xsub counts as 0 here and in sp_objective_kernel
template <typename T, int KMAX>
__global__ void __launch_bounds__(SP_T) sp_pass_kernel(const T* __restrict__ D, const T* __restrict__ Ust, const T* __restrict__ Vst,
                                                       long long u_rstride, long long v_rstride, long long su_o, long long su_a,
                                                       long long sv_t, long long sv_a, int nown, int nred, int k, T xsub,
                                                       double lambda, double beta, int bmode, const UnitState* st, T* __restrict__ Aest,
                                                       T* __restrict__ Ax) {
    __shared__ T Vs[SP_TT][KMAX + 1];
    const int r = blockIdx.y, tid = threadIdx.x;
    if (st[r].stop != 0) return;
    const int o = blockIdx.x * SP_T + tid;
    const bool valid = o < nown;
    const T* U = Ust + (long long)r * u_rstride;
    const T* V = Vst + (long long)r * v_rstride;
    T u[KMAX], ae[KMAX], ax[KMAX];
#pragma unroll
    for (int b = 0; b < KMAX; ++b) {
        u[b] = (valid && b < k) ? U[(long long)o * su_o + (long long)b * su_a] : (T)0;
        ae[b] = (T)0;
        ax[b] = (T)0;
    }
    const T lam = (T)lambda;
    for (int t0 = 0; t0 < nred; t0 += SP_TT) {
        __syncthreads();
        for (int e = tid; e < SP_TT * KMAX; e += SP_T) {
            const int tt = e / KMAX, b = e % KMAX;
            Vs[tt][b] = (t0 + tt < nred && b < k) ? V[(long long)(t0 + tt) * sv_t + (long long)b * sv_a] : (T)0;
        }
        __syncthreads();
        if (valid) {
            const int cnt = min(SP_TT, nred - t0);
            for (int tt = 0; tt < cnt; ++tt) {
                T p = (T)0;
#pragma unroll
                for (int b = 0; b < KMAX; ++b) p = fma(u[b], Vs[tt][b], p);
                const T e = p > lam ? p : lam;  // max.(W*H, lambda)
                T x = D[(long long)o + (long long)(t0 + tt) * nown];
                if (x == xsub) x = (T)0;
                T est, xt;
                sp_terms<T>(x, e, beta, bmode, est, xt);
#pragma unroll
                for (int b = 0; b < KMAX; ++b) {
                    ae[b] = fma(est, Vs[tt][b], ae[b]);
                    ax[b] = fma(xt, Vs[tt][b], ax[b]);
                }
            }
        }
    }
    if (!valid) return;
    T* de = Aest + ((long long)r * nown + o) * KMAX;
    T* dx = Ax + ((long long)r * nown + o) * KMAX;
#pragma unroll
    for (int b = 0; b < KMAX; ++b) {
        de[b] = ae[b];
        dx[b] = ax[b];
    }
}

// H[a,j] *= A_x / max(A_est + sparsity, lambda)   (:69-70)
template <typename T, int KMAX>
__global__ void sp_apply_H_kernel(T* __restrict__ Hst, int k, int m, const T* __restrict__ Aest, const T* __restrict__ Ax, double sparsity,
                                  double lambda, const UnitState* st) {
    const int r = blockIdx.y;
    if (st[r].stop != 0) return;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    T* h = Hst + (long long)r * k * m + (long long)j * k;
    const T* ae = Aest + ((long long)r * m + j) * KMAX;
    const T* ax = Ax + ((long long)r * m + j) * KMAX;
    for (int a = 0; a < k; ++a) {
        T dph = ae[a] + (T)sparsity;
        dph = dph > (T)lambda ? dph : (T)lambda;
        h[a] = h[a] * (ax[a] / dph);
    }
}

// c1[a] = sum_i A_x[i,a] W[i,a], c2[a] = sum_i A_est[i,a] W[i,a]  (the colsum terms of :78-79); one CTA per restart
template <typename T, int KMAX>
__global__ void __launch_bounds__(256) sp_colstats_kernel(const T* __restrict__ Wst, int n, int k, const T* __restrict__ Aest,
                                                          const T* __restrict__ Ax, const UnitState* st, double* __restrict__ cst) {
    __shared__ double red[40];
    const int r = blockIdx.x, tid = threadIdx.x;
    if (st[r].stop != 0) return;
    const T* W = Wst + (long long)r * n * k;
    for (int a = 0; a < k; ++a) {
        double s1 = 0.0, s2 = 0.0;
        for (int i = tid; i < n; i += 256) {
            const double w = (double)W[(long long)i + (long long)a * n];
            s1 += (double)Ax[((long long)r * n + i) * KMAX + a] * w;
            s2 += (double)Aest[((long long)r * n + i) * KMAX + a] * w;
        }
        s1 = block_sum(s1, red);
        s2 = block_sum(s2, red);
        if (tid == 0) {
            cst[(long long)r * 64 + a] = s1;
            cst[(long long)r * 64 + 32 + a] = s2;
        }
    }
}

// W[i,a] *= (A_x + c2[a] W) / max(A_est + c1[a] W, lambda)   (:78-85)
template <typename T, int KMAX>
__global__ void sp_apply_W_kernel(T* __restrict__ Wst, int n, int k, const T* __restrict__ Aest, const T* __restrict__ Ax,
                                  const double* __restrict__ cst, double lambda, const UnitState* st) {
    const int r = blockIdx.y;
    if (st[r].stop != 0) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    T* W = Wst + (long long)r * n * k;
    for (int a = 0; a < k; ++a) {
        const T w = W[(long long)i + (long long)a * n];
        const T dmw = Ax[((long long)r * n + i) * KMAX + a] + (T)cst[(long long)r * 64 + 32 + a] * w;
        T dpw = Aest[((long long)r * n + i) * KMAX + a] + (T)cst[(long long)r * 64 + a] * w;
        dpw = dpw > (T)lambda ? dpw : (T)lambda;
        W[(long long)i + (long long)a * n] = w * (dmw / dpw);
    }
}

// W ./= sqrt.(sum(W.^2; dims=1)) (:86; with scaleH also H .*= Wn' for the initial normalisation :44-46); one CTA per restart
template <typename T>
__global__ void __launch_bounds__(256) sp_colnorm_kernel(T* __restrict__ Wst, T* __restrict__ Hst, int n, int m, int k, int scaleH,
                                                         const UnitState* st) {
    __shared__ double red[40];
    __shared__ double nrm[32];
    const int r = blockIdx.x, tid = threadIdx.x;
    if (st[r].stop != 0) return;
    T* W = Wst + (long long)r * n * k;
    for (int a = 0; a < k; ++a) {
        double s = 0.0;
        for (int i = tid; i < n; i += 256) {
            const double w = (double)W[(long long)i + (long long)a * n];
            s = fma(w, w, s);
        }
        s = block_sum(s, red);
        if (tid == 0) nrm[a] = (double)(T)sqrt(s);
    }
    __syncthreads();
    for (long long e = tid; e < (long long)n * k; e += 256) W[e] = W[e] / (T)nrm[e / n];
    if (scaleH) {
        T* H = Hst + (long long)r * k * m;
        for (long long e = tid; e < (long long)k * m; e += 256) H[e] = H[e] * (T)nrm[e % k];
    }
}

// divergence(X, max(W*H, lambda)) of rows [128 b, 128 b + 128) -> part[(r * nblk + b)]   (:89-98).  With zeros in X (x == xsub
// counts as 0) the kl divergence is NaN and the is divergence Inf, as in the reference: the relative-change test then never
// stops the run
template <typename T, int KMAX>
__global__ void __launch_bounds__(SP_T) sp_objective_kernel(const T* __restrict__ X, int n, int m, int k, const T* __restrict__ Wst,
                                                            const T* __restrict__ Hst, T xsub, double lambda, double beta, int bmode,
                                                            const UnitState* st, double* __restrict__ part) {
    __shared__ T Hs[SP_TT][KMAX + 1];
    __shared__ double red[8];
    const int r = blockIdx.y, tid = threadIdx.x;
    if (st[r].stop != 0) return;
    const int i = blockIdx.x * SP_T + tid;
    const bool valid = i < n;
    const T* W = Wst + (long long)r * n * k;
    const T* H = Hst + (long long)r * k * m;
    T w[KMAX];
#pragma unroll
    for (int b = 0; b < KMAX; ++b) w[b] = (valid && b < k) ? W[(long long)i + (long long)b * n] : (T)0;
    double s = 0.0;
    for (int j0 = 0; j0 < m; j0 += SP_TT) {
        __syncthreads();
        for (int e = tid; e < SP_TT * KMAX; e += SP_T) {
            const int jj = e / KMAX, b = e % KMAX;
            Hs[jj][b] = (j0 + jj < m && b < k) ? H[(long long)(j0 + jj) * k + b] : (T)0;
        }
        __syncthreads();
        if (valid) {
            const int cnt = min(SP_TT, m - j0);
            for (int jj = 0; jj < cnt; ++jj) {
                T p = (T)0;
#pragma unroll
                for (int b = 0; b < KMAX; ++b) p = fma(w[b], Hs[jj][b], p);
                const double e = (double)(p > (T)lambda ? p : (T)lambda);
                const T xs = X[(long long)i + (long long)(j0 + jj) * n];
                const double x = xs == xsub ? 0.0 : (double)xs;
                double d;
                if (bmode == 2)
                    d = (x - e) * (x - e);
                else if (bmode == 1)
                    d = x * log(x / e) - x + e;
                else if (bmode == 0)
                    d = x / e - log(x / e) - 1.0;
                else
                    d = (pow(x, beta) + (beta - 1.0) * pow(e, beta) - beta * x * pow(e, beta - 1.0)) / (beta * (beta - 1.0));
                s += d;
            }
        }
    }
    s = warp_sum(s);
    if ((tid & 31) == 0) red[tid >> 5] = s;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w2 = 0; w2 < SP_T / 32; ++w2) t += red[w2];
        part[(long long)r * gridDim.x + blockIdx.x] = t;
    }
}

// of = divergence + sparsity * sum(H); relative-change test against the previous iteration (:99-107); one CTA per restart
template <typename T>
__global__ void __launch_bounds__(256) sp_state_kernel(UnitState* stv, const T* __restrict__ Hst, int k, int m, const double* __restrict__ part,
                                                       int nblk, double sparsity, double tol, int it) {
    __shared__ double red[40];
    const int r = blockIdx.x, tid = threadIdx.x;
    UnitState* st = stv + r;
    if (st->stop != 0) return;
    const T* H = Hst + (long long)r * k * m;
    double sh = 0.0;
    for (long long e = tid; e < (long long)k * m; e += 256) sh += (double)H[e];
    sh = block_sum(sh, red);
    if (tid == 0) {
        double div = 0.0;
        for (int b = 0; b < nblk; ++b) div += part[(long long)r * nblk + b];
        const double of = div + sparsity * sh;
        const double last = st->best;  // last_of (Inf before the first iteration)
        st->it = it;
        st->obj_chk = of;
        if (it > 1 && tol > 0 && (fabs(of - last) / last) < tol) st->stop = 2;
        st->best = of;
    }
}

template <typename T, int KMAX>
cudaError_t sp_iteration(const SolveArgs& a, double beta, int bmode, double sparsity, double lam, T* Aest, T* Ax, double* cst, double* part,
                         int nblk, int it, cudaStream_t s, int64_t* launches) {
    const int n = a.n, m = a.m, k = a.k, R = a.R;
    T* W = static_cast<T*>(a.W);
    T* H = static_cast<T*>(a.H);
    cudaError_t e;
    if (!a.Hfixed) {  // own = columns of H: D = X^T, U = H (su_o = k, su_a = 1), V = W (sv_t = 1, sv_a = n)
        sp_pass_kernel<T, KMAX><<<dim3((m + SP_T - 1) / SP_T, R), SP_T, 0, s>>>(static_cast<const T*>(a.Xt), H, W, (long long)k * m,
                                                                               (long long)n * k, k, 1, 1, n, m, n, k, (T)a.lambda, lam, beta,
                                                                               bmode, a.st, Aest, Ax);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        sp_apply_H_kernel<T, KMAX><<<dim3((m + 255) / 256, R), 256, 0, s>>>(H, k, m, Aest, Ax, sparsity, lam, a.st);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        *launches += 2;
    }
    if (!a.Wfixed) {  // own = rows of W: D = X, U = W (su_o = 1, su_a = n), V = H' (sv_t = k, sv_a = 1)
        sp_pass_kernel<T, KMAX><<<dim3((n + SP_T - 1) / SP_T, R), SP_T, 0, s>>>(static_cast<const T*>(a.X), W, H, (long long)n * k,
                                                                               (long long)k * m, 1, n, k, 1, n, m, k, (T)a.lambda, lam, beta,
                                                                               bmode, a.st, Aest, Ax);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        sp_colstats_kernel<T, KMAX><<<R, 256, 0, s>>>(W, n, k, Aest, Ax, a.st, cst);
        sp_apply_W_kernel<T, KMAX><<<dim3((n + 255) / 256, R), 256, 0, s>>>(W, n, k, Aest, Ax, cst, lam, a.st);
        sp_colnorm_kernel<T><<<R, 256, 0, s>>>(W, H, n, m, k, 0, a.st);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        *launches += 4;
    }
    sp_objective_kernel<T, KMAX><<<dim3(nblk, R), SP_T, 0, s>>>(static_cast<const T*>(a.X), n, m, k, W, H, (T)a.lambda, lam, beta, bmode,
                                                                   a.st, part);
    sp_state_kernel<T><<<R, 256, 0, s>>>(a.st, H, k, m, part, nblk, sparsity, a.tol, it);
    *launches += 2;
    return cudaGetLastError();
}

template <typename T>
cudaError_t solve_sparsity_t(const SolveArgs& a, double beta, double sparsity, double lam, cudaStream_t s, int64_t* launches) {
    const int n = a.n, m = a.m, k = a.k, R = a.R;
    if (k > 32) return cudaErrorInvalidValue;
    const int bmode = beta == 2.0 ? 2 : (beta == 1.0 ? 1 : (beta == 0.0 ? 0 : -1));
    const int KM = k <= 8 ? 8 : (k <= 16 ? 16 : 32);
    const int nblk = (n + SP_T - 1) / SP_T, nblkObj = (n + 127) / 128;
    cudaError_t err = cudaSuccess;
    T *Aest = nullptr, *Ax = nullptr;
    double *cst = nullptr, *part = nullptr, *objp = nullptr;
    int *d_active = nullptr, *h_active = nullptr;
    std::vector<UnitState> hst((size_t)R);
    bool any_running = false;
    int it = 0;
#define SP_TRY(call)                        \
    do {                                    \
        cudaError_t e__ = (call);           \
        if (e__ != cudaSuccess) {           \
            err = e__;                      \
            goto done;                      \
        }                                   \
    } while (0)
    SP_TRY(scratch_alloc(&Aest, (size_t)R * std::max(n, m) * KM * sizeof(T), s));
    SP_TRY(scratch_alloc(&Ax, (size_t)R * std::max(n, m) * KM * sizeof(T), s));
    SP_TRY(scratch_alloc(&cst, (size_t)R * 64 * sizeof(double), s));
    SP_TRY(scratch_alloc(&part, (size_t)R * nblk * sizeof(double), s));
    SP_TRY(scratch_alloc(&objp, (size_t)R * nblkObj * 2 * sizeof(double), s));
    SP_TRY(scratch_alloc(&d_active, sizeof(int), s));
    h_active = pinned_flags();
    if (h_active == nullptr) SP_TRY(cudaErrorMemoryAllocation);
    SP_TRY(cudaMemcpyAsync(hst.data(), a.st, (size_t)R * sizeof(UnitState), cudaMemcpyDeviceToHost, s));
    SP_TRY(cudaStreamSynchronize(s));
    for (auto& u : hst)
        if (u.stop == 0 && !u.done) {
            any_running = true;
            it = std::max(it, (int)u.it);
        }
    if (any_running) {
        if (it == 0) {  // Wn = sqrt.(sum(W.^2; dims=1)); W ./= Wn; H .*= Wn' (:44-46)
            sp_colnorm_kernel<T><<<R, 256, 0, s>>>(static_cast<T*>(a.W), static_cast<T*>(a.H), n, m, k, 1, a.st);
            SP_TRY(cudaGetLastError());
            ++*launches;
        }
        bool need_guard = true;
        while (true) {
            if (need_guard) {
                SP_TRY(cudaMemsetAsync(d_active, 0, sizeof(int), s));
                tiled_guard_kernel<<<(R + 127) / 128, 128, 0, s>>>(a.st, R, it, a.maxiter, INT_MAX, INT_MAX, a.iter_limit, d_active);
                SP_TRY(cudaGetLastError());
                SP_TRY(cudaMemcpyAsync(h_active, d_active, sizeof(int), cudaMemcpyDeviceToHost, s));
                SP_TRY(cudaStreamSynchronize(s));
                ++*launches;
                if (*h_active == 0) break;
                need_guard = false;
            }
            ++it;
            if (KM == 8)
                SP_TRY((sp_iteration<T, 8>(a, beta, bmode, sparsity, lam, Aest, Ax, cst, part, nblk, it, s, launches)));
            else if (KM == 16)
                SP_TRY((sp_iteration<T, 16>(a, beta, bmode, sparsity, lam, Aest, Ax, cst, part, nblk, it, s, launches)));
            else
                SP_TRY((sp_iteration<T, 32>(a, beta, bmode, sparsity, lam, Aest, Ax, cst, part, nblk, it, s, launches)));
            if (it % a.check_every == 0 || it >= a.maxiter || (a.iter_limit > 0 && it >= a.iter_limit)) need_guard = true;
        }
    }
    {
        dim3 g(nblkObj, R);  // objvalue = normnan(X - W*H) (NMFkExecute.jl:791-792) + normalisation (:800-804)
        tiled_objective_kernel<T, T><<<g, 128, (size_t)k * 128 * sizeof(T), s>>>(static_cast<const T*>(a.X), n, m, k, static_cast<const T*>(a.W),
                                                                                 static_cast<const T*>(a.H), a.st, (T)a.lambda, 1, 0, 1.0,
                                                                                 WeightRef{nullptr, nullptr, nullptr}, objp);
        SP_TRY(cudaGetLastError());
        tiled_finish_kernel<T><<<R, 256, 0, s>>>(a.W, a.H, a.st, objp, n, m, k, nblkObj, a.normalize);
        SP_TRY(cudaGetLastError());
        *launches += 2;
        SP_TRY(cudaStreamSynchronize(s));
    }
done:
#undef SP_TRY
    scratch_free(Aest, s);
    scratch_free(Ax, s);
    scratch_free(cst, s);
    scratch_free(part, s);
    scratch_free(objp, s);
    scratch_free(d_active, s);
    return err;
}

}  // namespace

cudaError_t solve_sparsity(const SolveArgs& a, int dtype, double beta, double sparsity, double lam, cudaStream_t s, int64_t* launches) {
    return dtype == 1 ? solve_sparsity_t<double>(a, beta, sparsity, lam, s, launches) : solve_sparsity_t<float>(a, beta, sparsity, lam, s, launches);
}

}  // namespace nmfk
