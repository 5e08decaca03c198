// Variant FRO: the Frobenius ("mse") multiplicative update for a batch of R stacked restarts.
//
// Replaces, for method=:nmf / algorithm=:multdiv (/root/reference/src/NMFkExecute.jl:763-766), the third-party
// NMF.solve!(NMF.MultUpdate{T}(obj=:mse, maxiter, tol), X, W, H) (NMF.jl `src/multupd.jl`, restated in
// oracle/nmfk_oracle.py::nmf_multupdate_mse) - the update BASELINE.json's north star spells out:
//     H <- H .* (W'X)  ./ (W'W*H  + d)          d = sqrt(eps(T))
//     W <- W .* (X*H') ./ (W*H*H' + d)          (with the new H)
//     stop when every column of W and every row of H moved by less than tol relative, or at maxiter.
// Unlike the KL update of method=:simple the numerators do not depend on the restart's own product W*H, so ALL restarts
// of a batch are stacked: the factor stacks are kept as [R*k x n] (W, which is the API layout itself) and [R*k x m] (H,
// transposed per restart for the duration of the solve), and one half-update is
//     N = stack_of_the_other_factor * X^(T)     ONE tensor-core GEMM over X for all restarts (fro_gemm.cu / fro_gemm_f64.cu)
//     G_r = V_r V_r^T  (k x k per restart)      fro_gram_kernel
//     U <- U .* N ./ (G_r U + d)                fro_apply_kernel (also writes the lo image of the 3-term split and the
//                                               per-row sums of the convergence test)
// The convergence test runs on the device after every iteration (fro_converge_kernel); the host looks at the number of
// running restarts every `check_every` iterations.  The post-run objective (normnan(X - W*H), NMFkExecute.jl:791-792) and the
// H-row normalisation (:800-804) are the tiled engine's kernels.
#include <climits>
#include <cmath>
#include <vector>

#include "fro.h"
#include "kl_tiled.cuh"  // tiled_objective_kernel, tiled_finish_kernel, block_sum

namespace nmfk {
namespace {

constexpr int FRO_TT = 128;  // columns of a stack handled by one CTA of the apply / gram kernels

__global__ void split_lo_kernel(const float* __restrict__ x, float* __restrict__ lo, long long len) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < len; i += (long long)gridDim.x * blockDim.x) {
        const float v = x[i];
        lo[i] = v - __uint_as_float(__float_as_uint(v) & 0xffffe000u);
    }
}

// H (k x m x R, column-major per restart) <-> Ht ([R*k x m] row-major)
template <typename T>
__global__ void fro_h_to_stack(const T* __restrict__ H, T* __restrict__ Ht, int k, int m) {
    const int r = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const T* src = H + (long long)r * k * m + (long long)j * k;
    for (int a = 0; a < k; ++a) Ht[((long long)r * k + a) * m + j] = src[a];
}
template <typename T>
__global__ void fro_stack_to_h(const T* __restrict__ Ht, T* __restrict__ H, int k, int m, const UnitState* st) {
    const int r = blockIdx.y;
    if (st[r].done != 0) return;  // finished in an earlier (resumed) solve: the API copy is already final
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    T* dst = H + (long long)r * k * m + (long long)j * k;
    for (int a = 0; a < k; ++a) dst[a] = Ht[((long long)r * k + a) * m + j];
}

// Gpart[r][s][a*k + b] = sum over the s-th slice of t of V[(r,a), t] V[(r,b), t]   (V: [R*k x len] row-major)
template <typename T>
__global__ void __launch_bounds__(256) fro_gram_kernel(const T* __restrict__ V, int k, long long len, int S, const UnitState* st,
                                                       double* __restrict__ Gpart) {
    extern __shared__ unsigned char gsm[];
    T* Vs = reinterpret_cast<T*>(gsm);  // [k][FRO_TT + 1]
    const int r = blockIdx.x, s = blockIdx.y, tid = threadIdx.x;
    if (st[r].stop != 0) return;
    const long long t_begin = len * s / S, t_end = len * (s + 1) / S;
    const int npairs = k * k;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};  // k <= 32: at most 4 pairs per thread
    for (long long t0 = t_begin; t0 < t_end; t0 += FRO_TT) {
        const int cnt = (int)min((long long)FRO_TT, t_end - t0);
        for (int e = tid; e < k * FRO_TT; e += 256) {
            const int a = e / FRO_TT, tt = e - a * FRO_TT;
            Vs[a * (FRO_TT + 1) + tt] = tt < cnt ? V[((long long)r * k + a) * len + t0 + tt] : (T)0;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int p = tid + q * 256;
            if (p < npairs) {
                const T* x = Vs + (p / k) * (FRO_TT + 1);
                const T* y = Vs + (p % k) * (FRO_TT + 1);
                double sum = 0.0;
                for (int tt = 0; tt < FRO_TT; ++tt) sum = fma((double)x[tt], (double)y[tt], sum);
                acc[q] += sum;
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int p = tid + q * 256;
        if (p < npairs) Gpart[((long long)r * S + s) * npairs + p] = acc[q];
    }
}

// U[(r,a), t] <- U * N / (sum_b G_r[a,b] U[(r,b), t] + delta) for one tile of FRO_TT columns t of one restart;
// conv[((r * ntile + tile) * k + a) * 2 + {0,1}] = sum_t (new - old)^2, sum_t (new + old)^2 (NMF.jl stop_condition)
template <typename T, int KMAX>
__global__ void __launch_bounds__(FRO_TT) fro_apply_kernel(T* __restrict__ U, float* __restrict__ Ulo, const T* __restrict__ Nm, int NS,
                                                           long long nstride, int k, long long len, const double* __restrict__ Gpart,
                                                           int S, double delta, const UnitState* st, double* __restrict__ conv) {
    __shared__ double Gs[32 * 32];
    __shared__ double red[2][FRO_TT / 32];
    const int r = blockIdx.y, tile = blockIdx.x, tid = threadIdx.x;
    if (st[r].stop != 0) return;
    for (int p = tid; p < k * k; p += FRO_TT) {
        double g = 0.0;
        for (int s = 0; s < S; ++s) g += Gpart[((long long)r * S + s) * k * k + p];  // slices in order: deterministic
        Gs[p] = g;
    }
    __syncthreads();
    const long long t = (long long)tile * FRO_TT + tid;
    const bool valid = t < len;
    T u[KMAX];
#pragma unroll
    for (int b = 0; b < KMAX; ++b) u[b] = (valid && b < k) ? U[((long long)r * k + b) * len + t] : (T)0;
    for (int a = 0; a < k; ++a) {
        double dv = 0.0, sv = 0.0;
        if (valid) {
            T den = (T)0;
#pragma unroll
            for (int b = 0; b < KMAX; ++b)
                if (b < k) den = fma((T)Gs[a * k + b], u[b], den);
            const long long idx = ((long long)r * k + a) * len + t;
            T uo = (T)0;
#pragma unroll
            for (int b = 0; b < KMAX; ++b)
                if (b == a) uo = u[b];
            T num = Nm[idx];
            for (int q = 1; q < NS; ++q) num += Nm[(long long)q * nstride + idx];  // split-K partial products, in slice order
            const T un = uo * (num / (den + (T)delta));
            U[idx] = un;
            if (Ulo != nullptr) {
                const float f = (float)un;
                Ulo[idx] = f - __uint_as_float(__float_as_uint(f) & 0xffffe000u);
            }
            const double d = (double)un - (double)uo, s2 = (double)un + (double)uo;
            dv = d * d;
            sv = s2 * s2;
        }
        dv = warp_sum(dv);
        sv = warp_sum(sv);
        if ((tid & 31) == 0) {
            red[0][tid >> 5] = dv;
            red[1][tid >> 5] = sv;
        }
        __syncthreads();
        if (tid == 0) {
            double x = 0.0, y = 0.0;
            for (int w = 0; w < FRO_TT / 32; ++w) {
                x += red[0][w];
                y += red[1][w];
            }
            double* dst = conv + (((long long)r * gridDim.x + tile) * k + a) * 2;
            dst[0] = x;
            dst[1] = y;
        }
        __syncthreads();
    }
}

// NMF.jl stop_condition after every iteration, one thread per restart
__global__ void fro_converge_kernel(UnitState* st, int R, int k, const double* __restrict__ convW, int tilesW,
                                    const double* __restrict__ convH, int tilesH, int wactive, int hactive, double tol, int it) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    UnitState* s = st + r;
    if (s->stop != 0) return;
    bool converged = true;
    for (int a = 0; a < k && converged; ++a) {
        double dw = 0.0, sw = 0.0, dh = 0.0, sh = 0.0;
        if (wactive)
            for (int t = 0; t < tilesW; ++t) {
                dw += convW[(((long long)r * tilesW + t) * k + a) * 2];
                sw += convW[(((long long)r * tilesW + t) * k + a) * 2 + 1];
            }
        if (hactive)
            for (int t = 0; t < tilesH; ++t) {
                dh += convH[(((long long)r * tilesH + t) * k + a) * 2];
                sh += convH[(((long long)r * tilesH + t) * k + a) * 2 + 1];
            }
        // `if sqrt(dev_w) > eps * sqrt(sum_w) || sqrt(dev_h) > eps * sqrt(sum_h) return false` (a NaN never is greater)
        if ((wactive && sqrt(dw) > tol * sqrt(sw)) || (hactive && sqrt(dh) > tol * sqrt(sh))) converged = false;
    }
    s->it = it;
    if (converged) s->stop = 2;
}

template <typename T>
cudaError_t apply_dispatch(T* U, float* Ulo, const T* Nm, int NS, long long nstride, int k, long long len, int R, const double* Gpart,
                           int S, double delta, const UnitState* st, double* conv, cudaStream_t s) {
    dim3 g((unsigned)((len + FRO_TT - 1) / FRO_TT), R);
    if (k <= 8)
        fro_apply_kernel<T, 8><<<g, FRO_TT, 0, s>>>(U, Ulo, Nm, NS, nstride, k, len, Gpart, S, delta, st, conv);
    else if (k <= 16)
        fro_apply_kernel<T, 16><<<g, FRO_TT, 0, s>>>(U, Ulo, Nm, NS, nstride, k, len, Gpart, S, delta, st, conv);
    else
        fro_apply_kernel<T, 32><<<g, FRO_TT, 0, s>>>(U, Ulo, Nm, NS, nstride, k, len, Gpart, S, delta, st, conv);
    return cudaGetLastError();
}

__global__ void sum_slices_kernel(float* __restrict__ C, int S, long long pstride, long long len) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < len; i += (long long)gridDim.x * blockDim.x) {
        float v = C[i];
        for (int q = 1; q < S; ++q) v += C[(long long)q * pstride + i];
        C[i] = v;
    }
}

#define FRO_TRY(call)                       \
    do {                                    \
        cudaError_t e__ = (call);           \
        if (e__ != cudaSuccess) {           \
            err = e__;                      \
            goto done;                      \
        }                                   \
    } while (0)

template <typename T>
cudaError_t solve_fro_t(const SolveArgs& a, const void* Xlo, const void* Xtlo, cudaStream_t s, int64_t* launches) {
    constexpr bool F32 = sizeof(T) == 4;
    const int n = a.n, m = a.m, k = a.k, R = a.R;
    const long long Rk = (long long)R * k;
    if (k > 32) return cudaErrorInvalidValue;
    cudaError_t err = cudaSuccess;
    const double delta = F32 ? std::sqrt((double)1.1920929e-07f) : std::sqrt(2.220446049250313e-16);
    const int tilesW = (n + FRO_TT - 1) / FRO_TT, tilesH = (m + FRO_TT - 1) / FRO_TT;
    // split-K slices of the two stacked GEMMs (Float32 / tcgen05 only): partial products side by side in Nbuf
    const int NSH = F32 ? fro_gemm_slices((int)Rk, m, n) : 1, NSW = F32 ? fro_gemm_slices((int)Rk, n, m) : 1;
    const int SW = std::max(1, std::min(64, n / 2048)), SH = std::max(1, std::min(64, m / 2048));  // Gram slices along the long dimension
    T* W = static_cast<T*>(a.W);
    T *Ht = nullptr, *Nbuf = nullptr;
    float *Wlo = nullptr, *Htlo = nullptr;
    double *Gpart = nullptr, *convW = nullptr, *convH = nullptr, *objp = nullptr;
    int *d_active = nullptr, *h_active = nullptr;
    int* errflag = nullptr;  // h_active + 1: barrier time-out site, written by the tcgen05 kernels through mapped pinned memory
    const char* flag_kernel = "fro_gemm_kernel";  // what can raise it in the current phase of the solve, for the error message
    const char* flag_where = "stacked GEMM of an iteration";
    const int nblkObj = (n + 127) / 128;
    std::vector<UnitState> hst((size_t)R);
    bool any_running = false;
    int it = 0;
    // NMFK_TILED_TIMING=1: per-phase device time (the phase names of the KL engine are reused: sums_* = Gram kernels, pass_* =
    // the stacked GEMMs, apply_H / impute = the two apply kernels, clamp_check = the convergence kernel)
    PhaseTimer pt;
    pt.on = getenv("NMFK_TILED_TIMING") != nullptr;
    FRO_TRY(scratch_alloc(&Ht, (size_t)Rk * m * sizeof(T), s));
    FRO_TRY(scratch_alloc(&Nbuf, std::max((size_t)NSH * Rk * m, (size_t)NSW * Rk * n) * sizeof(T), s));
    if (F32) {
        FRO_TRY(scratch_alloc(&Wlo, (size_t)Rk * n * sizeof(float), s));
        FRO_TRY(scratch_alloc(&Htlo, (size_t)Rk * m * sizeof(float), s));
    }
    FRO_TRY(scratch_alloc(&Gpart, (size_t)R * std::max(SW, SH) * k * k * sizeof(double), s));
    FRO_TRY(scratch_alloc(&convW, (size_t)R * tilesW * k * 2 * sizeof(double), s));
    FRO_TRY(scratch_alloc(&convH, (size_t)R * tilesH * k * 2 * sizeof(double), s));
    FRO_TRY(scratch_alloc(&objp, (size_t)R * nblkObj * 2 * sizeof(double), s));
    FRO_TRY(scratch_alloc(&d_active, sizeof(int), s));
    h_active = pinned_flags();
    if (h_active == nullptr) FRO_TRY(cudaErrorMemoryAllocation);
    h_active[0] = h_active[1] = 0;
    errflag = h_active + 1;
    FRO_TRY(cudaMemcpyAsync(hst.data(), a.st, (size_t)R * sizeof(UnitState), cudaMemcpyDeviceToHost, s));
    FRO_TRY(cudaStreamSynchronize(s));
    for (auto& u : hst)
        if (u.stop == 0 && !u.done) {
            any_running = true;
            it = std::max(it, (int)u.it);
        }
    if (any_running) {
        fro_h_to_stack<T><<<dim3((m + 255) / 256, R), 256, 0, s>>>(static_cast<const T*>(a.H), Ht, k, m);
        FRO_TRY(cudaGetLastError());
        ++*launches;
        if (F32) {
            const int blocks = 148 * 8;
            split_lo_kernel<<<blocks, 256, 0, s>>>(reinterpret_cast<const float*>(W), Wlo, Rk * n);
            split_lo_kernel<<<blocks, 256, 0, s>>>(reinterpret_cast<const float*>(Ht), Htlo, Rk * m);
            FRO_TRY(cudaGetLastError());
            *launches += 2;
        }
        const size_t gsmem = (size_t)k * (FRO_TT + 1) * sizeof(T);
        bool need_guard = true;
        while (true) {
            if (need_guard) {  // loop guard on the host every check_every iterations (and before the first one)
                FRO_TRY(cudaMemsetAsync(d_active, 0, sizeof(int), s));
                // `while !converged && t < maxiter`: restarts the convergence kernel has stopped are skipped, the others stop
                // at maxiter or pause at iter_limit; counts the ones that go on
                tiled_guard_kernel<<<(R + 127) / 128, 128, 0, s>>>(a.st, R, it, a.maxiter, INT_MAX, INT_MAX, a.iter_limit, d_active);
                FRO_TRY(cudaGetLastError());
                ++*launches;
                FRO_TRY(cudaMemcpyAsync(h_active, d_active, sizeof(int), cudaMemcpyDeviceToHost, s));
                pt.mark(s, 10);
                FRO_TRY(cudaStreamSynchronize(s));
                if (a.prof) a.prof->harvest();
                pt.harvest();
                if (h_active[1] != 0) goto done;
                if (h_active[0] == 0) break;
                need_guard = false;
                pt.mark(s, -1);
            }
            ++it;
            if (!a.Hfixed) {  // H <- H .* (W'X) ./ (W'W H + d)
                fro_gram_kernel<T><<<dim3(R, SW), 256, gsmem, s>>>(W, k, n, SW, a.st, Gpart);
                FRO_TRY(cudaGetLastError());
                pt.mark(s, 0);
                if (a.prof) a.prof->begin(s);
                if (F32)
                    FRO_TRY(launch_fro_gemm(reinterpret_cast<const float*>(W), Wlo, n, static_cast<const float*>(a.X),
                                            static_cast<const float*>(Xlo), n, reinterpret_cast<float*>(Nbuf), m, (int)Rk, m, n, NSH, Rk * m, errflag, s));
                else
                    FRO_TRY(launch_fro_gemm_f64(reinterpret_cast<const double*>(W), n, static_cast<const double*>(a.X), n,
                                                reinterpret_cast<double*>(Nbuf), m, (int)Rk, m, n, s));
                if (a.prof) a.prof->end(s);
                pt.mark(s, 1);
                FRO_TRY(apply_dispatch<T>(Ht, Htlo, Nbuf, NSH, Rk * m, k, m, R, Gpart, SW, delta, a.st, convH, s));
                pt.mark(s, 3);
                *launches += 3;
            }
            if (!a.Wfixed) {  // W <- W .* (X H') ./ (W H H' + d)
                fro_gram_kernel<T><<<dim3(R, SH), 256, gsmem, s>>>(Ht, k, m, SH, a.st, Gpart);
                FRO_TRY(cudaGetLastError());
                pt.mark(s, 4);
                if (a.prof) a.prof->begin(s);
                if (F32)
                    FRO_TRY(launch_fro_gemm(reinterpret_cast<const float*>(Ht), Htlo, m, static_cast<const float*>(a.Xt),
                                            static_cast<const float*>(Xtlo), m, reinterpret_cast<float*>(Nbuf), n, (int)Rk, n, m, NSW, Rk * n, errflag, s));
                else
                    FRO_TRY(launch_fro_gemm_f64(reinterpret_cast<const double*>(Ht), m, static_cast<const double*>(a.Xt), m,
                                                reinterpret_cast<double*>(Nbuf), n, (int)Rk, n, m, s));
                if (a.prof) a.prof->end(s);
                pt.mark(s, 5);
                FRO_TRY(apply_dispatch<T>(W, Wlo, Nbuf, NSW, Rk * n, k, n, R, Gpart, SH, delta, a.st, convW, s));
                pt.mark(s, 6);
                *launches += 3;
            }
            fro_converge_kernel<<<(R + 127) / 128, 128, 0, s>>>(a.st, R, k, convW, tilesW, convH, tilesH, !a.Wfixed, !a.Hfixed, a.tol, it);
            FRO_TRY(cudaGetLastError());
            pt.mark(s, 9);
            ++*launches;
            if (it % a.check_every == 0 || it >= a.maxiter || (a.iter_limit > 0 && it >= a.iter_limit)) need_guard = true;
        }
        fro_stack_to_h<T><<<dim3((m + 255) / 256, R), 256, 0, s>>>(Ht, static_cast<T*>(a.H), k, m, a.st);
        FRO_TRY(cudaGetLastError());
        ++*launches;
    }
    {
        // post-run objective on the caller's X (normnan(X - W*H), NMFkExecute.jl:791-792) + normalisation (:800-804)
        pt.mark(s, -1);
        // the tensor-core objective kernels of the tiled KL engine when they apply (the scalar kernel takes 39 ms on C3, the
        // tcgen05 one 4 ms), the scalar kernel otherwise
        TiledPassArgs po{};
        po.U = a.W;
        po.V = a.H;
        po.st = a.st;
        po.u_rstride = (long long)n * k;
        po.v_rstride = (long long)k * m;
        po.su_o = 1;
        po.su_a = n;
        po.sv_t = k;
        po.sv_a = 1;
        po.nown = n;
        po.nred = m;
        po.k = k;
        po.R = R;
        po.S = 1;
        po.nblocks = nblkObj;
        po.lambda = a.lambda;
        po.ktmpl = resident_template_k(k);
        po.obj_partials = objp;
        po.obj_weight = 1.0;
        po.obj_restore = 1;
        po.obj_sel = 1;
        po.wait_hint_ns = (32 << 16) | 64;
        bool done_obj = false;
        if (F32) {
            po.D = a.X;
            if (tc_pass_supported(po)) {
                flag_kernel = "tc_pass_kernel";
                flag_where = "post-run objective";
                FRO_TRY(launch_tc_objective(po, errflag, s));
                done_obj = true;
            }
        } else if (k >= 4) {
            po.D = a.Xt;  // the DMMA kernel reads the step-contiguous copy
            FRO_TRY(launch_tiled_dmma_objective(po, s));
            done_obj = true;
        }
        if (!done_obj) {
            dim3 g(nblkObj, R);
            tiled_objective_kernel<T, T><<<g, 128, (size_t)k * 128 * sizeof(T), s>>>(static_cast<const T*>(a.X), n, m, k, W,
                                                                                     static_cast<const T*>(a.H), a.st, (T)a.lambda, 1, 0, 1.0,
                                                                                     WeightRef{nullptr, nullptr, nullptr}, objp);
        }
        FRO_TRY(cudaGetLastError());
        tiled_finish_kernel<T><<<R, 256, 0, s>>>(a.W, a.H, a.st, objp, n, m, k, nblkObj, a.normalize);
        FRO_TRY(cudaGetLastError());
        *launches += 2;
        pt.mark(s, 11);
        FRO_TRY(cudaStreamSynchronize(s));
        if (a.prof) a.prof->harvest();
        pt.harvest();
        pt.report(it, 0);
    }
done:
    // a time-out ends in a trap: the solve has usually failed with that CUDA error already, the flag says where
    if (h_active && h_active[1] != 0) err = solve_timeout(a, err, flag_kernel, flag_where, h_active[1]);
    scratch_free(Ht, s);
    scratch_free(Nbuf, s);
    scratch_free(Wlo, s);
    scratch_free(Htlo, s);
    scratch_free(Gpart, s);
    scratch_free(convW, s);
    scratch_free(convH, s);
    scratch_free(objp, s);
    scratch_free(d_active, s);
    return err;
}

}  // namespace

cudaError_t launch_sum_slices(float* C, int S, long long pstride, long long len, cudaStream_t s) {
    if (S <= 1) return cudaSuccess;
    sum_slices_kernel<<<148 * 8, 256, 0, s>>>(C, S, pstride, len);
    return cudaGetLastError();
}

cudaError_t launch_split_lo(const float* x, float* lo, long long len, cudaStream_t s) {
    split_lo_kernel<<<148 * 8, 256, 0, s>>>(x, lo, len);
    return cudaGetLastError();
}

cudaError_t solve_fro(const SolveArgs& a, int dtype, const void* Xlo, const void* Xtlo, cudaStream_t s, int64_t* launches) {
    return dtype == 1 ? solve_fro_t<double>(a, nullptr, nullptr, s, launches) : solve_fro_t<float>(a, Xlo, Xtlo, s, launches);
}

}  // namespace nmfk
