// Resident KL engine: one CTA runs ONE restart of NMFmultiplicative from start to stop.
//
// Replaces the body of NMFk.NMFmultiplicative (/root/reference/src/NMFkMultiplicative.jl:56-127)
// and the post-run objective + normalisation of execute_singlerun_compute
// (/root/reference/src/NMFkExecute.jl:791-804) for problems whose factors fit in one SM's shared
// memory (BASELINE configs C1, C2): W (n x k) and H^T (m x k) stay in shared memory for the whole
// solve, X (and its transpose) is streamed from L2 with fully coalesced loads, the stop-state
// machine runs on the device, and all R restarts of all k run concurrently as independent CTAs.
// No host synchronisation happens between iterations.
//
// Both half-updates of the KL multiplicative rule are the same operation under transposition:
//     U[o,a] <- U[o,a] * ( sum_t (D[o,t] / (U[o,:].V[t,:])) * V[t,a] ) / ( sum_t V[t,a] )
//   H-update (:67): D = X^T (m x n), U = H^T (m x k), V = W   (n x k)
//   W-update (:70): D = X   (n x m), U = W   (n x k), V = H^T (m x k)   (uses the NEW H)
// A thread owns one "own" index o (its U row and its k partial sums live in registers), walks the
// reduction index t, reads D[o,t] coalesced (lanes = consecutive o) and V[t,:] as a shared-memory
// broadcast.  If fewer own indices than threads exist the reduction range is split in S slices
// that are combined in a fixed order (deterministic: no floating-point atomics anywhere).
#pragma once
#include <cfloat>
#include <climits>
#include <cmath>

#include "nmfk_internal.h"

namespace nmfk {

template <typename T>
struct VecOf;
template <>
struct VecOf<double> {
    using type = double2;
    static constexpr int N = 2;
};
template <>
struct VecOf<float> {
    using type = float4;
    static constexpr int N = 4;
};

template <typename TC, int KP>
__device__ __forceinline__ void load_row(const TC* __restrict__ p, TC (&v)[KP]) {
    using V = typename VecOf<TC>::type;
    constexpr int N = VecOf<TC>::N;
    const V* pv = reinterpret_cast<const V*>(p);
#pragma unroll
    for (int i = 0; i < KP / N; ++i) {
        V t = pv[i];
        if constexpr (N == 2) {
            v[2 * i] = t.x;
            v[2 * i + 1] = t.y;
        } else {
            v[4 * i] = t.x;
            v[4 * i + 1] = t.y;
            v[4 * i + 2] = t.z;
            v[4 * i + 3] = t.w;
        }
    }
}

__device__ __forceinline__ void cp_async_8(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_4(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem));
}
template <typename T>
__device__ __forceinline__ void cp_async_elem(T* smem, const T* gmem) {
    if constexpr (sizeof(T) == 8)
        cp_async_8(smem, gmem);
    else
        cp_async_4(smem, gmem);
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N));
}

// IEEE division kept out of line where it is not on the hot loop (the inlined sequence is ~25
// instructions plus a slow path; the factor-update epilogues would otherwise unroll K copies of it)
template <typename TC>
__device__ __noinline__ TC div_cold(TC a, TC b) {
    return a / b;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// deterministic block-wide sum of one double per thread; result broadcast to all threads.
// red must hold >= 33 doubles.
__device__ __forceinline__ double block_sum(double v, double* red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < nw; ++i) s += red[i];
        red[32] = s;
    }
    __syncthreads();
    return red[32];
}

// den[a] = sum_t V[t][a], a < K  (sum(W; dims=1) / sum(H; dims=2) of :67,:70)
template <typename TC, int K, int KP>
__device__ __forceinline__ void factor_sums(const TC* __restrict__ V, int nred, TC* den) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int a = w; a < K; a += nw) {
        double s = 0.0;
        for (int t = lane; t < nred; t += 32) s += (double)V[(size_t)t * KP + a];
        s = warp_sum(s);
        if (lane == 0) den[a] = (TC)s;
    }
}

// x / p on the hot loop.  The compiler's IEEE division carries a slow-path CALL that splits the
// loop body into basic blocks and serialises the unrolled steps; here the quotient is
// x * (1/p) with 1/p from MUFU.RCP64H + two Newton steps (relative error ~2^-52, well inside the
// 1e-9 parity budget), straight-line.  `unsafe` flags operands outside the range where that is
// valid (zero, subnormal, huge, Inf, NaN): the caller redoes those with the IEEE division so that
// degenerate restarts produce the same Inf/NaN pattern as the reference's `X ./ (W*H)`.
__device__ __forceinline__ double fast_div(double x, double p, bool& unsafe) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(p));
    double e = fma(-p, r, 1.0);
    r = fma(r, e, r);
    e = fma(-p, r, 1.0);
    r = fma(r, e, r);
    const unsigned ex = ((unsigned)__double2hiint(p) >> 20) & 0x7ffu;
    unsafe = (ex < 2u) | (ex > 0x7fbu) | (__double2hiint(p) < 0);
    return x * r;
}
__device__ __forceinline__ float fast_div(float x, float p, bool& unsafe) {
    unsafe = !(p > 1e-37f && p < 1e37f);
    return __fdividef(x, p);
}

// dot product u.v with two interleaved partial sums (halves the dependent-FMA chain)
template <typename TC, int K, int KP>
__device__ __forceinline__ TC dot2(const TC (&u)[KP], const TC (&v)[KP]) {
    TC p0 = (TC)0, p1 = (TC)0;
#pragma unroll
    for (int a = 0; a + 1 < K; a += 2) {
        p0 = fma(u[a], v[a], p0);
        p1 = fma(u[a + 1], v[a + 1], p1);
    }
    if (K & 1) p0 = fma(u[K - 1], v[K - 1], p0);
    return p0 + p1;
}

// One straight-line group of UNR reduction steps: UNR independent dot products, UNR independent
// divisions, then K independent accumulator chains (acc[a] += V[t][a] * x_t / (u . V[t,:])).
// V rows are re-read from shared memory for the accumulation phase instead of being kept live
// (registers are the scarce resource: u and acc already hold 2K values).
// DIV: the quotient of NMF.jl's KL update (Variant KL_DIV), x / (u . V[t,:] + kKlDivDelta).
template <typename TC, int K, int KP, int UNR, bool DIV = false>
__device__ __forceinline__ void kl_group(const TC (&x)[UNR], const TC* const (&vrow)[UNR], const bool (&live)[UNR],
                                         const TC (&u)[KP], TC (&acc)[KP]) {
    TC p[UNR], qv[UNR];
    bool bad = false;
#pragma unroll
    for (int q = 0; q < UNR; ++q) {
        TC v[KP];
        load_row<TC, KP>(vrow[q], v);
        p[q] = dot2<TC, K, KP>(u, v);
        if constexpr (DIV) p[q] += kKlDivDelta<TC>;
    }
#pragma unroll
    for (int q = 0; q < UNR; ++q) {
        bool uq;
        qv[q] = fast_div(x[q], p[q], uq);
        bad |= uq;
    }
    if (bad) {  // rare: operands outside the fast path's range -> IEEE semantics
#pragma unroll
        for (int q = 0; q < UNR; ++q) qv[q] = div_cold<TC>(x[q], p[q]);
    }
#pragma unroll
    for (int q = 0; q < UNR; ++q)
        if (!live[q]) qv[q] = (TC)0;
    if (K > 4) asm volatile("" ::: "memory");  // do not keep the UNR V rows live: re-read them
#pragma unroll
    for (int q = 0; q < UNR; ++q) {
        TC v[KP];
        load_row<TC, KP>(vrow[q], v);
#pragma unroll
        for (int a = 0; a < K; ++a) acc[a] = fma(v[a], qv[q], acc[a]);
    }
}

// Sweep of one thread over reduction indices [t0,t1) for own index o:
//   acc[a] += sum_t V[t][a] * (D[o,t] / (u . V[t,:]))
// UNR consecutive t form one straight-line group: UNR independent dot products, UNR independent
// divisions, then K independent accumulator chains - enough ILP to keep the FP64 pipe busy with
// 4 warps per scheduler.  X values of the next group are prefetched while the current one
// computes.  V rows are re-read from shared memory for the accumulation phase instead of being
// kept live (registers are the scarce resource: u and acc already hold 2K values).
constexpr int kRingGroups = 8;  // cp.async groups in flight per thread (each group = UNR steps)

template <typename TX, typename TC, int K, int KP, bool TRANSPOSED, bool HASNAN, int UNR>
__device__ __forceinline__ void sweep(const TX* __restrict__ dcol, int nown, int o, int t0, int t1, const TC (&u)[KP],
                                      TC (&acc)[KP], const TC* __restrict__ V, bool first_iter, TC lambda,
                                      const TC* __restrict__ ximp, int ldimp, TX* __restrict__ ring, int NT) {
    // ring[(slot*UNR + q)*NT] is private to this thread (the pointer already includes threadIdx.x):
    // X is L2-resident but ~600 cycles away, so every thread keeps (G-1)*UNR of its own X values in
    // flight with cp.async instead of holding them in registers.
    constexpr int G = kRingGroups;
    const int ngroups = (t1 - t0 + UNR - 1) / UNR;
    auto issue = [&](int g) {
#pragma unroll
        for (int q = 0; q < UNR; ++q) {
            const int t = t0 + g * UNR + q;
            if (t < t1) cp_async_elem<TX>(ring + ((g & (G - 1)) * UNR + q) * NT, dcol + (size_t)t * nown);
        }
    };
#pragma unroll
    for (int g = 0; g < G - 1; ++g) {
        if (g < ngroups) issue(g);
        cp_async_commit();
    }
    for (int g = 0; g < ngroups; ++g) {
        cp_async_wait<G - 2>();  // group g has landed
        const int t = t0 + g * UNR;
        TC x[UNR];
        const TC* vrow[UNR];
        bool live[UNR];
#pragma unroll
        for (int q = 0; q < UNR; ++q) {
            live[q] = (t + q < t1);
            const TX xr = live[q] ? ring[((g & (G - 1)) * UNR + q) * NT] : (TX)1;
            x[q] = (TC)xr;
            if (HASNAN) {
                if (xr != xr)
                    x[q] = first_iter ? lambda
                                      : ximp[TRANSPOSED ? ((size_t)(t + q) + (size_t)o * ldimp)
                                                        : ((size_t)o + (size_t)(t + q) * ldimp)];
            }
            vrow[q] = V + (size_t)(live[q] ? (t + q) : t) * KP;  // tail: a valid row, contribution zeroed
        }
        // refill the slot consumed in the PREVIOUS iteration (its values are already in registers)
        if (g + G - 1 < ngroups) issue(g + G - 1);
        cp_async_commit();
        kl_group<TC, K, KP, UNR>(x, vrow, live, u, acc);
    }
    cp_async_wait<0>();
}

// One half-update.  D is column-major with leading dimension = nown (own index contiguous).
// TRANSPOSED tells how to address the imputation buffer (always stored in X layout, ld = n).
template <typename TX, typename TC, int K, int KP, bool TRANSPOSED, bool HASNAN>
__device__ __forceinline__ void half_update(const TX* __restrict__ D, int nown, int nred, int kact,
                                            TC* __restrict__ U, const TC* __restrict__ V, const TC* __restrict__ den,
                                            TC* __restrict__ scr, bool first_iter, TC lambda,
                                            const TC* __restrict__ ximp, int ldimp, TX* __restrict__ ring) {
    const int tid = threadIdx.x, NT = blockDim.x;
    int S = NT / nown;
    if (S > nred) S = nred;
    if (S < 1) S = 1;
    constexpr int UNR = 2;
    if (S == 1) {
        // every thread sweeps the whole reduction range for own rows tid, tid+NT, ...
        for (int o = tid; o < nown; o += NT) {
            TC u[KP], acc[KP];
            load_row<TC, KP>(U + (size_t)o * KP, u);
#pragma unroll
            for (int a = 0; a < KP; ++a) acc[a] = (TC)0;
            sweep<TX, TC, K, KP, TRANSPOSED, HASNAN, UNR>(D + o, nown, o, 0, nred, u, acc, V, first_iter, lambda, ximp,
                                                          ldimp, ring + tid, NT);
            // (U .* acc) ./ den : Julia's left-to-right broadcast of `H .* (...) ./ sum`
            TC* urow = U + (size_t)o * KP;
#pragma unroll
            for (int a = 0; a < K; ++a)
                if (a < kact) urow[a] = div_cold<TC>(u[a] * acc[a], den[a]);
        }
        __syncthreads();
        return;
    }
    // S > 1: thread = (own index o, slice s); slices combined in order through shared memory
    const int s = tid / nown, o = tid - s * nown;
    const bool active = s < S;
    TC u[KP], acc[KP];
#pragma unroll
    for (int a = 0; a < KP; ++a) acc[a] = (TC)0;
    if (active) {
        load_row<TC, KP>(U + (size_t)o * KP, u);
        const int t0 = (int)(((long long)nred * s) / S), t1 = (int)(((long long)nred * (s + 1)) / S);
        sweep<TX, TC, K, KP, TRANSPOSED, HASNAN, UNR>(D + o, nown, o, t0, t1, u, acc, V, first_iter, lambda, ximp,
                                                      ldimp, ring + tid, NT);
        if (s > 0) {
            TC* dst = scr + ((size_t)(s - 1) * nown + o) * KP;
#pragma unroll
            for (int a = 0; a < K; ++a) dst[a] = acc[a];
        }
    }
    __syncthreads();
    if (active && s == 0) {
        for (int ss = 1; ss < S; ++ss) {
            const TC* src = scr + ((size_t)(ss - 1) * nown + o) * KP;
#pragma unroll
            for (int a = 0; a < K; ++a) acc[a] += src[a];
        }
        TC* urow = U + (size_t)o * KP;
#pragma unroll
        for (int a = 0; a < K; ++a)
            if (a < kact) urow[a] = div_cold<TC>(u[a] * acc[a], den[a]);
    }
    __syncthreads();
}

// sum over non-NaN entries of ((x - (W*H)) * weight)^2 and of (x - W*H)^2.
// RESTORE: x == lambda (a substituted zero) counts as 0, i.e. the caller's restored X
// (NMFkMultiplicative.jl:123-125, NMFkExecute.jl:791-792); otherwise the lambda-substituted X of :74.
template <typename TX, typename TC, int K, int KP, bool RESTORE>
__device__ __forceinline__ double2 objective_pass(const TX* __restrict__ X, int n, int m, const TC* __restrict__ Ws,
                                                  const TC* __restrict__ Hs, TC lambda, double weight, double* red) {
    double sw = 0.0, s1 = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        TC u[KP];
        load_row<TC, KP>(Ws + (size_t)i * KP, u);
        for (int j = 0; j < m; ++j) {
            const TX xr = __ldg(X + (size_t)i + (size_t)j * n);
            if (xr != xr) continue;  // [.!inan]
            TC x = (TC)xr;
            if (RESTORE && x == lambda) x = (TC)0;
            TC v[KP];
            load_row<TC, KP>(Hs + (size_t)j * KP, v);
            TC p = (TC)0;
#pragma unroll
            for (int a = 0; a < K; ++a) p = fma(u[a], v[a], p);
            const double e = (double)(x - p);
            s1 = fma(e, e, s1);
            const double ew = e * weight;
            sw = fma(ew, ew, sw);
        }
    }
    double2 out;
    out.x = block_sum(sw, red);
    out.y = block_sum(s1, red);
    return out;
}

// X[inan] = (W*H)[inan]  (NMFkMultiplicative.jl:72), into the per-restart imputation buffer
template <typename TX, typename TC, int K, int KP>
__device__ __forceinline__ void impute_pass(const TX* __restrict__ X, int n, int m, const TC* __restrict__ Ws,
                                            const TC* __restrict__ Hs, TC* __restrict__ ximp) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        TC u[KP];
        load_row<TC, KP>(Ws + (size_t)i * KP, u);
        for (int j = 0; j < m; ++j) {
            const TX xr = __ldg(X + (size_t)i + (size_t)j * n);
            if (xr == xr) continue;
            TC v[KP];
            load_row<TC, KP>(Hs + (size_t)j * KP, v);
            TC p = (TC)0;
#pragma unroll
            for (int a = 0; a < K; ++a) p = fma(u[a], v[a], p);
            ximp[(size_t)i + (size_t)j * n] = p;
        }
    }
    __syncthreads();
}

struct ResidentSmem {
    // byte offsets of the carve-up; computed identically on host (resident_smem_bytes) and device
    size_t off_W, off_H, off_den, off_scr, off_red, off_idx, off_first, off_ring, total;
    __host__ __device__ static ResidentSmem make(int n, int m, int KP, size_t szTC, size_t szTX, int nthreads) {
        ResidentSmem r;
        auto al = [](size_t x) { return (x + 15) & ~size_t(15); };
        size_t o = 0;
        r.off_W = o;
        o = al(o + (size_t)n * KP * szTC);
        r.off_H = o;
        o = al(o + (size_t)m * KP * szTC);
        r.off_den = o;
        o = al(o + (size_t)KP * szTC);
        r.off_scr = o;
        // cross-slice partials: only when a pass has fewer own indices than threads (S > 1)
        size_t scr = 0;
        {
            int S = nthreads / m;  // H-update: own = m, reduction = n
            if (S > n) S = n;
            if (S > 1) scr = (size_t)(S - 1) * m * KP;
            S = nthreads / n;  // W-update: own = n, reduction = m
            if (S > m) S = m;
            if (S > 1 && (size_t)(S - 1) * n * KP > scr) scr = (size_t)(S - 1) * n * KP;
        }
        o = al(o + scr * szTC);
        r.off_red = o;
        o = al(o + 40 * sizeof(double));
        r.off_idx = o;
        o = al(o + (size_t)m * sizeof(int));
        r.off_first = o;
        o = al(o + (size_t)(KP + 4) * sizeof(int));
        r.off_ring = o;
        o = al(o + (size_t)kRingGroups * 2 * nthreads * szTX);  // UNR = 2 steps per group
        r.total = o;
        return r;
    }
};

template <typename TX, typename TC, int K, bool HASNAN>
__global__ void __launch_bounds__(resident_threads(K), 1) kl_resident_kernel(const SolveArgs a) {
    constexpr int VEC = VecOf<TC>::N;
    constexpr int KP = (K + VEC - 1) / VEC * VEC;
    extern __shared__ __align__(16) unsigned char smem[];
    const int n = a.n, m = a.m, k = a.k;
    const int r = blockIdx.x;
    const int tid = threadIdx.x, NT = blockDim.x;
    UnitState* stg = a.st + r;
    if (stg->done) return;  // finished in an earlier (resumed) solve
    if (a.iter_limit > 0 && a.iter_limit < a.maxiter && stg->it >= a.iter_limit) return;  // paused beyond this launch

    const ResidentSmem L = ResidentSmem::make(n, m, KP, sizeof(TC), sizeof(TX), NT);
    TC* Ws = reinterpret_cast<TC*>(smem + L.off_W);
    TC* Hs = reinterpret_cast<TC*>(smem + L.off_H);
    TC* den = reinterpret_cast<TC*>(smem + L.off_den);
    TC* scr = reinterpret_cast<TC*>(smem + L.off_scr);
    double* red = reinterpret_cast<double*>(smem + L.off_red);
    int* idx = reinterpret_cast<int*>(smem + L.off_idx);
    int* first = reinterpret_cast<int*>(smem + L.off_first);
    TX* ring = reinterpret_cast<TX*>(smem + L.off_ring);

    const TX* X = static_cast<const TX*>(a.X);
    const TX* Xt = static_cast<const TX*>(a.Xt);
    TC* Wg = static_cast<TC*>(a.W) + (size_t)r * n * k;
    TC* Hg = static_cast<TC*>(a.H) + (size_t)r * k * m;
    int* canon_old = a.canon + (size_t)r * m;
    TC* ximp = HASNAN ? static_cast<TC*>(a.ximp) + (size_t)r * n * m : nullptr;
    constexpr bool has_nan = HASNAN;
    const TC lambda = (TC)a.lambda;

    // ---- load factors (column-major global -> row-of-k shared), zero the padding ----
    for (int e = tid; e < n * KP; e += NT) Ws[e] = (TC)0;
    for (int e = tid; e < m * KP; e += NT) Hs[e] = (TC)0;
    __syncthreads();
    for (int e = tid; e < n * k; e += NT) {
        const int i = e % n, c = e / n;
        Ws[(size_t)i * KP + c] = Wg[e];
    }
    for (int e = tid; e < k * m; e += NT) {
        const int c = e % k, j = e / k;
        Hs[(size_t)j * KP + c] = Hg[e];
    }
    __syncthreads();

    // every thread carries an identical copy of the scalar state (uniform control flow)
    int it = stg->it, bad = stg->bad, re = stg->re, inc = stg->inc, has_cons = stg->has_cons;
    double best = stg->best, obj_chk = stg->obj_chk;
    int stop = 0;
    __syncthreads();

    if (has_nan && it > 0) impute_pass<TX, TC, K, KP>(X, n, m, Ws, Hs, ximp);  // resume: rebuild X[inan]

    while (true) {
        // while iters < maxiter && baditers < maxbaditers && reattempts < maxreattempts  (:64)
        if (it >= a.maxiter) {
            stop = 1;
            break;
        }
        if (bad >= a.maxbad) {
            stop = 5;
            break;
        }
        if (re >= a.maxre) {
            stop = 3;
            break;
        }
        if (a.iter_limit > 0 && it >= a.iter_limit) break;  // paused
        ++it;
        const bool first_iter = (it == 1);
        if (!a.Hfixed) {  // :66-68
            factor_sums<TC, K, KP>(Ws, n, den);
            __syncthreads();
            half_update<TX, TC, K, KP, true, HASNAN>(Xt, m, n, k, Hs, Ws, den, scr, first_iter, lambda, ximp, n, ring);
        }
        if (!a.Wfixed) {  // :69-71
            factor_sums<TC, K, KP>(Hs, m, den);
            __syncthreads();
            half_update<TX, TC, K, KP, false, HASNAN>(X, n, m, k, Ws, Hs, den, scr, first_iter, lambda, ximp, n, ring);
        }
        if (has_nan) impute_pass<TX, TC, K, KP>(X, n, m, Ws, Hs, ximp);  // :72
        if (it % a.check_every == 0) {                                    // :73
            const double2 ob = objective_pass<TX, TC, K, KP, false>(X, n, m, Ws, Hs, lambda, a.weight, red);
            const double obj = ob.x;  // :74
            obj_chk = obj;
            if (obj < a.tol) {  // :75-78
                stop = 2;
                break;
            }
            if (obj < best) {  // :79-89
                if ((best - obj) < a.tolOF)
                    ++bad;
                else
                    bad = 0;
                best = obj;
            } else {
                ++bad;
            }
            if (bad >= a.maxbad) {  // :90-95
                ++re;
                bad = 0;
            }
            // H = max.(H, eps()); W = max.(W, eps())  (:99-100)
            const TC epsc = (TC)a.eps_clamp;
            for (int e = tid; e < n * KP; e += NT) {
                const int c = e % KP;
                if (c < k) {
                    const TC v = Ws[e];
                    Ws[e] = (v != v) ? v : (v < epsc ? epsc : v);
                }
            }
            for (int e = tid; e < m * KP; e += NT) {
                const int c = e % KP;
                if (c < k) {
                    const TC v = Hs[e];
                    Hs[e] = (v != v) ? v : (v < epsc ? epsc : v);
                }
            }
            if (tid < KP + 1) first[tid] = INT_MAX;
            __syncthreads();
            // index[q] = argmin(H[:, q]) (:101-103): first minimum, NaN counts as smallest
            for (int j = tid; j < m; j += NT) {
                const TC* h = Hs + (size_t)j * KP;
                TC bv = h[0];
                int bi = 0;
                for (int c = 1; c < k; ++c) {
                    const TC v = h[c];
                    const bool take = (bv != bv) ? false : ((v != v) ? true : (v < bv));
                    if (take) {
                        bv = v;
                        bi = c;
                    }
                }
                idx[j] = bi;
                atomicMin(&first[bi], j);
            }
            __syncthreads();
            // cons[i,j] = (index[i] == index[j]) (:105) <=> canonical label = first column with that argmin
            int same = 1;
            for (int j = tid; j < m; j += NT) {
                const int c = first[idx[j]];
                if (!has_cons || canon_old[j] != c) same = 0;
                idx[j] = c;
            }
            same = __syncthreads_and(same);
            if (same)  // :106-111
                ++inc;
            else
                inc = 0;
            if (inc > a.stopconv) {  // :112-115
                stop = 4;
                break;
            }
            for (int j = tid; j < m; j += NT) canon_old[j] = idx[j];  // consold = cons (:116)
            has_cons = 1;
            __syncthreads();
        }
    }

    // ---- epilogue ----
    double obj_ssq = stg->obj_ssq, obj_norm = stg->obj_norm;
    int done = 0;
    if (stop != 0) {
        // X[izero] = 0; X[inan] = NaN; objvalue = sum((((X - W*H) .* weight)[.!inan]).^2)  (:123-125)
        // E = X - W*H; objvalue = normnan(E)  (NMFkExecute.jl:791-792)
        const double2 ob = objective_pass<TX, TC, K, KP, true>(X, n, m, Ws, Hs, lambda, a.weight, red);
        obj_ssq = ob.x;
        obj_norm = sqrt(ob.y);
        if (a.normalize == 1) {  // total = sum(H; dims=2); W .*= total'; H ./= total  (NMFkExecute.jl:800-804)
            factor_sums<TC, K, KP>(Hs, m, den);
            __syncthreads();
            for (int e = tid; e < n * KP; e += NT) {
                const int c = e % KP;
                if (c < k) Ws[e] = Ws[e] * den[c];
            }
            for (int e = tid; e < m * KP; e += NT) {
                const int c = e % KP;
                if (c < k) Hs[e] = div_cold<TC>(Hs[e], den[c]);
            }
        } else if (a.normalize == 2) {  // total = sum(W; dims=1); W ./= total; H .*= total'  (:796-799)
            factor_sums<TC, K, KP>(Ws, n, den);
            __syncthreads();
            for (int e = tid; e < n * KP; e += NT) {
                const int c = e % KP;
                if (c < k) Ws[e] = div_cold<TC>(Ws[e], den[c]);
            }
            for (int e = tid; e < m * KP; e += NT) {
                const int c = e % KP;
                if (c < k) Hs[e] = Hs[e] * den[c];
            }
        }
        done = 1;
        __syncthreads();
    }
    for (int e = tid; e < n * k; e += NT) {
        const int i = e % n, c = e / n;
        Wg[e] = Ws[(size_t)i * KP + c];
    }
    for (int e = tid; e < k * m; e += NT) {
        const int c = e % k, j = e / k;
        Hg[e] = Hs[(size_t)j * KP + c];
    }
    if (tid == 0) {
        stg->it = it;
        stg->bad = bad;
        stg->re = re;
        stg->inc = inc;
        stg->stop = stop;
        stg->has_cons = has_cons;
        stg->done = done;
        stg->best = best;
        stg->obj_chk = obj_chk;
        stg->obj_ssq = obj_ssq;
        stg->obj_norm = obj_norm;
    }
}

template <typename TX, typename TC, int K>
cudaError_t launch_resident_k(const SolveArgs& a, cudaStream_t s) {
    constexpr int VEC = VecOf<TC>::N;
    constexpr int KP = (K + VEC - 1) / VEC * VEC;
    constexpr int NT = resident_threads(K);
    const size_t smem = ResidentSmem::make(a.n, a.m, KP, sizeof(TC), sizeof(TX), NT).total;
    cudaError_t e;
    if (a.has_nan) {
        e = cudaFuncSetAttribute(kl_resident_kernel<TX, TC, K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem);
        if (e != cudaSuccess) return e;
        kl_resident_kernel<TX, TC, K, true><<<a.R, NT, smem, s>>>(a);
    } else {
        e = cudaFuncSetAttribute(kl_resident_kernel<TX, TC, K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem);
        if (e != cudaSuccess) return e;
        kl_resident_kernel<TX, TC, K, false><<<a.R, NT, smem, s>>>(a);
    }
    return cudaGetLastError();
}

#define NMFK_DISPATCH_K(FN, TX, TC, KT, ...)                      \
    switch (KT) {                                                 \
        case 1: return FN<TX, TC, 1>(__VA_ARGS__);                \
        case 2: return FN<TX, TC, 2>(__VA_ARGS__);                \
        case 3: return FN<TX, TC, 3>(__VA_ARGS__);                \
        case 4: return FN<TX, TC, 4>(__VA_ARGS__);                \
        case 5: return FN<TX, TC, 5>(__VA_ARGS__);                \
        case 6: return FN<TX, TC, 6>(__VA_ARGS__);                \
        case 7: return FN<TX, TC, 7>(__VA_ARGS__);                \
        case 8: return FN<TX, TC, 8>(__VA_ARGS__);                \
        case 9: return FN<TX, TC, 9>(__VA_ARGS__);                \
        case 10: return FN<TX, TC, 10>(__VA_ARGS__);              \
        case 11: return FN<TX, TC, 11>(__VA_ARGS__);              \
        case 12: return FN<TX, TC, 12>(__VA_ARGS__);              \
        case 16: return FN<TX, TC, 16>(__VA_ARGS__);              \
        case 20: return FN<TX, TC, 20>(__VA_ARGS__);              \
        case 24: return FN<TX, TC, 24>(__VA_ARGS__);              \
        case 32: return FN<TX, TC, 32>(__VA_ARGS__);              \
        default: return cudaErrorInvalidValue;                    \
    }

}  // namespace nmfk
