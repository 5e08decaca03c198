// Tiled KL engine: the same multiplicative updates as kl_resident.cuh for problems whose factors
// do NOT fit in one SM's shared memory (BASELINE configs C3, C4, C5).
//
// Replaces the loop body of NMFk.NMFmultiplicative (/root/reference/src/NMFkMultiplicative.jl:64-118)
// with one kernel launch per half-update for ALL restarts of a batch:
//   grid = slices x own-blocks x R, restart index fastest, so the CTAs that are resident at the
//   same time work on the SAME block of X for different restarts: X is fetched from HBM once and
//   re-read from the 126 MB L2 by the other restarts.
//   A CTA owns 256 consecutive "own" indices (rows of W, or columns of H) of one restart and walks
//   the reduction index in chunks of TCH: the X tile (TCH x 256) and the other factor's rows
//   (TCH x k) are staged into shared memory by a 3-stage cp.async pipeline (every thread fetches
//   exactly the X elements it will consume, fully coalesced), the two thin products and the
//   element-wise division happen in registers.
//   If the own dimension alone cannot fill the GPU the reduction range is split in slices whose
//   partial sums are combined in slice order by a second kernel (deterministic; it is also the
//   hook for row-sharding X across GPUs: all-reduce the partials between the two kernels).
// The stop-state machine (tolOF / baditers / reattempts / co-clustering consistency, :73-116) runs
// in a per-restart check kernel every `check_every` iterations; finished restarts are skipped by
// every later launch.
#pragma once
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <chrono>
#include <vector>

#include "kl_resident.cuh"  // load_row, warp_sum, block_sum, div_cold, VecOf
#include "kl_tiled_args.h"

namespace nmfk {

constexpr int kTiledThreads = 256;
constexpr int kTiledStages = 3;

template <typename TX>
struct TiledCfg {
    static constexpr int TCH = sizeof(TX) == 8 ? 16 : 32;  // reduction indices per pipeline stage
};


// DIV (HASNAN = false only): the quotient of NMF.jl's KL update (Variant KL_DIV), x / (p + delta); a.den already holds the sums
// + delta
template <typename TX, typename TC, int K, bool HASNAN, bool DIV = false>
__global__ void __launch_bounds__(kTiledThreads, (K <= 12 ? 2 : 1)) tiled_pass_kernel(const TiledPassArgs a) {
    constexpr int VEC = VecOf<TC>::N;
    constexpr int KP = (K + VEC - 1) / VEC * VEC;
    constexpr int TCH = TiledCfg<TX>::TCH;
    constexpr int NT = kTiledThreads;
    constexpr int ST = kTiledStages;
    extern __shared__ __align__(16) unsigned char smem[];
    TC* Vs = reinterpret_cast<TC*>(smem);                                      // [ST][TCH][KP]
    TX* Ds = reinterpret_cast<TX*>(smem + (size_t)ST * TCH * KP * sizeof(TC));  // [ST][TCH][NT]

    const int tid = threadIdx.x;
    const int r = blockIdx.x % a.R;
    const int rest = blockIdx.x / a.R;
    const int ob = rest % a.nblocks;
    const int slice = rest / a.nblocks;
    if (a.st[r].stop != 0) return;  // finished restarts are frozen
    const int k = a.k;
    const int o = ob * NT + tid;
    const bool valid = o < a.nown;
    const int t_begin = (int)(((long long)a.nred * slice) / a.S);
    const int t_end = (int)(((long long)a.nred * (slice + 1)) / a.S);
    const int nchunks = (t_end - t_begin + TCH - 1) / TCH;

    const TX* D = static_cast<const TX*>(a.D);
    TC* U = static_cast<TC*>(a.U) + (long long)r * a.u_rstride;
    const TC* V = static_cast<const TC*>(a.V) + (long long)r * a.v_rstride;
    const TC* ximp = HASNAN ? static_cast<const TC*>(a.ximp) + (long long)r * a.nown * a.nred : nullptr;
    const TC lambda = (TC)a.lambda;

    // padding columns of the broadcast rows stay zero for the whole kernel
    for (int e = tid; e < ST * TCH * KP; e += NT) Vs[e] = (TC)0;
    __syncthreads();

    auto issue = [&](int chunk) {
        const int stage = chunk % ST;
        const int t0 = t_begin + chunk * TCH;
        const int cnt = min(TCH, t_end - t0);
        TC* vs = Vs + (size_t)stage * TCH * KP;
        TX* ds = Ds + (size_t)stage * TCH * NT;
        // the other factor's rows t0..t0+cnt: coalesced along whichever index is contiguous
        if (a.sv_t == 1) {
            for (int e = tid; e < cnt * k; e += NT) {
                const int tl = e % cnt, c = e / cnt;
                cp_async_elem<TC>(vs + tl * KP + c, V + (long long)(t0 + tl) + (long long)c * a.sv_a);
            }
        } else {
            for (int e = tid; e < cnt * k; e += NT) {
                const int c = e % k, tl = e / k;
                cp_async_elem<TC>(vs + tl * KP + c, V + (long long)(t0 + tl) * a.sv_t + c);
            }
        }
        // the X elements this thread will consume
        if (valid) {
            const TX* src = D + (long long)o + (long long)t0 * a.nown;
#pragma unroll 4
            for (int tl = 0; tl < cnt; ++tl) cp_async_elem<TX>(ds + tl * NT + tid, src + (long long)tl * a.nown);
        }
    };

    TC u[KP], acc[KP];
#pragma unroll
    for (int c = 0; c < KP; ++c) {
        u[c] = (TC)0;
        acc[c] = (TC)0;
    }
    if (valid) {
#pragma unroll
        for (int c = 0; c < K; ++c)
            if (c < k) u[c] = U[(long long)o * a.su_o + (long long)c * a.su_a];
    }

#pragma unroll
    for (int c = 0; c < ST - 1; ++c) {
        if (c < nchunks) issue(c);
        cp_async_commit();
    }
    for (int chunk = 0; chunk < nchunks; ++chunk) {
        cp_async_wait<ST - 2>();
        __syncthreads();  // chunk's data visible to all; everyone is done with the stage refilled below
        if (chunk + ST - 1 < nchunks) issue(chunk + ST - 1);
        cp_async_commit();
        const int stage = chunk % ST;
        const int t0 = t_begin + chunk * TCH;
        const int cnt = min(TCH, t_end - t0);
        const TC* vs = Vs + (size_t)stage * TCH * KP;
        const TX* ds = Ds + (size_t)stage * TCH * NT + tid;
        if (valid) {
            constexpr int UNR = 2;
            for (int tl = 0; tl < cnt; tl += UNR) {
                TC x[UNR];
                const TC* vrow[UNR];
                bool live[UNR];
#pragma unroll
                for (int q = 0; q < UNR; ++q) {
                    live[q] = (tl + q < cnt);
                    const int tq = live[q] ? (tl + q) : tl;
                    const TX xr = ds[tq * NT];
                    x[q] = (TC)xr;
                    if (HASNAN) {
                        if (xr != xr)
                            x[q] = a.first_iter ? lambda
                                                : ximp[a.transposed ? ((long long)(t0 + tq) + (long long)o * a.ldimp)
                                                                    : ((long long)o + (long long)(t0 + tq) * a.ldimp)];
                    }
                    vrow[q] = vs + tq * KP;
                }
                kl_group<TC, K, KP, UNR, DIV>(x, vrow, live, u, acc);
            }
        }
    }
    cp_async_wait<0>();
    if (!valid) return;
    if (a.partial == nullptr) {
        const TC* den = static_cast<const TC*>(a.den) + (long long)r * kTiledMaxK;
#pragma unroll
        for (int c = 0; c < K; ++c)
            if (c < k) U[(long long)o * a.su_o + (long long)c * a.su_a] = div_cold<TC>(u[c] * acc[c], den[c]);
    } else {
        TC* dst = static_cast<TC*>(a.partial) + (((long long)slice * a.R + r) * a.nown + o) * K;
#pragma unroll
        for (int c = 0; c < K; ++c) dst[c] = acc[c];
    }
}

// U[o,a] <- (U[o,a] * sum_slices partial) / den, slices added in order.
// red != nullptr (row-sharded X): the slice sum is written to red[r][o][K] instead (the numerators of
// this rank's rows; all-reduced across ranks before tiled_apply_kernel finishes the update).
template <typename TC, int K>
__global__ void tiled_combine_kernel(const TiledPassArgs a, TC* __restrict__ red) {
    const int r = blockIdx.y;
    if (a.st[r].stop != 0) return;
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= a.nown) return;
    TC* U = static_cast<TC*>(a.U) + (long long)r * a.u_rstride;
    const TC* den = static_cast<const TC*>(a.den) + (long long)r * kTiledMaxK;
    TC acc[K];
#pragma unroll
    for (int c = 0; c < K; ++c) acc[c] = (TC)0;
    for (int s = 0; s < a.S; ++s) {
        const TC* src = static_cast<const TC*>(a.partial) + (((long long)s * a.R + r) * a.nown + o) * K;
#pragma unroll
        for (int c = 0; c < K; ++c) acc[c] += src[c];
    }
    if (red != nullptr) {
        TC* dst = red + ((long long)r * a.nown + o) * K;
#pragma unroll
        for (int c = 0; c < K; ++c) dst[c] = acc[c];
        return;
    }
#pragma unroll
    for (int c = 0; c < K; ++c)
        if (c < a.k) {
            const long long idx = (long long)o * a.su_o + (long long)c * a.su_a;
            U[idx] = div_cold<TC>(U[idx] * acc[c], den[c]);
        }
}

// row-sharded X: U[o,a] <- (U[o,a] * red[r][o][a]) / den[r][a] with the all-reduced numerators / sums
template <typename TC, int K>
__global__ void tiled_apply_kernel(const TiledPassArgs a, const TC* __restrict__ red) {
    const int r = blockIdx.y;
    if (a.st[r].stop != 0) return;
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= a.nown) return;
    TC* U = static_cast<TC*>(a.U) + (long long)r * a.u_rstride;
    const TC* den = static_cast<const TC*>(a.den) + (long long)r * kTiledMaxK;
    const TC* src = red + ((long long)r * a.nown + o) * K;
#pragma unroll
    for (int c = 0; c < K; ++c)
        if (c < a.k) {
            const long long idx = (long long)o * a.su_o + (long long)c * a.su_a;
            U[idx] = div_cold<TC>(U[idx] * src[c], den[c]);
        }
}

// row-sharded X: obj2[r][0..1] = sum over this rank's row blocks of the objective partials
static __global__ void tiled_objsum_kernel(const double* __restrict__ partials, int nblk, int R, double* __restrict__ obj2) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    double a0 = 0.0, a1 = 0.0;
    for (int b = 0; b < nblk; ++b) {
        a0 += partials[((long long)r * nblk + b) * 2];
        a1 += partials[((long long)r * nblk + b) * 2 + 1];
    }
    obj2[2 * r] = a0;
    obj2[2 * r + 1] = a1;
}

// den[r][a] = sum_t V_r[t,a] : grid (k, R), fixed-order block reduction
template <typename TC>
__global__ void __launch_bounds__(256) tiled_sums_kernel(const void* Vv, long long v_rstride, long long sv_t,
                                                         long long sv_a, int nred, const UnitState* st, void* denv) {
    __shared__ double red[40];
    const int c = blockIdx.x, r = blockIdx.y;
    if (st[r].stop != 0) return;
    const TC* V = static_cast<const TC*>(Vv) + (long long)r * v_rstride + (long long)c * sv_a;
    // four independent chains keep four loads in flight per thread (fixed order: deterministic)
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const int NT = blockDim.x;
    int t = threadIdx.x;
    for (; t + 3 * NT < nred; t += 4 * NT) {
        s0 += (double)V[(long long)t * sv_t];
        s1 += (double)V[(long long)(t + NT) * sv_t];
        s2 += (double)V[(long long)(t + 2 * NT) * sv_t];
        s3 += (double)V[(long long)(t + 3 * NT) * sv_t];
    }
    for (; t < nred; t += NT) s0 += (double)V[(long long)t * sv_t];
    double s = (s0 + s1) + (s2 + s3);
    s = block_sum(s, red);
    if (threadIdx.x == 0) static_cast<TC*>(denv)[(long long)r * kTiledMaxK + c] = (TC)s;
}

// sum over non-NaN entries of ((x - W_r H_r) w)^2 and (x - W_r H_r)^2 for 128 rows x all columns;
// partials[(r*nblk + b)*2 + {0,1}].  only_running: skip finished restarts (the :74 check);
// restore: substituted zeros count as 0 (final objective).
template <typename TX, typename TC>
__global__ void __launch_bounds__(128) tiled_objective_kernel(const TX* __restrict__ X, int n, int m, int k,
                                                              const TC* __restrict__ Wst, const TC* __restrict__ Hst,
                                                              const UnitState* st, TC lambda, int restore,
                                                              int only_running, double weight, const WeightRef wref,
                                                              double* __restrict__ partials) {
    extern __shared__ unsigned char smraw[];
    TC* Ws = reinterpret_cast<TC*>(smraw);  // [k][128]
    __shared__ double red[2][4];
    const int r = blockIdx.y, b = blockIdx.x, tid = threadIdx.x;
    const bool stopped = st[r].stop != 0;
    if (only_running ? stopped : (st[r].done != 0 || !stopped)) return;
    const TC* W = Wst + (long long)r * n * k;
    const TC* H = Hst + (long long)r * k * m;
    const int i = b * 128 + tid;
    for (int c = 0; c < k; ++c) Ws[c * 128 + tid] = (i < n) ? W[(long long)i + (long long)c * n] : (TC)0;
    __syncthreads();
    double sw = 0.0, s1 = 0.0;
    const bool wany = wref.any();
    if (i < n) {
        for (int j = 0; j < m; ++j) {
            const TX xr = X[(long long)i + (long long)j * n];
            if (xr != xr) continue;
            TC x = (TC)xr;
            if (restore && x == lambda) x = (TC)0;
            const TC* h = H + (long long)j * k;
            TC p = (TC)0;
            for (int c = 0; c < k; ++c) p = fma(Ws[c * 128 + tid], __ldg(h + c), p);
            const double e = (double)(x - p);
            s1 = fma(e, e, s1);
            const double ew = e * (wany ? weight_at<TX>(wref, weight, i, j, n) : weight);
            sw = fma(ew, ew, sw);
        }
    }
    sw = warp_sum(sw);
    s1 = warp_sum(s1);
    if ((tid & 31) == 0) {
        red[0][tid >> 5] = sw;
        red[1][tid >> 5] = s1;
    }
    __syncthreads();
    if (tid == 0) {
        double a0 = 0.0, a1 = 0.0;
        for (int w = 0; w < 4; ++w) {
            a0 += red[0][w];
            a1 += red[1][w];
        }
        partials[((long long)r * gridDim.x + b) * 2] = a0;
        partials[((long long)r * gridDim.x + b) * 2 + 1] = a1;
    }
}

// the rows of W a block of tiled_objective_kernel keeps in shared memory: with the static sums above 48 KB (Float64, k >= 48)
// only with the attribute
template <typename TX, typename TC>
cudaError_t tiled_objective_smem(int k) {
    const size_t smem = (size_t)k * 128 * sizeof(TC);
    if (smem + sizeof(double) * 2 * 4 <= 48 * 1024) return cudaSuccess;
    return cudaFuncSetAttribute(tiled_objective_kernel<TX, TC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

// X[inan] = (W*H)[inan] (:72) for every running restart
template <typename TX, typename TC>
__global__ void __launch_bounds__(128) tiled_impute_kernel(const TX* __restrict__ X, int n, int m, int k,
                                                           const TC* __restrict__ Wst, const TC* __restrict__ Hst,
                                                           const UnitState* st, TC* __restrict__ ximp) {
    const int r = blockIdx.y;
    if (st[r].stop != 0) return;
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n) return;
    const TC* W = Wst + (long long)r * n * k;
    const TC* H = Hst + (long long)r * k * m;
    TC* xi = ximp + (long long)r * n * m;
    for (int j = 0; j < m; ++j) {
        const TX xr = X[(long long)i + (long long)j * n];
        if (xr == xr) continue;
        TC p = (TC)0;
        for (int c = 0; c < k; ++c) p = fma(W[(long long)i + (long long)c * n], H[(long long)j * k + c], p);
        xi[(long long)i + (long long)j * n] = p;
    }
}

struct TiledCheckArgs {
    void* W;
    void* H;
    UnitState* st;
    int32_t* canon;
    const double* partials;  // R x nblk x 2
    int n, m, k, nblk;
    int it;                  // iteration just completed
    int maxbad, stopconv;
    double tol, tolOF, eps_clamp;
    int* active_count;
    int w_clamped;           // 1: W was clamped by tiled_clampW_kernel (tall matrices: n*k elements per restart)
};

// W = max(W, eps()) of :100 for every restart that goes on (running and objective >= tol: a restart that stops on the
// tolerance keeps its unclamped factors, :75-78), spread over the whole GPU: one CTA per restart is 22 ms at n = 500 000.
// obj2[2r] is the SAME objective sum the check kernel reads, so the two kernels take the same decision.
template <typename TC>
__global__ void __launch_bounds__(256) tiled_clampW_kernel(TC* __restrict__ Wst, long long nk, const UnitState* st,
                                                            const double* __restrict__ obj2, double tol, TC epsc) {
    const int r = blockIdx.y;
    if (st[r].stop != 0 || obj2[2 * r] < tol) return;
    TC* W = Wst + (long long)r * nk;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nk; e += (long long)gridDim.x * blockDim.x) {
        const TC v = W[e];
        W[e] = (v != v) ? v : (v < epsc ? epsc : v);
    }
}

// the every-10th-iteration block of NMFmultiplicative (:73-116) for one restart per CTA
template <typename TC>
__global__ void __launch_bounds__(256) tiled_check_kernel(const TiledCheckArgs a) {
    extern __shared__ int smi[];
    int* idx = smi;           // m
    int* first = smi + a.m;   // k
    __shared__ double s_obj;
    __shared__ int s_stop;
    const int r = blockIdx.x, tid = threadIdx.x, NT = blockDim.x;
    UnitState* st = a.st + r;
    if (st->stop != 0) return;
    const int n = a.n, m = a.m, k = a.k;
    TC* W = static_cast<TC*>(a.W) + (long long)r * n * k;
    TC* H = static_cast<TC*>(a.H) + (long long)r * k * m;
    int32_t* canon_old = a.canon + (long long)r * m;
    if (tid == 0) {
        double obj = 0.0;
        for (int b = 0; b < a.nblk; ++b) obj += a.partials[((long long)r * a.nblk + b) * 2];
        s_obj = obj;
        int stop = 0;
        int bad = st->bad, re = st->re;
        double best = st->best;
        st->obj_chk = obj;
        if (obj < a.tol) {
            stop = 2;  // :75-78 (before the clamp)
        } else {
            if (obj < best) {
                if ((best - obj) < a.tolOF)
                    ++bad;
                else
                    bad = 0;
                best = obj;
            } else {
                ++bad;
            }
            if (bad >= a.maxbad) {
                ++re;
                bad = 0;
            }
            st->bad = bad;
            st->re = re;
            st->best = best;
        }
        s_stop = stop;
    }
    __syncthreads();
    if (s_stop == 2) {
        if (tid == 0) {
            st->stop = 2;
            st->it = a.it;
        }
        return;
    }
    const TC epsc = (TC)a.eps_clamp;
    if (!a.w_clamped)
        for (long long e = tid; e < (long long)n * k; e += NT) {
            const TC v = W[e];
            W[e] = (v != v) ? v : (v < epsc ? epsc : v);
        }
    for (long long e = tid; e < (long long)k * m; e += NT) {
        const TC v = H[e];
        H[e] = (v != v) ? v : (v < epsc ? epsc : v);
    }
    for (int c = tid; c < k; c += NT) first[c] = INT_MAX;
    __syncthreads();
    for (int j = tid; j < m; j += NT) {
        const TC* h = H + (long long)j * k;
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
    const int has_cons = st->has_cons;
    int same = 1;
    for (int j = tid; j < m; j += NT) {
        const int c = first[idx[j]];
        if (!has_cons || canon_old[j] != c) same = 0;
        idx[j] = c;
    }
    same = __syncthreads_and(same);
    int inc = st->inc;
    __syncthreads();
    inc = same ? inc + 1 : 0;
    const bool stopc = inc > a.stopconv;
    if (!stopc)
        for (int j = tid; j < m; j += NT) canon_old[j] = idx[j];
    if (tid == 0) {
        st->inc = inc;
        st->it = a.it;
        if (stopc)
            st->stop = 4;
        else
            st->has_cons = 1;
    }
}

// post-run: objective sums -> state, then normalisation (NMFkExecute.jl:791-804); one CTA per restart
// wide W .*= total' of the finish step for tall matrices (one CTA per restart took 18 ms at n = 250 000): the finish kernel
// leaves the k totals and a flag per restart, this one scales W with the whole GPU
template <typename TC>
__global__ void __launch_bounds__(256) tiled_scaleW_kernel(TC* __restrict__ Wst, long long n, int k, const double* __restrict__ tot,
                                                            const int* __restrict__ wflag) {
    const int r = blockIdx.y;
    if (!wflag[r]) return;
    TC* W = Wst + (long long)r * n * k;
    const double* t = tot + (long long)r * kTiledMaxK;
    const long long nk = n * k;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nk; e += (long long)gridDim.x * blockDim.x)
        W[e] = W[e] * (TC)t[e / n];
}

template <typename TC>
__global__ void __launch_bounds__(256) tiled_finish_kernel(void* Wv, void* Hv, UnitState* stv, const double* partials,
                                                           int n, int m, int k, int nblk, int normalize, double* tot_out = nullptr,
                                                           int* wflag = nullptr) {
    __shared__ double red[40];
    __shared__ double tot[kTiledMaxK];
    const int r = blockIdx.x, tid = threadIdx.x, NT = blockDim.x;
    UnitState* st = stv + r;
    if (st->stop == 0 || st->done != 0) return;
    TC* W = static_cast<TC*>(Wv) + (long long)r * n * k;
    TC* H = static_cast<TC*>(Hv) + (long long)r * k * m;
    if (tid == 0) {
        double a0 = 0.0, a1 = 0.0;
        for (int b = 0; b < nblk; ++b) {
            a0 += partials[((long long)r * nblk + b) * 2];
            a1 += partials[((long long)r * nblk + b) * 2 + 1];
        }
        st->obj_ssq = a0;
        st->obj_norm = sqrt(a1);
    }
    if (normalize == 1) {  // total = sum(H; dims=2); W .*= total'; H ./= total
        for (int c = 0; c < k; ++c) {
            double s = 0.0;
            for (int j = tid; j < m; j += NT) s += (double)H[(long long)j * k + c];
            s = block_sum(s, red);
            if (tid == 0) tot[c] = (double)(TC)s;
        }
        __syncthreads();
        if (wflag != nullptr) {  // W is scaled by tiled_scaleW_kernel over the whole GPU
            for (int c = tid; c < k; c += NT) tot_out[(long long)r * kTiledMaxK + c] = tot[c];
            if (tid == 0) wflag[r] = 1;
        } else {
            for (long long e = tid; e < (long long)n * k; e += NT) W[e] = W[e] * (TC)tot[e / n];
        }
        for (long long e = tid; e < (long long)k * m; e += NT) H[e] = div_cold<TC>(H[e], (TC)tot[e % k]);
    } else if (normalize == 2) {  // total = sum(W; dims=1); W ./= total; H .*= total'
        for (int c = 0; c < k; ++c) {
            double s = 0.0;
            for (int i = tid; i < n; i += NT) s += (double)W[(long long)i + (long long)c * n];
            s = block_sum(s, red);
            if (tid == 0) tot[c] = (double)(TC)s;
        }
        __syncthreads();
        for (long long e = tid; e < (long long)n * k; e += NT) W[e] = div_cold<TC>(W[e], (TC)tot[e / n]);
        for (long long e = tid; e < (long long)k * m; e += NT) H[e] = H[e] * (TC)tot[e % k];
    }
    __syncthreads();
    if (tid == 0) st->done = 1;
}

// Variant KL_DIV: den[r][a] += delta (NMF.jl's colsum(W) .+ delta / rowsum(H) .+ delta) for every running restart
template <typename TC>
__global__ void tiled_den_delta_kernel(TC* __restrict__ den, int k, const UnitState* st) {
    const int r = blockIdx.x, c = threadIdx.x;
    if (st[r].stop != 0 || c >= k) return;
    den[(long long)r * kTiledMaxK + c] += kKlDivDelta<TC>;
}

// Variant KL_DIV: the sums of NMF.jl's stop_condition for one factor against its snapshot from before the iteration, in the
// layout fro_converge_kernel reads: conv[((r * gridDim.x + tile) * k + a) * 2 + {0,1}] = sum over the tile's 256 own indices o of
// (new - old)^2, (new + old)^2 for column a of W (o = row) or row a of H (o = column).
template <typename TC>
__global__ void __launch_bounds__(256) tiled_conv_kernel(const TC* __restrict__ U, const TC* __restrict__ Uold, long long rstride,
                                                          long long s_o, long long s_a, int nown, int k, const UnitState* st,
                                                          double* __restrict__ conv) {
    __shared__ double red[40];
    const int r = blockIdx.y, tile = blockIdx.x;
    if (st[r].stop != 0) return;
    const int o = tile * 256 + threadIdx.x;
    const long long base = (long long)r * rstride + (long long)o * s_o;
    for (int c = 0; c < k; ++c) {
        double d2 = 0.0, s2 = 0.0;
        if (o < nown) {
            const double un = (double)U[base + (long long)c * s_a], uo = (double)Uold[base + (long long)c * s_a];
            d2 = (un - uo) * (un - uo);
            s2 = (un + uo) * (un + uo);
        }
        d2 = block_sum(d2, red);
        s2 = block_sum(s2, red);
        if (threadIdx.x == 0) {
            double* dst = conv + (((long long)r * gridDim.x + tile) * k + c) * 2;
            dst[0] = d2;
            dst[1] = s2;
        }
    }
}

// loop guard of :64 evaluated on the device between iterations: marks restarts that must not start
// another iteration and counts the ones still running
static __global__ void tiled_guard_kernel(UnitState* st, int R, int it, int maxiter, int maxbad, int maxre, int iter_limit,
                                   int* active_count) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    UnitState* s = st + r;
    if (s->stop != 0) return;
    s->it = it;
    if (it >= maxiter)
        s->stop = 1;
    else if (s->bad >= maxbad)
        s->stop = 5;
    else if (s->re >= maxre)
        s->stop = 3;
    else if (!(iter_limit > 0 && it >= iter_limit))
        atomicAdd(active_count, 1);
}

// red == nullptr: the complete half-update.  red != nullptr (row-sharded X, H-update): the pass leaves
// the numerators of this rank's rows in red[R][nown][K]; launch_tiled_apply_k finishes after the all-reduce.
template <typename TX, typename TC, int K>
cudaError_t launch_tiled_pass_k(const TiledPassArgs& a, void* red, cudaStream_t s, bool div = false) {
    constexpr int VEC = VecOf<TC>::N;
    constexpr int KP = (K + VEC - 1) / VEC * VEC;
    constexpr int TCH = TiledCfg<TX>::TCH;
    const size_t smem = (size_t)kTiledStages * TCH * (KP * sizeof(TC) + kTiledThreads * sizeof(TX));
    const long long grid = (long long)a.S * a.nblocks * a.R;
    if (grid > 2147483647ll) return cudaErrorInvalidValue;
    cudaError_t e;
    if (div) {
        e = cudaFuncSetAttribute(tiled_pass_kernel<TX, TC, K, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        tiled_pass_kernel<TX, TC, K, false, true><<<(unsigned)grid, kTiledThreads, smem, s>>>(a);
    } else if (a.has_nan) {
        e = cudaFuncSetAttribute(tiled_pass_kernel<TX, TC, K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        tiled_pass_kernel<TX, TC, K, true><<<(unsigned)grid, kTiledThreads, smem, s>>>(a);
    } else {
        e = cudaFuncSetAttribute(tiled_pass_kernel<TX, TC, K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        tiled_pass_kernel<TX, TC, K, false><<<(unsigned)grid, kTiledThreads, smem, s>>>(a);
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (a.partial != nullptr) {
        dim3 g((a.nown + 255) / 256, a.R);
        tiled_combine_kernel<TC, K><<<g, 256, 0, s>>>(a, static_cast<TC*>(red));
        e = cudaGetLastError();
    }
    return e;
}

template <typename TX, typename TC, int K>
cudaError_t launch_tiled_combine_k(const TiledPassArgs& a, void* red, cudaStream_t s) {
    dim3 g((a.nown + 255) / 256, a.R);
    tiled_combine_kernel<TC, K><<<g, 256, 0, s>>>(a, static_cast<TC*>(red));
    return cudaGetLastError();
}

template <typename TX, typename TC, int K>
cudaError_t launch_tiled_apply_k(const TiledPassArgs& a, void* red, cudaStream_t s) {
    dim3 g((a.nown + 255) / 256, a.R);
    tiled_apply_kernel<TC, K><<<g, 256, 0, s>>>(a, static_cast<const TC*>(red));
    return cudaGetLastError();
}

}  // namespace nmfk

// ------------------------------------------------------------------------------------------
// host driver (one instantiation per dtype)
// ------------------------------------------------------------------------------------------
namespace nmfk {

// template K of the tiled engine's kernels (tiled_template_k): the resident set up to 32, then 40 / 48 / 56 / 64.  Kept
// apart from NMFK_DISPATCH_K so that no resident kernel is instantiated above 32.
#define NMFK_DISPATCH_TILED_K(FN, TX, TC, KT, ...)                \
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
        case 40: return FN<TX, TC, 40>(__VA_ARGS__);              \
        case 48: return FN<TX, TC, 48>(__VA_ARGS__);              \
        case 56: return FN<TX, TC, 56>(__VA_ARGS__);              \
        case 64: return FN<TX, TC, 64>(__VA_ARGS__);              \
        default: return cudaErrorInvalidValue;                    \
    }

template <typename TX, typename TC>
cudaError_t dispatch_tiled_combine(const TiledPassArgs& a, void* red, cudaStream_t s) {
    const int kt = tiled_template_k(a.k);
    NMFK_DISPATCH_TILED_K(launch_tiled_combine_k, TX, TC, kt, a, red, s)
}
// use_tc: Float32 without NaN -> the tcgen05 kernel of kl_tiled_tc.cu (a.nblocks counts 128-index tiles)
// use_td: Float64 without NaN, k >= 4 -> the DMMA kernel of kl_tiled_dmma.cu (a.nblocks counts 128-index blocks, a.D is
// the step-contiguous copy of the data)
// div: the pass kernels' Variant KL_DIV flavour (quotient x / (p + delta); a.den holds the sums + delta)
template <typename TX, typename TC>
cudaError_t dispatch_tiled_pass(const TiledPassArgs& a, void* red, cudaStream_t s, bool use_tc, int* errflag, bool use_td = false,
                                bool div = false) {
    const int kt = tiled_template_k(a.k);
    if (use_tc) {
        cudaError_t e = launch_tc_pass(a, errflag, s, div);
        if (e != cudaSuccess || a.partial == nullptr) return e;
        return dispatch_tiled_combine<TX, TC>(a, red, s);
    }
    if (use_td) {
        cudaError_t e = launch_tiled_dmma_pass(a, s, div);
        if (e != cudaSuccess || a.partial == nullptr) return e;
        return dispatch_tiled_combine<TX, TC>(a, red, s);
    }
    NMFK_DISPATCH_TILED_K(launch_tiled_pass_k, TX, TC, kt, a, red, s, div)
}
// the same, bracketed by the profile events (one "launch" = the pass kernel, plus the small slice-combine kernel when the
// reduction range is sliced)
template <typename TX, typename TC>
cudaError_t timed_tiled_pass(const TiledPassArgs& a, void* red, cudaStream_t s, bool use_tc, int* errflag, bool use_td,
                             PassProfile* prof, bool div = false) {
    if (prof) prof->begin(s);
    const cudaError_t e = dispatch_tiled_pass<TX, TC>(a, red, s, use_tc, errflag, use_td, div);
    if (prof) prof->end(s);
    return e;
}
template <typename TX, typename TC>
cudaError_t dispatch_tiled_apply(const TiledPassArgs& a, void* red, cudaStream_t s) {
    const int kt = tiled_template_k(a.k);
    NMFK_DISPATCH_TILED_K(launch_tiled_apply_k, TX, TC, kt, a, red, s)
}

// NMFK_TILED_TIMING=1: device time of every phase of the tiled engine's iteration (CUDA events between the launches, read at
// the host synchronisation points), printed per solve - the timeline that says what bounds an iteration (row-sharded runs).
struct PhaseTimer {
    static constexpr int NPH = 14;
    bool on = false;
    std::vector<cudaEvent_t> idle;
    std::vector<std::pair<cudaEvent_t, int>> marks;
    double ms[NPH] = {0};
    long long cnt[NPH] = {0};
    void mark(cudaStream_t s, int phase) {  // `phase` = what ran since the previous mark (-1: start of a timed stretch)
        if (!on) return;
        cudaEvent_t e = nullptr;
        if (!idle.empty()) {
            e = idle.back();
            idle.pop_back();
        } else {
            cudaEventCreate(&e);
        }
        cudaEventRecord(e, s);
        marks.emplace_back(e, phase);
    }
    void harvest() {
        for (size_t i = 1; i < marks.size(); ++i) {
            float t = 0.f;
            if (marks[i].second >= 0 && cudaEventElapsedTime(&t, marks[i - 1].first, marks[i].first) == cudaSuccess) {
                ms[marks[i].second] += t;
                ++cnt[marks[i].second];
            }
        }
        for (auto& m : marks) idle.push_back(m.first);
        marks.clear();
    }
    void report(int iters, int rank) {
        if (!on) return;
        static const char* names[NPH] = {"sums_W", "pass_H", "allreduce_H", "apply_H", "sums_H", "pass_W", "impute", "objective",
                                         "objsum_allreduce", "clamp_check", "guard_sync", "finish", "snapshot", "converge"};
        fprintf(stderr, "[nmfk timing rank %d] %d iterations:", rank, iters);
        for (int i = 0; i < NPH; ++i)
            if (cnt[i]) fprintf(stderr, " %s=%.3fms/%lld", names[i], ms[i], cnt[i]);
        fprintf(stderr, "\n");
        for (auto e : idle) cudaEventDestroy(e);
        idle.clear();
    }
};

#define NMFK_TRY(call)                      \
    do {                                    \
        cudaError_t e__ = (call);           \
        if (e__ != cudaSuccess) {           \
            err = e__;                      \
            goto done;                      \
        }                                   \
    } while (0)

// div: Variant KL_DIV (NMF.jl's MultUpdate(obj=:div)) instead of NMFmultiplicative: the same passes in their delta flavour,
// no NaN imputation, clamp or objective checks; NMF.jl's stop_condition after every iteration against a snapshot of the factors
// taken before it (fro_converge_kernel), the host looking at the running count every check_every iterations
template <typename TX, typename TC>
cudaError_t solve_tiled_t(const SolveArgs& a, cudaStream_t s, int64_t* launches, bool div) {
    const int n = a.n, m = a.m, k = a.k, R = a.R;
    const int kt = tiled_template_k(k);
    if (kt < 0) return cudaErrorInvalidValue;
    if (div && (a.has_nan || a.shard != nullptr)) return cudaErrorNotSupported;
    cudaError_t err = cudaSuccess;
    int sms = 148;
    {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    // Float32 without NaN: both half-updates run on the tensor cores (kl_tiled_tc.cu), 128 own indices per CTA and
    // groups of restarts that share the X tiles; everything else (sums, combine, objective, check) is unchanged
    bool use_tc = false;
    if (std::is_same<TX, float>::value && std::is_same<TC, float>::value && a.tiled_tc && !a.has_nan) {
        TiledPassArgs probe{};
        probe.k = k;
        probe.nown = m;
        probe.D = a.Xt;
        use_tc = tc_pass_supported(probe);
        probe.nown = n;
        probe.D = a.X;
        use_tc = use_tc && tc_pass_supported(probe);
    }
    // Float64 without NaN, k >= 4: both half-updates run on the FP64 tensor pipe (kl_tiled_dmma.cu)
    const bool use_td = std::is_same<TX, double>::value && std::is_same<TC, double>::value && a.tiled_tc && !a.has_nan && k >= 4;
    const int ownper = use_tc ? 128 : (use_td ? tiled_dmma_own() : kTiledThreads);
    const int units = use_tc ? (R + tc_pass_group(k) - 1) / tc_pass_group(k) : R;  // CTAs per own block and slice
    const int nblkH = (m + ownper - 1) / ownper;  // H-update: own = columns
    const int nblkW = (n + ownper - 1) / ownper;  // W-update: own = rows
    constexpr int TCH = TiledCfg<TX>::TCH;
    const double slice_gain = getenv("NMFK_TILED_SLICE_GAIN") ? atof(getenv("NMFK_TILED_SLICE_GAIN")) : 0.05;
    auto slices = [&](int nblk, int nred) {
        const long long target = (use_tc ? 3ll * tc_pass_ctas_per_sm(k) : (use_td ? 3ll : 4ll)) * sms;
        long long S = (target + (long long)nblk * units - 1) / ((long long)nblk * units);
        const long long smax = std::max(1, nred / ((use_tc ? tc_pass_chunk(k) : (use_td ? tiled_dmma_chunk() : TCH)) * 8));
        if (S > smax) S = smax;
        if (S < 1) S = 1;
        // wave quantisation: one CTA per SM, so a grid of 3.46 waves (C4, 32 restarts per GPU: 16 own blocks x 32) runs as 4.  A few
        // more slices are worth their combine pass when they fill the last wave (>= 5 % of the launch; on C3, 8.54 waves, three
        // slices would gain 3.6 % of the grid and measured 1.3 % SLOWER with their partial sums and combine pass).
        auto eff = [&](long long s_) {
            const long long ctas = (long long)nblk * units * s_;
            return (double)ctas / (double)(((ctas + sms - 1) / sms) * sms);
        };
        long long best = S;
        for (long long s2 = S + 1; s2 <= std::min(smax, S + 3); ++s2)
            if (eff(s2) > eff(best) + slice_gain) best = s2;
        return (int)best;
    };
    const int SH = slices(nblkH, n), SW = slices(nblkW, m);
    const int nblkObj = (n + 127) / 128;
    const bool wobj = a.wref.any();  // per-row / per-column / per-entry weights: the scalar objective kernel applies them

    // row-sharded X: den and the H-update numerators are contiguous so that one all-reduce moves both
    const ShardComm* sh = a.shard;
    const bool sharded = sh != nullptr;
    PhaseTimer pt;
    pt.on = getenv("NMFK_TILED_TIMING") != nullptr;
    const auto host_t0 = std::chrono::steady_clock::now();
    auto host_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count(); };
    double host_setup_ms = 0.0;
    const int it_begin_report = 0;
    (void)it_begin_report;
    TC* den = nullptr;  // R x kTiledMaxK, followed by red (R x m x kt) when sharded
    TC* red = nullptr;
    double* obj2 = nullptr;
    TC* partial = nullptr;
    double* objp = nullptr;
    int* d_active = nullptr;
    double* fin_tot = nullptr;  // wide finish: the k totals of every restart
    int* fin_flag = nullptr;    //              ... and which restarts tiled_scaleW_kernel has to scale
    TC* Wold = nullptr;         // Variant KL_DIV: the factors before the iteration ...
    TC* Hold = nullptr;
    double* convW = nullptr;    // ... and the per-tile sums of the stop condition
    double* convH = nullptr;
    const int ctW = (n + 255) / 256, ctH = (m + 255) / 256;
    void* vimg = nullptr;       // tcgen05 pass (k <= 16): V operand images, rebuilt before every half-update
    int* h_active = nullptr;  // [0] running restarts, [1] barrier time-out site reported by the tcgen05 kernel
    // the tcgen05 kernels that can raise h_active[1] in the current phase of the solve, for the error message
    const char* flag_kernel = use_tc && tc2_pass_enabled(k) ? "tc2_pass_kernel or tc_pass_kernel" : "tc_pass_kernel";
    const char* flag_where = "half-update pass or stop-check objective";
    std::vector<UnitState> hst((size_t)R);
    int it = 0;
    bool any_running = false;
    const size_t psz = std::max((size_t)((SH > 1 || sharded) ? (size_t)SH * R * m * kt : 0),
                                (size_t)(SW > 1 ? (size_t)SW * R * n * kt : 0));
    const size_t redsz = sharded ? (size_t)R * m * kt : 0;
    if (sharded && a.normalize == 2) return cudaErrorNotSupported;
    // Float32 objective on the tensor cores: D = X, U = W, V = H (the W-update orientation), P = W H by MMA#1 and
    // (x - p)^2 by the quotient warps; partial sums per block of 128 rows like tiled_objective_kernel
    // nanosleep between barrier polls of the roles that run ahead of the critical path: low 16 bits = X producer,
    // high 16 bits = V stagers (NMFK_TC_WAIT_HINT_NS overrides; 64 / 32 ns measured best or equal on C3, C3 k=32, C5)
    const int wait_hint = getenv("NMFK_TC_WAIT_HINT_NS") ? atoi(getenv("NMFK_TC_WAIT_HINT_NS")) : ((32 << 16) | 64);
    const int qwait = getenv("NMFK_TC_QWAIT_NS") ? atoi(getenv("NMFK_TC_QWAIT_NS")) : 0;
    auto obj_args = [&](int restore, int sel) {
        TiledPassArgs po{};
        po.D = use_td ? a.Xt : a.X;  // the DMMA kernel reads the step-contiguous copy
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
        po.ktmpl = kt;
        po.obj_partials = objp;
        po.obj_weight = a.weight;
        po.obj_restore = restore;
        po.obj_sel = sel;
        po.wait_hint_ns = wait_hint;
        po.qwait_ns = qwait;
        return po;
    };
  // column sums of W would need another exchange

    NMFK_TRY(scratch_alloc(&den, ((size_t)R * kTiledMaxK + redsz) * sizeof(TC), s));
    if (sharded) red = den + (size_t)R * kTiledMaxK;
    NMFK_TRY(scratch_alloc(&obj2, (size_t)R * 2 * sizeof(double), s));
    if (psz) NMFK_TRY(scratch_alloc(&partial, psz * sizeof(TC), s));
    NMFK_TRY(scratch_alloc(&objp, (size_t)R * nblkObj * 2 * sizeof(double), s));
    NMFK_TRY(scratch_alloc(&d_active, sizeof(int), s));
    NMFK_TRY(scratch_alloc(&fin_tot, (size_t)R * kTiledMaxK * sizeof(double), s));
    NMFK_TRY(scratch_alloc(&fin_flag, (size_t)R * sizeof(int), s));
    if (div) {
        NMFK_TRY(scratch_alloc(&Wold, (size_t)R * n * k * sizeof(TC), s));
        NMFK_TRY(scratch_alloc(&Hold, (size_t)R * k * m * sizeof(TC), s));
        NMFK_TRY(scratch_alloc(&convW, (size_t)R * ctW * k * 2 * sizeof(double), s));
        NMFK_TRY(scratch_alloc(&convH, (size_t)R * ctH * k * 2 * sizeof(double), s));
    }
    if (use_tc) {
        const size_t vb = std::max(tc2_image_bytes(k, R, n), tc2_image_bytes(k, R, m));
        if (vb) NMFK_TRY(scratch_alloc(&vimg, vb, s));
    }
    h_active = pinned_flags();
    if (h_active == nullptr) NMFK_TRY(cudaErrorMemoryAllocation);
    h_active[0] = h_active[1] = 0;
    h_active[1] = 0;
    NMFK_TRY(cudaMemcpyAsync(hst.data(), a.st, (size_t)R * sizeof(UnitState), cudaMemcpyDeviceToHost, s));
    NMFK_TRY(cudaStreamSynchronize(s));
    for (auto& u : hst)
        if (u.stop == 0 && !u.done) {
            any_running = true;
            it = std::max(it, (int)u.it);
        }
    if (any_running) {
        // restarts of one batch advance in lockstep
        TiledPassArgs ph{}, pw{};
        ph.D = use_td ? a.X : a.Xt;  // the DMMA kernel reads the STEP-contiguous copy, the others the OWN-contiguous one
        ph.Dstep = a.X;              // ... except the tc2 pass, which reads the step-contiguous one through Dstep
        ph.U = a.H;
        ph.V = a.W;
        ph.den = den;
        ph.partial = (SH > 1 || sharded) ? partial : nullptr;
        ph.st = a.st;
        ph.ximp = a.ximp;
        ph.u_rstride = (long long)k * m;
        ph.v_rstride = (long long)n * k;
        ph.su_o = k;
        ph.su_a = 1;
        ph.sv_t = 1;
        ph.sv_a = n;
        ph.nown = m;
        ph.nred = n;
        ph.k = k;
        ph.R = R;
        ph.S = SH;
        ph.nblocks = nblkH;
        ph.transposed = 1;
        ph.ldimp = n;
        ph.has_nan = a.has_nan;
        ph.lambda = a.lambda;
        ph.ktmpl = kt;
        ph.vimg = vimg;
        ph.wait_hint_ns = wait_hint;
        ph.qwait_ns = qwait;
        pw = ph;
        pw.D = use_td ? a.Xt : a.X;
        pw.Dstep = a.Xt;
        pw.U = a.W;
        pw.V = a.H;
        pw.partial = SW > 1 ? partial : nullptr;
        pw.u_rstride = (long long)n * k;
        pw.v_rstride = (long long)k * m;
        pw.su_o = 1;
        pw.su_a = n;
        pw.sv_t = k;
        pw.sv_a = 1;
        pw.nown = n;
        pw.nred = m;
        pw.S = SW;
        pw.nblocks = nblkW;
        pw.transposed = 0;

        if (a.has_nan && it > 0) {  // resume: rebuild X[inan] = (W*H)[inan]
            dim3 g((n + 127) / 128, R);
            tiled_impute_kernel<TX, TC><<<g, 128, 0, s>>>((const TX*)a.X, n, m, k, (const TC*)a.W, (const TC*)a.H, a.st,
                                                          (TC*)a.ximp);
            NMFK_TRY(cudaGetLastError());
            ++*launches;
        }
        // NMFK_TC_TRACE=<file>: clock64 stamps of CTA 0 of the first tcgen05 H-update (tools/tc_trace.py reads them)
        long long* d_trace = nullptr;
        const char* trace_path = use_tc ? getenv("NMFK_TC_TRACE") : nullptr;
        if (trace_path != nullptr) {
            NMFK_TRY(cudaMalloc(&d_trace, 3 * 64 * 8 * sizeof(long long)));
            NMFK_TRY(cudaMemsetAsync(d_trace, 0, 3 * 64 * 8 * sizeof(long long), s));
            ph.trace = d_trace;
        }
        bool need_guard = true;
        host_setup_ms = host_ms();
        while (true) {
            if (need_guard) {
                NMFK_TRY(cudaMemsetAsync(d_active, 0, sizeof(int), s));
                tiled_guard_kernel<<<(R + 127) / 128, 128, 0, s>>>(a.st, R, it, a.maxiter, div ? INT_MAX : a.maxbad,
                                                                   div ? INT_MAX : a.maxre, a.iter_limit, d_active);
                NMFK_TRY(cudaGetLastError());
                ++*launches;
                NMFK_TRY(cudaMemcpyAsync(h_active, d_active, sizeof(int), cudaMemcpyDeviceToHost, s));
                pt.mark(s, 10);
                NMFK_TRY(cudaStreamSynchronize(s));
                if (a.prof) a.prof->harvest();
                pt.harvest();
                if (h_active[1] != 0) goto done;  // written by the tcgen05 kernels through the mapped pinned flags
                if (*h_active == 0) break;
                need_guard = false;
                pt.mark(s, -1);
            }
            ++it;
            ph.first_iter = pw.first_iter = (it == 1);
            if (div) {
                if (!a.Wfixed) NMFK_TRY(cudaMemcpyAsync(Wold, a.W, (size_t)R * n * k * sizeof(TC), cudaMemcpyDeviceToDevice, s));
                if (!a.Hfixed) NMFK_TRY(cudaMemcpyAsync(Hold, a.H, (size_t)R * k * m * sizeof(TC), cudaMemcpyDeviceToDevice, s));
                pt.mark(s, 12);
            }
            if (!a.Hfixed) {
                tiled_sums_kernel<TC><<<dim3(k, R), 256, 0, s>>>(a.W, (long long)n * k, 1, n, n, a.st, den);
                NMFK_TRY(cudaGetLastError());
                if (div) {
                    tiled_den_delta_kernel<TC><<<R, kTiledMaxK, 0, s>>>(den, k, a.st);
                    NMFK_TRY(cudaGetLastError());
                    ++*launches;
                }
                pt.mark(s, 0);
                NMFK_TRY((timed_tiled_pass<TX, TC>(ph, red, s, use_tc, h_active + 1, use_td, a.prof, div)));
                pt.mark(s, 1);
                *launches += 2 + (SH > 1 || sharded) + (vimg != nullptr);  // + the image producer of the tc2 pass
                if (d_trace != nullptr) {
                    std::vector<long long> ht(3 * 64 * 8);
                    NMFK_TRY(cudaMemcpyAsync(ht.data(), d_trace, ht.size() * sizeof(long long), cudaMemcpyDeviceToHost, s));
                    NMFK_TRY(cudaStreamSynchronize(s));
                    if (FILE* f = fopen(trace_path, "wb")) {
                        fwrite(ht.data(), sizeof(long long), ht.size(), f);
                        fclose(f);
                    }
                    cudaFree(d_trace);
                    d_trace = nullptr;
                    ph.trace = nullptr;
                }
                if (sharded) {
                    // colsum(W) and W' * (X ./ (W*H)) over this rank's rows -> sums over all rows, then the update
                    NMFK_TRY(sh->allreduce(sh->comm, den, (size_t)R * kTiledMaxK + redsz, sizeof(TC) == 8 ? 1 : 0, s));
                    pt.mark(s, 2);
                    NMFK_TRY((dispatch_tiled_apply<TX, TC>(ph, red, s)));
                    pt.mark(s, 3);
                    ++*launches;
                }
            }
            if (!a.Wfixed) {
                tiled_sums_kernel<TC><<<dim3(k, R), 256, 0, s>>>(a.H, (long long)k * m, k, 1, m, a.st, den);
                NMFK_TRY(cudaGetLastError());
                if (div) {
                    tiled_den_delta_kernel<TC><<<R, kTiledMaxK, 0, s>>>(den, k, a.st);
                    NMFK_TRY(cudaGetLastError());
                    ++*launches;
                }
                pt.mark(s, 4);
                NMFK_TRY((timed_tiled_pass<TX, TC>(pw, nullptr, s, use_tc, h_active + 1, use_td, a.prof, div)));
                pt.mark(s, 5);
                *launches += 2 + (SW > 1) + (vimg != nullptr);
            }
            if (a.has_nan) {
                dim3 g((n + 127) / 128, R);
                tiled_impute_kernel<TX, TC><<<g, 128, 0, s>>>((const TX*)a.X, n, m, k, (const TC*)a.W, (const TC*)a.H,
                                                              a.st, (TC*)a.ximp);
                NMFK_TRY(cudaGetLastError());
                ++*launches;
            }
            if (div) {
                if (!a.Wfixed) {
                    tiled_conv_kernel<TC><<<dim3(ctW, R), 256, 0, s>>>((const TC*)a.W, Wold, (long long)n * k, 1, n, n, k, a.st, convW);
                    NMFK_TRY(cudaGetLastError());
                    ++*launches;
                }
                if (!a.Hfixed) {
                    tiled_conv_kernel<TC><<<dim3(ctH, R), 256, 0, s>>>((const TC*)a.H, Hold, (long long)k * m, k, 1, m, k, a.st, convH);
                    NMFK_TRY(cudaGetLastError());
                    ++*launches;
                }
                NMFK_TRY(launch_fro_converge(a.st, R, k, convW, ctW, convH, ctH, !a.Wfixed, !a.Hfixed, a.tol, it, s));
                ++*launches;
                pt.mark(s, 13);
                if (it % a.check_every == 0) need_guard = true;
            } else if (it % a.check_every == 0) {
                if (use_tc && !wobj) {
                    NMFK_TRY(launch_tc_objective(obj_args(0, 0), h_active + 1, s));
                } else if (use_td && !wobj) {
                    NMFK_TRY(launch_tiled_dmma_objective(obj_args(0, 0), s));
                } else {
                    dim3 g(nblkObj, R);
                    NMFK_TRY((tiled_objective_smem<TX, TC>(k)));
                    tiled_objective_kernel<TX, TC><<<g, 128, (size_t)k * 128 * sizeof(TC), s>>>(
                        (const TX*)a.X, n, m, k, (const TC*)a.W, (const TC*)a.H, a.st, (TC)a.lambda, 0, 1, a.weight, a.wref, objp);
                }
                NMFK_TRY(cudaGetLastError());
                pt.mark(s, 7);
                // per-restart objective sums in block order (and, row-sharded, over all ranks)
                tiled_objsum_kernel<<<(R + 127) / 128, 128, 0, s>>>(objp, nblkObj, R, obj2);
                NMFK_TRY(cudaGetLastError());
                ++*launches;
                if (sharded) NMFK_TRY(sh->allreduce(sh->comm, obj2, (size_t)R * 2, 1, s));
                pt.mark(s, 8);
                const bool wide_clamp = (long long)n * k >= (1ll << 18) && !a.Wfixed;
                if (wide_clamp) {
                    const long long nk = (long long)n * k;
                    dim3 g((unsigned)std::min<long long>((nk + 2047) / 2048, 4096), R);
                    tiled_clampW_kernel<TC><<<g, 256, 0, s>>>((TC*)a.W, nk, a.st, obj2, a.tol, (TC)a.eps_clamp);
                    NMFK_TRY(cudaGetLastError());
                    ++*launches;
                }
                TiledCheckArgs c{};
                c.W = a.W;
                c.H = a.H;
                c.st = a.st;
                c.canon = a.canon;
                c.partials = obj2;
                c.n = n;
                c.m = m;
                c.k = k;
                c.nblk = 1;
                c.w_clamped = wide_clamp ? 1 : 0;
                c.it = it;
                c.maxbad = a.maxbad;
                c.stopconv = a.stopconv;
                c.tol = a.tol;
                c.tolOF = a.tolOF;
                c.eps_clamp = a.eps_clamp;
                {
                    // canonical co-clustering labels of the m columns live in shared memory (m <= ~58000)
                    const size_t csm = (size_t)(m + k) * sizeof(int);
                    if (csm > 48 * 1024)
                        NMFK_TRY(cudaFuncSetAttribute(tiled_check_kernel<TC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)csm));
                    tiled_check_kernel<TC><<<R, 256, csm, s>>>(c);
                }
                NMFK_TRY(cudaGetLastError());
                pt.mark(s, 9);
                *launches += 2;
                need_guard = true;
            }
            if (it >= a.maxiter || (a.iter_limit > 0 && it >= a.iter_limit)) need_guard = true;
        }
    }
    {
        // post-run objective on the restored X + normalisation for restarts that stopped in this call
        pt.mark(s, -1);
        flag_kernel = "tc_pass_kernel";
        flag_where = "post-run objective";
        if (use_tc && !wobj) {
            NMFK_TRY(launch_tc_objective(obj_args(1, 1), h_active + 1, s));
        } else if (use_td && !wobj) {
            NMFK_TRY(launch_tiled_dmma_objective(obj_args(1, 1), s));
        } else {
            dim3 g(nblkObj, R);
            NMFK_TRY((tiled_objective_smem<TX, TC>(k)));
            tiled_objective_kernel<TX, TC><<<g, 128, (size_t)k * 128 * sizeof(TC), s>>>(
                (const TX*)a.X, n, m, k, (const TC*)a.W, (const TC*)a.H, a.st, (TC)a.lambda, 1, 0, a.weight, a.wref, objp);
        }
        NMFK_TRY(cudaGetLastError());
        if (sharded) {
            tiled_objsum_kernel<<<(R + 127) / 128, 128, 0, s>>>(objp, nblkObj, R, obj2);
            NMFK_TRY(cudaGetLastError());
            NMFK_TRY(sh->allreduce(sh->comm, obj2, (size_t)R * 2, 1, s));
            ++*launches;
        }
        const bool wide_finish = a.normalize == 1 && (long long)n * k >= (1ll << 18);
        if (wide_finish) NMFK_TRY(cudaMemsetAsync(fin_flag, 0, (size_t)R * sizeof(int), s));
        tiled_finish_kernel<TC><<<R, 256, 0, s>>>(a.W, a.H, a.st, sharded ? obj2 : objp, n, m, k, sharded ? 1 : nblkObj,
                                                  a.normalize, wide_finish ? fin_tot : nullptr, wide_finish ? fin_flag : nullptr);
        NMFK_TRY(cudaGetLastError());
        if (wide_finish) {
            const long long nk = (long long)n * k;
            dim3 g((unsigned)std::min<long long>((nk + 2047) / 2048, 1024), R);
            tiled_scaleW_kernel<TC><<<g, 256, 0, s>>>((TC*)a.W, n, k, fin_tot, fin_flag);
            NMFK_TRY(cudaGetLastError());
            ++*launches;
        }
        *launches += 2;
        pt.mark(s, 11);
        NMFK_TRY(cudaStreamSynchronize(s));
        if (a.prof) a.prof->harvest();
        pt.harvest();
        if (pt.on) fprintf(stderr, "[nmfk timing] host wall clock: set-up %.1f ms, whole solve %.1f ms\n", host_setup_ms, host_ms());
        pt.report(it, sharded ? sh->rank : 0);
    }
done:
    // a time-out ends in a trap: the solve has usually failed with that CUDA error already, the flag says where
    if (h_active && h_active[1] != 0) err = solve_timeout(a, err, flag_kernel, flag_where, h_active[1]);
    scratch_free(den, s);
    scratch_free(partial, s);
    scratch_free(objp, s);
    scratch_free(obj2, s);
    scratch_free(d_active, s);
    scratch_free(fin_tot, s);
    scratch_free(fin_flag, s);
    scratch_free(vimg, s);
    scratch_free(Wold, s);
    scratch_free(Hold, s);
    scratch_free(convW, s);
    scratch_free(convH, s);
    return err;
}

}  // namespace nmfk
