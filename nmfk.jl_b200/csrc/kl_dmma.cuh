// Resident KL engine, Float64, FP64-pipe formulation in DMMA fragment layout
// (mma.sync.aligned.m8n8k4.f64 for the aligned part of k, DFMA for the remainder columns).
//
// Same contract as kl_resident.cuh (one CTA = one restart of NMFmultiplicative,
// /root/reference/src/NMFkMultiplicative.jl:56-127 + NMFkExecute.jl:791-804), different hot loop.
// The ncu capture of the scalar kernel (profiles/r01_resident_scalar_k10.txt) shows the
// shared-memory LSU data pipe at 66 % and the FP64 pipe at 31 %: every element-step needs a
// broadcast read of a k-vector.  Here a WARP owns a group of 8 "own" indices and walks the
// reduction index in tiles of 8 steps; lane (g = lane/4, q = lane%4) holds the two elements
// (own g, steps 2q and 2q+1) of the tile, the C-fragment layout of m8n8k4:
//
//   P[8 own x 8 steps]  = U[8 x k] * V[steps, :]^T           (KD/4 DMMAs + (k-KD) DFMAs per element)
//   Q = X ./ P                                               (2 elements per lane)
//   ACC[8 own x k]     += Q[8 x 8 steps] * V[steps, :]       (2 * ND/8 DMMAs + (k-ND) DFMAs per element)
//
// The C-fragment column a lane holds after the first product is exactly the A-fragment element
// it must supply to the second one if the second product's k-index q is bound to step 2q+s
// (s = 0,1), so Q never moves between lanes.
//
// On B200 DMMA and DFMA run on the SAME FP64 datapath (37.0 vs 33.9 TFLOP/s measured; ncu's
// sm__throughput equals the SUM of the dmma sub-pipe and fp64 pipe percentages), so a DMMA is only
// worth issuing when its 8x8x4 block is full: the k columns are split at compile time (DmmaCfg<K>)
// in a DMMA part (multiples of 4 for P, of 8 for ACC) and a remainder of <= 4 columns done with
// plain DFMAs on the same two elements; their 4 per-quad partial sums are combined once per item.
// k <= 3 is all-DFMA in fragment layout.
//
// X is L2-resident (1.6 MB for C2) but ~800 cycles away: every lane keeps PF tiles of its own X
// values in flight in registers, and the prefetch cursor runs ahead ACROSS work items, so a warp
// never drains its pipeline between row groups.  The NaN test of the fast reciprocal is deferred
// to the end of an item (a NaN quotient poisons the accumulators), where the item is redone with
// IEEE divisions - no data-dependent branch on the hot loop.
//
// Shared-memory layout: W rows and H^T rows with pitch = 4*odd doubles (zero padded columns; rows
// padded to a multiple of 8 with ONES so that steps beyond the end see p > 0 and x = 0): the
// B-fragment loads of both products hit all 32 banks in the minimum 2 wavefronts.
#pragma once
#include <type_traits>

#include "kl_resident.cuh"

namespace nmfk {

__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c[0]), "+d"(c[1])
        : "d"(a), "d"(b));
}

__host__ __device__ constexpr int dmma_pitch(int KC) { return (KC & 1) ? KC * 4 : KC * 4 + 4; }
__host__ __device__ constexpr int dmma_cmax(int a, int b) { return a > b ? a : b; }

// compile-time split of the k columns between DMMA blocks and DFMA remainder columns
template <int K>
struct DmmaCfg {
    static constexpr int KC = (K + 3) / 4;
    static constexpr int pitch = dmma_pitch(KC);
    // ACC += Q V: columns [0,ND) by DMMA (8 per instruction pair), [ND,K) by DFMA when few remain.
    // The DFMA columns cost 4 LSU wavefronts per 16-byte row read (LDS.128 is served per quarter
    // warp), so 3-4 remainder columns only pay once the DMMA part keeps the FP64 pipe the bound (K > 8).
    static constexpr int ND =
        (K % 8 == 0) ? K : ((K % 8 <= 2 || (K % 8 <= 4 && K > 8)) ? 8 * (K / 8) : 8 * ((K + 7) / 8));
    static constexpr bool hasSA = ND < K;
    static constexpr int NSA = hasSA ? K - ND : 0;
    // P = U V^T: columns [0,KD) by DMMA (4 per instruction), [KD,K) by DFMA
    static constexpr int KD = (K % 4 == 0) ? K : ((K % 4 == 3 && !hasSA) ? 4 * KC : 4 * (K / 4));
    static constexpr bool hasSP = KD < K;
    static constexpr int NSP = hasSP ? K - KD : 0;
    static constexpr int C0 = hasSA ? ND : KD;                  // first V column the DFMA part reads
    static constexpr int NS = (hasSA || hasSP) ? K - C0 : 0;    // <= 4
    static constexpr int NAD = ND / 8;
    static constexpr int KCD = KD / 4;
    static constexpr int NV = 2 * NAD + (hasSA ? 1 : 0);        // update values a lane ends up with
    static_assert(NS <= 4 && C0 % 4 == 0, "remainder layout");
};

#ifndef NMFK_DMMA_MAXT
#define NMFK_DMMA_MAXT 640
#endif
__host__ __device__ constexpr int dmma_max_threads(int K) { return K <= 12 ? NMFK_DMMA_MAXT : 512; }
__host__ __device__ constexpr int dmma_nv_max(int KC) { return 2 * ((KC + 1) / 2) + 1; }
__host__ __device__ constexpr int round8(int x) { return (x + 7) & ~7; }

struct DmmaSmem {
    size_t off_W, off_H, off_den, off_scr, off_red, off_idx, off_first, off_ticket, total;
    __host__ __device__ static DmmaSmem make(int n, int m, int KC, int SH, int SW) {
        DmmaSmem r;
        auto al = [](size_t x) { return (x + 15) & ~size_t(15); };
        const int pitch = dmma_pitch(KC), NV = dmma_nv_max(KC);
        size_t o = 0;
        r.off_W = o;
        o = al(o + (size_t)round8(n) * pitch * 8);
        r.off_H = o;
        o = al(o + (size_t)round8(m) * pitch * 8);
        r.off_den = o;
        o = al(o + 40 * 8);
        r.off_scr = o;
        size_t scr = 0;
        if (SH > 1) scr = (size_t)SH * ((m + 7) / 8) * NV * 32;
        if (SW > 1 && (size_t)SW * ((n + 7) / 8) * NV * 32 > scr) scr = (size_t)SW * ((n + 7) / 8) * NV * 32;
        o = al(o + scr * 8);
        r.off_red = o;
        o = al(o + 40 * 8);
        r.off_idx = o;
        o = al(o + (size_t)m * 4);
        r.off_first = o;
        o = al(o + 40 * 4);
        r.off_ticket = o;
        o = al(o + 16);
        r.total = o;
        return r;
    }
};

// den[a] = sum_t V[t][a] for a < k (runtime pitch version of factor_sums)
__device__ __forceinline__ void factor_sums_p(const double* __restrict__ V, int nred, int pitch, int k, double* den) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int a = w; a < k; a += nw) {
        double s0 = 0.0, s1 = 0.0;
        int t = lane;
        for (; t + 32 < nred; t += 64) {
            s0 += V[(size_t)t * pitch + a];
            s1 += V[(size_t)(t + 32) * pitch + a];
        }
        if (t < nred) s0 += V[(size_t)t * pitch + a];
        const double s = warp_sum(s0 + s1);
        if (lane == 0) den[a] = s;
    }
}

// x / p as x * (1/p): MUFU.RCP64H seed r0 (relative error e, |e| <= ~2^-20: the unit works on the upper
// 32 bits of p) refined by one cubic step r = r0 (1 + e + e^2), error e^3 < 2^-60, then rounded once more
// by the multiplication: <= 1 ulp from the IEEE quotient with 3 DFMA + 1 DMUL (the Newton pair needs 5).
// No range check: operands outside the valid range (0, subnormal, Inf, NaN) turn the quotient into
// NaN, which the caller detects.
__device__ __forceinline__ double div_fast(double x, double p) {
    double r0;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"(p));
    const double e = fma(-p, r0, 1.0);
    const double t = fma(e, e, e);
    const double q0 = x * r0;
    return fma(q0, t, q0);
}

// Registers of one work item: A-fragments of U (DMMA part), U remainder columns, accumulators.
// (SETS = 2 would give even / odd tiles their own accumulators; measured: the dependent-issue latency
// of a DMMA is 26 cycles against 16 issue cycles, 5 warps per scheduler hide it, and the second set
// only costs registers - tools/probe/dmma_lat.cu.)
template <int K>
struct DmmaRegs {
    using C = DmmaCfg<K>;
    static constexpr int NADx = dmma_cmax(C::NAD, 1), NSAx = dmma_cmax(C::NSA, 1);
    double ua[dmma_cmax(C::KCD, 1)];
    double us[dmma_cmax(C::NSP, 1)];
    static constexpr int SETS = 1;  // accumulator sets a caller may alternate between (dmma_tiles SET0)
    double acc[SETS][NADx][2];
    double as[SETS][NSAx];
    __device__ __forceinline__ void load(const double* __restrict__ urow, int q) {
#pragma unroll
        for (int kc = 0; kc < C::KCD; ++kc) ua[kc] = urow[kc * 4 + q];
#pragma unroll
        for (int j = 0; j < C::NSP; ++j) us[j] = urow[C::KD + j];
    }
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int s = 0; s < SETS; ++s) {
#pragma unroll
            for (int na = 0; na < NADx; ++na) acc[s][na][0] = acc[s][na][1] = 0.0;
#pragma unroll
            for (int j = 0; j < NSAx; ++j) as[s][j] = 0.0;
        }
    }
    // fold the second accumulator set into the first and combine the 4 per-quad partial sums of the
    // DFMA columns; afterwards value(v) is valid
    __device__ __forceinline__ void finish() {
        if constexpr (SETS == 2) {
#pragma unroll
            for (int na = 0; na < C::NAD; ++na) {
                acc[0][na][0] += acc[SETS - 1][na][0];
                acc[0][na][1] += acc[SETS - 1][na][1];
            }
        }
#pragma unroll
        for (int j = 0; j < C::NSA; ++j) {
            double v = SETS == 2 ? as[0][j] + as[SETS - 1][j] : as[0][j];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            as[0][j] = v;
        }
    }
    // NaN anywhere in this lane's (finished) accumulators?
    __device__ __forceinline__ bool poisoned() const {
        double s = 0.0;
#pragma unroll
        for (int na = 0; na < C::NAD; ++na) s += acc[0][na][0] + acc[0][na][1];
#pragma unroll
        for (int j = 0; j < C::NSA; ++j) s += as[0][j];
        return s != s;
    }
    // v-th update value of this lane and its column: v < 2*NAD -> DMMA accumulator, else the DFMA column ND+q
    __device__ __forceinline__ double value(int v, int q) const {
        if (v < 2 * C::NAD) return acc[0][v >> 1][v & 1];
        double r = as[0][0];
#pragma unroll
        for (int j = 1; j < C::NSA; ++j) r = (q == j) ? as[0][j] : r;
        return r;
    }
    __device__ __forceinline__ static int column(int v, int q) {
        if (v < 2 * C::NAD) return (v >> 1) * 8 + 2 * q + (v & 1);
        return (q < C::NSA) ? C::ND + q : K;  // K = no column
    }
};

// Column c of a tile's P / Q block is step sigma(c) of the tile, sigma = (0,1,2,3,5,4,7,6): shared
// memory serves 64-bit loads per HALF warp, and with the row pitch 4*odd both B-fragment patterns
// (rows sigma(g) for P, rows sigma(2q+e) for ACC) then touch 16 distinct bank pairs per half warp.
__device__ __forceinline__ int dmma_sigma(int c) { return c < 4 ? c : (c ^ 1); }

// NT (1 or 2) consecutive 8-own x 8-step tiles, instruction streams interleaved.  For tile j:
// vp1 + j*8*pitch -> V[t0+sigma(g)][q]; vp2a/vp2b -> V[t0+sigma(2q)][g], V[t0+sigma(2q+1)][g];
// x[j][0..1] = this lane's X values at those two steps.  Tile j accumulates into set (SET0 + j) % SETS.
// MODE 0: fast reciprocal, no range check (the caller tests the accumulators for NaN and redoes the item);
// MODE 1: IEEE divisions, steps beyond the end masked; MODE 2: fast reciprocal with a warp-uniform range
// check that falls back to IEEE divisions (tiled engine: an item cannot be redone once its V chunks are gone).
// DIV: the quotient of NMF.jl's KL update (Variant KL_DIV), x / (p + kKlDivDelta).
template <int K, int MODE, int NT, int SET0, bool DIV = false>
__device__ __forceinline__ void dmma_tiles(DmmaRegs<K>& R, const double (&x)[NT][2], const double* __restrict__ vp1,
                                           const double* __restrict__ vp2a, const double* __restrict__ vp2b, int g,
                                           const bool (&in)[NT][2], bool hi_ok) {
    using C = DmmaCfg<K>;
    constexpr int TS = 8 * C::pitch;  // doubles between consecutive tiles
    double vs[NT][2][4];
    double p[NT][2], qv[NT][2];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
        const double* vpsa = vp2a + j * TS + (C::C0 - g);
        const double* vpsb = vp2b + j * TS + (C::C0 - g);
        if constexpr (C::NS == 1) {
            vs[j][0][0] = vpsa[0];
            vs[j][1][0] = vpsb[0];
        } else if constexpr (C::NS > 1) {
#pragma unroll
            for (int i = 0; i < (C::NS + 1) / 2; ++i) {
                const double2 a = *reinterpret_cast<const double2*>(vpsa + 2 * i);
                const double2 b = *reinterpret_cast<const double2*>(vpsb + 2 * i);
                vs[j][0][2 * i] = a.x;
                vs[j][0][2 * i + 1] = a.y;
                vs[j][1][2 * i] = b.x;
                vs[j][1][2 * i + 1] = b.y;
            }
        }
        p[j][0] = p[j][1] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < C::NSP; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            p[j][0] = fma(R.us[i], vs[j][0][C::KD - C::C0 + i], p[j][0]);
            p[j][1] = fma(R.us[i], vs[j][1][C::KD - C::C0 + i], p[j][1]);
        }
#pragma unroll
    for (int kc = 0; kc < C::KCD; ++kc)
#pragma unroll
        for (int j = 0; j < NT; ++j) dmma884(p[j], R.ua[kc], vp1[j * TS + kc * 4]);
    if constexpr (DIV) {
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            p[j][0] += kKlDivDelta<double>;
            p[j][1] += kKlDivDelta<double>;
        }
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) {
        if constexpr (MODE == 1) {
            qv[j][0] = in[j][0] ? div_cold<double>(x[j][0], p[j][0]) : 0.0;  // steps beyond the end contribute nothing
            qv[j][1] = in[j][1] ? div_cold<double>(x[j][1], p[j][1]) : 0.0;
        } else if constexpr (MODE == 2) {
            qv[j][0] = div_fast(x[j][0], p[j][0]);
            qv[j][1] = div_fast(x[j][1], p[j][1]);
            const bool ok = p[j][0] > 1e-290 && p[j][0] < 1e290 && p[j][1] > 1e-290 && p[j][1] < 1e290 &&
                            x[j][0] < 1e290 && x[j][1] < 1e290;  // false for NaN operands too
            if (__any_sync(0xffffffffu, !ok)) {
                qv[j][0] = div_cold<double>(x[j][0], p[j][0]);
                qv[j][1] = div_cold<double>(x[j][1], p[j][1]);
            }
        } else {
            qv[j][0] = div_fast(x[j][0], p[j][0]);
            qv[j][1] = div_fast(x[j][1], p[j][1]);
        }
    }
#pragma unroll
    for (int na = 0; na < C::NAD; ++na) {
        double b[NT][2];
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            if constexpr (C::ND <= C::pitch) {
                b[j][0] = vp2a[j * TS + na * 8];
                b[j][1] = vp2b[j * TS + na * 8];
            } else {
                // K = 3, 4: the row pitch is 4, lanes whose B column lies beyond it supply zeros.  The
                // selected values are pinned in registers: the compiler otherwise predicates the
                // (warp-collective) DMMA itself on the per-lane condition, which hangs the warp.
                const bool ok = (na * 8 + 8 <= C::pitch) || hi_ok;
                b[j][0] = ok ? vp2a[j * TS + na * 8] : 0.0;
                b[j][1] = ok ? vp2b[j * TS + na * 8] : 0.0;
                asm volatile("" : "+d"(b[j][0]), "+d"(b[j][1]));
            }
        }
#pragma unroll
        for (int e = 0; e < 2; ++e)
#pragma unroll
            for (int j = 0; j < NT; ++j) dmma884(R.acc[(SET0 + j) % DmmaRegs<K>::SETS][na], qv[j][e], b[j][e]);
    }
#pragma unroll
    for (int i = 0; i < C::NSA; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            double& d = R.as[(SET0 + j) % DmmaRegs<K>::SETS][i];
            d = fma(qv[j][0], vs[j][0][i], d);
            d = fma(qv[j][1], vs[j][1][i], d);
        }
}

// One half-update.  D: STEP-contiguous data (element (o,t) at D[t + o*nred]).
// Work items = (row group of 8 own indices) x (slice of the reduction range), dealt round-robin
// to the warps.
template <int K, bool TRANSPOSED, bool HASNAN>
__device__ __forceinline__ void dmma_half_update(const double* __restrict__ D, int nown, int nred, int k, int S,
                                                 double* __restrict__ U, const double* __restrict__ V,
                                                 const double* __restrict__ den, double* __restrict__ scr,
                                                 bool first_iter, double lambda, const double* __restrict__ ximp,
                                                 int ldimp, int* __restrict__ ticket) {
    using C = DmmaCfg<K>;
    constexpr int pitch = C::pitch;
    constexpr int NV = C::NV;
    constexpr int PF = 8;  // tiles of X kept in flight per lane (X is L2-resident but ~800 cycles away)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int G = (nown + 7) >> 3;
    const unsigned tiles_total = (unsigned)(nred + 7) >> 3;
    const int tiles_full = ((nred & 1) == 0) ? (nred >> 3) : 0;  // tiles a lane can fetch with one 16-byte load
    const int items = G * S;
    const bool hi_ok = (C::ND - 8 + g) < pitch;
    const int sw = q >> 1;                          // sigma swaps the two steps of a lane for q >= 2
    const int sa = 2 * q + sw, sb = 2 * q + 1 - sw;  // steps (within a tile) of this lane's columns 2q, 2q+1
    const int off1 = dmma_sigma(g) * pitch + q;
    const int off2a = sa * pitch + g, off2b = sb * pitch + g;

    // .x / .y of a loaded pair are the steps 2q, 2q+1 of the tile (memory order)
    auto load_tail = [&](const double* ptr, int tile) -> double2 {  // partial / unaligned tile
        const int t = tile * 8 + 2 * q;
        double2 r;
        r.x = (t < nred) ? __ldg(ptr) : 0.0;
        r.y = (t + 1 < nred) ? __ldg(ptr + 1) : 0.0;
        return r;
    };
    auto fix_nan = [&](double& x, int t, int rowc) {
        if (HASNAN) {
            if (x != x)
                x = first_iter ? lambda
                               : ximp[TRANSPOSED ? ((size_t)t + (size_t)rowc * ldimp) : ((size_t)rowc + (size_t)t * ldimp)];
        }
    };

    // items are handed out dynamically (the first NW statically): *ticket was set to NW before the
    // barrier that precedes this call.  Which warp runs an item does not affect the result.
    int item = warp;
    while (item < items) {
        const int grp = item % G, slice = item / G;
        const int row = grp * 8 + g;
        const bool rvalid = row < nown;
        const int rowc = rvalid ? row : nown - 1;  // invalid rows shadow the last valid one; never stored
        const int tb = (int)((tiles_total * (unsigned)slice) / (unsigned)S);
        const int te = (int)((tiles_total * (unsigned)(slice + 1)) / (unsigned)S);
        const int tef = min(te, tiles_full);  // tiles [tb, tef) take the vector load
        DmmaRegs<K> R;
        R.load(U + (size_t)rowc * pitch, q);
        R.zero();
        const double* xrow = D + (size_t)rowc * nred + 2 * q;
        const double* xp = xrow + (size_t)tb * 8;  // advances with the consumed tile
        double2 xq[PF];
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            const int tile = tb + u;
            if (tile < tef)
                xq[u] = __ldg(reinterpret_cast<const double2*>(xp + u * 8));
            else if (tile < te)
                xq[u] = load_tail(xp + u * 8, tile);
            else
                xq[u] = make_double2(0.0, 0.0);
        }
        const double* vb = V + (size_t)tb * (8 * pitch);
        const double* vp1 = vb + off1;
        const double* vp2a = vb + off2a;
        const double* vp2b = vb + off2b;
        const bool inall[1][2] = {{true, true}};
        auto take = [&](int u, int tile, double (&x)[2]) {  // consume ring slot u, refill it PF tiles ahead
            x[0] = sw ? xq[u].y : xq[u].x;
            x[1] = sw ? xq[u].x : xq[u].y;
            if (tile + PF < tef)
                xq[u] = __ldg(reinterpret_cast<const double2*>(xp + PF * 8));
            else if (tile + PF < te)
                xq[u] = load_tail(xp + PF * 8, tile + PF);
            fix_nan(x[0], tile * 8 + sa, rowc);
            fix_nan(x[1], tile * 8 + sb, rowc);
        };
        for (int tile0 = tb; tile0 < te; tile0 += PF) {
#pragma unroll
            for (int u = 0; u < PF; ++u) {
                const int tile = tile0 + u;
                if (tile < te) {  // warp-uniform
                    double x[1][2];
                    take(u, tile, x[0]);
                    dmma_tiles<K, 0, 1, 0>(R, x, vp1, vp2a, vp2b, g, inall, hi_ok);
                    xp += 8;
                    vp1 += 8 * pitch;
                    vp2a += 8 * pitch;
                    vp2b += 8 * pitch;
                }
            }
        }
        R.finish();
        if (__any_sync(0xffffffffu, R.poisoned())) {
            // rare: some quotient left the fast reciprocal's range -> redo the item with IEEE semantics
            // (x/0 = Inf, 0/0 = NaN, ...) so degenerate restarts match the reference's Inf/NaN pattern
            R.zero();
            for (int tile = tb; tile < te; ++tile) {
                const double2 x = load_tail(xrow + (size_t)tile * 8, tile);
                double x0 = sw ? x.y : x.x, x1 = sw ? x.x : x.y;
                const int ta = tile * 8 + sa, tb2 = tile * 8 + sb;
                fix_nan(x0, ta, rowc);
                fix_nan(x1, tb2, rowc);
                const double* vt = V + (size_t)tile * (8 * pitch);
                const double xx[1][2] = {{x0, x1}};
                const bool in1[1][2] = {{ta < nred, tb2 < nred}};
                dmma_tiles<K, 1, 1, 0>(R, xx, vt + off1, vt + off2a, vt + off2b, g, in1, hi_ok);
            }
            R.finish();
        }
        if (S == 1) {
            // (U .* acc) ./ den : the rows of this group are read by this warp only
#pragma unroll
            for (int v = 0; v < NV; ++v) {
                const int a = DmmaRegs<K>::column(v, q);
                if (rvalid && a < k) {
                    double* up = U + (size_t)row * pitch + a;
                    *up = div_cold<double>(*up * R.value(v, q), den[a]);
                }
            }
        } else {
            double* dst = scr + (size_t)(slice * G + grp) * (NV * 32) + lane;
#pragma unroll
            for (int v = 0; v < NV; ++v) dst[v * 32] = R.value(v, q);
        }
        int nxt = 0;
        if (lane == 0) nxt = atomicAdd(ticket, 1);
        item = __shfl_sync(0xffffffffu, nxt, 0);
    }
    __syncthreads();
    if (S > 1) {
        for (int grp = warp; grp < G; grp += NW) {
            const int row = grp * 8 + g;
            const bool rvalid = row < nown;
#pragma unroll
            for (int v = 0; v < NV; ++v) {
                double s = 0.0;
                for (int sl = 0; sl < S; ++sl) s += scr[(size_t)(sl * G + grp) * (NV * 32) + v * 32 + lane];
                const int a = DmmaRegs<K>::column(v, q);
                if (rvalid && a < k) {
                    double* up = U + (size_t)row * pitch + a;
                    *up = div_cold<double>(*up * s, den[a]);
                }
            }
        }
        __syncthreads();
    }
}

// MODE 0: sum over non-NaN of ((x-p)w)^2 and (x-p)^2 (RESTORE: substituted zeros count as 0);
// MODE 1: imputation X[inan] = (W*H)[inan] into ximp (X layout).
// Xt is the step-contiguous copy of X (element (row i, column t) at Xt[t + i*m]): a lane's two
// elements of a tile are one 16-byte load, 4 tiles in flight.
template <int K, int MODE, bool RESTORE>
__device__ __forceinline__ double2 dmma_residual_pass(const double* __restrict__ Xt, int n, int m,
                                                      const double* __restrict__ Ws, const double* __restrict__ Hs,
                                                      double lambda, double weight, double* __restrict__ ximp,
                                                      double* red) {
    constexpr int KC = DmmaCfg<K>::KC;
    constexpr int pitch = DmmaCfg<K>::pitch;
    constexpr int UN = 4;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int G = (n + 7) >> 3, tiles = (m + 7) >> 3, tiles_full = m >> 3;
    const bool vec_ok = ((m & 1) == 0);
    double sw = 0.0, s1 = 0.0;
    for (int grp = warp; grp < G; grp += NW) {
        const int row = grp * 8 + g;
        const bool rvalid = row < n;
        const int rowc = rvalid ? row : n - 1;
        double ua[KC];
#pragma unroll
        for (int kc = 0; kc < KC; ++kc) ua[kc] = Ws[(size_t)rowc * pitch + kc * 4 + q];
        for (int tile0 = 0; tile0 < tiles; tile0 += UN) {
            double2 xv[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int tile = tile0 + u;
                const double* ptr = Xt + (size_t)rowc * m + (size_t)tile * 8 + 2 * q;
                const int t = tile * 8 + 2 * q;
                if (vec_ok && tile < tiles_full) {
                    xv[u] = __ldg(reinterpret_cast<const double2*>(ptr));
                } else {
                    xv[u].x = (t < m) ? __ldg(ptr) : 0.0;
                    xv[u].y = (t + 1 < m) ? __ldg(ptr + 1) : 0.0;
                }
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int tile = tile0 + u;
                if (tile < tiles) {  // warp-uniform
                    double p[2] = {0.0, 0.0};
                    const double* vrow = Hs + (size_t)(tile * 8 + g) * pitch + q;  // pad rows exist (ones)
#pragma unroll
                    for (int kc = 0; kc < KC; ++kc) dmma884(p, ua[kc], vrow[kc * 4]);
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int t = tile * 8 + 2 * q + e;
                        const double xr = e ? xv[u].y : xv[u].x;
                        if (!rvalid || t >= m) continue;
                        if (MODE == 0) {
                            if (xr != xr) continue;
                            double x = xr;
                            if (RESTORE && x == lambda) x = 0.0;
                            const double d = x - p[e];
                            s1 = fma(d, d, s1);
                            const double dw = d * weight;
                            sw = fma(dw, dw, sw);
                        } else {
                            if (xr != xr) ximp[(size_t)row + (size_t)t * n] = p[e];
                        }
                    }
                }
            }
        }
    }
    double2 out;
    out.x = out.y = 0.0;
    if (MODE == 0) {
        out.x = block_sum(sw, red);
        out.y = block_sum(s1, red);
    } else {
        __syncthreads();
    }
    return out;
}

template <int K, bool HASNAN>
__global__ void __launch_bounds__(dmma_max_threads(K), 1) kl_resident_dmma_kernel(const SolveArgs a) {
    constexpr int KC = DmmaCfg<K>::KC;
    constexpr int pitch = DmmaCfg<K>::pitch;
    extern __shared__ __align__(16) unsigned char smem[];
    const int n = a.n, m = a.m, k = a.k;
    const int r = blockIdx.x;
    const int tid = threadIdx.x, NT = blockDim.x;
    UnitState* stg = a.st + r;
    if (stg->done) return;
    if (a.iter_limit > 0 && a.iter_limit < a.maxiter && stg->it >= a.iter_limit) return;  // paused beyond this launch

    const DmmaSmem L = DmmaSmem::make(n, m, KC, a.SH, a.SW);
    double* Ws = reinterpret_cast<double*>(smem + L.off_W);
    double* Hs = reinterpret_cast<double*>(smem + L.off_H);
    double* den = reinterpret_cast<double*>(smem + L.off_den);
    double* scr = reinterpret_cast<double*>(smem + L.off_scr);
    double* red = reinterpret_cast<double*>(smem + L.off_red);
    int* idx = reinterpret_cast<int*>(smem + L.off_idx);
    int* first = reinterpret_cast<int*>(smem + L.off_first);
    int* ticket = reinterpret_cast<int*>(smem + L.off_ticket);

    const double* X = static_cast<const double*>(a.X);
    const double* Xt = static_cast<const double*>(a.Xt);
    double* Wg = static_cast<double*>(a.W) + (size_t)r * n * k;
    double* Hg = static_cast<double*>(a.H) + (size_t)r * k * m;
    int* canon_old = a.canon + (size_t)r * m;
    double* ximp = HASNAN ? static_cast<double*>(a.ximp) + (size_t)r * n * m : nullptr;
    const double lambda = a.lambda;

    // padding columns zero; padding rows (n..round8(n), m..round8(m)) ones: see the file header
    const int n8 = round8(n), m8 = round8(m);
    for (int e = tid; e < n8 * pitch; e += NT) Ws[e] = (e >= n * pitch) ? 1.0 : 0.0;
    for (int e = tid; e < m8 * pitch; e += NT) Hs[e] = (e >= m * pitch) ? 1.0 : 0.0;
    __syncthreads();
    for (int e = tid; e < n * k; e += NT) Ws[(size_t)(e % n) * pitch + e / n] = Wg[e];
    for (int e = tid; e < k * m; e += NT) Hs[(size_t)(e / k) * pitch + e % k] = Hg[e];
    __syncthreads();

    int it = stg->it, bad = stg->bad, re = stg->re, inc = stg->inc, has_cons = stg->has_cons;
    double best = stg->best, obj_chk = stg->obj_chk;
    int stop = 0;
    __syncthreads();

    if (HASNAN && it > 0) dmma_residual_pass<K, 1, false>(Xt, n, m, Ws, Hs, lambda, 1.0, ximp, red);

    while (true) {
        if (it >= a.maxiter) {  // :64
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
        if (a.iter_limit > 0 && it >= a.iter_limit) break;
        ++it;
        const bool first_iter = (it == 1);
        if (!a.Hfixed) {  // :66-68
            factor_sums_p(Ws, n, pitch, k, den);
            if (tid == 0) *ticket = NT >> 5;
            __syncthreads();
            dmma_half_update<K, true, HASNAN>(X, m, n, k, a.SH, Hs, Ws, den, scr, first_iter, lambda, ximp, n, ticket);
        }
        if (!a.Wfixed) {  // :69-71
            factor_sums_p(Hs, m, pitch, k, den);
            if (tid == 0) *ticket = NT >> 5;
            __syncthreads();
            dmma_half_update<K, false, HASNAN>(Xt, n, m, k, a.SW, Ws, Hs, den, scr, first_iter, lambda, ximp, n, ticket);
        }
        if (HASNAN) dmma_residual_pass<K, 1, false>(Xt, n, m, Ws, Hs, lambda, 1.0, ximp, red);  // :72
        if (it % a.check_every == 0) {                                                          // :73
            const double2 ob = dmma_residual_pass<K, 0, false>(Xt, n, m, Ws, Hs, lambda, a.weight, nullptr, red);
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
            const double epsc = a.eps_clamp;  // :99-100
            for (int e = tid; e < n * pitch; e += NT) {
                if (e % pitch < k) {
                    const double v = Ws[e];
                    Ws[e] = (v != v) ? v : (v < epsc ? epsc : v);
                }
            }
            for (int e = tid; e < m * pitch; e += NT) {
                if (e % pitch < k) {
                    const double v = Hs[e];
                    Hs[e] = (v != v) ? v : (v < epsc ? epsc : v);
                }
            }
            if (tid < 36) first[tid] = INT_MAX;
            __syncthreads();
            for (int j = tid; j < m; j += NT) {  // :101-103
                const double* h = Hs + (size_t)j * pitch;
                double bv = h[0];
                int bi = 0;
                for (int c = 1; c < k; ++c) {
                    const double v = h[c];
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
            int same = 1;  // :105-111
            for (int j = tid; j < m; j += NT) {
                const int c = first[idx[j]];
                if (!has_cons || canon_old[j] != c) same = 0;
                idx[j] = c;
            }
            same = __syncthreads_and(same);
            if (same)
                ++inc;
            else
                inc = 0;
            if (inc > a.stopconv) {  // :112-115
                stop = 4;
                break;
            }
            for (int j = tid; j < m; j += NT) canon_old[j] = idx[j];  // :116
            has_cons = 1;
            __syncthreads();
        }
    }

    double obj_ssq = stg->obj_ssq, obj_norm = stg->obj_norm;
    int done = 0;
    if (stop != 0) {
        const double2 ob = dmma_residual_pass<K, 0, true>(Xt, n, m, Ws, Hs, lambda, a.weight, nullptr, red);
        obj_ssq = ob.x;           // NMFkMultiplicative.jl:125
        obj_norm = sqrt(ob.y);    // NMFkExecute.jl:792
        if (a.normalize == 1) {   // NMFkExecute.jl:800-804
            factor_sums_p(Hs, m, pitch, k, den);
            __syncthreads();
            for (int e = tid; e < n * pitch; e += NT)
                if (e % pitch < k) Ws[e] = Ws[e] * den[e % pitch];
            for (int e = tid; e < m * pitch; e += NT)
                if (e % pitch < k) Hs[e] = div_cold<double>(Hs[e], den[e % pitch]);
        } else if (a.normalize == 2) {  // :796-799
            factor_sums_p(Ws, n, pitch, k, den);
            __syncthreads();
            for (int e = tid; e < n * pitch; e += NT)
                if (e % pitch < k) Ws[e] = div_cold<double>(Ws[e], den[e % pitch]);
            for (int e = tid; e < m * pitch; e += NT)
                if (e % pitch < k) Hs[e] = Hs[e] * den[e % pitch];
        }
        done = 1;
        __syncthreads();
    }
    for (int e = tid; e < n * k; e += NT) Wg[e] = Ws[(size_t)(e % n) * pitch + e / n];
    for (int e = tid; e < k * m; e += NT) Hg[e] = Hs[(size_t)(e / k) * pitch + e % k];
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

}  // namespace nmfk
