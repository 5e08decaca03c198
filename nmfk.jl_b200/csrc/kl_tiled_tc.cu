// Float32 half-update of the tiled KL engine on the 5th-generation tensor cores (tcgen05 / tensor memory).
//
// Replaces, for Float32 data without NaN, the loop body of NMFk.NMFmultiplicative
// (/root/reference/src/NMFkMultiplicative.jl:67,70) exactly like tiled_pass_kernel (kl_tiled.cuh) does:
//   ACC[o,a] = sum_t (D[o,t] / (U[o,:] . V[t,:])) V[t,a]      then  U[o,a] <- U[o,a] ACC[o,a] / den[a]
// (H-update: D = X^T, U = H^T, V = W;  W-update: D = X, U = W, V = H^T).
//
// One CTA = 128 own indices (the 128 lanes of tensor memory) x one slice of the reduction range x a GROUP of
// RB restarts that share every X tile.  The reduction range is walked in chunks of TS = 64 steps; a "unit" is
// one (chunk, restart) pair:
//   MMA#1  P[128 x 64]  = U_r[128 x k] V_r[64 x k]^T      A = U (hi, lo) in tensor memory, B = V chunk in smem
//   quot.  Q = X_tile ./ P  in registers (tcgen05.ld, MUFU.RCP, tcgen05.st), split Q = Qhi + Qlo (TF32 + rest)
//   MMA#2  ACC_r[128 x k] += Q[128 x 64] V_r[64 x k]      A = Q (hi, lo) in tensor memory, B = V chunk in smem
// Both products use the 3-term TF32 split (hi*hi + lo*hi + hi*lo, FP32 accumulation; never plain TF32).
// Warp roles (704 threads): warp 0 = bulk-copy producer of X tiles (cp.async.bulk + mbarrier transaction
// counts, 3 stages), warp 1 = tcgen05.mma issuer (elect.sync regions), warps 2-5 = V stagers (cp.async two units
// ahead -> hi/lo split -> the two canonical un-swizzled K-major images MMA#1 and MMA#2 read), warps 6-21 =
// quotient warps (lane quarter = warp % 4): two GROUPS of 8 warps that alternate units (32 of the 64 columns per
// thread), so one group divides while the other waits for the tensor-pipe round trip of its P tile.  P/Q tiles are
// double-buffered in tensor memory (one buffer per group; a third one when k <= 8).  With OBJ the same machinery
// computes the objective sums (MMA#1 only, 16 warps x 16 columns in lockstep).
// tcgen05.mma accumulates with round-toward-zero (measured: -0.47 ulp per chained instruction, tools/umma_selftest.py
// --timing), so numerators are NOT chained across units: MMA#2 of every unit starts a fresh tensor-memory
// accumulator (8 chained K-steps) that the quotient warps add into FP32 registers with round-to-nearest.
// Tensor-memory map (512 columns): [0,256) two P/Q buffers (64 P->Qhi + 64 Qlo), then two per-unit numerator
// buffers (NST*N2 columns each; k <= 16 stacks Qhi*[Vhi;Vlo] into one N = 32 instruction), then U hi | U lo
// (K8 each) per restart of the group.
// 32 < k <= 64 (N2 = 64): 256 + 128 + 2 K8 columns leave room for ONE restart per CTA (RB = 1; X tiles are no longer shared
// between restarts, they come from L2 for the other restarts' CTAs); the two quotient groups then alternate chunks of the
// same restart and add their numerators at the end.  Shared memory: 2 X stages + 2 V images (64 KB each at K8 = 64) + 2 raw
// chunks = 224 KB.
#include <algorithm>

#include "kl_tiled_args.h"
#include "tc_ptx.cuh"
#include "tc_stage.cuh"

namespace nmfk {
namespace {

constexpr int TC_M = 128;

// K8 / N2: k rounded up to the K granularity of MMA#1 (8) / the N granularity of MMA#2 (16).
// One CTA per SM: chunks of 64 steps, 16 quotient + 4 stager warps, all 512 tensor-memory columns.  (A configuration with
// TWO CTAs per SM - chunks of 32 steps, 8 quotient + 2 stager warps, 256 columns each - measured slower on C3, 3083 vs
// 3489 restart-iterations/s at the time: the per-unit hand-offs are paid twice as often.  It was removed.)
template <int K8, int N2>
struct TcCfg {
    static constexpr int TS = 64;                                     // steps per chunk
    // X tile stages, raw V chunk buffers, V image buffers: fewer as the V images grow (shared memory budget for k > 16 / 32)
    static constexpr int NXS = K8 <= 32 ? 3 : 2;
    static constexpr int NRAW = K8 <= 32 ? 4 : 2;
    static constexpr int NVB = K8 <= 16 ? 4 : (K8 <= 32 ? 3 : 2);
    static constexpr int RPAD = K8 > 24 ? 0 : 4;                      // raw V chunk padding (shared memory budget at K8 = 32)
    static constexpr int QW = TS / 4;                                 // quotient warps: lane quarter = warp % 4, 16 columns each
    static constexpr int SW = 4;                                      // V stager warps
    static constexpr int QW0 = 2 + SW;                                // first quotient warp
    static constexpr int THREADS = (QW0 + QW) * 32;
    static constexpr int TCOLS = 512;                                 // tensor-memory columns of the CTA
    static constexpr int NCS = QW / 4;                                // column groups of quotient warps
    static constexpr int NST = N2 == 16 ? 2 : 1;                      // MMA#2: Qhi * [Vhi ; Vlo] stacked along N
    static constexpr int ACOLS = NST * N2;                            // columns of one per-unit numerator buffer
    static constexpr int PQ = 2 * TS;                                 // one P/Q buffer: P -> Qhi | Qlo
    // P/Q buffers.  With two, MMA#1(u) can only be issued after MMA#2(u-2) (same buffer), i.e. after the quotient group of
    // unit u has finished its previous unit.  A third buffer lets MMA#1 run three units ahead.  Tensor memory has room
    // for it with RB = 4 restarts per CTA only when k <= 8 (C3 shape at k = 8: 6494 against 5982 restart-iterations/s);
    // at k = 16 it would leave RB = 2 and measured 5030-5100 against 5460 with two buffers and RB = 4.
    static constexpr int NPQ = K8 <= 8 ? 3 : 2;
    static constexpr int NAB3 = 2;                                    // per-unit numerator buffers (one per quotient group)
    static constexpr int ABASE = NPQ * PQ, UBASE = ABASE + NAB3 * ACOLS;  // tensor-memory columns
    static constexpr int PERB = 2 * K8;                               // U hi | U lo per restart
    static constexpr int NCQ = N2 / NCS;                              // numerator columns per quotient thread
    static constexpr int RBT = (TCOLS - UBASE) / PERB;
    static constexpr int RBR = 16 / NCQ;                              // 16 accumulator registers per quotient thread
    static constexpr int RB0 = RBT < RBR ? RBT : RBR;
    static constexpr int RB = RB0 < NCS ? RB0 : NCS;                  // restarts per CTA (they share the X tiles)
    static constexpr uint32_t SBO1 = (K8 / 4) * 128;                  // MMA#1 B: rows = steps, K extent = K8
    static constexpr uint32_t SBO2 = (TS / 4) * 128;                  // MMA#2 B: rows = columns a, K extent = TS
    static constexpr uint32_t B1_BYTES = TS * K8 * 4;
    static constexpr uint32_t B2_BYTES = N2 * TS * 4;
    static constexpr uint32_t V_BYTES = 2 * B1_BYTES + 2 * B2_BYTES;  // B1 hi | B1 lo | B2 hi | B2 lo
    static constexpr uint32_t X_BYTES = TS * TC_M * 4;
    static constexpr int RAWP_T = TS + RPAD;                          // raw V chunk [column][step], padded pitch (floats)
    static constexpr int RAWP_A = K8 + RPAD;                          // raw V chunk [step][column], padded pitch
    static constexpr uint32_t RAW_BYTES = (K8 * TS + RPAD * (K8 > TS ? K8 : TS)) * 4;
    static constexpr size_t SMEM =
        (size_t)NXS * X_BYTES + (size_t)NVB * V_BYTES + (size_t)NRAW * RAW_BYTES + 32 * 8 + 64;
    static_assert(RB >= 1 && RB <= 4, "restart group");
    static_assert(SMEM <= 232448, "shared memory budget of one CTA");
};

__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(lo), "f"(hi));
    return v;
}

__device__ __forceinline__ float rcp_fast(float p) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p));
    return r;
}

// OBJ = true: objective mode.  Only MMA#1 runs (P = U V^T); the quotient warps accumulate (x - p)^2 instead of dividing,
// nothing is written back to the factors: replaces tiled_objective_kernel (NMFkMultiplicative.jl:74,125) for Float32.
template <int K8, int N2, bool OBJ>
__global__ void __launch_bounds__((TcCfg<K8, N2>::THREADS), 1) tc_pass_kernel(const TiledPassArgs a, int* errflag) {
    using C = TcCfg<K8, N2>;
    constexpr int TC_NXS = C::NXS, TC_NVB = C::NVB;
    constexpr int TC_TS = C::TS, TC_QWARPS = C::QW, TC_SWARPS = C::SW, TC_QW0 = C::QW0, TC_THREADS = C::THREADS;
    constexpr int RB = C::RB;
    extern __shared__ __align__(1024) unsigned char smem[];
    float* Xs = reinterpret_cast<float*>(smem);                         // [NXS][TS][M]
    unsigned char* Vs = smem + (size_t)TC_NXS * C::X_BYTES;              // [NVB][V_BYTES]
    float* Raw = reinterpret_cast<float*>(Vs + (size_t)TC_NVB * C::V_BYTES);  // [NRAW][RAW_BYTES]
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(Raw) + (size_t)C::NRAW * C::RAW_BYTES);
    uint64_t* x_full = bars;                 // [NXS]  X tile landed (bulk-copy transaction count)
    uint64_t* x_empty = x_full + TC_NXS;     // [NXS]  quotient warps are done with the tile
    uint64_t* v_full = x_empty + TC_NXS;     // [NVB]  V images staged
    uint64_t* v_empty = v_full + TC_NVB;     // [NVB]  MMA#1 and MMA#2 of the unit have read them
    uint64_t* p_full = v_empty + TC_NVB;     // [NPQ]  MMA#1 done: P readable
    uint64_t* q_full = p_full + C::NPQ;      // [NPQ]  Q written (and the numerator buffer of unit u-2 drained)
    uint64_t* a_full = q_full + C::NPQ;      // [2]    MMA#2 done: the unit's numerators readable
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 32);
    int* s_act = reinterpret_cast<int*>(tmem_slot + 1);  // [RB] restart of every unit slot, then the number of real ones

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t hint = (uint32_t)a.wait_hint_ns;
    long long* const trc = (a.trace != nullptr && blockIdx.x == 0) ? a.trace : nullptr;
    const int ngroups = (a.R + RB - 1) / RB;
    const int g = blockIdx.x % ngroups;
    const int rest = blockIdx.x / ngroups;
    const int ob = rest % a.nblocks;
    const int slice = rest / a.nblocks;
    const int o0 = ob * TC_M;
    const int k = a.k;
    // slices are whole chunks: every chunk starts at a multiple of 64 steps (16-byte aligned V rows)
    const int chunks_all = (a.nred + TC_TS - 1) / TC_TS;
    const int t_begin = (int)(((long long)chunks_all * slice) / a.S) * TC_TS;
    const int t_end = min(a.nred, (int)(((long long)chunks_all * (slice + 1)) / a.S) * TC_TS);
    const int nchunks = (t_end - t_begin + TC_TS - 1) / TC_TS;

    if (tid == 0) {
        int nact = 0;
        for (int b = 0; b < RB; ++b) {
            const int r = g * RB + b;
            if (r >= a.R) continue;
            const bool stopped = a.st[r].stop != 0;
            const bool take = (OBJ && a.obj_sel == 1) ? (stopped && a.st[r].done == 0) : !stopped;  // finished restarts are frozen
            if (take) s_act[nact++] = r;
        }
        s_act[RB] = nact;
        // pass mode: the two quotient groups alternate units, so a chunk holds an EVEN number of units; an odd group of
        // restarts (ragged last group, frozen restarts) gets a shadow unit that recomputes its first restart and is dropped
        // (one restart per CTA, k > 32: the groups alternate chunks instead)
        if (!OBJ && RB > 1 && (nact & 1)) s_act[nact] = s_act[0];
    }
    __syncthreads();
    const int nreal = s_act[RB];
    const int nact = (OBJ || RB == 1) ? nreal : nreal + (nreal & 1);
    if (nreal == 0 || nchunks <= 0) return;
    const int total = nchunks * nact;

    if (warp == 0) tc::tmem_alloc<C::TCOLS>(tmem_slot);
    if (tid == 32) {
        for (int i = 0; i < TC_NXS; ++i) {
            tc::mbar_init(&x_full[i], 1);
            tc::mbar_init(&x_empty[i], TC_QWARPS);
        }
        for (int i = 0; i < TC_NVB; ++i) {
            tc::mbar_init(&v_full[i], TC_SWARPS);
            tc::mbar_init(&v_empty[i], 1);
        }
        for (int i = 0; i < C::NPQ; ++i) {
            tc::mbar_init(&p_full[i], 1);
            tc::mbar_init(&q_full[i], OBJ ? TC_QWARPS : TC_QWARPS / 2);
        }
        for (int i = 0; i < 2; ++i) tc::mbar_init(&a_full[i], 1);
        tc::mbar_fence_init();
    }
    // padding rows / columns of the V images stay zero for the whole kernel; so do the own indices past the
    // edge of X in the X stages (the bulk copies of an edge tile are shorter than 128 indices)
    for (uint32_t e = tid; e < TC_NVB * C::V_BYTES / 16; e += TC_THREADS) reinterpret_cast<uint4*>(Vs)[e] = make_uint4(0, 0, 0, 0);
    if (o0 + TC_M > a.nown)
        for (uint32_t e = tid; e < TC_NXS * C::X_BYTES / 16; e += TC_THREADS) reinterpret_cast<uint4*>(Xs)[e] = make_uint4(0, 0, 0, 0);
    tc::fence_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tbase = *tmem_slot;

    const float* D = static_cast<const float*>(a.D);
    const float* Vg = static_cast<const float*>(a.V);
    float* Ug = static_cast<float*>(a.U);

    // own factor rows -> tensor memory (A operand of MMA#1), split hi / lo: quotient warp group cs loads restart
    // slot cs.  Own indices past the edge get U = 1 (finite P; their X is 0 and their rows are never stored).
    if (warp >= TC_QW0) {
        const int lq = warp & 3, cs = (warp - TC_QW0) >> 2;
        const int o = o0 + lq * 32 + lane;
        const bool valid = o < a.nown;
        const uint32_t lane_base = tbase + ((uint32_t)(lq * 32) << 16);
        if (cs < nact) {
            const float* U = Ug + (long long)s_act[cs] * a.u_rstride;
            const uint32_t col = C::UBASE + cs * C::PERB;
#pragma unroll
            for (int c0 = 0; c0 < K8; c0 += 8) {
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float u = !valid ? 1.f : (c0 + c < k ? U[(long long)o * a.su_o + (long long)(c0 + c) * a.su_a] : 0.f);
                    hi[c] = __float_as_uint(u) & 0xffffe000u;
                    lo[c] = __float_as_uint(u - __uint_as_float(hi[c]));
                }
                tc::tmem_st8(lane_base + col + c0, hi);
                tc::tmem_st8(lane_base + col + K8 + c0, lo);
            }
        }
        tc::tmem_wait_st();
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();

    if (warp == 0) {
        // ===== X producer: one bulk copy per step row (128 consecutive own indices = 512 bytes).  The whole warp runs
        // the loop; the copies are issued from an elect.sync region (single thread, uniform registers) =====
        {
            const uint32_t row_bytes = (uint32_t)min(TC_M, a.nown - o0) * 4u;
            for (int c = 0; c < nchunks; ++c) {
                const int s = c % TC_NXS;
                if (c >= TC_NXS) tc::mbar_wait_relaxed(&x_empty[s], (uint32_t)((c / TC_NXS - 1) & 1), hint & 0xffffu, errflag, 10);
                const int t0 = t_begin + c * TC_TS;
                const int cnt = min(TC_TS, t_end - t0);
                if (tc::elect_one()) {
                    tc::mbar_arrive_expect_tx(&x_full[s], (uint32_t)cnt * row_bytes);
                    float* dst = Xs + (size_t)s * TC_TS * TC_M;
                    const float* src = D + (long long)o0 + (long long)t0 * a.nown;
                    for (int j = 0; j < cnt; ++j) tc::bulk_g2s(dst + j * TC_M, src + (long long)j * a.nown, row_bytes, &x_full[s]);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the whole warp runs the (warp-uniform) control flow, lane 0 issues; descriptors are built once,
        // the unrolled issue loops only add constants =====
        {
            constexpr uint32_t idP = tc::idesc_tf32(TC_M, TC_TS, 0);
            constexpr uint32_t idA1 = tc::idesc_tf32(TC_M, C::ACOLS, 0);  // Qhi * [Vhi ; Vlo] (or Qhi * Vhi when not stacked)
            constexpr uint32_t idA2 = tc::idesc_tf32(TC_M, N2, 0);
            const uint32_t vs0 = tc::smem_u32(Vs);
            const uint64_t d1 = tc::smem_desc(vs0, TC_LBO, C::SBO1);                     // MMA#1 image of buffer 0, hi
            const uint64_t d2 = tc::smem_desc(vs0 + 2 * C::B1_BYTES, TC_LBO, C::SBO2);   // MMA#2 image of buffer 0, hi
            constexpr uint64_t KSTEP = (2 * TC_LBO) >> 4;                                // one K-step = two 16-byte chunks
            auto mma1 = [&](int u, int b) {
                const int vb = u % TC_NVB;
                TC_STAMP(1, u, 3);
                tc::mbar_wait_h(0u, &v_full[vb], (uint32_t)((u / TC_NVB) & 1), errflag, 20);
                tc::tc_fence_after_sync();
                TC_STAMP(1, u, 4);
                const uint32_t d = tbase + (uint32_t)(u % C::NPQ) * C::PQ;
                const uint32_t uh = tbase + C::UBASE + b * C::PERB, ul = uh + K8;
                const uint64_t bh = d1 + (uint64_t)((vb * C::V_BYTES) >> 4), bl = bh + (C::B1_BYTES >> 4);
                if (tc::elect_one()) {
#pragma unroll
                for (int ks = 0; ks < K8 / 8; ++ks) {
                    tc::mma_tf32_ts(d, ul + ks * 8, bh + ks * KSTEP, idP, ks > 0);
                    tc::mma_tf32_ts(d, uh + ks * 8, bl + ks * KSTEP, idP, 1);
                    tc::mma_tf32_ts(d, uh + ks * 8, bh + ks * KSTEP, idP, 1);
                }
                tc::mma_commit(&p_full[u % C::NPQ]);
                if (OBJ) tc::mma_commit(&v_empty[vb]);  // MMA#1 is the only reader of the V images
                }
                __syncwarp();
                TC_STAMP(1, u, 5);
            };
            auto mma2 = [&](int u) {
                const int vb = u % TC_NVB;
                TC_STAMP(1, u, 0);
                tc::mbar_wait_h(0u, &q_full[u % C::NPQ], (uint32_t)((u / C::NPQ) & 1), errflag, 21);
                tc::tc_fence_after_sync();
                TC_STAMP(1, u, 1);
                const uint32_t d = tbase + C::ABASE + (uint32_t)(u % C::NAB3) * C::ACOLS;
                const uint32_t qh = tbase + (uint32_t)(u % C::NPQ) * C::PQ, ql = qh + TC_TS;
                const uint64_t bh = d2 + (uint64_t)((vb * C::V_BYTES) >> 4), bl = bh + (C::B2_BYTES >> 4);
                if (tc::elect_one()) {
#pragma unroll
                for (int ks = 0; ks < TC_TS / 8; ++ks) tc::mma_tf32_ts(d, qh + ks * 8, bh + ks * KSTEP, idA1, ks > 0);
                if (C::NST == 1) {
#pragma unroll
                    for (int ks = 0; ks < TC_TS / 8; ++ks) tc::mma_tf32_ts(d, qh + ks * 8, bl + ks * KSTEP, idA2, 1);
                }
#pragma unroll
                for (int ks = 0; ks < TC_TS / 8; ++ks) tc::mma_tf32_ts(d, ql + ks * 8, bh + ks * KSTEP, idA2, 1);
                tc::mma_commit(&v_empty[vb]);
                tc::mma_commit(&a_full[u & 1]);
                }
                __syncwarp();
                TC_STAMP(1, u, 2);
            };
            // unit u = c * nact + b; MMA#1 runs NPQ units ahead of MMA#2
            int b1 = 0;  // restart slot of the next MMA#1
            auto next_b = [&](int b) { return b + 1 == nact ? 0 : b + 1; };
            for (int u0 = 0; u0 < C::NPQ && u0 < total; ++u0) {
                mma1(u0, b1);
                b1 = next_b(b1);
            }
            for (int u = 0; u < total; ++u) {
                if (OBJ) {  // no MMA#2: the P buffer is free once the quotient warps have read it
                    tc::mbar_wait_h(0u, &q_full[u % C::NPQ], (uint32_t)((u / C::NPQ) & 1), errflag, 22);
                    tc::tc_fence_after_sync();
                } else {
                    mma2(u);
                }
                if (u + C::NPQ < total) {
                    mma1(u + C::NPQ, b1);
                    b1 = next_b(b1);
                }
            }
        }
        __syncwarp();
    } else if (warp < TC_QW0) {
        tc_stager_role<C, K8, OBJ>(a, Vs, Raw, v_full, v_empty, s_act, nact, total, t_begin, t_end, 64, hint, errflag, trc);
    } else {
        // ===== quotient warps: 128 lanes x 16 columns each =====
        const int lq = warp & 3, cs = (warp - TC_QW0) >> 2;
        const int o_loc = lq * 32 + lane;
        const int o = o0 + o_loc;
        const bool valid = o < a.nown;
        const uint32_t lane_base = tbase + ((uint32_t)(lq * 32) << 16);
        const int j0 = cs * 16;
        if constexpr (OBJ) {
            // ----- objective mode: sum over this thread's (own index, 16 steps) of (x - p)^2, per restart slot -----
            double sacc[RB];
#pragma unroll
            for (int b = 0; b < RB; ++b) sacc[b] = 0.0;
            const float lambda = (float)a.lambda;
            const bool restore = a.obj_restore != 0;
            int u = 0;
            for (int c = 0; c < nchunks; ++c) {
                const int s = c % TC_NXS;
                const int cnt = min(TC_TS, t_end - (t_begin + c * TC_TS));
                tc::mbar_wait_h(0u, &x_full[s], (uint32_t)((c / TC_NXS) & 1), errflag, 40);
                const float* xs = Xs + (size_t)s * TC_TS * TC_M + (size_t)j0 * TC_M + o_loc;
                for (int b = 0; b < nact; ++b, ++u) {
                    const uint32_t col = lane_base + (uint32_t)(u % C::NPQ) * C::PQ + j0;
                    tc::mbar_wait_h(0u, &p_full[u % C::NPQ], (uint32_t)((u / C::NPQ) & 1), errflag, 41);
                    tc::tc_fence_after_sync();
                    uint32_t p[16];
                    tc::tmem_ld16(col, p);
                    tc::tmem_wait_ld();
                    tc::tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(&q_full[u % C::NPQ]);  // P is in registers: the buffer is free
                    float su = 0.f;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float x = xs[j * TC_M];
                        if (restore && x == lambda) x = 0.f;
                        float e = x - __uint_as_float(p[j]);
                        e = (valid && j0 + j < cnt) ? e : 0.f;
                        su = fmaf(e, e, su);
                    }
#pragma unroll
                    for (int bb = 0; bb < RB; ++bb)
                        if (bb == b) sacc[bb] += (double)su;
                }
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&x_empty[s]);
            }
            // fixed-order reduction: lanes (shuffle tree), then the 16 quotient warps in warp order
            double* red = reinterpret_cast<double*>(Xs);  // the X stages are idle now: [RB][QWARPS]
            __syncwarp();
            tc::named_bar_sync(2, TC_QWARPS * 32);  // every quotient warp is past its last X tile
#pragma unroll
            for (int b = 0; b < RB; ++b) {
                double v = sacc[b];
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                if (lane == 0) red[b * TC_QWARPS + (warp - TC_QW0)] = v;
            }
            tc::named_bar_sync(2, TC_QWARPS * 32);
            if (warp == TC_QW0 && lane < nact) {
                double t = 0.0;
                for (int w = 0; w < TC_QWARPS; ++w) t += red[lane * TC_QWARPS + w];
                double* dst = a.obj_partials + ((long long)s_act[lane] * a.nblocks + ob) * 2;
                dst[0] = t * a.obj_weight * a.obj_weight;
                dst[1] = t;
            }
        } else {
        // Two GROUPS of 8 warps (4 lane quarters x 2 column halves of 32) alternate units: group 0 takes the even units
        // (P/Q and numerator buffers 0), group 1 the odd ones (buffers 1).  While one group divides, the other waits for
        // its P tile / loads / stores: the division stage no longer runs in lockstep over the whole CTA.
        const int grp = cs >> 1, hh = cs & 1;
        const int jh = hh * 32;                     // this thread's 32 columns of a unit
        constexpr int NC2 = N2 / 2;                 // numerator columns per thread
        constexpr int SL = (RB + 1) / 2;            // restart slots a group accumulates (slot b -> group b % 2, index b / 2)
        float acc[SL][NC2];
#pragma unroll
        for (int i = 0; i < SL; ++i)
#pragma unroll
            for (int c = 0; c < NC2; ++c) acc[i][c] = 0.f;
        // numerators of a unit -> registers, round-to-nearest adds.  A group drains its previous unit u-2 while it divides
        // unit u (the tensor pipe is quieter then: a tensor-memory load issued while MMAs run was measured ~300 clk
        // slower); the a_full wait that precedes it has normally completed long before.
        // The 16 numerator values of a thread (NST = 2: 8 columns of Qhi*Vhi+Qlo*Vhi and the same 8 of Qhi*Vlo; NST = 1:
        // 16 columns) are fetched in two parts of 8, one per 16-column round of the division, to keep registers down.
        // N2 = 64 (k > 32, one restart slot): 32 numerator values, added before the division in four loads of 8 (DRAIN32) - with
        // 32 accumulators, a prefetch next to the 2 x 16 quotient registers spilled part of them to local memory.
        constexpr bool DRAIN32 = NC2 == 32;
        static_assert(NC2 * C::NST == 16 || (DRAIN32 && SL == 1), "numerator values per quotient thread");
        uint32_t v[8];
        const uint32_t acol = lane_base + C::ABASE + (uint32_t)grp * C::ACOLS + hh * NC2;
        auto drain_load = [&](int part) { tc::tmem_ld8(acol + part * (C::NST == 2 ? N2 : 8), v); };
        auto drain_add = [&](int slot, int part) {
#pragma unroll
            for (int i = 0; i < SL; ++i)
                if (i == slot) {
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        if (C::NST == 2) {
                            acc[i][c] += __uint_as_float(v[c]);
                        } else {
#pragma unroll
                            for (int pp = 0; pp < 2; ++pp)
                                if (pp == part) acc[i][pp * 8 + c] += __uint_as_float(v[c]);
                        }
                    }
                }
        };
        auto drain32 = [&]() {
#pragma unroll
            for (int q = 0; q < NC2 / 8; ++q) {
                tc::tmem_ld8(acol + q * 8, v);
                tc::tmem_wait_ld();
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[0][q * 8 + c] += __uint_as_float(v[c]);
            }
        };
        // One restart per CTA (RB = 1, k > 32): the groups take the even / odd CHUNKS, both accumulate the same restart and
        // their sums are added at the end.
        int prev_slot = -1;  // restart slot index (b / 2) of this group's previous unit, -1: none yet
        int ulast = -1;      // this group's last unit
        for (int c = 0; c < nchunks; ++c) {
            const int s = c % TC_NXS;
            const int cnt = min(TC_TS, t_end - (t_begin + c * TC_TS));
            tc::mbar_wait_h(0u, &x_full[s], (uint32_t)((c / TC_NXS) & 1), errflag, 40);
            const float* xs = Xs + (size_t)s * TC_TS * TC_M + (size_t)jh * TC_M + o_loc;
            for (int b = RB == 1 ? 0 : grp; b < nact; b += 2) {
                const int u = c * nact + b;  // u % 2 == grp when nact is even
                if (RB == 1 && (u & 1) != grp) continue;
                const int pq = u % C::NPQ;
                const uint32_t col = lane_base + (uint32_t)pq * C::PQ + jh;
                if (warp == TC_QW0) TC_STAMP(0, u, 0);
                if (a.qwait_ns > 0)  // a waiting group sleeps between polls: its spinning takes issue slots from the dividing group
                    tc::mbar_wait_relaxed(&p_full[pq], (uint32_t)((u / C::NPQ) & 1), (unsigned)a.qwait_ns, errflag, 41);
                else
                    tc::mbar_wait_h(0u, &p_full[pq], (uint32_t)((u / C::NPQ) & 1), errflag, 41);
                // the numerators of this group's previous unit u-2: wait for the commit behind MMA#2(u-2) (with three P/Q
                // buffers the commit behind p_full(u) only covers MMA#2(u-3)); it has normally completed long ago
                if (prev_slot >= 0) tc::mbar_wait_h(0u, &a_full[grp], (uint32_t)((((u - 2) >> 1)) & 1), errflag, 44);
                tc::tc_fence_after_sync();
                if (warp == TC_QW0) TC_STAMP(0, u, 1);
                if constexpr (DRAIN32)
                    if (prev_slot >= 0) drain32();
#pragma unroll 1
                for (int half = 0; half < 2; ++half) {
                    uint32_t p[16], lo[16];
                    tc::tmem_ld16(col + half * 16, p);
                    tc::tmem_wait_ld();
                    if (!DRAIN32 && prev_slot >= 0) drain_load(half);
                    if (half == 0 && warp == TC_QW0) TC_STAMP(0, u, 2);
                    const float* xh = xs + half * 16 * TC_M;
                    if (cnt == TC_TS) {
                        // (one MUFU.RCP per PAIR of quotients, r = 1/(p0 p1), was measured slower: this loop is bound by
                        // instruction issue, not by the MUFU unit.)  Packed FP32x2 arithmetic of sm_100 (FMUL2 / FADD2) for
                        // the quotient and the low part: 8 instead of 10 issue slots per pair of elements.
#pragma unroll
                        for (int j = 0; j < 16; j += 2) {
                            const float r0 = rcp_fast(__uint_as_float(p[j])), r1 = rcp_fast(__uint_as_float(p[j + 1]));
                            const unsigned long long x2 = pack2(xh[j * TC_M], xh[(j + 1) * TC_M]), r2 = pack2(r0, r1);
                            unsigned long long q2, l2;
                            asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(q2) : "l"(x2), "l"(r2));
                            const unsigned long long h2 = q2 & 0xffffe000ffffe000ull;
                            asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(l2) : "l"(q2), "l"(h2));
                            p[j] = (uint32_t)h2;
                            p[j + 1] = (uint32_t)(h2 >> 32);
                            lo[j] = (uint32_t)l2;
                            lo[j + 1] = (uint32_t)(l2 >> 32);
                        }
                    } else {  // last chunk of the slice: steps past the end contribute nothing
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            float q = xh[j * TC_M] * rcp_fast(__uint_as_float(p[j]));
                            q = (jh + half * 16 + j < cnt) ? q : 0.f;
                            const uint32_t h = __float_as_uint(q) & 0xffffe000u;
                            lo[j] = __float_as_uint(q - __uint_as_float(h));
                            p[j] = h;
                        }
                    }
                    if (!DRAIN32 && prev_slot >= 0) {
                        tc::tmem_wait_ld();
                        drain_add(prev_slot, half);
                    }
                    tc::tmem_st16(col + half * 16, p);
                    tc::tmem_st16(col + TC_TS + half * 16, lo);
                }
                if (warp == TC_QW0) TC_STAMP(0, u, 3);
                tc::tmem_wait_st();
                tc::tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&q_full[pq]);
                if (warp == TC_QW0) TC_STAMP(0, u, 4);
                prev_slot = b >> 1;
                ulast = u;
            }
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&x_empty[s]);
        }
        // tail: this group's last unit waits for the commit behind its own MMA#2
        if (ulast >= 0) {
            tc::mbar_wait_h(0u, &a_full[grp], (uint32_t)((ulast >> 1) & 1), errflag, 43);
            tc::tc_fence_after_sync();
            if constexpr (DRAIN32) {
                drain32();
            } else {
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                    drain_load(part);
                    tc::tmem_wait_ld();
                    drain_add(prev_slot, part);
                }
            }
        }
        if constexpr (RB == 1) {  // group 1's sums -> group 0 through the idle X stages, added in a fixed order
            float* xch = Xs;
            const int slot = (lq * 2 + hh) * 32 + lane;
            __syncwarp();
            tc::named_bar_sync(2, TC_QWARPS * 32);  // every quotient warp is past its last X tile
            if (grp == 1)
#pragma unroll
                for (int c = 0; c < NC2; ++c) xch[c * 256 + slot] = acc[0][c];
            tc::named_bar_sync(2, TC_QWARPS * 32);
            if (grp == 0)
#pragma unroll
                for (int c = 0; c < NC2; ++c) acc[0][c] += xch[c * 256 + slot];
        }
        // numerators -> factor update (or the slice's partial sums): this thread's NC2 columns of this group's restarts
#pragma unroll
        for (int i = 0; i < SL; ++i) {
            const int b = 2 * i + grp;
            if (b < nreal && valid) {
                const int r = s_act[b];
                if (a.partial == nullptr) {
                    float* U = Ug + (long long)r * a.u_rstride;
                    const float* den = static_cast<const float*>(a.den) + (long long)r * kTiledMaxK;
#pragma unroll
                    for (int c = 0; c < NC2; ++c) {
                        const int col = hh * NC2 + c;
                        if (col < k) {
                            const long long idx = (long long)o * a.su_o + (long long)col * a.su_a;
                            U[idx] = (U[idx] * acc[i][c]) / den[col];
                        }
                    }
                } else {
                    float* dst = static_cast<float*>(a.partial) + (((long long)slice * a.R + r) * a.nown + o) * a.ktmpl;
#pragma unroll
                    for (int c = 0; c < NC2; ++c) {
                        const int col = hh * NC2 + c;
                        if (col < a.ktmpl) dst[col] = acc[i][c];
                    }
                }
            }
        }
        }
        __syncwarp();
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<C::TCOLS>(tbase);
}

template <int K8, int N2, bool OBJ>
cudaError_t launch_tc(const TiledPassArgs& a, int* d_errflag, cudaStream_t s) {
    using C = TcCfg<K8, N2>;
    const int ngroups = (a.R + C::RB - 1) / C::RB;
    const long long grid = (long long)a.S * a.nblocks * ngroups;
    if (grid > 2147483647ll) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(tc_pass_kernel<K8, N2, OBJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
    if (e != cudaSuccess) return e;
    tc_pass_kernel<K8, N2, OBJ><<<(unsigned)grid, C::THREADS, C::SMEM, s>>>(a, d_errflag);
    return cudaGetLastError();
}

}  // namespace

int tc_pass_group(int k) {
    if (k <= 8) return TcCfg<8, 16>::RB;
    if (k <= 16) return TcCfg<16, 16>::RB;
    if (k <= 24) return TcCfg<24, 32>::RB;
    if (k <= 32) return TcCfg<32, 32>::RB;
    if (k <= 48) return TcCfg<48, 64>::RB;
    return TcCfg<64, 64>::RB;
}
int tc_pass_ctas_per_sm(int) { return 1; }
int tc_pass_chunk(int) { return 64; }

// bulk copies need 16-byte aligned rows of 128 own indices: nown % 4 == 0
bool tc_pass_supported(const TiledPassArgs& a) {
    return !a.has_nan && a.k >= 1 && a.k <= kTiledMaxK && (a.nown % 4) == 0 && (reinterpret_cast<uintptr_t>(a.D) % 16) == 0;
}

cudaError_t launch_tc_pass(const TiledPassArgs& a, int* d_errflag, cudaStream_t s) {
    if (tc2_pass_enabled(a.k)) return launch_tc2_pass(a, d_errflag, s);
    if (a.k <= 8) return launch_tc<8, 16, false>(a, d_errflag, s);
    if (a.k <= 16) return launch_tc<16, 16, false>(a, d_errflag, s);
    if (a.k <= 24) return launch_tc<24, 32, false>(a, d_errflag, s);
    if (a.k <= 32) return launch_tc<32, 32, false>(a, d_errflag, s);
    if (a.k <= 48) return launch_tc<48, 64, false>(a, d_errflag, s);
    return launch_tc<64, 64, false>(a, d_errflag, s);
}

cudaError_t launch_tc_objective(const TiledPassArgs& a, int* d_errflag, cudaStream_t s) {
    if (a.k <= 8) return launch_tc<8, 16, true>(a, d_errflag, s);
    if (a.k <= 16) return launch_tc<16, 16, true>(a, d_errflag, s);
    if (a.k <= 24) return launch_tc<24, 32, true>(a, d_errflag, s);
    if (a.k <= 32) return launch_tc<32, 32, true>(a, d_errflag, s);
    if (a.k <= 48) return launch_tc<48, 64, true>(a, d_errflag, s);
    return launch_tc<64, 64, true>(a, d_errflag, s);
}

}  // namespace nmfk
