// Second generation of the Float32 tcgen05 half-update (k <= 16: C3).  Same mathematics, same unit decomposition and the
// same 3-term TF32 split as tc_pass_kernel (kl_tiled_tc.cu; NMFkMultiplicative.jl:67,70); what changes is the tensor-memory
// plan, so that the stages of a unit stop waiting for one another:
//
//   * P (the product tile MMA#1 writes) gets its OWN columns (one tile per quotient group) instead of being overwritten by
//     Q in place.  In tc_pass_kernel MMA#1 of unit u+2 could only be issued after MMA#2 of unit u had read Q(u): every
//     quotient group sat idle for the round trip  Q(u) stored -> MMA#2(u) -> MMA#1(u+2) -> P(u+2)  (measured 1400 of the 3300
//     clk a group spends per unit, profiles/r01_tc_trace_v17_c3.txt).  Here MMA#1(u+2) is issued as soon as the group has
//     pulled P(u) into registers (p_empty), a whole division earlier; the only other thing a group waits for is the
//     completion of MMA#2(u-2) before its FIRST store of Q(u), half a division after it started on u;
//   * the 128 columns for the P tiles come from the own factor: only U hi stays in tensor memory, U lo (needed by one of the
//     three MMA#1 terms) is an image in shared memory.  (All of U in shared memory was tried first: MMA#1 as an smem x smem
//     instruction reads 6 KB per instruction and ran at half speed.  A single P tile shared by both groups was tried second:
//     the pulls of P and MMA#1 then alternate strictly and the issuer thread becomes the critical path.)
//   * TWO threads issue the MMAs (warp 0: MMA#1, warp 1: MMA#2): one thread issuing both spends ~740 clk per unit issuing
//     (the commit behind the 16 small MMAs of MMA#2 alone costs 75 clk) plus ~450 clk in barrier waits and fences, and was
//     the critical path of every single-issuer variant;
//   * a THIRD thread (warp 18) does all the loading, so the MMA#2 thread only waits for Q: with the X and V loads and
//     their barrier waits on it as well, it reached each unit ~1300 clk after Q was stored, and the quotient groups waited
//     for its a_full (profiles/r05_tc2_trace_c3_main.txt);
//   * X tiles arrive by tensor-map TMA loads from the STEP-contiguous copy of the data, two boxes of 128 own indices x 32
//     steps per chunk, swizzled (SWIZZLE_128B): a quotient thread reads 4 consecutive steps of its own row with one 16-byte
//     shared load (8 per unit instead of 32 scalar ones), and the 8 threads of a quarter-warp hit 8 different bank groups;
//   * the V operand images of a unit (hi / lo split, the K-major layouts of MMA#1 and MMA#2, zeros past k and past the last
//     step) are built once per launch by tc2_images_kernel for every (restart, chunk) and fetched by ONE 1-D bulk copy per
//     unit; no warp of the pass converts V any more (four stager warps did, and took registers and issue slots from the
//     quotient warps);
//   * the numerators of the previous unit are fetched behind the stores of Q and consumed one half-division later.
// What bounds it now is the quotient stage itself (DESIGN.md 4a).
//
// Tensor-memory map (512 columns): P0 | P1 (64 each), Q0 | Q1 (Qhi 64 + Qlo 64 each), two per-unit numerator buffers of 32, U hi of
// the 4 restarts of the CTA (16 each).  Warps: 0 = MMA#1 issuer, 1 = MMA#2 issuer, 2-17 = two alternating quotient groups,
// 18 = load warp (X tiles and V images; last, because a warp reaches only the tensor-memory lanes of its warp % 4 quarter and
// this one touches none).  The objective sums keep using tc_pass_kernel<.., OBJ = true>.
#include <algorithm>
#include <cstdlib>
#include <mutex>

#include "kl_tiled_args.h"
#include "tc_ptx.cuh"
#include "tc_stage.cuh"
#include "tma.cuh"

namespace nmfk {
namespace {

constexpr int T2_M = 128;

template <int K8>
struct Tc2Cfg {
    static constexpr int N2 = 16;
    static constexpr int TS = 64;
    static constexpr int NXS = 3;                                     // X tile stages
    static constexpr int NVB = 6;                                     // V image buffers: an image lives from MMA#1(u) to MMA#2(u), ~4 units
    static constexpr int QW = TS / 4;
    static constexpr int QW0 = 2;                                     // warps 0, 1: the two MMA issuers
    static constexpr int LW = QW0 + QW;                               // the load warp, after the quotient warps
    static constexpr int THREADS = (LW + 1) * 32;
    static constexpr int TCOLS = 512;
    static constexpr int RB = 4;                                      // restarts per CTA (they share the X tiles)
    static constexpr int ACOLS = 2 * N2;                              // Qhi * [Vhi ; Vlo] stacked along N
    static constexpr int PBASE = 0, QBASE = 2 * TS, ABASE = QBASE + 2 * 2 * TS, UBASE = ABASE + 2 * ACOLS;
    static constexpr int PERB = K8;                                   // U hi per restart (U lo lives in shared memory)
    static_assert(UBASE + RB * PERB <= TCOLS, "tensor memory");
    static constexpr uint32_t U1_BYTES = T2_M * K8 * 4;               // U lo image of one restart's 128 own rows
    static constexpr uint32_t SBO1 = (K8 / 4) * 128;                  // K extent K8: the V image of MMA#1 and the U images
    static constexpr uint32_t SBO2 = (TS / 4) * 128;
    static constexpr uint32_t B1_BYTES = TS * K8 * 4;
    static constexpr uint32_t B2_BYTES = N2 * TS * 4;
    static constexpr uint32_t V_BYTES = 2 * B1_BYTES + 2 * B2_BYTES;  // one unit's images: B1 hi, B1 lo, B2 hi, B2 lo
    static constexpr uint32_t X_BYTES = TS * T2_M * 4;                // two swizzled boxes of [128 own][32 steps]
    static constexpr int XBOX = 32;                                   // steps per box: 128 bytes, the swizzle span
    static constexpr size_t SMEM = (size_t)NXS * X_BYTES + (size_t)NVB * V_BYTES + (size_t)RB * U1_BYTES + 32 * 8 + 64;
    static_assert(SMEM <= 232448, "shared memory budget of one CTA");
};

__device__ __forceinline__ unsigned long long pack2f(float lo, float hi) {
    unsigned long long v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(lo), "f"(hi));
    return v;
}
__device__ __forceinline__ float rcp_approx(float p) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p));
    return r;
}

// V operand images of every running restart r and chunk c of the reduction range (block (c, r)), at
// vimg + (r * chunks + c) * V_BYTES: B1 = [steps][K8 columns] (MMA#1, K = columns), B2 = [N2 columns][steps] (MMA#2, K = steps),
// each as hi = the TF32 part and lo = the rest, in the canonical un-swizzled K-major layout.  Item it = 16 bytes = 4 values at
// byte it * 16 of its image (8 rows x 16 bytes per core matrix, core matrices along K first), so a warp writes 512 contiguous bytes.
template <int K8>
__global__ void __launch_bounds__(256) tc2_images_kernel(const TiledPassArgs a, int chunks) {
    using C = Tc2Cfg<K8>;
    const int c = blockIdx.x, r = blockIdx.y;
    if (a.st[r].stop != 0) return;  // frozen: the pass does not read it
    const float* V = static_cast<const float*>(a.V) + (long long)r * a.v_rstride;
    float4* img = reinterpret_cast<float4*>(static_cast<unsigned char*>(a.vimg) + ((size_t)r * chunks + c) * C::V_BYTES);
    const int t0 = c * C::TS;
    auto val = [&](int t, int col) {
        return (t0 + t < a.nred && col < a.k) ? V[(long long)(t0 + t) * a.sv_t + (long long)col * a.sv_a] : 0.f;
    };
    constexpr int NAB = K8 / 4, NTB = C::TS / 4;
    constexpr int NA = C::TS * NAB, NB = C::N2 * NTB;
    for (int it = threadIdx.x; it < NA + NB; it += blockDim.x) {
        float v[4];
        int hi, lo;
        if (it < NA) {  // B1: row = step t, 4 columns 4 ab ..
            const int t = (it & 7) + 8 * (it / (8 * NAB)), ab = (it >> 3) % NAB;
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = val(t, ab * 4 + j);
            hi = it;
            lo = it + C::B1_BYTES / 16;
        } else {  // B2: row = column, 4 steps 4 tb ..
            const int ib = it - NA;
            const int col = (ib & 7) + 8 * (ib / (8 * NTB)), tb = (ib >> 3) % NTB;
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = val(tb * 4 + i, col);
            hi = 2 * C::B1_BYTES / 16 + ib;
            lo = hi + C::B2_BYTES / 16;
        }
        float h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            h[j] = __uint_as_float(__float_as_uint(v[j]) & 0xffffe000u);
            l[j] = v[j] - h[j];
        }
        img[hi] = make_float4(h[0], h[1], h[2], h[3]);
        img[lo] = make_float4(l[0], l[1], l[2], l[3]);
    }
}

template <int K8>
__global__ void __launch_bounds__((Tc2Cfg<K8>::THREADS), 1) tc2_pass_kernel(const TiledPassArgs a, const __grid_constant__ CUtensorMap mX,
                                                                            int* errflag) {
    using C = Tc2Cfg<K8>;
    constexpr int NXS = C::NXS, NVB = C::NVB, TS = C::TS, QWARPS = C::QW, QW0 = C::QW0;
    constexpr int RB = C::RB, N2 = C::N2;
    extern __shared__ __align__(1024) unsigned char smem[];
    float* Xs = reinterpret_cast<float*>(smem);                                   // [NXS][2][M][XBOX] (swizzled)
    unsigned char* Vs = smem + (size_t)NXS * C::X_BYTES;                           // [NVB][V_BYTES]
    unsigned char* Us = Vs + (size_t)NVB * C::V_BYTES;                             // [RB] U lo images
    uint64_t* bars = reinterpret_cast<uint64_t*>(Us + (size_t)RB * C::U1_BYTES);
    uint64_t* x_full = bars;             // [NXS]
    uint64_t* x_empty = x_full + NXS;    // [NXS]
    uint64_t* v_full = x_empty + NXS;    // [NVB]
    uint64_t* v_empty = v_full + NVB;    // [NVB]  MMA#2 of the unit is done with the images
    uint64_t* p_full = v_empty + NVB;    // [2]    MMA#1 done: P readable
    uint64_t* p_empty = p_full + 2;      // [2]    the group has P in registers: MMA#1 of unit u+2 may overwrite the tile
    uint64_t* q_full = p_empty + 2;      // [2]    Q stored
    uint64_t* a_full = q_full + 2;       // [2]    MMA#2 done: numerators readable, Q buffer free
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 32);
    int* s_act = reinterpret_cast<int*>(tmem_slot + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    long long* const trc = (a.trace != nullptr && blockIdx.x == 0) ? a.trace : nullptr;
    const int ngroups = (a.R + RB - 1) / RB;
    const int g = blockIdx.x % ngroups;
    const int rest = blockIdx.x / ngroups;
    const int ob = rest % a.nblocks;
    const int slice = rest / a.nblocks;
    const int o0 = ob * T2_M;
    const int k = a.k;
    const int chunks_all = (a.nred + TS - 1) / TS;  // chunks of the whole reduction range (the image scratch is indexed by them)
    const int t_begin = (int)(((long long)chunks_all * slice) / a.S) * TS;
    const int t_end = min(a.nred, (int)(((long long)chunks_all * (slice + 1)) / a.S) * TS);
    const int nchunks = (t_end - t_begin + TS - 1) / TS;

    if (tid == 0) {
        int nact = 0;
        for (int b = 0; b < RB; ++b) {
            const int r = g * RB + b;
            if (r >= a.R) continue;
            if (a.st[r].stop == 0) s_act[nact++] = r;  // finished restarts are frozen
        }
        s_act[RB] = nact;
        if (nact & 1) s_act[nact] = s_act[0];  // shadow unit: the two groups alternate, a chunk holds an even number of units
    }
    __syncthreads();
    const int nreal = s_act[RB];
    const int nact = nreal + (nreal & 1);
    if (nreal == 0 || nchunks <= 0) return;
    const int total = nchunks * nact;

    if (warp == 0) tc::tmem_alloc<C::TCOLS>(tmem_slot);
    if (tid == 32) {
        for (int i = 0; i < NXS; ++i) {
            tc::mbar_init(&x_full[i], 1);
            tc::mbar_init(&x_empty[i], QWARPS);
        }
        for (int i = 0; i < NVB; ++i) {
            tc::mbar_init(&v_full[i], 1);
            tc::mbar_init(&v_empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            tc::mbar_init(&p_full[i], 1);
            tc::mbar_init(&p_empty[i], QWARPS / 2);
            tc::mbar_init(&q_full[i], QWARPS / 2);
            tc::mbar_init(&a_full[i], 1);
        }
        tc::mbar_fence_init();
    }
    if (tid == 0) tma_prefetch_map(&mX);

    float* Ug = static_cast<float*>(a.U);

    tc::fence_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tbase = *tmem_slot;

    // own factor rows, split hi / lo: hi -> tensor memory, lo -> the canonical K-major image in shared memory (the A operands
    // of MMA#1); quotient warp column group cs loads restart slot cs.  Own indices past the edge get U = 1 (finite P; their X
    // is 0 and their rows are never stored).
    if (warp >= QW0 && warp < C::LW) {
        const int lq = warp & 3, cs = (warp - QW0) >> 2;
        const int ol = lq * 32 + lane;
        const int o = o0 + ol;
        const bool valid = o < a.nown;
        const uint32_t lane_base = tbase + ((uint32_t)(lq * 32) << 16);
        if (cs < nact) {
            const float* U = Ug + (long long)s_act[cs] * a.u_rstride;
            const uint32_t col = C::UBASE + cs * C::PERB;
            unsigned char* img = Us + (size_t)cs * C::U1_BYTES + (ol & 7) * 16 + (ol >> 3) * C::SBO1;
#pragma unroll
            for (int c0 = 0; c0 < K8; c0 += 8) {
                uint32_t hi[8];
                float lo[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float u = !valid ? 1.f : (c0 + c < k ? U[(long long)o * a.su_o + (long long)(c0 + c) * a.su_a] : 0.f);
                    hi[c] = __float_as_uint(u) & 0xffffe000u;
                    lo[c] = u - __uint_as_float(hi[c]);
                }
                tc::tmem_st8(lane_base + col + c0, hi);
                *reinterpret_cast<float4*>(img + (c0 / 4) * TC_LBO) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                *reinterpret_cast<float4*>(img + (c0 / 4 + 1) * TC_LBO) = make_float4(lo[4], lo[5], lo[6], lo[7]);
            }
        }
        tc::tmem_wait_st();
    }
    tc::fence_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();

    if (warp == 0) {
        // ===== MMA#1 issuer: P(u) = U V^T as soon as the group two units back has pulled its P tile and the V images of u are
        // staged.  (One thread issuing both MMA#1 and MMA#2 is the bottleneck of tc_pass_kernel: ~740 clk of issue + ~450 clk of
        // barrier / fence overhead per unit with the tensor pipe 21 % busy; two issuing threads halve that.) =====
        constexpr uint32_t idP = tc::idesc_tf32(T2_M, TS, 0);
        const uint64_t d1 = tc::smem_desc(tc::smem_u32(Vs), TC_LBO, C::SBO1);
        const uint64_t du = tc::smem_desc(tc::smem_u32(Us), TC_LBO, C::SBO1);
        constexpr uint64_t KSTEP = (2 * TC_LBO) >> 4;
        int b = 0;
        for (int u = 0; u < total; ++u) {
            const int vb = u % NVB;
            TC_STAMP(1, u, 3);
            if (u >= 2) tc::mbar_wait_h(0u, &p_empty[u & 1], (uint32_t)(((u - 2) >> 1) & 1), errflag, 23);
            tc::mbar_wait_h(0u, &v_full[vb], (uint32_t)((u / NVB) & 1), errflag, 20);
            tc::tc_fence_after_sync();
            TC_STAMP(1, u, 4);
            const uint32_t d = tbase + C::PBASE + (uint32_t)(u & 1) * TS;
            const uint32_t uh = tbase + C::UBASE + b * C::PERB;
            const uint64_t al = du + (uint64_t)((b * C::U1_BYTES) >> 4);
            const uint64_t bh = d1 + (uint64_t)((vb * C::V_BYTES) >> 4), bl = bh + (C::B1_BYTES >> 4);
            if (tc::elect_one()) {
#pragma unroll
                for (int ks = 0; ks < K8 / 8; ++ks) {
                    tc::mma_tf32_ss(d, al + ks * KSTEP, bh + ks * KSTEP, idP, ks > 0);
                    tc::mma_tf32_ts(d, uh + ks * 8, bl + ks * KSTEP, idP, 1);
                    tc::mma_tf32_ts(d, uh + ks * 8, bh + ks * KSTEP, idP, 1);
                }
                tc::mma_commit(&p_full[u & 1]);
            }
            __syncwarp();
            TC_STAMP(1, u, 5);
            b = b + 1 == nact ? 0 : b + 1;
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===== MMA#2 issuer: ACC(u) = Q(u) V as soon as Q(u) is stored.  Nothing else: every clk this thread spends elsewhere
        // delays a_full(u), and with it the quotient group's first store of Q(u+2) =====
        constexpr uint32_t idA1 = tc::idesc_tf32(T2_M, C::ACOLS, 0);
        constexpr uint32_t idA2 = tc::idesc_tf32(T2_M, N2, 0);
        const uint64_t d2 = tc::smem_desc(tc::smem_u32(Vs) + 2 * C::B1_BYTES, TC_LBO, C::SBO2);
        constexpr uint64_t KSTEP = (2 * TC_LBO) >> 4;
        int vb = 0;  // u % NVB
        for (int u = 0; u < total; ++u) {
            const uint32_t h = (uint32_t)(u & 1);
            TC_STAMP(1, u, 0);
            tc::mbar_wait_h(0u, &q_full[h], (uint32_t)((u >> 1) & 1), errflag, 21);
            tc::tc_fence_after_sync();
            TC_STAMP(1, u, 1);
            const uint32_t d = tbase + C::ABASE + h * C::ACOLS;
            const uint32_t qh = tbase + C::QBASE + h * 2 * TS, ql = qh + TS;
            const uint64_t bh = d2 + (uint64_t)((vb * C::V_BYTES) >> 4);
            if (tc::elect_one()) {
#pragma unroll
                for (int ks = 0; ks < TS / 8; ++ks) tc::mma_tf32_ts(d, qh + ks * 8, bh + ks * KSTEP, idA1, ks > 0);
#pragma unroll
                for (int ks = 0; ks < TS / 8; ++ks) tc::mma_tf32_ts(d, ql + ks * 8, bh + ks * KSTEP, idA2, 1);
                tc::mma_commit(&v_empty[vb]);
                tc::mma_commit(&a_full[h]);
            }
            __syncwarp();
            TC_STAMP(1, u, 2);
            vb = vb + 1 == NVB ? 0 : vb + 1;
        }
        __syncwarp();
    } else if (warp == C::LW) {
        // ===== load warp, in unit order: before the first unit of chunk c its X tile (two tensor-map TMA loads, boxes of 32
        // steps x 128 own indices, zero fill past the edges of X) once both groups are through chunk c-NXS, the previous user
        // of the stage; then the V images of each unit w (one bulk copy into the ring) once MMA#2(w-NVB) is done with the
        // buffer.
        // Deadlock-freedom: every role handles its units in increasing order, and every wait is for a stage of an earlier
        // unit or of an earlier step of the same unit, so the lowest unfinished unit can always progress.  The waits:
        //   load warp  V(w): v_empty = MMA#2(w-NVB) done.  X(c): x_empty = both groups through the units of chunk c-NXS, all
        //              below c*nact, the unit it loads next (X(c) goes out before V(c*nact), so a group never waits for an X
        //              tile behind a V wait of a later unit);
        //   MMA#1(u)   p_empty = the group has P(u-2) in registers; v_full = V(u) loaded;
        //   MMA#2(u)   q_full = Q(u) stored;
        //   group, u   x_full of its chunk, p_full = MMA#1(u) done, a_full = MMA#2(u-2) done.
        // The edge cases keep this order:
        //   * nact = 2 with the shadow unit: nact counts it, so all roles see the same total = nchunks * nact units and the same
        //     chunk boundaries; the shadow unit loads the images of slot 0 again, and its numerators are never stored;
        //   * nchunks < NXS: only nchunks tiles are loaded and no x_empty is waited for; the arrivals on them are never awaited;
        //   * slices (S > 1): every role counts its chunks from the same [t_begin, t_end), the images from chunk t_begin / TS;
        //   * restarts frozen by stop are left out of s_act before any role starts, and a CTA with none running returns before
        //     the barriers are initialised. =====
        auto load_x = [&](int c, int s) {
            if (tc::elect_one()) {
                tc::mbar_arrive_expect_tx(&x_full[s], C::X_BYTES);
                tma_load_2d(Xs + (size_t)s * TS * T2_M, &mX, t_begin + c * TS, o0, &x_full[s]);
                tma_load_2d(Xs + (size_t)s * TS * T2_M + C::XBOX * T2_M, &mX, t_begin + c * TS + C::XBOX, o0, &x_full[s]);
            }
            __syncwarp();
        };
        for (int c = 0; c < NXS && c < nchunks; ++c) load_x(c, c);
        const unsigned char* vimg = static_cast<const unsigned char*>(a.vimg) + (size_t)(t_begin / TS) * C::V_BYTES;
        int c = 0, b = 0, s = 0;  // chunk of unit w, w % nact, c % NXS
        int vb = 0, vround = 0;   // w % NVB, w / NVB
        for (int w = 0; w < total; ++w) {
            if (b == 0 && c >= NXS) {
                TC_STAMP(2, w, 4);
                tc::mbar_wait_h(0u, &x_empty[s], (uint32_t)((c / NXS - 1) & 1), errflag, 10);
                TC_STAMP(2, w, 5);
                load_x(c, s);
                TC_STAMP(2, w, 6);
            }
            TC_STAMP(2, w, 0);
            if (vround > 0) tc::mbar_wait_h(0u, &v_empty[vb], (uint32_t)((vround - 1) & 1), errflag, 22);
            TC_STAMP(2, w, 1);
            if (tc::elect_one()) {
                tc::mbar_arrive_expect_tx(&v_full[vb], C::V_BYTES);
                tc::bulk_g2s(Vs + (size_t)vb * C::V_BYTES, vimg + ((size_t)s_act[b] * chunks_all + c) * C::V_BYTES, C::V_BYTES,
                             &v_full[vb]);
            }
            __syncwarp();
            TC_STAMP(2, w, 2);
            if (++vb == NVB) vb = 0, ++vround;
            if (++b == nact) {
                b = 0;
                ++c;
                s = s + 1 == NXS ? 0 : s + 1;
            }
        }
        __syncwarp();
    } else {
        // ===== quotient warps: two GROUPS of 8 warps (4 lane quarters x 2 column halves of 32) alternate units =====
        const int lq = warp & 3, cs = (warp - QW0) >> 2;
        const int o_loc = lq * 32 + lane;
        const int o = o0 + o_loc;
        const bool valid = o < a.nown;
        const uint32_t lane_base = tbase + ((uint32_t)(lq * 32) << 16);
        const int grp = cs >> 1, hh = cs & 1;
        const int jh = hh * 32;
        constexpr int NC2 = N2 / 2;       // numerator columns per thread
        constexpr int SL = (RB + 1) / 2;  // restart slots a group accumulates
        float acc[SL][NC2];
#pragma unroll
        for (int i = 0; i < SL; ++i)
#pragma unroll
            for (int c = 0; c < NC2; ++c) acc[i][c] = 0.f;
        // numerators of the group's previous unit: 8 columns of Qhi*Vhi + Qlo*Vhi (part 0) and the same 8 of Qhi*Vlo (part 1)
        uint32_t v[8];
        const uint32_t acol = lane_base + C::ABASE + (uint32_t)grp * C::ACOLS + hh * NC2;
        auto drain_load = [&](int part) { tc::tmem_ld8(acol + part * N2, v); };
        auto drain_add = [&](int slot) {
#pragma unroll
            for (int i = 0; i < SL; ++i)
                if (i == slot) {
#pragma unroll
                    for (int c = 0; c < 8; ++c) acc[i][c] += __uint_as_float(v[c]);
                }
        };
        const uint32_t pcol = lane_base + C::PBASE + (uint32_t)grp * TS + jh;
        const uint32_t qcol = lane_base + C::QBASE + (uint32_t)grp * 2 * TS + jh;
        // X row of this thread in each stage: box hh (steps jh .. jh+31), 128 bytes at o_loc; 16-byte piece i of the row (steps
        // jh+4i .. jh+4i+3) sits at piece i ^ (address bits 7-9), the SWIZZLE_128B pattern of the TMA load
        const uint32_t xrow = (uint32_t)(hh * C::XBOX * T2_M + o_loc * C::XBOX) * 4;
        const uint32_t xsw = ((tc::smem_u32(Xs) + xrow) >> 7) & 7;
        int prev_slot = -1;
        for (int c = 0; c < nchunks; ++c) {
            const int s = c % NXS;
            const int cnt = min(TS, t_end - (t_begin + c * TS));
            tc::mbar_wait_h(0u, &x_full[s], (uint32_t)((c / NXS) & 1), errflag, 40);
            const unsigned char* xs = reinterpret_cast<const unsigned char*>(Xs + (size_t)s * TS * T2_M) + xrow;
            for (int b = grp; b < nact; b += 2) {
                const int u = c * nact + b;  // u % 2 == grp (nact is even)
                if (warp == QW0) TC_STAMP(0, u, 0);
                tc::mbar_wait_h(0u, &p_full[grp], (uint32_t)((u >> 1) & 1), errflag, 41);
                tc::tc_fence_after_sync();
                if (warp == QW0) TC_STAMP(0, u, 1);
#pragma unroll 1
                for (int half = 0; half < 2; ++half) {
                    uint32_t p[16];
                    tc::tmem_ld16(pcol + half * 16, p);
                    tc::tmem_wait_ld();
                    if (half == 1) {  // P(u) is in registers: MMA#1 of unit u+2 may overwrite the tile (the MMA#1 issuer has slack)
                        tc::tc_fence_before_sync();
                        __syncwarp();
                        if (lane == 0) tc::mbar_arrive(&p_empty[grp]);
                    }
                    if (half == 0 && warp == QW0) TC_STAMP(0, u, 2);
                    uint32_t lo[16];
                    float xv[16];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float4 x4 = *reinterpret_cast<const float4*>(xs + (((uint32_t)(half * 4 + i) ^ xsw) << 4));
                        xv[4 * i] = x4.x, xv[4 * i + 1] = x4.y, xv[4 * i + 2] = x4.z, xv[4 * i + 3] = x4.w;
                    }
                    if (cnt == TS) {
#pragma unroll
                        for (int j = 0; j < 16; j += 2) {
                            // packed FP32x2 arithmetic of sm_100 (FMUL2 / FADD2) for the quotient and its low part.  (One MUFU.RCP
                            // per PAIR of quotients, r = 1 / (p0 p1), was measured: no gain - the MUFU pipe is not what bounds this
                            // stage - and p0 p1 underflows for the tiny products of all-zero rows.)
                            const int jj = j;
                            const float r0 = rcp_approx(__uint_as_float(p[jj])), r1 = rcp_approx(__uint_as_float(p[jj + 1]));
                            const unsigned long long x2 = pack2f(xv[j], xv[j + 1]), r2 = pack2f(r0, r1);
                            unsigned long long q2, l2;
                            asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(q2) : "l"(x2), "l"(r2));
                            const unsigned long long h2 = q2 & 0xffffe000ffffe000ull;
                            asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(l2) : "l"(q2), "l"(h2));
                            p[jj] = (uint32_t)h2;
                            p[jj + 1] = (uint32_t)(h2 >> 32);
                            lo[j] = (uint32_t)l2;
                            lo[j + 1] = (uint32_t)(l2 >> 32);
                        }
                    } else {  // last chunk of the slice: steps past the end contribute nothing
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int jj = j;
                            float q = xv[j] * rcp_approx(__uint_as_float(p[jj]));
                            q = (jh + half * 16 + jj < cnt) ? q : 0.f;
                            const uint32_t h = __float_as_uint(q) & 0xffffe000u;
                            lo[j] = __float_as_uint(q - __uint_as_float(h));
                            p[jj] = h;
                        }
                    }
                    if (prev_slot >= 0) {
                        if (half == 0) {
                            // MMA#2 of this group's previous unit u-2 has completed: its numerators are readable and it no
                            // longer reads the Q buffer that the stores below overwrite
                            if (warp == QW0) TC_STAMP(0, u, 5);
                            tc::mbar_wait_h(0u, &a_full[grp], (uint32_t)(((u - 2) >> 1) & 1), errflag, 44);
                            tc::tc_fence_after_sync();
                            if (warp == QW0) TC_STAMP(0, u, 6);
                        } else {  // the numerators fetched behind the stores of the first half have had a half-division to arrive
                            tc::tmem_wait_ld();
                            drain_add(prev_slot);
                        }
                        drain_load(half);
                    }
                    tc::tmem_st16(qcol + half * 16, p);
                    tc::tmem_st16(qcol + TS + half * 16, lo);
                    if (half == 0 && warp == QW0) TC_STAMP(0, u, 7);
                }
                if (prev_slot >= 0) {
                    tc::tmem_wait_ld();
                    drain_add(prev_slot);
                }
                if (warp == QW0) TC_STAMP(0, u, 3);
                tc::tmem_wait_st();
                tc::tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&q_full[grp]);
                if (warp == QW0) TC_STAMP(0, u, 4);
                prev_slot = b >> 1;
            }
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&x_empty[s]);
        }
        {  // tail: the group's last unit
            const int ulast = (nchunks - 1) * nact + (nact - 2 + grp);
            tc::mbar_wait_h(0u, &a_full[grp], (uint32_t)((ulast >> 1) & 1), errflag, 43);
            tc::tc_fence_after_sync();
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                drain_load(part);
                tc::tmem_wait_ld();
                drain_add(prev_slot);
            }
        }
        // numerators -> factor update (or the slice's partial sums)
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
        __syncwarp();
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<C::TCOLS>(tbase);
}

template <int K8>
cudaError_t launch2(const TiledPassArgs& a, int* d_errflag, cudaStream_t s) {
    using C = Tc2Cfg<K8>;
    const int ngroups = (a.R + C::RB - 1) / C::RB;
    const long long grid = (long long)a.S * a.nblocks * ngroups;
    const int chunks = (a.nred + C::TS - 1) / C::TS;
    if (grid > 2147483647ll || a.vimg == nullptr || a.R > 65535) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(tc2_pass_kernel<K8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
    if (e != cudaSuccess) return e;
    // Dstep: element (own o, step t) at Dstep[t + o * nred].  The map is a pure function of (Dstep, nown, nred): the two maps of
    // a solve (X and its transpose) are encoded once and reused by every launch.
    struct Cached {
        const void* base;
        int nown, nred;
        CUtensorMap map;
    };
    static std::mutex mu;
    static Cached cache[4];
    static int next = 0;
    CUtensorMap mX;
    {
        std::lock_guard<std::mutex> lock(mu);
        int hit = -1;
        for (int i = 0; i < 4; ++i)
            if (cache[i].base == a.Dstep && cache[i].nown == a.nown && cache[i].nred == a.nred) hit = i;
        if (hit < 0) {
            hit = next;
            next = (next + 1) % 4;
            cache[hit].base = nullptr;
            if (!tma_make_map_f32(&cache[hit].map, a.Dstep, a.nred, a.nown, a.nred, C::XBOX, T2_M, CU_TENSOR_MAP_SWIZZLE_128B))
                return cudaErrorNotSupported;
            cache[hit].base = a.Dstep;
            cache[hit].nown = a.nown;
            cache[hit].nred = a.nred;
        }
        mX = cache[hit].map;
    }
    tc2_images_kernel<K8><<<dim3((unsigned)chunks, (unsigned)a.R), 256, 0, s>>>(a, chunks);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    tc2_pass_kernel<K8><<<(unsigned)grid, C::THREADS, C::SMEM, s>>>(a, mX, d_errflag);
    return cudaGetLastError();
}

}  // namespace

// NMFK_TC_GEN=1 selects the first-generation kernel (tc_pass_kernel) for k <= 16 as well
bool tc2_pass_enabled(int k) {
    static const int gen = [] {
        const char* e = std::getenv("NMFK_TC_GEN");
        return e ? std::atoi(e) : 2;
    }();
    return gen >= 2 && k <= 16 && tma_encode_fn() != nullptr;
}

size_t tc2_image_bytes(int k, int R, int nred) {
    const size_t per = k <= 8 ? Tc2Cfg<8>::V_BYTES : Tc2Cfg<16>::V_BYTES;
    constexpr int TS = Tc2Cfg<16>::TS;
    return tc2_pass_enabled(k) ? (size_t)R * (size_t)((nred + TS - 1) / TS) * per : 0;
}

void tc2_pass_prepare() {
    static bool done = false;
    if (done) return;
    done = true;
    CUtensorMap m;  // a first (dummy) encode and the function look-ups: the driver does lazy work on both
    float* dummy = nullptr;
    if (cudaMalloc(&dummy, 1 << 20) == cudaSuccess) {
        (void)tma_make_map_f32(&m, dummy, 512, 512, 512, 32, T2_M, CU_TENSOR_MAP_SWIZZLE_128B);
        cudaFree(dummy);
    }
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, tc2_pass_kernel<8>);
    cudaFuncGetAttributes(&fa, tc2_pass_kernel<16>);
    cudaFuncSetAttribute(tc2_pass_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc2Cfg<8>::SMEM);
    cudaFuncSetAttribute(tc2_pass_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc2Cfg<16>::SMEM);
}

cudaError_t launch_tc2_pass(const TiledPassArgs& a, int* d_errflag, cudaStream_t s) {
    if (a.k <= 8) return launch2<8>(a, d_errflag, s);
    return launch2<16>(a, d_errflag, s);
}

}  // namespace nmfk
