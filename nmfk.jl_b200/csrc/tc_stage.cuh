// V stager role of the first-generation tcgen05 tiled pass (kl_tiled_tc.cu): 128 threads cp.async the raw chunk of the
// broadcast factor two units ahead (16 bytes at a time along whichever index is contiguous in global memory), then split it
// hi / lo (TF32 + rest) into the two canonical un-swizzled K-major images that MMA#1 (rows = steps, K = columns) and MMA#2
// (rows = columns, K = steps) read.  Work item = half a 4 x 4 block.
#pragma once
#include "kl_tiled_args.h"
#include "tc_ptx.cuh"

namespace nmfk {

constexpr uint32_t TC_LBO = 128;  // leading-dimension byte offset of the canonical layouts

#define TC_STAMP(role, unit, ev)                                                                    \
    do {                                                                                            \
        if (trc != nullptr && (unit) < 64 && lane == 0) trc[((role) * 64 + (unit)) * 8 + (ev)] = clock64(); \
    } while (0)

// C: configuration (TS, NVB, NRAW, SW, K8, V_BYTES, B1_BYTES, B2_BYTES, SBO1, SBO2, RAW_BYTES, RAWP_T, RAWP_A); first = thread id of the
// first stager thread; unit u = chunk * nact + restart slot.
template <class C, int K8, bool OBJ>
__device__ __forceinline__ void tc_stager_role(const TiledPassArgs& a, unsigned char* Vs, float* Raw, uint64_t* v_full, uint64_t* v_empty,
                                               const int* s_act, int nact, int total, int t_begin, int t_end, int first, uint32_t hint,
                                               int* errflag, long long* trc) {
    constexpr int TC_TS = C::TS, TC_NVB = C::NVB, TC_SWARPS = C::SW;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int k = a.k;
    const float* Vg = static_cast<const float*>(a.V);
    constexpr int NS = TC_SWARPS * 32;
    const int sid = tid - first;
    const bool t_major = a.sv_t == 1;  // raw layout [column][step] (H-update: V = W) instead of [step][column]
    const bool vec16 = t_major ? ((a.sv_a & 3) == 0 && (a.v_rstride & 3) == 0)
                               : (a.sv_a == 1 && (k & 3) == 0 && (a.sv_t & 3) == 0 && (a.v_rstride & 3) == 0);
    constexpr int RAWF = C::RAW_BYTES / 4, PT = C::RAWP_T, PA = C::RAWP_A;
    constexpr int NAB = K8 / 4, NTB = TC_TS / 4;
    constexpr int ITA = TC_TS * NAB / NS, ITB = K8 * NTB / NS;  // items per thread and pass
    static_assert(ITA * NS == TC_TS * NAB && ITB * NS == K8 * NTB && ITA >= 1, "stager work split");
    // per-thread constants of the two conversion passes (the items of a thread never change): raw index of the first
    // of the 4 values, image byte offset
    int rawA[ITA], rawB[ITB > 0 ? ITB : 1];
    uint32_t offA[ITA], offB[ITB > 0 ? ITB : 1];
#pragma unroll
    for (int q = 0; q < ITA; ++q) {
        const int it = sid + q * NS;
        const int t = (it & 7) + 8 * (it / (8 * NAB)), ab = (it >> 3) % NAB;
        rawA[q] = t_major ? (ab * 4) * PT + t : t * PA + ab * 4;
        offA[q] = (t & 7) * 16 + (t >> 3) * C::SBO1 + ab * TC_LBO;
    }
#pragma unroll
    for (int q = 0; q < ITB; ++q) {
        const int it = sid + q * NS;
        const int col = (it & 7) + 8 * (it / (8 * NTB)), tb = (it >> 3) % NTB;
        rawB[q] = t_major ? col * PT + tb * 4 : (tb * 4) * PA + col;
        offB[q] = 2 * C::B1_BYTES + (col & 7) * 16 + (col >> 3) * C::SBO2 + tb * TC_LBO;
    }
    // ... and of the 16-byte copies of the raw chunk: element offset in V relative to the first step of the unit,
    // raw index, step within the unit, column in range.  K8 > 32: recomputed per copy instead (kept in registers, the tables
    // of 8 copies spilled to local memory)
    constexpr int NCP = K8 * (TC_TS / 4) / NS;
    static_assert(NCP * NS == K8 * (TC_TS / 4), "copy split");
    constexpr bool CPTAB = K8 <= 32;
    constexpr int NCPT = CPTAB ? NCP : 1;
    long long cpg[NCPT];
    int cps[NCPT], cpt[NCPT];
    bool cpok[NCPT];
    auto cp_item = [&](int i, long long& g, int& sidx, int& t, bool& ok) {
        const int e = sid + i * NS;
        if (t_major) {
            const int col = e / (TC_TS / 4), t4 = (e % (TC_TS / 4)) * 4;
            g = (long long)t4 + (long long)col * a.sv_a;
            sidx = col * PT + t4;
            t = t4;
            ok = col < k;
        } else {
            const int tl = e / (K8 / 4), a4 = (e % (K8 / 4)) * 4;
            g = (long long)tl * a.sv_t + a4;
            sidx = tl * PA + a4;
            t = tl;
            ok = a4 < k;
        }
    };
    if constexpr (CPTAB) {
#pragma unroll
        for (int i = 0; i < NCP; ++i) cp_item(i, cpg[i], cps[i], cpt[i], cpok[i]);
    }
    auto issue_raw = [&](int c, int b, int stage) {
        const float* V = Vg + (long long)s_act[b] * a.v_rstride;
        const int t0 = t_begin + c * TC_TS;
        float* dst = Raw + (size_t)stage * RAWF;
        if (vec16) {
            const float* Vu = V + (long long)t0 * (t_major ? 1 : a.sv_t);
#pragma unroll
            for (int i = 0; i < NCP; ++i) {
                long long g;
                int sidx, t;
                bool ok;
                if constexpr (CPTAB) {
                    g = cpg[i], sidx = cps[i], t = cpt[i], ok = cpok[i];
                } else {
                    cp_item(i, g, sidx, t, ok);
                }
                const bool live = ok && (t0 + t < t_end);
                tc::cp_async16_zfill(dst + sidx, live ? Vu + g : V, live ? 16u : 0u);
            }
        } else {
            for (int e = sid; e < TC_TS * K8; e += NS) {
                int tl, col;
                if (t_major) {
                    tl = e % TC_TS;
                    col = e / TC_TS;
                } else {
                    col = e % K8;
                    tl = e / K8;
                }
                const bool live = (t0 + tl < t_end) && (col < k);
                tc::cp_async4_zfill(dst + (t_major ? col * PT + tl : tl * PA + col),
                                    live ? V + (long long)(t0 + tl) * a.sv_t + (long long)col * a.sv_a : V, live ? 4u : 0u);
            }
        }
    };
    int ci = 0, bi = 0;  // (chunk, restart slot) of the next unit to issue
    auto advance = [&]() {
        if (++bi == nact) {
            bi = 0;
            ++ci;
        }
    };
    issue_raw(ci, bi, 0);
    advance();
    tc::cp_async_commit();
    if (total > 1) {
        issue_raw(ci, bi, 1);
        advance();
    }
    tc::cp_async_commit();
    for (int u = 0; u < total; ++u) {
        tc::cp_async_wait<1>();           // this thread's copies of unit u have landed (unit u + 1 may be in flight)
        tc::named_bar_sync(1, NS);        // ... and everybody else's
        if (warp == (first >> 5)) TC_STAMP(2, u, 1);
        const int vb = u % TC_NVB;
        if (u >= TC_NVB) tc::mbar_wait_relaxed(&v_empty[vb], (uint32_t)((u / TC_NVB - 1) & 1), hint >> 16, errflag, 30);
        if (warp == (first >> 5)) TC_STAMP(2, u, 2);
        unsigned char* base = Vs + (size_t)vb * C::V_BYTES;
        const float* raw = Raw + (size_t)(u % C::NRAW) * RAWF;
        // Two passes with shared-memory-conflict-free lane mappings (a warp touches 8 consecutive 16-byte rows of
        // 4 different core matrices = 512 contiguous bytes per store); all loads of a pass are issued up front.
        // pass A -> MMA#1 images: item = (step t, 4 columns 4 ab ..): row = step, 16 bytes = 4 columns
        {
            float v[ITA][4];
#pragma unroll
            for (int q = 0; q < ITA; ++q) {
                if (t_major) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[q][j] = raw[rawA[q] + j * PT];
                } else {
                    const float4 w = *reinterpret_cast<const float4*>(raw + rawA[q]);
                    v[q][0] = w.x, v[q][1] = w.y, v[q][2] = w.z, v[q][3] = w.w;
                }
            }
#pragma unroll
            for (int q = 0; q < ITA; ++q) {
                float h[4], l[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    h[j] = __uint_as_float(__float_as_uint(v[q][j]) & 0xffffe000u);
                    l[j] = v[q][j] - h[j];
                }
                const uint32_t off = offA[q];
                *reinterpret_cast<float4*>(base + off) = make_float4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<float4*>(base + C::B1_BYTES + off) = make_float4(l[0], l[1], l[2], l[3]);
            }
        }
        // pass B -> MMA#2 images: item = (column, 4 steps 4 tb ..): row = column, 16 bytes = 4 steps
        if (!OBJ) {
            float v[ITB][4];
#pragma unroll
            for (int q = 0; q < ITB; ++q) {
                if (t_major) {
                    const float4 w = *reinterpret_cast<const float4*>(raw + rawB[q]);
                    v[q][0] = w.x, v[q][1] = w.y, v[q][2] = w.z, v[q][3] = w.w;
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) v[q][i] = raw[rawB[q] + i * PA];
                }
            }
#pragma unroll
            for (int q = 0; q < ITB; ++q) {
                float h[4], l[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    h[i] = __uint_as_float(__float_as_uint(v[q][i]) & 0xffffe000u);
                    l[i] = v[q][i] - h[i];
                }
                const uint32_t off = offB[q];
                *reinterpret_cast<float4*>(base + off) = make_float4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<float4*>(base + C::B2_BYTES + off) = make_float4(l[0], l[1], l[2], l[3]);
            }
        }
        tc::fence_async_smem();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&v_full[vb]);
        if (warp == (first >> 5)) TC_STAMP(2, u, 3);
        if (u + 2 < total) {
            // two raw buffers (k > 32: shared memory budget): the one refilled below is the one every stager just read
            if constexpr (C::NRAW < 3) tc::named_bar_sync(1, NS);
            issue_raw(ci, bi, (u + 2) % C::NRAW);
            advance();
        }
        tc::cp_async_commit();
        if (warp == (first >> 5)) TC_STAMP(2, u, 0);
    }
    tc::cp_async_wait<0>();
    __syncwarp();
}

}  // namespace nmfk
