// Float64 half-update of the tiled KL engine on the FP64 tensor pipe (DMMA m8n8k4), for factors that do not fit
// in shared memory (BASELINE config C4: 100000 x 2000 Float64, k = 2:32, nNMF = 256; the tiled engine takes k up to 64).
//
// Replaces, for Float64 data without NaN, the loop body of NMFk.NMFmultiplicative
// (/root/reference/src/NMFkMultiplicative.jl:67,70) exactly like tiled_pass_kernel (kl_tiled.cuh):
//   ACC[o,a] = sum_t (D[o,t] / (U[o,:] . V[t,:])) V[t,a]      then  U[o,a] <- U[o,a] ACC[o,a] / den[a]
// in the fragment formulation of the resident engine (kl_dmma.cuh): a WARP owns 8 own indices and walks the
// reduction range in tiles of 8 steps, P = U V^T and ACC += Q V are DMMAs (plus DFMA remainder columns), the
// quotient never leaves the lane that computed it.  What changes against the resident kernel:
//   * V (the other factor) is streamed: chunks of 64 steps x k are staged into shared memory in the padded-pitch
//     layout the B-fragment loads want, by a 3-stage cp.async pipeline shared by the 16 warps of the CTA
//     (128 own indices per CTA); rows past the end of the slice are ONES and their X is 0 (quotient 0);
//   * D is the STEP-contiguous copy of the data (H-update: X, W-update: X^T), each lane loads the two X values
//     of its tile column pair with one 16-byte load, 8 tiles in flight across chunk boundaries;
//   * the fast reciprocal is range-checked per tile (warp vote) instead of redoing a poisoned item;
//   * grid = slices x own-blocks x R with the restart index fastest (X tiles shared through L2), partial sums of
//     the slices are combined by tiled_combine_kernel in slice order (deterministic).
#include "kl_dmma.cuh"
#include "kl_tiled_args.h"

namespace nmfk {
namespace {

constexpr int TD_WARPS = 16;           // 8 own indices each
constexpr int TD_THREADS = TD_WARPS * 32;
constexpr int TD_OWN = TD_WARPS * 8;   // own indices per CTA
constexpr int TD_TCH = 64;             // steps per staged chunk (8 tiles)
constexpr int TD_ST = 3;               // cp.async stages

// P = U V^T for one tile (the first product of dmma_tiles): p[e] = value at (own g, step sigma(2q+e))
template <int K>
__device__ __forceinline__ void dmma_p_tile(const DmmaRegs<K>& R, const double* __restrict__ vp1, const double* __restrict__ vp2a,
                                            const double* __restrict__ vp2b, int g, double (&p)[2]) {
    using C = DmmaCfg<K>;
    p[0] = p[1] = 0.0;
    if constexpr (C::NSP > 0) {
        const double* vpsa = vp2a + (C::C0 - g);
        const double* vpsb = vp2b + (C::C0 - g);
#pragma unroll
        for (int i = 0; i < C::NSP; ++i) {
            p[0] = fma(R.us[i], vpsa[C::KD - C::C0 + i], p[0]);
            p[1] = fma(R.us[i], vpsb[C::KD - C::C0 + i], p[1]);
        }
    }
#pragma unroll
    for (int kc = 0; kc < C::KCD; ++kc) dmma884(p, R.ua[kc], vp1[kc * 4]);
}

// OBJ = true: objective mode (NMFkMultiplicative.jl:74,125): only P = U V^T, the lanes accumulate (x - p)^2; nothing is
// written to the factors.  a = the W-update arguments with S = 1; partial sums per block of 128 rows.
// DIV (pass mode only): the quotient of NMF.jl's KL update (Variant KL_DIV), x / (p + delta); a.den already holds the sums + delta
template <int K, bool OBJ, bool DIV = false>
__global__ void __launch_bounds__(TD_THREADS, 1) tiled_dmma_pass_kernel(const TiledPassArgs a) {
    using C = DmmaCfg<K>;
    constexpr int pitch = C::pitch;
    constexpr int NV = C::NV;
    constexpr int PF = 8;
    extern __shared__ __align__(16) unsigned char smem[];
    double* Vs = reinterpret_cast<double*>(smem);  // [ST][TCH][pitch]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int r = blockIdx.x % a.R;
    const int rest = blockIdx.x / a.R;
    const int ob = rest % a.nblocks;
    const int slice = rest / a.nblocks;
    {
        const bool stopped = a.st[r].stop != 0;
        const bool take = (OBJ && a.obj_sel == 1) ? (stopped && a.st[r].done == 0) : !stopped;  // finished restarts are frozen
        if (!take) return;
    }
    const int k = a.k, nown = a.nown, nred = a.nred;
    double ssum = 0.0;
    const double lambda = a.lambda;
    const bool restore = OBJ && a.obj_restore != 0;

    const double* D = static_cast<const double*>(a.D);  // element (o, t) at D[t + o * nred]
    double* U = static_cast<double*>(a.U) + (long long)r * a.u_rstride;
    const double* V = static_cast<const double*>(a.V) + (long long)r * a.v_rstride;

    // slice = whole tiles of 8 steps
    const unsigned tiles_total = (unsigned)(nred + 7) >> 3;
    const int tb = (int)(((unsigned long long)tiles_total * (unsigned)slice) / (unsigned)a.S);
    const int te = (int)(((unsigned long long)tiles_total * (unsigned)(slice + 1)) / (unsigned)a.S);
    const int tiles_full = ((nred & 1) == 0) ? (nred >> 3) : 0;  // tiles a lane can fetch with one 16-byte load
    const int tef = min(te, tiles_full);
    const int nchunks = (te - tb + 7) / 8;

    // padding columns of the staged rows stay zero for the whole kernel
    for (int e = tid; e < TD_ST * TD_TCH * pitch; e += TD_THREADS) Vs[e] = 0.0;
    __syncthreads();

    auto issue = [&](int chunk) {
        double* vs = Vs + (size_t)(chunk % TD_ST) * TD_TCH * pitch;
        const int t0 = (tb + chunk * 8) * 8;
        // coalesced along whichever index is contiguous in global memory
        for (int e = tid; e < TD_TCH * k; e += TD_THREADS) {
            int tl, c;
            if (a.sv_t == 1) {
                tl = e % TD_TCH;
                c = e / TD_TCH;
            } else {
                c = e % k;
                tl = e / k;
            }
            const int t = t0 + tl;
            if (t < nred)
                cp_async_8(vs + tl * pitch + c, V + (long long)t * a.sv_t + (long long)c * a.sv_a);
            else
                vs[tl * pitch + c] = 1.0;  // steps past the end: p > 0, x = 0
        }
    };

    const int row = ob * TD_OWN + warp * 8 + g;
    const bool rvalid = row < nown;
    const int rowc = rvalid ? row : nown - 1;  // invalid rows shadow the last valid one; never stored
    const int sw = q >> 1;
    const int sa = 2 * q + sw, sb = 2 * q + 1 - sw;
    const int off1 = dmma_sigma(g) * pitch + q;
    const int off2a = sa * pitch + g, off2b = sb * pitch + g;
    const bool hi_ok = (C::ND - 8 + g) < pitch;

    DmmaRegs<K> R;
    {
        // this lane's U fragment straight from global memory (column kc*4+q of the DMMA part, the remainder columns)
        const double* up = U + (long long)rowc * a.su_o;
#pragma unroll
        for (int kc = 0; kc < C::KCD; ++kc) R.ua[kc] = (kc * 4 + q < k) ? up[(long long)(kc * 4 + q) * a.su_a] : 0.0;
#pragma unroll
        for (int j = 0; j < C::NSP; ++j) R.us[j] = (C::KD + j < k) ? up[(long long)(C::KD + j) * a.su_a] : 0.0;
    }
    R.zero();

    auto load_tail = [&](const double* ptr, int tile) -> double2 {  // partial / unaligned tile
        const int t = tile * 8 + 2 * q;
        double2 v;
        v.x = (t < nred) ? __ldg(ptr) : 0.0;
        v.y = (t + 1 < nred) ? __ldg(ptr + 1) : 0.0;
        return v;
    };
    const double* xp = D + (long long)rowc * nred + 2 * q + (long long)tb * 8;  // advances with the consumed tile
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

#pragma unroll
    for (int c = 0; c < TD_ST - 1; ++c) {
        if (c < nchunks) issue(c);
        cp_async_commit();
    }
    const bool inall[1][2] = {{true, true}};
    int tile = tb;
    for (int chunk = 0; chunk < nchunks; ++chunk) {
        cp_async_wait<TD_ST - 2>();
        __syncthreads();  // the chunk is visible to all; everyone is done with the stage refilled below
        if (chunk + TD_ST - 1 < nchunks) issue(chunk + TD_ST - 1);
        cp_async_commit();
        const double* vb = Vs + (size_t)(chunk % TD_ST) * TD_TCH * pitch;
#pragma unroll
        for (int u = 0; u < PF; ++u) {  // 8 tiles per chunk == PF: ring slot u <-> tile u of the chunk
            if (tile < te) {            // warp-uniform
                double x[1][2];
                x[0][0] = sw ? xq[u].y : xq[u].x;
                x[0][1] = sw ? xq[u].x : xq[u].y;
                if (tile + PF < tef)
                    xq[u] = __ldg(reinterpret_cast<const double2*>(xp + PF * 8));
                else if (tile + PF < te)
                    xq[u] = load_tail(xp + PF * 8, tile + PF);
                const double* vt = vb + (size_t)u * 8 * pitch;
                if constexpr (OBJ) {
                    double p[2];
                    dmma_p_tile<K>(R, vt + off1, vt + off2a, vt + off2b, g, p);
                    double x0 = x[0][0], x1 = x[0][1];
                    if (restore) {
                        x0 = (x0 == lambda) ? 0.0 : x0;
                        x1 = (x1 == lambda) ? 0.0 : x1;
                    }
                    const double e0 = (rvalid && tile * 8 + sa < nred) ? x0 - p[0] : 0.0;
                    const double e1 = (rvalid && tile * 8 + sb < nred) ? x1 - p[1] : 0.0;
                    ssum = fma(e0, e0, ssum);
                    ssum = fma(e1, e1, ssum);
                } else {
                    dmma_tiles<K, 2, 1, 0, DIV>(R, x, vt + off1, vt + off2a, vt + off2b, g, inall, hi_ok);
                }
                xp += 8;
                ++tile;
            }
        }
    }
    cp_async_wait<0>();
    if constexpr (OBJ) {
        // fixed-order reduction: lanes (shuffle tree), then the 16 warps in warp order
        __shared__ double red[TD_WARPS];
        ssum = warp_sum(ssum);
        if (lane == 0) red[warp] = ssum;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int w = 0; w < TD_WARPS; ++w) t += red[w];
            double* dst = a.obj_partials + ((long long)r * a.nblocks + ob) * 2;
            dst[0] = t * a.obj_weight * a.obj_weight;
            dst[1] = t;
        }
        return;
    }
    R.finish();
    if (!rvalid) return;
    if (a.partial == nullptr) {
        const double* den = static_cast<const double*>(a.den) + (long long)r * kTiledMaxK;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            const int c = DmmaRegs<K>::column(v, q);
            if (c < k) {
                double* up = U + (long long)row * a.su_o + (long long)c * a.su_a;
                *up = div_cold<double>(*up * R.value(v, q), den[c]);
            }
        }
    } else {
        double* dst = static_cast<double*>(a.partial) + (((long long)slice * a.R + r) * nown + row) * a.ktmpl;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            const int c = DmmaRegs<K>::column(v, q);
            if (c < a.ktmpl) dst[c] = (c < k) ? R.value(v, q) : 0.0;
        }
    }
}

template <int K, bool OBJ, bool DIV>
cudaError_t launch_td(const TiledPassArgs& a, cudaStream_t s) {
    constexpr auto kernel = tiled_dmma_pass_kernel<K, OBJ, DIV>;
    const size_t smem = (size_t)TD_ST * TD_TCH * DmmaCfg<K>::pitch * sizeof(double);
    const long long grid = (long long)a.S * a.nblocks * a.R;
    if (grid > 2147483647ll) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<(unsigned)grid, TD_THREADS, smem, s>>>(a);
    return cudaGetLastError();
}

template <bool OBJ, bool DIV = false>
cudaError_t dispatch_td(const TiledPassArgs& a, cudaStream_t s) {
    switch (a.ktmpl) {
        case 4: return launch_td<4, OBJ, DIV>(a, s);
        case 5: return launch_td<5, OBJ, DIV>(a, s);
        case 6: return launch_td<6, OBJ, DIV>(a, s);
        case 7: return launch_td<7, OBJ, DIV>(a, s);
        case 8: return launch_td<8, OBJ, DIV>(a, s);
        case 9: return launch_td<9, OBJ, DIV>(a, s);
        case 10: return launch_td<10, OBJ, DIV>(a, s);
        case 11: return launch_td<11, OBJ, DIV>(a, s);
        case 12: return launch_td<12, OBJ, DIV>(a, s);
        case 16: return launch_td<16, OBJ, DIV>(a, s);
        case 20: return launch_td<20, OBJ, DIV>(a, s);
        case 24: return launch_td<24, OBJ, DIV>(a, s);
        case 32: return launch_td<32, OBJ, DIV>(a, s);
        case 40: return launch_td<40, OBJ, DIV>(a, s);
        case 48: return launch_td<48, OBJ, DIV>(a, s);
        case 56: return launch_td<56, OBJ, DIV>(a, s);
        case 64: return launch_td<64, OBJ, DIV>(a, s);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace

int tiled_dmma_own() { return TD_OWN; }
int tiled_dmma_chunk() { return TD_TCH; }

// a.k in 4..64 (smaller k are all-DFMA in the resident formulation and stay on the scalar pass); K = the template K of
// the combine kernel (tiled_template_k), a.nblocks = ceil(nown / 128), a.D step-contiguous
cudaError_t launch_tiled_dmma_pass(const TiledPassArgs& a, cudaStream_t s, bool div) {
    return div ? dispatch_td<false, true>(a, s) : dispatch_td<false>(a, s);
}
// objective sums: a = the W-update arguments (D = X^T step-contiguous, U = W, V = H), S = 1
cudaError_t launch_tiled_dmma_objective(const TiledPassArgs& a, cudaStream_t s) { return dispatch_td<true>(a, s); }

}  // namespace nmfk
