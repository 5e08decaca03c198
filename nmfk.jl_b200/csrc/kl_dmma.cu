// Float64 DMMA/DFMA fragment-layout instantiations of the resident engine + the host heuristic that
// picks the CTA width and the reduction slices per half-update (see kl_dmma.cuh).
#include <cstdio>
#include <cstdlib>

#include "kl_dmma.cuh"

namespace nmfk {

namespace {

constexpr size_t kSmemLimit = 227u * 1024u;

struct DmmaPlan {
    int nthreads, SH, SW;
    size_t smem;
    bool ok;
};

// template K instantiated for a requested k: exact up to 12, then multiples of 4
int dmma_template_k(int k) {
    if (k < 1 || k > kResidentMaxK) return -1;
    if (k <= 12) return k;
    return (k + 3) / 4 * 4;
}

// Makespan (in 8-step tiles) of one half-update: G = ceil(own/8) row groups x S slices work items are
// handed out dynamically to NW warps (list scheduling of equal items), + the per-item epilogue and,
// for S > 1, the ordered combination of the slices.
long long half_cost(int G, int T, int S, int NW) {
    const long long items = (long long)G * S;
    const long long per_item = (T + S - 1) / S + 3;
    long long cost = ((items + NW - 1) / NW) * per_item;
    if (S > 1) cost += ((G + NW - 1) / NW) * (long long)(S + 1);
    return cost;
}

DmmaPlan plan_dmma(int n, int m, int K) {
    const int KC = (K + 3) / 4;
    const int maxthreads = dmma_max_threads(K);
    const int GH = (m + 7) / 8, TH = (n + 7) / 8;  // H-update: own = columns, reduction = rows
    const int GW = (n + 7) / 8, TW = (m + 7) / 8;
    DmmaPlan best{0, 1, 1, 0, false};
    long long bestcost = LLONG_MIN;
    if (const char* ov = std::getenv("NMFK_DMMA_PLAN")) {  // measurement hook: "NW,SH,SW"
        int NW = 0, SH = 1, SW = 1;
        if (std::sscanf(ov, "%d,%d,%d", &NW, &SH, &SW) == 3 && NW >= 1 && NW * 32 <= maxthreads && SH >= 1 && SW >= 1 &&
            SH <= TH && SW <= TW) {
            const size_t smem = DmmaSmem::make(n, m, KC, SH, SW).total;
            if (smem <= kSmemLimit) return DmmaPlan{NW * 32, SH, SW, smem, true};
        }
    }
    for (int NW = 8; NW * 32 <= maxthreads; ++NW) {
        for (int SH = 1; SH <= 8 && SH <= TH; ++SH)
            for (int SW = 1; SW <= 8 && SW <= TW; ++SW) {
                const size_t smem = DmmaSmem::make(n, m, KC, SH, SW).total;
                if (smem > kSmemLimit) continue;
                long long cost = (half_cost(GH, TH, SH, NW) + half_cost(GW, TW, SW, NW)) * 64;
                cost = cost * NW / (NW & ~3);   // the four schedulers get unequal warp counts
                if (NW < 16) cost += cost / 4;  // too few warps to cover the dependent chain of a tile
                cost -= NW;                     // ties -> more warps
                if (bestcost == LLONG_MIN || cost < bestcost) {
                    bestcost = cost;
                    best = DmmaPlan{NW * 32, SH, SW, smem, true};
                }
            }
    }
    return best;
}

template <int K>
cudaError_t launch_dmma_k(SolveArgs a, cudaStream_t s) {
    const DmmaPlan pl = plan_dmma(a.n, a.m, K);
    if (!pl.ok) return cudaErrorInvalidConfiguration;
    a.SH = pl.SH;
    a.SW = pl.SW;
    cudaError_t e;
    if (a.has_nan) {
        e = cudaFuncSetAttribute(kl_resident_dmma_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem);
        if (e != cudaSuccess) return e;
        kl_resident_dmma_kernel<K, true><<<a.R, pl.nthreads, pl.smem, s>>>(a);
    } else {
        e = cudaFuncSetAttribute(kl_resident_dmma_kernel<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem);
        if (e != cudaSuccess) return e;
        kl_resident_dmma_kernel<K, false><<<a.R, pl.nthreads, pl.smem, s>>>(a);
    }
    return cudaGetLastError();
}

}  // namespace

bool resident_dmma_fits(int n, int m, int k) {
    const int K = dmma_template_k(k);
    if (K < 0) return false;
    return plan_dmma(n, m, K).ok;
}

cudaError_t launch_kl_resident_dmma(const SolveArgs& a, cudaStream_t s) {
    switch (dmma_template_k(a.k)) {
        case 1: return launch_dmma_k<1>(a, s);
        case 2: return launch_dmma_k<2>(a, s);
        case 3: return launch_dmma_k<3>(a, s);
        case 4: return launch_dmma_k<4>(a, s);
        case 5: return launch_dmma_k<5>(a, s);
        case 6: return launch_dmma_k<6>(a, s);
        case 7: return launch_dmma_k<7>(a, s);
        case 8: return launch_dmma_k<8>(a, s);
        case 9: return launch_dmma_k<9>(a, s);
        case 10: return launch_dmma_k<10>(a, s);
        case 11: return launch_dmma_k<11>(a, s);
        case 12: return launch_dmma_k<12>(a, s);
        case 16: return launch_dmma_k<16>(a, s);
        case 20: return launch_dmma_k<20>(a, s);
        case 24: return launch_dmma_k<24>(a, s);
        case 28: return launch_dmma_k<28>(a, s);
        case 32: return launch_dmma_k<32>(a, s);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace nmfk
