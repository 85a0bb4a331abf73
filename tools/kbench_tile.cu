// kbench_tile.cu -- developer micro-benchmark: tile_kernel<Op,...> configurations (PPT, THREADS, STAGES, CTAs/SM)
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <vector>

#include "dct_jsd_kernels.cuh"
#include "dct_pixelwise.cuh"

namespace dct {
#define DCT_KBENCH 1
}
// pull in the KL ops (defined in dct_kl.cu) without its extern "C" part clashing: include the TU
#include "dct_kl.cu"
#include "dct_ce.cu"
static bool g_pdl = true;
static int g_pool_div = 0;
static int g_refill = 0;
static bool g_static = false;  // 1: no workspace -> static round-robin tile schedule (and no loss sum)
namespace dct { bool pdl_enabled() { return g_pdl; } unsigned long long* trace_next(int) { return nullptr; } }

using namespace dct;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1); } } while (0)

__global__ void fillf(float* p, size_t n, unsigned seed, float scale) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        unsigned h = (unsigned)i * 2654435761u + seed; h ^= h >> 13; h *= 0x5bd1e995u; h ^= h >> 15;
        p[i] = ((h & 0xffff) / 65535.0f - 0.5f) * scale;
    }
}
__global__ void filll(long long* p, size_t n, int C) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        unsigned h = (unsigned)i * 2654435761u; h ^= h >> 13; h *= 0x5bd1e995u; h ^= h >> 15;
        p[i] = h % C;
    }
}

struct DiceOpB {
    static constexpr int NIN = 1, NOUT = 0, NDICE = 1;
    static constexpr bool HAS_MAP = false, USES_UP = false, CHECKS_SIMPLEX = false, GMAP = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&)[1][CM], int, T, float, bool&) { return vset<T>(0.0f); }
};

// pure copy through the pipeline (NIN*C planes in, same planes out): the skeleton's own ceiling
template <int N>
struct CopyOp {
    static constexpr int NIN = N, NOUT = N, NDICE = 0;
    static constexpr bool HAS_MAP = false, USES_UP = false, CHECKS_SIMPLEX = false, GMAP = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&)[N][CM], int, T, float, bool&) { return vset<T>(0.0f); }
};

template <class Op, int CT, int PPT, int NCW, int STAGES, int MINB, bool TMAP = false>
void run(const char* tag, int64_t B, int64_t HW, int reps, double bytes_per_px, bool labels) {
    constexpr int THREADS = NCW * 32 + 32;
    using Cfg = TileCfg<Op, CT, PPT, NCW * 32, STAGES, float, TMAP>;
    auto kern = tile_kernel<Op, CT, PPT, NCW, STAGES, MINB, float, false, TMAP>;
    if (Cfg::kSmemBytes * MINB > 227 * 1024) { printf("%-14s skip (smem)\n", tag); return; }
    const int R = 4;
    size_t n = (size_t)B * CT * HW;
    std::vector<TileArgs> sets(R);
    std::vector<TileMaps<TMAP>> maps(R);
    Workspace* ws; CK(cudaMalloc(&ws, sizeof(Workspace))); CK(cudaMemset(ws, 0, sizeof(Workspace)));
    double* sum; CK(cudaMalloc(&sum, 8));
    unsigned long long* counts; CK(cudaMalloc(&counts, 8 * 8 * B * CT * 3)); CK(cudaMemset(counts, 0, 8 * 8 * B * CT * 3));
    std::vector<void*> allocs;
    for (int r = 0; r < R; ++r) {
        TileArgs a{};
        for (int k = 0; k < Op::NIN; ++k) {
            float* in; CK(cudaMalloc(&in, n * 4)); allocs.push_back(in);
            fillf<<<1024, 256>>>(in, n, 17u * r + k, 12.0f);
            a.in[k] = in;
        }
        for (int k = 0; k < Op::NOUT; ++k) { float* g; CK(cudaMalloc(&g, n * 4)); allocs.push_back(g); a.out[k] = g; }
        if (labels) { long long* l; CK(cudaMalloc(&l, (size_t)B * HW * 8)); allocs.push_back(l); filll<<<1024, 256>>>(l, (size_t)B * HW, CT); a.labels = (const int64_t*)l; }
        a.counts = counts; a.count_view_stride = B * CT * 3;
        a.HW = HW; a.map = nullptr; a.sum = Op::HAS_MAP ? sum : nullptr; a.up = Upstream{nullptr, nullptr, 1e-6f};
        a.eps = 1e-10f; a.ignore_index = 255; a.class_w = nullptr; a.flags = nullptr; a.ws = ws; a.force_static = g_static ? 1 : 0; a.pool_div = g_pool_div;
        tile_set_geometry(a, B, Cfg::TP); a.refill = g_refill;
        sets[r] = a;
        if constexpr (TMAP) {
            for (int k = 0; k < Op::NIN; ++k) if (!make_tmap_bchw(&maps[r].in[k], a.in[k], 4, HW, CT, B, Cfg::TP)) { printf("tensor map refused\n"); return; }
            for (int k = 0; k < Op::NOUT; ++k) if (!make_tmap_bchw(&maps[r].out[k], a.out[k], 4, HW, CT, B, Cfg::TP)) { printf("tensor map refused\n"); return; }
        }
    }
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes));
    int grid = 148 * MINB; if (grid > sets[0].num_tiles) grid = sets[0].num_tiles;
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    for (int i = 0; i < 5; ++i) launch_pdl(kern, dim3(grid), dim3(THREADS), Cfg::kSmemBytes, (cudaStream_t)0, sets[i % R], maps[i % R]);
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(e0));
    for (int i = 0; i < reps; ++i) launch_pdl(kern, dim3(grid), dim3(THREADS), Cfg::kSmemBytes, (cudaStream_t)0, sets[i % R], maps[i % R]);
    CK(cudaEventRecord(e1));
    CK(cudaDeviceSynchronize());
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
    double us = ms * 1e3 / reps;
    // in-kernel trace of a chain of 8 launches: CTA residency window vs launch-to-launch spacing
    {
        const int NL = 8;
        unsigned long long* tr; CK(cudaMalloc(&tr, (size_t)NL * grid * 8 * kTraceSlots));
        for (int i = 0; i < NL; ++i) { TileArgs t = sets[i % R]; t.trace = tr + (size_t)i * grid * kTraceSlots; launch_pdl(kern, dim3(grid), dim3(THREADS), Cfg::kSmemBytes, (cudaStream_t)0, t, maps[i % R]); }
        CK(cudaDeviceSynchronize());
        std::vector<unsigned long long> h((size_t)NL * grid * kTraceSlots);
        CK(cudaMemcpy(h.data(), tr, h.size() * 8, cudaMemcpyDeviceToHost));
        double win = 0, gap = 0, cta = 0, spread_s = 0, spread_e = 0; unsigned long long prev_end = 0, prev_start = 0; double spacing = 0;
        for (int i = 0; i < NL; ++i) {
            unsigned long long s0 = ~0ull, s1 = 0, e0_ = ~0ull, e1_ = 0; double d = 0;
            for (int c = 0; c < grid; ++c) { auto a0 = h[((size_t)i * grid + c) * kTraceSlots], a1 = h[((size_t)i * grid + c) * kTraceSlots + 3]; s0 = std::min(s0, a0); s1 = std::max(s1, a0); e0_ = std::min(e0_, a1); e1_ = std::max(e1_, a1); d += (double)(a1 - a0); }
            if (i >= 2) { win += (double)(e1_ - s0); gap += (double)(s0 - prev_end); cta += d / grid; spread_s += (double)(s1 - s0); spread_e += (double)(e1_ - e0_); spacing += (double)(s0 - prev_start); }
            prev_end = e1_; prev_start = s0;
        }
        if (getenv("KB_DUMP")) {   // per-CTA detail of the last traced launch: end time after the launch's first start, tiles, pool draws, SM
            int i = NL - 1;
            unsigned long long s0 = ~0ull;
            for (int c = 0; c < grid; ++c) s0 = std::min(s0, h[((size_t)i * grid + c) * kTraceSlots]);
            std::vector<std::pair<double, int>> ends;
            for (int c = 0; c < grid; ++c) ends.push_back({(double)(h[((size_t)i * grid + c) * kTraceSlots + 3] - s0) / 1e3, c});
            std::sort(ends.begin(), ends.end());
            printf("      per-CTA (sorted by end): end_us cta sm tiles pool_draws first_data_us\n");
            for (int k = 0; k < grid; ++k) {
                if (k >= 12 && k < grid - 24 && (k % 16) != 0) continue;
                int c = ends[k].second; unsigned long long w = h[((size_t)i * grid + c) * kTraceSlots + 2];
                printf("        %7.2f %4d sm%3llu tiles %3llu pool %3llu first %5.2f\n", ends[k].first, c, w >> 32, w & 0xffff, (w >> 16) & 0xffff,
                       (double)(h[((size_t)i * grid + c) * kTraceSlots + 1] - s0) / 1e3);
            }
            // per SM: latest end and total tiles
            std::vector<double> sm_end(256, 0); std::vector<int> sm_tiles(256, 0);
            for (int c = 0; c < grid; ++c) { unsigned long long w = h[((size_t)i * grid + c) * kTraceSlots + 2]; int sm = (int)(w >> 32) & 255;
                sm_end[sm] = std::max(sm_end[sm], (double)(h[((size_t)i * grid + c) * kTraceSlots + 3] - s0) / 1e3); sm_tiles[sm] += (int)(w & 0xffff); }
            printf("      per-SM (sm: last end us / tiles):");
            for (int sm = 0; sm < 160; ++sm) if (sm_tiles[sm]) printf(" %d:%.1f/%d", sm, sm_end[sm], sm_tiles[sm]);
            printf("\n");
        }
        int n = NL - 2;
        printf("      trace: spacing %.2f us = window %.2f (first start -> last end) + gap %.2f | mean CTA life %.2f, start spread %.2f, end spread %.2f\n",
               spacing / n / 1e3, win / n / 1e3, gap / n / 1e3, cta / n / 1e3, spread_s / n / 1e3, spread_e / n / 1e3);
        cudaFree(tr);
    }
    cudaFuncAttributes fa; CK(cudaFuncGetAttributes(&fa, kern));
    printf("%-14s %s C=%d PPT=%d thr=%4d stages=%d minb=%d regs=%3d smem=%3zuKB grid=%3d  %8.2f us  %7.1f GB/s  %6.2f Gpix/s\n", tag, TMAP ? "tmap" : "rows", CT, PPT,
           THREADS, STAGES, MINB, fa.numRegs, Cfg::kSmemBytes / 1024, grid, us, bytes_per_px * B * HW / us / 1e3, B * HW / us / 1e3);
    for (void* p : allocs) cudaFree(p);
    cudaFree(ws); cudaFree(sum); cudaFree(counts);
}

static int g_only = -1, g_idx = 0;
// STAGES = 0: as many as fit
template <class Op, int CT, int PPT, int NCW, int MINB, bool TMAP = false>
void run_auto(const char* tag, int64_t B, int64_t HW, int reps, double bpp, bool labels) {
    constexpr int S = tile_stages<tile_stage_bytes<Op, CT, NCW * 32 * PPT, float, TMAP>(), MINB>();
    if (g_only < 0 || g_only == g_idx) run<Op, CT, PPT, NCW, S, MINB, TMAP>(tag, B, HW, reps, bpp, labels);
    ++g_idx;
}
// c2-sized launches (C <= 4): tile of 256 pixels, 4 consumer warps, 3..4 CTAs / SM, row copies vs one box per tensor
template <class Op, int CT>
void sweep_small(const char* tag, int64_t B, int64_t HW, int reps, double bpp, bool labels) {
    run_auto<Op, CT, 2, 8, 2>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 4, 4>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 4, 4, true>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 4, 3, true>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 4, 2, true>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 1, 8, 2, true>(tag, B, HW, reps, bpp, labels);
}
template <class Op, int CT>
void sweep(const char* tag, int64_t B, int64_t HW, int reps, double bpp, bool labels) {
    run_auto<Op, CT, 2, 8, 2>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 4, 8, 2>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 8, 1>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 16, 1>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 4, 16, 1>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 4, 3>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 6, 3>(tag, B, HW, reps, bpp, labels);
    run_auto<Op, CT, 2, 12, 1>(tag, B, HW, reps, bpp, labels);
}
#ifndef KB_NO_MAIN
int main(int argc, char** argv) {
    int reps = argc > 1 ? atoi(argv[1]) : 40;
    if (argc > 2) g_only = atoi(argv[2]);
    int64_t B = argc > 3 ? atoi(argv[3]) : 32;
    if (argc > 4) g_pdl = atoi(argv[4]) != 0;
    int which = argc > 5 ? atoi(argv[5]) : 0;
    if (argc > 6) g_static = atoi(argv[6]) != 0;
    if (argc > 7) g_pool_div = atoi(argv[7]);
    if (const char* e = getenv("DCT_TILE_REFILL")) g_refill = atoi(e);  // 0: C=4 family, 1: C=19 family
    const int64_t HW = 65536;
    if (which == 0) {
        sweep<JsdOp<3, true, kFwdBwd, true>, 4>("jsd+dice c2", B, HW, reps, 104, true);
        sweep<JsdOp<3, true, kFwdBwd, false>, 4>("jsd c2", B, HW, reps, 96, false);
        sweep<CopyOp<3>, 4>("copy3x4", B, HW, reps, 96, false);
        sweep<CopyOp<1>, 4>("copy1x4", B, HW, reps, 32, false);
        sweep<KlFromLogits, 4>("klfromlogits", B, HW, reps, 48, false);
        sweep<KlLogit<true>, 4>("kllogit", B, HW, reps, 64, false);
        sweep<DiceOpB, 4>("dice", B, HW, reps, 24, true);
        sweep<JsdOp<2, true, kFwdBwd, true>, 2>("jsd+dice c3", B / 4, 262144, reps, 40, true);
        sweep<JsdOp<2, true, kFwdBwd, true>, 4>("jsd+dice c1x8", B, 65536, reps, 72, true);
    } else if (which <= 2) {
        // Cityscapes-like: C = 19, 512x1024 images
        const int64_t HWc = 512 * 1024;
        using J19 = JsdOp<2, true, kFwdBwd, false>;
        run_auto<J19, 19, 1, 8, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 1, 4, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 1, 4, 2>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 2, 4, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 1, 16, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 1, 2, 2>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<CopyOp<2>, 19, 1, 8, 1>("copy2x19", B, HWc, reps, 304, false);
        run_auto<CopyOp<2>, 19, 1, 4, 2>("copy2x19", B, HWc, reps, 304, false);
        run_auto<CopyOp<2>, 19, 4, 4, 1>("copy2x19", B, HWc, reps, 304, false);
        run_auto<KlFromLogits, 19, 1, 8, 1>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlFromLogits, 19, 1, 4, 2>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlLogit<true>, 19, 1, 8, 1>("kllogit19", B, HWc, reps, 304, false);
    }
    if (which == 2) {
        const int64_t HWc = 512 * 1024;
        using J3 = JsdOp<3, true, kFwdBwd, false>;
        using J4 = JsdOp<4, true, kFwdBwd, false>;
        run_auto<J3, 19, 1, 4, 1>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 1, 4, 2>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 1, 8, 1>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 2, 2, 2>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 2, 4, 1>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J4, 19, 1, 4, 1>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<J4, 19, 1, 2, 2>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<J4, 19, 1, 8, 1>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<KlFromLogits, 19, 2, 4, 1>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlFromLogits, 19, 2, 4, 2>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlFromLogits, 19, 2, 8, 1>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlLogit<true>, 19, 2, 4, 1>("kllogit19", B, HWc, reps, 304, false);
        run_auto<KlLogit<true>, 19, 2, 4, 2>("kllogit19", B, HWc, reps, 304, false);
        run_auto<JsdOp<2, true, kFwdBwd, false>, 19, 2, 4, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<JsdOp<2, true, kFwdBwd, false>, 19, 2, 6, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<JsdOp<2, true, kFwd, false>, 19, 2, 4, 1>("jsdfwd K2 C19", B, HWc, reps, 152, false);
        run_auto<JsdOp<2, true, kFwd, false>, 19, 2, 8, 1>("jsdfwd K2 C19", B, HWc, reps, 152, false);
    }
    if (which == 3) {
        // rows = 38 family (Cityscapes C = 19, two tensors) and the C = 19 cross-entropy: consumer warps vs stages
        const int64_t HWc = 512 * 1024;
        using J19 = JsdOp<2, true, kFwdBwd, false>;
        run_auto<J19, 19, 2, 5, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 2, 6, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 2, 7, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 2, 8, 1>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 2, 3, 2>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<J19, 19, 2, 4, 2>("jsd K2 C19", B, HWc, reps, 304, false);
        run_auto<KlFromLogits, 19, 2, 6, 1>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlFromLogits, 19, 2, 8, 1>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlFromLogits, 19, 2, 3, 2>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlFromLogits, 19, 2, 6, 2>("klfromlogits19", B, HWc, reps, 228, false);
        run_auto<KlLogit<true>, 19, 2, 6, 1>("kllogit19", B, HWc, reps, 304, false);
        run_auto<KlLogit<true>, 19, 2, 8, 1>("kllogit19", B, HWc, reps, 304, false);
        run_auto<KlLogit<true>, 19, 2, 3, 2>("kllogit19", B, HWc, reps, 304, false);
        using CE = CeOp<true, false, false>;
        run_auto<CE, 19, 2, 4, 1>("ce C19", B, HWc, reps, 160, true);
        run_auto<CE, 19, 2, 8, 1>("ce C19", B, HWc, reps, 160, true);
        run_auto<CE, 19, 2, 4, 2>("ce C19", B, HWc, reps, 160, true);
        run_auto<CE, 19, 2, 6, 2>("ce C19", B, HWc, reps, 160, true);
        run_auto<CE, 19, 4, 4, 2>("ce C19", B, HWc, reps, 160, true);
        using J3 = JsdOp<3, true, kFwdBwd, false>;
        run_auto<J3, 19, 2, 5, 1>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 2, 6, 1>("jsd K3 C19", B, HWc, reps, 456, false);
    }
    if (which == 5) {
        const int64_t HWc = 512 * 1024;
        using JF = JsdOp<2, true, kFwd, false>;
        run_auto<JF, 19, 2, 8, 1>("jsdfwd K2 C19", B, HWc, reps, 152, false);
        run_auto<JF, 19, 2, 3, 2>("jsdfwd K2 C19", B, HWc, reps, 152, false);
        run_auto<JF, 19, 2, 4, 2>("jsdfwd K2 C19", B, HWc, reps, 152, false);
        run_auto<JF, 19, 2, 6, 1>("jsdfwd K2 C19", B, HWc, reps, 152, false);
        using J4 = JsdOp<4, true, kFwdBwd, false>;
        run_auto<J4, 19, 1, 6, 1>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<J4, 19, 1, 3, 2>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<J4, 19, 1, 4, 2>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<J4, 19, 1, 5, 1>("jsd K4 C19", B, HWc, reps, 608, false);
        using J3 = JsdOp<3, true, kFwdBwd, false>;
        run_auto<J3, 19, 2, 5, 1>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 1, 6, 2>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 1, 8, 1>("jsd K3 C19", B, HWc, reps, 456, false);
        using CF = CeOp<false, false, false>;
        run_auto<CF, 19, 2, 4, 2>("cefwd C19", B, HWc, reps, 84, true);
        run_auto<CF, 19, 4, 4, 2>("cefwd C19", B, HWc, reps, 84, true);
        run_auto<CF, 19, 2, 8, 1>("cefwd C19", B, HWc, reps, 84, true);
    }
    if (which == 7) {  // K = 4, C = 19: remaining shapes around the r08 winner (one pixel/thread, 6 warps, 3 stages)
        const int64_t HWc = 512 * 1024;
        using J4 = JsdOp<4, true, kFwdBwd, false>;
        run_auto<J4, 19, 1, 6, 1>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<J4, 19, 1, 3, 2>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<J4, 19, 1, 5, 1>("jsd K4 C19", B, HWc, reps, 608, false);
        run_auto<J4, 19, 1, 7, 1>("jsd K4 C19", B, HWc, reps, 608, false);
        using J3 = JsdOp<3, true, kFwdBwd, false>;
        run_auto<J3, 19, 1, 5, 2>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 1, 4, 2>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 1, 6, 2>("jsd K3 C19", B, HWc, reps, 456, false);
        run_auto<J3, 19, 1, 3, 3>("jsd K3 C19", B, HWc, reps, 456, false);
    }
    if (which == 8) {
        sweep_small<JsdOp<3, true, kFwdBwd, true>, 4>("jsd+dice c2", B, HW, reps, 104, true);
        sweep_small<KlFromLogits, 4>("klfromlogits", B, HW, reps, 48, false);
        sweep_small<KlLogit<true>, 4>("kllogit", B, HW, reps, 64, false);
        sweep_small<CopyOp<3>, 4>("copy3x4", B, HW, reps, 96, false);
        sweep_small<JsdOp<2, true, kFwdBwd, true>, 2>("jsd+dice c3", B / 4, 262144, reps, 40, true);
        sweep_small<JsdOp<2, true, kFwdBwd, true>, 4>("jsd+dice c1", B / 8, 65536, reps, 72, true);
    }
    if (which == 4) {
        // ACDC-sized cross-entropy + Dice (C = 4, 256x256) and the plain variant
        using CED = CeOp<true, true, false>;
        using CE = CeOp<true, false, false>;
        sweep<CED, 4>("ce+dice C4", B, HW, reps, 40, true);
        sweep<CE, 4>("ce C4", B, HW, reps, 40, true);
        sweep<CED, 2>("ce+dice C2", B / 4, 262144, reps, 24, true);
    }
    return 0;
}
#endif  // KB_NO_MAIN
