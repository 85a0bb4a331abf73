// dct_pixelwise.cuh -- one launch skeleton for every "per pixel over the class axis" op of the
// adversarial branch (KL family, softmax, entropy).  Same memory plan as the JSD kernel: all
// NIN*C planes of VEC consecutive pixels are fetched with independent coalesced streaming loads,
// the math runs in registers, results go back with streaming stores, the optional map sum is a
// deterministic two-stage reduction.  CT == 0 instantiates the runtime-C fallback (VEC = 1,
// per-thread arrays in local memory) so every C <= DCT_MAX_CLASSES is served.
#pragma once
#include "dct_common.cuh"
#include "dct_tile.cuh"

namespace dct {

struct PixArgs {
    const float* in[2];
    float* out[2];      // each nullable
    int C;
    int64_t B, HW;      // images b = blockIdx.y, blockIdx.y + gridDim.y, ... (image_grid)
    float* map;         // nullable
    double* sum;        // nullable
    Upstream up;
    float eps;
    int32_t* flags;     // nullable
    Workspace* ws;
};

// (NIN*CT <= 16 has no register-tiled instantiation: the tile pipeline takes every call such a kernel could, see pix_launch_ct)
template <int NIN, int CT>
constexpr int pix_vec() {
    return CT == 0 ? 1 : (NIN * CT <= 40 ? 2 : 1);
}

// Op interface:
//   static constexpr int NIN, NOUT (NOUT <= NIN: outputs reuse the input registers);
//   static constexpr bool HAS_MAP  (produces a per-pixel scalar), USES_UP (consumes an upstream);
//   template <int CM, class T> static T apply(T (&x)[NIN][CM], int C, T g, float eps, bool& bad)   (T = float | f2)
//       in: x = inputs; out: x[0..NOUT) = outputs; returns the map value.
template <class Op, int CT, int VEC>
__global__ void __launch_bounds__(256) pix_kernel(const PixArgs a) {
    constexpr int CM = CT ? CT : DCT_MAX_CLASSES;
    constexpr int NIN = Op::NIN, NOUT = Op::NOUT;
    const int C = CT ? CT : a.C;
    const int64_t HW = a.HW;
    const int64_t gpi = HW / VEC;
    float gs = 1.0f;
    if constexpr (Op::USES_UP) gs = upstream_scalar(a.up);
    double acc = 0.0;
    bool bad = false;
    for (int64_t b = blockIdx.y; b < a.B; b += gridDim.y) {
        const int64_t img = b * C * HW;
        for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < gpi; g += (int64_t)gridDim.x * blockDim.x) {
            const int64_t i = g * VEC;
            FVec<VEC> xin[NIN][CM];
#pragma unroll
            for (int n = 0; n < NIN; ++n)
#pragma unroll
                for (int c = 0; c < CM; ++c)
                    if (c < C) xin[n][c] = ld_stream<VEC>(a.in[n] + img + (int64_t)c * HW + i);
            FVec<VEC> gm;
#pragma unroll
            for (int v = 0; v < VEC; ++v) gm.v[v] = 1.0f;
            if constexpr (Op::USES_UP) {
                if (a.up.gmap != nullptr) gm = ld_stream<VEC>(a.up.gmap + b * HW + i);
            }
            FVec<VEC> mapv;
            float part = 0.0f;
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                float x[NIN][CM];
#pragma unroll
                for (int n = 0; n < NIN; ++n)
#pragma unroll
                    for (int c = 0; c < CM; ++c)
                        if (c < C) x[n][c] = xin[n][c].v[v];
                float mv = Op::template apply<CM, float>(x, C, gs * gm.v[v], a.eps, bad);
                mapv.v[v] = mv;
                part += mv;
#pragma unroll
                for (int n = 0; n < NOUT; ++n)
#pragma unroll
                    for (int c = 0; c < CM; ++c)
                        if (c < C) xin[n][c].v[v] = x[n][c];
            }
            acc += (double)part;
            if constexpr (Op::HAS_MAP) {
                if (a.map != nullptr) st_stream<VEC>(a.map + b * HW + i, mapv);
            }
#pragma unroll
            for (int n = 0; n < NOUT; ++n)
                if (a.out[n] != nullptr) {
#pragma unroll
                    for (int c = 0; c < CM; ++c)
                        if (c < C) st_stream<VEC>(a.out[n] + img + (int64_t)c * HW + i, xin[n][c]);
                }
        }
    }
    if constexpr (Op::CHECKS_SIMPLEX) {
        if (a.flags != nullptr && __syncthreads_or(bad)) {
            if (bad) atomicAdd(&a.flags[DCT_FLAG_SIMPLEX], 1);
        }
    }
    if constexpr (Op::HAS_MAP) grid_sum_to(acc, a.ws, a.sum, blockIdx.y * gridDim.x + blockIdx.x, gridDim.x * gridDim.y);
}

template <class Op, int CT>
int pix_launch_ct(const PixArgs& a, int64_t B, cudaStream_t stream) {
    if constexpr (CT > 0 && Op::NIN * CT <= kTileMaxRows) {
        TileArgs t{};
        for (int n = 0; n < Op::NIN; ++n) t.in[n] = a.in[n];
        for (int n = 0; n < Op::NOUT; ++n) t.out[n] = a.out[n];
        t.HW = a.HW; t.map = a.map; t.sum = a.sum; t.up = a.up; t.eps = a.eps; t.flags = a.flags; t.ws = a.ws;
        if (tile_eligible<Op>(t, B)) return tile_launch_ct<Op, CT>(t, B, stream);
    }
    if constexpr (CT > 0 && Op::NIN * CT <= 16) {
        return DCT_ERR_UNSUPPORTED;   // refused by the tile pipeline: the caller falls back to pix_kernel<Op, 0, 1>
    } else {
        constexpr int VEC = pix_vec<Op::NIN, CT>();
        bool al = (a.HW % VEC) == 0 && (a.map == nullptr || aligned(a.map, 4 * VEC)) &&
                  (a.up.gmap == nullptr || aligned(a.up.gmap, 4 * VEC));
        for (int n = 0; n < Op::NIN; ++n) al = al && aligned(a.in[n], 4 * VEC);
        for (int n = 0; n < Op::NOUT; ++n) al = al && (a.out[n] == nullptr || aligned(a.out[n], 4 * VEC));
        if (!al) return DCT_ERR_UNSUPPORTED;
        const int threads = 256;
        dim3 grid = image_grid(B, a.HW / VEC, threads);
        if (Op::HAS_MAP && !fits_partials(grid)) return DCT_ERR_UNSUPPORTED;
        PixArgs ab = a;
        ab.B = B;
        pix_kernel<Op, CT, VEC><<<grid, threads, 0, stream>>>(ab);
        return check_launch();
    }
}

template <class Op>
int pix_launch(const PixArgs& a, int64_t B, cudaStream_t stream) {
    if (a.C < 1 || B < 1 || a.HW < 1) return DCT_ERR_BAD_ARG;
    if (a.C > DCT_MAX_CLASSES || B > 65535) return DCT_ERR_UNSUPPORTED;
    for (int n = 0; n < Op::NIN; ++n) {
        if (a.in[n] == nullptr) return DCT_ERR_BAD_ARG;
        if (!aligned(a.in[n], 4)) return DCT_ERR_MISALIGNED;
    }
    if (Op::HAS_MAP && a.sum != nullptr && a.ws == nullptr) return DCT_ERR_BAD_ARG;
    int rc = DCT_ERR_UNSUPPORTED;
    switch (a.C) {
        case 2: rc = pix_launch_ct<Op, 2>(a, B, stream); break;
        case 3: rc = pix_launch_ct<Op, 3>(a, B, stream); break;
        case 4: rc = pix_launch_ct<Op, 4>(a, B, stream); break;
        case 19: rc = pix_launch_ct<Op, 19>(a, B, stream); break;
        default: break;
    }
    if (rc == DCT_ERR_UNSUPPORTED) rc = pix_launch_ct<Op, 0>(a, B, stream);
    return rc;
}

}  // namespace dct
