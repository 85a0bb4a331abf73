// dct_hausdorff.cu -- Hausdorff distance between two class maps on the device (evaluation path, Summary.py:25).
//
// Definition: medpy.metric.binary.hd (the ACDC challenge's evaluation code), per class c on a grid (one H x W slice, or the
// B x H x W batch as one volume):  A = {pred == c}, G = {gt == c};  border(M) = M xor binary_erosion(M) with the cross
// structuring element and cells outside the grid as background (medpy's __surface_distances);  d(x, S) = min over y in S of
// ||(x - y) * spacing||_2;  HD = max(max_{x in border(A)} d(x, border(G)), max_{y in border(G)} d(y, border(A))).  NaN if A or
// G is empty (medpy raises).  Since every pixel carries exactly one class, a pixel is a border pixel of its class exactly when
// one of its 4 (6) neighbours holds another value or lies off the grid.
//
// Work per call (2 sides x C classes = 2C feature sets, each the border set of one class on one side):
//   hd_classify_kernel   one pass over both int64 maps: a 2-byte record per pixel (per side: class | 0x80 on the border,
//                        0x7F for a value outside [0,C)); zeroes the per-(row, class, side) maxima and presence words.
//   hd_column_kernel     one thread per (side, class, image, column): two sweeps along H give the distance in rows to the
//                        nearest feature of the column (uint16, 0xFFFF = none); coalesced across columns.
//   hd_envelope_kernel   exact squared EDT along one more axis: lower envelope of the parabolas f(q) + w (x - q)^2
//                        (Felzenszwalb-Huttenlocher) restricted to integer positions, one thread per line with its stack in
//                        shared memory.  Along W it either writes the float map (volume) or is the last pass; along B
//                        (volume) it is the last pass.  The last pass folds max over the other side's border pixels of d^2
//                        into the (row, class, side) maximum with an integer atomicMax on the float bits (non-negative
//                        floats order like their bit patterns): order-independent, so bit-reproducible.
//   hd_finish_kernel     HD = __fsqrt_rn(max of the two sides), NaN where a side's set is empty.
// Launches: 4 for '2d', 5 for a volume.  Envelope arithmetic is double; at unit spacing every d^2 is an integer, exact in
// the float maxima up to 2^24, so the result is the correctly rounded square root of the exact squared distance.
#include <math_constants.h>

#include <algorithm>
#include <climits>
#include <cmath>

#include "dct_common.cuh"

namespace dct {

constexpr int kHdMaxAxis = 32768;                 // stack entries hold (position, region start) as two uint16
constexpr uint16_t kNone = 0xFFFF;                // hd_column_kernel: no feature in the column
constexpr unsigned char kOutOfRange = 0x7F;       // record byte of a value outside [0,C): matches no (class | 0x80)
constexpr int kEnvSmemBudget = 48 * 1024;         // per CTA; a line of n positions takes 4n bytes of stack

struct HdGeom {
    int C;
    int64_t B, H, W, N;   // N = B*H*W
    int volume;
};

// shapes the kernels take: axes within the 16-bit stack entries, every grid within 2^31 - 1 threads
inline bool hd_supported(int C, int64_t B, int64_t H, int64_t W, int volume) {
    if (C > DCT_MAX_CLASSES || H > kHdMaxAxis || W > kHdMaxAxis || (volume && B > kHdMaxAxis)) return false;
    const int64_t lines = 2 * (int64_t)C * B * std::max(H, W);   // column and row passes
    return lines <= INT_MAX && (!volume || 2 * (int64_t)C * H * W <= INT_MAX);
}

inline size_t hd_align256(size_t v) { return (v + 255) & ~(size_t)255; }

struct HdLayout {
    size_t hdr, rec, g, f, total;
};
inline HdLayout hd_layout(int C, int64_t B, int64_t H, int64_t W, int volume) {
    const size_t N = (size_t)B * H * W, rows = volume ? 1 : (size_t)B;
    HdLayout L;
    L.hdr = 0;                                          // uint32 rowmax[rows][C][2], present[rows][C][2]
    L.rec = hd_align256(L.hdr + rows * C * 2 * 2 * 4);     // uint16 [N]: pred byte | gt byte << 8
    L.g = hd_align256(L.rec + N * 2);                      // uint16 [2][C][N]
    L.f = hd_align256(L.g + 2 * (size_t)C * N * 2);        // float  [2][C][N] (volume only)
    L.total = volume ? hd_align256(L.f + 2 * (size_t)C * N * 4) : L.f;
    return L;
}

__device__ __forceinline__ unsigned side_byte(uint16_t r, int side) { return side ? (r >> 8) : (r & 0xFFu); }

__global__ void __launch_bounds__(256) hd_classify_kernel(const int64_t* __restrict__ pred, const int64_t* __restrict__ gt,
                                                           const HdGeom g, uint16_t* __restrict__ rec, unsigned* hdr, int nhdr,
                                                           int32_t* flags) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < nhdr; i += nthr) hdr[i] = 0u;
    const int64_t HW = g.H * g.W;
    int bad_pred = 0, bad_gt = 0;
    for (int64_t p = tid; p < g.N; p += nthr) {
        const int64_t b = p / HW, yx = p - b * HW, y = yx / g.W, x = yx - y * g.W;
        unsigned byte[2];
        const int64_t* maps[2] = {pred, gt};
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int64_t* m = maps[s];
            const long long v = m[p];
            if (v < 0 || v >= g.C) {
                byte[s] = kOutOfRange;
                if (s) ++bad_gt; else ++bad_pred;
                continue;
            }
            bool border = x == 0 || x == g.W - 1 || y == 0 || y == g.H - 1;
            if (!border) border = m[p - 1] != v || m[p + 1] != v || m[p - g.W] != v || m[p + g.W] != v;
            if (!border && g.volume) border = b == 0 || b == g.B - 1 || m[p - HW] != v || m[p + HW] != v;
            byte[s] = (unsigned)v | (border ? 0x80u : 0u);
        }
        rec[p] = (uint16_t)(byte[0] | (byte[1] << 8));
    }
    if (flags != nullptr) {
        bad_pred = __reduce_add_sync(0xffffffffu, bad_pred);
        bad_gt = __reduce_add_sync(0xffffffffu, bad_gt);
        if ((threadIdx.x & 31) == 0) {
            if (bad_pred) atomicAdd(&flags[DCT_FLAG_PRED], bad_pred);
            if (bad_gt) atomicAdd(&flags[DCT_FLAG_LABEL], bad_gt);
        }
    }
}

// one thread per (side, class, image, column); adjacent threads take adjacent columns
__global__ void __launch_bounds__(128) hd_column_kernel(const uint16_t* __restrict__ rec, const HdGeom g,
                                                        uint16_t* __restrict__ gdist, unsigned* present) {
    const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t per_sc = g.B * g.W;
    if (line >= 2 * g.C * per_sc) return;
    const int sc = (int)(line / per_sc), side = sc / g.C, c = sc - side * g.C;
    const int64_t r = line - sc * per_sc, b = r / g.W, x = r - b * g.W;
    const int64_t base = b * g.H * g.W + x;
    const unsigned want = (unsigned)c | 0x80u;
    const uint16_t* in = rec + base;
    uint16_t* out = gdist + (int64_t)sc * g.N + base;
    int last = -1;
    for (int y = 0; y < g.H; ++y) {
        if (side_byte(in[(int64_t)y * g.W], side) == want) last = y;
        out[(int64_t)y * g.W] = last < 0 ? kNone : (uint16_t)(y - last);
    }
    if (last < 0) return;   // no feature in this column
    present[((g.volume ? 0 : b) * g.C + c) * 2 + side] = 1u;
    int next = -1;
    for (int y = (int)g.H - 1; y >= 0; --y) {
        const int64_t o = (int64_t)y * g.W;
        if (side_byte(in[o], side) == want) next = y;
        if (next >= 0) {
            const uint16_t d = (uint16_t)(next - y);
            if (d < out[o]) out[o] = d;
        }
    }
}

struct EnvArgs {
    const uint16_t* gdist;   // FROM_G: input distances in rows (weight w_in)
    const float* fin;        // !FROM_G: input squared distances
    float* fout;             // !FOLD: output squared distances
    const uint16_t* rec;     // FOLD: border records of the queries
    unsigned* rowmax;        // FOLD: [rows][C][2] float bits
    HdGeom g;
    int64_t lines_per_plane, line_step, stride, lines_per_row;
    int n;
    double w_in, w;          // squared spacing of the previous axis (FROM_G) and of this one
};

template <bool FROM_G>
__device__ __forceinline__ double env_load(const EnvArgs& a, int64_t plane, int64_t off) {
    if constexpr (FROM_G) {
        const uint16_t d = a.gdist[plane + off];
        return d == kNone ? CUDART_INF : a.w_in * (double)d * (double)d;
    } else {
        return (double)a.fin[plane + off];
    }
}

// Lower envelope of {f(q) + w (x - q)^2} over the finite f(q) of one line, evaluated at the integer positions x of the
// line.  Stack entry k = (position v_k, first integer position z_k at which parabola v_k is the lowest); a new parabola q
// (to the right of every stacked one) is at or below v_k from ceil(sep) on, so v_k is popped when ceil(sep) <= z_k and q is
// only pushed when ceil(sep) < n.
template <bool FROM_G, bool FOLD>
__global__ void __launch_bounds__(64) hd_envelope_kernel(const EnvArgs a) {
    extern __shared__ unsigned stk_all[];
    const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= 2 * a.g.C * a.lines_per_plane) return;
    const int sc = (int)(line / a.lines_per_plane), side = sc / a.g.C, c = sc - side * a.g.C;
    const int64_t l = line - sc * a.lines_per_plane;
    const int64_t plane = (int64_t)sc * a.g.N, base = l * a.line_step, stride = a.stride;
    const int n = a.n, R = blockDim.x;
    unsigned* stk = stk_all + threadIdx.x;   // entry k at stk[k * R]
    const double w = a.w;
    int top = -1;
    for (int q = 0; q < n; ++q) {
        const double fq = env_load<FROM_G>(a, plane, base + q * stride);
        if (isinf(fq)) continue;
        const double hq = fq + w * (double)q * (double)q;
        int zq = 0;
        bool push = true;
        while (top >= 0) {
            const unsigned e = stk[top * R];
            const int v = (int)(e & 0xFFFFu), zv = (int)(e >> 16);
            const double hv = env_load<FROM_G>(a, plane, base + v * stride) + w * (double)v * (double)v;
            const double cs = ceil((hq - hv) / (2.0 * w * (double)(q - v)));
            if (cs <= (double)zv) { --top; continue; }
            if (cs >= (double)n) push = false;
            else zq = (int)cs;
            break;
        }
        if (push) stk[++top * R] = (unsigned)q | ((unsigned)zq << 16);
    }
    const unsigned want = (unsigned)c | 0x80u;
    float m = 0.0f;
    bool any = false;
    int k = 0;
    for (int x = 0; x < n; ++x) {
        const int64_t off = base + x * stride;
        if constexpr (FOLD) {
            if (side_byte(a.rec[off], 1 - side) != want) continue;   // queries: the other side's border pixels of c
        }
        float d = CUDART_INF_F;
        if (top >= 0) {
            while (k < top && (int)(stk[(k + 1) * R] >> 16) <= x) ++k;
            const int v = (int)(stk[k * R] & 0xFFFFu);
            d = (float)(env_load<FROM_G>(a, plane, base + v * stride) + w * (double)(x - v) * (double)(x - v));
        }
        if constexpr (FOLD) { m = fmaxf(m, d); any = true; }
        else a.fout[plane + off] = d;
    }
    if constexpr (FOLD) {
        if (any) {
            const int64_t row = l / a.lines_per_row;
            atomicMax(&a.rowmax[(row * a.g.C + c) * 2 + side], __float_as_uint(m));
        }
    }
}

__global__ void hd_finish_kernel(const unsigned* __restrict__ rowmax, const unsigned* __restrict__ present, int64_t n,
                                 float* __restrict__ hd) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        const bool both = present[2 * j] != 0u && present[2 * j + 1] != 0u;
        const unsigned bits = max(rowmax[2 * j], rowmax[2 * j + 1]);
        hd[j] = both ? __fsqrt_rn(__uint_as_float(bits)) : CUDART_NAN_F;
    }
}

template <bool FROM_G, bool FOLD>
cudaError_t launch_envelope(const EnvArgs& a, cudaStream_t s) {
    const int64_t lines = 2 * a.g.C * a.lines_per_plane;
    int R = kEnvSmemBudget / (4 * a.n);
    R = R > 64 ? 64 : (R < 1 ? 1 : R);
    const size_t smem = (size_t)R * a.n * 4;
    if (smem > (size_t)kEnvSmemBudget) {
        cudaError_t e = cudaFuncSetAttribute(hd_envelope_kernel<FROM_G, FOLD>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem);
        if (e != cudaSuccess) return e;
    }
    hd_envelope_kernel<FROM_G, FOLD><<<(unsigned)((lines + R - 1) / R), R, smem, s>>>(a);
    return cudaGetLastError();
}

}  // namespace dct

using namespace dct;

extern "C" size_t dct_hausdorff_scratch_bytes(int C, int64_t B, int64_t H, int64_t W, int volume) {
    if (C < 1 || B < 1 || H < 1 || W < 1 || !hd_supported(C, B, H, W, volume)) return 0;
    return hd_layout(C, B, H, W, volume).total;
}

extern "C" int dct_hausdorff_i64(const int64_t* pred, const int64_t* labels, int C, int64_t B, int64_t H, int64_t W,
                                 int volume, const double* spacing, float* hd, int32_t* flags, void* scratch, void* stream) {
    if (pred == nullptr || labels == nullptr || hd == nullptr || scratch == nullptr) return DCT_ERR_BAD_ARG;
    if (C < 1 || B < 1 || H < 1 || W < 1) return DCT_ERR_BAD_ARG;
    if (!hd_supported(C, B, H, W, volume)) return DCT_ERR_UNSUPPORTED;
    double sp[3] = {1.0, 1.0, 1.0};   // (sz,) sy, sx
    if (spacing != nullptr) {
        for (int i = 0; i < (volume ? 3 : 2); ++i) {
            const double v = spacing[i];
            if (!(v > 0.0) || !std::isfinite(v)) return DCT_ERR_BAD_ARG;   // also rejects NaN
            sp[volume ? i : i + 1] = v;
        }
    }
    if (!aligned(pred, 8) || !aligned(labels, 8) || !aligned(hd, 4) || !aligned(flags, 4) || !aligned(scratch, 256))
        return DCT_ERR_MISALIGNED;
    const HdGeom g{C, B, H, W, B * H * W, volume ? 1 : 0};
    const HdLayout L = hd_layout(C, B, H, W, volume);
    char* base = static_cast<char*>(scratch);
    unsigned* rowmax = reinterpret_cast<unsigned*>(base + L.hdr);
    const int64_t rows = volume ? 1 : B, nrc = rows * C;
    unsigned* present = rowmax + 2 * nrc;
    uint16_t* rec = reinterpret_cast<uint16_t*>(base + L.rec);
    uint16_t* gdist = reinterpret_cast<uint16_t*>(base + L.g);
    float* f = reinterpret_cast<float*>(base + L.f);
    cudaStream_t s = static_cast<cudaStream_t>(stream);

    const int64_t cls_blocks = std::min<int64_t>((g.N + 255) / 256, (int64_t)kSMs * 16);
    hd_classify_kernel<<<(unsigned)cls_blocks, 256, 0, s>>>(pred, labels, g, rec, rowmax, (int)(4 * nrc), flags);
    const int64_t col_lines = 2 * (int64_t)C * B * W;
    hd_column_kernel<<<(unsigned)((col_lines + 127) / 128), 128, 0, s>>>(rec, g, gdist, present);
    cudaError_t e = cudaGetLastError();

    EnvArgs a{};
    a.gdist = gdist; a.rec = rec; a.rowmax = rowmax; a.g = g;
    a.lines_per_plane = B * H; a.line_step = W; a.stride = 1; a.n = (int)W;
    a.w_in = sp[1] * sp[1]; a.w = sp[2] * sp[2];
    if (e == cudaSuccess) {
        if (!volume) {
            a.lines_per_row = H;   // line l = b * H + y lies in image b
            e = launch_envelope<true, true>(a, s);
        } else {
            a.fout = f;
            e = launch_envelope<true, false>(a, s);
            EnvArgs z{};
            z.fin = f; z.rec = rec; z.rowmax = rowmax; z.g = g;
            z.lines_per_plane = H * W; z.line_step = 1; z.stride = H * W; z.n = (int)B;
            z.lines_per_row = H * W;   // one row: the volume
            z.w = sp[0] * sp[0];
            if (e == cudaSuccess) e = launch_envelope<false, true>(z, s);
        }
    }
    if (e == cudaSuccess) {
        hd_finish_kernel<<<(unsigned)std::min<int64_t>((nrc + 127) / 128, 1024), 128, 0, s>>>(rowmax, present, nrc, hd);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return DCT_OK;
}
