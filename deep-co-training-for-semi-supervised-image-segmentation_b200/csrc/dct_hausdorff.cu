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
//
// dct_surface_distances_i64 (HD95, ASD, ASSD; medpy.metric.binary hd95 / asd / assd) runs the same passes with the last
// one in its SURF mode, which also keeps every query's d^2 and per-line sums, then:
//   sd_sum_kernel        fixed-order reduction of the per-line sums and counts per (row, class, side); rank to select.
//   sd_select_kernel<P>  P = 0..3: radix histogram of 8 key bits under the selected prefix; P = 4: least key above it.
//   sd_pick_kernel<P>    narrows prefix and rank from the histogram of pass P.
//   sd_finish_kernel     hd, hd95, asd, assd.
// Launches: 14 for '2d', 15 for a volume.
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
    size_t hdr, rec, g, f, total;              // dct_hausdorff_i64
    size_t qd, lsum, lcnt, hist, st, surf_total;   // dct_surface_distances_i64: the same, then these
};
constexpr size_t kSdStateBytes = 64;   // sizeof(SdState)
inline HdLayout hd_layout(int C, int64_t B, int64_t H, int64_t W, int volume) {
    const size_t N = (size_t)B * H * W, rows = volume ? 1 : (size_t)B;
    const size_t fold_lines = 2 * (size_t)C * (volume ? (size_t)H * W : (size_t)B * H);   // lines of the last pass
    HdLayout L;
    L.hdr = 0;                                          // uint32 rowmax[rows][C][2], present[rows][C][2]
    L.rec = hd_align256(L.hdr + rows * C * 2 * 2 * 4);     // uint16 [N]: pred byte | gt byte << 8
    L.g = hd_align256(L.rec + N * 2);                      // uint16 [2][C][N]
    L.f = hd_align256(L.g + 2 * (size_t)C * N * 2);        // float  [2][C][N] (volume only)
    L.total = volume ? hd_align256(L.f + 2 * (size_t)C * N * 4) : L.f;
    L.qd = L.total;                                        // float  [2][N]
    L.lsum = hd_align256(L.qd + 2 * N * 4);                // double [fold_lines]
    L.lcnt = hd_align256(L.lsum + fold_lines * 8);         // uint32 [fold_lines]
    L.hist = hd_align256(L.lcnt + fold_lines * 4);         // uint64 [rows][C][256]
    L.st = hd_align256(L.hist + rows * C * 256 * 8);       // SdState [rows][C]
    L.surf_total = hd_align256(L.st + rows * C * kSdStateBytes);
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
    float* qd;               // SURF: [2][N] squared distance of each query pixel to the border set of that side
    double* lsum;            // SURF: per line of the last pass, sum of sqrt(d^2) over its queries
    unsigned* lcnt;          // SURF: per line of the last pass, number of its queries
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
// only pushed when ceil(sep) < n.  SURF (last pass of dct_surface_distances_i64): also keep every query's d^2 and the
// line's sum of distances and query count.
template <bool FROM_G, bool FOLD, bool SURF = false>
__global__ void __launch_bounds__(64) hd_envelope_kernel(const EnvArgs a) {
    static_assert(FOLD || !SURF, "only the last pass has queries");
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
    double dsum = 0.0;
    unsigned cnt = 0;
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
        if constexpr (SURF) {
            a.qd[side * a.g.N + off] = d;   // a pixel is a query of one class per side: no other line writes here
            dsum += sqrt((double)d);
            ++cnt;
        }
    }
    if constexpr (FOLD) {
        if (any) {
            const int64_t row = l / a.lines_per_row;
            atomicMax(&a.rowmax[(row * a.g.C + c) * 2 + side], __float_as_uint(m));
        }
    }
    if constexpr (SURF) { a.lsum[line] = dsum; a.lcnt[line] = cnt; }
}

__device__ __forceinline__ float hd_value(const unsigned* __restrict__ rowmax, const unsigned* __restrict__ present,
                                          int64_t j) {
    const bool both = present[2 * j] != 0u && present[2 * j + 1] != 0u;
    const unsigned bits = max(rowmax[2 * j], rowmax[2 * j + 1]);
    return both ? __fsqrt_rn(__uint_as_float(bits)) : CUDART_NAN_F;
}

__global__ void hd_finish_kernel(const unsigned* __restrict__ rowmax, const unsigned* __restrict__ present, int64_t n,
                                 float* __restrict__ hd) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x)
        hd[j] = hd_value(rowmax, present, j);
}

// ---- surface distances (dct_surface_distances_i64): HD95, ASD, ASSD from the last pass's per-query d^2 -------------
//
// Per (row, class) the keys are the float bits of the d^2 of both sides' queries (non-negative floats order like their
// bits).  HD95 is numpy's 'linear' percentile of the distances: with n keys, v = (n - 1) * 0.95, lo = floor(v), the
// keys at ranks lo and lo + 1 are found by a radix select (4 passes of 8 bits, integer histograms) and, when the run of
// keys equal to the one at rank lo ends there, one pass for the least key above it.
struct SdState {
    double sum[2];                // per side: sum of the distances of its queries (fixed-order reduction of the lines)
    unsigned long long cnt[2];    // per side: number of its queries
    long long k;                  // rank still to skip below the selected prefix
    unsigned long long run;       // after the last pass: number of keys equal to the one at rank lo
    unsigned prefix;              // high bits selected so far; after the last pass the key at rank lo
    unsigned hikey;               // need_hi: the least key above it (atomicMin target)
    unsigned active;              // some key to select from
    unsigned need_hi;             // the key at rank lo + 1 is above the one at rank lo
};
static_assert(sizeof(SdState) == kSdStateBytes, "scratch layout");

// numpy.percentile(x, 95) with the default method 'linear': virtual index (n - 1) * 0.95, its floor and fraction
__device__ __forceinline__ double sd_rank95(unsigned long long n, long long* lo) {
    const double v = (double)(n - 1) * 0.95, f = floor(v);
    *lo = (long long)f;
    return v - f;
}

// one CTA per (row, class): both sides' per-line sums and counts in a fixed order (bit-reproducible), the rank to
// select, and a zeroed histogram for the first select pass
constexpr int kSumThreads = 512;
__global__ void __launch_bounds__(kSumThreads) sd_sum_kernel(const double* __restrict__ lsum,
                                                             const unsigned* __restrict__ lcnt, const HdGeom g,
                                                             int64_t lines_per_plane, int64_t lines_per_row, int64_t nrc,
                                                             SdState* st, unsigned long long* hist) {
    __shared__ double ssum[kSumThreads];
    __shared__ unsigned long long scnt[kSumThreads];
    const int t = threadIdx.x;
    for (int64_t rc = blockIdx.x; rc < nrc; rc += gridDim.x) {
        const int64_t row = rc / g.C;
        const int c = (int)(rc - row * g.C);
        double tot[2];
        unsigned long long num[2];
        for (int side = 0; side < 2; ++side) {
            const int64_t base = (int64_t)(side * g.C + c) * lines_per_plane + row * lines_per_row;
            double s = 0.0;
            unsigned long long n = 0;
            for (int64_t j = t; j < lines_per_row; j += kSumThreads) { s += lsum[base + j]; n += lcnt[base + j]; }
            ssum[t] = s; scnt[t] = n;
            __syncthreads();
            for (int h = kSumThreads / 2; h > 0; h >>= 1) {
                if (t < h) { ssum[t] += ssum[t + h]; scnt[t] += scnt[t + h]; }
                __syncthreads();
            }
            tot[side] = ssum[0]; num[side] = scnt[0];
            __syncthreads();
        }
        for (int i = t; i < 256; i += kSumThreads) hist[rc * 256 + i] = 0ull;
        if (t == 0) {
            SdState& s = st[rc];
            const unsigned long long n = num[0] + num[1];
            long long lo = 0;
            if (n > 0) sd_rank95(n, &lo);
            s.sum[0] = tot[0]; s.sum[1] = tot[1]; s.cnt[0] = num[0]; s.cnt[1] = num[1];
            s.k = lo; s.run = 0; s.prefix = 0u; s.hikey = 0xFFFFFFFFu; s.active = n > 0; s.need_hi = 0u;
        }
    }
}

struct SdTasks {
    int64_t rowpix, chunk, chunks_per_row, tasks;   // a task: `chunk` pixels of one row
};

// PASS 0..3: per-(row, class) histogram of key bits [24 - 8 PASS, 32 - 8 PASS) over the keys whose higher bits equal
// the selected prefix, counted in shared memory per task and added to `hist`.  PASS 4: least key above the selected one
// for the (row, class) that need it.  Every block runs the same number of iterations per task (whole warps vote).
template <int PASS>
__global__ void __launch_bounds__(256) sd_select_kernel(const uint16_t* __restrict__ rec, const float* __restrict__ qd,
                                                        const HdGeom g, const SdTasks tk, unsigned long long* hist,
                                                        SdState* st) {
    constexpr bool MIN = PASS == 4;
    extern __shared__ unsigned sm[];
    const int nb = MIN ? g.C : g.C * 256;
    unsigned* bins = sm;          // PASS < 4: [C][256] counts; PASS 4: [C] least key above the selected one
    unsigned* pre = sm + nb;      // [C] selected prefix (PASS 4: the selected key)
    unsigned* act = pre + g.C;    // [C] the class takes part in this pass
    const int lane = threadIdx.x & 31;
    for (int64_t task = blockIdx.x; task < tk.tasks; task += gridDim.x) {
        const int64_t row = task / tk.chunks_per_row;
        const int64_t p0 = row * tk.rowpix + (task - row * tk.chunks_per_row) * tk.chunk;
        const int64_t p1 = min(p0 + tk.chunk, (row + 1) * tk.rowpix);
        __syncthreads();   // the previous task's bins have been flushed
        for (int i = threadIdx.x; i < nb; i += blockDim.x) bins[i] = MIN ? 0xFFFFFFFFu : 0u;
        for (int c = threadIdx.x; c < g.C; c += blockDim.x) {
            const SdState& s = st[row * g.C + c];
            pre[c] = s.prefix;
            act[c] = MIN ? s.need_hi : s.active;
        }
        __syncthreads();
        for (int64_t q = p0; q < p1; q += blockDim.x) {
            const int64_t p = q + threadIdx.x;
            const unsigned r = p < p1 ? rec[p] : 0u;   // 0: a border pixel on neither side
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const unsigned byte = side_byte((uint16_t)r, 1 - s);   // query of side s's border set (last envelope pass)
                const int c = (int)(byte & 0x7Fu);
                unsigned tag = 0xFFFFFFFFu, key = 0u;
                if ((byte & 0x80u) && act[c]) {
                    key = __float_as_uint(qd[s * g.N + p]);
                    if constexpr (PASS == 0) {
                        tag = (unsigned)c * 256u + (key >> 24);
                    } else if constexpr (!MIN) {
                        if ((key >> (32 - 8 * PASS)) == pre[c]) tag = (unsigned)c * 256u + ((key >> (24 - 8 * PASS)) & 0xFFu);
                    } else {
                        if (key > pre[c]) tag = (unsigned)c;
                    }
                }
                if constexpr (!MIN) {
                    // salt-and-pepper maps put most keys of a warp into one bin: one shared atomic per distinct bin
                    const unsigned peers = __match_any_sync(0xffffffffu, tag);
                    if (tag != 0xFFFFFFFFu && lane == __ffs(peers) - 1) atomicAdd(&bins[tag], (unsigned)__popc(peers));
                } else {
                    if (tag != 0xFFFFFFFFu && key < bins[tag]) atomicMin(&bins[tag], key);
                }
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < nb; i += blockDim.x) {
            if constexpr (!MIN) {
                if (bins[i] != 0u) atomicAdd(&hist[row * g.C * 256 + i], (unsigned long long)bins[i]);
            } else {
                if (bins[i] != 0xFFFFFFFFu) atomicMin(&st[row * g.C + i].hikey, bins[i]);
            }
        }
    }
}

// one warp per (row, class): the bin holding rank k of the PASS histogram (lane l scans bins 8l..8l+7), which narrows the
// prefix and the rank; the histogram is zeroed for the next pass
template <int PASS>
__global__ void __launch_bounds__(256) sd_pick_kernel(unsigned long long* hist, SdState* st, int64_t nrc) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t rc = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; rc < nrc; rc += warps) {
        SdState& s = st[rc];
        if (!s.active) continue;   // nothing counted: the histogram is still zero
        unsigned long long* hb = hist + rc * 256 + lane * 8;
        unsigned long long h[8], sum = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { h[i] = hb[i]; sum += h[i]; hb[i] = 0ull; }
        unsigned long long incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const long long k = s.k;
        const unsigned hit = __ballot_sync(0xffffffffu, incl > (unsigned long long)k);
        if (lane == __ffs(hit) - 1) {
            long long kk = k - (long long)(incl - sum);
            int bin = -1;
            unsigned long long run = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (bin < 0) {
                    if (kk < (long long)h[i]) { bin = lane * 8 + i; run = h[i]; }
                    else kk -= (long long)h[i];
                }
            }
            s.prefix = (PASS == 0 ? 0u : s.prefix << 8) | (unsigned)bin;
            s.k = kk;
            if (PASS == 3) {
                s.run = run;
                s.need_hi = s.cnt[0] + s.cnt[1] >= 2 && (unsigned long long)kk + 1 >= run;
            }
        }
    }
}

// out [4][n]: hd (as hd_finish_kernel), hd95, asd = mean of side 1's queries (pred border -> label border), assd
__global__ void sd_finish_kernel(const unsigned* __restrict__ rowmax, const unsigned* __restrict__ present,
                                 const SdState* __restrict__ st, int64_t n, float* __restrict__ out) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        const bool both = present[2 * j] != 0u && present[2 * j + 1] != 0u;
        float hd95 = CUDART_NAN_F, asd = CUDART_NAN_F, assd = CUDART_NAN_F;
        if (both) {   // both border sets exist, so both sides have queries
            const SdState& s = st[j];
            long long lo;
            const double t = sd_rank95(s.cnt[0] + s.cnt[1], &lo);
            const double a = sqrt((double)__uint_as_float(s.prefix));
            const double b = s.need_hi ? sqrt((double)__uint_as_float(s.hikey)) : a;
            const double d = b - a;
            hd95 = (float)(t >= 0.5 ? b - d * (1.0 - t) : a + d * t);   // numpy's _lerp
            const double m1 = s.sum[1] / (double)s.cnt[1], m0 = s.sum[0] / (double)s.cnt[0];
            asd = (float)m1;
            assd = (float)((m1 + m0) / 2.0);
        }
        out[j] = hd_value(rowmax, present, j);
        out[n + j] = hd95;
        out[2 * n + j] = asd;
        out[3 * n + j] = assd;
    }
}

template <bool FROM_G, bool FOLD, bool SURF = false>
cudaError_t launch_envelope(const EnvArgs& a, cudaStream_t s) {
    const int64_t lines = 2 * a.g.C * a.lines_per_plane;
    int R = kEnvSmemBudget / (4 * a.n);
    R = R > 64 ? 64 : (R < 1 ? 1 : R);
    const size_t smem = (size_t)R * a.n * 4;
    if (smem > (size_t)kEnvSmemBudget) {
        cudaError_t e = cudaFuncSetAttribute(hd_envelope_kernel<FROM_G, FOLD, SURF>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    hd_envelope_kernel<FROM_G, FOLD, SURF><<<(unsigned)((lines + R - 1) / R), R, smem, s>>>(a);
    return cudaGetLastError();
}

// argument checks of both entry points; fills the spacing (sz, sy, sx)
inline int hd_check_args(const int64_t* pred, const int64_t* labels, int C, int64_t B, int64_t H, int64_t W, int volume,
                         const double* spacing, const void* out, const int32_t* flags, const void* scratch, double sp[3]) {
    if (pred == nullptr || labels == nullptr || out == nullptr || scratch == nullptr) return DCT_ERR_BAD_ARG;
    if (C < 1 || B < 1 || H < 1 || W < 1) return DCT_ERR_BAD_ARG;
    if (!hd_supported(C, B, H, W, volume)) return DCT_ERR_UNSUPPORTED;
    sp[0] = sp[1] = sp[2] = 1.0;
    if (spacing != nullptr) {
        for (int i = 0; i < (volume ? 3 : 2); ++i) {
            const double v = spacing[i];
            if (!(v > 0.0) || !std::isfinite(v)) return DCT_ERR_BAD_ARG;   // also rejects NaN
            sp[volume ? i : i + 1] = v;
        }
    }
    if (!aligned(pred, 8) || !aligned(labels, 8) || !aligned(out, 4) || !aligned(flags, 4) || !aligned(scratch, 256))
        return DCT_ERR_MISALIGNED;
    return DCT_OK;
}

// classify, column and envelope passes (3 launches for '2d', 4 for a volume): leave the per-(row, class, side) maxima
// and presence words in the scratch header and, with SURF, every query's d^2 and the last pass's per-line slots
template <bool SURF>
cudaError_t hd_distance_passes(const int64_t* pred, const int64_t* labels, const HdGeom& g, const double sp[3],
                               const HdLayout& L, char* base, int32_t* flags, cudaStream_t s) {
    const int64_t B = g.B, H = g.H, W = g.W, nrc = (g.volume ? 1 : B) * g.C;
    unsigned* rowmax = reinterpret_cast<unsigned*>(base + L.hdr);
    unsigned* present = rowmax + 2 * nrc;
    uint16_t* rec = reinterpret_cast<uint16_t*>(base + L.rec);
    uint16_t* gdist = reinterpret_cast<uint16_t*>(base + L.g);
    float* f = reinterpret_cast<float*>(base + L.f);

    const int64_t cls_blocks = std::min<int64_t>((g.N + 255) / 256, (int64_t)kSMs * 16);
    hd_classify_kernel<<<(unsigned)cls_blocks, 256, 0, s>>>(pred, labels, g, rec, rowmax, (int)(4 * nrc), flags);
    const int64_t col_lines = 2 * (int64_t)g.C * B * W;
    hd_column_kernel<<<(unsigned)((col_lines + 127) / 128), 128, 0, s>>>(rec, g, gdist, present);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;

    EnvArgs a{};
    a.gdist = gdist; a.rec = rec; a.rowmax = rowmax; a.g = g;
    a.lines_per_plane = B * H; a.line_step = W; a.stride = 1; a.n = (int)W;
    a.w_in = sp[1] * sp[1]; a.w = sp[2] * sp[2];
    if (SURF) {
        a.qd = reinterpret_cast<float*>(base + L.qd);
        a.lsum = reinterpret_cast<double*>(base + L.lsum);
        a.lcnt = reinterpret_cast<unsigned*>(base + L.lcnt);
    }
    if (!g.volume) {
        a.lines_per_row = H;   // line l = b * H + y lies in image b
        return launch_envelope<true, true, SURF>(a, s);
    }
    a.fout = f;
    e = launch_envelope<true, false>(a, s);
    EnvArgs z = a;
    z.gdist = nullptr; z.fout = nullptr; z.fin = f;
    z.lines_per_plane = H * W; z.line_step = 1; z.stride = H * W; z.n = (int)B;
    z.lines_per_row = H * W;   // one row: the volume
    z.w_in = 0.0; z.w = sp[0] * sp[0];
    if (e == cudaSuccess) e = launch_envelope<false, true, SURF>(z, s);
    return e;
}

// a task per `chunk` pixels of one row, about 4 per SM, no fewer pixels than the per-task histogram has bins
inline SdTasks sd_tasks(const HdGeom& g) {
    SdTasks t;
    const int64_t rows = g.volume ? 1 : g.B;
    t.rowpix = g.volume ? g.N : g.H * g.W;
    int64_t chunk = std::max<int64_t>((g.N + kSMs * 4 - 1) / (kSMs * 4), (int64_t)g.C * 256);
    chunk = std::min<int64_t>((chunk + 255) & ~(int64_t)255, (int64_t)1 << 30);   // per-task counts stay in uint32
    t.chunk = std::min(chunk, t.rowpix);
    t.chunks_per_row = (t.rowpix + t.chunk - 1) / t.chunk;
    t.tasks = rows * t.chunks_per_row;
    return t;
}

template <int PASS>
cudaError_t launch_select(const uint16_t* rec, const float* qd, const HdGeom& g, const SdTasks& tk,
                          unsigned long long* hist, SdState* st, cudaStream_t s) {
    const size_t smem = ((PASS == 4 ? (size_t)g.C : (size_t)g.C * 256) + 2 * (size_t)g.C) * 4;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(sd_select_kernel<PASS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem);
        if (e != cudaSuccess) return e;
    }
    sd_select_kernel<PASS><<<(unsigned)std::min<int64_t>(tk.tasks, (int64_t)kSMs * 8), 256, smem, s>>>(rec, qd, g, tk,
                                                                                                     hist, st);
    return cudaGetLastError();
}

template <int PASS>
cudaError_t launch_pick(unsigned long long* hist, SdState* st, int64_t nrc, cudaStream_t s) {
    sd_pick_kernel<PASS><<<(unsigned)std::min<int64_t>((nrc + 7) / 8, (int64_t)kSMs * 16), 256, 0, s>>>(hist, st, nrc);
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
    double sp[3];
    const int rc = hd_check_args(pred, labels, C, B, H, W, volume, spacing, hd, flags, scratch, sp);
    if (rc != DCT_OK) return rc;
    const HdGeom g{C, B, H, W, B * H * W, volume ? 1 : 0};
    const HdLayout L = hd_layout(C, B, H, W, volume);
    char* base = static_cast<char*>(scratch);
    const unsigned* rowmax = reinterpret_cast<const unsigned*>(base + L.hdr);
    const int64_t nrc = (volume ? 1 : B) * C;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaError_t e = hd_distance_passes<false>(pred, labels, g, sp, L, base, flags, s);
    if (e == cudaSuccess) {
        hd_finish_kernel<<<(unsigned)std::min<int64_t>((nrc + 127) / 128, 1024), 128, 0, s>>>(rowmax, rowmax + 2 * nrc,
                                                                                               nrc, hd);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return DCT_OK;
}

extern "C" size_t dct_surface_distance_scratch_bytes(int C, int64_t B, int64_t H, int64_t W, int volume) {
    if (C < 1 || B < 1 || H < 1 || W < 1 || !hd_supported(C, B, H, W, volume)) return 0;
    return hd_layout(C, B, H, W, volume).surf_total;
}

extern "C" int dct_surface_distances_i64(const int64_t* pred, const int64_t* labels, int C, int64_t B, int64_t H,
                                         int64_t W, int volume, const double* spacing, float* out, int32_t* flags,
                                         void* scratch, void* stream) {
    double sp[3];
    const int rc = hd_check_args(pred, labels, C, B, H, W, volume, spacing, out, flags, scratch, sp);
    if (rc != DCT_OK) return rc;
    const HdGeom g{C, B, H, W, B * H * W, volume ? 1 : 0};
    const HdLayout L = hd_layout(C, B, H, W, volume);
    char* base = static_cast<char*>(scratch);
    const unsigned* rowmax = reinterpret_cast<const unsigned*>(base + L.hdr);
    const uint16_t* rec = reinterpret_cast<const uint16_t*>(base + L.rec);
    const float* qd = reinterpret_cast<const float*>(base + L.qd);
    unsigned long long* hist = reinterpret_cast<unsigned long long*>(base + L.hist);
    SdState* st = reinterpret_cast<SdState*>(base + L.st);
    const int64_t nrc = (volume ? 1 : B) * C;
    cudaStream_t s = static_cast<cudaStream_t>(stream);

    cudaError_t e = hd_distance_passes<true>(pred, labels, g, sp, L, base, flags, s);
    if (e == cudaSuccess) {
        const int64_t lines_per_plane = volume ? H * W : B * H, lines_per_row = volume ? H * W : H;
        sd_sum_kernel<<<(unsigned)std::min<int64_t>(nrc, (int64_t)kSMs * 8), kSumThreads, 0, s>>>(
            reinterpret_cast<const double*>(base + L.lsum), reinterpret_cast<const unsigned*>(base + L.lcnt), g,
            lines_per_plane, lines_per_row, nrc, st, hist);
        e = cudaGetLastError();
    }
    const SdTasks tk = sd_tasks(g);
    if (e == cudaSuccess) e = launch_select<0>(rec, qd, g, tk, hist, st, s);
    if (e == cudaSuccess) e = launch_pick<0>(hist, st, nrc, s);
    if (e == cudaSuccess) e = launch_select<1>(rec, qd, g, tk, hist, st, s);
    if (e == cudaSuccess) e = launch_pick<1>(hist, st, nrc, s);
    if (e == cudaSuccess) e = launch_select<2>(rec, qd, g, tk, hist, st, s);
    if (e == cudaSuccess) e = launch_pick<2>(hist, st, nrc, s);
    if (e == cudaSuccess) e = launch_select<3>(rec, qd, g, tk, hist, st, s);
    if (e == cudaSuccess) e = launch_pick<3>(hist, st, nrc, s);
    if (e == cudaSuccess) e = launch_select<4>(rec, qd, g, tk, hist, st, s);
    if (e == cudaSuccess) {
        sd_finish_kernel<<<(unsigned)std::min<int64_t>((nrc + 127) / 128, 1024), 128, 0, s>>>(rowmax, rowmax + 2 * nrc,
                                                                                              st, nrc, out);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return DCT_OK;
}
