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
//                        shared memory.  Along W it either writes the d^2 map (volume) or is the last pass; along B
//                        (volume) it is the last pass.  The last pass folds max over the other side's border pixels of d^2
//                        into the (row, class, side) maximum with an integer atomicMax on the d^2 key (d2_key):
//                        order-independent, so bit-reproducible.
//   hd_finish_kernel     HD = square root of the max of the two sides, NaN where a side's set is empty.
// Launches: 4 for '2d', 5 for a volume.  Envelope arithmetic is double.  Every d^2 that leaves a pass is a 32-bit key that
// orders like the value: at unit spacing the exact integer (3 * 32767^2 < 2^32), otherwise the bits of the float d^2.  So
// at unit spacing the result is the correctly rounded square root of the exact squared distance for every accepted shape
// (a float d^2 would be rounded from 4096 pixels of distance on).
//
// dct_surface_distances_i64 (HD95, ASD, ASSD; medpy.metric.binary hd95 / asd / assd) runs the same passes with the last
// one in its SURF mode, which also keeps every query's d^2 and per-line sums, then:
//   sd_sum_kernel        fixed-order reduction of the per-line sums and counts per (row, class, side); rank to select.
//   sd_select_kernel<P>  P = 0..3: radix histogram of 8 key bits under the selected prefix; P = 4: least key above it.
//   sd_pick_kernel<P>    narrows prefix and rank from the histogram of pass P.
//   sd_finish_kernel     hd, hd95, asd, assd.
// Launches: 14 for '2d', 15 for a volume.
//
// dct_surface_dice_i64 (normalized surface Dice at tolerance tol[c]) runs the same passes with the last one in its TOL
// mode, which only counts per line the queries and the queries with sqrt((double)d^2) <= tol[c], then:
//   nsd_finish_kernel    per (row, class): 64-bit sums of both sides' line counts; nsd, overlap_pg, overlap_gp, counts.
// Launches: 4 for '2d', 5 for a volume.
//
// dct_distance_map_i64 (signed / inside Euclidean distance maps of one class map, scipy's EDT semantics: cells off the
// grid are not features) runs the same transform on the sets {map != c} and, for signed maps, {map == c}:
//   dm_classify_kernel   one class byte per pixel; zeroes the presence words.
//   dm_column_kernel     hd_column_kernel with those feature sets.
//   hd_envelope_kernel   as above; the last pass in its MAP mode writes each query's distance into the float map.
// Launches: 3 for '2d', 4 for a volume.
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
constexpr unsigned kInfKey = 0xFFFFFFFFu;         // d2_key of +inf at unit spacing

struct HdGeom {
    int C;
    int64_t B, H, W, N;   // N = B*H*W
    int volume;
    int exact;            // unit spacing: d^2 keys are the exact integers
};

// d^2 as a 32-bit key that orders like the value (maxima by integer atomicMax, percentiles by a radix select on the key):
// at unit spacing (exact) the integer d^2 itself, which fits since every axis is at most 32768 long, with kInfKey for
// +inf; otherwise the bits of the float d^2 (non-negative floats order like their bits)
__device__ __forceinline__ unsigned d2_key(double d2, bool exact) {
    if (exact) return isinf(d2) ? kInfKey : (unsigned)d2;
    return __float_as_uint((float)d2);
}
__device__ __forceinline__ double d2_value(unsigned key, bool exact) {
    if (exact) return key == kInfKey ? CUDART_INF : (double)key;
    return (double)__uint_as_float(key);
}

// shapes the kernels take: axes within the 16-bit stack entries, every grid within 2^31 - 1 threads (B is bounded
// first so that the line count cannot overflow int64)
inline bool hd_supported(int C, int64_t B, int64_t H, int64_t W, int volume) {
    if (C > DCT_MAX_CLASSES || H > kHdMaxAxis || W > kHdMaxAxis || B > (volume ? kHdMaxAxis : INT_MAX)) return false;
    const int64_t lines = 2 * (int64_t)C * B * std::max(H, W);   // column and row passes
    return lines <= INT_MAX && (!volume || 2 * (int64_t)C * H * W <= INT_MAX);
}

inline size_t hd_align256(size_t v) { return (v + 255) & ~(size_t)255; }

struct HdLayout {
    size_t hdr, rec, g, f, total;              // dct_hausdorff_i64
    size_t qd, lsum, lcnt, hist, st, surf_total;   // dct_surface_distances_i64: the same, then these
    size_t tq, tw, dice_total;                 // dct_surface_dice_i64: the Hausdorff scratch, then these
};
constexpr size_t kSdStateBytes = 64;   // sizeof(SdState)
inline HdLayout hd_layout(int C, int64_t B, int64_t H, int64_t W, int volume) {
    const size_t N = (size_t)B * H * W, rows = volume ? 1 : (size_t)B;
    const size_t fold_lines = 2 * (size_t)C * (volume ? (size_t)H * W : (size_t)B * H);   // lines of the last pass
    HdLayout L;
    L.hdr = 0;                                          // uint32 rowmax[rows][C][2], present[rows][C][2]
    L.rec = hd_align256(L.hdr + rows * C * 2 * 2 * 4);     // uint16 [N]: pred byte | gt byte << 8
    L.g = hd_align256(L.rec + N * 2);                      // uint16 [2][C][N]
    L.f = hd_align256(L.g + 2 * (size_t)C * N * 2);        // uint32 [2][C][N] d^2 keys (volume only)
    L.total = volume ? hd_align256(L.f + 2 * (size_t)C * N * 4) : L.f;
    L.qd = L.total;                                        // uint32 [2][N] d^2 keys
    L.lsum = hd_align256(L.qd + 2 * N * 4);                // double [fold_lines]
    L.lcnt = hd_align256(L.lsum + fold_lines * 8);         // uint32 [fold_lines]
    L.hist = hd_align256(L.lcnt + fold_lines * 4);         // uint64 [rows][C][256]
    L.st = hd_align256(L.hist + rows * C * 256 * 8);       // SdState [rows][C]
    L.surf_total = hd_align256(L.st + rows * C * kSdStateBytes);
    L.tq = L.total;                                        // uint32 [fold_lines] queries
    L.tw = hd_align256(L.tq + fold_lines * 4);             // uint32 [fold_lines] queries within the tolerance
    L.dice_total = hd_align256(L.tw + fold_lines * 4);
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

// ---- distance maps (dct_distance_map_i64): classify and column passes of one class map --------------------------------
//
// g.C counts the computed classes first_class .. first_class + g.C - 1; `sides` feature sets per class: side 0's
// features are out_c = {byte != c} (the inside distances), side 1's, in signed mode only, in_c = {byte == c}.

// scratch: uint32 present[rows][Cc][2], uint8 class byte [N], uint16 column distances [sides][Cc][N], and for a volume
// uint32 d^2 keys [sides][Cc][N] after the row pass
struct DmLayout {
    size_t cls, g, f, total;
};
inline DmLayout dm_layout(int Cc, int64_t B, int64_t H, int64_t W, int volume, int sides) {
    const size_t N = (size_t)B * H * W, rows = volume ? 1 : (size_t)B, sets = (size_t)sides * Cc;
    DmLayout L;
    L.cls = hd_align256(rows * Cc * 2 * 4);
    L.g = hd_align256(L.cls + N);
    L.f = hd_align256(L.g + sets * N * 2);
    L.total = volume ? hd_align256(L.f + sets * N * 4) : L.f;
    return L;
}

// one class byte per pixel (kOutOfRange for a value outside [0,C), counted in flags[DCT_FLAG_PRED]); zeroes the
// presence words
__global__ void __launch_bounds__(256) dm_classify_kernel(const int64_t* __restrict__ map, int64_t N, int C,
                                                          unsigned char* __restrict__ cls, unsigned* present, int npres,
                                                          int32_t* flags) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = tid; i < npres; i += nthr) present[i] = 0u;
    int bad = 0;
    for (int64_t p = tid; p < N; p += nthr) {
        const long long v = map[p];
        const bool in = v >= 0 && v < C;
        bad += !in;
        cls[p] = in ? (unsigned char)v : kOutOfRange;
    }
    if (flags != nullptr) {
        bad = __reduce_add_sync(0xffffffffu, bad);
        if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&flags[DCT_FLAG_PRED], bad);
    }
}

// hd_column_kernel with the map's feature sets: one thread per (side, class, image, column)
__global__ void __launch_bounds__(128) dm_column_kernel(const unsigned char* __restrict__ cls, const HdGeom g, int sides,
                                                        int first_class, uint16_t* __restrict__ gdist,
                                                        unsigned* present) {
    const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t per_sc = g.B * g.W;
    if (line >= sides * g.C * per_sc) return;
    const int sc = (int)(line / per_sc), side = sc / g.C, c = sc - side * g.C;
    const int64_t r = line - sc * per_sc, b = r / g.W, x = r - b * g.W;
    const int64_t base = b * g.H * g.W + x;
    const unsigned char want = (unsigned char)(first_class + c);
    const bool feat_in = side == 1;   // side 1: features in_c; side 0: out_c
    const unsigned char* in = cls + base;
    uint16_t* out = gdist + (int64_t)sc * g.N + base;
    int last = -1;
    for (int y = 0; y < g.H; ++y) {
        if ((in[(int64_t)y * g.W] == want) == feat_in) last = y;
        out[(int64_t)y * g.W] = last < 0 ? kNone : (uint16_t)(y - last);
    }
    if (last < 0) return;   // no feature in this column
    present[((g.volume ? 0 : b) * g.C + c) * 2 + side] = 1u;
    int next = -1;
    for (int y = (int)g.H - 1; y >= 0; --y) {
        const int64_t o = (int64_t)y * g.W;
        if ((in[o] == want) == feat_in) next = y;
        if (next >= 0) {
            const uint16_t d = (uint16_t)(next - y);
            if (d < out[o]) out[o] = d;
        }
    }
}

struct EnvArgs {
    const uint16_t* gdist;   // FROM_G: input distances in rows (weight w_in)
    const unsigned* fin;     // !FROM_G: input d^2 keys
    unsigned* fout;          // !FOLD: output d^2 keys
    const uint16_t* rec;     // FOLD: border records of the queries
    unsigned* rowmax;        // FOLD: [rows][C][2] d^2 keys
    HdGeom g;
    int64_t lines_per_plane, line_step, stride, lines_per_row;
    int n;
    double w_in, w;          // squared spacing of the previous axis (FROM_G) and of this one
    unsigned* qd;            // SURF: [2][N] d^2 key of each query pixel to the border set of that side
    double* lsum;            // SURF: per line of the last pass, sum of sqrt(d^2) over its queries
    unsigned* lcnt;          // SURF, TOL: per line of the last pass, number of its queries
};

// TOL (last pass of dct_surface_dice_i64): the tolerances travel by value in the kernel arguments (no copy, graph-safe);
// only this mode's instantiations take the larger argument block
struct EnvTolArgs : EnvArgs {
    unsigned* lwin;                  // per line of the last pass, number of its queries within tol[c]
    double tol[DCT_MAX_CLASSES];     // per class, in spacing units
};
// MAP (dct_distance_map_i64): g.C counts the computed classes first_class .. first_class + g.C - 1, and only `sides`
// feature sets per class exist (1: the inside distances alone); the last pass writes the map itself
struct EnvMapArgs : EnvArgs {
    const unsigned char* cls;   // class byte per pixel (kOutOfRange outside [0,C))
    const unsigned* present;    // [rows][g.C][2]: the column pass found a feature of that side
    float* out;                 // [B][g.C][H][W]
    int64_t HW, ostride;        // out index of pixel base + x * stride: base + (row * (g.C - 1) + c) * HW + x * ostride
    int sides, first_class;
};
template <bool TOL, bool MAP = false>
using EnvParams = std::conditional_t<TOL, EnvTolArgs, std::conditional_t<MAP, EnvMapArgs, EnvArgs>>;

// lines of one envelope pass: one per (side, class, line of a plane)
template <bool MAP>
__host__ __device__ __forceinline__ int64_t env_lines(const EnvParams<false, MAP>& a) {
    if constexpr (MAP) return (int64_t)a.sides * a.g.C * a.lines_per_plane;
    else return 2 * a.g.C * a.lines_per_plane;
}

template <bool FROM_G>
__device__ __forceinline__ double env_load(const EnvArgs& a, int64_t plane, int64_t off) {
    if constexpr (FROM_G) {
        const uint16_t d = a.gdist[plane + off];
        return d == kNone ? CUDART_INF : a.w_in * (double)d * (double)d;
    } else {
        return d2_value(a.fin[plane + off], a.g.exact);
    }
}

// MAP, last pass: the values of one line of class c's plane of the map, from the line's envelope (stack entries
// stk[k * R], k <= top).  Side 0's features are out_c and its queries in_c: it writes -d (signed) or d (unsigned), and in
// unsigned mode also the 0 of every other position.  Side 1's features are in_c and its queries out_c: it writes +d.
// So every element of the plane is written by exactly one thread.  A signed plane is 0 where either feature set is
// empty on the grid; an unsigned query with no out_c on the grid gets +inf, the d of the empty envelope.
template <bool FROM_G>
__device__ __forceinline__ void env_write_map(const EnvMapArgs& a, const unsigned* stk, int R, int top, int64_t plane,
                                              int64_t base, int side, int c, int64_t l) {
    const int64_t row = l / a.lines_per_row;
    const bool is_signed = a.sides == 2;
    const unsigned* pr = a.present + (row * a.g.C + c) * 2;
    const bool empty = is_signed && (pr[0] == 0u || pr[1] == 0u);
    const unsigned cls = (unsigned)(a.first_class + c);
    float* out = a.out + base + (row * (a.g.C - 1) + c) * a.HW;
    const int n = a.n;
    const int64_t stride = a.stride, ostride = a.ostride;
    const double w = a.w;
    int k = 0;
    for (int x = 0; x < n; ++x) {
        const bool inside = a.cls[base + x * stride] == cls;
        float v = 0.0f;
        if (inside == (side == 0)) {   // a query of this side
            if (!empty) {
                while (k < top && (int)(stk[(k + 1) * R] >> 16) <= x) ++k;
                double d2 = CUDART_INF;
                if (top >= 0) {
                    const int q = (int)(stk[k * R] & 0xFFFFu);
                    d2 = env_load<FROM_G>(a, plane, base + q * stride) + w * (double)(x - q) * (double)(x - q);
                }
                v = (float)sqrt(d2);
                if (is_signed && side == 0) v = -v;
            }
        } else if (is_signed) {
            continue;   // the other side's line writes this position
        }
        out[x * ostride] = v;
    }
}

// Lower envelope of {f(q) + w (x - q)^2} over the finite f(q) of one line, evaluated at the integer positions x of the
// line.  Stack entry k = (position v_k, first integer position z_k at which parabola v_k is the lowest); a new parabola q
// (to the right of every stacked one) is at or below v_k from ceil(sep) on, so v_k is popped when ceil(sep) <= z_k and q is
// only pushed when ceil(sep) < n.  SURF (last pass of dct_surface_distances_i64): also keep every query's d^2 and the
// line's sum of distances and query count.  TOL (last pass of dct_surface_dice_i64): instead of the maximum, only the
// line's query count and the number of its queries with sqrt((double)d^2) <= tol[c].  MAP (dct_distance_map_i64): the
// line count follows a.sides and, in the last pass, env_write_map writes the line's values of the map.
template <bool FROM_G, bool FOLD, bool SURF = false, bool TOL = false, bool MAP = false>
__global__ void __launch_bounds__(64) hd_envelope_kernel(const EnvParams<TOL, MAP> a) {
    static_assert(FOLD || !(SURF || TOL), "only the last pass has queries");
    static_assert(!(SURF && TOL), "one query mode per pass");
    static_assert(!(MAP && (SURF || TOL)), "the map is its own query mode");
    extern __shared__ unsigned stk_all[];
    const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= env_lines<MAP>(a)) return;
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
    if constexpr (MAP && FOLD) {
        env_write_map<FROM_G>(a, stk, R, top, plane, base, side, c, l);
        return;
    }
    const unsigned want = (unsigned)c | 0x80u;
    const bool exact = a.g.exact;
    unsigned m = 0u;
    bool any = false;
    double dsum = 0.0;
    unsigned cnt = 0, win = 0;
    double tol = 0.0;
    if constexpr (TOL) tol = a.tol[c];
    int k = 0;
    for (int x = 0; x < n; ++x) {
        const int64_t off = base + x * stride;
        if constexpr (FOLD) {
            if (side_byte(a.rec[off], 1 - side) != want) continue;   // queries: the other side's border pixels of c
        }
        double d2 = CUDART_INF;
        if (top >= 0) {
            while (k < top && (int)(stk[(k + 1) * R] >> 16) <= x) ++k;
            const int v = (int)(stk[k * R] & 0xFFFFu);
            d2 = env_load<FROM_G>(a, plane, base + v * stride) + w * (double)(x - v) * (double)(x - v);
        }
        const unsigned key = d2_key(d2, exact);
        if constexpr (FOLD) { m = max(m, key); any = true; }
        else a.fout[plane + off] = key;
        if constexpr (SURF || TOL) d2 = d2_value(key, exact);   // the d^2 the maxima and keys hold
        if constexpr (SURF) {
            a.qd[side * a.g.N + off] = key;   // a pixel is a query of one class per side: no other line writes here
            dsum += sqrt(d2);
            ++cnt;
        }
        if constexpr (TOL) {
            ++cnt;
            if (sqrt(d2) <= tol) ++win;   // d2 = +inf (no border on this side) is never within
        }
    }
    if constexpr (FOLD && !TOL) {
        if (any) {
            const int64_t row = l / a.lines_per_row;
            atomicMax(&a.rowmax[(row * a.g.C + c) * 2 + side], m);
        }
    }
    if constexpr (SURF) { a.lsum[line] = dsum; a.lcnt[line] = cnt; }
    if constexpr (TOL) { a.lcnt[line] = cnt; a.lwin[line] = win; }
}

// the square root of the larger side's maximum, correctly rounded: at unit spacing of the exact integer d^2 (the double
// square root rounded to float is the correctly rounded float square root, as 53 >= 2 * 24 + 2)
__device__ __forceinline__ float hd_value(const unsigned* __restrict__ rowmax, const unsigned* __restrict__ present,
                                          int64_t j, bool exact) {
    const bool both = present[2 * j] != 0u && present[2 * j + 1] != 0u;
    const unsigned key = max(rowmax[2 * j], rowmax[2 * j + 1]);
    if (!both) return CUDART_NAN_F;
    return exact ? (float)sqrt((double)key) : __fsqrt_rn(__uint_as_float(key));
}

__global__ void hd_finish_kernel(const unsigned* __restrict__ rowmax, const unsigned* __restrict__ present, int64_t n,
                                 int exact, float* __restrict__ hd) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x)
        hd[j] = hd_value(rowmax, present, j, exact);
}

// ---- surface distances (dct_surface_distances_i64): HD95, ASD, ASSD from the last pass's per-query d^2 -------------
//
// Per (row, class) the keys are the d2_key of the d^2 of both sides' queries.  HD95 is numpy's 'linear' percentile of the distances: with n keys, v = (n - 1) * 0.95, lo = floor(v), the
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
__global__ void __launch_bounds__(256) sd_select_kernel(const uint16_t* __restrict__ rec, const unsigned* __restrict__ qd,
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
                    key = qd[s * g.N + p];
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
                                 const SdState* __restrict__ st, int64_t n, int exact, float* __restrict__ out) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        const bool both = present[2 * j] != 0u && present[2 * j + 1] != 0u;
        float hd95 = CUDART_NAN_F, asd = CUDART_NAN_F, assd = CUDART_NAN_F;
        if (both) {   // both border sets exist, so both sides have queries
            const SdState& s = st[j];
            long long lo;
            const double t = sd_rank95(s.cnt[0] + s.cnt[1], &lo);
            const double a = sqrt(d2_value(s.prefix, exact));
            const double b = s.need_hi ? sqrt(d2_value(s.hikey, exact)) : a;
            const double d = b - a;
            hd95 = (float)(t >= 0.5 ? b - d * (1.0 - t) : a + d * t);   // numpy's _lerp
            const double m1 = s.sum[1] / (double)s.cnt[1], m0 = s.sum[0] / (double)s.cnt[0];
            asd = (float)m1;
            assd = (float)((m1 + m0) / 2.0);
        }
        out[j] = hd_value(rowmax, present, j, exact);
        out[n + j] = hd95;
        out[2 * n + j] = asd;
        out[3 * n + j] = assd;
    }
}

// ---- normalized surface Dice (dct_surface_dice_i64): counts of the TOL last pass -------------------------------------

// one CTA per (row, class): 64-bit sums of both sides' per-line query and within-tolerance counts (integers: the order
// does not matter), then nsd = (W_pg + W_gp) / (|S_pg| + |S_gp|), overlap_pg = W_pg / |S_pg|, overlap_gp = W_gp / |S_gp|
// as double ratios rounded once to float (NaN for a zero denominator).  Side 1's queries are the prediction's border
// pixels (S_pg), side 0's the label's (S_gp).  out [3][nrc]; counts (nullable) [nrc][4] = W_pg, |S_pg|, W_gp, |S_gp|.
constexpr int kNsdThreads = 256;
__global__ void __launch_bounds__(kNsdThreads) nsd_finish_kernel(const unsigned* __restrict__ lq,
                                                                 const unsigned* __restrict__ lw, int C,
                                                                 int64_t lines_per_plane, int64_t lines_per_row,
                                                                 int64_t nrc, float* __restrict__ out,
                                                                 long long* __restrict__ counts) {
    __shared__ unsigned long long part[kNsdThreads / 32][4];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int64_t rc = blockIdx.x; rc < nrc; rc += gridDim.x) {
        const int64_t row = rc / C;
        const int c = (int)(rc - row * C);
        unsigned long long v[4] = {0ull, 0ull, 0ull, 0ull};   // W_pg, |S_pg|, W_gp, |S_gp|
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            const int64_t base = (int64_t)(side * C + c) * lines_per_plane + row * lines_per_row;
            const int slot = side ? 0 : 2;
            for (int64_t j = t; j < lines_per_row; j += kNsdThreads) {
                v[slot] += lw[base + j];
                v[slot + 1] += lq[base + j];
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            for (int o = 16; o > 0; o >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
            if (lane == 0) part[warp][i] = v[i];
        }
        __syncthreads();
        if (t == 0) {
            unsigned long long s[4] = {0ull, 0ull, 0ull, 0ull};
            for (int w = 0; w < kNsdThreads / 32; ++w)
                for (int i = 0; i < 4; ++i) s[i] += part[w][i];
            const unsigned long long n = s[1] + s[3];
            out[rc] = n ? (float)((double)(s[0] + s[2]) / (double)n) : CUDART_NAN_F;
            out[nrc + rc] = s[1] ? (float)((double)s[0] / (double)s[1]) : CUDART_NAN_F;
            out[2 * nrc + rc] = s[3] ? (float)((double)s[2] / (double)s[3]) : CUDART_NAN_F;
            if (counts != nullptr)
                for (int i = 0; i < 4; ++i) counts[rc * 4 + i] = (long long)s[i];
        }
        __syncthreads();   // part[] is reused by the next (row, class)
    }
}

template <bool FROM_G, bool FOLD, bool SURF = false, bool TOL = false, bool MAP = false>
cudaError_t launch_envelope(const EnvParams<TOL, MAP>& a, cudaStream_t s) {
    const int64_t lines = env_lines<MAP>(a);
    int R = kEnvSmemBudget / (4 * a.n);
    R = R > 64 ? 64 : (R < 1 ? 1 : R);
    const size_t smem = (size_t)R * a.n * 4;
    if (smem > (size_t)kEnvSmemBudget) {
        cudaError_t e = cudaFuncSetAttribute(hd_envelope_kernel<FROM_G, FOLD, SURF, TOL, MAP>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    hd_envelope_kernel<FROM_G, FOLD, SURF, TOL, MAP><<<(unsigned)((lines + R - 1) / R), R, smem, s>>>(a);
    return cudaGetLastError();
}

// the last envelope pass of one entry point: plain (Hausdorff), SURF, or TOL with the per-class tolerances
template <bool FROM_G, bool SURF, bool TOL>
cudaError_t launch_last_pass(const EnvArgs& a, const double* tol, const HdLayout& L, char* base, cudaStream_t s) {
    if constexpr (TOL) {
        EnvTolArgs t{};
        static_cast<EnvArgs&>(t) = a;
        t.lcnt = reinterpret_cast<unsigned*>(base + L.tq);
        t.lwin = reinterpret_cast<unsigned*>(base + L.tw);
        for (int c = 0; c < a.g.C; ++c) t.tol[c] = tol[c];
        return launch_envelope<FROM_G, true, false, true>(t, s);
    } else {
        return launch_envelope<FROM_G, true, SURF>(a, s);
    }
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

inline HdGeom hd_geom(int C, int64_t B, int64_t H, int64_t W, int volume, const double sp[3]) {
    return HdGeom{C, B, H, W, B * H * W, volume ? 1 : 0, sp[0] == 1.0 && sp[1] == 1.0 && sp[2] == 1.0};
}

// classify, column and envelope passes (3 launches for '2d', 4 for a volume): leave the per-(row, class, side) maxima
// and presence words in the scratch header and, with SURF, every query's d^2 and the last pass's per-line slots; with
// TOL (tolerances `tol`, C host values) only the last pass's per-line query and within-tolerance counts
template <bool SURF, bool TOL = false>
cudaError_t hd_distance_passes(const int64_t* pred, const int64_t* labels, const HdGeom& g, const double sp[3],
                               const HdLayout& L, char* base, int32_t* flags, cudaStream_t s,
                               const double* tol = nullptr) {
    const int64_t B = g.B, H = g.H, W = g.W, nrc = (g.volume ? 1 : B) * g.C;
    unsigned* rowmax = reinterpret_cast<unsigned*>(base + L.hdr);
    unsigned* present = rowmax + 2 * nrc;
    uint16_t* rec = reinterpret_cast<uint16_t*>(base + L.rec);
    uint16_t* gdist = reinterpret_cast<uint16_t*>(base + L.g);
    unsigned* f = reinterpret_cast<unsigned*>(base + L.f);

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
        a.qd = reinterpret_cast<unsigned*>(base + L.qd);
        a.lsum = reinterpret_cast<double*>(base + L.lsum);
        a.lcnt = reinterpret_cast<unsigned*>(base + L.lcnt);
    }
    if (!g.volume) {
        a.lines_per_row = H;   // line l = b * H + y lies in image b
        return launch_last_pass<true, SURF, TOL>(a, tol, L, base, s);
    }
    a.fout = f;
    e = launch_envelope<true, false>(a, s);
    EnvArgs z = a;
    z.gdist = nullptr; z.fout = nullptr; z.fin = f;
    z.lines_per_plane = H * W; z.line_step = 1; z.stride = H * W; z.n = (int)B;
    z.lines_per_row = H * W;   // one row: the volume
    z.w_in = 0.0; z.w = sp[0] * sp[0];
    if (e == cudaSuccess) e = launch_last_pass<false, SURF, TOL>(z, tol, L, base, s);
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
cudaError_t launch_select(const uint16_t* rec, const unsigned* qd, const HdGeom& g, const SdTasks& tk,
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
    const HdGeom g = hd_geom(C, B, H, W, volume, sp);
    const HdLayout L = hd_layout(C, B, H, W, volume);
    char* base = static_cast<char*>(scratch);
    const unsigned* rowmax = reinterpret_cast<const unsigned*>(base + L.hdr);
    const int64_t nrc = (volume ? 1 : B) * C;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaError_t e = hd_distance_passes<false>(pred, labels, g, sp, L, base, flags, s);
    if (e == cudaSuccess) {
        hd_finish_kernel<<<(unsigned)std::min<int64_t>((nrc + 127) / 128, 1024), 128, 0, s>>>(rowmax, rowmax + 2 * nrc,
                                                                                               nrc, g.exact, hd);
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
    const HdGeom g = hd_geom(C, B, H, W, volume, sp);
    const HdLayout L = hd_layout(C, B, H, W, volume);
    char* base = static_cast<char*>(scratch);
    const unsigned* rowmax = reinterpret_cast<const unsigned*>(base + L.hdr);
    const uint16_t* rec = reinterpret_cast<const uint16_t*>(base + L.rec);
    const unsigned* qd = reinterpret_cast<const unsigned*>(base + L.qd);
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
                                                                                              st, nrc, g.exact, out);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return DCT_OK;
}

extern "C" size_t dct_surface_dice_scratch_bytes(int C, int64_t B, int64_t H, int64_t W, int volume) {
    if (C < 1 || B < 1 || H < 1 || W < 1 || !hd_supported(C, B, H, W, volume)) return 0;
    return hd_layout(C, B, H, W, volume).dice_total;
}

extern "C" int dct_surface_dice_i64(const int64_t* pred, const int64_t* labels, int C, int64_t B, int64_t H, int64_t W,
                                    int volume, const double* spacing, const double* tolerance, float* out,
                                    int64_t* counts, int32_t* flags, void* scratch, void* stream) {
    double sp[3];
    const int rc = hd_check_args(pred, labels, C, B, H, W, volume, spacing, out, flags, scratch, sp);
    if (rc != DCT_OK) return rc;
    if (tolerance == nullptr) return DCT_ERR_BAD_ARG;
    for (int c = 0; c < C; ++c)
        if (!(tolerance[c] >= 0.0) || !std::isfinite(tolerance[c])) return DCT_ERR_BAD_ARG;   // also rejects NaN
    if (!aligned(counts, 8)) return DCT_ERR_MISALIGNED;
    const HdGeom g = hd_geom(C, B, H, W, volume, sp);
    const HdLayout L = hd_layout(C, B, H, W, volume);
    char* base = static_cast<char*>(scratch);
    const int64_t nrc = (volume ? 1 : B) * C;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaError_t e = hd_distance_passes<false, true>(pred, labels, g, sp, L, base, flags, s, tolerance);
    if (e == cudaSuccess) {
        const int64_t lines_per_plane = volume ? H * W : B * H, lines_per_row = volume ? H * W : H;
        nsd_finish_kernel<<<(unsigned)std::min<int64_t>(nrc, (int64_t)kSMs * 8), kNsdThreads, 0, s>>>(
            reinterpret_cast<const unsigned*>(base + L.tq), reinterpret_cast<const unsigned*>(base + L.tw), C,
            lines_per_plane, lines_per_row, nrc, out, reinterpret_cast<long long*>(counts));
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return DCT_OK;
}

extern "C" size_t dct_distance_map_scratch_bytes(int C, int first_class, int64_t B, int64_t H, int64_t W, int volume,
                                                 int signed_map) {
    if (C < 1 || C > DCT_MAX_CLASSES || first_class < 0 || first_class >= C || (signed_map != 0 && signed_map != 1))
        return 0;
    if (B < 1 || H < 1 || W < 1 || !hd_supported(C - first_class, B, H, W, volume)) return 0;
    return dm_layout(C - first_class, B, H, W, volume, signed_map ? 2 : 1).total;
}

extern "C" int dct_distance_map_i64(const int64_t* map, int C, int first_class, int64_t B, int64_t H, int64_t W,
                                    int volume, const double* spacing, int signed_map, float* out, int32_t* flags,
                                    void* scratch, void* stream) {
    if (C < 1 || first_class < 0 || first_class >= C || (signed_map != 0 && signed_map != 1)) return DCT_ERR_BAD_ARG;
    if (C > DCT_MAX_CLASSES) return DCT_ERR_UNSUPPORTED;
    const int Cc = C - first_class, sides = signed_map ? 2 : 1;
    double sp[3];
    const int rc = hd_check_args(map, map, Cc, B, H, W, volume, spacing, out, flags, scratch, sp);
    if (rc != DCT_OK) return rc;
    const HdGeom g = hd_geom(Cc, B, H, W, volume, sp);
    const DmLayout L = dm_layout(Cc, B, H, W, volume, sides);
    char* base = static_cast<char*>(scratch);
    unsigned* present = reinterpret_cast<unsigned*>(base);
    unsigned char* cls = reinterpret_cast<unsigned char*>(base + L.cls);
    uint16_t* gdist = reinterpret_cast<uint16_t*>(base + L.g);
    unsigned* f = reinterpret_cast<unsigned*>(base + L.f);
    const int64_t nrc = (volume ? 1 : B) * Cc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);

    const int64_t cls_blocks = std::min<int64_t>((g.N + 255) / 256, (int64_t)kSMs * 16);
    dm_classify_kernel<<<(unsigned)cls_blocks, 256, 0, s>>>(map, g.N, C, cls, present, (int)(2 * nrc), flags);
    const int64_t col_lines = (int64_t)sides * Cc * B * W;
    dm_column_kernel<<<(unsigned)((col_lines + 127) / 128), 128, 0, s>>>(cls, g, sides, first_class, gdist, present);
    cudaError_t e = cudaGetLastError();

    EnvMapArgs a{};
    a.gdist = gdist; a.g = g;
    a.lines_per_plane = B * H; a.line_step = W; a.stride = 1; a.n = (int)W;
    a.w_in = sp[1] * sp[1]; a.w = sp[2] * sp[2];
    a.cls = cls; a.present = present; a.out = out; a.HW = H * W; a.ostride = 1;
    a.sides = sides; a.first_class = first_class;
    if (e == cudaSuccess && !volume) {
        a.lines_per_row = H;   // line l = b * H + y lies in image b
        e = launch_envelope<true, true, false, false, true>(a, s);
    } else if (e == cudaSuccess) {
        a.fout = f;
        e = launch_envelope<true, false, false, false, true>(a, s);
        EnvMapArgs z = a;
        z.gdist = nullptr; z.fout = nullptr; z.fin = f;
        z.lines_per_plane = H * W; z.line_step = 1; z.stride = H * W; z.n = (int)B;
        z.lines_per_row = H * W;   // one row: the volume
        z.w_in = 0.0; z.w = sp[0] * sp[0];
        z.ostride = (int64_t)Cc * H * W;
        if (e == cudaSuccess) e = launch_envelope<false, true, false, false, true>(z, s);
    }
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return DCT_OK;
}
