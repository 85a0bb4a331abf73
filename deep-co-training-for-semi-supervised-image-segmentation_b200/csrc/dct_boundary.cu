// dct_boundary.cu -- Boundary IoU (Cheng et al., CVPR 2021) of a class map against a label map on the device
// (evaluation path of the Cityscapes trainers, next to IoU.add).
//
// Definition (boundary-iou-api mask_to_boundary): for class c with mask M, the band of width d is
//   dM = M - erode(pad(M, 1, 0), ones(3, 3), iterations = d)[1:H+1, 1:W+1],
// i.e. x is in dM when x is in M and some cell of the (2d+1) x (2d+1) square centred on x is off the grid or outside M.
// Per (image, class): (I, G, P) = (|dP & dG & valid|, |dG|, |dP & valid|), valid = label != ignore_index.
//
// The square test is separable into run-length tests on lines: with u(r, j) = "rows r-d .. r+d of column j are on the
// grid and hold the value of (r, j)", x = (r, j) is interior iff columns j-d .. j+d of row r are on the grid, hold the
// class of x and have u = 1.  A position p of a line lies in a run reaching d cells to both sides iff
//   p - P(p) >= d  and  N(p) - p > d,
// with P(p) the last break <= p and N(p) the first break > p (a break at q: value(q) != value(q - 1); the line's ends
// are breaks).  Both are a prefix max / suffix min of break positions, so the work per pixel does not depend on d.
//
// Launches (3, whatever C is):
//   biou_col_kernel   along H.  A CTA owns 32 columns x kColSeg rows (lane = column, so every load and store is a
//                     256-byte / 64-byte row of the strip); each of its 16 warps takes 16 consecutive rows, the break
//                     positions are scanned across warps in shared memory.  The rows up to d above and below the
//                     segment are searched for their nearest break only (early exit once every column has one).  Writes
//                     one record byte per map and pixel: class in 7 bits (0x7E ignore label, 0x7F no class), u in bit
//                     7; raises the range flags; zeroes the (I, G, P) accumulators.
//   biou_row_kernel   along W.  A warp owns kRowSeg consecutive pixels of one row (loaded coalesced, transposed through
//                     shared memory so that each lane holds 8 consecutive pixels); warp shuffles scan the break
//                     positions of the records; halo search as above.  Classifies every pixel as band or interior for
//                     its class in both maps and counts I, G, P in per-CTA shared histograms (one shared atomic per
//                     run of a key within a lane's 8 pixels), flushed with 64-bit integer atomics: order-independent,
//                     bit-reproducible.
//   biou_finish_kernel  biou = float(double(I) / (G + P - I)), NaN for an empty union; copies the counts out.
// Scratch: 2 B per pixel of records + 24 B per (image, class) of accumulators, each rounded up to 256 B.  No host
// synchronisation, allocation or copy: a call captures into a CUDA graph.
#include <algorithm>
#include <climits>
#include <cmath>

#include "dct_common.cuh"

namespace dct {

constexpr int kColWarps = 16, kColRows = 16, kColSeg = kColWarps * kColRows;   // 256 rows per CTA
constexpr int kColThreads = kColWarps * 32;
constexpr int kRowWarps = 8, kRowPer = 8, kRowSeg = 32 * kRowPer;             // 256 pixels per warp
constexpr int kRowThreads = kRowWarps * 32;
constexpr int kHaloPer = 4;               // halo positions per thread and search step
constexpr int kSent = 0x100;              // value of a cell off the line (differs from every record byte)
constexpr int kNoClass = 0x7F, kIgnore = 0x7E, kUBit = 0x80;
constexpr int kFar = INT_MAX / 2;         // "no break" in segment-relative positions

template <typename T> __host__ __device__ __forceinline__ T bmax(T a, T b) { return a < b ? b : a; }
template <typename T> __host__ __device__ __forceinline__ T bmin(T a, T b) { return b < a ? b : a; }

struct BiouGeom {
    int C;
    int64_t B, H, W;
    int d;                   // dilation; meaningful only along an axis that can hold a (2d+1) window
    int none_h, none_w;      // 2d+1 > H (no u = 1) / 2d+1 > W (no interior pixel)
    int has_ignore;
    int64_t ignore;
    int64_t nstrip, nseg_h, nseg_w;
};

__device__ __forceinline__ int pred_code(long long v, int C) { return v >= 0 && v < C ? (int)v : kNoClass; }
__device__ __forceinline__ int label_code(long long v, const BiouGeom& g) {
    if (g.has_ignore && v == g.ignore) return kIgnore;
    return v >= 0 && v < g.C ? (int)v : kNoClass;
}

// ---- along H ----------------------------------------------------------------------------------------------------

// codes of (row y, column x) of image b, kSent off the grid
__device__ __forceinline__ void col_codes(const int64_t* __restrict__ pred, const int64_t* __restrict__ labels,
                                          const BiouGeom& g, int64_t img, int64_t x, int64_t y, int& vp, int& vg) {
    if (x < g.W && y >= 0 && y < g.H) {
        const int64_t i = img + y * g.W + x;
        vp = pred_code(pred[i], g.C);
        vg = label_code(labels[i], g);
    } else {
        vp = vg = kSent;
    }
}

__global__ void __launch_bounds__(kColThreads) biou_col_kernel(const int64_t* __restrict__ pred,
                                                               const int64_t* __restrict__ labels, const BiouGeom g,
                                                               uint16_t* __restrict__ rec,
                                                               unsigned long long* __restrict__ acc, int64_t nacc,
                                                               int32_t* flags) {
    __shared__ int s_a[2][kColWarps][32];   // per warp and column: first / last code, then break scans (pred, label)
    __shared__ int s_b[2][kColWarps][32];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nacc; i += (int64_t)gridDim.x * blockDim.x)
        acc[i] = 0ull;

    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t seg = (int64_t)blockIdx.x % g.nseg_h, rest = (int64_t)blockIdx.x / g.nseg_h;
    const int64_t b = rest / g.nstrip, x = (rest % g.nstrip) * 32 + lane;
    const int64_t img = b * g.H * g.W;
    const int64_t s0 = seg * kColSeg;
    const int64_t e0 = bmax<int64_t>(0, s0 - g.d), e1 = bmin<int64_t>(g.H, s0 + kColSeg + g.d);

    int vp[kColRows], vg[kColRows];
    int bad_p = 0, bad_l = 0;
#pragma unroll
    for (int i = 0; i < kColRows; ++i) {
        col_codes(pred, labels, g, img, x, s0 + w * kColRows + i, vp[i], vg[i]);
        bad_p += vp[i] == kNoClass;
        bad_l += vg[i] == kNoClass;
    }
    if (flags != nullptr) {
        bad_p = __reduce_add_sync(0xffffffffu, bad_p);
        bad_l = __reduce_add_sync(0xffffffffu, bad_l);
        if (lane == 0 && bad_p) atomicAdd(&flags[DCT_FLAG_PRED], bad_p);
        if (lane == 0 && bad_l) atomicAdd(&flags[DCT_FLAG_LABEL], bad_l);
    }

    bool up_p[kColRows], up_g[kColRows];
    if (g.none_h) {
#pragma unroll
        for (int i = 0; i < kColRows; ++i) up_p[i] = up_g[i] = false;
    } else {
        // nearest break above the segment: the largest q in (e0, s0) with code(q) != code(q-1), else e0
        int64_t top_p = e0, top_g = e0;
        bool found_p = s0 - 1 <= e0 || x >= g.W, found_g = found_p;   // nothing to search
        for (int64_t hi = s0 - 1; hi > e0; hi -= kColWarps * kHaloPer) {
            int64_t best_p = -1, best_g = -1;
#pragma unroll
            for (int k = 0; k < kHaloPer; ++k) {
                const int64_t q = hi - (w * kHaloPer + k);
                if (q > e0) {
                    int a_p, a_g, c_p, c_g;
                    col_codes(pred, labels, g, img, x, q, a_p, a_g);
                    col_codes(pred, labels, g, img, x, q - 1, c_p, c_g);
                    if (a_p != c_p) best_p = bmax(best_p, q);
                    if (a_g != c_g) best_g = bmax(best_g, q);
                }
            }
            s_a[0][w][lane] = (int)(best_p < 0 ? -1 : hi - best_p);   // distances below hi fit in int
            s_a[1][w][lane] = (int)(best_g < 0 ? -1 : hi - best_g);
            __syncthreads();
            int dp = INT_MAX, dg = INT_MAX;
            for (int v = 0; v < kColWarps; ++v) {
                if (s_a[0][v][lane] >= 0) dp = bmin(dp, s_a[0][v][lane]);
                if (s_a[1][v][lane] >= 0) dg = bmin(dg, s_a[1][v][lane]);
            }
            if (!found_p && dp != INT_MAX) { top_p = hi - dp; found_p = true; }
            if (!found_g && dg != INT_MAX) { top_g = hi - dg; found_g = true; }
            if (__syncthreads_and(found_p && found_g)) break;
        }
        // nearest break below the segment: the smallest q in (s0 + kColSeg, e1) with code(q) != code(q-1), else e1
        int64_t bot_p = e1, bot_g = e1;
        found_p = s0 + kColSeg + 1 >= e1 || x >= g.W; found_g = found_p;
        for (int64_t lo = s0 + kColSeg + 1; lo < e1; lo += kColWarps * kHaloPer) {
            int64_t best_p = LLONG_MAX, best_g = LLONG_MAX;
#pragma unroll
            for (int k = 0; k < kHaloPer; ++k) {
                const int64_t q = lo + (w * kHaloPer + k);
                if (q < e1) {
                    int a_p, a_g, c_p, c_g;
                    col_codes(pred, labels, g, img, x, q, a_p, a_g);
                    col_codes(pred, labels, g, img, x, q - 1, c_p, c_g);
                    if (a_p != c_p) best_p = bmin(best_p, q);
                    if (a_g != c_g) best_g = bmin(best_g, q);
                }
            }
            s_a[0][w][lane] = (int)(best_p == LLONG_MAX ? -1 : best_p - lo);
            s_a[1][w][lane] = (int)(best_g == LLONG_MAX ? -1 : best_g - lo);
            __syncthreads();
            int dp = INT_MAX, dg = INT_MAX;
            for (int v = 0; v < kColWarps; ++v) {
                if (s_a[0][v][lane] >= 0) dp = bmin(dp, s_a[0][v][lane]);
                if (s_a[1][v][lane] >= 0) dg = bmin(dg, s_a[1][v][lane]);
            }
            if (!found_p && dp != INT_MAX) { bot_p = lo + dp; found_p = true; }
            if (!found_g && dg != INT_MAX) { bot_g = lo + dg; found_g = true; }
            if (__syncthreads_and(found_p && found_g)) break;
        }

        // neighbours of this thread's rows: the previous warp's last row / the next warp's first row, or the halo
        s_a[0][w][lane] = vp[kColRows - 1]; s_a[1][w][lane] = vg[kColRows - 1];
        s_b[0][w][lane] = vp[0];            s_b[1][w][lane] = vg[0];
        __syncthreads();
        int prev_p, prev_g, next_p, next_g;
        if (w > 0) { prev_p = s_a[0][w - 1][lane]; prev_g = s_a[1][w - 1][lane]; }
        else if (s0 > 0) col_codes(pred, labels, g, img, x, s0 - 1, prev_p, prev_g);
        else prev_p = prev_g = kSent;
        if (w < kColWarps - 1) { next_p = s_b[0][w + 1][lane]; next_g = s_b[1][w + 1][lane]; }
        else if (s0 + kColSeg < e1) col_codes(pred, labels, g, img, x, s0 + kColSeg, next_p, next_g);
        else next_p = next_g = kSent;
        __syncthreads();

        // last break at or before each row: local scan, then the carry of the warps above (segment-relative rows)
        const int r0 = w * kColRows;
        int lb_p = -kFar, lb_g = -kFar, fb_p = kFar, fb_g = kFar;
#pragma unroll
        for (int i = 0; i < kColRows; ++i) {
            if (vp[i] != (i ? vp[i - 1] : prev_p)) lb_p = r0 + i;
            if (vg[i] != (i ? vg[i - 1] : prev_g)) lb_g = r0 + i;
        }
#pragma unroll
        for (int i = kColRows - 1; i >= 0; --i) {
            if (vp[i] != (i < kColRows - 1 ? vp[i + 1] : next_p)) fb_p = r0 + i + 1;
            if (vg[i] != (i < kColRows - 1 ? vg[i + 1] : next_g)) fb_g = r0 + i + 1;
        }
        s_a[0][w][lane] = lb_p; s_a[1][w][lane] = lb_g;
        s_b[0][w][lane] = fb_p; s_b[1][w][lane] = fb_g;
        __syncthreads();
        int P_p = (int)(top_p - s0), P_g = (int)(top_g - s0);   // >= -d
        int N_p = (int)(bot_p - s0), N_g = (int)(bot_g - s0);   // <= kColSeg + d
        for (int v = 0; v < w; ++v) { P_p = bmax(P_p, s_a[0][v][lane]); P_g = bmax(P_g, s_a[1][v][lane]); }
        for (int v = w + 1; v < kColWarps; ++v) {
            N_p = bmin(N_p, s_b[0][v][lane]); N_g = bmin(N_g, s_b[1][v][lane]);
        }
        bool upf_p[kColRows], upf_g[kColRows];
#pragma unroll
        for (int i = 0; i < kColRows; ++i) {
            if (vp[i] != (i ? vp[i - 1] : prev_p)) P_p = r0 + i;
            if (vg[i] != (i ? vg[i - 1] : prev_g)) P_g = r0 + i;
            upf_p[i] = r0 + i - P_p >= g.d;
            upf_g[i] = r0 + i - P_g >= g.d;
        }
#pragma unroll
        for (int i = kColRows - 1; i >= 0; --i) {
            if (vp[i] != (i < kColRows - 1 ? vp[i + 1] : next_p)) N_p = r0 + i + 1;
            if (vg[i] != (i < kColRows - 1 ? vg[i + 1] : next_g)) N_g = r0 + i + 1;
            up_p[i] = upf_p[i] && N_p - (r0 + i) > g.d;
            up_g[i] = upf_g[i] && N_g - (r0 + i) > g.d;
        }
    }

    if (x < g.W) {
#pragma unroll
        for (int i = 0; i < kColRows; ++i) {
            const int64_t y = s0 + w * kColRows + i;
            if (y < g.H)
                rec[img + y * g.W + x] = (uint16_t)((vp[i] | (up_p[i] ? kUBit : 0)) |
                                                    ((vg[i] | (up_g[i] ? kUBit : 0)) << 8));
        }
    }
}

// ---- along W ----------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(kRowThreads) biou_row_kernel(const uint16_t* __restrict__ rec, const BiouGeom g,
                                                               unsigned long long* __restrict__ acc) {
    __shared__ __align__(16) uint16_t s_buf[kRowWarps][kRowSeg];
    __shared__ unsigned s_hist[kRowWarps][3][DCT_MAX_CLASSES];   // [image slot][I, G, P][class]
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int C = g.C;
    const int64_t ntasks = g.B * g.H * g.nseg_w;
    const int64_t t0 = (int64_t)blockIdx.x * kRowWarps;
    const int64_t b_first = t0 / g.nseg_w / g.H;
    const int64_t b_last = bmin(t0 + kRowWarps, ntasks) - 1;
    const int nslots = (int)(b_last / g.nseg_w / g.H - b_first + 1);
    for (int i = threadIdx.x; i < nslots * 3 * DCT_MAX_CLASSES; i += blockDim.x) (&s_hist[0][0][0])[i] = 0u;
    __syncthreads();

    const int64_t t = t0 + w;
    if (t < ntasks) {   // warp-uniform
        const int64_t line = t / g.nseg_w, s0 = (t % g.nseg_w) * kRowSeg;
        const int slot = (int)(line / g.H - b_first);
        const uint16_t* row = rec + line * g.W;
        const int64_t W = g.W;
        const int64_t e0 = bmax<int64_t>(0, s0 - g.d), e1 = bmin<int64_t>(W, s0 + kRowSeg + g.d);
#pragma unroll
        for (int k = 0; k < kRowPer; ++k) {
            const int64_t p = s0 + k * 32 + lane;
            s_buf[w][k * 32 + lane] = p < W ? row[p] : (uint16_t)0;
        }
        __syncwarp();
        const uint4 packed = reinterpret_cast<const uint4*>(s_buf[w])[lane];
        const unsigned words[4] = {packed.x, packed.y, packed.z, packed.w};
        const int r0 = lane * kRowPer;
        int kp[kRowPer], kg[kRowPer];
#pragma unroll
        for (int i = 0; i < kRowPer; ++i) {
            const unsigned v = (words[i >> 1] >> ((i & 1) * 16)) & 0xFFFFu;
            const bool on = s0 + r0 + i < W;
            kp[i] = on ? (int)(v & 0xFFu) : kSent;
            kg[i] = on ? (int)(v >> 8) : kSent;
        }

        bool int_p[kRowPer], int_g[kRowPer];
        if (g.none_w) {
#pragma unroll
            for (int i = 0; i < kRowPer; ++i) int_p[i] = int_g[i] = false;
        } else {
            auto key = [&](int64_t q, int& a, int& c) {
                const unsigned v = row[q];
                a = (int)(v & 0xFFu); c = (int)(v >> 8);
            };
            // nearest break left of the segment: largest q in (e0, s0) with key(q) != key(q-1), else e0
            int64_t top_p = e0, top_g = e0;
            bool found_p = s0 - 1 <= e0, found_g = found_p;
            for (int64_t hi = s0 - 1; hi > e0 && !(found_p && found_g); hi -= 32 * kHaloPer) {
                int dp = INT_MAX, dg = INT_MAX;
#pragma unroll
                for (int k = 0; k < kHaloPer; ++k) {
                    const int off = k * 32 + lane;
                    if (hi - off > e0) {
                        int a_p, a_g, c_p, c_g;
                        key(hi - off, a_p, a_g);
                        key(hi - off - 1, c_p, c_g);
                        if (a_p != c_p) dp = bmin(dp, off);
                        if (a_g != c_g) dg = bmin(dg, off);
                    }
                }
                dp = (int)__reduce_min_sync(0xffffffffu, (unsigned)dp);
                dg = (int)__reduce_min_sync(0xffffffffu, (unsigned)dg);
                if (!found_p && dp != INT_MAX) { top_p = hi - dp; found_p = true; }
                if (!found_g && dg != INT_MAX) { top_g = hi - dg; found_g = true; }
            }
            // nearest break right of the segment: smallest q in (s0 + kRowSeg, e1) with key(q) != key(q-1), else e1
            int64_t bot_p = e1, bot_g = e1;
            found_p = s0 + kRowSeg + 1 >= e1; found_g = found_p;
            for (int64_t lo = s0 + kRowSeg + 1; lo < e1 && !(found_p && found_g); lo += 32 * kHaloPer) {
                int dp = INT_MAX, dg = INT_MAX;
#pragma unroll
                for (int k = 0; k < kHaloPer; ++k) {
                    const int off = k * 32 + lane;
                    if (lo + off < e1) {
                        int a_p, a_g, c_p, c_g;
                        key(lo + off, a_p, a_g);
                        key(lo + off - 1, c_p, c_g);
                        if (a_p != c_p) dp = bmin(dp, off);
                        if (a_g != c_g) dg = bmin(dg, off);
                    }
                }
                dp = (int)__reduce_min_sync(0xffffffffu, (unsigned)dp);
                dg = (int)__reduce_min_sync(0xffffffffu, (unsigned)dg);
                if (!found_p && dp != INT_MAX) { bot_p = lo + dp; found_p = true; }
                if (!found_g && dg != INT_MAX) { bot_g = lo + dg; found_g = true; }
            }

            int prev_p = __shfl_up_sync(0xffffffffu, kp[kRowPer - 1], 1);
            int prev_g = __shfl_up_sync(0xffffffffu, kg[kRowPer - 1], 1);
            int next_p = __shfl_down_sync(0xffffffffu, kp[0], 1);
            int next_g = __shfl_down_sync(0xffffffffu, kg[0], 1);
            if (lane == 0) {
                if (s0 > 0) key(s0 - 1, prev_p, prev_g);
                else prev_p = prev_g = kSent;
            }
            if (lane == 31) {
                if (s0 + kRowSeg < e1) key(s0 + kRowSeg, next_p, next_g);
                else next_p = next_g = kSent;
            }
            int lb_p = -kFar, lb_g = -kFar, fb_p = kFar, fb_g = kFar;
#pragma unroll
            for (int i = 0; i < kRowPer; ++i) {
                if (kp[i] != (i ? kp[i - 1] : prev_p)) lb_p = r0 + i;
                if (kg[i] != (i ? kg[i - 1] : prev_g)) lb_g = r0 + i;
            }
#pragma unroll
            for (int i = kRowPer - 1; i >= 0; --i) {
                if (kp[i] != (i < kRowPer - 1 ? kp[i + 1] : next_p)) fb_p = r0 + i + 1;
                if (kg[i] != (i < kRowPer - 1 ? kg[i + 1] : next_g)) fb_g = r0 + i + 1;
            }
            // exclusive prefix max of the last breaks / suffix min of the first breaks over the lanes
            int P_p = (int)(top_p - s0), P_g = (int)(top_g - s0), N_p = (int)(bot_p - s0), N_g = (int)(bot_g - s0);
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int a = __shfl_up_sync(0xffffffffu, lb_p, o), c = __shfl_up_sync(0xffffffffu, lb_g, o);
                const int e = __shfl_down_sync(0xffffffffu, fb_p, o), f = __shfl_down_sync(0xffffffffu, fb_g, o);
                if (lane >= o) { lb_p = bmax(lb_p, a); lb_g = bmax(lb_g, c); }
                if (lane + o < 32) { fb_p = bmin(fb_p, e); fb_g = bmin(fb_g, f); }
            }
            const int xl_p = __shfl_up_sync(0xffffffffu, lb_p, 1), xl_g = __shfl_up_sync(0xffffffffu, lb_g, 1);
            const int xf_p = __shfl_down_sync(0xffffffffu, fb_p, 1), xf_g = __shfl_down_sync(0xffffffffu, fb_g, 1);
            if (lane > 0) { P_p = bmax(P_p, xl_p); P_g = bmax(P_g, xl_g); }
            if (lane < 31) { N_p = bmin(N_p, xf_p); N_g = bmin(N_g, xf_g); }
            bool upf_p[kRowPer], upf_g[kRowPer];
#pragma unroll
            for (int i = 0; i < kRowPer; ++i) {
                if (kp[i] != (i ? kp[i - 1] : prev_p)) P_p = r0 + i;
                if (kg[i] != (i ? kg[i - 1] : prev_g)) P_g = r0 + i;
                upf_p[i] = r0 + i - P_p >= g.d;
                upf_g[i] = r0 + i - P_g >= g.d;
            }
#pragma unroll
            for (int i = kRowPer - 1; i >= 0; --i) {
                if (kp[i] != (i < kRowPer - 1 ? kp[i + 1] : next_p)) N_p = r0 + i + 1;
                if (kg[i] != (i < kRowPer - 1 ? kg[i + 1] : next_g)) N_g = r0 + i + 1;
                int_p[i] = (kp[i] & kUBit) && upf_p[i] && N_p - (r0 + i) > g.d;
                int_g[i] = (kg[i] & kUBit) && upf_g[i] && N_g - (r0 + i) > g.d;
            }
        }

        // each lane holds 8 consecutive pixels: count runs of one key per kind in registers, one shared atomic per run
        unsigned* hist = &s_hist[slot][0][0];
        int cur[3] = {-1, -1, -1};
        unsigned run[3] = {0u, 0u, 0u};
#pragma unroll
        for (int i = 0; i < kRowPer; ++i) {
            const int cp = kp[i] & 0x7F, cg = kg[i] & 0x7F;   // kSent & 0x7F == 0: masked by `on` below
            const bool on = kp[i] != kSent;
            const bool band_p = on && cp < C && !int_p[i], band_g = on && cg < C && !int_g[i];
            const int keys[3] = {band_p && band_g && cp == cg ? cp : -1, band_g ? cg : -1,
                                 band_p && cg != kIgnore ? cp : -1};
#pragma unroll
            for (int kind = 0; kind < 3; ++kind) {
                if (keys[kind] != cur[kind]) {
                    if (cur[kind] >= 0) atomicAdd(&hist[kind * DCT_MAX_CLASSES + cur[kind]], run[kind]);
                    cur[kind] = keys[kind];
                    run[kind] = 0u;
                }
                ++run[kind];
            }
        }
#pragma unroll
        for (int kind = 0; kind < 3; ++kind)
            if (cur[kind] >= 0) atomicAdd(&hist[kind * DCT_MAX_CLASSES + cur[kind]], run[kind]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nslots * 3 * C; i += blockDim.x) {
        const int slot = i / (3 * C), rem = i - slot * 3 * C, kind = rem / C, c = rem - kind * C;
        const unsigned v = s_hist[slot][kind][c];
        if (v) atomicAdd(&acc[((b_first + slot) * C + c) * 3 + kind], (unsigned long long)v);
    }
}

__global__ void biou_finish_kernel(const unsigned long long* __restrict__ acc, int64_t nrc, float* __restrict__ biou,
                                   long long* __restrict__ counts) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nrc; j += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long I = acc[3 * j], G = acc[3 * j + 1], P = acc[3 * j + 2];
        const unsigned long long U = G + P - I;
        biou[j] = U ? (float)((double)I / (double)U) : __int_as_float(0x7fffffff);
        if (counts != nullptr) {
            counts[3 * j] = (long long)I;
            counts[3 * j + 1] = (long long)G;
            counts[3 * j + 2] = (long long)P;
        }
    }
}

inline size_t biou_align256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace dct

using namespace dct;

static bool biou_supported(int C, int64_t B, int64_t H, int64_t W) {
    if (C > DCT_MAX_CLASSES) return false;
    if (B > INT_MAX || H > INT_MAX || W > INT_MAX) return false;
    return B * H <= INT_MAX && B * H * W <= INT_MAX;
}

extern "C" size_t dct_boundary_iou_scratch_bytes(int C, int64_t B, int64_t H, int64_t W) {
    if (C < 1 || B < 1 || H < 1 || W < 1 || !biou_supported(C, B, H, W)) return 0;
    return biou_align256((size_t)(B * H * W) * 2) + biou_align256((size_t)B * C * 24);
}

extern "C" int dct_boundary_iou_i64(const int64_t* pred, const int64_t* labels, int C, int64_t B, int64_t H,
                                    int64_t W, int64_t dilation, int64_t ignore_index, float* biou, int64_t* counts,
                                    int32_t* flags, void* scratch, void* stream) {
    if (pred == nullptr || labels == nullptr || biou == nullptr || scratch == nullptr) return DCT_ERR_BAD_ARG;
    if (C < 1 || B < 1 || H < 1 || W < 1 || dilation < 1) return DCT_ERR_BAD_ARG;
    if (ignore_index >= 0 && ignore_index < C) return DCT_ERR_BAD_ARG;
    if (!biou_supported(C, B, H, W)) return DCT_ERR_UNSUPPORTED;
    if (!aligned(pred, 8) || !aligned(labels, 8) || !aligned(biou, 4) || !aligned(counts, 8) || !aligned(flags, 4) ||
        !aligned(scratch, 256))
        return DCT_ERR_MISALIGNED;

    BiouGeom g{};
    g.C = C; g.B = B; g.H = H; g.W = W;
    g.none_h = dilation > (H - 1) / 2;   // 2d+1 > H, without overflow
    g.none_w = dilation > (W - 1) / 2;
    g.d = (g.none_h && g.none_w) ? 1 : (int)dilation;   // < 2^30 whenever an axis can hold the window
    g.has_ignore = ignore_index >= 0;
    g.ignore = ignore_index;
    g.nstrip = (W + 31) / 32;
    g.nseg_h = (H + kColSeg - 1) / kColSeg;
    g.nseg_w = (W + kRowSeg - 1) / kRowSeg;

    const int64_t N = B * H * W, nrc = B * C;
    char* base = static_cast<char*>(scratch);
    uint16_t* rec = reinterpret_cast<uint16_t*>(base);
    unsigned long long* acc = reinterpret_cast<unsigned long long*>(base + biou_align256((size_t)N * 2));
    cudaStream_t s = static_cast<cudaStream_t>(stream);

    const int64_t col_ctas = B * g.nstrip * g.nseg_h;          // <= N
    const int64_t row_ctas = (B * H * g.nseg_w + kRowWarps - 1) / kRowWarps;
    biou_col_kernel<<<(unsigned)col_ctas, kColThreads, 0, s>>>(pred, labels, g, rec, acc, 3 * nrc, flags);
    biou_row_kernel<<<(unsigned)row_ctas, kRowThreads, 0, s>>>(rec, g, acc);
    biou_finish_kernel<<<(unsigned)std::min<int64_t>((nrc + 255) / 256, (int64_t)kSMs * 8), 256, 0, s>>>(
        acc, nrc, biou, reinterpret_cast<long long*>(counts));
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return DCT_OK;
}
