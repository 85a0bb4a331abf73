// dct_jsd_kernels.cuh -- K-view Jensen-Shannon divergence, forward / backward / fused, sm_100a.
//
// Replaces JSD_2D / JSD / Entropy_2D (generalframework/loss/loss.py:53-84,165-196) and, in logits
// mode, the F.softmax that feeds them (generalframework/models/segmentators.py:46-50).
//
// Data layout: K tensors [B,C,HW] (NCHW): for a fixed (k,c) the HW pixels are contiguous, so a
// warp reading VEC consecutive pixels per lane issues one fully coalesced 128*VEC-byte request
// per (k,c) plane.  All K*C planes of a pixel group are loaded up front (K*C independent
// streaming loads in flight per thread), the per-pixel math runs entirely in registers, and the
// gradients are stored back with the same access pattern.  No shared memory, no tensor cores:
// the kernel is an HBM-bound map/reduce (see DESIGN.md, "JSD kernel").
#pragma once
#include <cstring>
#include "dct_common.cuh"
#include "dct_tile.cuh"

namespace dct {

enum JsdMode { kFwd = 0, kBwd = 1, kFwdBwd = 2 };

template <int K>
struct JsdArgs {
    Views<K> v;
    int64_t B, HW;          // images b = blockIdx.y, blockIdx.y + gridDim.y, ... (image_grid)
    float* map;             // [B,HW] or null
    double* sum;            // or null
    Upstream up;            // kBwd: full upstream; kFwdBwd: gconst only
    int32_t* flags;         // or null
    Workspace* ws;
};

struct JsdArgsRt {          // runtime-(K,C) fallback
    const float* in[DCT_MAX_VIEWS];
    float* grad[DCT_MAX_VIEWS];
    int K, C;
    int64_t B, HW;
    float* map;
    double* sum;
    Upstream up;
    int32_t* flags;
    Workspace* ws;
};

// s / K.  Powers of two are exact; otherwise one multiply by the rounded reciprocal (<= 1 ulp from the
// reference's true division, far inside the 1e-5 budget, and ~10 instructions cheaper per call).
template <int K>
__device__ __forceinline__ float div_by_K(float s) {
    return s * (1.0f / (float)K);
}

// One pixel (T = float) or one pixel PAIR (T = f2, packed FP32x2 math -- see dct_common.cuh).
// In: x[k][c] (probs or logits).  Out: returns the JSD value (nats); if GRAD, x[k][c] is
// overwritten with gK * d JSD / d x[k][c]  (gK = upstream / K).  `bad` is set when a view fails
// the reference's simplex predicate (probs mode only).
//
// All logarithms are taken in base 2 (one MUFU.LG2 / MUFU.EX2 each, flush-to-zero) and the
// ln 2 factor is applied once per pixel: H = -ln2 * sum p*lg2(p).
template <int K, int C, bool LOGITS, bool GRAD, class T>
__device__ __forceinline__ T jsd_pixel(T (&x)[K][C], T gK, bool& bad) {
    constexpr float invK = 1.0f / (float)K;  // exact for powers of two; else <= 1 ulp from the true division
    T p[K][C];
    T hsum = vset<T>(0.0f);  // sum_k sum_c p*lg2 p   (= -sum_k H_k / ln2)
    if constexpr (LOGITS) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            T mx = x[k][0];
#pragma unroll
            for (int c = 1; c < C; ++c) mx = vmax(mx, x[k][c]);
            const T nmxl = vmuls(mx, -kLog2e);
            T Z;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                T t = vfmas(x[k][c], kLog2e, nmxl);  // (x - max) * log2(e), one rounding
                T e = vex2(t);
                x[k][c] = t;
                p[k][c] = e;
                Z = (c == 0) ? e : vadd(Z, e);
            }
            const T inv = vrcp(Z);
            const T lZ = vlg2(Z);
            T hk = vset<T>(0.0f);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                T pv = vmul(p[k][c], inv);
                T lp = vsub(x[k][c], lZ);  // lg2 softmax: differs from lg2(p+1e-16) by < 1e-16/p, and
                p[k][c] = pv;              // only ever multiplied by p  ->  absolute error < 1e-16
                x[k][c] = lp;
                hk = vfma(pv, lp, hk);
            }
            hsum = vadd(hsum, hk);
        }
    } else {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            T s = vset<T>(0.0f), hk = vset<T>(0.0f);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                T pv = x[k][c];
                s = vadd(s, pv);
                T lp = vlg2(vadds(pv, kEntEps));
                p[k][c] = pv;
                x[k][c] = lp;
                hk = vfma(pv, lp, hk);
            }
            bad |= vsimplex_bad(s);
            hsum = vadd(hsum, hk);
        }
    }
    T hm = vset<T>(0.0f);  // sum_c m*lg2(m+eps)  (= -H(m)/ln2)
    T am[C];               // per class: lg2(m+eps) [probs mode with GRAD: ln2*lg2(m+eps) + m/(m+eps)]
#pragma unroll
    for (int c = 0; c < C; ++c) {
        T s = p[0][c];
#pragma unroll
        for (int k = 1; k < K; ++k) s = vadd(s, p[k][c]);
        T m = vmuls(s, invK);
        T me = vadds(m, kEntEps);
        T lm = vlg2(me);
        hm = vfma(m, lm, hm);
        if constexpr (GRAD && !LOGITS) lm = vfmas(lm, kLn2, vmul(m, vrcp(me)));
        am[c] = lm;
    }
    const T jsd = vmuls(vsub(vmuls(hsum, invK), hm), kLn2);
    if constexpr (GRAD) {
        if constexpr (LOGITS) {
            // d/dz_kc = gK * p_kc * ((ln p_kc - ln m_c) - KL(p_k || m));  the +1 terms of
            // d(p log p)/dp cancel inside the softmax backward.  ln = ln2 * lg2 folded into gK.
            const T g2 = vmuls(gK, kLn2);
#pragma unroll
            for (int k = 0; k < K; ++k) {
                T kl = vset<T>(0.0f);
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    T t = vsub(x[k][c], am[c]);
                    x[k][c] = t;
                    kl = vfma(p[k][c], t, kl);
                }
#pragma unroll
                for (int c = 0; c < C; ++c) x[k][c] = vmul(vmul(g2, p[k][c]), vsub(x[k][c], kl));
            }
        } else {
            // d/dp_kc = gK * [(ln(p+e) + p/(p+e)) - (ln(m+e) + m/(m+e))]
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    T pv = p[k][c];
                    T a = vfmas(x[k][c], kLn2, vmul(pv, vrcp(vadds(pv, kEntEps))));
                    x[k][c] = vmul(gK, vsub(a, am[c]));
                }
        }
    }
    return jsd;
}

// K-view JSD forward + backward from logits on a pixel (pair) whose K*C values stay in the shared-memory stage (K*C > 40:
// a register-resident pair would need > 255 registers and spills).  Four sweeps over the stage, in place:
//   A  per view: max_c x                                                    (LDS)
//   B  per view: e = 2^((x - max) log2 e) written over x; Z = sum e; S = sum e*t       -> sum_c p lg p = S/Z - lg Z
//   C  per class: m = (1/K) sum_k e_k/Z_k; lg m; H(m); per view sum_c e lg m           -> KL(p_k||m) without another pass
//   D  per class: lg m again (K multiplies + one MUFU), lg p = lg2(e) - lg Z; gradient written over e
// MUFU per pixel: 2*K*C (ex2, lg2 of e) + 2*C (lg m) + 2*K -- 155 at K=3, 190 at K=4, against ~360-480 issue slots.
// e underflows to 0 below 2^-126: lg2(0) = -inf is clamped so that 0 * (...) stays 0 (the register path's 0 * finite).
template <int K, int C, class T>
__device__ __forceinline__ T jsd_stream_pair(unsigned char* st, size_t row_bytes, int p0, float g) {
    auto at = [&](int k, int c) -> T* { return reinterpret_cast<T*>(st + (size_t)(k * C + c) * row_bytes + (size_t)p0 * 4); };
    const float invK = 1.0f / (float)K;
    T rZ[K], lZ[K], hp[K];
    T hsum = vset<T>(0.0f);
#pragma unroll
    for (int k = 0; k < K; ++k) {
        T mx = *at(k, 0);
#pragma unroll
        for (int c = 1; c < C; ++c) mx = vmax(mx, *at(k, c));
        const T nmxl = vmuls(mx, -kLog2e);
        T Z = vset<T>(0.0f), S = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const T t = vfmas(*at(k, c), kLog2e, nmxl);  // (x - max) * log2(e), one rounding
            const T e = vex2(t);
            *at(k, c) = e;
            Z = vadd(Z, e);
            S = vfma(e, t, S);
        }
        rZ[k] = vrcp(Z);
        lZ[k] = vlg2(Z);
        hp[k] = vsub(vmul(rZ[k], S), lZ[k]);     // sum_c p lg2 p
        hsum = vadd(hsum, hp[k]);
        // compiler barrier: the next sweeps re-read e from the stage instead of keeping K*C pairs in (255) registers
        // across them -- the point of this body is a small register footprint
        asm volatile("" ::: "memory");
    }
    T hm = vset<T>(0.0f);
    T plm[K];
#pragma unroll
    for (int k = 0; k < K; ++k) plm[k] = vset<T>(0.0f);
    T rZK[K];                                    // 1 / (K Z_k): m_c = sum_k e_kc * rZK_k
#pragma unroll
    for (int k = 0; k < K; ++k) rZK[k] = vmuls(rZ[k], invK);
#pragma unroll
    for (int c = 0; c < C; ++c) {
        T e[K];
#pragma unroll
        for (int k = 0; k < K; ++k) e[k] = *at(k, c);
        T m = vmul(e[0], rZK[0]);
#pragma unroll
        for (int k = 1; k < K; ++k) m = vfma(e[k], rZK[k], m);
        const T lm = vlg2(vadds(m, kEntEps));
        hm = vfma(m, lm, hm);
#pragma unroll
        for (int k = 0; k < K; ++k) plm[k] = vfma(e[k], lm, plm[k]);
    }
    const T jsd = vmuls(vsub(vmuls(hsum, invK), hm), kLn2);
    asm volatile("" ::: "memory");
    // gradient: (g/K) ln2 * p_kc * ((lg p_kc - lg m_c) - KL_k),  KL_k = hp_k - sum_c p_kc lg m_c  (in lg2 units)
    T off[K], gr[K];
    const float g2 = g * invK * kLn2;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const T kl = vsub(hp[k], vmul(rZ[k], plm[k]));
        off[k] = vadd(lZ[k], kl);                // (lg2 e - lg Z) - lg m - KL  =  lg2 e - lg m - off
        gr[k] = vmuls(rZ[k], g2);                // g2 * p = gr * e
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
        T e[K];
#pragma unroll
        for (int k = 0; k < K; ++k) e[k] = *at(k, c);
        T m = vmul(e[0], rZK[0]);
#pragma unroll
        for (int k = 1; k < K; ++k) m = vfma(e[k], rZK[k], m);
        const T lm = vlg2(vadds(m, kEntEps));
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const T le = vmax(vlg2(e[k]), vset<T>(-1.0e4f));   // e == 0 (underflow): keep 0 * finite == 0
            *at(k, c) = vmul(vmul(gr[k], e[k]), vsub(vsub(le, lm), off[k]));
        }
    }
    return jsd;
}

// JSD as a tile-pipeline Op (dct_tile.cuh): NIN = K views; gradients overwrite the views' rows.
template <int K, bool LOGITS, int MODE, bool DICEF>
struct JsdOp {
    static constexpr int NIN = K, NOUT = (MODE != kFwd) ? K : 0;
    static constexpr bool HAS_MAP = (MODE != kBwd), USES_UP = (MODE != kFwd), CHECKS_SIMPLEX = !LOGITS;
    static constexpr int NDICE = DICEF ? K : 0;
    static constexpr bool GMAP = (MODE == kBwd);
    // logits in, loss + gradients out, no meters: the shape the shared-memory-resident body (jsd_stream_pair) serves
    static constexpr bool STREAM_CAPABLE = LOGITS && MODE == kFwdBwd && !DICEF;
    template <int CM, class T>   // T = f2: a pixel pair per thread (p0 even); T = float: one pixel per thread
    static __device__ __forceinline__ T stream(unsigned char* st, size_t row_bytes, int p0, float g) {
        return jsd_stream_pair<K, CM, T>(st, row_bytes, p0, g);
    }
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[K][CM], int, T g, float, bool& bad) {
        return jsd_pixel<K, CM, LOGITS, MODE != kFwd, T>(x, vmuls(g, 1.0f / (float)K), bad);
    }
};

template <int K, int C>
constexpr int jsd_vec() {
    return K * C <= 16 ? 4 : (K * C <= 40 ? 2 : 1);
}

template <int K, int C, int VEC, bool LOGITS, int MODE, int MINB = 1>
__global__ void __launch_bounds__(256, MINB) jsd_kernel(const JsdArgs<K> a) {
    const int64_t HW = a.HW;
    const int64_t gpi = HW / VEC;  // pixel groups per image (host guarantees HW % VEC == 0)
    float gs = 0.0f;
    if constexpr (MODE == kBwd) gs = upstream_scalar(a.up);
    if constexpr (MODE == kFwdBwd) gs = a.up.gconst;
    gs = div_by_K<K>(gs);
    double acc = 0.0;
    bool bad = false;
    for (int64_t b = blockIdx.y; b < a.B; b += gridDim.y) {
        const int64_t img = b * C * HW;
        for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < gpi; g += (int64_t)gridDim.x * blockDim.x) {
            const int64_t i = g * VEC;
            FVec<VEC> xin[K][C];
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int c = 0; c < C; ++c) xin[k][c] = ld_stream<VEC>(a.v.in[k] + img + (int64_t)c * HW + i);
            FVec<VEC> gm;
            if constexpr (MODE == kBwd) {
                if (a.up.gmap != nullptr) gm = ld_stream<VEC>(a.up.gmap + b * HW + i);
                else {
#pragma unroll
                    for (int v = 0; v < VEC; ++v) gm.v[v] = 1.0f;
                }
            }
            FVec<VEC> mapv;
            float part = 0.0f;
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                float x[K][C];
#pragma unroll
                for (int k = 0; k < K; ++k)
#pragma unroll
                    for (int c = 0; c < C; ++c) x[k][c] = xin[k][c].v[v];
                float gK = gs;
                if constexpr (MODE == kBwd) gK *= gm.v[v];
                float j = jsd_pixel<K, C, LOGITS, MODE != kFwd, float>(x, gK, bad);
                mapv.v[v] = j;
                part += j;
                if constexpr (MODE != kFwd) {
#pragma unroll
                    for (int k = 0; k < K; ++k)
#pragma unroll
                        for (int c = 0; c < C; ++c) xin[k][c].v[v] = x[k][c];
                }
            }
            acc += (double)part;
            if constexpr (MODE != kBwd) {
                if (a.map != nullptr) st_stream<VEC>(a.map + b * HW + i, mapv);
            }
            if constexpr (MODE != kFwd) {
#pragma unroll
                for (int k = 0; k < K; ++k)
#pragma unroll
                    for (int c = 0; c < C; ++c) st_stream<VEC>(a.v.grad[k] + img + (int64_t)c * HW + i, xin[k][c]);
            }
        }
    }
    if constexpr (MODE != kBwd) {
        if constexpr (!LOGITS) {
            if (a.flags != nullptr && __syncthreads_or(bad)) {
                // count per pixel-group is not needed: the contract is "non-zero == violated"
                if (bad) atomicAdd(&a.flags[DCT_FLAG_SIMPLEX], 1);
            }
        }
        grid_sum_to(acc, a.ws, a.sum, blockIdx.y * gridDim.x + blockIdx.x, gridDim.x * gridDim.y);
    }
}

// ---------------------------------------------------------------------------------------------
// Runtime-(K,C) fallback: one pixel per thread, three sweeps over the class axis re-reading the
// inputs (L1/L2 hits).  Correctness path for shapes without a register-tiled instantiation.
// ---------------------------------------------------------------------------------------------
template <bool LOGITS, int MODE>
__global__ void __launch_bounds__(256) jsd_kernel_rt(const JsdArgsRt a) {
    const int K = a.K, C = a.C;
    const int64_t HW = a.HW;
    const float invK = 1.0f / (float)K;
    float gs = 0.0f;
    if constexpr (MODE == kBwd) gs = upstream_scalar(a.up);
    if constexpr (MODE == kFwdBwd) gs = a.up.gconst;
    double acc = 0.0;
    bool bad = false;
    for (int64_t b = blockIdx.y; b < a.B; b += gridDim.y) {
        const int64_t img = b * C * HW;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (int64_t)gridDim.x * blockDim.x) {
            float mx[DCT_MAX_VIEWS], inv[DCT_MAX_VIEWS], lZ[DCT_MAX_VIEWS], kl[DCT_MAX_VIEWS];
            float hsum = 0.0f;
#pragma unroll
            for (int k = 0; k < DCT_MAX_VIEWS; ++k) {
                mx[k] = 0.0f; inv[k] = 1.0f; lZ[k] = 0.0f; kl[k] = 0.0f;
                if (k < K) {
                    const float* xb = a.in[k] + img + i;
                    if constexpr (LOGITS) {
                        float m = xb[0];
                        for (int c = 1; c < C; ++c) m = fmaxf(m, xb[(int64_t)c * HW]);
                        float Z = 0.0f;
                        for (int c = 0; c < C; ++c) Z += fexp(xb[(int64_t)c * HW] - m);
                        mx[k] = m; inv[k] = fdiv(1.0f, Z); lZ[k] = flog(Z);
                    } else {
                        float s = 0.0f;
                        for (int c = 0; c < C; ++c) s += xb[(int64_t)c * HW];
                        bad |= !simplex_ok(s);
                    }
                }
            }
            float hm = 0.0f;
            for (int c = 0; c < C; ++c) {
                float s = 0.0f;
                float pv[DCT_MAX_VIEWS], lp[DCT_MAX_VIEWS];
#pragma unroll
                for (int k = 0; k < DCT_MAX_VIEWS; ++k) {
                    pv[k] = 0.0f; lp[k] = 0.0f;
                    if (k < K) {
                        float xv = a.in[k][img + (int64_t)c * HW + i];
                        if constexpr (LOGITS) { float d = xv - mx[k]; pv[k] = fexp(d) * inv[k]; lp[k] = d - lZ[k]; }
                        else { pv[k] = xv; lp[k] = flog(xv + kEntEps); }
                        s = (k == 0) ? pv[k] : s + pv[k];
                        hsum = fmaf(pv[k], lp[k], hsum);
                    }
                }
                float m = ((K & (K - 1)) == 0) ? s * invK : s / (float)K;
                float lm = flog(m + kEntEps);
                hm = fmaf(m, lm, hm);
#pragma unroll
                for (int k = 0; k < DCT_MAX_VIEWS; ++k)
                    if (k < K) kl[k] = fmaf(pv[k], lp[k] - lm, kl[k]);
            }
            float hs = ((K & (K - 1)) == 0) ? hsum * invK : hsum / (float)K;
            const float jsd = hs - hm;
            acc += (double)jsd;
            if constexpr (MODE != kBwd) {
                if (a.map != nullptr) a.map[(int64_t)b * HW + i] = jsd;
            }
            if constexpr (MODE != kFwd) {
                float g = gs;
                if constexpr (MODE == kBwd) { if (a.up.gmap != nullptr) g *= a.up.gmap[(int64_t)b * HW + i]; }
                float gK = ((K & (K - 1)) == 0) ? g * invK : g / (float)K;
                for (int c = 0; c < C; ++c) {
                    float s = 0.0f;
                    float pv[DCT_MAX_VIEWS], lp[DCT_MAX_VIEWS];
#pragma unroll
                    for (int k = 0; k < DCT_MAX_VIEWS; ++k) {
                        pv[k] = 0.0f; lp[k] = 0.0f;
                        if (k < K) {
                            float xv = a.in[k][img + (int64_t)c * HW + i];
                            if constexpr (LOGITS) { float d = xv - mx[k]; pv[k] = fexp(d) * inv[k]; lp[k] = d - lZ[k]; }
                            else { pv[k] = xv; lp[k] = flog(xv + kEntEps); }
                            s = (k == 0) ? pv[k] : s + pv[k];
                        }
                    }
                    float m = ((K & (K - 1)) == 0) ? s * invK : s / (float)K;
                    float lm = flog(m + kEntEps);
#pragma unroll
                    for (int k = 0; k < DCT_MAX_VIEWS; ++k)
                        if (k < K) {
                            float gv;
                            if constexpr (LOGITS) gv = gK * pv[k] * ((lp[k] - lm) - kl[k]);
                            else gv = gK * ((lp[k] + fdiv(pv[k], pv[k] + kEntEps)) - (lm + fdiv(m, m + kEntEps)));
                            a.grad[k][img + (int64_t)c * HW + i] = gv;
                        }
                }
            }
        }
    }
    if constexpr (MODE != kBwd) {
        if constexpr (!LOGITS) {
            if (a.flags != nullptr && __syncthreads_or(bad)) {
                if (bad) atomicAdd(&a.flags[DCT_FLAG_SIMPLEX], 1);
            }
        }
        grid_sum_to(acc, a.ws, a.sum, blockIdx.y * gridDim.x + blockIdx.x, gridDim.x * gridDim.y);
    }
}

// ---------------------------------------------------------------------------------------------
// host-side launch of one (K,C) instantiation; defined per K in dct_jsd_k*.cu
// ---------------------------------------------------------------------------------------------
struct JsdCall {
    const int64_t* labels;      // fused Dice (kFwdBwd / kFwd with logits): nullable
    int64_t* counts;            // [K][B][C][3]
    bool* dice_done;            // set to true when the launch also produced the Dice counts
    const float* const* views;
    float* const* grads;
    int K, C;
    int64_t B, HW;
    int in_kind, mode;
    float* map;
    double* sum;
    Upstream up;
    int32_t* flags;
    Workspace* ws;
    cudaStream_t stream;
    int elem = 0;               // 0: float32 tensors; 1: bfloat16 tensors (views / grads point to bf16; tile pipeline only)
    bool counts_overwrite = false;   // DCT_COUNTS_OVERWRITE: the fused launch clears `counts` itself
    const dct_peer_pub* pub = nullptr;   // dct_jsd_fwdbwd_pub_f32: sums (final before this launch) its first finishing CTA publishes
    bool* pub_done = nullptr;            // set to true when the launch carried the publication
};

// returns DCT_ERR_UNSUPPORTED when (K,C) has no register-tiled instantiation
int jsd_launch_k2(const JsdCall& c);
int jsd_launch_k3(const JsdCall& c);
int jsd_launch_k4(const JsdCall& c);

template <int K, int C, class ET = float>
int jsd_launch_tile(const JsdCall& c) {
    TileArgs a{};
    for (int k = 0; k < K; ++k) {
        a.in[k] = c.views[k];
        a.out[k] = c.grads ? c.grads[k] : nullptr;
    }
    a.HW = c.HW; a.map = c.map; a.sum = c.sum; a.up = c.up; a.eps = 0.0f; a.flags = c.flags; a.ws = c.ws;
    a.labels = nullptr; a.counts = nullptr; a.count_view_stride = c.B * C * 3; a.counts_overwrite = c.counts_overwrite ? 1 : 0;
    const bool lg = c.in_kind == DCT_IN_LOGITS;
    if constexpr (!std::is_same<ET, float>::value) {
        // bf16 tensors: the one-pass-over-logits forms only (fused forward+backward [+ Dice], or forward for eval)
        if (!lg || c.mode == kBwd) return DCT_ERR_UNSUPPORTED;
        if (c.mode == kFwd) {
            if (!tile_eligible<JsdOp<K, true, kFwd, false>, ET>(a, c.B)) return DCT_ERR_UNSUPPORTED;
            return tile_launch_ct<JsdOp<K, true, kFwd, false>, C, ET>(a, c.B, c.stream);
        }
        if constexpr (C <= 4) {
            if (c.labels != nullptr && aligned(c.labels, 16)) {
                a.labels = c.labels;
                a.counts = reinterpret_cast<unsigned long long*>(c.counts);
                if (!tile_eligible<JsdOp<K, true, kFwdBwd, true>, ET>(a, c.B)) return DCT_ERR_UNSUPPORTED;
                int rc = tile_launch_ct<JsdOp<K, true, kFwdBwd, true>, C, ET>(a, c.B, c.stream);
                if (rc == DCT_OK && c.dice_done) *c.dice_done = true;
                return rc;
            }
        }
        if (!tile_eligible<JsdOp<K, true, kFwdBwd, false>, ET>(a, c.B)) return DCT_ERR_UNSUPPORTED;
        return tile_launch_ct<JsdOp<K, true, kFwdBwd, false>, C, ET>(a, c.B, c.stream);
    } else {
    if (c.mode == kFwdBwd) {
        // logits in, with a loss sum: the launch can also carry the early publication of the previous step's sums (PUB kernels)
        const bool pub = lg && c.pub != nullptr && c.sum != nullptr && c.ws != nullptr;
        if (pub) {
            std::memcpy(&a.pub, c.pub, sizeof(a.pub));
            a.pub_early = 1;
        }
        if constexpr (C <= 4) {
            if (lg && c.labels != nullptr && aligned(c.labels, 16)) {
                a.labels = c.labels;
                a.counts = reinterpret_cast<unsigned long long*>(c.counts);
                if (!tile_eligible<JsdOp<K, true, kFwdBwd, true>, ET>(a, c.B)) return DCT_ERR_UNSUPPORTED;
                int rc = pub ? tile_launch_ct<JsdOp<K, true, kFwdBwd, true>, C, ET, true>(a, c.B, c.stream)
                             : tile_launch_ct<JsdOp<K, true, kFwdBwd, true>, C, ET>(a, c.B, c.stream);
                if (rc == DCT_OK && c.dice_done) *c.dice_done = true;
                if (rc == DCT_OK && pub && c.pub_done) *c.pub_done = true;
                return rc;
            }
        }
        if (!tile_eligible<JsdOp<K, true, kFwdBwd, false>, ET>(a, c.B)) return DCT_ERR_UNSUPPORTED;
        if (pub) {
            int rc = tile_launch_ct<JsdOp<K, true, kFwdBwd, false>, C, ET, true>(a, c.B, c.stream);
            if (rc == DCT_OK && c.pub_done) *c.pub_done = true;
            return rc;
        }
        return lg ? tile_launch_ct<JsdOp<K, true, kFwdBwd, false>, C, ET>(a, c.B, c.stream)
                  : tile_launch_ct<JsdOp<K, false, kFwdBwd, false>, C, ET>(a, c.B, c.stream);
    }
    if (c.mode == kBwd) {
        if (!tile_eligible<JsdOp<K, true, kBwd, false>, ET>(a, c.B)) return DCT_ERR_UNSUPPORTED;
        return lg ? tile_launch_ct<JsdOp<K, true, kBwd, false>, C, ET>(a, c.B, c.stream)
                  : tile_launch_ct<JsdOp<K, false, kBwd, false>, C, ET>(a, c.B, c.stream);
    }
    if (!tile_eligible<JsdOp<K, true, kFwd, false>, ET>(a, c.B)) return DCT_ERR_UNSUPPORTED;
    return lg ? tile_launch_ct<JsdOp<K, true, kFwd, false>, C, ET>(a, c.B, c.stream)
              : tile_launch_ct<JsdOp<K, false, kFwd, false>, C, ET>(a, c.B, c.stream);
    }
}

template <int K, int C>
int jsd_launch_kc(const JsdCall& c) {
    if (c.elem == 1) {
        if constexpr (K * C <= kTileMaxRows) return jsd_launch_tile<K, C, bf16>(c);
        return DCT_ERR_UNSUPPORTED;
    }
    if constexpr (K * C <= kTileMaxRows) {
        // TMA tile pipeline (falls through to the register-tiled kernel when rows are not 16-byte aligned)
        int rc = jsd_launch_tile<K, C>(c);
        if (rc != DCT_ERR_UNSUPPORTED) return rc;
    }
    constexpr int VEC = jsd_vec<K, C>();
    JsdArgs<K> a;
    bool al = (c.HW % VEC) == 0 && (c.map == nullptr || aligned(c.map, 4 * VEC)) &&
              (c.up.gmap == nullptr || aligned(c.up.gmap, 4 * VEC));
    for (int k = 0; k < K; ++k) {
        a.v.in[k] = c.views[k];
        a.v.grad[k] = c.grads ? c.grads[k] : nullptr;
        al = al && aligned(a.v.in[k], 4 * VEC) && (a.v.grad[k] == nullptr || aligned(a.v.grad[k], 4 * VEC));
    }
    a.B = c.B; a.HW = c.HW; a.map = c.map; a.sum = c.sum; a.up = c.up; a.flags = c.flags; a.ws = c.ws;
    const int threads = 256;
    auto go = [&](auto vec_tag) -> int {
        constexpr int V = decltype(vec_tag)::value;
        dim3 grid = image_grid(c.B, c.HW / V, threads);
        if (!fits_partials(grid)) return DCT_ERR_UNSUPPORTED;
#define DCT_JSD_GO(LG, MD) jsd_kernel<K, C, V, LG, MD, (V == 4 ? 3 : 2)><<<grid, threads, 0, c.stream>>>(a)
        if (c.in_kind == DCT_IN_LOGITS) {
            if (c.mode == kFwd) DCT_JSD_GO(true, kFwd);
            else if (c.mode == kBwd) DCT_JSD_GO(true, kBwd);
            else DCT_JSD_GO(true, kFwdBwd);
        } else {
            if (c.mode == kFwd) DCT_JSD_GO(false, kFwd);
            else if (c.mode == kBwd) DCT_JSD_GO(false, kBwd);
            else DCT_JSD_GO(false, kFwdBwd);
        }
#undef DCT_JSD_GO
        return check_launch();
    };
    if (al) return go(std::integral_constant<int, VEC>{});
    return DCT_ERR_UNSUPPORTED;  // odd HW / misaligned views: the caller falls back to jsd_kernel_rt
}

}  // namespace dct
