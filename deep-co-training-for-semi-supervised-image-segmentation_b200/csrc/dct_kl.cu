// dct_kl.cu -- the adversarial branch's KL family, entropy and softmax as pixelwise ops
// (dct_pixelwise.cuh) plus their C-ABI entry points (include/dct_b200.h).
#include <cstring>

#include "dct_kl_logit.cuh"
#include "dct_pixelwise.cuh"

namespace dct {

// KL_Divergence_2D.forward -- generalframework/loss/loss.py:117-134
struct KlProbFwd {
    static constexpr int NIN = 2, NOUT = 0;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = false;
    static constexpr bool HAS_MAP = true, USES_UP = false, CHECKS_SIMPLEX = true;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[2][CM], int C, T, float eps, bool& bad) {
        T yy = vset<T>(0.0f), yp = vset<T>(0.0f), sp = vset<T>(0.0f), sy = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                T pv = x[0][c], yv = x[1][c];
                sp = vadd(sp, pv); sy = vadd(sy, yv);
                yy = vfma(yv, vlog(vadds(yv, eps)), yy);
                yp = vfma(yv, vlog(vadds(pv, eps)), yp);
            }
        bad |= vsimplex_bad(sp) | vsimplex_bad(sy);
        return vsub(yy, yp);
    }
};

// its derivative: d/dp = -y/(p+eps); d/dy = log(y+eps) + y/(y+eps) - log(p+eps)
template <bool WANT_Y>
struct KlProbBwd {
    static constexpr int NIN = 2, NOUT = 2;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = true;
    static constexpr bool HAS_MAP = false, USES_UP = true, CHECKS_SIMPLEX = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[2][CM], int C, T g, float eps, bool&) {
        const T ng = vneg(g);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                T pv = x[0][c], yv = x[1][c];
                T pe = vadds(pv, eps);
                x[0][c] = vmul(ng, vdiv(yv, pe));
                if constexpr (WANT_Y) {
                    T ye = vadds(yv, eps);
                    x[1][c] = vmul(g, vsub(vadd(vlog(ye), vdiv(yv, ye)), vlog(pe)));
                }
            }
        return vset<T>(0.0f);
    }
};

// KL_Divergence_2D(reduce=True)(softmax(p_logit), y.detach()) + backward to p_logit in one pass
// (generalframework/trainer/cotraining_totalloss.py:391-392).  in[0] = p_logit, in[1] = y_prob; out[0] = grad p_logit.
struct KlFromLogits {
    static constexpr int NIN = 2, NOUT = 1;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = false;
    static constexpr bool HAS_MAP = true, USES_UP = true, CHECKS_SIMPLEX = true;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[2][CM], int C, T g, float eps, bool& bad) {
        T e[CM];
        T inv, lZ;
        softmax_stats<CM, T>(x[0], e, C, inv, lZ);
        const T ng = vneg(g);
        T yy = vset<T>(0.0f), yp = vset<T>(0.0f), sy = vset<T>(0.0f), dot = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                T pv = vmul(e[c], inv), yv = x[1][c];
                sy = vadd(sy, yv);
                T pe = vadds(pv, eps);
                yy = vfma(yv, vlog(vadds(yv, eps)), yy);
                yp = vfma(yv, vlog(pe), yp);
                T gp = vmul(ng, vdiv(yv, pe));
                e[c] = pv;
                x[0][c] = gp;
                dot = vfma(pv, gp, dot);
            }
        bad |= vsimplex_bad(sy);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) x[0][c] = vmul(e[c], vsub(x[0][c], dot));
        return vsub(yy, yp);
    }
};

// KL_div.forward -- loss.py:99-107: sum_c -p*log(q/p + eps)
struct KlDivFwd {
    static constexpr int NIN = 2, NOUT = 0;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = false;
    static constexpr bool HAS_MAP = true, USES_UP = false, CHECKS_SIMPLEX = true;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[2][CM], int C, T, float eps, bool& bad) {
        T s = vset<T>(0.0f), sp = vset<T>(0.0f), sq = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                T pv = x[0][c], qv = x[1][c];
                sp = vadd(sp, pv); sq = vadd(sq, qv);
                // IEEE divide and libdevice logf: 0/0 -> NaN exactly like the reference
                T l = vmap([eps](float q, float p) { return logf(q / p + eps); }, qv, pv);
                s = vfma(vneg(pv), l, s);
            }
        bad |= vsimplex_bad(sp) | vsimplex_bad(sq);
        return s;
    }
};

// its derivative (what autograd builds for loss.py:105): with r = q/p and u = r + eps,
//   d/dp_c = -(log u) + r/u        d/dq_c = -1/u
// IEEE divide / libdevice logf like the forward (p == 0 gives the reference's NaN / inf pattern, not a fast-math variant)
template <bool WANT_Q>
struct KlDivBwd {
    static constexpr int NIN = 2, NOUT = 2;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = true;
    static constexpr bool HAS_MAP = false, USES_UP = true, CHECKS_SIMPLEX = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[2][CM], int C, T g, float eps, bool&) {
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                const T pv = x[0][c], qv = x[1][c];
                const T r = vmap([](float q, float p) { return q / p; }, qv, pv);
                const T u = vadds(r, eps);
                const T dp = vmap([](float rr, float uu) { return rr / uu - logf(uu); }, r, u);
                x[0][c] = vmul(g, dp);
                if constexpr (WANT_Q) x[1][c] = vmul(g, vmap([](float uu, float) { return -1.0f / uu; }, u, u));
            }
        return vset<T>(0.0f);
    }
};

// Entropy_2D / Entropy forward -- loss.py:53-84
struct EntropyFwd {
    static constexpr int NIN = 1, NOUT = 0;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = false;
    static constexpr bool HAS_MAP = true, USES_UP = false, CHECKS_SIMPLEX = true;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[1][CM], int C, T, float, bool& bad) {
        T h = vset<T>(0.0f), s = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                T pv = x[0][c];
                s = vadd(s, pv);
                h = vfma(pv, vlog(vadds(pv, kEntEps)), h);
            }
        bad |= vsimplex_bad(s);
        return vneg(h);
    }
};
struct EntropyBwd {
    static constexpr int NIN = 1, NOUT = 1;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = true;
    static constexpr bool HAS_MAP = false, USES_UP = true, CHECKS_SIMPLEX = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[1][CM], int C, T g, float, bool&) {
        const T ng = vneg(g);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                T pv = x[0][c];
                T pe = vadds(pv, kEntEps);
                x[0][c] = vmul(ng, vadd(vlog(pe), vdiv(pv, pe)));
            }
        return vset<T>(0.0f);
    }
};

// F.softmax(x, 1) as a standalone product op uses the accurate libdevice expf and IEEE division
struct SoftmaxFwd {
    static constexpr int NIN = 1, NOUT = 1;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = false;
    static constexpr bool HAS_MAP = false, USES_UP = false, CHECKS_SIMPLEX = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[1][CM], int C, T, float, bool&) {
        T mx = x[0][0];
#pragma unroll
        for (int c = 1; c < CM; ++c)
            if (c < C) mx = vmax(mx, x[0][c]);
        T Z = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) {
                x[0][c] = vmap([](float a, float m) { return expf(a - m); }, x[0][c], mx);
                Z = vadd(Z, x[0][c]);
            }
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) x[0][c] = vmap([](float a, float z) { return a / z; }, x[0][c], Z);
        return vset<T>(0.0f);
    }
};
struct SoftmaxBwd {  // in[0] = p, in[1] = gp ; out[0] = gx
    static constexpr int NIN = 2, NOUT = 1;
    static constexpr int NDICE = 0;
    static constexpr bool GMAP = false;
    static constexpr bool HAS_MAP = false, USES_UP = false, CHECKS_SIMPLEX = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[2][CM], int C, T, float, bool&) {
        T dot = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) dot = vfma(x[0][c], x[1][c], dot);
#pragma unroll
        for (int c = 0; c < CM; ++c)
            if (c < C) x[0][c] = vmul(x[0][c], vsub(x[1][c], dot));
        return vset<T>(0.0f);
    }
};

static PixArgs make_args(const float* in0, const float* in1, float* out0, float* out1, int C, int64_t HW, float* map,
                         double* sum, Upstream up, float eps, int32_t* flags, void* ws) {
    PixArgs a;
    a.in[0] = in0; a.in[1] = in1; a.out[0] = out0; a.out[1] = out1;
    a.C = C; a.HW = HW; a.map = map; a.sum = sum; a.up = up; a.eps = eps; a.flags = flags;
    a.ws = static_cast<Workspace*>(ws);
    return a;
}

// bf16 tensors: the tile pipeline only (DCT_ERR_UNSUPPORTED otherwise: the caller converts to float32)
template <class Op>
static int tile_bf16(const void* in0, const void* in1, void* out0, void* out1, int C, int64_t B, int64_t HW, float* map,
                     double* sum, Upstream up, float eps, int32_t* flags, void* ws, cudaStream_t stream) {
    if (in0 == nullptr || (Op::NIN > 1 && in1 == nullptr) || C < 1 || B < 1 || HW < 1) return DCT_ERR_BAD_ARG;
    if (Op::HAS_MAP && sum != nullptr && ws == nullptr) return DCT_ERR_BAD_ARG;
    if (B > 65535) return DCT_ERR_UNSUPPORTED;
    TileArgs t{};
    t.in[0] = in0; t.in[1] = in1; t.out[0] = out0; t.out[1] = out1;
    t.HW = HW; t.map = map; t.sum = sum; t.up = up; t.eps = eps; t.flags = flags; t.ws = static_cast<Workspace*>(ws);
    if (!tile_eligible<Op, bf16>(t, B)) return DCT_ERR_UNSUPPORTED;
    switch (C) {
        case 2: return tile_launch_ct<Op, 2, bf16>(t, B, stream);
        case 3: return tile_launch_ct<Op, 3, bf16>(t, B, stream);
        case 4: return tile_launch_ct<Op, 4, bf16>(t, B, stream);
        case 19: return tile_launch_ct<Op, 19, bf16>(t, B, stream);
        default: return DCT_ERR_UNSUPPORTED;
    }
}

}  // namespace dct

using namespace dct;

extern "C" int dct_kl_fwd_f32(const float* p, const float* y, int C, int64_t B, int64_t HW, float eps, float* map,
                              double* sum, int32_t* flags, void* workspace, void* stream) {
    PixArgs a = make_args(p, y, nullptr, nullptr, C, HW, map, sum, Upstream{nullptr, nullptr, 1.0f}, eps, flags, workspace);
    return pix_launch<KlProbFwd>(a, B, static_cast<cudaStream_t>(stream));
}

extern "C" int dct_kl_bwd_f32(const float* p, const float* y, int C, int64_t B, int64_t HW, float eps,
                              const float* gmap, const float* gscalar, float gconst, float* grad_p, float* grad_y,
                              void* stream) {
    PixArgs a = make_args(p, y, grad_p, grad_y, C, HW, nullptr, nullptr, Upstream{gmap, gscalar, gconst}, eps, nullptr, nullptr);
    if (grad_y != nullptr) return pix_launch<KlProbBwd<true>>(a, B, static_cast<cudaStream_t>(stream));
    return pix_launch<KlProbBwd<false>>(a, B, static_cast<cudaStream_t>(stream));
}

extern "C" int dct_kl_logit_f32(const float* q_logit, const float* p_logit, int C, int64_t B, int64_t HW, float* map,
                                double* sum, int has_upstream, const float* gmap, const float* gscalar, float gconst,
                                float* grad_p_logit, float* grad_q_logit, void* workspace, void* stream) {
    PixArgs a = make_args(q_logit, p_logit, grad_q_logit, grad_p_logit, C, HW, map, sum,
                          Upstream{gmap, gscalar, gconst}, 0.0f, nullptr, workspace);
    if (has_upstream) return pix_launch<KlLogit<true>>(a, B, static_cast<cudaStream_t>(stream));
    a.out[0] = a.out[1] = nullptr;
    return pix_launch<KlLogit<false>>(a, B, static_cast<cudaStream_t>(stream));
}

extern "C" int dct_kl_from_logits_fwdbwd_f32(const float* p_logit, const float* y_prob, int C, int64_t B, int64_t HW,
                                             float eps, float gconst, float* map, double* sum, float* grad_p_logit,
                                             int32_t* flags, void* workspace, void* stream) {
    PixArgs a = make_args(p_logit, y_prob, grad_p_logit, nullptr, C, HW, map, sum, Upstream{nullptr, nullptr, gconst},
                          eps, flags, workspace);
    return pix_launch<KlFromLogits>(a, B, static_cast<cudaStream_t>(stream));
}

#ifndef DCT_KBENCH  // (tools/kbench_tile.cu includes this file without dct_abi.cu)
// The adversarial KL is the LAST kernel of a consistency step (JSD -> VAT -> KL): this variant's last CTA also pushes the
// step's loss sums into every data-parallel rank's mailbox over NVLink (include/dct_b200.h, "Fused cross-rank exchange").
extern "C" int dct_kl_from_logits_fwdbwd_pub_f32(const float* p_logit, const float* y_prob, int C, int64_t B, int64_t HW,
                                                 float eps, float gconst, float* map, double* sum, float* grad_p_logit,
                                                 int32_t* flags, void* workspace, const dct_peer_pub* pub_desc,
                                                 void* stream) {
    if (sum == nullptr) return DCT_ERR_BAD_ARG;
    int prc = check_pub(pub_desc);
    if (prc != DCT_OK) return prc;
    PixArgs a = make_args(p_logit, y_prob, grad_p_logit, nullptr, C, HW, map, sum, Upstream{nullptr, nullptr, gconst},
                          eps, flags, workspace);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (C >= 1 && B >= 1 && HW >= 1 && p_logit != nullptr && y_prob != nullptr && workspace != nullptr && B <= 65535) {
        TileArgs t{};
        t.in[0] = a.in[0]; t.in[1] = a.in[1]; t.out[0] = a.out[0];
        t.HW = a.HW; t.map = a.map; t.sum = a.sum; t.up = a.up; t.eps = a.eps; t.flags = a.flags; t.ws = a.ws;
        std::memcpy(&t.pub, pub_desc, sizeof(t.pub));
        if (tile_eligible<KlFromLogits>(t, B)) {
            switch (C) {
                case 2: return tile_launch_ct<KlFromLogits, 2, float, true>(t, B, st);
                case 3: return tile_launch_ct<KlFromLogits, 3, float, true>(t, B, st);
                case 4: return tile_launch_ct<KlFromLogits, 4, float, true>(t, B, st);
                case 19: return tile_launch_ct<KlFromLogits, 19, float, true>(t, B, st);
                default: break;
            }
        }
    }
    // shapes outside the tile pipeline: the plain kernels, then the stand-alone publication
    int rc = pix_launch<KlFromLogits>(a, B, st);
    if (rc != DCT_OK) return rc;
    return dct_exchange_publish(pub_desc, stream);
}

#endif  // DCT_KBENCH

extern "C" int dct_kl_div_fwd_f32(const float* p, const float* q, int C, int64_t B, int64_t HW, float eps, float* map,
                                  double* sum, int32_t* flags, void* workspace, void* stream) {
    PixArgs a = make_args(p, q, nullptr, nullptr, C, HW, map, sum, Upstream{nullptr, nullptr, 1.0f}, eps, flags, workspace);
    return pix_launch<KlDivFwd>(a, B, static_cast<cudaStream_t>(stream));
}

extern "C" int dct_kl_div_bwd_f32(const float* p, const float* q, int C, int64_t B, int64_t HW, float eps,
                                  const float* gmap, const float* gscalar, float gconst, float* grad_p, float* grad_q,
                                  void* stream) {
    if (grad_p == nullptr) return DCT_ERR_BAD_ARG;
    PixArgs a = make_args(p, q, grad_p, grad_q, C, HW, nullptr, nullptr, Upstream{gmap, gscalar, gconst}, eps, nullptr, nullptr);
    if (grad_q != nullptr) return pix_launch<KlDivBwd<true>>(a, B, static_cast<cudaStream_t>(stream));
    return pix_launch<KlDivBwd<false>>(a, B, static_cast<cudaStream_t>(stream));
}

extern "C" int dct_entropy_fwd_f32(const float* p, int C, int64_t B, int64_t HW, float* map, double* sum,
                                   int32_t* flags, void* workspace, void* stream) {
    PixArgs a = make_args(p, nullptr, nullptr, nullptr, C, HW, map, sum, Upstream{nullptr, nullptr, 1.0f}, 0.0f, flags, workspace);
    return pix_launch<EntropyFwd>(a, B, static_cast<cudaStream_t>(stream));
}

extern "C" int dct_entropy_bwd_f32(const float* p, int C, int64_t B, int64_t HW, const float* gmap,
                                   const float* gscalar, float gconst, float* grad_p, void* stream) {
    if (grad_p == nullptr) return DCT_ERR_BAD_ARG;
    PixArgs a = make_args(p, nullptr, grad_p, nullptr, C, HW, nullptr, nullptr, Upstream{gmap, gscalar, gconst}, 0.0f, nullptr, nullptr);
    return pix_launch<EntropyBwd>(a, B, static_cast<cudaStream_t>(stream));
}

extern "C" int dct_softmax_fwd_f32(const float* x, int C, int64_t B, int64_t HW, float* p, void* stream) {
    if (p == nullptr) return DCT_ERR_BAD_ARG;
    PixArgs a = make_args(x, nullptr, p, nullptr, C, HW, nullptr, nullptr, Upstream{nullptr, nullptr, 1.0f}, 0.0f, nullptr, nullptr);
    return pix_launch<SoftmaxFwd>(a, B, static_cast<cudaStream_t>(stream));
}

extern "C" int dct_softmax_bwd_f32(const float* p, const float* gp, int C, int64_t B, int64_t HW, float* gx, void* stream) {
    if (gx == nullptr) return DCT_ERR_BAD_ARG;
    PixArgs a = make_args(p, gp, gx, nullptr, C, HW, nullptr, nullptr, Upstream{nullptr, nullptr, 1.0f}, 0.0f, nullptr, nullptr);
    return pix_launch<SoftmaxBwd>(a, B, static_cast<cudaStream_t>(stream));
}

// ---- bf16 twins of the two one-pass-over-logits ops of the adversarial branch (fp32 math, fp32 map / sum) ----
extern "C" int dct_kl_logit_bf16(const void* q_logit, const void* p_logit, int C, int64_t B, int64_t HW, float* map,
                                 double* sum, int has_upstream, const float* gmap, const float* gscalar, float gconst,
                                 void* grad_p_logit, void* grad_q_logit, void* workspace, void* stream) {
    const Upstream up{gmap, gscalar, gconst};
    if (has_upstream)
        return tile_bf16<KlLogit<true>>(q_logit, p_logit, grad_q_logit, grad_p_logit, C, B, HW, map, sum, up, 0.0f, nullptr,
                                        workspace, static_cast<cudaStream_t>(stream));
    return tile_bf16<KlLogit<false>>(q_logit, p_logit, nullptr, nullptr, C, B, HW, map, sum, up, 0.0f, nullptr, workspace,
                                     static_cast<cudaStream_t>(stream));
}

extern "C" int dct_kl_from_logits_fwdbwd_bf16(const void* p_logit, const void* y_prob, int C, int64_t B, int64_t HW,
                                              float eps, float gconst, float* map, double* sum, void* grad_p_logit,
                                              int32_t* flags, void* workspace, void* stream) {
    return tile_bf16<KlFromLogits>(p_logit, y_prob, grad_p_logit, nullptr, C, B, HW, map, sum,
                                   Upstream{nullptr, nullptr, gconst}, eps, flags, workspace, static_cast<cudaStream_t>(stream));
}
