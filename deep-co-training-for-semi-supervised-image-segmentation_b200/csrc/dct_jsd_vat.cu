// dct_jsd_vat.cu -- the consistency step's JSD launch with the VAT KL folded in (dct_jsd_vat_kl_fwdbwd_f32).
//
// The VAT KL (VATGenerator.kl_div_with_logit(pred.detach(), yhat), AEGenerator.py:93-119) reads pred = the first view's
// logits, which the JSD launch reads as well.  One tile launch over [views..., yhat] reads them once and saves the ~3.5 us
// ramp and drain of a second launch (DESIGN.md 8).  Per pixel it runs the two unchanged op bodies one after the other
// (KlLogit<true> on a copy of view 0 and yhat, then jsd_pixel on the K views), so every value is the one the two
// stand-alone launches produce: bit for bit wherever their tiles have the same shape.
#include <cstring>

#include "dct_jsd_kernels.cuh"
#include "dct_kl_logit.cuh"

namespace dct {

// in[0..K) = the K view logits, in[K] = yhat; out[0..K) = the JSD gradients, out[K] = grad yhat (overwriting the rows read).
// Map value / `sum`: the JSD (upstream g = jsd_gconst); second value / `sum2`: the VAT KL, whose upstream constant travels in
// `eps` (neither body reads eps in logits mode).  grad of pred is not produced: pred is detached.
template <int K, bool DICEF>
struct JsdVatKlOp {
    static constexpr int NIN = K + 1, NOUT = K + 1;
    static constexpr bool HAS_MAP = true, USES_UP = true, CHECKS_SIMPLEX = false, SUM2 = true;
    static constexpr int NDICE = DICEF ? K : 0;
    static constexpr bool GMAP = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&x)[K + 1][CM], int C, T g, float kl_g, bool& bad, T& kl) {
        T kx[2][CM];
#pragma unroll
        for (int c = 0; c < CM; ++c) { kx[0][c] = x[0][c]; kx[1][c] = x[K][c]; }
        kl = KlLogit<true>::template apply<CM, T>(kx, C, vset<T>(kl_g), 0.0f, bad);
        T jx[K][CM];
#pragma unroll
        for (int c = 0; c < CM; ++c) {
            x[K][c] = kx[1][c];
#pragma unroll
            for (int k = 0; k < K; ++k) jx[k][c] = x[k][c];
        }
        const T j = JsdOp<K, true, kFwdBwd, false>::template apply<CM, T>(jx, C, g, 0.0f, bad);
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int c = 0; c < CM; ++c) x[k][c] = jx[k][c];
        return j;
    }
};

template <int K, int C, bool DICEF>
static int jsd_vat_kl_launch(TileArgs& a, int64_t B, bool pub, cudaStream_t stream) {
    using Op = JsdVatKlOp<K, DICEF>;
    static_assert((K + 1) * C <= 16 && C <= 4, "the fused launch is instantiated for the 5-16-row stages only");
    if (!tile_eligible<Op>(a, B)) return DCT_ERR_UNSUPPORTED;
    return pub ? tile_launch_ct<Op, C, float, true>(a, B, stream) : tile_launch_ct<Op, C, float, false>(a, B, stream);
}

template <int K, int C>
static int jsd_vat_kl_kc(TileArgs& a, int64_t B, bool pub, cudaStream_t stream) {
    return a.labels != nullptr ? jsd_vat_kl_launch<K, C, true>(a, B, pub, stream) : jsd_vat_kl_launch<K, C, false>(a, B, pub, stream);
}

// DCT_ERR_UNSUPPORTED (nothing launched) when the shape is outside the fused launch's bracket
static int jsd_vat_kl_tile(TileArgs& a, int K, int C, int64_t B, bool pub, cudaStream_t stream) {
    switch (K * 8 + C) {
        case 2 * 8 + 2: return jsd_vat_kl_kc<2, 2>(a, B, pub, stream);
        case 2 * 8 + 3: return jsd_vat_kl_kc<2, 3>(a, B, pub, stream);
        case 2 * 8 + 4: return jsd_vat_kl_kc<2, 4>(a, B, pub, stream);
        case 3 * 8 + 2: return jsd_vat_kl_kc<3, 2>(a, B, pub, stream);
        case 3 * 8 + 3: return jsd_vat_kl_kc<3, 3>(a, B, pub, stream);
        case 3 * 8 + 4: return jsd_vat_kl_kc<3, 4>(a, B, pub, stream);
        case 4 * 8 + 2: return jsd_vat_kl_kc<4, 2>(a, B, pub, stream);
        case 4 * 8 + 3: return jsd_vat_kl_kc<4, 3>(a, B, pub, stream);
        default: return DCT_ERR_UNSUPPORTED;
    }
}

}  // namespace dct

using namespace dct;

extern "C" int dct_jsd_vat_kl_fwdbwd_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, float jsd_gconst,
                                         double* jsd_sum, float* const* grad_views, const int64_t* labels, int64_t* counts,
                                         int counts_mode, const float* yhat, float kl_gconst, double* kl_sum, float* grad_yhat,
                                         int32_t* flags, void* workspace, const dct_peer_pub* pub_desc, void* stream) {
    // everything either half would refuse is refused before anything is launched
    if (views == nullptr || grad_views == nullptr || yhat == nullptr || K < 1 || C < 1 || B < 1 || HW < 1) return DCT_ERR_BAD_ARG;
    if (K > DCT_MAX_VIEWS || C > DCT_MAX_CLASSES || B > 65535) return DCT_ERR_UNSUPPORTED;
    for (int k = 0; k < K; ++k) {
        if (views[k] == nullptr || grad_views[k] == nullptr) return DCT_ERR_BAD_ARG;
        if (!aligned(views[k], 4) || !aligned(grad_views[k], 4)) return DCT_ERR_MISALIGNED;
    }
    if (!aligned(yhat, 4)) return DCT_ERR_MISALIGNED;
    if ((jsd_sum != nullptr || kl_sum != nullptr) && workspace == nullptr) return DCT_ERR_BAD_ARG;
    if (labels != nullptr && counts == nullptr) return DCT_ERR_BAD_ARG;
    if (counts_mode != DCT_COUNTS_ACCUMULATE && counts_mode != DCT_COUNTS_OVERWRITE) return DCT_ERR_BAD_ARG;
    if (labels != nullptr && counts_mode == DCT_COUNTS_OVERWRITE && workspace == nullptr) return DCT_ERR_BAD_ARG;
    if (pub_desc != nullptr) {
        const int prc = check_pub(pub_desc);
        if (prc != DCT_OK) return prc;
    }
    // the fused launch: 5-16-row stages ((K + 1) * C <= 16, C <= 4); it needs the workspace for its schedule and publication
    if ((K + 1) * C <= 16 && C <= 4 && workspace != nullptr) {
        TileArgs a{};
        for (int k = 0; k < K; ++k) {
            a.in[k] = views[k];
            a.out[k] = grad_views[k];
        }
        a.in[K] = yhat;
        a.out[K] = grad_yhat;
        a.HW = HW; a.map = nullptr; a.sum = jsd_sum; a.sum2 = kl_sum; a.up = Upstream{nullptr, nullptr, jsd_gconst};
        a.eps = kl_gconst; a.flags = flags; a.ws = static_cast<Workspace*>(workspace);
        a.labels = labels; a.counts = reinterpret_cast<unsigned long long*>(counts); a.count_view_stride = B * C * 3;
        a.counts_overwrite = counts_mode == DCT_COUNTS_OVERWRITE ? 1 : 0;
        if (pub_desc != nullptr) {
            std::memcpy(&a.pub, pub_desc, sizeof(a.pub));
            a.pub_early = 1;
        }
        const int rc = jsd_vat_kl_tile(a, K, C, B, pub_desc != nullptr, static_cast<cudaStream_t>(stream));
        if (rc != DCT_ERR_UNSUPPORTED) return rc;
    }
    // outside the fused bracket (shape, alignment, HW % 4, a refused tensor-map encode): the two stand-alone launches
    int rc = pub_desc != nullptr
                 ? dct_jsd_fwdbwd_pub_f32(views, K, C, B, HW, DCT_IN_LOGITS, jsd_gconst, nullptr, jsd_sum, grad_views, labels,
                                          counts, counts_mode, flags, workspace, pub_desc, stream)
                 : dct_jsd_fwdbwd_f32(views, K, C, B, HW, DCT_IN_LOGITS, jsd_gconst, nullptr, jsd_sum, grad_views, labels,
                                      counts, counts_mode, flags, workspace, stream);
    if (rc != DCT_OK) return rc;
    return dct_kl_logit_f32(views[0], yhat, C, B, HW, nullptr, kl_sum, 1, nullptr, nullptr, kl_gconst, grad_yhat, nullptr,
                            workspace, stream);
}
