// dct_jsd.cu -- C-ABI entry points of the JSD family (include/dct_b200.h), argument validation and
// dispatch to the register-tiled instantiations (dct_jsd_k*.cu) or the runtime-(K,C) fallback.
#include "dct_jsd_kernels.cuh"

namespace dct {

static int jsd_launch_rt(const JsdCall& c) {
    JsdArgsRt a;
    for (int k = 0; k < DCT_MAX_VIEWS; ++k) {
        a.in[k] = k < c.K ? c.views[k] : nullptr;
        a.grad[k] = (k < c.K && c.grads) ? c.grads[k] : nullptr;
    }
    a.K = c.K; a.C = c.C; a.B = c.B; a.HW = c.HW; a.map = c.map; a.sum = c.sum; a.up = c.up; a.flags = c.flags; a.ws = c.ws;
    const int threads = 256;
    dim3 grid = image_grid(c.B, c.HW, threads);
    if (!fits_partials(grid)) return DCT_ERR_UNSUPPORTED;
#define DCT_JSD_RT(LG, MD) jsd_kernel_rt<LG, MD><<<grid, threads, 0, c.stream>>>(a)
    if (c.in_kind == DCT_IN_LOGITS) {
        if (c.mode == kFwd) DCT_JSD_RT(true, kFwd);
        else if (c.mode == kBwd) DCT_JSD_RT(true, kBwd);
        else DCT_JSD_RT(true, kFwdBwd);
    } else {
        if (c.mode == kFwd) DCT_JSD_RT(false, kFwd);
        else if (c.mode == kBwd) DCT_JSD_RT(false, kBwd);
        else DCT_JSD_RT(false, kFwdBwd);
    }
#undef DCT_JSD_RT
    return check_launch();
}

static int jsd_dispatch(const JsdCall& c) {
    if (c.views == nullptr || c.K < 1 || c.C < 1 || c.B < 1 || c.HW < 1) return DCT_ERR_BAD_ARG;
    if (c.K > DCT_MAX_VIEWS || c.C > DCT_MAX_CLASSES || c.B > 65535) return DCT_ERR_UNSUPPORTED;
    if (c.in_kind != DCT_IN_PROBS && c.in_kind != DCT_IN_LOGITS) return DCT_ERR_BAD_ARG;
    for (int k = 0; k < c.K; ++k) {
        if (c.views[k] == nullptr) return DCT_ERR_BAD_ARG;
        if (!aligned(c.views[k], 4)) return DCT_ERR_MISALIGNED;
        if (c.mode != kFwd) {
            if (c.grads == nullptr || c.grads[k] == nullptr) return DCT_ERR_BAD_ARG;
            if (!aligned(c.grads[k], 4)) return DCT_ERR_MISALIGNED;
        }
    }
    if (c.mode != kBwd && c.sum != nullptr && c.ws == nullptr) return DCT_ERR_BAD_ARG;
    int rc = DCT_ERR_UNSUPPORTED;
    switch (c.K) {
        case 2: rc = jsd_launch_k2(c); break;
        case 3: rc = jsd_launch_k3(c); break;
        case 4: rc = jsd_launch_k4(c); break;
        default: break;
    }
    if (rc == DCT_ERR_UNSUPPORTED && c.elem == 0) rc = jsd_launch_rt(c);
    return rc;
}

}  // namespace dct

using namespace dct;

extern "C" int dct_jsd_fwd_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                               float* map, double* sum, int32_t* flags, void* workspace, void* stream) {
    JsdCall c{nullptr, nullptr, nullptr, views, nullptr, K, C, B, HW, in_kind, kFwd, map, sum, Upstream{nullptr, nullptr, 0.0f}, flags,
              static_cast<Workspace*>(workspace), static_cast<cudaStream_t>(stream)};
    return jsd_dispatch(c);
}

extern "C" int dct_jsd_bwd_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                               const float* gmap, const float* gscalar, float gconst, float* const* grad_views,
                               void* stream) {
    JsdCall c{nullptr, nullptr, nullptr, views, grad_views, K, C, B, HW, in_kind, kBwd, nullptr, nullptr, Upstream{gmap, gscalar, gconst},
              nullptr, nullptr, static_cast<cudaStream_t>(stream)};
    return jsd_dispatch(c);
}

static int jsd_fwdbwd_f32_impl(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                               float gconst, float* map, double* sum, float* const* grad_views,
                               const int64_t* labels, int64_t* counts, int counts_mode, int32_t* flags,
                               void* workspace, const dct_peer_pub* pub, void* stream) {
    if (labels != nullptr && counts == nullptr) return DCT_ERR_BAD_ARG;
    if (counts_mode != DCT_COUNTS_ACCUMULATE && counts_mode != DCT_COUNTS_OVERWRITE) return DCT_ERR_BAD_ARG;
    if (labels != nullptr && counts_mode == DCT_COUNTS_OVERWRITE && workspace == nullptr) return DCT_ERR_BAD_ARG;
    bool dice_done = false;
    JsdCall c{labels, counts, &dice_done, views, grad_views, K, C, B, HW, in_kind, kFwdBwd, map, sum,
              Upstream{nullptr, nullptr, gconst}, flags, static_cast<Workspace*>(workspace),
              static_cast<cudaStream_t>(stream)};
    c.counts_overwrite = counts_mode == DCT_COUNTS_OVERWRITE;
    bool pub_done = false;
    c.pub = pub;
    c.pub_done = &pub_done;
    int rc = jsd_dispatch(c);
    if (rc != DCT_OK) return rc;
    if (pub != nullptr && !pub_done) {   // shapes outside the tile pipeline: the stand-alone publication behind the launch
        rc = dct_exchange_publish(pub, stream);
        if (rc != DCT_OK) return rc;
    }
    if (labels != nullptr && !dice_done) {
        // Dice counting of the K views against the same labels (unlabdiceMeters,
        // generalframework/trainer/cotraining_totalloss.py:224).  C <= 4 with aligned rows is fused
        // into the loss kernel itself (JsdOp<.., DICEF>); other shapes count in K extra launches.
        for (int k = 0; k < K; ++k) {
            rc = dct_dice_counts_f32(views[k], labels, C, B, HW, counts + (int64_t)k * B * C * 3,
                                     counts_mode == DCT_COUNTS_OVERWRITE ? 0 : 1, flags, stream);
            if (rc != DCT_OK) return rc;
        }
    }
    return DCT_OK;
}

extern "C" int dct_jsd_fwdbwd_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                                  float gconst, float* map, double* sum, float* const* grad_views,
                                  const int64_t* labels, int64_t* counts, int counts_mode, int32_t* flags,
                                  void* workspace, void* stream) {
    return jsd_fwdbwd_f32_impl(views, K, C, B, HW, in_kind, gconst, map, sum, grad_views, labels, counts, counts_mode, flags,
                               workspace, nullptr, stream);
}

// The fused JSD launch is the FIRST kernel of a consistency step: this variant also carries the publication of sums that
// were final before the launch (the previous step's): its first finishing CTA pushes them into every rank's mailbox while
// the rest of the grid is still working (include/dct_b200.h, "Fused cross-rank exchange").
extern "C" int dct_jsd_fwdbwd_pub_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                                      float gconst, float* map, double* sum, float* const* grad_views,
                                      const int64_t* labels, int64_t* counts, int counts_mode, int32_t* flags,
                                      void* workspace, const dct_peer_pub* pub_desc, void* stream) {
    const int prc = check_pub(pub_desc);
    if (prc != DCT_OK) return prc;
    return jsd_fwdbwd_f32_impl(views, K, C, B, HW, in_kind, gconst, map, sum, grad_views, labels, counts, counts_mode, flags,
                               workspace, pub_desc, stream);
}

// bf16 tensors (networks under autocast): logits in, fp32 math in registers, bf16 gradients out; the tile pipeline
// only.  grad_views == NULL: forward only (evaluation).  Returns DCT_ERR_UNSUPPORTED for shapes outside the pipeline
// (K*C > 80, C not in {2,3,4,19}, HW % 8 != 0, rows not 16-byte aligned): the caller converts to float32 then.
extern "C" int dct_jsd_fwdbwd_bf16(const void* const* views, int K, int C, int64_t B, int64_t HW, float gconst,
                                   float* map, double* sum, void* const* grad_views, const int64_t* labels,
                                   int64_t* counts, int counts_mode, int32_t* flags, void* workspace, void* stream) {
    if (labels != nullptr && counts == nullptr) return DCT_ERR_BAD_ARG;
    if (counts_mode != DCT_COUNTS_ACCUMULATE && counts_mode != DCT_COUNTS_OVERWRITE) return DCT_ERR_BAD_ARG;
    if (labels != nullptr && counts_mode == DCT_COUNTS_OVERWRITE && workspace == nullptr) return DCT_ERR_BAD_ARG;
    if (labels != nullptr && (C > 4 || !aligned(labels, 16) || grad_views == nullptr)) return DCT_ERR_UNSUPPORTED;
    bool dice_done = false;
    JsdCall c{labels, counts, &dice_done, reinterpret_cast<const float* const*>(views),
              reinterpret_cast<float* const*>(grad_views), K, C, B, HW, DCT_IN_LOGITS, grad_views ? kFwdBwd : kFwd, map, sum,
              Upstream{nullptr, nullptr, gconst}, flags, static_cast<Workspace*>(workspace),
              static_cast<cudaStream_t>(stream), 1};
    c.counts_overwrite = counts_mode == DCT_COUNTS_OVERWRITE;
    int rc = jsd_dispatch(c);
    if (rc == DCT_OK && labels != nullptr && !dice_done) return DCT_ERR_UNSUPPORTED;  // (not reachable: C <= 4 fuses)
    return rc;
}
