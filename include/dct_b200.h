/*
 * dct_b200.h -- C ABI of libdct_b200.so: the B200 (sm_100a) kernels for the
 * consistency hot path of Deep Co-Training for semi-supervised segmentation.
 *
 * The reference (jizongFox/Deep-Co-Training-for-Semi-Supervised-Image-Segmentation,
 * pure Python/PyTorch) has no FFI: its "plugin interface" for this path is the
 * set of duck-typed Python objects the trainers call (SURVEY.md section 8b).  Each
 * entry point below names the reference function(s) it replaces, as file:line
 * into the reference tree.  The Python mirror of the reference interface lives in
 * deep-co-training-for-semi-supervised-image-segmentation_b200/ and calls ONLY
 * these functions (ctypes); INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer unless marked "host".  Tensors are NCHW
 *    contiguous float32: element (b,c,i) of a [B,C,HW] tensor at (b*C+c)*HW+i;
 *    maps are [B,HW] float32; labels are [B,HW] int64 (the reference's dtype).
 *  - No allocation, no ownership transfer, no global state, re-entrant.  All
 *    buffers belong to the caller and must stay alive until the stream reaches
 *    the end of the call's work.  Calls enqueue on `stream` (a cudaStream_t,
 *    NULL = legacy default stream) and never synchronise.
 *  - `workspace`: >= dct_workspace_bytes() bytes, zero-initialised ONCE by the
 *    caller, private to one stream at a time (kernels leave it zeroed again).
 *  - `flags`: int32[DCT_NUM_FLAGS], caller-zeroed; kernels only ever add to it.
 *      flags[DCT_FLAG_SIMPLEX]  += #pixels whose class sum fails the reference's
 *                                  utils.simplex allclose(sum,1) (utils/utils.py:142-151)
 *      flags[DCT_FLAG_LABEL]    += #labels outside [0,C) (class2one_hot's assert, utils.py:190)
 *      flags[DCT_FLAG_PRED]     += #integer predictions outside [0,C) (ConfusionMatrix's bincount assert)
 *      flags[DCT_FLAG_ONEHOT]   += #violations of utils.one_hot (a value outside {0,1}, or a pixel whose class
 *                                  column does not hold exactly one 1; utils.py:154-161)
 *    May be NULL (checks compiled out of the launch).
 *  - Upstream gradient of a [B,HW] map output ("dct_upstream"): the per-pixel
 *    incoming gradient is   gconst * (gscalar ? *gscalar : 1) * (gmap ? gmap[b,i] : 1).
 *  - Return value: DCT_OK (0) or a negative DCT_ERR_* code; nothing was launched
 *    on error except where noted.
 */
#ifndef DCT_B200_H
#define DCT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCT_ABI_VERSION 2

#if defined(__GNUC__)
#define DCT_API __attribute__((visibility("default")))
#else
#define DCT_API
#endif

enum {
    DCT_OK = 0,
    DCT_ERR_BAD_ARG = -1,      /* null pointer / non-positive size / K or C out of range */
    DCT_ERR_UNSUPPORTED = -2,  /* shape not supported by any kernel (K > 8 or C > 64) */
    DCT_ERR_MISALIGNED = -3,   /* a pointer is not 4-byte (float) / 8-byte (int64) aligned */
    DCT_ERR_CUDA = -4,         /* the launch itself failed; see dct_last_cuda_error() */
    DCT_ERR_NO_DEVICE = -5     /* no CUDA device / not an sm_100 device */
};

enum { DCT_FLAG_SIMPLEX = 0, DCT_FLAG_LABEL = 1, DCT_FLAG_PRED = 2, DCT_FLAG_ONEHOT = 3, DCT_NUM_FLAGS = 4 };

/* input kind of the K view tensors handed to the JSD entry points */
enum { DCT_IN_PROBS = 0, DCT_IN_LOGITS = 1 };

#define DCT_MAX_VIEWS 8
#define DCT_MAX_CLASSES 64

DCT_API int dct_abi_version(void);
DCT_API const char* dct_error_string(int code);
/* cudaGetErrorString of the last failing CUDA call made by this library on the calling thread */
DCT_API const char* dct_last_cuda_error(void);
/* DCT_OK if device `ordinal` is usable by this library (compute capability 10.x) */
DCT_API int dct_device_check(int ordinal);
DCT_API size_t dct_workspace_bytes(void);

/* ------------------------------------------------------------------------------------------
 * Fused cross-rank exchange of the step's loss sums (SURVEY.md 8e; the reference never shards
 * this path -- nn.DataParallel gathers to cuda:0, generalframework/models/segmentators.py:34-36 --
 * and reads every loss with .item() per iteration, trainer/cotraining_totalloss.py:251-264).
 *
 * Under batch sharding the only cross-rank coupling of the path is a handful of scalars
 * (sum of the JSD map, of the KL maps).  Instead of a collective launched after the step, the
 * step's LAST kernel (dct_kl_from_logits_fwdbwd_pub_f32: the adversarial KL) also pushes all
 * sums into every rank's "mailbox" with plain stores through NVLink / NVSwitch peer mappings
 * (one process per GPU; mailboxes are shared with CUDA IPC).  No extra launch, no NCCL kernel
 * competing for SMs.  Steps that end with another kernel use dct_exchange_publish (one thread).
 *
 *   mailbox (device memory of each rank):  uint64 [nslots][world][DCT_PUB_ROW_WORDS]
 *     publication number q (1, 2, ...) of rank r lands in slot q % nslots, row r, of EVERY
 *     rank's mailbox.  Value j travels as two words {seq32 << 32 | low 32 data bits},
 *     {seq32 << 32 | high 32 data bits} with seq32 = q mod 2^32: a reader that finds seq32 in
 *     a word holds valid data (aligned 8-byte stores are single-copy atomic); summing the rows
 *     in rank order gives every rank the same bits.
 *   dct_peer_pub: the descriptor (a HOST struct, copied into the kernel parameters) handed to a
 *     *_pub launch, which publishes src[0..n) when its last CTA has written the launch's own sum.
 *     `src`, `seq`, `mailbox_table` are device pointers; `seq` is a device counter the kernels
 *     increment (zero it once; shared by a rank's descriptors).
 * ------------------------------------------------------------------------------------------ */
#define DCT_MAX_PEERS 8
#define DCT_PUB_ROW_WORDS 16
#define DCT_PUB_MAX_VALUES 8
#define DCT_IPC_HANDLE_BYTES 64
typedef struct dct_peer_pub {
    const double* src;                          /* device: the n sums to publish */
    unsigned long long* seq;                    /* device: publication counter */
    unsigned long long* const* mailbox_table;   /* device array of `world` mailbox pointers, mailbox_table[r] = rank r's */
    int32_t n, rank, world, nslots;
} dct_peer_pub;
DCT_API size_t dct_peer_pub_bytes(void);
/* cudaMalloc + zero a mailbox of `bytes` on the current device; *dev_ptr receives it and ipc_handle
 * (host, DCT_IPC_HANDLE_BYTES) the CUDA IPC handle another process of this node opens it with. */
DCT_API int dct_mailbox_create(size_t bytes, void** dev_ptr, void* ipc_handle);
/* map a peer's mailbox into this process (peer access enabled lazily); *dev_ptr receives the mapping */
DCT_API int dct_mailbox_open(const void* ipc_handle, void** dev_ptr);
/* owned != 0: cudaFree of a created mailbox; owned == 0: unmap an opened one */
DCT_API int dct_mailbox_close(void* dev_ptr, int owned);
/* stand-alone publication of desc->src[0..n): a one-CTA (64-thread) kernel chained to the previous launch of `stream` with
 * programmatic dependent launch (its scheduling overlaps that kernel's tail) */
DCT_API int dct_exchange_publish(const dct_peer_pub* desc, void* stream);
/* dct_kl_from_logits_fwdbwd_f32 (below) whose last CTA, after writing *sum, publishes the step's sums through
 * `pub_desc` (host struct; sum must be non-NULL and is normally one of desc->src[0..n)). */
DCT_API int dct_kl_from_logits_fwdbwd_pub_f32(const float* p_logit, const float* y_prob, int C, int64_t B, int64_t HW,
                                              float eps, float gconst, float* map, double* sum, float* grad_p_logit,
                                              int32_t* flags, void* workspace, const dct_peer_pub* pub_desc,
                                              void* stream);
/* dct_jsd_fwdbwd_f32 (below) that also carries an EARLY publication: desc->src[0..n) must be final before the launch starts
 * (the previous step's sums, written by earlier launches of `stream`); the first CTA of the grid to finish publishes them while
 * the others are still working, so the publication adds nothing between two launches of the stream (the product's choice at
 * world > 1: every step's first kernel publishes the step before; the caller publishes the last step with
 * dct_exchange_publish).  Shapes outside the tile pipeline: the plain launch followed by dct_exchange_publish. */
DCT_API int dct_jsd_fwdbwd_pub_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                                   float gconst, float* map, double* sum, float* const* grad_views,
                                   const int64_t* labels, int64_t* counts, int counts_mode, int32_t* flags,
                                   void* workspace, const dct_peer_pub* pub_desc, void* stream);

/* ------------------------------------------------------------------------------------------
 * K-view Jensen-Shannon divergence.
 * Replaces JSD_2D.forward (generalframework/loss/loss.py:183-196), JSD.forward (:165-180)
 * and, with DCT_IN_LOGITS, the
 * F.softmax(logits, 1) that produces their inputs (generalframework/models/segmentators.py:46-50).
 *   m = ((x0+x1)+..)/K ; out = H(m) - (H(x0)+..)/K ; H(p) = -sum_c p*log(p+1e-16)
 * `views`: HOST array of K device pointers, each [B,C,HW].
 * ------------------------------------------------------------------------------------------ */

/* forward only: map (nullable) [B,HW]; sum (nullable) double[1] = sum over all pixels of the map
 * (deterministic: fixed-order two-stage reduction). */
DCT_API int dct_jsd_fwd_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                    float* map, double* sum, int32_t* flags, void* workspace, void* stream);

/* backward: grad_views[k] = upstream * d out / d views[k]  (w.r.t. probs, or through the softmax
 * w.r.t. logits when in_kind == DCT_IN_LOGITS).  `grad_views`: HOST array of K device pointers. */
DCT_API int dct_jsd_bwd_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                    const float* gmap, const float* gscalar, float gconst,
                    float* const* grad_views, void* stream);

/* one pass: forward (map nullable, sum nullable) AND gradient with a per-pixel upstream `gconst`
 * known up front (e.g. cot_weight / N for `weight * JSD_2D(..).mean()`,
 * generalframework/trainer/cotraining_totalloss.py:225-226,246).
 * Optional fused Dice counting for the K views on the same read (unlabdiceMeters,
 * cotraining_totalloss.py:224): if `labels` != NULL, `counts` int64 [K][B][C][3] (I, G, P) receives the counts with
 * pred_k = argmax softmax(views[k]) exactly as dct_dice_counts_f32.  `counts_mode`: DCT_COUNTS_ACCUMULATE adds to what
 * `counts` holds; DCT_COUNTS_OVERWRITE makes the launch itself clear the counters first (its first CTA zeroes them and
 * releases a flag in the workspace that every other CTA acquires before its first add -- needs `workspace`), so a
 * training loop needs no fill launch per step (ABI 2; ABI 1 always accumulated). */
#define DCT_COUNTS_ACCUMULATE 0
#define DCT_COUNTS_OVERWRITE 1
DCT_API int dct_jsd_fwdbwd_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int in_kind,
                       float gconst, float* map, double* sum, float* const* grad_views,
                       const int64_t* labels, int64_t* counts, int counts_mode,
                       int32_t* flags, void* workspace, void* stream);

/* grad[i] *= *gscalar for i < n, skipped entirely (no memory traffic) when *gscalar == 1.0f.
 * Used by the fused loss' backward: the upstream of `total = sup + fused_loss` is exactly 1. */
DCT_API int dct_scale_if_not_one_f32(float* grad, int64_t n, const float* gscalar, void* stream);

/* ------------------------------------------------------------------------------------------
 * KL family of the adversarial step.
 * ------------------------------------------------------------------------------------------ */

/* KL_Divergence_2D.forward (loss.py:110-134): out = sum_c y*log(y+eps) - sum_c y*log(p+eps).
 * map nullable, sum nullable (as above). */
DCT_API int dct_kl_fwd_f32(const float* p, const float* y, int C, int64_t B, int64_t HW, float eps,
                   float* map, double* sum, int32_t* flags, void* workspace, void* stream);
/* its backward: grad_p (nullable) = up * (-y/(p+eps)); grad_y (nullable) = up * (log(y+eps)+y/(y+eps)-log(p+eps)) */
DCT_API int dct_kl_bwd_f32(const float* p, const float* y, int C, int64_t B, int64_t HW, float eps,
                   const float* gmap, const float* gscalar, float gconst,
                   float* grad_p, float* grad_y, void* stream);

/* VATGenerator.kl_div_with_logit(q_logit, p_logit) (generalframework/utils/AEGenerator.py:78-91) and
 * KL_Divergence_2D_Logit(p_logit, y_logit) (loss.py:137-162, with q := y):
 *   q = softmax(q_logit); out = sum_c q*(log_softmax(q_logit) - log_softmax(p_logit)).
 * One pass: map (nullable), sum (nullable), and if has_upstream != 0 the gradients
 *   grad_p_logit (nullable) = up*(softmax(p_logit) - q),  grad_q_logit (nullable) = up*q*((logq-logp) - out). */
DCT_API int dct_kl_logit_f32(const float* q_logit, const float* p_logit, int C, int64_t B, int64_t HW,
                     float* map, double* sum,
                     int has_upstream, const float* gmap, const float* gscalar, float gconst,
                     float* grad_p_logit, float* grad_q_logit, void* workspace, void* stream);

/* the trainers' composite  KL_Divergence_2D(reduce=True)(softmax(adv_logits), real_probs.detach())
 * (cotraining_totalloss.py:391-392, vattrainer.py:152-154) in one pass over logits:
 * sum (nullable) of the KL map, grad_logits (nullable) = gconst * softmax_backward(-y/(p+eps)). */
DCT_API int dct_kl_from_logits_fwdbwd_f32(const float* p_logit, const float* y_prob, int C, int64_t B, int64_t HW,
                                  float eps, float gconst, float* map, double* sum, float* grad_p_logit,
                                  int32_t* flags, void* workspace, void* stream);

/* Entropy_2D.forward / Entropy.forward (loss.py:53-84): H = -sum_c p*log(p+1e-16); map/sum nullable;
 * backward grad_p = up * -(log(p+1e-16) + p/(p+1e-16)). */
DCT_API int dct_entropy_fwd_f32(const float* p, int C, int64_t B, int64_t HW, float* map, double* sum,
                                int32_t* flags, void* workspace, void* stream);
DCT_API int dct_entropy_bwd_f32(const float* p, int C, int64_t B, int64_t HW, const float* gmap,
                                const float* gscalar, float gconst, float* grad_p, void* stream);

/* KL_div.forward (loss.py:87-107): out = sum_c -p*log(q/p + eps) (unused by the trainers; differentiable like the
 * reference's autograd graph: with r = q/p, u = r + eps: grad_p = up * (r/u - log u), grad_q = up * (-1/u); grad_q nullable) */
DCT_API int dct_kl_div_fwd_f32(const float* p, const float* q, int C, int64_t B, int64_t HW, float eps,
                       float* map, double* sum, int32_t* flags, void* workspace, void* stream);
DCT_API int dct_kl_div_bwd_f32(const float* p, const float* q, int C, int64_t B, int64_t HW, float eps,
                       const float* gmap, const float* gscalar, float gconst, float* grad_p, float* grad_q,
                       void* stream);

/* F.softmax(x, 1) forward (segmentators.py:50) and its backward gx = p*(gp - sum_c p*gp) */
DCT_API int dct_softmax_fwd_f32(const float* x, int C, int64_t B, int64_t HW, float* p, void* stream);
DCT_API int dct_softmax_bwd_f32(const float* p, const float* gp, int C, int64_t B, int64_t HW, float* gx, void* stream);

/* ------------------------------------------------------------------------------------------
 * VAT / FGSM perturbation arithmetic (image-shaped tensors: B samples of M = Cin*H*W floats).
 * ------------------------------------------------------------------------------------------ */

/* VATGenerator._l2_normalize (AEGenerator.py:68-76): out_b = scale * (d_b / (||d_b||_2 + 1e-16)).
 * `out` may alias `d` (the reference normalises in place); scale = 1 for the bare function,
 * xi / eps for `xi * _l2_normalize(d)` (:103) and `eps * d` (:113-114).
 * passes = 2 applies the normalisation twice before scaling -- the reference's
 * `d = _l2_normalize(d)` (:98) immediately followed by `xi * _l2_normalize(d)` (:103) -- in one launch.
 * If img != NULL also writes adv = clamp(img + out, 0, 1) (:116-117). */
DCT_API int dct_l2_normalize_f32(const float* d, float* out, int64_t B, int64_t M, int passes, float scale,
                         const float* img, float* adv, void* workspace, void* stream);

/* FSGMGenerator.adversarial_fgsm (AEGenerator.py:35-51): noise = eps*sign(grad); adv = img + noise */
DCT_API int dct_fgsm_f32(const float* img, const float* grad, float eps, float* adv, float* noise,
                 int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------
 * Integer metric reductions (bit-exact).
 * ------------------------------------------------------------------------------------------ */

/* DiceMeter.add counting (generalframework/metrics/dice_meter.py:12-33,50-55; utils/utils.py:154-217):
 *   pred = argmax_c softmax(x)_c (first index on ties; pinned arithmetic, see DESIGN.md "Dice spec")
 *   counts[b][c] = (I, G, P) = (#{pred==c & gt==c}, #{gt==c}, #{pred==c})  int64 [B][C][3]
 * counts is zeroed first unless accumulate != 0.  Out-of-range labels are counted in
 * flags[DCT_FLAG_LABEL] and excluded from I and G. */
DCT_API int dct_dice_counts_f32(const float* x, const int64_t* labels, int C, int64_t B, int64_t HW,
                        int64_t* counts, int accumulate, int32_t* flags, void* stream);

/* meta_dice's final arithmetic (dice_meter.py:17-20): dice = (2*f32(I)+1e-8)/(f32(G+P)+1e-8).
 * batch_sum == 0: rows = B ('2d', einsum bcwh->bc); != 0: counts summed over b first, 1 row ('3d', bcwh->c).
 * dice float32 [rows][C]. */
DCT_API int dct_dice_from_counts_f32(const int64_t* counts, int64_t B, int C, int batch_sum, float* dice, void* stream);

/* IoU.add -> ConfusionMatrix.add (generalframework/metrics/iou.py:43-69, confusionmatrix.py:32-85):
 *   pred = argmax_c x_c on the RAW scores (first index on ties, NaN maximal as torch.max);
 *   over pixels with 0 <= gt < C:  conf[gt][pred] += 1.   conf int64 [C][C], ACCUMULATED into. */
DCT_API int dct_confusion_f32(const float* x, const int64_t* labels, int C, int64_t B, int64_t HW,
                      int64_t* conf, void* stream);
/* same for an integer prediction map ([N] int64, iou.py:49-50); predictions outside [0,C) on a
 * valid-label pixel are counted in flags[DCT_FLAG_PRED] (the reference's bincount-size assert). */
DCT_API int dct_confusion_labels_i64(const int64_t* pred, const int64_t* labels, int64_t n, int C,
                             int64_t* conf, int32_t* flags, void* stream);

/* ------------------------------------------------------------------------------------------
 * Supervised branch (SURVEY.md 8f.1): pixel-wise cross-entropy fused with the Dice counting of the
 * same (logits, labels) pair.
 * Replaces CrossEntropyLoss2d.forward (generalframework/loss/loss.py:12-25) =
 *   nn.NLLLoss(weight, ignore_index)(F.log_softmax(outputs, 1), targets)
 * as called at generalframework/trainer/cotraining_totalloss.py:211 (and :294, trainer.py:171), and the
 * diceMeters[k].add(pred, gt) of the next line (:212) when `dice_counts` is given.
 *   l_i = -w[t_i] * log_softmax(x_i)[t_i]  (0 where t_i == ignore_index; w = 1 without class_weight)
 *   d l_i / d x_ic = w[t_i] * (softmax(x_i)_c - [c == t_i])
 * The 'mean' reduction divides by W = sum_i w[t_i] over the non-ignored pixels: W comes from
 * dct_label_hist_i64 (8 B/pixel) or is simply the pixel count when there is neither a class weight nor an
 * ignored pixel; the caller folds 1/W into the upstream (gscalar / gconst).
 * `class_weight`: device float[C] or NULL.  Labels outside [0,C) other than ignore_index are counted in
 * flags[DCT_FLAG_LABEL] (PyTorch raises "Target out of bounds") and treated as ignored.
 * ------------------------------------------------------------------------------------------ */

/* hist int64[C+2], overwritten: hist[c] = #{label == c} (c < C, the ignore_index excluded even if it is < C),
 * hist[C] = #{label == ignore_index}, hist[C+1] = #{other labels outside [0,C)}. */
DCT_API int dct_label_hist_i64(const int64_t* labels, int64_t n, int C, int64_t ignore_index, int64_t* hist,
                               void* stream);

/* forward: map (nullable) [B,HW] = l_i; sum (nullable) double[1] = sum_i l_i (bit-reproducible). */
DCT_API int dct_ce_fwd_f32(const float* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                           const float* class_weight, int64_t ignore_index, float* map, double* sum,
                           int32_t* flags, void* workspace, void* stream);

/* backward: grad_logits = upstream * d l_i / d x  (upstream as "dct_upstream": gmap for reduce=False). */
DCT_API int dct_ce_bwd_f32(const float* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                           const float* class_weight, int64_t ignore_index, const float* gmap,
                           const float* gscalar, float gconst, float* grad_logits, int32_t* flags, void* stream);

/* one pass: forward (map / sum nullable) AND grad_logits = gconst * (gscalar ? *gscalar : 1) * d l_i / d x.
 * If dice_counts != NULL (int64 [B][C][3], ACCUMULATED into) the Dice counts (I, G, P) of
 * argmax softmax(logits) against `labels` are produced from the same read, exactly as
 * dct_dice_counts_f32 (every label outside [0,C), the ignore_index included, then raises
 * flags[DCT_FLAG_LABEL] as DiceMeter.add's class2one_hot assert does). */
DCT_API int dct_ce_fwdbwd_f32(const float* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                              const float* class_weight, int64_t ignore_index, const float* gscalar, float gconst,
                              float* map, double* sum, float* grad_logits, int64_t* dice_counts, int32_t* flags,
                              void* workspace, void* stream);

/* Cityscapes flavour of the labeled loop (generalframework/trainer/cotraining_city.py:236-241; trainer_city.py:141):
 *   sup_loss = criterions['sup'](pred, gt.squeeze(1));   metrics[k].add(predicted=pred, target=gt)
 * with metrics[k] = IoU(C, ignore_index=255) (generalframework/metrics/iou.py:43-69 -> confusionmatrix.py:32-85).
 * Same loss / gradient arguments as dct_ce_fwdbwd_f32; `confusion` is int64 [C,C] (rows = ground truth), ACCUMULATED
 * into: conf[t][argmax_c logits] += 1 for every pixel with 0 <= t < C (raw arg-max with torch.max semantics: first
 * index on ties, NaN maximal; ignore-255 pixels fall outside [0,C) and are dropped).  One pass over logits + labels. */
DCT_API int dct_ce_fwdbwd_conf_f32(const float* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                                   const float* class_weight, int64_t ignore_index, const float* gscalar, float gconst,
                                   float* map, double* sum, float* grad_logits, int64_t* confusion, int32_t* flags,
                                   void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------
 * Class maps, one-hot tensors and the functional Dice on one-hot inputs (SURVEY.md 8a11 / 8b "Functional Dice").
 * Replaces generalframework/utils/utils.py: pred2class :73-80, probs2class :178-184, class2one_hot :187-198,
 * probs2one_hot :201-207, predlogit2one_hot :210-217, one_hot :154-161, intersection :164-168,
 * meta_dice / dice_coef / dice_batch :221-235 (called by trainer/trainer.py:171-175,222-227).
 * ------------------------------------------------------------------------------------------ */

/* scores [B,C,HW] -> class map and/or one-hot (each output nullable, at least one given):
 *   cls int64 [B,HW], cls_u8 uint8 [B,HW] (save_images' uint8 PNG plane, utils.py:238-250), onehot int32 [B,C,HW].
 *   mode 0: raw arg-max with torch.max semantics (first index on ties, NaN maximal)      -- pred2class
 *   mode 1: arg-max of softmax(x) in the pinned Dice arithmetic (DESIGN.md "Dice spec")  -- predlogit2one_hot
 *   mode 2: mode 0 + flags[DCT_FLAG_SIMPLEX] on columns failing utils.simplex             -- probs2class / probs2one_hot */
DCT_API int dct_classmap_f32(const float* x, int C, int64_t B, int64_t HW, int mode, int64_t* cls, uint8_t* cls_u8,
                             int32_t* onehot, int32_t* flags, void* stream);

/* class2one_hot: int64 labels [B,HW] -> int32 one-hot [B,C,HW]; labels outside [0,C) are counted in
 * flags[DCT_FLAG_LABEL] (the reference's sset assert) and produce an all-zero column. */
DCT_API int dct_onehot_from_labels_i64(const int64_t* labels, int C, int64_t B, int64_t HW, int32_t* onehot,
                                       int32_t* flags, void* stream);

/* meta_dice's counting on int32 one-hot tensors [B,C,HW]: counts int64 [B][C][3] = (sum label&pred, sum label,
 * sum pred), OVERWRITTEN (nullable: predicate only); flags[DCT_FLAG_ONEHOT] += violations of utils.one_hot in
 * either tensor.  pred_onehot may be NULL (one_hot(label) alone).  dct_dice_from_counts_f32 finishes
 * dice_coef (batch_sum = 0) / dice_batch (batch_sum = 1). */
DCT_API int dct_onehot_dice_counts_i32(const int32_t* label_onehot, const int32_t* pred_onehot, int C, int64_t B,
                                       int64_t HW, int64_t* counts, int32_t* flags, void* stream);

/* Ensemble voting over K views [B,C,HW] (HOST array of K device pointers) -- SURVEY.md 8f.4, replaces
 * Ensembleway._softVoting / _hardVoting (Summary.py:88-120).
 *   hard = 0: out (nullable) [B,C,HW] = ((x_0 + x_1) + ...) / K; cls / cls_u8 (nullable) = raw arg-max of the mean
 *   hard = 1: per-view raw arg-max, most voted class per pixel (smallest class on ties, np.bincount(...).argmax());
 *             out (nullable) = one-hot of the winner as float; cls / cls_u8 (nullable) = the winner.
 * (The reference's hard vote concatenates the views along the batch axis, i.e. it assumes B = 1; here every
 * image of the batch is voted on its own, which is the same thing at B = 1.) */
DCT_API int dct_vote_f32(const float* const* views, int K, int C, int64_t B, int64_t HW, int hard, float* out,
                         int64_t* cls, uint8_t* cls_u8, void* stream);

/* ------------------------------------------------------------------------------------------
 * Boundary distance (evaluation path, Summary.py:25: the reference reports the Hausdorff distance of every view and
 * ensemble through the external deepclustering package).  Definition: medpy.metric.binary.hd, the ACDC challenge's
 * evaluation code.  Per class c on a grid -- one H x W slice (volume == 0) or the whole batch as one B x H x W volume
 * (volume != 0; DiceMeter's '2d' / '3d') -- with A = {pred == c}, G = {labels == c}:
 *   border(M) = M xor binary_erosion(M), cross structuring element (4 / 6 neighbours), off-grid cells are background;
 *   d(x, S)   = min over y in S of ||(x - y) * spacing||_2, spacing (sy, sx) or (sz, sy, sx) along the tensor axes;
 *   hd        = max(max over border(A) of d(., border(G)), max over border(G) of d(., border(A))); NaN if A or G is empty.
 * Values outside [0,C) belong to no class (a non-c neighbour for every c) and are counted in flags[DCT_FLAG_PRED]
 * (pred) / flags[DCT_FLAG_LABEL] (labels).  Exact separable Euclidean distance transforms of the 2C border sets:
 * 4 launches for a slice batch, 5 for a volume; no host synchronisation.  At unit spacing hd is the correctly rounded
 * square root of the exact squared distance (while that stays below 2^24).
 * Limits (DCT_ERR_UNSUPPORTED): C <= DCT_MAX_CLASSES; H, W (and B when volume != 0) <= 32768 (each line's envelope stack
 * keeps 16-bit positions); 2*C*B*max(H,W) (and 2*C*H*W for a volume) <= 2^31 - 1.
 * ------------------------------------------------------------------------------------------ */

/* bytes of `scratch` dct_hausdorff_i64 needs for this shape (about 4*C + 2 bytes per pixel, 12*C + 2 for a volume);
 * 0 for a shape it rejects.  Host only. */
DCT_API size_t dct_hausdorff_scratch_bytes(int C, int64_t B, int64_t H, int64_t W, int volume);
/* pred, labels int64 [B,H,W]; spacing: HOST array of 2 (volume == 0) or 3 positive finite values, NULL = all ones;
 * hd float32 [volume ? 1 : B][C], overwritten; scratch: >= dct_hausdorff_scratch_bytes() bytes, 256-byte aligned, no
 * initial state required, private to the call until the stream reaches its end. */
DCT_API int dct_hausdorff_i64(const int64_t* pred, const int64_t* labels, int C, int64_t B, int64_t H, int64_t W,
                              int volume, const double* spacing, float* hd, int32_t* flags, void* scratch, void* stream);

/* Surface distances of the same borders, grids and spacing (medpy.metric.binary hd95 / asd / assd, connectivity 1).
 * Per (row, class): S_pg = d(x, border(G)) for every x in border(A), S_gp = d(y, border(A)) for every y in border(G);
 *   hd   = max(max S_pg, max S_gp), bit-identical to dct_hausdorff_i64;
 *   hd95 = numpy.percentile(concat(S_pg, S_gp), 95) with the default 'linear' method: n = |S_pg| + |S_gp|,
 *          v = (n - 1) * 0.95, lo = floor(v), t = v - lo, a = sorted[lo], b = sorted[min(lo + 1, n - 1)], d = b - a,
 *          (t >= 0.5 ? b - d * (1 - t) : a + d * t) in double, rounded once to float;
 *   asd  = mean(S_pg) (directional: prediction border to label border), assd = (mean(S_pg) + mean(S_gp)) / 2.
 * All four are NaN where A or G is empty.  Same limits, flags, argument checks and error codes as dct_hausdorff_i64.
 * The last distance pass keeps each border pixel's d^2 and per-line sums; a radix select on the d^2 bits (4 passes of
 * 8 bits, integer histograms) and a fixed-order reduction of the sums make the result bit-reproducible.  14 launches
 * for a slice batch, 15 for a volume; no host synchronisation, no allocation. */

/* bytes of `scratch` dct_surface_distances_i64 needs: dct_hausdorff_scratch_bytes() + 8 per pixel (d^2 of the queries
 * of both sides) + 12 per line of the last pass (2*C*B*H lines for a slice batch, 2*C*H*W for a volume) + 2112 per
 * (row, class), each region rounded up to 256 bytes; 0 for a shape it rejects.  Host only. */
DCT_API size_t dct_surface_distance_scratch_bytes(int C, int64_t B, int64_t H, int64_t W, int volume);
/* pred, labels, spacing, flags, scratch as for dct_hausdorff_i64 (scratch >= dct_surface_distance_scratch_bytes());
 * out float32 [4][volume ? 1 : B][C] = hd, hd95, asd, assd, overwritten. */
DCT_API int dct_surface_distances_i64(const int64_t* pred, const int64_t* labels, int C, int64_t B, int64_t H, int64_t W,
                                      int volume, const double* spacing, float* out, int32_t* flags, void* scratch,
                                      void* stream);

/* ------------------------------------------------------------------------------------------
 * bfloat16 twins of the one-pass-over-logits entry points (networks under torch.autocast emit bf16 logits;
 * north_star: "within 1e-2 relative in bf16").  Tensors [B,C,HW] are bfloat16 (2-byte elements, same NCHW
 * layout), gradients are written as bfloat16 (round-to-nearest-even); ALL arithmetic is fp32 in registers and the
 * map / sum outputs, labels, counts, flags and workspace are exactly as in the _f32 functions.  Only the TMA tile
 * pipeline serves these: HW % 8 == 0, 16-byte aligned tensors, C in {2,3,4,19}, K*C <= 80; any other shape
 * returns DCT_ERR_UNSUPPORTED with nothing launched and the caller converts to float32.
 * Algorithmic traffic: 2*K*C*2 (+8 with labels) B/pixel for the JSD step, 3*C*2 for the adversarial KL.
 * ------------------------------------------------------------------------------------------ */

/* dct_jsd_fwdbwd_f32 with DCT_IN_LOGITS on bf16 views (HOST arrays of K device pointers).  grad_views == NULL:
 * forward only (evaluation; `labels` must be NULL then).  Fused Dice counting needs C <= 4. */
DCT_API int dct_jsd_fwdbwd_bf16(const void* const* views, int K, int C, int64_t B, int64_t HW, float gconst,
                                float* map, double* sum, void* const* grad_views, const int64_t* labels,
                                int64_t* counts, int counts_mode, int32_t* flags, void* workspace, void* stream);

/* dct_kl_logit_f32 (VATGenerator.kl_div_with_logit, AEGenerator.py:78-91) on bf16 logits; bf16 gradients. */
DCT_API int dct_kl_logit_bf16(const void* q_logit, const void* p_logit, int C, int64_t B, int64_t HW, float* map,
                              double* sum, int has_upstream, const float* gmap, const float* gscalar, float gconst,
                              void* grad_p_logit, void* grad_q_logit, void* workspace, void* stream);

/* dct_kl_from_logits_fwdbwd_f32 (cotraining_totalloss.py:391-392) on bf16 p_logit / y_prob; bf16 gradient. */
DCT_API int dct_kl_from_logits_fwdbwd_bf16(const void* p_logit, const void* y_prob, int C, int64_t B, int64_t HW,
                                           float eps, float gconst, float* map, double* sum, void* grad_p_logit,
                                           int32_t* flags, void* workspace, void* stream);

/* dct_ce_fwdbwd_f32 (CrossEntropyLoss2d, loss.py:12-25, + DiceMeter.add) on bf16 logits; bf16 gradient. */
DCT_API int dct_ce_fwdbwd_bf16(const void* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                               const float* class_weight, int64_t ignore_index, const float* gscalar, float gconst,
                               float* map, double* sum, void* grad_logits, int64_t* dice_counts, int32_t* flags,
                               void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------
 * Developer tracing (tools/step_trace.py; not used by the product).  Between _begin and _end every launch of the tile
 * pipeline and of the perturbation normalisation takes the next 4 * max_ctas uint64 words of `buf` (device memory, zeroed
 * by the caller) and each of its CTAs stamps %globaltimer (ns) there: [0] after the programmatic-dependency wait,
 * [1] first tile landed / after the first per-sample exchange, [2] tile pipeline: (SM id << 32) | (pool draws << 16) | tiles
 * processed; normalisation: after the last exchange, [3] at its end.  _end returns the number of launches recorded.
 * Process-global state: do not trace from two host threads at once.
 * ------------------------------------------------------------------------------------------ */
DCT_API int dct_dev_trace_begin(void* buf, int max_ctas, int max_launches);
DCT_API int dct_dev_trace_end(void);
/* Developer check, host only (no GPU): the image index the tile schedule derives for `tile` with `tiles_per_image` tiles per
 * image (a multiply-shift form of the division; csrc/dct_tile.cuh tile_image).  Negative: DCT_ERR_BAD_ARG. */
DCT_API int dct_dev_tile_image(int tiles_per_image, int tile);

#ifdef __cplusplus
}
#endif
#endif /* DCT_B200_H */
