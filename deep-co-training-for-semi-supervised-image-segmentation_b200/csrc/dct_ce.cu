// dct_ce.cu -- the supervised branch's pixel-wise cross-entropy (SURVEY.md 8f.1), fused with the Dice counting
// of the same (logits, labels) pair:
//   sup_loss = CrossEntropyLoss2d(pred, gt.squeeze(1))        generalframework/trainer/cotraining_totalloss.py:211
//   diceMeters[k].add(pred, gt)                               :212
// CrossEntropyLoss2d (generalframework/loss/loss.py:12-25) = nn.NLLLoss(weight, ignore_index)(F.log_softmax(x, 1), t):
//   l_i = -w[t_i] * log_softmax(x_i)[t_i]   (0 where t_i == ignore_index);   'mean' = sum_i l_i / sum_i w[t_i]
//   d l_i / d x_ic = w[t_i] * (softmax(x_i)_c - [c == t_i])
// One pass over the logits: read C planes + the int64 label, write C gradient planes (2*C*4 + 8 B/pixel).
#include "dct_tile.cuh"

namespace dct {

// per-component select for the packed lane type
__device__ __forceinline__ float vsel(const bool (&c)[1], float a, float b) { return c[0] ? a : b; }
__device__ __forceinline__ f2 vsel(const bool (&c)[2], f2 a, f2 b) { return mk2(c[0] ? a.v.x : b.v.x, c[1] ? a.v.y : b.v.y); }
template <class T> struct lanes_of { static constexpr int value = 1; };
template <> struct lanes_of<f2> { static constexpr int value = 2; };
__device__ __forceinline__ float vfrom(const float (&w)[1]) { return w[0]; }
__device__ __forceinline__ f2 vfrom(const float (&w)[2]) { return mk2(w[0], w[1]); }

// GRAD: x[0][c] <- g * w * (p_c - onehot_c);  DICEF: the tile kernel also counts Dice (I,G,P) of the same logits;
// CONFV: it also counts the confusion matrix of arg-max(logits) against the labels (the Cityscapes trainers' IoU meter)
template <bool GRAD, bool DICEF, bool GMAPV, bool CONFV = false>
struct CeOp {
    static constexpr int NIN = 1, NOUT = GRAD ? 1 : 0;
    static constexpr int NDICE = DICEF ? 1 : 0;
    static constexpr bool GMAP = GMAPV, LABELS = true, CONF = CONFV;
    static constexpr bool HAS_MAP = true, USES_UP = GRAD, CHECKS_SIMPLEX = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&)[1][CM], int, T, float, bool&) { return vset<T>(0.0f); }  // unused
    template <int CM, class T, int LW>
    static __device__ __forceinline__ T apply_lab(T (&x)[1][CM], int, T g, const int (&cls)[LW], const float (&cw)[LW], bool&) {
        static_assert(LW == lanes_of<T>::value, "one label per lane");
        // log-softmax in base 2 (one MUFU.EX2 per class, one LG2 + one RCP per pixel), as the JSD kernel
        T mx = x[0][0];
#pragma unroll
        for (int c = 1; c < CM; ++c) mx = vmax(mx, x[0][c]);
        const T nmxl = vmuls(mx, -kLog2e);
        T e[CM];
        T Z, sel = vset<T>(0.0f);
#pragma unroll
        for (int c = 0; c < CM; ++c) {
            const T t = vfmas(x[0][c], kLog2e, nmxl);  // (x - max) * log2(e)
            const T ev = vex2(t);
            e[c] = ev;
            Z = (c == 0) ? ev : vadd(Z, ev);
            bool is[LW];
#pragma unroll
            for (int j = 0; j < LW; ++j) is[j] = cls[j] == c;
            sel = vsel(is, t, sel);
        }
        const T lZ = vlg2(Z);
        const T w = vfrom(cw);
        bool on[LW];
#pragma unroll
        for (int j = 0; j < LW; ++j) on[j] = cls[j] >= 0;
        // -w * ln2 * (lg2 e_t - lg2 Z); exactly 0 for ignored pixels whatever their logits hold
        const T loss = vsel(on, vmul(w, vmuls(vsub(lZ, sel), kLn2)), vset<T>(0.0f));
        if constexpr (GRAD) {
            const T inv = vrcp(Z);
            const T gw = vmul(g, w);
#pragma unroll
            for (int c = 0; c < CM; ++c) {
                bool is[LW];
#pragma unroll
                for (int j = 0; j < LW; ++j) is[j] = cls[j] == c;
                const T oh = vsel(is, vset<T>(1.0f), vset<T>(0.0f));
                x[0][c] = vsel(on, vmul(gw, vsub(vmul(e[c], inv), oh)), vset<T>(0.0f));
            }
        }
        return loss;
    }
};

struct CeArgs {
    const float* x;
    const int64_t* labels;
    const float* class_w;
    int64_t ignore_index;
    int C;
    int64_t HW;
    float* map;
    double* sum;
    float* grad;
    Upstream up;
    int32_t* flags;
    Workspace* ws;
    int64_t B;          // ce_launch_rt: images b = blockIdx.y, blockIdx.y + gridDim.y, ... (image_grid)
};

// Correctness path for shapes the tile pipeline does not take (C outside {2,3,4,19}, odd HW, misaligned pointers):
// one pixel per thread, two sweeps over the pixel's class column (the second one is served by L1/L2).
template <bool GRAD>
__global__ void __launch_bounds__(256) ce_kernel_rt(const CeArgs a) {
    const int C = a.C;
    const int64_t HW = a.HW;
    float gs = 1.0f;
    if constexpr (GRAD) gs = upstream_scalar(a.up);
    double acc = 0.0;
    int nbad = 0;
    for (int64_t b = blockIdx.y; b < a.B; b += gridDim.y) {
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (int64_t)gridDim.x * blockDim.x) {
            const float* xb = a.x + b * C * HW + i;
            const long long t = a.labels[b * HW + i];
            const bool valid = t >= 0 && t < C, ign = t == a.ignore_index;
            nbad += (!valid) & (!ign);
            const bool use = valid & !ign;
            const float w = use ? (a.class_w != nullptr ? __ldg(a.class_w + t) : 1.0f) : 0.0f;
            float mx = xb[0];
            for (int c = 1; c < C; ++c) mx = fmaxf(mx, xb[(int64_t)c * HW]);
            float Z = 0.0f, sel = 0.0f;
            for (int c = 0; c < C; ++c) {
                const float tt = fmaf(xb[(int64_t)c * HW], kLog2e, -mx * kLog2e);
                Z += ex2_ftz(tt);
                if (use && c == (int)t) sel = tt;
            }
            const float lZ = lg2_ftz(Z);
            const float loss = use ? w * ((lZ - sel) * kLn2) : 0.0f;
            acc += (double)loss;
            if (a.map != nullptr) a.map[b * HW + i] = loss;
            if constexpr (GRAD) {
                float g = gs * w;
                if (a.up.gmap != nullptr) g *= a.up.gmap[b * HW + i];
                const float inv = rcp_ftz(Z);
                float* gb = a.grad + b * C * HW + i;
                for (int c = 0; c < C; ++c) {
                    const float p = ex2_ftz(fmaf(xb[(int64_t)c * HW], kLog2e, -mx * kLog2e)) * inv;
                    gb[(int64_t)c * HW] = use ? g * (p - ((int)t == c ? 1.0f : 0.0f)) : 0.0f;
                }
            }
        }
    }
    nbad = __reduce_add_sync(0xffffffffu, nbad);
    if ((threadIdx.x & 31) == 0 && nbad != 0 && a.flags != nullptr) atomicAdd(&a.flags[DCT_FLAG_LABEL], nbad);
    grid_sum_to(acc, a.ws, a.sum, blockIdx.y * gridDim.x + blockIdx.x, gridDim.x * gridDim.y);
}

template <class Op, class ET = float>
static int ce_tile(const CeArgs& c, int64_t B, unsigned long long* counts, cudaStream_t stream, bool& done,
                   unsigned long long* conf = nullptr) {
    done = false;
    TileArgs t{};
    t.conf = conf;
    t.in[0] = c.x; t.out[0] = c.grad;
    t.HW = c.HW; t.map = c.map; t.sum = c.sum; t.up = c.up; t.eps = 0.0f; t.flags = c.flags; t.ws = c.ws;
    t.labels = c.labels; t.counts = counts; t.count_view_stride = B * c.C * 3;
    t.class_w = c.class_w; t.ignore_index = c.ignore_index;
    if (!tile_eligible<Op, ET>(t, B)) return DCT_OK;
    int rc = DCT_ERR_UNSUPPORTED;
    switch (c.C) {
        case 2: rc = tile_launch_ct<Op, 2, ET>(t, B, stream); break;
        case 3: rc = tile_launch_ct<Op, 3, ET>(t, B, stream); break;
        case 4: rc = tile_launch_ct<Op, 4, ET>(t, B, stream); break;
        case 19:
            if constexpr (Op::NDICE == 0) rc = tile_launch_ct<Op, 19, ET>(t, B, stream);
            break;
        default: break;
    }
    if (rc == DCT_ERR_UNSUPPORTED) return DCT_OK;  // not a tile shape: the caller falls back
    done = rc == DCT_OK;
    return rc;
}

template <bool GRAD>
static int ce_launch_rt(CeArgs c, int64_t B, cudaStream_t s) {
    c.B = B;
    const dim3 grid = image_grid(B, c.HW, 256);
    if (!fits_partials(grid)) return DCT_ERR_UNSUPPORTED;
    ce_kernel_rt<GRAD><<<grid, 256, 0, s>>>(c);
    return check_launch();
}

static int ce_check(const float* x, const int64_t* labels, int C, int64_t B, int64_t HW) {
    if (x == nullptr || labels == nullptr || C < 1 || B < 1 || HW < 1) return DCT_ERR_BAD_ARG;
    if (C > DCT_MAX_CLASSES || B > 65535) return DCT_ERR_UNSUPPORTED;
    if (!aligned(x, 4) || !aligned(labels, 8)) return DCT_ERR_MISALIGNED;
    return DCT_OK;
}

// ---- label histogram: hist[c] = #{label == c}, c < C; hist[C] = #{label == ignore_index}; hist[C+1] = #other ----
__global__ void __launch_bounds__(256) label_hist_kernel(const int64_t* __restrict__ labels, int64_t n, int C,
                                                         int64_t ignore_index, unsigned long long* hist) {
    __shared__ unsigned int s_h[DCT_MAX_CLASSES + 2];
    for (int i = threadIdx.x; i < C + 2; i += blockDim.x) s_h[i] = 0u;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    // <= 2^31 labels per CTA between flushes is guaranteed by the grid size chosen on the host
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        long long t;
        asm volatile("ld.global.nc.L1::no_allocate.s64 %0, [%1];" : "=l"(t) : "l"(labels + i));
        const int slot = (t == ignore_index) ? C : ((t >= 0 && t < C) ? (int)t : C + 1);
        // warp-aggregated: lanes with the same slot elect one to add the group's population count
        const unsigned int peers = __match_any_sync(__activemask(), slot);
        if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_h[slot], (unsigned int)__popc(peers));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C + 2; i += blockDim.x)
        if (s_h[i] != 0u) atomicAdd(&hist[i], (unsigned long long)s_h[i]);
}

}  // namespace dct

#ifndef DCT_KBENCH  // tools/kbench_tile.cu includes this file for the ops only
using namespace dct;

extern "C" int dct_label_hist_i64(const int64_t* labels, int64_t n, int C, int64_t ignore_index, int64_t* hist,
                                  void* stream) {
    if (labels == nullptr || hist == nullptr || n < 1 || C < 1) return DCT_ERR_BAD_ARG;
    if (C > DCT_MAX_CLASSES) return DCT_ERR_UNSUPPORTED;
    if (!aligned(labels, 8) || !aligned(hist, 8)) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(hist, 0, (size_t)(C + 2) * 8, s);
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    int64_t ctas = (n + 256 * 16 - 1) / (256 * 16);
    if (ctas > kSMs * 8) ctas = kSMs * 8;
    label_hist_kernel<<<(unsigned)ctas, 256, 0, s>>>(labels, n, C, ignore_index, reinterpret_cast<unsigned long long*>(hist));
    return check_launch();
}

extern "C" int dct_ce_fwd_f32(const float* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                              const float* class_weight, int64_t ignore_index, float* map, double* sum,
                              int32_t* flags, void* workspace, void* stream) {
    int rc = ce_check(logits, labels, C, B, HW);
    if (rc != DCT_OK) return rc;
    if (sum != nullptr && workspace == nullptr) return DCT_ERR_BAD_ARG;
    if (map != nullptr && !aligned(map, 4)) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CeArgs c{logits, labels, class_weight, ignore_index, C, HW, map, sum, nullptr, Upstream{nullptr, nullptr, 1.0f}, flags,
             static_cast<Workspace*>(workspace)};
    bool done;
    rc = ce_tile<CeOp<false, false, false>>(c, B, nullptr, s, done);
    if (rc != DCT_OK || done) return rc;
    return ce_launch_rt<false>(c, B, s);
}

extern "C" int dct_ce_bwd_f32(const float* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                              const float* class_weight, int64_t ignore_index, const float* gmap,
                              const float* gscalar, float gconst, float* grad_logits, int32_t* flags, void* stream) {
    int rc = ce_check(logits, labels, C, B, HW);
    if (rc != DCT_OK) return rc;
    if (grad_logits == nullptr) return DCT_ERR_BAD_ARG;
    if (!aligned(grad_logits, 4) || (gmap != nullptr && !aligned(gmap, 4))) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CeArgs c{logits, labels, class_weight, ignore_index, C, HW, nullptr, nullptr, grad_logits, Upstream{gmap, gscalar, gconst},
             flags, nullptr};
    bool done;
    rc = ce_tile<CeOp<true, false, true>>(c, B, nullptr, s, done);
    if (rc != DCT_OK || done) return rc;
    return ce_launch_rt<true>(c, B, s);
}

extern "C" int dct_ce_fwdbwd_f32(const float* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                                 const float* class_weight, int64_t ignore_index, const float* gscalar, float gconst,
                                 float* map, double* sum, float* grad_logits, int64_t* dice_counts, int32_t* flags,
                                 void* workspace, void* stream) {
    int rc = ce_check(logits, labels, C, B, HW);
    if (rc != DCT_OK) return rc;
    if (grad_logits == nullptr || (sum != nullptr && workspace == nullptr)) return DCT_ERR_BAD_ARG;
    if (!aligned(grad_logits, 4) || (map != nullptr && !aligned(map, 4))) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CeArgs c{logits, labels, class_weight, ignore_index, C, HW, map, sum, grad_logits, Upstream{nullptr, gscalar, gconst}, flags,
             static_cast<Workspace*>(workspace)};
    bool done = false;
    if (dice_counts != nullptr && C <= 4) {
        rc = ce_tile<CeOp<true, true, false>>(c, B, reinterpret_cast<unsigned long long*>(dice_counts), s, done);
        if (rc != DCT_OK || done) return rc;
    }
    rc = ce_tile<CeOp<true, false, false>>(c, B, nullptr, s, done);
    if (rc != DCT_OK) return rc;
    if (!done) {
        rc = ce_launch_rt<true>(c, B, s);
        if (rc != DCT_OK) return rc;
    }
    if (dice_counts != nullptr)  // Dice counting of the same logits in its own launch (C > 4 or a non-tile shape)
        return dct_dice_counts_f32(logits, labels, C, B, HW, dice_counts, 1, flags, stream);
    return DCT_OK;
}

// Cityscapes flavour of the labeled loop (generalframework/trainer/cotraining_city.py:236-241, trainer_city.py:141):
//   sup_loss = criterions['sup'](pred, gt.squeeze(1));  metrics[k].add(predicted=pred, target=gt)      (IoU meter)
// One read of the logits + labels gives the loss, its gradient and conf[gt][argmax pred] (int64 [C,C], accumulated).
extern "C" int dct_ce_fwdbwd_conf_f32(const float* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                                      const float* class_weight, int64_t ignore_index, const float* gscalar, float gconst,
                                      float* map, double* sum, float* grad_logits, int64_t* confusion, int32_t* flags,
                                      void* workspace, void* stream) {
    int rc = ce_check(logits, labels, C, B, HW);
    if (rc != DCT_OK) return rc;
    if (grad_logits == nullptr || confusion == nullptr || (sum != nullptr && workspace == nullptr)) return DCT_ERR_BAD_ARG;
    if (!aligned(grad_logits, 4) || !aligned(confusion, 8) || (map != nullptr && !aligned(map, 4))) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CeArgs c{logits, labels, class_weight, ignore_index, C, HW, map, sum, grad_logits, Upstream{nullptr, gscalar, gconst}, flags,
             static_cast<Workspace*>(workspace)};
    bool done = false;
    rc = ce_tile<CeOp<true, false, false, true>>(c, B, nullptr, s, done, reinterpret_cast<unsigned long long*>(confusion));
    if (rc != DCT_OK || done) return rc;
    // not a tile shape: the loss kernels, then the counting kernel on the same tensors
    rc = dct_ce_fwdbwd_f32(logits, labels, C, B, HW, class_weight, ignore_index, gscalar, gconst, map, sum, grad_logits,
                           nullptr, flags, workspace, stream);
    if (rc != DCT_OK) return rc;
    return dct_confusion_f32(logits, labels, C, B, HW, confusion, stream);
}

// bf16 logits / gradients (fp32 math, fp32 map / sum): the tile pipeline only; DCT_ERR_UNSUPPORTED for other shapes
// (C not in {2,3,4,19}, HW % 8 != 0, misaligned rows, Dice counts with C > 4): the caller converts to float32 then.
extern "C" int dct_ce_fwdbwd_bf16(const void* logits, const int64_t* labels, int C, int64_t B, int64_t HW,
                                  const float* class_weight, int64_t ignore_index, const float* gscalar, float gconst,
                                  float* map, double* sum, void* grad_logits, int64_t* dice_counts, int32_t* flags,
                                  void* workspace, void* stream) {
    if (logits == nullptr || labels == nullptr || grad_logits == nullptr || C < 1 || B < 1 || HW < 1) return DCT_ERR_BAD_ARG;
    if (sum != nullptr && workspace == nullptr) return DCT_ERR_BAD_ARG;
    if (C > DCT_MAX_CLASSES || B > 65535 || (dice_counts != nullptr && C > 4)) return DCT_ERR_UNSUPPORTED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CeArgs c{reinterpret_cast<const float*>(logits), labels, class_weight, ignore_index, C, HW, map, sum,
             reinterpret_cast<float*>(grad_logits), Upstream{nullptr, gscalar, gconst}, flags, static_cast<Workspace*>(workspace)};
    bool done = false;
    int rc;
    if (dice_counts != nullptr)
        rc = ce_tile<CeOp<true, true, false>, bf16>(c, B, reinterpret_cast<unsigned long long*>(dice_counts), s, done);
    else
        rc = ce_tile<CeOp<true, false, false>, bf16>(c, B, nullptr, s, done);
    if (rc != DCT_OK) return rc;
    return done ? DCT_OK : DCT_ERR_UNSUPPORTED;
}
#endif  // DCT_KBENCH
