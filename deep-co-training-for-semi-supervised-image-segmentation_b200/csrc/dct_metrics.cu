// dct_metrics.cu -- integer metric reductions (bit-exact): Dice counts and confusion matrix.
//
// Replaces DiceMeter.add / meta_dice / toOneHot (generalframework/metrics/dice_meter.py:12-55), the
// helper chain class2one_hot / probs2one_hot / intersection / one_hot / simplex / uniq
// (generalframework/utils/utils.py:130-217) and IoU.add -> ConfusionMatrix.add
// (generalframework/metrics/iou.py:43-69, confusionmatrix.py:32-85).  The reference materialises
// int32 one-hot tensors, copies them to the host nine times for torch.unique and runs numpy
// bincount on the CPU; here each (scores, int64 labels) pixel is read once from HBM
// (C*4 + 8 bytes) and only 3*B*C (or C*C) int64 counters leave the SMs.
//
// Counting never touches floating point after the arg-max, so any summation order gives the same
// integers: per-thread packed counters (C <= 4) or a per-CTA shared-memory histogram (C > 4) are
// merged into global int64 counters with atomics.
#include "dct_common.cuh"
#include "dct_tile.cuh"

namespace dct {

struct MetricArgs {
    const float* x;
    const int64_t* labels;
    int C;
    int64_t HW;
    int64_t* out;      // dice: [B][C][3] (I,G,P) ; confusion: [C][C]
    int32_t* flags;    // nullable
};

template <int CT>
constexpr int metric_vec() {
    return CT == 0 ? 1 : (CT <= 8 ? 4 : 2);
}

template <int VEC, int CM>
__device__ __forceinline__ void load_pixels(const float* xb, int C, int64_t HW, int64_t i, FVec<VEC> (&xin)[CM]) {
#pragma unroll
    for (int c = 0; c < CM; ++c)
        if (c < C) xin[c] = ld_stream<VEC>(xb + (int64_t)c * HW + i);
}

// ---------------------------------------------------------------------------------------------
// Dice counts of the shapes the tile pipeline's DiceOp does not take (C > 4, or rows it refuses).  grid = (gx, B): a CTA
// only sees pixels of image blockIdx.y.  Shared-memory histogram over (label row incl. one "invalid" row) x (prediction),
// one shared atomic per pixel; I/G/P are its diagonal, row sums and column sums.
// ---------------------------------------------------------------------------------------------
template <int CT, int VEC>
__global__ void __launch_bounds__(256) dice_kernel(const MetricArgs a) {
    constexpr int CM = CT ? CT : DCT_MAX_CLASSES;
    const int C = CT ? CT : a.C;
    const int64_t HW = a.HW;
    const int64_t gpi = HW / VEC;
    const int b = blockIdx.y;
    const float* xb = a.x + (int64_t)b * C * HW;
    const int64_t* lb = a.labels + (int64_t)b * HW;

    extern __shared__ int s_hist[];  // (C+1)*C ints
    const int nbins = (C + 1) * C;
    for (int j = threadIdx.x; j < nbins; j += blockDim.x) s_hist[j] = 0;
    __syncthreads();

    int nbad = 0;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < gpi; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = g * VEC;
        FVec<VEC> xin[CM];
        if constexpr (CT > 0) load_pixels<VEC, CM>(xb, C, HW, i, xin);
        long long lab[VEC];
        ld_labels<VEC>(lb + i, lab);
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            int pred;
            if constexpr (CT > 0) {
                float x[CM];
#pragma unroll
                for (int c = 0; c < CM; ++c) x[c] = xin[c].v[v];
                pred = spec_softmax_argmax<CM>(x);
            } else {
                pred = spec_softmax_argmax_rt(xb + i + v, C, HW);
            }
            const long long gl = lab[v];
            const bool valid = (gl >= 0) & (gl < C);
            nbad += !valid;
            const int row = valid ? (int)gl : C;
            atomicAdd(&s_hist[row * C + pred], 1);
        }
    }
    nbad = __reduce_add_sync(0xffffffffu, nbad);
    if ((threadIdx.x & 31) == 0 && nbad != 0 && a.flags != nullptr) atomicAdd(&a.flags[DCT_FLAG_LABEL], nbad);
    __syncthreads();
    unsigned long long* out = reinterpret_cast<unsigned long long*>(a.out) + (int64_t)b * C * 3;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        int vI = s_hist[c * C + c], vG = 0, vP = 0;
        for (int j = 0; j < C; ++j) vG += s_hist[c * C + j];
        for (int r = 0; r <= C; ++r) vP += s_hist[r * C + c];
        if (vI) atomicAdd(&out[c * 3 + 0], (unsigned long long)vI);
        if (vG) atomicAdd(&out[c * 3 + 1], (unsigned long long)vG);
        if (vP) atomicAdd(&out[c * 3 + 2], (unsigned long long)vP);
    }
}

// ---------------------------------------------------------------------------------------------
// Confusion matrix from raw scores: conf[gt][argmax x] += 1 over pixels with 0 <= gt < C.
// ---------------------------------------------------------------------------------------------
template <int CT, int VEC>
__global__ void __launch_bounds__(256) confusion_kernel(const MetricArgs a) {
    constexpr int CM = CT ? CT : DCT_MAX_CLASSES;
    const int C = CT ? CT : a.C;
    const int64_t HW = a.HW;
    const int64_t gpi = HW / VEC;
    const int b = blockIdx.y;
    const float* xb = a.x + (int64_t)b * C * HW;
    const int64_t* lb = a.labels + (int64_t)b * HW;
    extern __shared__ int s_hist[];
    for (int j = threadIdx.x; j < C * C; j += blockDim.x) s_hist[j] = 0;
    __syncthreads();
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < gpi; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = g * VEC;
        FVec<VEC> xin[CM];
        if constexpr (CT > 0) load_pixels<VEC, CM>(xb, C, HW, i, xin);
        long long lab[VEC];
        ld_labels<VEC>(lb + i, lab);
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            int pred;
            if constexpr (CT > 0) {
                float x[CM];
#pragma unroll
                for (int c = 0; c < CM; ++c) x[c] = xin[c].v[v];
                pred = raw_argmax<CM>(x);
            } else {
                pred = raw_argmax_rt(xb + i + v, C, HW);
            }
            const long long gl = lab[v];
            if ((gl >= 0) & (gl < C)) atomicAdd(&s_hist[(int)gl * C + pred], 1);
        }
    }
    __syncthreads();
    unsigned long long* out = reinterpret_cast<unsigned long long*>(a.out);
    for (int j = threadIdx.x; j < C * C; j += blockDim.x) {
        int v = s_hist[j];
        if (v) atomicAdd(&out[j], (unsigned long long)v);
    }
}

// integer prediction map variant (IoU.add with [N,H,W] ints, iou.py:49-50)
__global__ void __launch_bounds__(256) confusion_labels_kernel(const int64_t* pred, const int64_t* labels, int64_t n, int C,
                                                               int64_t* conf, int32_t* flags) {
    extern __shared__ int s_hist[];
    for (int j = threadIdx.x; j < C * C; j += blockDim.x) s_hist[j] = 0;
    __syncthreads();
    int nbad = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const long long gl = labels[i];
        if ((gl >= 0) & (gl < C)) {
            const long long key = pred[i] + (long long)C * gl;
            if ((key >= 0) & (key < (long long)C * C)) atomicAdd(&s_hist[(int)key], 1);
            else ++nbad;
        }
    }
    nbad = __reduce_add_sync(0xffffffffu, nbad);
    if ((threadIdx.x & 31) == 0 && nbad != 0 && flags != nullptr) atomicAdd(&flags[DCT_FLAG_PRED], nbad);
    __syncthreads();
    unsigned long long* out = reinterpret_cast<unsigned long long*>(conf);
    for (int j = threadIdx.x; j < C * C; j += blockDim.x) {
        int v = s_hist[j];
        if (v) atomicAdd(&out[j], (unsigned long long)v);
    }
}

// meta_dice's closing arithmetic in float32 (dice_meter.py:17-20)
__global__ void dice_from_counts_kernel(const int64_t* counts, int64_t B, int C, int batch_sum, float* dice) {
    const int64_t rows = batch_sum ? 1 : B;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < rows * C; j += (int64_t)gridDim.x * blockDim.x) {
        long long I = 0, G = 0, P = 0;
        if (batch_sum) {
            for (int64_t b = 0; b < B; ++b) {
                const int64_t* r = counts + (b * C + j) * 3;
                I += r[0]; G += r[1]; P += r[2];
            }
        } else {
            const int64_t* r = counts + j * 3;
            I = r[0]; G = r[1]; P = r[2];
        }
        const float inter = (float)I;
        const float sum = (float)(G + P);
        dice[j] = __fdiv_rn(__fadd_rn(__fmul_rn(2.0f, inter), 1e-8f), __fadd_rn(sum, 1e-8f));
    }
}

// Dice counting as a tile-pipeline Op (C <= 4): no outputs, one counted tensor
struct DiceOp {
    static constexpr int NIN = 1, NOUT = 0, NDICE = 1;
    static constexpr bool HAS_MAP = false, USES_UP = false, CHECKS_SIMPLEX = false, GMAP = false;
    template <int CM, class T>
    static __device__ __forceinline__ T apply(T (&)[1][CM], int, T, float, bool&) { return vset<T>(0.0f); }
};

template <int CT>
static int dice_launch_ct(const MetricArgs& a, int64_t B, cudaStream_t s) {
    if constexpr (CT > 0 && CT <= 4) {
        TileArgs t{};
        t.in[0] = a.x; t.HW = a.HW; t.flags = a.flags; t.labels = a.labels;
        t.counts = reinterpret_cast<unsigned long long*>(a.out); t.count_view_stride = B * CT * 3;
        if (tile_eligible<DiceOp>(t, B)) return tile_launch_ct<DiceOp, CT>(t, B, s);
        return DCT_ERR_UNSUPPORTED;   // the caller falls back to dice_kernel<0, 1>
    } else {
        constexpr int VEC = metric_vec<CT>();
        if ((a.HW % VEC) != 0 || !aligned(a.x, 4 * VEC) || !aligned(a.labels, VEC >= 2 ? 16 : 8)) return DCT_ERR_UNSUPPORTED;
        const int C = CT ? CT : a.C;
        const size_t smem = sizeof(int) * (C + 1) * C;
        // each thread takes ~4 pixel groups so that the per-CTA merge (<= 3C global atomics) amortises
        int64_t gpi = a.HW / VEC;
        int64_t gx = (gpi + 256 * 4 - 1) / (256 * 4);
        if (gx > 65535) gx = 65535;
        dice_kernel<CT, VEC><<<dim3((unsigned)gx, (unsigned)B), 256, smem, s>>>(a);
        return check_launch();
    }
}

template <int CT>
static int confusion_launch_ct(const MetricArgs& a, int64_t B, cudaStream_t s) {
    constexpr int VEC = metric_vec<CT>();
    if ((a.HW % VEC) != 0 || !aligned(a.x, 4 * VEC) || !aligned(a.labels, VEC >= 2 ? 16 : 8)) return DCT_ERR_UNSUPPORTED;
    const int C = CT ? CT : a.C;
    const size_t smem = sizeof(int) * C * C;
    int64_t gpi = a.HW / VEC;
    int64_t gx = (gpi + 256 * 8 - 1) / (256 * 8);   // C*C global atomics per CTA: give each CTA more pixels
    if (gx > 65535) gx = 65535;
    confusion_kernel<CT, VEC><<<dim3((unsigned)gx, (unsigned)B), 256, smem, s>>>(a);
    return check_launch();
}

static int metric_validate(const float* x, const int64_t* labels, int C, int64_t B, int64_t HW, const void* out) {
    if (x == nullptr || labels == nullptr || out == nullptr || C < 1 || B < 1 || HW < 1) return DCT_ERR_BAD_ARG;
    if (C > DCT_MAX_CLASSES || B > 65535) return DCT_ERR_UNSUPPORTED;
    if (!aligned(x, 4) || !aligned(labels, 8) || !aligned(out, 8)) return DCT_ERR_MISALIGNED;
    return DCT_OK;
}

}  // namespace dct

using namespace dct;

extern "C" int dct_dice_counts_f32(const float* x, const int64_t* labels, int C, int64_t B, int64_t HW,
                                   int64_t* counts, int accumulate, int32_t* flags, void* stream) {
    int rc = metric_validate(x, labels, C, B, HW, counts);
    if (rc != DCT_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!accumulate) {
        cudaError_t e = cudaMemsetAsync(counts, 0, sizeof(int64_t) * (size_t)(B * C * 3), s);
        if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    }
    MetricArgs a{x, labels, C, HW, counts, flags};
    rc = DCT_ERR_UNSUPPORTED;
    switch (C) {
        case 2: rc = dice_launch_ct<2>(a, B, s); break;
        case 3: rc = dice_launch_ct<3>(a, B, s); break;
        case 4: rc = dice_launch_ct<4>(a, B, s); break;
        case 19: rc = dice_launch_ct<19>(a, B, s); break;
        default: break;
    }
    if (rc == DCT_ERR_UNSUPPORTED) rc = dice_launch_ct<0>(a, B, s);
    return rc;
}

extern "C" int dct_dice_from_counts_f32(const int64_t* counts, int64_t B, int C, int batch_sum, float* dice,
                                        void* stream) {
    if (counts == nullptr || dice == nullptr || B < 1 || C < 1) return DCT_ERR_BAD_ARG;
    const int64_t n = (batch_sum ? 1 : B) * C;
    const int threads = 128;
    const int blocks = (int)((n + threads - 1) / threads);
    dice_from_counts_kernel<<<blocks > 1024 ? 1024 : blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(
        counts, B, C, batch_sum, dice);
    return check_launch();
}

extern "C" int dct_confusion_f32(const float* x, const int64_t* labels, int C, int64_t B, int64_t HW,
                                 int64_t* conf, void* stream) {
    int rc = metric_validate(x, labels, C, B, HW, conf);
    if (rc != DCT_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    MetricArgs a{x, labels, C, HW, conf, nullptr};
    rc = DCT_ERR_UNSUPPORTED;
    switch (C) {
        case 2: rc = confusion_launch_ct<2>(a, B, s); break;
        case 3: rc = confusion_launch_ct<3>(a, B, s); break;
        case 4: rc = confusion_launch_ct<4>(a, B, s); break;
        case 19: rc = confusion_launch_ct<19>(a, B, s); break;
        default: break;
    }
    if (rc == DCT_ERR_UNSUPPORTED) rc = confusion_launch_ct<0>(a, B, s);
    return rc;
}

extern "C" int dct_confusion_labels_i64(const int64_t* pred, const int64_t* labels, int64_t n, int C,
                                        int64_t* conf, int32_t* flags, void* stream) {
    if (pred == nullptr || labels == nullptr || conf == nullptr || n < 1 || C < 1) return DCT_ERR_BAD_ARG;
    if (C > DCT_MAX_CLASSES) return DCT_ERR_UNSUPPORTED;
    if (!aligned(pred, 8) || !aligned(labels, 8) || !aligned(conf, 8)) return DCT_ERR_MISALIGNED;
    int64_t blocks = (n + 256 * 8 - 1) / (256 * 8);
    if (blocks > 148 * 8) blocks = 148 * 8;
    confusion_labels_kernel<<<(unsigned)blocks, 256, sizeof(int) * C * C, static_cast<cudaStream_t>(stream)>>>(
        pred, labels, n, C, conf, flags);
    return check_launch();
}

// Developer check (host only, no GPU needed): the image index the tile pipeline's schedule computes for `tile` when an image
// holds `tiles_per_image` tiles -- the multiplier form of tile / tiles_per_image (tile_set_geometry / tile_image, dct_tile.cuh).
// tests/test_abi_and_host.py compares it with the integer division over the whole range of divisors and edge tiles.
extern "C" int dct_dev_tile_image(int tiles_per_image, int tile) {
    if (tiles_per_image < 1 || tile < 0) return DCT_ERR_BAD_ARG;
    TileArgs a{};
    a.HW = tiles_per_image;   // one-pixel tiles: tiles_per_image == HW
    tile_set_geometry(a, 1, 1);
    return tile_image(a, tile);
}
