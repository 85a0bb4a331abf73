// dct_tile.cuh -- the tile pipeline: one persistent-CTA skeleton for every per-pixel op of the path.
//
//   HBM --(TMA: tensor-map boxes or 1-D bulk copies, mbarrier)--> smem stage [NIN*C][TP] --> registers --> math
//   HBM <--(TMA stores, bulk groups)------------------------------- smem stage (results written in place) <----'
//
// A tile is TP = THREADS*PPT consecutive pixels of one image; in NCHW every (tensor, class) plane
// contributes one contiguous TP*4-byte row segment.  Stages of 5 or more rows whose tile is one box of
// <= 256 pixels are moved by ONE cp.async.bulk.tensor per tensor (SASS UTMALDG / UTMASTG, dct_tmap.cuh);
// the 4-row stages by one cp.async.bulk per row (SASS UBLKCP).
// STAGES-1 tiles are in flight per CTA at all times, so HBM latency is covered by shared-memory
// depth rather than by resident warps and registers (the register-tiled kernels top out at
// ~68% of the measured HBM peak on ACDC-sized inputs because raising occupancy forces spills).
// Results go back through the same stage with bulk stores; a stage is refilled once its store
// group has finished reading it.  Grid = min(#tiles, 148 * MINB) persistent CTAs, each owning a
// CONTIGUOUS range of tiles (so per-image integer counters rarely need flushing).
//
// Ops plug in through a small static interface (see dct_pixelwise.cuh for the same Ops on the
// register-tiled fallback):
//   NIN, NOUT        number of [B,C,HW] input / output tensors (output n reuses input n's rows)
//   HAS_MAP          produces a per-pixel scalar (map store and/or deterministic grid sum)
//   USES_UP          consumes an upstream gradient (gconst * *gscalar [* gmap[pixel] if GMAP])
//   GMAP             the upstream may carry a per-pixel map (reserves one side row per stage)
//   CHECKS_SIMPLEX   sets the simplex flag through `bad`
//   NDICE            number of leading input tensors whose Dice counts are accumulated (0 = none)
//   apply<CM>(x[NIN][CM], C, g, eps, bad) -> map value; outputs left in x[0..NOUT)
//   LABELS (optional) the op itself consumes the int64 label of every pixel (supervised cross-entropy): it then
//                    provides apply_lab<CM>(x, C, g, cls[LW], w[LW], bad) instead, with cls = label in [0,C) or -1
//                    (ignored / out of range) and w = class weight of the label (0 when cls < 0 or ignored)
//   SUM2 (optional)  a second per-pixel scalar with its own deterministic grid sum (TileArgs::sum2): the op then provides
//                    apply<CM>(x, C, g, eps, bad, v2) instead, which also leaves the second value in v2
//   CONF (optional)  the kernel also counts the confusion matrix conf[gt][argmax x] of input tensor 0 against the labels
//                    (IoU.add / ConfusionMatrix.add, generalframework/metrics/iou.py:43-69, confusionmatrix.py:32-85):
//                    raw arg-max with torch.max semantics, labels outside [0,C) dropped (ignore-255 included)
#pragma once
#include <cuda_bf16.h>

#include "dct_common.cuh"
#include "dct_tma.cuh"
#include "dct_tmap.cuh"

namespace dct {

// Element type of the [B,C,HW] tensors a tile kernel moves: float (the reference's dtype) or __nv_bfloat16 (networks
// under autocast; the math is fp32 in registers either way, only the HBM / shared-memory rows are 2-byte).
using bf16 = __nv_bfloat16;

// PPT consecutive elements of one shared-memory row -> fp32 registers, and back (round-to-nearest-even)
template <int PPT, class ET>
__device__ __forceinline__ FVec<PPT> tile_ld_row(const unsigned char* row, int p0) {
    if constexpr (std::is_same<ET, float>::value) {
        return *reinterpret_cast<const FVec<PPT>*>(row + (size_t)p0 * 4);
    } else {
        FVec<PPT> r;
        const uint32_t* w = reinterpret_cast<const uint32_t*>(row + (size_t)p0 * 2);
        if constexpr (PPT == 1) {
            r.v[0] = __uint_as_float((uint32_t)(*reinterpret_cast<const uint16_t*>(row + (size_t)p0 * 2)) << 16);
        } else if constexpr (PPT == 2) {
            const uint32_t u = w[0];
            r.v[0] = __uint_as_float(u << 16); r.v[1] = __uint_as_float(u & 0xffff0000u);
        } else {
            const uint2 u = *reinterpret_cast<const uint2*>(w);
            r.v[0] = __uint_as_float(u.x << 16); r.v[1] = __uint_as_float(u.x & 0xffff0000u);
            r.v[2] = __uint_as_float(u.y << 16); r.v[3] = __uint_as_float(u.y & 0xffff0000u);
        }
        return r;
    }
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t u;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(u) : "f"(hi), "f"(lo));
    return u;
}
template <int PPT, class ET>
__device__ __forceinline__ void tile_st_row(unsigned char* row, int p0, const FVec<PPT>& r) {
    if constexpr (std::is_same<ET, float>::value) {
        *reinterpret_cast<FVec<PPT>*>(row + (size_t)p0 * 4) = r;
    } else {
        uint32_t* w = reinterpret_cast<uint32_t*>(row + (size_t)p0 * 2);
        if constexpr (PPT == 1) *reinterpret_cast<uint16_t*>(row + (size_t)p0 * 2) = (uint16_t)(pack_bf16x2(r.v[0], 0.0f) & 0xffffu);
        else if constexpr (PPT == 2) w[0] = pack_bf16x2(r.v[0], r.v[1]);
        else *reinterpret_cast<uint2*>(w) = make_uint2(pack_bf16x2(r.v[0], r.v[1]), pack_bf16x2(r.v[2], r.v[3]));
    }
}

// Fused Dice counters (NDICE > 0): every consumer thread keeps its packed 8-bit counters in registers ACROSS tiles.  The
// producer marks the tiles after which they must be handed over (the CTA's next tile belongs to another image or does not
// exist, or a field could overflow); only on a marked tile do the consumer warps reduce their counters into their slice of
// the stage's label row, and the producer warp adds the 8 warps' numbers to the global int64 counters -- a handful of
// times per CTA, nothing Dice-related in the other tiles but the per-pixel arg-max.  Measured (profiles/r19, r20): a fold
// through the producer on EVERY tile 41.9 us at c2; consumer warps adding to global memory themselves 41.6 us at c2 but
// +1 us at c1 / +2.7 us at c3-sized inputs (8x the atomics on a few dozen addresses at the kernel's end); marked tiles:
// see profiles/r20/kbench_dice_ab.log.
// (An experiment that handed the last level(s) of the tail pool out as 2 or 4 sub-tiles per tile -- to shrink the CTAs' end
// spread below one tile's service time -- was measured and removed: the extra indirection in the tile loop cost far more
// than the tail it saved: c2 step 106.2 -> 124.2 (2 sub-tiles) / 136.4 us (4), c4 1.385 -> 1.738 ms; profiles/r26/ab_split.log.)
constexpr int kTileMaxTensors = 8;
constexpr int kTileMaxRows = 80;   // NIN*C rows per stage

struct TileArgs {
    const void* in[kTileMaxTensors];   // [B,C,HW] of the kernel's element type (float or bf16)
    void* out[kTileMaxTensors];        // each nullable; same element type
    int64_t HW;
    float* map;                    // nullable
    double* sum;                   // nullable
    Upstream up;
    float eps;
    int32_t* flags;                // nullable
    Workspace* ws;
    const int64_t* labels;         // Dice: [B,HW] int64 (NDICE > 0 and non-null => count)
    unsigned long long* counts;    // Dice: [NDICE][B][C][3] (I,G,P), accumulated into
    int64_t count_view_stride;     // B*C*3
    int counts_overwrite;          // Dice: 1 = this launch clears `counts` first (CTA 0; the others wait for ws->counts_zeroed)
    PeerPub pub;                   // *_pub launches (PUB kernels): publication descriptor of the step's sums, by value
    int pub_early;                 // PUB kernels: 1 = `pub.src` is already final (the PREVIOUS step's sums): the first CTA to finish
                                   // publishes it; 0 = the last CTA publishes, with the sum this launch has just produced
    unsigned long long* conf;      // CONF ops: [C][C] int64 (rows = ground truth), accumulated into; null = not counted
    const float* class_w;          // LABELS ops: per-class weight [C] (device) or null = 1
    int64_t ignore_index;          // LABELS ops: label value that contributes nothing (nn.NLLLoss ignore_index)
    int tiles_per_image;
    int num_tiles;
    unsigned int tpi_mul;          // tile / tiles_per_image without a division (tile_set_geometry): q = (t + ((n - t) >> tpi_sh1)) >> tpi_sh2,
    int tpi_sh1, tpi_sh2;          //   t = umulhi(tpi_mul, n) -- exact for every 32-bit n
    int refill;                    // 1: a drained stage is refilled as soon as ITS OWN store group has been read; 0: one tile later
    int pool_div;                  // developer switch (tools/kbench_*.cu): the tail pool is 1/pool_div of every CTA's range (0 = default 5)
    int prefetch;                  // tiles of this CTA's range whose rows are prefetched into L2 before the dependency wait
    int force_static;              // developer switch (tools/kbench_tile.cu): 1 = no tail pool (purely static contiguous ranges) even with a workspace
    unsigned long long* trace;     // developer tracing: kTraceSlots words per CTA (start, first tile landed, -, end, tiles done,
                                   // stores read out, ticket drawn) in ns; null in the product
    double* sum2;                  // SUM2 ops: grid sum of the second per-pixel value (nullable)
};

// Tensor maps of a launch whose stages are filled / drained by tensor-map TMA (dct_tmap.cuh): second kernel parameter,
// __grid_constant__ (the copy instructions take the descriptors' addresses in parameter space).  Empty otherwise.
template <bool TMAP>
struct TileMaps {
    int unused;
};
template <>
struct alignas(64) TileMaps<true> {
    CUtensorMap in[kTileMaxTensors];
    CUtensorMap out[kTileMaxTensors];
};

// does the op read the labels itself (Op::LABELS == true)?  Ops without the member do not.
template <class Op, class = void>
struct op_labels : std::false_type {};
template <class Op>
struct op_labels<Op, std::enable_if_t<Op::LABELS>> : std::true_type {};
template <class Op, class = void>
struct op_conf : std::false_type {};
template <class Op>
struct op_conf<Op, std::enable_if_t<Op::CONF>> : std::true_type {};
template <class Op, class = void>
struct op_sum2 : std::false_type {};
template <class Op>
struct op_sum2<Op, std::enable_if_t<Op::SUM2>> : std::true_type {};
template <class Op>
constexpr bool op_label_row() { return Op::NDICE > 0 || op_labels<Op>::value || op_conf<Op>::value; }

// data rows + optional side rows: int64 labels (Dice / label ops) and the fp32 upstream-gradient map (backward ops);
// in BYTES per pixel
template <class Op, int CT, class ET = float>
constexpr int tile_row_bytes() {
    return Op::NIN * CT * (int)sizeof(ET) + (op_label_row<Op>() ? 8 : 0) + (Op::GMAP ? 4 : 0);
}
template <class Op, int CT>
constexpr int tile_row_words() { return tile_row_bytes<Op, CT, float>() / 4; }

// one tensor's C rows of a tile; with tensor-map TMA every tensor's box starts on a 128-byte boundary of the stage
template <int CT, int TP, class ET, bool TMAP>
constexpr size_t tile_tensor_stride() {
    constexpr size_t raw = (size_t)CT * TP * sizeof(ET);
    return TMAP ? (raw + 127) / 128 * 128 : raw;
}
template <class Op, int CT, int TP, class ET, bool TMAP>
constexpr size_t tile_stage_bytes() {
    return Op::NIN * tile_tensor_stride<CT, TP, ET, TMAP>() + (op_label_row<Op>() ? (size_t)TP * 8 : 0) + (Op::GMAP ? (size_t)TP * 4 : 0);
}

template <size_t STAGE_BYTES, int MINB>
constexpr int tile_stages() {
    // as many stages as fit in this CTA's share of shared memory, between 2 and 8
    // 228 KB per SM, 1 KB reserved per CTA, < 1 KB of static shared memory + barriers + alignment slack
    constexpr size_t n = (233472 / MINB - 2048) / STAGE_BYTES;
    return n < 2 ? 2 : (n > 8 ? 8 : (int)n);
}

template <class Op, int CT, int PPT, int CTHREADS, int STAGES, class ET = float, bool TMAP = false>
struct TileCfg {
    static constexpr int TP = CTHREADS * PPT;                       // pixels per tile
    static constexpr int ROWS = Op::NIN * CT;                       // data rows (element type ET)
    static constexpr int ES = (int)sizeof(ET);
    static constexpr size_t kTensorStride = tile_tensor_stride<CT, TP, ET, TMAP>();   // tensor n's rows start at n * kTensorStride
    static constexpr size_t kStageBytes = tile_stage_bytes<Op, CT, TP, ET, TMAP>();
    static constexpr size_t kRowBytes = (size_t)TP * ES;            // one data row
    static constexpr size_t kLabelOffB = Op::NIN * kTensorStride;   // in bytes; labels are 8-byte, TP*8 bytes
    static constexpr size_t kGmapOffB = kLabelOffB + (op_label_row<Op>() ? (size_t)TP * 8 : 0);  // valid when Op::GMAP (fp32 row)
    static constexpr size_t kSmemBytes = kStageBytes * STAGES + 16 * STAGES;
    static_assert(!TMAP || (TP <= 256 && kStageBytes % 128 == 0), "tensor-map stages: one box per tensor, 128-byte aligned");
    __host__ __device__ static constexpr size_t row_off(int n, int c) { return (size_t)n * kTensorStride + (size_t)c * kRowBytes; }
};

// image index of a tile: division by the launch's tiles_per_image through a precomputed multiplier (the hardware has no
// integer divide: `tile / tpi` is ~25 dependent instructions incl. a MUFU.RCP, once per tile in the producer lane's critical
// path and -- before the producer published the image index with the tile -- once per tile in every consumer thread)
__host__ __device__ __forceinline__ int tile_image(const TileArgs& a, int tile) {
    const unsigned int n = (unsigned int)tile;
#ifdef __CUDA_ARCH__
    const unsigned int t = __umulhi(a.tpi_mul, n);
#else
    const unsigned int t = (unsigned int)(((unsigned long long)a.tpi_mul * n) >> 32);   // (dct_dev_tile_image: host-side check)
#endif
    return (int)((t + ((n - t) >> a.tpi_sh1)) >> a.tpi_sh2);
}
inline void tile_set_geometry(TileArgs& a, int64_t B, int tile_pixels) {
    a.tiles_per_image = (int)((a.HW + tile_pixels - 1) / tile_pixels);
    a.num_tiles = (int)(a.tiles_per_image * B);
    const unsigned int d = (unsigned int)a.tiles_per_image;
    int l = 0;
    while ((1ull << l) < d) ++l;                                   // ceil(log2 d)
    a.tpi_mul = (unsigned int)((((1ull << l) - d) << 32) / d + 1);   // Granlund-Montgomery round-up multiplier (33-bit form)
    a.tpi_sh1 = l < 1 ? l : 1;
    a.tpi_sh2 = l < 1 ? 0 : l - 1;
}

// Warp-specialised persistent kernel: NCW consumer warps + 1 producer warp per CTA.
//   producer: lane 0 owns the tile schedule (a contiguous range per CTA whose last fifth is shared through an
//       atomic counter, see draw() below), publishes each tile index in the stage's shared-memory slot, issues every
//       bulk load / store, and recycles a stage when its `done` mbarrier (NCW arrivals) has completed and, for ops
//       with outputs, when the bulk store group that drains it has finished reading shared memory.  Fused Dice: lane 0
//       marks the last tile of every run of one image (s_info.w); on those tiles all 32 lanes add the counters the
//       consumer warps hand over through the label row to the global int64 counters (see "Fused Dice counters" above).
//   consumers: wait on the stage's `full` mbarrier (transaction bytes), read the stage's info word (tile -1 = no more work),
//       compute in registers, write results back in place, fence to the async proxy, arrive on `done`.
//       No CTA-wide barrier in the tile loop: a fast warp runs ahead by up to STAGES-1 tiles.
// Nothing depends on WHICH CTA processes a tile: Dice counts are integer atomics, the loss sum is accumulated in
// exact fixed point (tile_grid_finish), so results are bit-reproducible under the dynamic part of the schedule.
// TMAP: the data rows move by tensor-map TMA, one copy per tensor and tile each way (dct_tmap.cuh); side rows (labels,
// upstream map) stay 1-D bulk copies.  A ragged last tile of an image needs no special casing for the data rows then:
// the box is filled with zeros beyond the image (the transaction count is always the whole box) and clipped on the way out.
template <class Op, int CT, int PPT, int NCW, int STAGES, int MINB = 1, class ET = float, bool PUB = false, bool TMAP = false>
__global__ void __launch_bounds__(NCW * 32 + 32, MINB) tile_kernel(const TileArgs a, const __grid_constant__ TileMaps<TMAP> maps) {
    constexpr int CTHREADS = NCW * 32;
    using Cfg = TileCfg<Op, CT, PPT, CTHREADS, STAGES, ET, TMAP>;
    constexpr int TP = Cfg::TP, ROWS = Cfg::ROWS, ES = Cfg::ES, NIN = Op::NIN, NOUT = Op::NOUT, C = CT;
    constexpr bool DICE = Op::NDICE > 0;         // fused Dice counts (see "Fused Dice counters" above)
    constexpr bool LAB = op_labels<Op>::value;   // the op consumes the labels itself
    constexpr bool CONF = op_conf<Op>::value;    // confusion counts of tensor 0 vs the labels (CTA-shared histogram)
    constexpr bool LROW = DICE || LAB || CONF;   // the stage carries a label row
    constexpr bool SUM2 = op_sum2<Op>::value;    // a second per-pixel value and grid sum
    constexpr int LW = (PPT % 2 == 0) ? 2 : 1;   // pixels per math lane group: pairs use packed FP32x2
    constexpr int NG = PPT / LW;
    using T = typename std::conditional<LW == 2, f2, float>::type;
    static_assert(!DICE || CT <= 4, "fused Dice counters are packed 8-bit fields: C <= 4");
    static_assert(!DICE || PPT <= 4, "per-tile packed Dice counters: 32 lanes * PPT must stay below 256");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char* stages = smem_raw;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + Cfg::kStageBytes * STAGES);
    uint64_t* done = full + STAGES;
    // per stage, written by the producer lane before the stage's `full` barrier is armed: x = tile index held by the stage
    // (-1 = end of work), y = its image, z = its pixel count (a ragged last tile of an image is shorter than TP),
    // w = Dice: 1 = hand the Dice counters over after this tile
    __shared__ int4 s_info[STAGES];
    __shared__ unsigned int s_conf[CONF ? CT * CT : 1];   // this CTA's confusion counts (flushed once, at the end)
    const int tid = threadIdx.x, lane = tid & 31;
    const bool is_producer = tid >= CTHREADS;
    const int64_t HW = a.HW;
    const int tpi = a.tiles_per_image;
    const bool do_lab = LROW && a.labels != nullptr;
    const bool do_dice = DICE && do_lab;
    const bool do_conf = CONF && do_lab && a.conf != nullptr;
    if constexpr (CONF) {
        for (int i = tid; i < CT * CT; i += (int)blockDim.x) s_conf[i] = 0u;
    }
    const bool has_gmap = Op::GMAP && a.up.gmap != nullptr;
    const bool dynamic = a.ws != nullptr && !a.force_static;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            tma::mbar_init(&full[s], 1);
            tma::mbar_init(&done[s], NCW);
        }
        tma::fence_barrier_init();
    }
    if constexpr (TMAP) {   // descriptor fetch overlaps the previous grid's tail (before the dependency wait)
        if (tid == CTHREADS) {
#pragma unroll
            for (int n = 0; n < NIN; ++n) tma::prefetch_tensormap(&maps.in[n]);
#pragma unroll
            for (int n = 0; n < NOUT; ++n) tma::prefetch_tensormap(&maps.out[n]);
        }
    }
    __syncthreads();
    // Ramp hiding.  This CTA's first tiles are known before anything of the previous grid is (contiguous static ranges), so
    // their rows are pulled into L2 while that grid is still draining: resident since its first CTAs left, this grid would
    // otherwise idle in the dependency wait and then pay a cold DRAM round trip for its first stage (first data 1.6-2.5 us
    // after the wait, profiles/r26).  A prefetch moves no value into the SM: ordering against the previous grid's writes is
    // untouched (L2 is the point of coherence; a line it still rewrites is simply updated in place).
    if (a.prefetch > 0 && tid == CTHREADS) {
        const int per = a.num_tiles / (int)gridDim.x, extra = a.num_tiles % (int)gridDim.x;
        const int my_begin = (int)blockIdx.x * per + min((int)blockIdx.x, extra);
        const int my_n = per + ((int)blockIdx.x < extra ? 1 : 0);
        const int npre = min(min(a.prefetch, STAGES), my_n);
        for (int s = 0; s < npre; ++s) {
            const int tile = my_begin + s, b = tile_image(a, tile);
            const int64_t off = (int64_t)(tile - b * tpi) * TP;
            const int64_t rem = HW - off;
            const uint32_t npix = (uint32_t)(rem < TP ? rem : TP);
            if constexpr (TMAP) {
#pragma unroll
                for (int n = 0; n < NIN; ++n) tma::tensor_prefetch_3d(&maps.in[n], (int)off, 0, b);
            } else {
#pragma unroll
                for (int n = 0; n < NIN; ++n)
#pragma unroll
                    for (int c = 0; c < C; ++c)
                        tma::bulk_prefetch_l2(static_cast<const ET*>(a.in[n]) + ((int64_t)b * C + c) * HW + off, npix * (uint32_t)ES);
            }
            if constexpr (LROW) {
                if (do_lab) tma::bulk_prefetch_l2(a.labels + (int64_t)b * HW + off, 8u * npix);
            }
            if constexpr (Op::GMAP) {
                if (has_gmap) tma::bulk_prefetch_l2(a.up.gmap + (int64_t)b * HW + off, 4u * npix);
            }
        }
    }
    pdl_wait();               // the previous grid has completed and its writes are visible (no-op without PDL)
    if (a.trace != nullptr && tid == 0) a.trace[kTraceSlots * blockIdx.x] = globaltimer_ns();
    if constexpr (DICE) {
        // DCT_COUNTS_OVERWRITE: the launch clears its own counters.  CTA 0 stores the zeros and releases a flag; every
        // other CTA's producer warp acquires it before its first add (by then -- a whole run of tiles later -- it has long
        // been set).  All CTAs of the persistent grid are co-resident and CTA 0 never waits on anybody: no deadlock.
        if (do_dice && a.counts_overwrite && blockIdx.x == 0) {
            const int64_t ncnt = (int64_t)Op::NDICE * a.count_view_stride;
            for (int64_t i = tid; i < ncnt; i += (int64_t)blockDim.x) a.counts[i] = 0ull;
            __threadfence();
            __syncthreads();
            if (tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(&a.ws->counts_zeroed), "r"(1u) : "memory");
        }
    }

    FxAcc acc_fx;             // this thread's share of the map sum, 2^-40 fixed point
    bool nonfinite = false;
    FxAcc acc_fx2;            // SUM2: the same for the second value
    bool nonfinite2 = false;
    bool bad = false;

    if (is_producer) {
        // scheduling state lives in lane 0; the other lanes only help with the Dice counter flush
        // Tile schedule: every CTA owns a CONTIGUOUS range of tiles (image locality: its Dice counters change image
        // once or twice), but the last fifth of every range goes to a pool that is handed out through an atomic counter
        // in the workspace: CTAs on faster SMs finish their own share early and drain the pool, which removes a
        // measured 10 us spread of CTA finishing times on a 40 us kernel.  Pool draws are made one tile ahead of use.
        const int per = a.num_tiles / (int)gridDim.x, extra = a.num_tiles % (int)gridDim.x;
        const int my_begin = (int)blockIdx.x * per + min((int)blockIdx.x, extra);
        const int my_n = per + ((int)blockIdx.x < extra ? 1 : 0);
        const int pool_q = dynamic ? per / (a.pool_div > 0 ? a.pool_div : 5) : 0;             // pool tiles taken from the end of every CTA's range
        const int my_static = my_n - pool_q;
        int draws = 0;
        // (A tapered look-ahead -- fewer loads in flight per CTA the deeper a draw lands in the pool, so that the last tiles
        // stay unclaimed for whichever CTA frees up first -- was measured and removed: the end spread did not shrink and the
        // thinner pipelines cost bandwidth: c2 step 102.3 -> 109.8 us, profiles/r30/ab_taper.log.)
        auto draw = [&]() -> int {  // next tile index for this CTA; >= num_tiles when there is no more work
            int t;
            if (draws < my_static) t = my_begin + draws;
            else if (pool_q == 0) t = a.num_tiles;
            else {
                // inline PTX: the compiler's warp-aggregated atomicAdd shuffles the result right away, which
                // would expose the atomic's round trip at every draw; this way it is consumed one tile later
                unsigned int got;
                asm volatile("atom.global.relaxed.gpu.add.u32 %0, [%1], 1;" : "=r"(got) : "l"(&a.ws->tile_counter) : "memory");
                const int j = (int)(got % gridDim.x), k = (int)(got / gridDim.x);  // k-th pool tile of CTA j's range
                t = k < pool_q ? j * per + min(j, extra) + per + (j < extra ? 1 : 0) - pool_q + k : a.num_tiles;
            }
            ++draws;
            return t;
        };
        int run_b = -1, run_len = 0;               // Dice: image and length of the current run of tiles (lane 0)
        constexpr int kDiceMaxTiles = 255 / PPT;   // a packed 8-bit field grows by at most PPT per tile
        int issued = 0;        // loads issued so far; the k-th goes to stage k % STAGES
        bool more = true;
        int pending = 0;       // drawn one ahead of its use
        auto try_issue = [&]() {  // lane 0 only
            if (!more) return;
            const int tile = pending, stage = issued % STAGES;
            if (tile >= a.num_tiles) {  // publish "no more work" through the same barrier
                more = false;
                s_info[stage] = make_int4(-1, 0, 0, 0);
                tma::mbar_arrive(&full[stage]);
                return;
            }
            pending = draw();
            const int b = tile_image(a, tile);
            int mark = 0;
            if constexpr (DICE) {
                // last tile of a run of one image (or of this CTA's work), or the run is as long as an 8-bit field allows
                run_len = (b == run_b) ? run_len + 1 : 1;
                run_b = b;
                mark = (pending >= a.num_tiles || tile_image(a, pending) != b || run_len == kDiceMaxTiles) ? 1 : 0;
                if (mark) run_b = -1;
            }
            const int64_t off = (int64_t)(tile - b * tpi) * TP;
            const int64_t rem = HW - off;
            const uint32_t npix = (uint32_t)(rem < TP ? rem : TP);
            s_info[stage] = make_int4(tile, b, (int)npix, mark);
            const uint32_t bytes = npix * (uint32_t)ES;   // one data row segment
            unsigned char* dst = stages + (size_t)stage * Cfg::kStageBytes;
            uint32_t total = TMAP ? (uint32_t)(ROWS * TP * ES) : bytes * ROWS;   // (a box always completes whole)
            if constexpr (LROW) total += do_lab ? 8u * npix : 0u;
            if constexpr (Op::GMAP) total += has_gmap ? 4u * npix : 0u;
            tma::mbar_expect_tx(&full[stage], total);  // release: the tile index above is visible to the waiters
            if constexpr (TMAP) {
#pragma unroll
                for (int n = 0; n < NIN; ++n)
                    tma::tensor_load_3d(dst + (size_t)n * Cfg::kTensorStride, &maps.in[n], (int)off, 0, b, &full[stage]);
            } else {
#pragma unroll
                for (int n = 0; n < NIN; ++n)
#pragma unroll
                    for (int c = 0; c < C; ++c)
                        tma::bulk_load(dst + Cfg::row_off(n, c),
                                       static_cast<const ET*>(a.in[n]) + ((int64_t)b * C + c) * HW + off, bytes, &full[stage]);
            }
            if constexpr (LROW) {
                if (do_lab) tma::bulk_load(dst + Cfg::kLabelOffB, a.labels + (int64_t)b * HW + off, 8u * npix, &full[stage]);
            }
            if constexpr (Op::GMAP) {
                if (has_gmap) tma::bulk_load(dst + Cfg::kGmapOffB, a.up.gmap + (int64_t)b * HW + off, 4u * npix, &full[stage]);
            }
            ++issued;
        };
        // Dice: producer lane r (and r + 32) owns counter r = (view, class, kind): it adds what the consumer warps hand over
        // on a marked tile straight to the global int64 counters (integer atomics: order-independent)
        constexpr int kDiceCounters = DICE ? Op::NDICE * C * 3 : 0;
        constexpr int kDiceRounds = (kDiceCounters + 31) / 32;
        bool counts_ready = !(DICE && do_dice && a.counts_overwrite) || blockIdx.x == 0;   // CTA 0 cleared them itself
        auto await_counts = [&]() {   // all lanes; once per CTA, right before its first add to the global counters
            if (!counts_ready) {
                unsigned int z;
                do {
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(z) : "l"(&a.ws->counts_zeroed) : "memory");
                } while (z == 0u);
                counts_ready = true;
            }
        };
        if (lane == 0) {
            pending = draw();
            // (A staggered initial fill -- only 1..3 stages up front, stage s following the landing of stage s - ramp, so that no
            // CTA's first tile queues behind its neighbours' whole look-ahead -- was measured and removed: the first data lands
            // 2.3 .. 4.7 us after the start either way (it is the memory system's queue, in-flight bytes / bandwidth, not the
            // order of issue), and the thinner start costs: c2 step 92.0 -> 101.6 (1 stage) / 93.9 (2) / 91.9 us (3);
            // profiles/r38/ab_ramp.log, kbench_ramp.log.)
#pragma unroll 1
            for (int s = 0; s < STAGES; ++s) try_issue();
        }
        __syncwarp();
#pragma unroll 1
        for (int i = 0;; ++i) {
            if (!__shfl_sync(0xffffffffu, (int)(i < issued), 0)) break;
            const int stage = i % STAGES;
            tma::mbar_wait(&done[stage], (uint32_t)(i / STAGES) & 1u);  // every consumer warp is through with load i
            const int4 info = s_info[stage];
            const int tile = info.x, b = info.y;
            // Dice counts handed over on a marked tile: every consumer warp left 2 * (1 + 2*NDICE) words of 16-bit fields
            // (classes 0,2 / 1,3 of |gt==c|, then I / P of every view) in its slice of the stage's label row; lane r sums
            // counter r over the warps (before the stage is refilled) and, AFTER this iteration's copies have been issued,
            // adds it to the global counter (the atomics then never sit in front of the release of the refill's barrier arrive).
            unsigned int dsum[kDiceRounds > 0 ? kDiceRounds : 1];
            bool hand_over = false;
            if constexpr (DICE) {
                hand_over = do_dice && info.w != 0;   // written by lane 0 at issue time (a __syncwarp() ago)
                if (hand_over) {
                    const unsigned int* pkw = reinterpret_cast<const unsigned int*>(stages + (size_t)stage * Cfg::kStageBytes + Cfg::kLabelOffB);
#pragma unroll
                    for (int rr = 0; rr < kDiceRounds; ++rr) {
                        const int r = rr * 32 + lane;
                        unsigned int sum = 0u;
                        if (r < kDiceCounters) {
                            const int n = r / (C * 3), rc = r - n * C * 3, c = rc / 3, kind = rc - c * 3;
                            const int widx = kind == 1 ? 0 : (kind == 0 ? 1 + 2 * n : 2 + 2 * n);
#pragma unroll
                            for (int w = 0; w < NCW; ++w) sum += (pkw[w * 64 * PPT + 2 * widx + (c & 1)] >> (16 * (c >> 1))) & 0xffffu;
                        }
                        dsum[rr] = sum;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) {
                if constexpr (NOUT > 0) {
                    const int64_t off = (int64_t)(tile - b * tpi) * TP;
                    const uint32_t bytes = (uint32_t)info.z * (uint32_t)ES;
                    const unsigned char* st = stages + (size_t)stage * Cfg::kStageBytes;
#pragma unroll
                    for (int n = 0; n < NOUT; ++n)
                        if (a.out[n] != nullptr) {
                            if constexpr (TMAP) {
                                tma::tensor_store_3d(&maps.out[n], (int)off, 0, b, st + (size_t)n * Cfg::kTensorStride);
                            } else {
#pragma unroll
                                for (int c = 0; c < C; ++c)
                                    tma::bulk_store(static_cast<ET*>(a.out[n]) + ((int64_t)b * C + c) * HW + off,
                                                    st + Cfg::row_off(n, c), bytes);
                            }
                        }
                    tma::bulk_commit();
                    if (a.refill) {
                        // immediate: wait until THIS tile's store group has been read out of shared memory (a few hundred
                        // ns; no other stage can need the producer sooner than one tile's compute time) and hand the very
                        // same stage to the next load: every stage spends one tile's compute time less empty
                        tma::bulk_wait_read<0>();
                        try_issue();
                    } else if (i >= 1) {
                        // lagged: load i-1's store group has drained its stage once at most one group is still reading:
                        // that stage (== issued % STAGES) takes the next load or the end marker
                        tma::bulk_wait_read<1>();
                        try_issue();
                    }
                } else {
                    try_issue();
                }
            }
            if constexpr (DICE) {
                if (hand_over) {   // uniform across the warp; after this iteration's copies have been issued
                    await_counts();
#pragma unroll
                    for (int rr = 0; rr < kDiceRounds; ++rr) {
                        const int r = rr * 32 + lane;
                        if (r < kDiceCounters && dsum[rr] != 0u) {
                            const int n = r / (C * 3), rc = r - n * C * 3;
                            atomicAdd(a.counts + (int64_t)n * a.count_view_stride + (int64_t)b * C * 3 + rc, (unsigned long long)dsum[rr]);
                        }
                    }
                }
            }
            __syncwarp();
        }
        if (a.trace != nullptr && lane == 0) a.trace[kTraceSlots * blockIdx.x + 4] = globaltimer_ns();   // tiles done
        if constexpr (NOUT > 0) {
            // the CTA may exit once its stores have been read out of shared memory; their writes are complete and visible
            // when the grid is (what the next grid's griddepcontrol.wait / stream order waits for)
            if (lane == 0) tma::bulk_wait_read<0>();
        }
        if (a.trace != nullptr && lane == 0) {   // developer tracing: tiles this CTA processed, pool draws among them, its SM
            a.trace[kTraceSlots * blockIdx.x + 5] = globaltimer_ns();
            unsigned int smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            const int pool_draws = draws > my_static ? draws - my_static : 0;
            a.trace[kTraceSlots * blockIdx.x + 2] = ((unsigned long long)smid << 32) | ((unsigned long long)(unsigned)pool_draws << 16) | (unsigned)(issued & 0xffff);
        }
        __syncwarp();
    } else {
        float gs = 1.0f;
        if constexpr (Op::USES_UP) gs = upstream_scalar(a.up);
        int nbad_label = 0;
        // Dice: packed 8-bit per-class counters of this thread, [view][I,P], and |gt == c| (the same for every view).
        // They live across tiles until the producer marks a tile (s_info.w).
        unsigned int pk[DICE ? Op::NDICE : 1][2] = {};
        unsigned int pkG = 0u;
#pragma unroll 1
        for (int i = 0;; ++i) {
            const int stage = i % STAGES;
            tma::mbar_wait(&full[stage], (uint32_t)(i / STAGES) & 1u);
            const int4 info = s_info[stage];   // one 16-byte shared load: tile, image, pixel count, Dice mark
            const int tile = info.x;
            if (a.trace != nullptr && i == 0 && tid == 0) a.trace[kTraceSlots * blockIdx.x + 1] = globaltimer_ns();
            if (tile < 0) break;
            const int b = info.y;
            const bool hand_over = do_dice && info.w != 0;   // uniform across the CTA's consumers
            const int64_t off = (int64_t)(tile - b * tpi) * TP;
            const int len = info.z;
            unsigned char* st = stages + (size_t)stage * Cfg::kStageBytes;
            const int p0 = tid * PPT;
            const bool active = p0 < len;
            const unsigned int amask = CONF ? __ballot_sync(0xffffffffu, active) : 0u;  // lanes that enter the block below
            if (active) {
                FVec<PPT> gm;
#pragma unroll
                for (int v = 0; v < PPT; ++v) gm.v[v] = 1.0f;
                if constexpr (Op::GMAP) {
                    if (has_gmap) gm = *reinterpret_cast<const FVec<PPT>*>(st + Cfg::kGmapOffB + (size_t)p0 * 4);
                }
                uint2 lab[PPT];  // int64 labels as (lo, hi) words
                if constexpr (LROW) {
                    if (do_lab) {
                        if constexpr (PPT % 2 == 0) {
#pragma unroll
                            for (int v = 0; v < PPT / 2; ++v) {  // two labels per 128-bit shared load
                                const uint4 q = reinterpret_cast<const uint4*>(st + Cfg::kLabelOffB)[(p0 >> 1) + v];
                                lab[2 * v] = make_uint2(q.x, q.y);
                                lab[2 * v + 1] = make_uint2(q.z, q.w);
                            }
                        } else {
#pragma unroll
                            for (int v = 0; v < PPT; ++v) lab[v] = reinterpret_cast<const uint2*>(st + Cfg::kLabelOffB)[p0 + v];
                        }
                    }
                }
                FVec<PPT> xin[NIN][C];
#pragma unroll
                for (int n = 0; n < NIN; ++n)
#pragma unroll
                    for (int c = 0; c < C; ++c) xin[n][c] = tile_ld_row<PPT, ET>(st + Cfg::row_off(n, c), p0);
                FVec<PPT> mapv;
                float part = 0.0f, part2 = 0.0f;
#pragma unroll
                for (int gi = 0; gi < NG; ++gi) {
                    T x[NIN][C];
#pragma unroll
                    for (int n = 0; n < NIN; ++n)
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            if constexpr (LW == 2) x[n][c] = mk2(xin[n][c].v[2 * gi], xin[n][c].v[2 * gi + 1]);
                            else x[n][c] = xin[n][c].v[gi];
                        }
                    if constexpr (DICE) {
                        if (do_dice) {
                            // One-hot byte of every (view, pixel) prediction.  All NDICE * LW fast-path tests (see
                            // spec_softmax_argmax_onehot4: the class within 2^-15 of the maximum is unique and the class sum
                            // is finite => the raw arg-max is the pinned answer) are evaluated first, branch-free, and ONE
                            // rare branch redoes the group with the pinned arithmetic.  With a branch per prediction the six
                            // ~10-deep dependent chains ran one after the other (ncu r33: the consumers issue every 7th
                            // cycle, top stalls `wait` / `branch_resolving`); side by side they fill each other's latencies,
                            // and the class maxima are shared with the op's own softmax.
                            unsigned int hot[LW][Op::NDICE];
                            unsigned int hsum = 0u;   // bytes: number of predictions naming class c (<= NDICE * LW <= 8)
                            bool fin = true;
#pragma unroll
                            for (int n = 0; n < Op::NDICE; ++n) {
                                T m = x[n][0], s = x[n][0];
#pragma unroll
                                for (int c = 1; c < C; ++c) { m = vmax(m, x[n][c]); s = vadd(s, x[n][c]); }
                                const T t = vadds(m, -3.0517578125e-05f);
#pragma unroll
                                for (int j = 0; j < LW; ++j) {
                                    const float tj = vget(t, j);
                                    unsigned int h = 0u;
#pragma unroll
                                    for (int c = 0; c < C; ++c) h += (vget(x[n][c], j) >= tj) ? (1u << (8 * c)) : 0u;
                                    hot[j][n] = h;
                                    hsum += h;
                                    fin &= fabsf(vget(s, j)) <= 3.4028234664e38f;
                                }
                            }
                            // finite sums => every mask names at least its maximum, so "NDICE * LW names in total" <=> each
                            // mask names exactly one class
                            const bool all_fast = fin & (((hsum * 0x01010101u) >> 24) == (unsigned int)(Op::NDICE * LW));
                            if (!all_fast) {
#pragma unroll
                                for (int j = 0; j < LW; ++j)
#pragma unroll
                                    for (int n = 0; n < Op::NDICE; ++n) {
                                        float xs[C];
#pragma unroll
                                        for (int c = 0; c < C; ++c) xs[c] = vget(x[n][c], j);
                                        hot[j][n] = spec_softmax_argmax_onehot4<C>(xs);
                                    }
                            }
#pragma unroll
                            for (int j = 0; j < LW; ++j) {
                                const uint2 lb = lab[gi * LW + j];
                                const bool valid = (lb.y == 0u) & (lb.x < (unsigned int)C);  // 0 <= int64 label < C
                                nbad_label += !valid;
                                const unsigned int gmask = valid ? (1u << (8u * (lb.x & 3u))) : 0u;  // one-hot byte of the label
                                pkG += gmask;
#pragma unroll
                                for (int n = 0; n < Op::NDICE; ++n) {
                                    pk[n][1] += hot[j][n];
                                    pk[n][0] += hot[j][n] & gmask;
                                }
                            }
                        }
                    }
                    if constexpr (CONF) {
                        if (do_conf) {
                            // lanes holding the same (gt, pred) cell elect a leader that adds their number to the CTA's
                            // histogram: one shared-memory atomic per distinct cell and warp instead of one per pixel
#pragma unroll
                            for (int j = 0; j < LW; ++j) {
                                const uint2 lb = lab[gi * LW + j];
                                const bool valid = (lb.y == 0u) & (lb.x < (unsigned int)C);  // 0 <= int64 label < C
                                float xs[C];
#pragma unroll
                                for (int c = 0; c < C; ++c) xs[c] = vget(x[0][c], j);
                                const int key = valid ? (int)lb.x * C + raw_argmax<C>(xs) : -1;
                                const unsigned int peers = __match_any_sync(amask, key);
                                if (key >= 0 && lane == __ffs((int)peers) - 1) atomicAdd(&s_conf[key], (unsigned int)__popc(peers));
                            }
                        }
                    }
                    T gv;
                    if constexpr (LW == 2) gv = mk2(gs * gm.v[2 * gi], gs * gm.v[2 * gi + 1]);
                    else gv = gs * gm.v[gi];
                    T mv;
                    if constexpr (LAB) {
                        int cls[LW];
                        float cw[LW];
#pragma unroll
                        for (int j = 0; j < LW; ++j) {
                            const uint2 lb = lab[gi * LW + j];
                            const bool valid = (lb.y == 0u) & (lb.x < (unsigned int)C);
                            const bool ign = (lb.x == (unsigned int)((unsigned long long)a.ignore_index & 0xffffffffull)) &
                                             (lb.y == (unsigned int)((unsigned long long)a.ignore_index >> 32));
                            if constexpr (!DICE) nbad_label += (!valid) & (!ign);  // (the Dice block counts every label outside [0,C))
                            const bool use = valid & !ign;
                            cls[j] = use ? (int)lb.x : -1;
                            cw[j] = use ? (a.class_w != nullptr ? __ldg(a.class_w + lb.x) : 1.0f) : 0.0f;
                        }
                        mv = Op::template apply_lab<C, T>(x, C, gv, cls, cw, bad);
                    } else if constexpr (SUM2) {
                        T mv2;
                        mv = Op::template apply<C, T>(x, C, gv, a.eps, bad, mv2);
                        part2 += vhsum(mv2);
                    } else {
                        mv = Op::template apply<C, T>(x, C, gv, a.eps, bad);
                    }
                    if constexpr (LW == 2) { mapv.v[2 * gi] = vget(mv, 0); mapv.v[2 * gi + 1] = vget(mv, 1); }
                    else mapv.v[gi] = vget(mv, 0);
                    part += vhsum(mv);
#pragma unroll
                    for (int n = 0; n < NOUT; ++n)
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            if constexpr (LW == 2) { xin[n][c].v[2 * gi] = vget(x[n][c], 0); xin[n][c].v[2 * gi + 1] = vget(x[n][c], 1); }
                            else xin[n][c].v[gi] = vget(x[n][c], 0);
                        }
                }
                if constexpr (Op::HAS_MAP) {
                    acc_fx.add(to_fixed(part, nonfinite));
                    if (a.map != nullptr) st_stream<PPT>(a.map + (int64_t)b * HW + off + p0, mapv);
                }
                if constexpr (SUM2) acc_fx2.add(to_fixed(part2, nonfinite2));
#pragma unroll
                for (int n = 0; n < NOUT; ++n)
                    if (a.out[n] != nullptr) {
#pragma unroll
                        for (int c = 0; c < C; ++c) tile_st_row<PPT, ET>(st + Cfg::row_off(n, c), p0, xin[n][c]);
                    }
            }
            if constexpr (NOUT > 0) tma::fence_proxy_async_smem();
            __syncwarp();
            if constexpr (DICE) {
                if (hand_over) {
                    // widen every packed word into two words of 16-bit fields (classes 0,2 and 1,3; 32 lanes * 255 < 2^16),
                    // reduce them across the warp (REDUX) and leave them in the warp's slice of the label row (its labels
                    // have all been read); the producer warp adds the warps' numbers once `done` has completed
                    constexpr int NW = 1 + 2 * Op::NDICE;
                    unsigned int mine = 0u;
#pragma unroll
                    for (int j = 0; j < NW; ++j) {
                        const unsigned int w = j == 0 ? pkG : pk[(j - 1) >> 1][(j - 1) & 1];
                        const unsigned int lo = __reduce_add_sync(0xffffffffu, w & 0x00ff00ffu);
                        const unsigned int hi = __reduce_add_sync(0xffffffffu, (w >> 8) & 0x00ff00ffu);
                        if (lane == 2 * j) mine = lo;
                        if (lane == 2 * j + 1) mine = hi;
                    }
                    static_assert(2 * NW <= 32, "one lane per reduced word");
                    if (lane < 2 * NW) reinterpret_cast<unsigned int*>(st + Cfg::kLabelOffB)[(tid >> 5) * 64 * PPT + lane] = mine;
                    pkG = 0u;
#pragma unroll
                    for (int n = 0; n < Op::NDICE; ++n) pk[n][0] = pk[n][1] = 0u;
                    __syncwarp();
                }
            }
            if (lane == 0) tma::mbar_arrive(&done[stage]);
        }
        if constexpr (LROW) {
            if (do_lab) {
                nbad_label = __reduce_add_sync(0xffffffffu, nbad_label);
                if (lane == 0 && nbad_label != 0 && a.flags != nullptr) atomicAdd(&a.flags[DCT_FLAG_LABEL], nbad_label);
            }
        }
        // this CTA's share of the loss sums goes to the workspace accumulators while the producer warp drains its stores
        if constexpr (SUM2)
            tile_grid_add<true>(acc_fx, nonfinite, a.ws, Op::HAS_MAP && a.sum != nullptr, CTHREADS, acc_fx2, nonfinite2,
                                a.sum2 != nullptr);
        else
            tile_grid_add(acc_fx, nonfinite, a.ws, Op::HAS_MAP && a.sum != nullptr, CTHREADS);
    }
    // this CTA's tiles are done: the next kernel in the stream may be scheduled onto the SMs that drain first and run
    // its prologue; its pdl_wait() still holds it until this whole grid (epilogue below included) has completed
    pdl_launch_dependents();
    if constexpr (CONF) {
        __syncthreads();  // every consumer warp's shared-memory atomics are done
        if (do_conf) {
            for (int i = tid; i < CT * CT; i += (int)blockDim.x) {
                const unsigned int v = s_conf[i];
                if (v != 0u) atomicAdd(a.conf + i, (unsigned long long)v);
            }
        }
    }
    if constexpr (Op::CHECKS_SIMPLEX) {
        if (a.flags != nullptr && __syncthreads_or(bad)) {
            if (bad) atomicAdd(&a.flags[DCT_FLAG_SIMPLEX], 1);
        }
    }
    __syncthreads();   // the producer's loop and thread 0's accumulator adds come before the ticket
    unsigned long long* const trace_ticket = a.trace != nullptr ? a.trace + kTraceSlots * blockIdx.x + 6 : nullptr;
    tile_grid_finish<PUB, SUM2>(a.ws, Op::HAS_MAP ? a.sum : nullptr, gridDim.x, trace_ticket, &a.pub, a.pub_early,
                                SUM2 ? a.sum2 : nullptr);
    if (a.trace != nullptr && tid == 0) a.trace[kTraceSlots * blockIdx.x + 3] = globaltimer_ns();
}

// Host side: does this problem fit the tile pipeline?  (16-byte aligned rows and segments)
template <class Op, class ET = float>
inline bool tile_eligible(const TileArgs& a, int64_t B) {
    if ((a.HW % (16 / (int)sizeof(ET))) != 0 || B * ((a.HW + 255) / 256) > 0x7fffffffLL) return false;
    for (int n = 0; n < Op::NIN; ++n)
        if (!aligned(a.in[n], 16)) return false;
    for (int n = 0; n < Op::NOUT; ++n)
        if (a.out[n] != nullptr && !aligned(a.out[n], 16)) return false;
    if (a.map != nullptr && !aligned(a.map, 16)) return false;
    if (a.up.gmap != nullptr && !aligned(a.up.gmap, 16)) return false;
    if (a.labels != nullptr && !aligned(a.labels, 16)) return false;
    return true;
}

template <class Op, int CT, class ET = float, bool PUB = false>
int tile_launch_ct(TileArgs a, int64_t B, cudaStream_t stream) {
    constexpr int ROWS = Op::NIN * CT;
    static_assert(ROWS <= kTileMaxRows, "tile pipeline instantiations are for NIN*C <= 80");
    // Launch shapes measured on B200 (tools/kbench_tile.cu; profiles/r01/kbench_c19_sweep.md).  What decides: the
    // consumer warps are latency-bound (ncu: 21% issue-slot use with one warp per scheduler), so the shape must put
    // >= 6 consumer warps on an SM while keeping >= 3 stages for ops with outputs (2 stages stall on the store drain);
    // two small CTAs per SM beat one large CTA (two independent producers).
    //   rows <= 4        4 pixels/thread, 8 consumer warps, 2 CTAs/SM, row copies (Dice counting, spleen K = C = 2)
    //   5 <= rows <= 16  ACDC: K*C = 8..16, the KL family: tiles of 256 pixels (2 pixels/thread, 4 consumer warps), 3 CTAs/SM,
    //                    one tensor-map box per tensor instead of C row copies: 3 independent producers per SM, 7 copies per
    //                    tile instead of 25 at c2 (round 1: 512-pixel tiles, 8 warps, 2 CTAs/SM, row copies;
    //                    profiles/r35/kbench_small.log: c2 JSD+Dice 40.9 -> 39.4 us, KL 25.4 -> 24.8, c1 9.4 -> 8.7)
    //   rows <= 24       one C = 19 tensor (cross-entropy): 4 warps, 2 CTAs/SM, 5 stages        (99% of the copy peak)
    //   rows <= 40       Cityscapes C = 19 with 2 tensors: 3 warps, 2 CTAs/SM, 3 stages           (JSD 4449 -> 5930 GB/s)
    //                    read-only ops: 8 warps, 1 CTA/SM, 2 stages
    //   rows <= 60       K = 3, C = 19: one pixel/thread (a pixel pair takes 255 registers), 5 warps, 2 CTAs/SM, 3 stages
    //                    (profiles/r08/kbench_wide_reg.log: 5244 GB/s against 4641 for the pixel-pair shape)
    //   rows <= 80       K = 4, C = 19: one pixel/thread, 7 warps, 1 CTA/SM, 3 stages of 68 KB (the most that fits)
    //                    (profiles/r09/kbench_wide_more.log: 4245 GB/s; 6 warps 3750, 2 x 3 warps 3744, 5 warps x 4 stages 3205)
    // (A shared-memory-resident JSD body for the > 40-row stages measured equal or slower than the register-resident one at
    // every shape and was removed: profiles/r08/kbench_wide_stream.log.)
    constexpr bool SMALL = ROWS > 4 && ROWS <= 16;
    constexpr int PPT = ROWS <= 4 ? 4 : (ROWS <= 40 ? 2 : 1);
    constexpr int NCW = ROWS <= 4 ? 8 : (ROWS <= 24 ? 4 : (ROWS <= 40 ? (Op::NOUT == 0 ? 8 : 3) : (ROWS <= 60 ? 5 : 7)));
    constexpr int MINB = SMALL ? 3 : (ROWS <= 24 ? 2 : (ROWS <= 40 ? (Op::NOUT == 0 ? 1 : 2) : (ROWS <= 60 ? 2 : 1)));
    constexpr int TPX = NCW * 32 * PPT;
    // stages whose tile is one box (<= 256 pixels): tensor-map TMA, one copy per tensor instead of one per row -- the wide
    // C = 19 stages and the small ACDC-sized ones
    constexpr bool TMAP = (CT > 4 || SMALL) && TPX <= 256;
    // bf16 tensors: same shapes (the register budget follows the number of rows, not their width); the 2-byte rows
    // simply buy more stages
    constexpr int STAGES = tile_stages<tile_stage_bytes<Op, CT, TPX, ET, TMAP>(), MINB>();
    using Cfg = TileCfg<Op, CT, PPT, NCW * 32, STAGES, ET, TMAP>;
    auto kern = tile_kernel<Op, CT, PPT, NCW, STAGES, MINB, ET, PUB, TMAP>;
    TileMaps<TMAP> maps{};
    if constexpr (TMAP) {
        // descriptors of this launch's tensors (host-side encode, ~1 us each; nothing is launched if the driver refuses)
        for (int n = 0; n < Op::NIN; ++n)
            if (!make_tmap_bchw(&maps.in[n], a.in[n], (int)sizeof(ET), a.HW, CT, B, Cfg::TP)) return DCT_ERR_UNSUPPORTED;
        for (int n = 0; n < Op::NOUT; ++n)
            if (a.out[n] != nullptr && !make_tmap_bchw(&maps.out[n], a.out[n], (int)sizeof(ET), a.HW, CT, B, Cfg::TP))
                return DCT_ERR_UNSUPPORTED;
    }
    static bool configured[64] = {};  // per instantiation and device (the attribute is per device function)
    int devid = 0;
    cudaGetDevice(&devid);
    if (devid < 0 || devid >= 64 || !configured[devid]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes);
        if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
        if (devid >= 0 && devid < 64) configured[devid] = true;
    }
    tile_set_geometry(a, B, Cfg::TP);
    // L2 prefetch of 2 tiles per CTA (measured, profiles/r30/ab_prefetch.log: c2 step 102.3 -> 101.9 us, c3 52.6 -> 51.8, c1 11.3
    // -> 10.5).  Deeper (3..4) makes the KL launches faster when timed alone (c2 kl_logit 19.0 -> 18.5 us) but not the chained
    // step (91.6 -> 91.6 / 91.9 us) and costs the JSD launch at c3 (12.9 -> 13.3 us): profiles/r39/ab_env.log, r42/ab_refill.log
    a.prefetch = 2;
    // Measured (profiles/r34/ab_refill.log): immediate refill pays where the store group is a fraction of the stage and the
    // stages are few -- the C = 19 KL kernels (2-3 tensors in, 1 out, 3 stages): c4 kl_adv 324 -> 305 us, kl_logit 301 -> 296;
    // it costs where the store drains the whole stage (JSD: c4 407 -> 418 us, c2 37.5 -> 37.9: the producer lane sits in
    // the read wait); on the short c2 / c3 KL launches it is neutral within 0.3 us either way (profiles/r42/ab_refill.log)
    a.refill = (TMAP && Op::NOUT < Op::NIN) ? 1 : 0;
    int grid = kSMs * MINB;
    if (grid > a.num_tiles) grid = a.num_tiles;
    if (a.trace == nullptr) a.trace = trace_next(grid);
    cudaError_t e = launch_pdl(kern, dim3(grid), dim3(NCW * 32 + 32), Cfg::kSmemBytes, stream, a, maps);
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return check_launch();
}

}  // namespace dct
