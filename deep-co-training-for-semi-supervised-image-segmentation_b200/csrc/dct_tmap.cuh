// dct_tmap.cuh -- tensor-map TMA (cp.async.bulk.tensor, SASS UTMALDG / UTMASTG) for the wide stages of the tile
// pipeline: ONE copy moves the C class rows of a tile of one [B,C,HW] tensor (box [TP, C, 1]) instead of C row copies.
//
// The 1-D bulk copies of dct_tma.cuh cost the producer lane one instruction per (tensor, class) row each way; at
// Cityscapes' C = 19 that is 76 + 76 issues per tile for K = 4 views, and that issue loop was measured to be the
// sensitive spot of those shapes (dct_common.cuh: R2UR 7 -> 100 cost 19 %).  With a tensor map the producer issues K + K.
//
// Host side: CUtensorMap descriptors are encoded per launch from the tensors' pointers (cuTensorMapEncodeTiled through
// cudaGetDriverEntryPoint: no link against libcuda) and travel in the kernel parameters (__grid_constant__).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dct_tma.cuh"

namespace dct {
namespace tma {

// global (tensor map, coordinates {x = pixel in image, y = class, z = image}) -> shared; completion as transaction bytes
// of the WHOLE box on `bar` (elements outside the tensor are written as zeros and count)
__device__ __forceinline__ void tensor_load_3d(void* smem_dst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
        : "memory");
}
// shared -> global (elements outside the tensor are not written), tracked by the thread's bulk async-group
__device__ __forceinline__ void tensor_store_3d(const CUtensorMap* map, int x, int y, int z, const void* smem_src) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(x), "r"(y), "r"(z), "r"(smem_u32(smem_src))
                 : "memory");
}
// hint: pull the box at {x, y, z} into L2 (see bulk_prefetch_l2)
__device__ __forceinline__ void tensor_prefetch_3d(const CUtensorMap* map, int x, int y, int z) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(x), "r"(y), "r"(z)
                 : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

}  // namespace tma

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult st = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &st) != cudaSuccess ||
            st != cudaDriverEntryPointSuccess)
            p = nullptr;
        (void)cudaGetLastError();
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// Tensor map of one contiguous [B, C, HW] tensor of `es`-byte elements (4: float32, 2: bfloat16) with box [box_w, C, 1].
// false: the driver entry point is missing or refused the shape (tile_launch_ct then launches nothing: DCT_ERR_UNSUPPORTED).
// Descriptors are pure functions of (pointer, element size, shape, box): a training loop presents the same few tensors'
// addresses step after step (caching allocator), so the last encodings are kept per host thread and a launch outside a
// CUDA graph pays a 128-byte copy instead of a driver call per tensor.
inline bool make_tmap_bchw(CUtensorMap* m, const void* base, int es, int64_t HW, int C, int64_t B, int box_w) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (enc == nullptr || box_w < 1 || box_w > 256 || C < 1 || C > 256) return false;
    struct Entry { const void* base; int64_t HW, B; int es, C, box_w; bool used; CUtensorMap map; };
    constexpr int kEntries = 32;
    thread_local Entry cache[kEntries] = {};
    thread_local int next = 0;
    for (int i = 0; i < kEntries; ++i) {
        const Entry& e = cache[i];
        if (e.used && e.base == base && e.HW == HW && e.B == B && e.es == es && e.C == C && e.box_w == box_w) {
            *m = e.map;
            return true;
        }
    }
    const cuuint64_t dims[3] = {(cuuint64_t)HW, (cuuint64_t)C, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)HW * es, (cuuint64_t)HW * C * es};   // bytes; multiples of 16 (checked by the caller)
    const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)C, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUresult r = enc(m, es == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3,
                           const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
    Entry& e = cache[next];
    next = (next + 1) % kEntries;
    e.base = base; e.HW = HW; e.B = B; e.es = es; e.C = C; e.box_w = box_w; e.map = *m; e.used = true;
    return true;
}

}  // namespace dct
