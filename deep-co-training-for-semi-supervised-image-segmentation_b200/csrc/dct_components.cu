// dct_components.cu -- connected-component labelling of a class map on the device, and the largest component per class
// (evaluation path: the post-processing in front of the Dice / surface distances; getLargestCC of the UA-MT / DTC /
// MC-Net test scripts, nnU-Net's "remove all but the largest component").
//
// Definition: per class c on a grid (one H x W slice, or the B x H x W batch as one volume), two pixels are in one
// component when both hold c and are joined through neighbours holding c; the neighbourhood is scipy's
// generate_binary_structure(rank, connectivity) (offsets in {-1,0,1}^rank with at most `connectivity` non-zero entries).
// Every class, 0 included, is labelled.  A component's label is the linear index, in the batch tensor, of its first
// pixel in raster order (its smallest index).  Values outside [0,C) belong to no component (label -1).
//
// Union-find with links from a larger root to a smaller one (atomicMin), so a component's final root is its smallest
// index whatever the scheduling, and every output is a bit-reproducible integer:
//   cc_local_kernel     one CTA per tile (TZ x TY x TX <= 1024 pixels): packs the int64 classes into a byte per pixel
//                       (0xFF out of range -> flags), union-find in shared memory over the tile's own neighbour pairs,
//                       writes each pixel's global parent; zeroes the per-pixel sizes and per-(row, class) statistics.
//   cc_merge_kernel     one CTA per tile: every pixel on a low face (or the last column / row, for the diagonals that
//                       point up-right or down) unions with its neighbours in other tiles, global atomicMin linking
//                       with path halving.
//   cc_compress_kernel  every pixel finds its root: label, size at the root (integer atomics, one per distinct root of a
//                       warp), roots counted per (row, class); parents are shortened towards the roots.
//   cc_winner_kernel    per root: 64-bit atomicMax of size << 32 | (INT32_MAX - root) into its (row, class): the largest
//                       component, ties to the smallest root, independent of order.
//   cc_finish_kernel    statistics (count, largest size) and the largest-component map (each pixel follows its
//                       parents to the root: a few steps at most after the compress pass).
// Launches: 5, or 3 when only labels are asked for.  No host synchronisation, no allocation, no float atomics.
#include <algorithm>
#include <climits>

#include "dct_common.cuh"

namespace dct {

constexpr int kCcTile = 1024;          // pixels per tile (shared memory: 5 B each)
constexpr int kCcThreads = 256;
constexpr unsigned char kCcNone = 0xFF;   // packed class byte of a value outside [0,C)

struct CcGeom {
    int C, volume, nofs;                 // nofs: backward neighbour offsets in use
    int64_t B, H, W, N;
    int TZ, TY, TX;                      // tile extents (powers of two)
    int ly_shift, lz_shift;              // log2(TX), log2(TX * TY)
    unsigned tiles_x, tiles_y, tiles;    // tiles <= N <= 2^31 - 1
};

// the backward half of the 26-neighbourhood (neighbours earlier in raster order), ordered so that a prefix is each
// connectivity's: 2d 1 -> 2, 2d 2 -> 4 (only dz = 0 used); 3d 1 -> 3, 2 -> 9, 3 -> 13
// each offset packed as (dz + 1) * 9 + (dy + 1) * 3 + (dx + 1)
__constant__ unsigned char kOfs2d[4] = {12, 10, 9, 11};
__constant__ unsigned char kOfs3d[13] = {12, 10, 4, 9, 11, 1, 7, 3, 5, 0, 2, 6, 8};
struct CcOfs { int dz, dy, dx; };
__device__ __forceinline__ CcOfs cc_ofs(const CcGeom& g, int k) {
    const int v = g.volume ? kOfs3d[k] : kOfs2d[k];
    return {v / 9 - 1, (v / 3) % 3 - 1, v % 3 - 1};
}

struct CcLayout {
    size_t cls, parent, size, count, best, total;
};
inline size_t cc_align256(size_t v) { return (v + 255) & ~(size_t)255; }
inline CcLayout cc_layout(int C, int64_t B, int64_t H, int64_t W, int volume) {
    const size_t N = (size_t)B * H * W, nrc = (volume ? 1 : (size_t)B) * C;
    CcLayout L;
    L.cls = 0;                                      // uint8 [N] packed classes
    L.parent = cc_align256(L.cls + N);              // int32 [N]
    L.size = cc_align256(L.parent + N * 4);         // uint32 [N] component size at its root
    L.count = cc_align256(L.size + N * 4);          // uint64 [rows][C] roots
    L.best = cc_align256(L.count + nrc * 8);        // uint64 [rows][C] size << 32 | (INT32_MAX - root)
    L.total = cc_align256(L.best + nrc * 8);
    return L;
}

inline int64_t pow2_at_least(int64_t v, int64_t cap) {
    int64_t p = 1;
    while (p < v && p < cap) p <<= 1;
    return p;
}

// tiles of at most kCcTile pixels: 32 x 32 per slice, 4 x 16 x 16 bricks in a volume, grown along the long axes of a
// thin grid (N x 1 x 1 or 1 x 1 x N) so that tiles stay full
inline CcGeom cc_geom(int C, int64_t B, int64_t H, int64_t W, int volume, int connectivity) {
    CcGeom g{};
    g.C = C; g.volume = volume; g.B = B; g.H = H; g.W = W; g.N = B * H * W;
    static const int nofs[2][4] = {{0, 2, 4, 0}, {0, 3, 9, 13}};
    g.nofs = nofs[volume ? 1 : 0][connectivity];
    int64_t tx = pow2_at_least(W, volume ? 16 : 32);
    int64_t ty = pow2_at_least(H, kCcTile / tx / (volume ? 4 : 1));
    const int64_t tz = pow2_at_least(B, kCcTile / (tx * ty));
    ty = pow2_at_least(H, kCcTile / (tx * tz));
    tx = pow2_at_least(W, kCcTile / (ty * tz));
    g.TZ = (int)tz; g.TY = (int)ty; g.TX = (int)tx;
    g.ly_shift = __builtin_ctzll(tx); g.lz_shift = __builtin_ctzll(tx * ty);
    g.tiles_x = (unsigned)((W + tx - 1) / tx);
    g.tiles_y = (unsigned)((H + ty - 1) / ty);
    g.tiles = g.tiles_x * g.tiles_y * (unsigned)((B + tz - 1) / tz);
    return g;
}

__device__ __forceinline__ void cc_tile_origin(const CcGeom& g, unsigned tile, int64_t& z0, int64_t& y0, int64_t& x0) {
    const unsigned per_z = g.tiles_x * g.tiles_y, tzi = tile / per_z, r = tile - tzi * per_z, tyi = r / g.tiles_x;
    z0 = (int64_t)tzi * g.TZ; y0 = (int64_t)tyi * g.TY; x0 = (int64_t)(r - tyi * g.tiles_x) * g.TX;
}

__device__ __forceinline__ void cc_local_xyz(const CcGeom& g, int i, int& lx, int& ly, int& lz) {
    lx = i & (g.TX - 1); ly = (i >> g.ly_shift) & (g.TY - 1); lz = i >> g.lz_shift;
}

// root of x with path halving.  Every write stores an ancestor of x, smaller than x, so concurrent unions stay correct:
// a link overwritten here is one whose atomicMin saw a non-root and is retried by its union.
__device__ __forceinline__ int cc_find(volatile int* par, int x) {
    while (true) {
        const int p = par[x];
        if (p == x) return x;
        const int gp = par[p];
        if (gp == p) return p;
        par[x] = gp;
        x = gp;
    }
}

template <typename P>
__device__ __forceinline__ void cc_union(P* par, int a, int b) {
    while (true) {
        a = cc_find(par, a);
        b = cc_find(par, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(const_cast<int*>(par + b), a);   // link the larger root to the smaller
        if (old == b) return;
        b = old;   // b was linked meanwhile: join its new parent with a
    }
}

__global__ void __launch_bounds__(kCcThreads) cc_local_kernel(const int64_t* __restrict__ map, const CcGeom g,
                                                             unsigned char* __restrict__ cls, int* __restrict__ parent,
                                                             unsigned* __restrict__ size, unsigned long long* stats,
                                                             int64_t nstats, int32_t* flags) {
    __shared__ int s_par[kCcTile];
    __shared__ unsigned char s_cls[kCcTile];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nstats; i += (int64_t)gridDim.x * blockDim.x)
        stats[i] = 0ull;
    const int TX = g.TX, TY = g.TY, n = g.TZ * TY * TX;
    const int64_t HW = g.H * g.W;
    int bad = 0;
    for (unsigned tile = blockIdx.x; tile < g.tiles; tile += gridDim.x) {
        int64_t z0, y0, x0;
        cc_tile_origin(g, tile, z0, y0, x0);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            int lx, ly, lz;
            cc_local_xyz(g, i, lx, ly, lz);
            const int64_t z = z0 + lz, y = y0 + ly, x = x0 + lx;
            unsigned char c = kCcNone;
            if (z < g.B && y < g.H && x < g.W) {
                const int64_t p = z * HW + y * g.W + x;
                const long long v = map[p];
                if (v >= 0 && v < g.C) c = (unsigned char)v;
                else ++bad;
                cls[p] = c;
                size[p] = 0u;
            }
            s_cls[i] = c;
            s_par[i] = i;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const unsigned char c = s_cls[i];
            if (c == kCcNone) continue;
            int lx, ly, lz;
            cc_local_xyz(g, i, lx, ly, lz);
            for (int k = 0; k < g.nofs; ++k) {
                const CcOfs o = cc_ofs(g, k);
                const int nz = lz + o.dz, ny = ly + o.dy, nx = lx + o.dx;
                if (nz < 0 || ny < 0 || nx < 0 || nx >= TX || ny >= TY) continue;   // another tile: cc_merge_kernel
                const int j = (nz * TY + ny) * TX + nx;
                if (s_cls[j] == c) cc_union<volatile int>(s_par, i, j);
            }
        }
        __syncthreads();
        // local raster order is global raster order within a tile, so the local root is the smallest global index
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            if (s_cls[i] == kCcNone) continue;
            const int r = cc_find(s_par, i);
            int lx, ly, lz;
            cc_local_xyz(g, i, lx, ly, lz);
            int rx, ry, rz;
            cc_local_xyz(g, r, rx, ry, rz);
            parent[(z0 + lz) * HW + (y0 + ly) * g.W + x0 + lx] = (int)((z0 + rz) * HW + (y0 + ry) * g.W + x0 + rx);
        }
        __syncthreads();   // shared arrays are reused by the next tile
    }
    if (flags != nullptr) {
        bad = __reduce_add_sync(0xffffffffu, bad);
        if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&flags[DCT_FLAG_PRED], bad);
    }
}

// pixels whose backward neighbours can lie in another tile: the first slice, row or column of the tile, its last column
// (offsets with dx = +1) and its last row (dy = +1, volumes); each unions with every such neighbour of its class
__global__ void __launch_bounds__(kCcThreads) cc_merge_kernel(const unsigned char* __restrict__ cls, const CcGeom g,
                                                             int* parent) {
    const int TX = g.TX, TY = g.TY, n = g.TZ * TY * TX;
    const int64_t HW = g.H * g.W;
    int64_t z0, y0, x0;   // one CTA per tile
    cc_tile_origin(g, blockIdx.x, z0, y0, x0);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        int lx, ly, lz;
        cc_local_xyz(g, i, lx, ly, lz);
        if (lx != 0 && ly != 0 && lz != 0 && lx != TX - 1 && ly != TY - 1) continue;
        const int64_t z = z0 + lz, y = y0 + ly, x = x0 + lx;
        if (z >= g.B || y >= g.H || x >= g.W) continue;
        const int64_t p = z * HW + y * g.W + x;
        const unsigned char c = cls[p];
        if (c == kCcNone) continue;
        for (int k = 0; k < g.nofs; ++k) {
            const CcOfs o = cc_ofs(g, k);
            const int nz = lz + o.dz, ny = ly + o.dy, nx = lx + o.dx;
            if (nz >= 0 && ny >= 0 && nx >= 0 && nx < TX && ny < TY) continue;   // same tile: cc_local_kernel
            if (z + o.dz < 0 || y + o.dy < 0 || y + o.dy >= g.H || x + o.dx < 0 || x + o.dx >= g.W) continue;
            const int64_t q = p + o.dz * HW + o.dy * g.W + o.dx;
            if (cls[q] == c) cc_union<volatile int>(parent, (int)p, (int)q);
        }
    }
}

__device__ __forceinline__ int64_t cc_row(const CcGeom& g, int64_t p) { return g.volume ? 0 : p / (g.H * g.W); }

__global__ void __launch_bounds__(kCcThreads) cc_compress_kernel(const unsigned char* __restrict__ cls, const CcGeom g,
                                                                int* parent, unsigned* size,
                                                                unsigned long long* count, int32_t* labels) {
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    // whole warps iterate together (the warp-aggregated atomics vote)
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < g.N; base += nthr) {
        const int64_t p = base + threadIdx.x;
        const unsigned char c = p < g.N ? cls[p] : kCcNone;
        int r = -1;
        if (c != kCcNone) {
            // no union runs now: halving only shortens paths.  The root stored here can still be overwritten by another
            // thread's halving step through p (with an ancestor of p), so later passes follow parents to the root.
            const int up = reinterpret_cast<volatile int*>(parent)[p];
            r = up == (int)p ? up : cc_find(parent, up);
            if (r != up) parent[p] = r;
            if (labels != nullptr) labels[p] = r;
        } else if (p < g.N && labels != nullptr) {
            labels[p] = -1;
        }
        if (size != nullptr) {
            const unsigned peers = __match_any_sync(0xffffffffu, r);
            if (r >= 0 && lane == __ffs(peers) - 1) atomicAdd(&size[r], (unsigned)__popc(peers));
            const long long tag = r == (int)p && r >= 0 ? cc_row(g, p) * g.C + c : -1;
            const unsigned same = __match_any_sync(0xffffffffu, tag);
            if (tag >= 0 && lane == __ffs(same) - 1) atomicAdd(&count[tag], (unsigned long long)__popc(same));
        }
    }
}

__device__ __forceinline__ unsigned long long cc_key(unsigned sz, int root) {
    return ((unsigned long long)sz << 32) | (unsigned)(INT_MAX - root);
}

__global__ void __launch_bounds__(kCcThreads) cc_winner_kernel(const unsigned char* __restrict__ cls, const CcGeom g,
                                                              const int* __restrict__ parent,
                                                              const unsigned* __restrict__ size,
                                                              unsigned long long* best) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < g.N; p += (int64_t)gridDim.x * blockDim.x) {
        const unsigned char c = cls[p];
        if (c == kCcNone || parent[p] != (int)p) continue;
        atomicMax(&best[cc_row(g, p) * g.C + c], cc_key(size[p], (int)p));
    }
}

__global__ void __launch_bounds__(kCcThreads) cc_finish_kernel(const int64_t* __restrict__ map,
                                                              const unsigned char* __restrict__ cls, const CcGeom g,
                                                              const int* __restrict__ parent,
                                                              const unsigned long long* __restrict__ count,
                                                              const unsigned long long* __restrict__ best,
                                                              int64_t nrc, int64_t* __restrict__ stats,
                                                              int64_t* __restrict__ largest) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
    if (stats != nullptr) {
        for (int64_t j = tid; j < nrc; j += nthr) {
            stats[2 * j] = (int64_t)count[j];
            stats[2 * j + 1] = (int64_t)(best[j] >> 32);
        }
    }
    if (largest == nullptr) return;
    for (int64_t p = tid; p < g.N; p += nthr) {
        const unsigned char c = cls[p];
        int64_t v;
        if (c == kCcNone) {
            v = map[p];   // copied unchanged
        } else if (c == 0) {
            v = 0;        // class 0 is never filtered
        } else {
            const int winner = INT_MAX - (int)(unsigned)(best[cc_row(g, p) * g.C + c] & 0xFFFFFFFFull);
            int r = parent[p];
            for (int up = parent[r]; up != r; up = parent[r]) r = up;   // at most a few steps after cc_compress_kernel
            v = r == winner ? (int64_t)c : 0;
        }
        largest[p] = v;
    }
}

}  // namespace dct

using namespace dct;

static bool cc_supported(int C, int64_t B, int64_t H, int64_t W) {
    if (C > DCT_MAX_CLASSES) return false;
    if (B > INT_MAX || H > INT_MAX || W > INT_MAX) return false;
    return B * H <= INT_MAX && B * H * W <= INT_MAX;   // labels and parents are int32 indices
}

extern "C" size_t dct_components_scratch_bytes(int C, int64_t B, int64_t H, int64_t W, int volume) {
    if (C < 1 || B < 1 || H < 1 || W < 1 || !cc_supported(C, B, H, W)) return 0;
    return cc_layout(C, B, H, W, volume).total;
}

extern "C" int dct_components_i64(const int64_t* map, int C, int64_t B, int64_t H, int64_t W, int volume,
                                  int connectivity, int32_t* labels, int64_t* stats, int64_t* largest_map,
                                  int32_t* flags, void* scratch, void* stream) {
    if (map == nullptr || scratch == nullptr || (labels == nullptr && stats == nullptr && largest_map == nullptr))
        return DCT_ERR_BAD_ARG;
    if (C < 1 || B < 1 || H < 1 || W < 1) return DCT_ERR_BAD_ARG;
    if (!cc_supported(C, B, H, W)) return DCT_ERR_UNSUPPORTED;
    volume = volume ? 1 : 0;
    if (connectivity < 1 || connectivity > (volume ? 3 : 2)) return DCT_ERR_BAD_ARG;
    const int64_t N = B * H * W;
    if (largest_map != nullptr) {
        const char *a = reinterpret_cast<const char*>(map), *b = reinterpret_cast<const char*>(largest_map);
        if (a < b + N * 8 && b < a + N * 8) return DCT_ERR_BAD_ARG;   // must not overlap the input
    }
    if (!aligned(map, 8) || !aligned(labels, 4) || !aligned(stats, 8) || !aligned(largest_map, 8) ||
        !aligned(flags, 4) || !aligned(scratch, 256))
        return DCT_ERR_MISALIGNED;

    const CcGeom g = cc_geom(C, B, H, W, volume, connectivity);
    const CcLayout L = cc_layout(C, B, H, W, volume);
    char* base = static_cast<char*>(scratch);
    unsigned char* cls = reinterpret_cast<unsigned char*>(base + L.cls);
    int* parent = reinterpret_cast<int*>(base + L.parent);
    unsigned* size = reinterpret_cast<unsigned*>(base + L.size);
    unsigned long long* count = reinterpret_cast<unsigned long long*>(base + L.count);
    unsigned long long* best = reinterpret_cast<unsigned long long*>(base + L.best);
    const int64_t nrc = (volume ? 1 : B) * C;
    const bool need_stats = stats != nullptr || largest_map != nullptr;
    cudaStream_t s = static_cast<cudaStream_t>(stream);

    const unsigned tile_blocks = (unsigned)std::min<int64_t>(g.tiles, (int64_t)kSMs * 64);
    const unsigned pix_blocks = (unsigned)std::min<int64_t>((N + kCcThreads - 1) / kCcThreads, (int64_t)kSMs * 32);
    // count and best are adjacent: one zeroing loop in the local pass
    cc_local_kernel<<<tile_blocks, kCcThreads, 0, s>>>(map, g, cls, parent, size, count,
                                                       (int64_t)((L.total - L.count) / 8), flags);
    cc_merge_kernel<<<g.tiles, kCcThreads, 0, s>>>(cls, g, parent);
    cc_compress_kernel<<<pix_blocks, kCcThreads, 0, s>>>(cls, g, parent, need_stats ? size : nullptr, count, labels);
    if (need_stats) {
        cc_winner_kernel<<<pix_blocks, kCcThreads, 0, s>>>(cls, g, parent, size, best);
        cc_finish_kernel<<<pix_blocks, kCcThreads, 0, s>>>(map, cls, g, parent, count, best, nrc, stats, largest_map);
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return DCT_OK;
}
