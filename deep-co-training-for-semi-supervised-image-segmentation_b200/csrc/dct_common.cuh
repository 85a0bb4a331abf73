// dct_common.cuh -- shared device/host helpers for the sm_100a kernels of libdct_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstddef>
#include <type_traits>

#include "../../include/dct_b200.h"

namespace dct {

constexpr int kSMs = 148;             // B200: 2 dies x 74 SMs
constexpr int kMaxPartials = 8192;    // per-launch CTA partial sums kept in the workspace
constexpr float kEntEps = 1e-16f;     // Entropy / Entropy_2D epsilon (generalframework/loss/loss.py:64,81)

// Peer publication descriptor ("dct_peer_pub" in include/dct_b200.h): where the last CTA of a *_pub launch pushes a
// step's loss sums -- straight into every data-parallel rank's mailbox over NVLink (see peer_publish below).
struct PeerPub {
    const double* src;                          // n doubles (local device memory) holding the step's sums
    unsigned long long* seq;                    // device counter of publications made so far (shared by a rank's descriptors)
    unsigned long long* const* mailbox_table;   // DEVICE array of `world` mailbox pointers (own one included), peer-mapped
    int n, rank, world, nslots;
};
static_assert(sizeof(PeerPub) == sizeof(dct_peer_pub), "PeerPub mirrors dct_peer_pub");

// workspace layout: 64-byte header (all fields zero between launches: the last CTA of a launch re-arms them)
// followed by kMaxPartials double partials
struct Workspace {
    unsigned int ticket;         // CTAs that have finished
    unsigned int tile_counter;   // dynamic tile scheduler of the tile pipeline (dct_tile.cuh)
    unsigned int nonfinite;      // #CTAs that saw a NaN / inf / out-of-range per-thread partial sum
    unsigned int counts_zeroed;  // DCT_COUNTS_OVERWRITE: set (release) by CTA 0 once the launch's counters are cleared
    unsigned long long fx_lo;    // order-independent loss sum in 2^-40 fixed point: sum of the low 32 bits ...
    long long fx_hi;             // ... and of the (signed) high bits of every partial
    unsigned int pad[8];
    double partials[kMaxPartials];
    // per-sample exchange of the one-launch perturbation normalisation (dct_vat.cu, l2_ll_kernel): a launch counter that
    // gives every launch fresh tags, its ticket, and kL2LLSamples x 2 passes x kL2LLSlots self-validating 8-byte words
    // {32-bit tag | fp32 partial sum of squares}.  Zero between allocations; only that kernel writes here.
    unsigned int l2_epoch;
    unsigned int l2_ticket;
    unsigned int pad2[14];
    unsigned long long l2_slots[256 * 2 * 32];
};
static_assert(offsetof(Workspace, partials) == 64, "workspace header is 64 bytes");
constexpr int kL2LLSamples = 256, kL2LLSlots = 32;
static_assert(sizeof(((Workspace*)nullptr)->l2_slots) == (size_t)kL2LLSamples * 2 * kL2LLSlots * 8, "l2 exchange area");

struct Upstream {          // see "dct_upstream" in include/dct_b200.h
    const float* gmap;     // [B,HW] or null
    const float* gscalar;  // device scalar or null
    float gconst;
};

template <int K>
struct Views {
    const float* in[K];
    float* grad[K];
};

thread_local inline cudaError_t g_last_cuda_error = cudaSuccess;
int check_pub(const dct_peer_pub* d);  // dct_abi.cu: validates a host-side publication descriptor

inline int check_launch() {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        g_last_cuda_error = e;
        return DCT_ERR_CUDA;
    }
    return DCT_OK;
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (sm_90+): the kernels of one consistency step are 15-45 us each,
// so the ~2 us launch latency + prologue of kernel N+1 is overlapped with the tail of kernel N.
// Every kernel launched through launch_pdl() executes pdl_wait() before its first global-memory
// access (full completion + visibility of the previous grid), so no data dependency is relaxed.
// DCT_B200_PDL=0 in the environment falls back to plain stream-ordered launches.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

bool pdl_enabled();  // dct_abi.cu

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

// Developer tracing (dct_dev_trace_begin / _end, include/dct_b200.h): while a trace buffer is registered every launch of a
// traced kernel gets the next kTraceSlots * max_ctas words of it and its CTAs stamp %globaltimer there:
// [0] after griddepcontrol.wait, [1] / [2] kernel-specific mid points, [3] at the CTA's end.  Null in the product.
constexpr int kTraceSlots = 4;
unsigned long long* trace_next(int grid);   // dct_abi.cu; nullptr when tracing is off or the buffer is exhausted

inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

// ---------------------------------------------------------------------------------------------
// streaming 128/64/32-bit global accesses: every tensor on this path is touched exactly once,
// so bypass L1 allocation on loads and mark stores streaming (evict-first in L2).
// ---------------------------------------------------------------------------------------------
template <int VEC>
struct FVec;
template <>
struct alignas(4) FVec<1> {
    float v[1];
};
template <>
struct alignas(8) FVec<2> {
    float v[2];
};
template <>
struct alignas(16) FVec<4> {
    float v[4];
};

template <int VEC>
__device__ __forceinline__ FVec<VEC> ld_stream(const float* p) {
    FVec<VEC> r;
    if constexpr (VEC == 4) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3])
                     : "l"(p));
    } else if constexpr (VEC == 2) {
        asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.v[0]), "=f"(r.v[1]) : "l"(p));
    } else {
        asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r.v[0]) : "l"(p));
    }
    return r;
}

template <int VEC>
__device__ __forceinline__ void st_stream(float* p, const FVec<VEC>& r) {
    if constexpr (VEC == 4) {
        asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]),
                     "f"(r.v[3])
                     : "memory");
    } else if constexpr (VEC == 2) {
        asm volatile("st.global.cs.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]) : "memory");
    } else {
        asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(r.v[0]) : "memory");
    }
}

// VEC int64 labels (VEC*8 bytes) as 128-bit streaming loads
template <int VEC>
__device__ __forceinline__ void ld_labels(const int64_t* p, long long (&g)[VEC]) {
    if constexpr (VEC % 2 == 0) {
#pragma unroll
        for (int j = 0; j < VEC; j += 2) {
            asm volatile("ld.global.nc.L1::no_allocate.v2.s64 {%0,%1}, [%2];" : "=l"(g[j]), "=l"(g[j + 1]) : "l"(p + j));
        }
    } else {
#pragma unroll
        for (int j = 0; j < VEC; ++j) asm volatile("ld.global.nc.L1::no_allocate.s64 %0, [%1];" : "=l"(g[j]) : "l"(p + j));
    }
}

// ---------------------------------------------------------------------------------------------
// reductions
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// Fused exchange (SURVEY.md 8e: the path's only cross-rank coupling is a handful of loss scalars).  Instead of a
// collective launched after the step, the thread that has just written the step's LAST sum pushes all n sums into
// row `rank` of every rank's mailbox with plain stores over NVLink / NVSwitch peer mappings.  Each double travels as
// two 8-byte words {32 data bits | 32-bit sequence number}: an aligned 8-byte store is single-copy atomic, so a
// reader that sees the expected sequence number in a word also sees its data -- no fence, no flag round trip
// (the "LL" scheme of NCCL's low-latency protocol).  Mailbox row: DCT_PUB_ROW_WORDS u64; slot = seq % nslots.
// Only the *_pub kernel variants contain this code (a compile-time switch): measured on B200, linking a hook into
// every kernel's finisher cost 5.6 us per c2 step.  The mailbox pointer table lives in device memory next to the
// sequence counter (`dct_peer_pub.mailbox_table`), so the descriptor is six scalars in the kernel parameters.
// ---------------------------------------------------------------------------------------------
// Out of line and fed scalars only.  Measured (profiles/r04/ab_publish.log, profiles/r05/ab_exchange_loopback.log):
// with this code in a tile kernel -- inlined or called -- ptxas demotes the kernel's uniform registers (SASS: R2UR 7 -> 100,
// PLOP3 230 -> 363 in the C=19 adversarial-KL kernel), the producer's bulk-copy issue loop slows down and the kernel
// loses 9 % (C=4) to 19 % (C=19).  The product therefore chains the one-thread publication kernel behind the plain
// kernel with programmatic dependent launch (+2.4 us per step); the fused *_pub variant stays available for A/B.  `fresh` is the sum the calling launch has just produced for slot `fresh_ptr`; the
// other slots are read back from `src` (written by earlier kernels of the stream).
static __device__ __noinline__ void peer_publish(const double* src, unsigned long long* seq, unsigned long long seq_old,
                                                 int n, int rank, int world, int nslots,
                                                 unsigned long long* const* mailbox_table, const double* fresh_ptr,
                                                 double fresh) {
    const unsigned long long q = seq_old + 1ull;
    const unsigned long long tag = (q & 0xffffffffull) << 32;
    const size_t row = ((size_t)(q % (unsigned long long)nslots) * world + rank) * DCT_PUB_ROW_WORDS;
    for (int j = 0; j < n; ++j) {
        const double val = (src + j == fresh_ptr) ? fresh : __ldcg(src + j);
        const unsigned long long bits = (unsigned long long)__double_as_longlong(val);
        const unsigned long long w0 = tag | (bits & 0xffffffffull), w1 = tag | (bits >> 32);
        for (int p = 0; p < world; ++p) {
            // volatile 8-byte stores = st.volatile (relaxed, system scope; SASS STG.E.64.STRONG.SYS); every word
            // carries its own tag
            volatile unsigned long long* vd = mailbox_table[p] + row + 2 * j;
            vd[0] = w0;
            vd[1] = w1;
        }
    }
    *seq = q;
}

// Deterministic grid-wide sum of one double per thread.  Every CTA writes its partial to the
// workspace; the CTA that draws the last ticket adds the partials in index order and writes
// *out, then re-arms the ticket.  `out` may be null (nothing is done).  num_ctas <= kMaxPartials
// (image_grid + fits_partials on the host): a larger grid would write past `partials` into the l2 area.
__device__ __forceinline__ void grid_sum_to(double v, Workspace* ws, double* out, int cta_linear, int num_ctas) {
    if (out == nullptr) return;
    __shared__ double s_warp[32];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    if (lane == 0) s_warp[wid] = v;
    __syncthreads();
    if (wid == 0) {
        double t = lane < nw ? s_warp[lane] : 0.0;
        t = warp_sum(t);
        if (lane == 0) {
            ws->partials[cta_linear] = t;
            __threadfence();
            unsigned int ticket = atomicAdd(&ws->ticket, 1u);
            s_last = (ticket == (unsigned int)num_ctas - 1u);
        }
    }
    __syncthreads();
    if (s_last) {
        __threadfence();
        double acc = 0.0;
        // fixed order: thread t sums partials t, t+T, ... ; then the same block tree as above
        for (int i = threadIdx.x; i < num_ctas; i += blockDim.x) acc += __ldcg(&ws->partials[i]);
        acc = warp_sum(acc);
        __syncthreads();
        if (lane == 0) s_warp[wid] = acc;
        __syncthreads();
        if (wid == 0) {
            double t = lane < nw ? s_warp[lane] : 0.0;
            t = warp_sum(t);
            if (lane == 0) {
                *out = t;
                ws->ticket = 0u;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Order-independent, bit-reproducible grid sum for the dynamically scheduled tile pipeline.
// Every per-thread fp32 partial (the sum of one thread's 1..4 pixel values of one tile) is
// converted exactly to 2^-40 fixed point (fp32 * 2^40 is exact; the int64 conversion is exact for
// |partial| < 2^23) and accumulated with integer adds, which are associative: the result does not
// depend on which CTA processed which tile.  Low and high halves are summed separately so that
// nothing can overflow (N < 2^31 partials).  NaN / inf partials poison the result (NaN).
// ---------------------------------------------------------------------------------------------
constexpr float kFxScale = 1099511627776.0f;  // 2^40
__device__ __forceinline__ long long to_fixed(float part, bool& nonfinite) {
    nonfinite |= !(fabsf(part) < 8388608.0f);
    return __float2ll_rn(part * kFxScale);
}
__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Called by every thread of the CTA at the end of a tile-pipeline kernel.  `out` may be null.
// Also re-arms the workspace header (ticket, tile counter, accumulators) when the last CTA is through.
template <bool PUB = false>
__device__ __forceinline__ void tile_grid_finish(long long acc_fx, bool nonfinite, Workspace* ws, double* out, int num_ctas,
                                                 const PeerPub* pub = nullptr, int pub_early = 0) {
    if (ws == nullptr) return;
    __shared__ long long s_lo[20], s_hi[20];  // <= 17 warps per CTA
    __shared__ int s_nf;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if (out != nullptr) {
        if (threadIdx.x == 0) s_nf = 0;
        long long lo = (long long)((unsigned long long)acc_fx & 0xffffffffull), hi = acc_fx >> 32;
        lo = warp_sum(lo);
        hi = warp_sum(hi);
        const bool wnf = __any_sync(0xffffffffu, nonfinite);
        __syncthreads();
        if (lane == 0) { s_lo[wid] = lo; s_hi[wid] = hi; if (wnf) s_nf = 1; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (out != nullptr) {
            long long lo = 0, hi = 0;
            for (int w = 0; w < nw; ++w) { lo += s_lo[w]; hi += s_hi[w]; }
            atomicAdd(&ws->fx_lo, (unsigned long long)lo);
            atomicAdd(reinterpret_cast<unsigned long long*>(&ws->fx_hi), (unsigned long long)hi);
            if (s_nf) atomicAdd(&ws->nonfinite, 1u);
        }
        __threadfence();
        const unsigned int ticket = atomicAdd(&ws->ticket, 1u);
        if constexpr (PUB) {
            // Early publication: `pub->src` holds sums that were final BEFORE this launch started (the previous step's: every
            // kernel that wrote them completed ahead of this grid's dependency wait).  The FIRST CTA to finish pushes them to
            // the peers while the other CTAs are still working -- the CTAs of a launch end 3-4 us apart, so the ~2 us of the
            // publication (counter and sums read back, remote stores) sit in the launch's own tail instead of between two
            // launches of the stream.
            if (pub_early && ticket == 0u)
                peer_publish(pub->src, pub->seq, __ldcg(pub->seq), pub->n, pub->rank, pub->world, pub->nslots,
                             pub->mailbox_table, nullptr, 0.0);
        }
        if (ticket == (unsigned int)num_ctas - 1u) {  // last CTA: publish the sum and re-arm the header
            __threadfence();
            if (out != nullptr) {
                const unsigned long long lo = __ldcg(&ws->fx_lo);
                const long long hi = __ldcg(&ws->fx_hi);
                const unsigned int nf = __ldcg(&ws->nonfinite);
                const double total = ((double)hi * 4294967296.0 + (double)lo) * (1.0 / 1099511627776.0);
                const double fin = nf ? __longlong_as_double(0x7ff8000000000000ll) : total;
                *out = fin;
                if constexpr (PUB)  // the step's sums -> every rank's mailbox (NVLink)
                    if (!pub_early) peer_publish(pub->src, pub->seq, __ldcg(pub->seq), pub->n, pub->rank, pub->world, pub->nslots,
                                 pub->mailbox_table, out, fin);
                ws->fx_lo = 0ull;
                ws->fx_hi = 0ll;
                ws->nonfinite = 0u;
            }
            ws->tile_counter = 0u;
            ws->counts_zeroed = 0u;
            __threadfence();
            ws->ticket = 0u;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// grid geometry: blockIdx.y = image b, blockIdx.x strides over the image's pixel groups, so a CTA
// never straddles two images (per-image integer counts and per-sample norms stay CTA-local).
// One pixel group per thread (thousands of small CTAs: the hardware block scheduler balances the
// tail); B <= 65535 is checked by the callers.  Every CTA of a grid_sum_to launch owns one of the
// kMaxPartials partial-sum slots, so the grid never has more CTAs than that: for B > max_ctas,
// gridDim.y = max_ctas and the kernels stride over images (b = blockIdx.y, blockIdx.y + gridDim.y, ...).
// For B <= max_ctas that loop runs once and the grid is one row per image.
// ---------------------------------------------------------------------------------------------
inline dim3 image_grid(int64_t B, int64_t groups_per_image, int threads, int64_t max_ctas = kMaxPartials) {
    const int64_t gy = B < 1 ? 1 : (B < max_ctas ? B : max_ctas);
    int64_t gx = (groups_per_image + threads - 1) / threads;  // one pixel group per thread ...
    const int64_t cap = max_ctas / gy;                         // ... unless that exceeds the partial-sum slots (cap >= 1)
    if (gx > cap) gx = cap;                                    // then threads stride over the image
    if (gx < 1) gx = 1;
    return dim3((unsigned)gx, (unsigned)gy, 1);
}

// host-side guard in front of every launch that ends in grid_sum_to: one partial-sum slot per CTA
inline bool fits_partials(dim3 grid) { return (int64_t)grid.x * grid.y * grid.z <= kMaxPartials; }

// ---------------------------------------------------------------------------------------------
// The pinned softmax arithmetic for the integer (Dice) path -- see DESIGN.md "Dice spec".
// Explicit round-to-nearest intrinsics: never contracted, never flushed, independent of flags.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float spec_expf(float d) {
    if (!(d >= -87.0f)) return (d != d) ? d : 0.0f;
    float t = __fmul_rn(d, 1.44269504088896341f);
    float n = rintf(t);
    float r = __fmaf_rn(n, -0.693359375f, d);
    r = __fmaf_rn(n, 2.12194440e-4f, r);
    float y = __fmaf_rn(1.9875691500e-4f, r, 1.3981999507e-3f);
    y = __fmaf_rn(y, r, 8.3334519073e-3f);
    y = __fmaf_rn(y, r, 4.1665795894e-2f);
    y = __fmaf_rn(y, r, 1.6666665459e-1f);
    y = __fmaf_rn(y, r, 5.0000001201e-1f);
    float z = __fmul_rn(r, r);
    y = __fmaf_rn(y, z, r);
    y = __fadd_rn(y, 1.0f);
    int e = (int)n + 127;
    float scale = __int_as_float(e << 23);
    return __fmul_rn(y, scale);
}

// The full pinned arithmetic (slow path of the arg-max below; the test-side CPU checker restates it operation for operation).
template <int C>
__device__ __forceinline__ int spec_softmax_argmax_full(const float (&x)[C]) {
    float m = x[0];
#pragma unroll
    for (int c = 1; c < C; ++c)
        if (x[c] > m) m = x[c];
    float S = 0.0f;
    bool any_nan = false;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        float d = __fsub_rn(x[c], m);
        any_nan |= (d != d);
        float e = spec_expf(d);
        S = (c == 0) ? e : __fadd_rn(S, e);
    }
    if (any_nan) return 0;
    int best = 0;
    float qb = __fdiv_rn(spec_expf(__fsub_rn(x[0], m)), S);
#pragma unroll
    for (int c = 1; c < C; ++c) {
        float q = __fdiv_rn(spec_expf(__fsub_rn(x[c], m)), S);
        if (q > qb) { qb = q; best = c; }
    }
    return best;
}

static __device__ __noinline__ int spec_full_upto4(float x0, float x1, float x2, float x3, int C) {
    float x[4] = {x0, x1, x2, x3};
    float m = x[0];
    for (int c = 1; c < C; ++c)
        if (x[c] > m) m = x[c];
    float S = 0.0f;
    bool any_nan = false;
    for (int c = 0; c < C; ++c) {
        float d = __fsub_rn(x[c], m);
        any_nan |= (d != d);
        float e = spec_expf(d);
        S = (c == 0) ? e : __fadd_rn(S, e);
    }
    if (any_nan) return 0;
    int best = 0;
    float qb = __fdiv_rn(spec_expf(__fsub_rn(x[0], m)), S);
    for (int c = 1; c < C; ++c) {
        float q = __fdiv_rn(spec_expf(__fsub_rn(x[c], m)), S);
        if (q > qb) { qb = q; best = c; }
    }
    return best;
}

// pred = argmax_c softmax_spec(x)_c, returned as a one-hot BYTE mask (1 << 8*pred) for C <= 4
// (what the packed Dice counters add), or as the index for larger C.
//
// Fast path.  Let t = fl(max - 2^-15).  If exactly one class satisfies x_c >= t and all inputs are
// finite, every other class has fl(x_c - max) <= -2^-17, so spec_expf(d_c) <= 1 - 2^-18 < 1 = spec_expf(0)
// and IEEE division by the common sum keeps q_c < q_max strictly: the raw arg-max IS the pinned
// answer.  Near-ties, exact ties, NaN and +-inf (detected through the finiteness of the class sum)
// run the full pinned arithmetic.  One-hot masks make "exactly one" a power-of-two test.
template <int C>
__device__ __forceinline__ unsigned int spec_softmax_argmax_onehot4(const float (&x)[C]) {
    static_assert(C <= 4, "one-hot byte mask needs C <= 4");
    float m = x[0], s = x[0];
#pragma unroll
    for (int c = 1; c < C; ++c) { m = fmaxf(m, x[c]); s += x[c]; }
    const float t = m - 3.0517578125e-05f;
    unsigned int hot = 0u;
#pragma unroll
    for (int c = 0; c < C; ++c) hot += (x[c] >= t) ? (1u << (8 * c)) : 0u;
    const bool fast = ((hot & (hot - 1u)) == 0u) & (hot != 0u) & (fabsf(s) <= 3.4028234664e38f);
    if (fast) return hot;
    // rare: scalars by value into an out-of-line call, so x[] never becomes address-taken
    return 1u << (8 * spec_full_upto4(x[0], C > 1 ? x[C > 1 ? 1 : 0] : 0.0f, C > 2 ? x[C > 2 ? 2 : 0] : 0.0f,
                                      C > 3 ? x[C > 3 ? 3 : 0] : 0.0f, C));
}

template <int C>
__device__ __forceinline__ int spec_softmax_argmax(const float (&x)[C]) {
    float m = x[0], s = x[0];
    int am = 0;
#pragma unroll
    for (int c = 1; c < C; ++c) {
        s += x[c];
        if (x[c] > m) { m = x[c]; am = c; }
    }
    const float t = m - 3.0517578125e-05f;
    int n_ge = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) n_ge += (x[c] >= t) ? 1 : 0;
    if ((n_ge == 1) & (fabsf(s) <= 3.4028234664e38f)) return am;
    return spec_softmax_argmax_full<C>(x);
}

// runtime-C variant reading a strided column (generic fallback kernels)
__device__ __forceinline__ int spec_softmax_argmax_rt(const float* xb, int C, int64_t HW) {
    float m = xb[0];
    for (int c = 1; c < C; ++c) { float v = xb[(int64_t)c * HW]; if (v > m) m = v; }
    float S = 0.0f;
    bool any_nan = false;
    for (int c = 0; c < C; ++c) {
        float d = __fsub_rn(xb[(int64_t)c * HW], m);
        any_nan |= (d != d);
        float e = spec_expf(d);
        S = (c == 0) ? e : __fadd_rn(S, e);
    }
    if (any_nan) return 0;
    int best = 0;
    float qb = __fdiv_rn(spec_expf(__fsub_rn(xb[0], m)), S);
    for (int c = 1; c < C; ++c) {
        float q = __fdiv_rn(spec_expf(__fsub_rn(xb[(int64_t)c * HW], m)), S);
        if (q > qb) { qb = q; best = c; }
    }
    return best;
}

// torch.max(dim) semantics on raw scores: first index on ties, NaN is maximal (first NaN wins)
template <int C>
__device__ __forceinline__ int raw_argmax(const float (&x)[C]) {
    float m = x[0];
    int best = 0;
    bool locked = (m != m);
#pragma unroll
    for (int c = 1; c < C; ++c) {
        float v = x[c];
        bool take = !locked && ((v != v) || (v > m));
        if (take) { m = v; best = c; }
        locked |= (v != v);
    }
    return best;
}

__device__ __forceinline__ int raw_argmax_rt(const float* xb, int C, int64_t HW) {
    float m = xb[0];
    int best = 0;
    if (m != m) return 0;
    for (int c = 1; c < C; ++c) {
        float v = xb[(int64_t)c * HW];
        if (v != v) return c;
        if (v > m) { m = v; best = c; }
    }
    return best;
}

// ---------------------------------------------------------------------------------------------
// transcendental wrappers for the floating-point kernels.  Default: MUFU-based intrinsics
// (ex2.approx / lg2.approx / rcp.approx; errors ~1e-7 relative, see DESIGN.md "Accuracy budget").
// -DDCT_ACCURATE_MATH switches to libdevice expf/logf and IEEE division for A/B checks.
// ---------------------------------------------------------------------------------------------
#ifdef DCT_ACCURATE_MATH
__device__ __forceinline__ float fexp(float x) { return expf(x); }
__device__ __forceinline__ float flog(float x) { return logf(x); }
__device__ __forceinline__ float fdiv(float a, float b) { return a / b; }
#else
__device__ __forceinline__ float fexp(float x) { return __expf(x); }
__device__ __forceinline__ float flog(float x) { return __logf(x); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdividef(a, b); }
#endif

// base-2 MUFU primitives with flush-to-zero (one SASS instruction each, no denormal fix-up code).
// Inputs on this path are never denormal where it matters: ex2 arguments are <= 0 (results below
// 2^-126 flush to 0 = a probability of 0), lg2 arguments are >= 1e-16.
__device__ __forceinline__ float ex2_ftz(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_ftz(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_ftz(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
constexpr float kLog2e = 1.44269504088896341f;
constexpr float kLn2 = 0.69314718055994531f;

// the reference's simplex predicate for one pixel: |sum - 1| <= 1e-8 + 1e-5 (utils/utils.py:142-151)
__device__ __forceinline__ bool simplex_ok(float s) { return fabsf(s - 1.0f) <= (1e-8f + 1e-5f); }

// ---------------------------------------------------------------------------------------------
// Lane types of the per-pixel math.  Every Op body is written once against the v*() helpers below
// and instantiated for T = float (one pixel) and T = f2 (TWO pixels in a 64-bit register pair).
// On sm_100 the f2 adds / multiplies / FMAs are single packed instructions (SASS FADD2 / FMUL2 /
// FFMA2 via __fadd2_rn / __fmul2_rn / __ffma2_rn): the tile kernels are issue-slot bound at their
// low occupancy, and packing halves the FP32 instruction count.  Per component the packed ops
// round exactly like their scalar twins, so both instantiations give bit-identical results.
// MUFU (ex2/lg2/rcp), min/max and compares stay per component.
// ---------------------------------------------------------------------------------------------
struct f2 {
    float2 v;
};
__device__ __forceinline__ f2 mk2(float a, float b) { return f2{make_float2(a, b)}; }

template <class T> __device__ __forceinline__ T vset(float s);
template <> __device__ __forceinline__ float vset<float>(float s) { return s; }
template <> __device__ __forceinline__ f2 vset<f2>(float s) { return mk2(s, s); }

__device__ __forceinline__ float vadd(float a, float b) { return a + b; }
__device__ __forceinline__ float vsub(float a, float b) { return a - b; }
__device__ __forceinline__ float vmul(float a, float b) { return a * b; }
__device__ __forceinline__ float vfma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ float vmax(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ float vneg(float a) { return -a; }
__device__ __forceinline__ float vex2(float a) { return ex2_ftz(a); }
__device__ __forceinline__ float vlg2(float a) { return lg2_ftz(a); }
__device__ __forceinline__ float vrcp(float a) { return rcp_ftz(a); }
__device__ __forceinline__ float vlog(float a) { return flog(a); }
__device__ __forceinline__ float vexp(float a) { return fexp(a); }
__device__ __forceinline__ float vdiv(float a, float b) { return fdiv(a, b); }
__device__ __forceinline__ float vhsum(float a) { return a; }
__device__ __forceinline__ bool vsimplex_bad(float s) { return !simplex_ok(s); }

__device__ __forceinline__ f2 vadd(f2 a, f2 b) { return f2{__fadd2_rn(a.v, b.v)}; }
__device__ __forceinline__ f2 vmul(f2 a, f2 b) { return f2{__fmul2_rn(a.v, b.v)}; }
__device__ __forceinline__ f2 vfma(f2 a, f2 b, f2 c) { return f2{__ffma2_rn(a.v, b.v, c.v)}; }
// a - b as fma(b, -1, a): one rounding of the exact difference, identical to a subtraction
__device__ __forceinline__ f2 vsub(f2 a, f2 b) { return f2{__ffma2_rn(b.v, make_float2(-1.0f, -1.0f), a.v)}; }
__device__ __forceinline__ f2 vmax(f2 a, f2 b) { return mk2(fmaxf(a.v.x, b.v.x), fmaxf(a.v.y, b.v.y)); }
__device__ __forceinline__ f2 vneg(f2 a) { return mk2(-a.v.x, -a.v.y); }
__device__ __forceinline__ f2 vex2(f2 a) { return mk2(ex2_ftz(a.v.x), ex2_ftz(a.v.y)); }
__device__ __forceinline__ f2 vlg2(f2 a) { return mk2(lg2_ftz(a.v.x), lg2_ftz(a.v.y)); }
__device__ __forceinline__ f2 vrcp(f2 a) { return mk2(rcp_ftz(a.v.x), rcp_ftz(a.v.y)); }
__device__ __forceinline__ f2 vlog(f2 a) { return mk2(flog(a.v.x), flog(a.v.y)); }
__device__ __forceinline__ f2 vexp(f2 a) { return mk2(fexp(a.v.x), fexp(a.v.y)); }
__device__ __forceinline__ f2 vdiv(f2 a, f2 b) { return mk2(fdiv(a.v.x, b.v.x), fdiv(a.v.y, b.v.y)); }
__device__ __forceinline__ float vhsum(f2 a) { return a.v.x + a.v.y; }
__device__ __forceinline__ float vget(float a, int) { return a; }
__device__ __forceinline__ float vget(f2 a, int j) { return j == 0 ? a.v.x : a.v.y; }
__device__ __forceinline__ bool vsimplex_bad(f2 s) { return !simplex_ok(s.v.x) | !simplex_ok(s.v.y); }

// scalar-operand forms (the scalar is broadcast for f2)
template <class T> __device__ __forceinline__ T vadds(T a, float s) { return vadd(a, vset<T>(s)); }
template <class T> __device__ __forceinline__ T vmuls(T a, float s) { return vmul(a, vset<T>(s)); }
template <class T> __device__ __forceinline__ T vfmas(T a, float s, T c) { return vfma(a, vset<T>(s), c); }

// apply a scalar function per component (for the rare exact-arithmetic ops)
template <class F> __device__ __forceinline__ float vmap(F f, float a, float b) { return f(a, b); }
template <class F> __device__ __forceinline__ f2 vmap(F f, f2 a, f2 b) { return mk2(f(a.v.x, b.v.x), f(a.v.y, b.v.y)); }

__device__ __forceinline__ float upstream_scalar(const Upstream& u) {
    float g = u.gconst;
    if (u.gscalar != nullptr) g *= __ldg(u.gscalar);
    return g;
}

}  // namespace dct
