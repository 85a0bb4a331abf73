// dct_vat.cu -- VAT / FGSM perturbation arithmetic on image-shaped tensors.
//
// Replaces VATGenerator._l2_normalize (generalframework/utils/AEGenerator.py:68-76), the scale /
// add / clamp tail of VATGenerator.__call__ (:103,:112-117) and FSGMGenerator.adversarial_fgsm
// (:35-51).
//
// _l2_normalize is a per-sample reduction followed by a per-sample rescale.  On B200 a sample of
// M*4 bytes is spread over a thread-block CLUSTER: every CTA of the cluster keeps its slice of
// the sample in registers, the partial sums of squares are exchanged through distributed shared
// memory, and each CTA rescales and stores its slice -- the sample is read from HBM once and
// written once (2*M*4 bytes, the algorithmic minimum) in a single launch.  Samples too large for
// 8 CTAs x 256 threads x 64 floats fall back to a two-launch path (sum of squares into the
// workspace, then rescale; the second read is served by the 126 MB L2).
#include <cooperative_groups.h>
#include <cuda_bf16.h>

#include "dct_common.cuh"

namespace cg = cooperative_groups;

namespace dct {

constexpr int kL2Threads = 256;
constexpr int kL2Cluster = 8;       // portable maximum cluster size
constexpr int kL2ClusterBig = 16;   // B200's non-portable maximum (opt-in per function): samples up to 1 MB stay one launch
constexpr int kL2MaxVecPerThread = 16;  // float4 per thread held in registers (64 floats)

struct L2Args {
    const float* d;
    float* out;
    int64_t M;
    int passes;        // 1, or 2 = normalise(normalise(d)) (AEGenerator.py:98 followed by :103)
    float scale;
    const float* img;  // nullable
    float* adv;        // nullable
    Workspace* ws;
    unsigned long long* trace;   // developer tracing (dct_common.cuh, trace_next); null in the product
    int prefetch;                // 1: the sample's lines are pulled into L2 before the dependency wait
};

__device__ __forceinline__ float block_sum_f(float v, float* s_warp) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_sum(v);
    if (lane == 0) s_warp[wid] = v;
    __syncthreads();
    float t = 0.0f;
    if (wid == 0) {
        t = lane < nw ? s_warp[lane] : 0.0f;
        t = warp_sum(t);
        if (lane == 0) s_warp[0] = t;
    }
    __syncthreads();
    t = s_warp[0];
    __syncthreads();
    return t;
}

// What one element goes through once the sample's sum of squares `ss` is known: d / n1 [/ n2] * scale, each step rounded
// like the reference's own sequence of ops (AEGenerator.py:72,103: `d /= norm`, again, `xi * d`), with the divisions as
// multiplications by the correctly rounded reciprocal (<= 1 ulp each; an IEEE divide per element is ~10 instructions and
// these launches are latency-bound).  n1 = sqrt(ss) + 1e-16; n2 = || d / n1 || + 1e-16 = sqrt(ss) / n1 + 1e-16.
struct L2Scale {
    float r1, r2, scale;
    bool twice;
};
__device__ __forceinline__ L2Scale l2_scales(float ss, int passes, float scale) {
    const float root = sqrtf(ss);
    const float n1 = root + 1e-16f;
    L2Scale s;
    s.r1 = __frcp_rn(n1);
    s.twice = passes > 1;
    s.r2 = s.twice ? __frcp_rn(__fdiv_rn(root, n1) + 1e-16f) : 1.0f;
    s.scale = scale;
    return s;
}
__device__ __forceinline__ float l2_apply(float x, const L2Scale& s) {
    float q = __fmul_rn(x, s.r1);
    if (s.twice) q = __fmul_rn(q, s.r2);
    return __fmul_rn(s.scale, q);
}

// One cluster per sample; NV float4 per thread (compile-time so the slice lives in registers).
// Critical path: warp shuffle tree -> one shared-memory word per warp -> ONE cluster barrier -> every warp gathers the
// 8 CTAs x 8 warps partials through distributed shared memory (2 per lane) and reduces them with the same shuffle tree
// (so all 2048 threads of the cluster hold bit-identical norms); the image (for the clamp(img + r) tail) is prefetched
// before the barrier.
template <int NV, bool IMG, int CL = kL2Cluster>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(kL2Threads, (NV <= 8 ? 3 : 1))   // <= 80 registers up to NV = 8
l2_cluster_kernel(const L2Args a) {
    constexpr int kL2Cluster = CL;   // (shadows the namespace constant: 8, or 16 for the large-sample instantiations)
    constexpr int kWarps = kL2Threads / 32;
    static_assert((CL * kWarps) % 32 == 0 && kWarps == 8, "gather: CL x 8 partials, CL / 4 per lane");
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ float s_wsum[2][kL2Threads / 32];  // [pass][warp], read by the cluster peers
    const unsigned int rank = cluster.block_rank();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t b = blockIdx.x / kL2Cluster;
    const int64_t base = b * a.M;
    const int64_t nvec = a.M / 4;
    FVec<4> v[NV];
    float ss = 0.0f;
    if (a.prefetch && (threadIdx.x & 7) == 0) {
        // ramp hiding (see dct_tile.cuh): this CTA's lines of `d` go to L2 while the previous grid drains; a prefetch moves
        // no value into the SM, so the ordering against that grid's writes is untouched
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int64_t q = ((int64_t)j * kL2Cluster + rank) * kL2Threads + threadIdx.x;
            if (q < nvec) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.d + base + q * 4));
        }
    }
    pdl_wait();
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * blockIdx.x] = globaltimer_ns();
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int64_t q = ((int64_t)j * kL2Cluster + rank) * kL2Threads + threadIdx.x;  // float4 index in sample
        if (q < nvec) {
            v[j] = ld_stream<4>(a.d + base + q * 4);
            // the image is only needed after the exchange: its lines are pulled into L2 now (one prefetch per 128-byte line)
            // and read from there later, instead of sitting in 4 * NV more registers per thread -- at 96 registers only
            // 31 of a 32-sample batch's clusters were co-resident and the last one started a whole kernel late (profiles/r25)
            if constexpr (IMG) {
                if ((threadIdx.x & 7) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.img + base + q * 4));
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int64_t q = ((int64_t)j * kL2Cluster + rank) * kL2Threads + threadIdx.x;
        if (q < nvec) ss += v[j].v[0] * v[j].v[0] + v[j].v[1] * v[j].v[1] + v[j].v[2] * v[j].v[2] + v[j].v[3] * v[j].v[3];
    }
    // ONE exchange per launch.  The second normalisation of passes == 2 (AEGenerator.py:98 followed by :103) divides by
    // || d / n1 ||: in exact arithmetic sqrt(ss) / n1, and any fp32 summation of the rounded quotients' squares sits within a
    // few 2^-24 of that (as do two different summation orders of it), far inside the 1e-5 budget -- so it is formed from the
    // first sum instead of a second read-reduce-exchange round (measured: 3 us of a 10.9 us launch, profiles/r25).
    const float w = warp_sum(ss);
    if (lane == 0) s_wsum[0][wid] = w;
    cluster.sync();
    float t = 0.0f;
#pragma unroll
    for (int i = 0; i < CL / 4; ++i)   // lane l reads warp (l & 7) of CTAs (l >> 3) + 4 i, in a fixed order
        t += *cluster.map_shared_rank(&s_wsum[0][lane & 7], 4 * i + (lane >> 3));
    // No CTA may exit (and free s_wsum) while a peer can still be reading it: this thread's peer reads are done -- it
    // arrives here and waits at the exit, by when the stores below have normally given every peer time to arrive.
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    t = warp_sum(t);
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * blockIdx.x + 2] = globaltimer_ns();
    const L2Scale sc = l2_scales(t, a.passes, a.scale);
    FVec<4> im[IMG ? NV : 1];
    if constexpr (IMG) {
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int64_t q = ((int64_t)j * kL2Cluster + rank) * kL2Threads + threadIdx.x;
            if (q < nvec) im[j] = ld_stream<4>(a.img + base + q * 4);   // L2 hits (prefetched above)
        }
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int64_t q = ((int64_t)j * kL2Cluster + rank) * kL2Threads + threadIdx.x;
        if (q < nvec) {
            const int64_t off = base + q * 4;
            FVec<4> o;
#pragma unroll
            for (int e = 0; e < 4; ++e) o.v[e] = l2_apply(v[j].v[e], sc);
            st_stream<4>(a.out + off, o);
            if constexpr (IMG) {
                FVec<4> ad;
#pragma unroll
                for (int e = 0; e < 4; ++e) ad.v[e] = fminf(fmaxf(im[j].v[e] + o.v[e], 0.0f), 1.0f);
                st_stream<4>(a.adv + off, ad);
            }
        }
    }
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * blockIdx.x + 4] = globaltimer_ns();   // stores issued
    pdl_launch_dependents();
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * blockIdx.x + 3] = globaltimer_ns();
}

// ---- one launch without a cluster: co-resident CTAs, per-sample exchange through self-validating words in L2 ----------------
// The cluster kernel above spends 35 % of its duration with no SM active (cluster launch / drain, profiles/r18).  Here a
// sample is spread over `cps` ordinary CTAs of one co-resident grid.  Per normalisation pass every CTA reduces its slice's
// sum of squares (shuffle tree -> one shared-memory word per warp -> warp 0) and stores it as ONE aligned 8-byte word
// {tag | fp32 bits} into its slot of the sample's row in the workspace; lanes 0..cps-1 of warp 0 then poll the sample's cps
// slots until each carries this launch's tag.  An aligned 8-byte store is single-copy atomic, so a matching tag implies the
// data (the scheme of the mailbox exchange, dct_common.cuh): no fence, no atomic, no flag round trip on the critical path.
// All CTAs add the cps partials with the same shuffle tree, so the whole sample sees one bit-identical norm.
// Tags: (launch epoch + 1) * 2 + pass; the epoch lives in the workspace and is bumped by the launch's last CTA (ticket), i.e.
// after every CTA has read it.  Co-residency (the polls would deadlock otherwise) is checked by the host: grid <= 148 x
// the kernel's resident CTAs per SM; larger problems take the cluster / grid-wide paths.
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

template <int NV, bool IMG, int THREADS>
__global__ void __launch_bounds__(THREADS) l2_ll_kernel(const L2Args a, int cps) {
    constexpr int kWarps = THREADS / 32;
    static_assert(kWarps <= 32, "one shared-memory word per warp, reduced by warp 0");
    __shared__ float s_w[kWarps];
    __shared__ float s_tot;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t b = blockIdx.x / cps;
    const int rank = (int)(blockIdx.x - b * cps);
    const int64_t base = b * a.M;
    const int64_t nvec = a.M / 4;
    FVec<4> v[NV];
    FVec<4> im[IMG ? NV : 1];
    if (a.prefetch && (threadIdx.x & 7) == 0) {   // ramp hiding, as in the cluster kernel
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int64_t q = ((int64_t)j * cps + rank) * THREADS + threadIdx.x;
            if (q < nvec) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(a.d + base + q * 4));
                if constexpr (IMG) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.img + base + q * 4));
            }
        }
    }
    pdl_wait();
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * blockIdx.x] = globaltimer_ns();
    const unsigned int epoch = __ldcg(&a.ws->l2_epoch);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int64_t q = ((int64_t)j * cps + rank) * THREADS + threadIdx.x;  // float4 index in sample
        if (q < nvec) {
            v[j] = ld_stream<4>(a.d + base + q * 4);
            if constexpr (IMG) im[j] = ld_stream<4>(a.img + base + q * 4);
        }
    }
    float ss = 0.0f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int64_t q = ((int64_t)j * cps + rank) * THREADS + threadIdx.x;
        if (q < nvec) ss += v[j].v[0] * v[j].v[0] + v[j].v[1] * v[j].v[1] + v[j].v[2] * v[j].v[2] + v[j].v[3] * v[j].v[3];
    }
    {   // one exchange per launch (the second norm of passes == 2 follows from the first sum, see l2_scales)
        const int pass = 0;
        const float w = warp_sum(ss);
        if (lane == 0) s_w[wid] = w;
        __syncthreads();
        if (wid == 0) {
            float t = lane < kWarps ? s_w[lane] : 0.0f;
            t = warp_sum(t);
            const unsigned long long tag = (unsigned long long)((epoch + 1u) * 2u + (unsigned int)pass) << 32;
            unsigned long long* row = a.ws->l2_slots + ((size_t)b * 2 + pass) * kL2LLSlots;
            if (lane == 0) st_relaxed_u64(row + rank, tag | (unsigned long long)__float_as_uint(t));
            float p = 0.0f;
            if (lane < cps) {
                unsigned long long got;
                do { got = ld_relaxed_u64(row + lane); } while ((got & 0xffffffff00000000ull) != tag);
                p = __uint_as_float((unsigned int)(got & 0xffffffffull));
            }
            __syncwarp();
            p = warp_sum(p);   // the same tree in every CTA of the sample: one bit-identical sum
            if (lane == 0) s_tot = p;
        }
        __syncthreads();
        if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * blockIdx.x + 2] = globaltimer_ns();
    }
    const L2Scale sc = l2_scales(s_tot, a.passes, a.scale);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int64_t q = ((int64_t)j * cps + rank) * THREADS + threadIdx.x;
        if (q < nvec) {
            const int64_t off = base + q * 4;
            FVec<4> o;
#pragma unroll
            for (int e = 0; e < 4; ++e) o.v[e] = l2_apply(v[j].v[e], sc);
            st_stream<4>(a.out + off, o);
            if constexpr (IMG) {
                FVec<4> ad;
#pragma unroll
                for (int e = 0; e < 4; ++e) ad.v[e] = fminf(fmaxf(im[j].v[e] + o.v[e], 0.0f), 1.0f);
                st_stream<4>(a.adv + off, ad);
            }
        }
    }
    pdl_launch_dependents();
    if (threadIdx.x == 0) {   // the launch's last CTA retires this launch's tags (every CTA has read the epoch long ago)
        const unsigned int ticket = atomicAdd(&a.ws->l2_ticket, 1u);
        if (ticket == gridDim.x - 1u) {
            a.ws->l2_ticket = 0u;
            a.ws->l2_epoch = epoch + 1u;
        }
        if (a.trace != nullptr) a.trace[kTraceSlots * blockIdx.x + 3] = globaltimer_ns();
    }
}

// host side of the kernel above: picks (cps, NV), checks co-residency once per instantiation; false = not served
template <int NV, bool IMG>
static bool l2_ll_try(const L2Args& a, int64_t B, int cps, cudaStream_t s, cudaError_t& err) {
    constexpr int THREADS = 256;
    auto kern = l2_ll_kernel<NV, IMG, THREADS>;
    static int resident = -1;   // CTAs of this instantiation one SM holds
    if (resident < 0) {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, THREADS, 0) != cudaSuccess) n = 0;
        resident = n;
    }
    if (B * cps > (int64_t)kSMs * resident) return false;
    L2Args at = a;
    at.trace = trace_next((int)(B * cps));
    err = launch_pdl(kern, dim3((unsigned)(B * cps)), dim3(THREADS), 0, s, at, cps);
    return true;
}

// ---- large / odd samples: two grid-wide launches through the workspace ------------------------------------------------
// Workspace layout of this path: sample b owns gx + 1 doubles: [0, gx) one partial per CTA of its row of the grid, [gx] the
// sample's sum of squares (as the float the scale launch works with).  The CTA that draws the last ticket of the first
// launch adds every sample's partials in a fixed order (one warp per sample: lane l takes partials l, l + 32, ...; shuffle
// tree) -- deterministic -- and re-arms the ticket.
__device__ __forceinline__ void l2_finish_sums(double ss, Workspace* ws, int gx) {
    __shared__ double s_warp[8];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    ss = warp_sum(ss);
    if (lane == 0) s_warp[wid] = ss;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += s_warp[w];
        ws->partials[(size_t)blockIdx.y * (gx + 1) + blockIdx.x] = t;
        __threadfence();
        const unsigned int ticket = atomicAdd(&ws->ticket, 1u);
        s_last = ticket == gridDim.x * gridDim.y - 1u;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int b = wid; b < (int)gridDim.y; b += 8) {
        const double* part = ws->partials + (size_t)b * (gx + 1);
        double t = 0.0;
        for (int i = lane; i < gx; i += 32) t += __ldcg(part + i);
        t = warp_sum(t);
        if (lane == 0) ws->partials[(size_t)b * (gx + 1) + gx] = (double)(float)t;
    }
    __syncthreads();
    if (threadIdx.x == 0) { __threadfence(); ws->ticket = 0u; }
}

// launch A: sum of squares of every sample.  VEC = 4: 128-bit streaming loads (M % 4 == 0, 16-byte aligned rows)
// (Four independent loads per thread and iteration, a grid stride apart, were measured and removed: c4 l2_direction 63 -> 68 us,
// l2_radv 89 -> 92 us -- 8 CTAs x 256 threads per SM already keep enough lines in flight, profiles/r43/bench_quick.log.)
template <int VEC>
__global__ void __launch_bounds__(256) l2_sumsq_kernel(const L2Args a, int gx) {
    pdl_wait();
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * (blockIdx.y * gridDim.x + blockIdx.x)] = globaltimer_ns();
    const float* x = a.d + (int64_t)blockIdx.y * a.M;
    double ss = 0.0;
    const int64_t n = a.M / VEC;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const FVec<VEC> v = ld_stream<VEC>(x + i * VEC);
        float s = 0.0f;
#pragma unroll
        for (int e = 0; e < VEC; ++e) s = fmaf(v.v[e], v.v[e], s);
        ss += (double)s;
    }
    pdl_launch_dependents();
    l2_finish_sums(ss, a.ws, gx);
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * (blockIdx.y * gridDim.x + blockIdx.x) + 3] = globaltimer_ns();
}

// launch B: out = scale * d / n1 [/ n2] [, adv = clamp(img + out, 0, 1)] -- both normalisations of passes == 2 in one sweep
// (the second norm follows from the first sum, l2_scales): d is read twice and written once per call, whatever `passes`.
template <int VEC, int kU = 4>
__global__ void __launch_bounds__(256) l2_scale_kernel(const L2Args a, int gx) {
    pdl_wait();
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * (blockIdx.y * gridDim.x + blockIdx.x)] = globaltimer_ns();
    const int64_t base = (int64_t)blockIdx.y * a.M;
    const L2Scale sc = l2_scales((float)__ldcg(&a.ws->partials[(size_t)blockIdx.y * (gx + 1) + gx]), a.passes, a.scale);
    const int64_t n = a.M / VEC;
    const bool tail = a.img != nullptr;
    // A CTA walks the sample in chunks of kU x 256 elements; every thread has kU loads in flight, 256 elements apart, so a warp
    // reads kU runs of 512 contiguous bytes out of one 16 KB chunk.  One load per thread and iteration (the loads cannot move
    // above the previous iteration's stores: `out` may alias `d`) left 32 KB in flight per SM: c4 l2_direction 63 -> 55 us
    // with kU = 4 (2: 58 us; profiles/r61/ab_DCT_L2_SCALE_U.log).  The launch with the clamp tail (four streams) does not
    // react (91 us either way), nor does the sum-of-squares launch.
    const int64_t nchunks = (n + kU * 256 - 1) / (kU * 256);
    for (int64_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
        const int64_t i0 = ch * (kU * 256) + threadIdx.x;
        FVec<VEC> v[kU], im[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            const int64_t i = i0 + u * 256;
            if (i < n) {
                v[u] = ld_stream<VEC>(a.d + base + i * VEC);
                if (tail) im[u] = ld_stream<VEC>(a.img + base + i * VEC);
            }
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            const int64_t i = i0 + u * 256;
            if (i < n) {
                const int64_t off = base + i * VEC;
                FVec<VEC> o;
#pragma unroll
                for (int e = 0; e < VEC; ++e) o.v[e] = l2_apply(v[u].v[e], sc);
                st_stream<VEC>(a.out + off, o);
                if (tail) {
                    FVec<VEC> ad;
#pragma unroll
                    for (int e = 0; e < VEC; ++e) ad.v[e] = fminf(fmaxf(im[u].v[e] + o.v[e], 0.0f), 1.0f);
                    st_stream<VEC>(a.adv + off, ad);
                }
            }
        }
    }
    pdl_launch_dependents();
    if (a.trace != nullptr && threadIdx.x == 0) a.trace[kTraceSlots * (blockIdx.y * gridDim.x + blockIdx.x) + 3] = globaltimer_ns();
}

template <int VEC>
__global__ void __launch_bounds__(256) fgsm_kernel(const float* img, const float* grad, float eps, float* adv,
                                                   float* noise, int64_t n) {
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC; i < n; i += (int64_t)gridDim.x * blockDim.x * VEC) {
        FVec<VEC> im = ld_stream<VEC>(img + i), g = ld_stream<VEC>(grad + i), nz, ad;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            float s = (float)((g.v[j] > 0.0f) - (g.v[j] < 0.0f));  // torch.sign: 0 -> 0, NaN -> 0
            nz.v[j] = eps * s;
            ad.v[j] = im.v[j] + nz.v[j];
        }
        st_stream<VEC>(noise + i, nz);
        st_stream<VEC>(adv + i, ad);
    }
}

template <int VEC>
__global__ void __launch_bounds__(256) scale_if_not_one_kernel(float* grad, int64_t n, const float* gscalar) {
    const float g = __ldg(gscalar);
    if (g == 1.0f) return;  // uniform: the whole grid leaves without touching `grad`
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC; i < n; i += (int64_t)gridDim.x * blockDim.x * VEC) {
        FVec<VEC> v = ld_stream<VEC>(grad + i);
#pragma unroll
        for (int j = 0; j < VEC; ++j) v.v[j] *= g;
        st_stream<VEC>(grad + i, v);
    }
}

// bf16 twin: grad[i] = RNE_bf16(float(grad[i]) * g) -- one fp32 multiply of the stored value and one rounding, so a
// gradient the tile pipeline wrote as RNE_bf16(v) ends as RNE_bf16(RNE_bf16(v) * g).  VEC = 8: one 16-byte word per step.
template <int VEC>
__global__ void __launch_bounds__(256) scale_if_not_one_bf16_kernel(__nv_bfloat16* grad, int64_t n, const float* gscalar) {
    const float g = __ldg(gscalar);
    if (g == 1.0f) return;  // uniform: the whole grid leaves without touching `grad`
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC; i < n; i += (int64_t)gridDim.x * blockDim.x * VEC) {
        if constexpr (VEC == 8) {
            uint4 u = __ldcs(reinterpret_cast<const uint4*>(grad + i));
            uint32_t* w = &u.x;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
                const __nv_bfloat162 r = __floats2bfloat162_rn(f.x * g, f.y * g);
                w[j] = *reinterpret_cast<const uint32_t*>(&r);
            }
            __stcs(reinterpret_cast<uint4*>(grad + i), u);
        } else {
            grad[i] = __float2bfloat16_rn(__bfloat162float(grad[i]) * g);
        }
    }
}

static inline unsigned ew_blocks(int64_t n, int vec) {
    int64_t b = (n / vec + 255) / 256;
    if (b < 1) b = 1;
    if (b > 148 * 16) b = 148 * 16;
    return (unsigned)b;
}

}  // namespace dct

using namespace dct;

extern "C" int dct_l2_normalize_f32(const float* d, float* out, int64_t B, int64_t M, int passes, float scale,
                                    const float* img, float* adv, void* workspace, void* stream) {
    if (d == nullptr || out == nullptr || B < 1 || M < 1 || passes < 1 || passes > 2) return DCT_ERR_BAD_ARG;
    if ((img == nullptr) != (adv == nullptr)) return DCT_ERR_BAD_ARG;
    if (!aligned(d, 4) || !aligned(out, 4) || !aligned(img, 4) || !aligned(adv, 4)) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // prefetch on: c2 l2 launches 5.93 -> 5.47 / 9.95 -> 8.64 us (profiles/r30)
    L2Args a{d, out, M, passes, scale, img, adv, static_cast<Workspace*>(workspace), nullptr, 1};
    const bool vec_ok = (M % 4) == 0 && aligned(d, 16) && aligned(out, 16) && aligned(img, 16) && aligned(adv, 16);
    // Which one-launch kernel (measured in the c2 / c3 steps, profiles/r24, r25): samples up to 512 KB -> one cluster of 8
    // CTAs (its exchange stays in distributed shared memory; the cluster-free kernel's tagged words go through an L2 that is
    // busy writing back the previous launch's gradients: 10.6 vs 13.5 us inside the c2 step); 512 KB - 1 MB -> the
    // cluster-free kernel (twice the CTAs of a 16-CTA cluster per sample: c3 step 61.0 vs 64.7 us), then the cluster of 16.
    const int64_t nv8 = (M + (int64_t)kL2Cluster * kL2Threads * 4 - 1) / ((int64_t)kL2Cluster * kL2Threads * 4);
    if (vec_ok && workspace != nullptr && B <= kL2LLSamples && nv8 > kL2MaxVecPerThread) {
        // cluster-free one-launch kernel: cps CTAs of 256 threads per sample, <= 8 float4 per thread, and as many more CTAs
        // (fewer float4 each) as still fit one co-resident wave
        const int64_t nvec = M / 4;
        int64_t cps = (nvec + 256 * 8 - 1) / (256 * 8);
        int nvt = 8;
        while (nvt > 1 && cps * 2 <= kL2LLSlots && B * cps * 2 <= 2 * kSMs && (nvec + cps * 2 * 256 - 1) / (cps * 2 * 256) <= nvt / 2) {
            cps *= 2;
            nvt /= 2;
        }
        if (cps <= kL2LLSlots) {
            cudaError_t e = cudaSuccess;
            bool served;
#define DCT_L2_LL(NVV) (img != nullptr ? l2_ll_try<NVV, true>(a, B, (int)cps, s, e) : l2_ll_try<NVV, false>(a, B, (int)cps, s, e))
            if (nvt == 8) served = DCT_L2_LL(8);
            else if (nvt == 4) served = DCT_L2_LL(4);
            else if (nvt == 2) served = DCT_L2_LL(2);
            else served = DCT_L2_LL(1);
#undef DCT_L2_LL
            if (served) {
                if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
                return check_launch();
            }
        }
    }
    const int64_t per_wave = (int64_t)kL2Cluster * kL2Threads * 4;  // floats covered by one float4 per thread
    const int64_t nv = (M + per_wave - 1) / per_wave;
    const int64_t nv_big = (nv + 1) / 2;   // float4 per thread with a cluster of 16
    if (vec_ok && nv > kL2MaxVecPerThread && nv_big <= kL2MaxVecPerThread && B * kL2ClusterBig <= 0x7fffffff) {
        // 512 KB < sample <= 1 MB (spleen 512 x 512 slices): one cluster of 16 CTAs per sample
        dim3 grid((unsigned)(B * kL2ClusterBig));
        auto go = [&](auto kern) -> cudaError_t {
            // the opt-in is per function and device; setting it again is harmless and costs a host-side table lookup
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e != cudaSuccess) return e;
            return launch_pdl(kern, grid, dim3(kL2Threads), 0, s, a);
        };
        cudaError_t e;
        if (nv_big <= 8) e = img != nullptr ? go(l2_cluster_kernel<8, true, kL2ClusterBig>) : go(l2_cluster_kernel<8, false, kL2ClusterBig>);
        else e = img != nullptr ? go(l2_cluster_kernel<16, true, kL2ClusterBig>) : go(l2_cluster_kernel<16, false, kL2ClusterBig>);
        if (e == cudaSuccess) return check_launch();
        (void)cudaGetLastError();   // cluster of 16 refused on this device / configuration: the grid-wide passes below
    }
    if (vec_ok && nv <= kL2MaxVecPerThread && B * kL2Cluster <= 0x7fffffff) {
        dim3 grid((unsigned)(B * kL2Cluster));
        a.trace = trace_next((int)grid.x);
        cudaError_t e;
#define DCT_L2_GO(NVV) (img != nullptr ? launch_pdl(l2_cluster_kernel<NVV, true>, grid, dim3(kL2Threads), 0, s, a) \
                                       : launch_pdl(l2_cluster_kernel<NVV, false>, grid, dim3(kL2Threads), 0, s, a))
        if (nv <= 1) e = DCT_L2_GO(1);
        else if (nv <= 2) e = DCT_L2_GO(2);
        else if (nv <= 4) e = DCT_L2_GO(4);
        else if (nv <= 8) e = DCT_L2_GO(8);
        else e = DCT_L2_GO(16);
#undef DCT_L2_GO
        if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
        return check_launch();
    }
    if (workspace == nullptr) return DCT_ERR_BAD_ARG;
    if (B > 65535 || B > kMaxPartials / 2) return DCT_ERR_UNSUPPORTED;
    // (Chunking the samples -- a pair of launches per 16 / 32 / 64 MB of `d`, so that the scale launch's read comes out of L2 --
    // was measured and removed: every extra pair of launches costs more in ramp and tail than the L2 hits save: c4 l2_direction
    // 64 -> 144 / 86 / 74 us, l2_radv 90 -> 170 / 115 / 102 us; profiles/r44/ab_DCT_L2_CHUNK_MB.log.)
    // CTAs per sample: about sixteen 256-thread CTAs per SM over the whole grid (two waves), grid-stride loops inside
    // (2 / 4 / 8 / 16 / 32 per SM at c4: l2_direction 63 / 58 / 57 / 57 / 59 us, l2_radv 99 / 94 / 93 / 90 / 91 us; profiles/r65)
    const int vec = vec_ok ? 4 : 1;
    int64_t gx = (kSMs * 16 + B - 1) / B;
    const int64_t need = (M / vec + 255) / 256;
    if (gx > need) gx = need;
    const int64_t cap = kMaxPartials / B - 1;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    const dim3 grid((unsigned)gx, (unsigned)B), block(256);
    L2Args a1 = a, a2 = a;
    a1.trace = trace_next((int)(gx * B));
    cudaError_t e = vec_ok ? launch_pdl(l2_sumsq_kernel<4>, grid, block, 0, s, a1, (int)gx)
                           : launch_pdl(l2_sumsq_kernel<1>, grid, block, 0, s, a1, (int)gx);
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    a2.trace = trace_next((int)(gx * B));
    e = vec_ok ? launch_pdl(l2_scale_kernel<4>, grid, block, 0, s, a2, (int)gx)
               : launch_pdl(l2_scale_kernel<1>, grid, block, 0, s, a2, (int)gx);
    if (e != cudaSuccess) { g_last_cuda_error = e; return DCT_ERR_CUDA; }
    return check_launch();
}

extern "C" int dct_fgsm_f32(const float* img, const float* grad, float eps, float* adv, float* noise, int64_t n,
                            void* stream) {
    if (img == nullptr || grad == nullptr || adv == nullptr || noise == nullptr || n < 1) return DCT_ERR_BAD_ARG;
    if (!aligned(img, 4) || !aligned(grad, 4) || !aligned(adv, 4) || !aligned(noise, 4)) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if ((n % 4) == 0 && aligned(img, 16) && aligned(grad, 16) && aligned(adv, 16) && aligned(noise, 16))
        fgsm_kernel<4><<<ew_blocks(n, 4), 256, 0, s>>>(img, grad, eps, adv, noise, n);
    else
        fgsm_kernel<1><<<ew_blocks(n, 1), 256, 0, s>>>(img, grad, eps, adv, noise, n);
    return check_launch();
}

extern "C" int dct_scale_if_not_one_f32(float* grad, int64_t n, const float* gscalar, void* stream) {
    if (grad == nullptr || gscalar == nullptr || n < 1) return DCT_ERR_BAD_ARG;
    if (!aligned(grad, 4) || !aligned(gscalar, 4)) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if ((n % 4) == 0 && aligned(grad, 16)) scale_if_not_one_kernel<4><<<ew_blocks(n, 4), 256, 0, s>>>(grad, n, gscalar);
    else scale_if_not_one_kernel<1><<<ew_blocks(n, 1), 256, 0, s>>>(grad, n, gscalar);
    return check_launch();
}

extern "C" int dct_scale_if_not_one_bf16(void* grad, int64_t n, const float* gscalar, void* stream) {
    if (grad == nullptr || gscalar == nullptr || n < 1) return DCT_ERR_BAD_ARG;
    if (!aligned(grad, 2) || !aligned(gscalar, 4)) return DCT_ERR_MISALIGNED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    __nv_bfloat16* g = static_cast<__nv_bfloat16*>(grad);
    if ((n % 8) == 0 && aligned(grad, 16)) scale_if_not_one_bf16_kernel<8><<<ew_blocks(n, 8), 256, 0, s>>>(g, n, gscalar);
    else scale_if_not_one_bf16_kernel<1><<<ew_blocks(n, 1), 256, 0, s>>>(g, n, gscalar);
    return check_launch();
}
