// Shared device helpers for the ngacf_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <mutex>
#include "../../include/ngacf_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "ngacf_b200 kernels are written for sm_100a (B200) only"
#endif

namespace ngacf {

constexpr int D = NGACF_D;
constexpr int CHUNK = NGACF_CHUNK;
constexpr float LRELU_ALPHA = 0.2f;   // SPUIGACF.py:22
constexpr int SCRATCH_STRIDE = D + 8; // per-slot partial: 64 accumulators + up to 8 per-head sums

void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define NGACF_REQUIRE(cond, ...)                       \
    do {                                               \
        if (!(cond)) {                                 \
            ngacf::set_error(__VA_ARGS__);             \
            return NGACF_ERR_INVALID_ARG;              \
        }                                              \
    } while (0)

// dense stage transforms: tcgen05 3xTF32 kernels (transform_tc.cu) unless NGACF_DENSE=ffma selects the CUDA-core kernels
// (kept for parity triage); read once per process
bool dense_on_tensor_cores();
void transform_fwd_tc(const float* Xu, const float* Xi, int apply_elu, const uint64_t* featmask, float scale, const float* const* wtab, int H,
                      int U, int I, float* h, float* s, cudaStream_t st);
void transform_bwd_dx_tc(const float* dh, const float* Zu, const float* Zi, int apply_elu, const uint64_t* featmask, float scale,
                         const float* const* wtab, int H, int U, int I, float* dXu, float* dXi, int accumulate, cudaStream_t st);

void transform_bwd_tc(const float* dh, const float* dS, const float* Xu, const float* Xi, int apply_elu, const uint64_t* featmask, float scale,
                      const float* const* wtab, int H, int U, int I, float* dXu, float* dXi, int accumulate_dx, float* partials,
                      int* nb_u, int* nb_i, cudaStream_t st);

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// cudaFuncSetAttribute is per DEVICE: a process that touches a second GPU must set it there too.  `first()` is true exactly once
// per device (and holds a lock while the caller sets the attributes, so a concurrent first launch cannot overtake them).
struct PerDeviceOnce {
    std::mutex mu;
    unsigned long long done = 0;
    template <class F>
    void run(F&& set_attributes) {
        int dev = 0;
        cudaGetDevice(&dev);
        const unsigned long long bit = 1ull << (dev & 63);
        std::lock_guard<std::mutex> lock(mu);
        if (done & bit) return;
        set_attributes();
        done |= bit;
    }
};

// ---------------------------------------------------------------------------------------------
// loads / stores with cache intent: gathered tables go through L1 (popular rows hit), streamed
// arrays do not allocate in L1.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ld_gather4(const float* p) {   // read-only path, L1 allocating
    return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ float4 ld_stream4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ int ld_stream_i32(const int* p) {
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream4(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 ld_cg4(const float* p) {   // L2-coherent (other SMs' writes in this launch)
    return __ldcg(reinterpret_cast<const float4*>(p));
}

// ELU.  expm1 for z <= 0 without libdevice's ~50-instruction expm1f (it was 75% of the dense kernels' instruction stream,
// profiles/r1e_dense_tc_ncu.txt): Taylor to z^6 on (-0.25, 0] (relative error < 6e-8), exp(z) - 1 below (|expm1| >= 0.22 there,
// so __expf's ~2^-22 absolute error stays < 1.2e-6 relative).  Forward and backward use this one definition.
__device__ __forceinline__ float elu(float z) {
    float p = fmaf(z, 1.f / 720.f, 1.f / 120.f);
    p = fmaf(p, z, 1.f / 24.f);
    p = fmaf(p, z, 1.f / 6.f);
    p = fmaf(p, z, 0.5f);
    p = fmaf(p, z, 1.f);
    p *= z;
    const float e = __expf(z) - 1.f;
    const float r = z > -0.25f ? p : e;
    return z > 0.f ? z : r;
}
__device__ __forceinline__ float elu_grad(float z) { return z > 0.f ? 1.f : __expf(z); }

// e = exp(-LeakyReLU(x)); the same expression is used by forward and backward so the recomputed
// weight is bit-identical to the one the forward normalised with.
__device__ __forceinline__ float edge_weight(float x) {
    float l = x > 0.f ? x : LRELU_ALPHA * x;
    return __expf(-l);
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (same constants/rounds as oracle/port.py:philox4x32_10)
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                       uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__host__ __device__ __forceinline__ uint32_t keep_threshold(float droprate) {
    double t = floor((1.0 - (double)droprate) * 65536.0 + 0.5);
    if (t < 0) t = 0;
    if (t > 65536.0) t = 65536.0;
    return (uint32_t)t;
}

// 16-lane group helpers: a "group" is one half of a warp; the two halves may diverge.
__device__ __forceinline__ unsigned group_mask() { return (threadIdx.x & 16) ? 0xFFFF0000u : 0x0000FFFFu; }

template <int H>
__device__ __forceinline__ float head_reduce(float v, unsigned mask) {
    // sum over the lanes that share a head: H=8 -> lane pairs, H=1 -> all 16 lanes (adjacent-pair tree)
    v += __shfl_xor_sync(mask, v, 1, 16);
    if (H == 1) {
        v += __shfl_xor_sync(mask, v, 2, 16);
        v += __shfl_xor_sync(mask, v, 4, 16);
        v += __shfl_xor_sync(mask, v, 8, 16);
    }
    return v;
}

// Issue fence: an empty asm that names one register of each of eight loaded vectors.  ptxas must have all eight loads issued
// before it and may not start consuming them earlier -- without it the consumers are interleaved with the loads (two or three
// registers are recycled), and since issue is in order every consumer stalls the loads behind it: eight independent gathers
// become a chain of three or four round trips.  Matters for the kernels that run few rows (latency-, not throughput-bound).
#define NGACF_ISSUE_FENCE8(v)                                                                                                   \
    asm volatile("" : "+f"((v)[0].x), "+f"((v)[1].x), "+f"((v)[2].x), "+f"((v)[3].x), "+f"((v)[4].x), "+f"((v)[5].x), \
                 "+f"((v)[6].x), "+f"((v)[7].x))
#define NGACF_ISSUE_FENCE4(v) asm volatile("" : "+f"((v)[0].x), "+f"((v)[1].x), "+f"((v)[2].x), "+f"((v)[3].x))

// ---------------------------------------------------------------------------------------------
// long rows (> CHUNK edges) are split into chunk tasks; every chunk writes its partial (64 accumulators + NSUM per-head sums) to
// its slot, and the group that arrives LAST sums the slots in slot order (deterministic, no atomics on data) and continues with
// the totals.  Returns false for every other group.  The counter is re-armed for the next launch by the last arriver.
// ---------------------------------------------------------------------------------------------
// release / acquire fence of the partial-sum hand-over (message passing: data stores -> fence -> counter atomic on the writer,
// counter atomic -> fence -> data loads (ld.cg) on the reader).  __threadfence() is the sequentially consistent fence
// (MEMBAR.SC.GPU + L1 invalidate), which this pattern does not need.
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

// FAST: eight slots in flight (32 more registers) -- for the kernels that run few rows, where this sum is the critical path; the
// throughput-bound full-graph kernels keep the plain loop (the extra registers cost them a resident CTA per SM: measured
// +8..18 % on the stage-0 kernels), their long rows are scheduled first and the sum hides behind the rest of the grid.
template <int H, int NSUM, bool FAST = false>
__device__ __forceinline__ bool long_row_combine(int lid, int chunk, const int* __restrict__ long_first_slot, int* long_counter,
                                                 float* scratch, int lane16, unsigned gm, float4& acc, float (&sums)[NSUM]) {
    const int head = H == 8 ? (lane16 >> 1) : 0;
    const int first = long_first_slot[lid];
    const int nslots = long_first_slot[lid + 1] - first;
    float* slot = scratch + (size_t)(first + chunk) * SCRATCH_STRIDE;
    *reinterpret_cast<float4*>(slot + lane16 * 4) = acc;
    // per-head scalars: NSUM values per head at [64 + j*H + head]: the slot has 8 floats of room => NSUM*H <= 8
    if ((H == 8 && (lane16 & 1) == 0) || (H == 1 && lane16 == 0)) {
#pragma unroll
        for (int j = 0; j < NSUM; ++j) slot[D + j * H + head] = sums[j];
    }
    fence_acq_rel_gpu();
    __syncwarp(gm);                          // every lane's partial is fenced before lane 0 publishes
    int old = 0;
    if (lane16 == 0) old = atomicAdd(long_counter + lid, 1);
    old = __shfl_sync(gm, old, 0, 16);
    if (old != nslots - 1) return false;
    fence_acq_rel_gpu();
    if constexpr (!FAST) {
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        float ts[NSUM];
#pragma unroll
        for (int j = 0; j < NSUM; ++j) ts[j] = 0.f;
        for (int c = 0; c < nslots; ++c) {
            const float* sl = scratch + (size_t)(first + c) * SCRATCH_STRIDE;
            float4 v = ld_cg4(sl + lane16 * 4);
            t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
#pragma unroll
            for (int j = 0; j < NSUM; ++j) ts[j] += __ldcg(sl + D + j * H + head);
        }
        acc = t;
#pragma unroll
        for (int j = 0; j < NSUM; ++j) sums[j] = ts[j];
    } else {
        // fixed summation order: four interleaved partial sums (slots c, c+4, ...), then ((0+1)+(2+3)).  Eight slots are in flight
        // at a time: the most popular item of the Gowalla-shape graph has 111 slots, and a dependent chain of 111 L2 round trips was
        // the critical path of every kernel that runs few rows (the pruned output stage)
        float4 t4[4];
        float ts4[4][NSUM];
    #pragma unroll
        for (int q = 0; q < 4; ++q) {
            t4[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    #pragma unroll
            for (int j = 0; j < NSUM; ++j) ts4[q][j] = 0.f;
        }
        for (int c0 = 0; c0 < nslots; c0 += 8) {
            float4 v[8];
            float sv[8][NSUM];
    #pragma unroll
            for (int q = 0; q < 8; ++q) {
                const bool in = c0 + q < nslots;
                const float* sl = scratch + (size_t)(first + (in ? c0 + q : 0)) * SCRATCH_STRIDE;
                v[q] = in ? ld_cg4(sl + lane16 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    #pragma unroll
                for (int j = 0; j < NSUM; ++j) sv[q][j] = in ? __ldcg(sl + D + j * H + head) : 0.f;
            }
            NGACF_ISSUE_FENCE8(v);
    #pragma unroll
            for (int q = 0; q < 8; ++q) {
                float4& a = t4[q & 3];
                a.x += v[q].x; a.y += v[q].y; a.z += v[q].z; a.w += v[q].w;
    #pragma unroll
                for (int j = 0; j < NSUM; ++j) ts4[q & 3][j] += sv[q][j];
            }
        }
        float4 t;
        t.x = (t4[0].x + t4[1].x) + (t4[2].x + t4[3].x);
        t.y = (t4[0].y + t4[1].y) + (t4[2].y + t4[3].y);
        t.z = (t4[0].z + t4[1].z) + (t4[2].z + t4[3].z);
        t.w = (t4[0].w + t4[1].w) + (t4[2].w + t4[3].w);
        acc = t;
    #pragma unroll
        for (int j = 0; j < NSUM; ++j) sums[j] = (ts4[0][j] + ts4[1][j]) + (ts4[2][j] + ts4[3][j]);
    }
    if (lane16 == 0) long_counter[lid] = 0;    // re-arm for the next launch
    return true;
}

// the same hand-over for W-wide single-head rows (W = 128: lane l owns columns W/16*l .. W/16*(l+1)-1, V float4 each); the slot
// stride is W + 8 floats.  The 64-wide kernels keep long_row_combine above.
template <int W, int NSUM>
__device__ __forceinline__ bool long_row_combine_wide(int lid, int chunk, const int* __restrict__ long_first_slot, int* long_counter,
                                                      float* scratch, int lane16, unsigned gm, float4 (&acc)[W / 64], float (&sums)[NSUM]) {
    constexpr int V = W / 64, STRIDE = W + 8;
    static_assert(NSUM <= 8, "per-slot room for 8 scalars");
    const int first = long_first_slot[lid];
    const int nslots = long_first_slot[lid + 1] - first;
    float* slot = scratch + (size_t)(first + chunk) * STRIDE;
#pragma unroll
    for (int v = 0; v < V; ++v) *reinterpret_cast<float4*>(slot + lane16 * 4 * V + 4 * v) = acc[v];
    if (lane16 == 0) {
#pragma unroll
        for (int j = 0; j < NSUM; ++j) slot[W + j] = sums[j];
    }
    fence_acq_rel_gpu();
    __syncwarp(gm);
    int old = 0;
    if (lane16 == 0) old = atomicAdd(long_counter + lid, 1);
    old = __shfl_sync(gm, old, 0, 16);
    if (old != nslots - 1) return false;
    fence_acq_rel_gpu();
    float4 t[V];
    float ts[NSUM];
#pragma unroll
    for (int v = 0; v < V; ++v) t[v] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < NSUM; ++j) ts[j] = 0.f;
    for (int c = 0; c < nslots; ++c) {
        const float* sl = scratch + (size_t)(first + c) * STRIDE;
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float4 x = ld_cg4(sl + lane16 * 4 * V + 4 * v);
            t[v].x += x.x; t[v].y += x.y; t[v].z += x.z; t[v].w += x.w;
        }
#pragma unroll
        for (int j = 0; j < NSUM; ++j) ts[j] += __ldcg(sl + W + j);
    }
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = t[v];
#pragma unroll
    for (int j = 0; j < NSUM; ++j) sums[j] = ts[j];
    if (lane16 == 0) long_counter[lid] = 0;
    return true;
}

// row widths of the width-generic (`_w`) entry points: 64 (every stage of the 64-wide models) and 128 (embedSize 128: the input
// of the first stage and the output of the single-head last stage)
static inline bool width_supported(int w) { return w == 64 || w == 128; }

// "active" rows of a pruned last stage (ngacf_mark_active): node n is active iff stamp[n] == value of this propagation
__device__ __forceinline__ int active_value(int val, const int64_t* __restrict__ val_dev) {
    return val_dev ? val + (int)*val_dev : val;
}

}  // namespace ngacf
