// Pieces shared by the exact CUDA-core rankers (eval_topk.cu: AllNeg top-20, recommend.cu: top-K recommendation lists): the
// ranking order, the specified adjacent-pair summation tree and the transposed item tile both score from.
#pragma once
#include "common.cuh"

namespace ngacf {

// order: score descending, item id ascending
__device__ __forceinline__ bool better(float s1, int i1, float s2, int i2) { return s1 > s2 || (s1 == s2 && i1 < i2); }

// 2^L-term adjacent-pair tree evaluated incrementally: `add(d, v)` with d compile-time after unrolling (L = 6: 64-wide rows,
// L = 7: 128-wide rows); the total ends in st[L-1]
template <int L>
struct TreeN {
    float st[L];
    __device__ __forceinline__ void add(int d, float v) {
#pragma unroll
        for (int l = 0; l < L; ++l) {
            if (((d >> l) & 1) == 0) { st[l] = v; return; }
            v = __fadd_rn(st[l], v);
        }
        st[L - 1] = v;   // d == 2^L - 1: v is the total (kept in st[L-1])
    }
};

// item tile of NI items, transposed: It[d][j] = F[U+i0+j][d] (zeros past I); every thread of the block takes part.  A macro, not a
// function: the inlined function gave eval_topk.cu's kernel a different register assignment
#define NGACF_LOAD_ITEM_TILE(W, NI, NT, It, F, U, I, i0, tid)                                       \
    for (int idx = (tid); idx < (NI) * ((W) / 4); idx += (NT)) {                                    \
        int j = idx / ((W) / 4), q = idx % ((W) / 4);                                               \
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);                                                 \
        if ((i0) + j < (I)) v = ld_gather4((F) + (int64_t)((U) + (i0) + j) * (W) + q * 4);          \
        (It)[(q * 4 + 0) * (NI) + j] = v.x; (It)[(q * 4 + 1) * (NI) + j] = v.y;                     \
        (It)[(q * 4 + 2) * (NI) + j] = v.z; (It)[(q * 4 + 3) * (NI) + j] = v.w;                     \
    }

}  // namespace ngacf
