// Forward propagation kernels of one SpUIGAT stage (all heads at once):
//   dropout masks (Philox), dense transform h = drop(act(X)) W with the rank-1 logit scalars s,
//   fused edge-softmax + neighbour aggregation over the unified node adjacency.
// Reference: graphattention/SPUIGACF.py:207-215 (SpUIGAT.forward), :340-400 (layer forward).
#include "common.cuh"

namespace ngacf {

// ------------------------------------------------------------------------------------------------
// dropout masks
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t decisions8(const uint32_t w[4], uint32_t thr) {
    // eight 16-bit fields, low half first (oracle/port.py:_decisions)
    uint32_t bits = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        uint32_t r16 = (w[j >> 1] >> (16 * (j & 1))) & 0xFFFFu;
        bits |= (uint32_t)(r16 < thr) << j;
    }
    return bits;
}

__global__ void feature_mask_kernel(uint64_t* __restrict__ out, int64_t N, uint32_t k0, uint32_t k1, uint32_t call,
                                    const int64_t* __restrict__ call_dev, uint32_t site, uint32_t thr) {
    if (call_dev) call += (uint32_t)*call_dev;
    // one thread per (row, 8-column group); 8 consecutive threads assemble a row's 64-bit word
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t n = t >> 3;
    int c = (int)(t & 7);
    uint32_t bits = 0;
    if (n < N) {
        uint64_t idx = (uint64_t)n * 8u + (uint64_t)c;
        uint32_t w[4];
        philox4x32_10((uint32_t)idx, (uint32_t)(idx >> 32), site, call, k0, k1, w);
        bits = decisions8(w, thr);
    }
    uint64_t word = (uint64_t)bits << (8 * c);
    // OR-reduce over the 8 threads of the row (aligned 8-lane segments)
    word |= __shfl_xor_sync(0xffffffffu, word, 1);
    word |= __shfl_xor_sync(0xffffffffu, word, 2);
    word |= __shfl_xor_sync(0xffffffffu, word, 4);
    if (n < N && c == 0) out[n] = word;
}

__global__ void edge_mask_kernel(uint8_t* __restrict__ out, int64_t E, int H, uint32_t k0, uint32_t k1, uint32_t call,
                                 const int64_t* __restrict__ call_dev, uint32_t site, uint32_t thr) {
    if (call_dev) call += (uint32_t)*call_dev;
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    uint32_t w[4];
    philox4x32_10((uint32_t)e, (uint32_t)((uint64_t)e >> 32), site, call, k0, k1, w);
    uint32_t bits = decisions8(w, thr);
    out[e] = (uint8_t)(bits & ((1u << H) - 1u));
}

// every mask of one propagation in a single launch: the grid is the concatenation of the per-stage
// feature blocks and edge blocks (same per-element streams as the two kernels above)
constexpr int MASK_MAX_STAGES = 8;
struct MaskPlan {
    uint64_t* feat[MASK_MAX_STAGES];
    uint8_t* edge[MASK_MAX_STAGES];
    int heads[MASK_MAX_STAGES];
    int wshift[MASK_MAX_STAGES];    // log2(input width / 64): a row has 8 << wshift Philox counters and 1 << wshift words
    int S;
    int feat_blocks, edge_blocks;   // per stage
};

__global__ void __launch_bounds__(256) dropout_masks_kernel(MaskPlan plan, int64_t N, int64_t E, uint32_t k0, uint32_t k1, uint32_t call,
                                                            const int64_t* __restrict__ call_dev, uint32_t thr) {
    if (call_dev) call += (uint32_t)*call_dev;
    int b = blockIdx.x;
    const int per_stage = plan.feat_blocks + plan.edge_blocks;
    const int site = b / per_stage;     // = stage; Philox sites are 2*stage (features) and 2*stage+1 (edges)
    b -= site * per_stage;
    uint32_t w[4];
    if (b < plan.feat_blocks) {
        // thread t = Philox counter t = (row n, 8-column group c) with t = n * (8 << wshift) + c; word t/8 of the mask holds the
        // decisions of counters 8*(t/8) .. 8*(t/8)+7 (a 64-wide row: word n, counters 8n .. 8n+7)
        const int64_t t = (int64_t)b * 256 + threadIdx.x;
        const bool in = t < (N << (3 + plan.wshift[site]));
        const int c = (int)(t & 7);
        uint32_t bits = 0;
        if (in) {
            const uint64_t idx = (uint64_t)t;
            philox4x32_10((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)site * 2u, call, k0, k1, w);
            bits = decisions8(w, thr);
        }
        uint64_t word = (uint64_t)bits << (8 * c);
        word |= __shfl_xor_sync(0xffffffffu, word, 1);
        word |= __shfl_xor_sync(0xffffffffu, word, 2);
        word |= __shfl_xor_sync(0xffffffffu, word, 4);
        if (in && c == 0) plan.feat[site][t >> 3] = word;
    } else {
        const int64_t e = (int64_t)(b - plan.feat_blocks) * 256 + threadIdx.x;
        if (e >= E) return;
        philox4x32_10((uint32_t)e, (uint32_t)((uint64_t)e >> 32), (uint32_t)site * 2u + 1u, call, k0, k1, w);
        plan.edge[site][e] = (uint8_t)(decisions8(w, thr) & ((1u << plan.heads[site]) - 1u));
    }
}

// the same streams restricted to two node ranges and one edge range, written at their GLOBAL positions (multi-GPU: a rank
// only needs the masks of the rows it transforms and of the edges it owns)
struct MaskRanges { int64_t fa0, fb0, fa1, fb1, e0, e1; int fb_blocks0, fb_blocks1, e_blocks; };

__global__ void __launch_bounds__(256) dropout_masks_ranges_kernel(MaskPlan plan, MaskRanges r, uint32_t k0, uint32_t k1, uint32_t call,
                                                                   const int64_t* __restrict__ call_dev, uint32_t thr) {
    if (call_dev) call += (uint32_t)*call_dev;
    int b = blockIdx.x;
    const int per_stage = r.fb_blocks0 + r.fb_blocks1 + r.e_blocks;
    const int site = b / per_stage;
    b -= site * per_stage;
    uint32_t w[4];
    if (b < r.fb_blocks0 + r.fb_blocks1) {
        const bool second = b >= r.fb_blocks0;
        const int64_t t = (int64_t)(second ? b - r.fb_blocks0 : b) * 256 + threadIdx.x;
        const int64_t n = (second ? r.fa1 : r.fa0) + (t >> 3);
        const int64_t hi = second ? r.fb1 : r.fb0;
        const int c = (int)(t & 7);
        uint32_t bits = 0;
        if (n < hi) {
            const uint64_t idx = (uint64_t)n * 8u + (uint64_t)c;
            philox4x32_10((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)site * 2u, call, k0, k1, w);
            bits = decisions8(w, thr);
        }
        uint64_t word = (uint64_t)bits << (8 * c);
        word |= __shfl_xor_sync(0xffffffffu, word, 1);
        word |= __shfl_xor_sync(0xffffffffu, word, 2);
        word |= __shfl_xor_sync(0xffffffffu, word, 4);
        if (n < hi && c == 0) plan.feat[site][n] = word;
    } else {
        const int64_t e = r.e0 + (int64_t)(b - r.fb_blocks0 - r.fb_blocks1) * 256 + threadIdx.x;
        if (e >= r.e1) return;
        philox4x32_10((uint32_t)e, (uint32_t)((uint64_t)e >> 32), (uint32_t)site * 2u + 1u, call, k0, k1, w);
        plan.edge[site][e] = (uint8_t)(decisions8(w, thr) & ((1u << plan.heads[site]) - 1u));
    }
}

// ------------------------------------------------------------------------------------------------
// dense transform: h = Xd @ Wcat, s = per-head a . h
// block = 256 threads, tile = TF_TM(DOUT) rows of one side; thread = TF_TM/16 rows x 4 columns of every 64-column group.
// (DIN, DOUT) = (64, 64) for every stage of the 64-wide models; embedSize 128 adds (128, 64) (first stage) and (64, 128) (last).
// ------------------------------------------------------------------------------------------------
template <int DOUT> __host__ __device__ constexpr int tf_tm() { return 128 * 64 / DOUT; }          // 8 rows x 4 columns per thread at DOUT = 64
template <int DIN, int DOUT> __host__ __device__ constexpr size_t tf_smem() { return (size_t)(DIN * DOUT + tf_tm<DOUT>() * (DIN + 4) + DOUT) * sizeof(float); }
constexpr int TF_TM = 128;
constexpr size_t TF_SMEM = tf_smem<64, 64>();

// load the H per-head (DIN,DH) matrices of one side into Ws[k][c], c = head*DH + j
template <int DIN, int DOUT>
__device__ __forceinline__ void load_wcat(float* Ws, const float* const* wptr, int H) {
    const int DH = DOUT / H;
    // 16-byte loads: every (DIN,DH) head matrix is contiguous and DH is a multiple of 4
    for (int idx = threadIdx.x; idx < DIN * DOUT / 4; idx += blockDim.x) {
        const int k = idx / (DOUT / 4), c = (idx % (DOUT / 4)) * 4;
        const float4 v = __ldg(reinterpret_cast<const float4*>(wptr[c / DH] + k * DH + (c % DH)));
        *reinterpret_cast<float4*>(Ws + k * DOUT + c) = v;
    }
}

// stage-input element: ELU on load for stage > 0, then dropout keep-bit and 1/(1-p); the mask has DIN/64 words per row
template <int DIN>
__device__ __forceinline__ float4 load_input4(const float* __restrict__ X, int64_t row, int q, bool apply_elu,
                                              const uint64_t* __restrict__ featmask, int64_t node, float scale) {
    float4 v = ld_stream4(X + row * DIN + q * 4);
    if (apply_elu) { v.x = elu(v.x); v.y = elu(v.y); v.z = elu(v.z); v.w = elu(v.w); }
    if (featmask) {
        uint32_t m = (uint32_t)(featmask[node * (DIN / 64) + (q >> 4)] >> ((q & 15) * 4)) & 0xFu;
        v.x = (m & 1u) ? v.x * scale : 0.f;
        v.y = (m & 2u) ? v.y * scale : 0.f;
        v.z = (m & 4u) ? v.z * scale : 0.f;
        v.w = (m & 8u) ? v.w * scale : 0.f;
    }
    return v;
}

template <int H, int DIN, int DOUT>
__global__ void __launch_bounds__(256, 4) transform_fwd_kernel(const float* __restrict__ Xu, const float* __restrict__ Xi, int apply_elu,
                                                            const uint64_t* __restrict__ featmask, float scale,
                                                            const float* const* __restrict__ wtab, int U, int I, int tiles_u,
                                                            float* __restrict__ h, float* __restrict__ s) {
    constexpr int TM = tf_tm<DOUT>(), XS = DIN + 4, RI = TM / 16, NC = DOUT / 64;
    extern __shared__ __align__(16) float smem[];
    float* Ws = smem;                    // [DIN][DOUT]
    float* Xs = smem + DIN * DOUT;       // [TM][DIN+4]
    float* av = Xs + TM * XS;            // [DOUT]
    constexpr int DH = DOUT / H;
    const bool item_side = (int)blockIdx.x >= tiles_u;
    const int tile = item_side ? blockIdx.x - tiles_u : blockIdx.x;
    const int rows_side = item_side ? I : U;
    const float* X = item_side ? Xi : Xu;
    const int64_t node0 = (item_side ? (int64_t)U : 0) + (int64_t)tile * TM;
    const int row0 = tile * TM;
    const int nrows = min(TM, rows_side - row0);

    load_wcat<DIN, DOUT>(Ws, wtab + (item_side ? H : 0), H);
    for (int c = threadIdx.x; c < DOUT; c += 256) {
        int k = c / DH, j = c % DH;
        av[c] = __ldg(wtab[2 * H + k] + (item_side ? DH : 0) + j);
    }
    for (int idx = threadIdx.x; idx < TM * (DIN / 4); idx += 256) {
        int r = idx / (DIN / 4), q = idx % (DIN / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < nrows) v = load_input4<DIN>(X, row0 + r, q, apply_elu != 0, featmask, node0 + r, scale);
        *reinterpret_cast<float4*>(Xs + r * XS + q * 4) = v;
    }
    __syncthreads();

    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[RI][NC][4];
#pragma unroll
    for (int i = 0; i < RI; ++i)
#pragma unroll
        for (int n = 0; n < NC; ++n) { acc[i][n][0] = acc[i][n][1] = acc[i][n][2] = acc[i][n][3] = 0.f; }
#pragma unroll 4
    for (int k4 = 0; k4 < DIN / 4; ++k4) {
        float4 w0[NC], w1[NC], w2[NC], w3[NC];
#pragma unroll
        for (int n = 0; n < NC; ++n) {
            w0[n] = *reinterpret_cast<const float4*>(Ws + (k4 * 4 + 0) * DOUT + 64 * n + tx * 4);
            w1[n] = *reinterpret_cast<const float4*>(Ws + (k4 * 4 + 1) * DOUT + 64 * n + tx * 4);
            w2[n] = *reinterpret_cast<const float4*>(Ws + (k4 * 4 + 2) * DOUT + 64 * n + tx * 4);
            w3[n] = *reinterpret_cast<const float4*>(Ws + (k4 * 4 + 3) * DOUT + 64 * n + tx * 4);
        }
#pragma unroll
        for (int i = 0; i < RI; ++i) {
            float4 x = *reinterpret_cast<const float4*>(Xs + (ty + 16 * i) * XS + k4 * 4);
#pragma unroll
            for (int n = 0; n < NC; ++n) {
                float* a = acc[i][n];
                a[0] = fmaf(x.x, w0[n].x, a[0]); a[1] = fmaf(x.x, w0[n].y, a[1]);
                a[2] = fmaf(x.x, w0[n].z, a[2]); a[3] = fmaf(x.x, w0[n].w, a[3]);
                a[0] = fmaf(x.y, w1[n].x, a[0]); a[1] = fmaf(x.y, w1[n].y, a[1]);
                a[2] = fmaf(x.y, w1[n].z, a[2]); a[3] = fmaf(x.y, w1[n].w, a[3]);
                a[0] = fmaf(x.z, w2[n].x, a[0]); a[1] = fmaf(x.z, w2[n].y, a[1]);
                a[2] = fmaf(x.z, w2[n].z, a[2]); a[3] = fmaf(x.z, w2[n].w, a[3]);
                a[0] = fmaf(x.w, w3[n].x, a[0]); a[1] = fmaf(x.w, w3[n].y, a[1]);
                a[2] = fmaf(x.w, w3[n].z, a[2]); a[3] = fmaf(x.w, w3[n].w, a[3]);
            }
        }
    }
    float4 a4[NC];
#pragma unroll
    for (int n = 0; n < NC; ++n) a4[n] = *reinterpret_cast<const float4*>(av + 64 * n + tx * 4);
    const unsigned gm = group_mask();
#pragma unroll
    for (int i = 0; i < RI; ++i) {
        int r = ty + 16 * i;
        float part = acc[i][0][0] * a4[0].x + acc[i][0][1] * a4[0].y + acc[i][0][2] * a4[0].z + acc[i][0][3] * a4[0].w;
#pragma unroll
        for (int n = 1; n < NC; ++n)
            part += acc[i][n][0] * a4[n].x + acc[i][n][1] * a4[n].y + acc[i][n][2] * a4[n].z + acc[i][n][3] * a4[n].w;
        part = head_reduce<H>(part, gm);     // every thread of the warp executes the shuffles
        if (r < nrows) {
            int64_t node = node0 + r;
#pragma unroll
            for (int n = 0; n < NC; ++n)
                st_stream4(h + node * DOUT + 64 * n + tx * 4, make_float4(acc[i][n][0], acc[i][n][1], acc[i][n][2], acc[i][n][3]));
            if (H == 8) { if ((tx & 1) == 0) s[node * 8 + (tx >> 1)] = part; }
            else        { if (tx == 0) s[node] = part; }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// fused edge softmax + aggregation.  One 16-lane group per task (a row, or a <=128-edge chunk of a
// long row); lane l owns columns 4l..4l+3 (16-byte vector loads of the gathered rows).
// ------------------------------------------------------------------------------------------------
template <int H>
__device__ __forceinline__ int lane_head(int lane16) { return H == 8 ? (lane16 >> 1) : 0; }

// body of one task; the kernels below call it for task t = group index (every row) or for the tasks of a compacted list
// LAT: latency-optimised variant for launches that run few rows (the pruned output stage)
template <int H, bool DROP, bool PARTIAL, bool LAT = false>
__device__ __forceinline__ void aggregate_task(const int t, const int4* __restrict__ tasks, const int* __restrict__ adj_ptr,
                                               const int* __restrict__ adj_idx, const int* __restrict__ adj_eid,
                                               const int* __restrict__ long_first_slot, int* long_counter, float* scratch,
                                               const float* __restrict__ h, const float* __restrict__ s,
                                               const uint8_t* __restrict__ edgemask, float scale,
                                               float* __restrict__ Z, float* __restrict__ norm, int partial_from) {
    const int lane16 = threadIdx.x & 15;
    const unsigned gm = group_mask();
    const int head = lane_head<H>(lane16);
    const int4 tk = __ldg(tasks + t);
    const int node = tk.x, beg = tk.y, end = tk.z, lid = tk.w;
    const float sn = __ldg(s + (int64_t)node * H + head);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float rs = 0.f;
    if constexpr (H == 1) {
        // One logit per edge: lane l owns edge base+l of the batch and computes its weight ONCE (before, all 16 lanes recomputed
        // every weight: ~30 instructions per visit, the kernel was issue-bound at 63 %); the visit loop is two shuffles, one
        // 16-byte gather and four FMAs.  The adjacency slice, logit and mask byte of batch b+1 are requested during batch b.
        // three-stage software pipeline (issue is in order: nothing the visit loop needs may still be in flight when a batch
        // starts): at the top of batch b the adjacency slice of b+2 and the logits / mask bytes of b+1 are requested, the weights
        // of b come from loads issued a whole batch earlier
        float rs_l = 0.f, s_c = 0.f;
        int m_c = 0, m_1 = 0, eid_1 = 0;
        unsigned mk_c = 1u;
        if (beg + lane16 < end) {
            m_c = ld_stream_i32(adj_idx + beg + lane16);
            if (DROP) mk_c = edgemask[ld_stream_i32(adj_eid + beg + lane16)];
        }
        if (beg + 16 + lane16 < end) {
            m_1 = ld_stream_i32(adj_idx + beg + 16 + lane16);
            if (DROP) eid_1 = ld_stream_i32(adj_eid + beg + 16 + lane16);
        }
        if (beg + lane16 < end) s_c = __ldg(s + m_c);
        for (int base = beg; base < end; base += 16) {
            const int i1x = base + 16 + lane16, i2x = base + 32 + lane16;
            int m_2 = 0, eid_2 = 0;
            float s_1 = 0.f;
            unsigned mk_1 = 1u;
            if (i2x < end) {
                m_2 = ld_stream_i32(adj_idx + i2x);
                if (DROP) eid_2 = ld_stream_i32(adj_eid + i2x);
            }
            if (i1x < end) {
                s_1 = __ldg(s + m_1);
                if (DROP) mk_1 = edgemask[eid_1];
            }
            const float w_l = base + lane16 < end ? edge_weight(sn + s_c) : 0.f;
            rs_l += w_l;
            const float wd_l = DROP ? ((mk_c & 1u) ? w_l * scale : 0.f) : w_l;
            const int cnt = min(16, end - base);
            if constexpr (LAT) {
                // eight row gathers in flight before the first is consumed (NGACF_ISSUE_FENCE8); predicated loads for the tail
                for (int j0 = 0; j0 < cnt; j0 += 8) {
                    float4 hm[8];
                    float wd[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const int j = (j0 + q) & 15;
                        const int m = __shfl_sync(gm, m_c, j, 16);
                        wd[q] = __shfl_sync(gm, wd_l, j, 16);
                        hm[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (j0 + q < cnt) hm[q] = ld_gather4(h + (int64_t)m * D + lane16 * 4);
                        else wd[q] = 0.f;
                    }
                    NGACF_ISSUE_FENCE8(hm);
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        acc.x = fmaf(wd[q], hm[q].x, acc.x); acc.y = fmaf(wd[q], hm[q].y, acc.y);
                        acc.z = fmaf(wd[q], hm[q].z, acc.z); acc.w = fmaf(wd[q], hm[q].w, acc.w);
                    }
                }
            } else {
#pragma unroll 8
                for (int j = 0; j < cnt; ++j) {
                    const int m = __shfl_sync(gm, m_c, j, 16);
                    const float wd = __shfl_sync(gm, wd_l, j, 16);
                    const float4 hm = ld_gather4(h + (int64_t)m * D + lane16 * 4);
                    acc.x = fmaf(wd, hm.x, acc.x); acc.y = fmaf(wd, hm.y, acc.y);
                    acc.z = fmaf(wd, hm.z, acc.z); acc.w = fmaf(wd, hm.w, acc.w);
                }
            }
            m_c = m_1; m_1 = m_2; eid_1 = eid_2; s_c = s_1; mk_c = mk_1;
        }
        rs_l += __shfl_xor_sync(gm, rs_l, 1, 16);
        rs_l += __shfl_xor_sync(gm, rs_l, 2, 16);
        rs_l += __shfl_xor_sync(gm, rs_l, 4, 16);
        rs_l += __shfl_xor_sync(gm, rs_l, 8, 16);
        rs = rs_l;
    } else {
        for (int base = beg; base < end; base += 16) {
            const int idx = base + lane16;
            int m_l = 0;
            unsigned mk_l = 0xFFu;
            if (idx < end) {
                m_l = ld_stream_i32(adj_idx + idx);
                if (DROP) mk_l = edgemask[ld_stream_i32(adj_eid + idx)];
            }
            const int cnt = min(16, end - base);
#pragma unroll 4
            for (int j = 0; j < cnt; ++j) {
                const int m = __shfl_sync(gm, m_l, j, 16);
                const float sm = __ldg(s + (int64_t)m * H + head);
                const float4 hm = ld_gather4(h + (int64_t)m * D + lane16 * 4);
                const float w = edge_weight(sn + sm);
                rs += w;
                float wd = w;
                if (DROP) {
                    const unsigned mk = __shfl_sync(gm, mk_l, j, 16);
                    wd = ((mk >> head) & 1u) ? w * scale : 0.f;
                }
                acc.x = fmaf(wd, hm.x, acc.x); acc.y = fmaf(wd, hm.y, acc.y);
                acc.z = fmaf(wd, hm.z, acc.z); acc.w = fmaf(wd, hm.w, acc.w);
            }
        }
    }
    if (lid >= 0) {
        float sums[1] = {rs};
        const int chunk = (beg - __ldg(adj_ptr + node)) / CHUNK;
        if (!long_row_combine<H, 1, LAT>(lid, chunk, long_first_slot, long_counter, scratch, lane16, gm, acc, sums)) return;
        rs = sums[0];
    }
    if (PARTIAL && t >= partial_from) {
        // multi-GPU: this rank only holds a slice of the row's edges -> emit the raw partial sums; they are summed
        // across ranks (NCCL) and normalised by aggregate_finalize_kernel
        st_stream4(Z + (int64_t)node * D + lane16 * 4, acc);
        if (H == 8) { if ((lane16 & 1) == 0) norm[(int64_t)node * 8 + head] = rs; }
        else        { if (lane16 == 0) norm[node] = rs; }
        return;
    }
    // epilogue: Z = h + agg / norm, NaN -> 0 for isolated nodes (SPUIGACF.py:383,388-390)
    const float inv = rs != 0.f ? 1.0f / rs : 0.f;
    const float4 hn = ld_stream4(h + (int64_t)node * D + lane16 * 4);
    st_stream4(Z + (int64_t)node * D + lane16 * 4,
               make_float4(fmaf(acc.x, inv, hn.x), fmaf(acc.y, inv, hn.y), fmaf(acc.z, inv, hn.z), fmaf(acc.w, inv, hn.w)));
    if (H == 8) { if ((lane16 & 1) == 0) norm[(int64_t)node * 8 + head] = rs; }
    else        { if (lane16 == 0) norm[node] = rs; }
}

template <int H, bool DROP, bool PARTIAL>
__global__ void __launch_bounds__(256) aggregate_fwd_kernel(const int4* __restrict__ tasks, int T, const int* __restrict__ adj_ptr,
                                                            const int* __restrict__ adj_idx, const int* __restrict__ adj_eid,
                                                            const int* __restrict__ long_first_slot, int* long_counter, float* scratch,
                                                            const float* __restrict__ h, const float* __restrict__ s,
                                                            const uint8_t* __restrict__ edgemask, float scale,
                                                            float* __restrict__ Z, float* __restrict__ norm, int partial_from) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    if (t >= T) return;                                  // whole 16-lane groups exit together
    aggregate_task<H, DROP, PARTIAL>(t, tasks, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, h, s, edgemask, scale, Z, norm,
                                     partial_from);
}

// the single-head aggregation on W-wide rows (W = 128: the last stage at embedSize 128): the algorithm of aggregate_task<1, DROP,
// false> (three-stage adjacency / logit / mask pipeline, one weight per lane and batch); lane l owns the W/16 columns W/16*l ..
template <bool DROP, int W>
__global__ void __launch_bounds__(256) aggregate_fwd_wide_kernel(const int4* __restrict__ tasks, int T, const int* __restrict__ adj_ptr,
                                                                 const int* __restrict__ adj_idx, const int* __restrict__ adj_eid,
                                                                 const int* __restrict__ long_first_slot, int* long_counter, float* scratch,
                                                                 const float* __restrict__ h, const float* __restrict__ s,
                                                                 const uint8_t* __restrict__ edgemask, float scale,
                                                                 float* __restrict__ Z, float* __restrict__ norm) {
    constexpr int V = W / 64;
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    if (t >= T) return;                                  // whole 16-lane groups exit together
    const int lane16 = threadIdx.x & 15;
    const unsigned gm = group_mask();
    const int col0 = lane16 * 4 * V;
    const int4 tk = __ldg(tasks + t);
    const int node = tk.x, beg = tk.y, end = tk.z, lid = tk.w;
    const float sn = __ldg(s + node);
    float4 acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    float rs_l = 0.f, s_c = 0.f;
    int m_c = 0, m_1 = 0, eid_1 = 0;
    unsigned mk_c = 1u;
    if (beg + lane16 < end) {
        m_c = ld_stream_i32(adj_idx + beg + lane16);
        if (DROP) mk_c = edgemask[ld_stream_i32(adj_eid + beg + lane16)];
    }
    if (beg + 16 + lane16 < end) {
        m_1 = ld_stream_i32(adj_idx + beg + 16 + lane16);
        if (DROP) eid_1 = ld_stream_i32(adj_eid + beg + 16 + lane16);
    }
    if (beg + lane16 < end) s_c = __ldg(s + m_c);
    for (int base = beg; base < end; base += 16) {
        const int i1x = base + 16 + lane16, i2x = base + 32 + lane16;
        int m_2 = 0, eid_2 = 0;
        float s_1 = 0.f;
        unsigned mk_1 = 1u;
        if (i2x < end) {
            m_2 = ld_stream_i32(adj_idx + i2x);
            if (DROP) eid_2 = ld_stream_i32(adj_eid + i2x);
        }
        if (i1x < end) {
            s_1 = __ldg(s + m_1);
            if (DROP) mk_1 = edgemask[eid_1];
        }
        const float w_l = base + lane16 < end ? edge_weight(sn + s_c) : 0.f;
        rs_l += w_l;
        const float wd_l = DROP ? ((mk_c & 1u) ? w_l * scale : 0.f) : w_l;
        const int cnt = min(16, end - base);
#pragma unroll 8
        for (int j = 0; j < cnt; ++j) {
            const int m = __shfl_sync(gm, m_c, j, 16);
            const float wd = __shfl_sync(gm, wd_l, j, 16);
            float4 hm[V];
#pragma unroll
            for (int v = 0; v < V; ++v) hm[v] = ld_gather4(h + (int64_t)m * W + col0 + 4 * v);
#pragma unroll
            for (int v = 0; v < V; ++v) {
                acc[v].x = fmaf(wd, hm[v].x, acc[v].x); acc[v].y = fmaf(wd, hm[v].y, acc[v].y);
                acc[v].z = fmaf(wd, hm[v].z, acc[v].z); acc[v].w = fmaf(wd, hm[v].w, acc[v].w);
            }
        }
        m_c = m_1; m_1 = m_2; eid_1 = eid_2; s_c = s_1; mk_c = mk_1;
    }
    rs_l += __shfl_xor_sync(gm, rs_l, 1, 16);
    rs_l += __shfl_xor_sync(gm, rs_l, 2, 16);
    rs_l += __shfl_xor_sync(gm, rs_l, 4, 16);
    rs_l += __shfl_xor_sync(gm, rs_l, 8, 16);
    float rs = rs_l;
    if (lid >= 0) {
        float sums[1] = {rs};
        const int chunk = (beg - __ldg(adj_ptr + node)) / CHUNK;
        if (!long_row_combine_wide<W, 1>(lid, chunk, long_first_slot, long_counter, scratch, lane16, gm, acc, sums)) return;
        rs = sums[0];
    }
    // epilogue: Z = h + agg / norm, NaN -> 0 for isolated nodes (SPUIGACF.py:383,388-390)
    const float inv = rs != 0.f ? 1.0f / rs : 0.f;
#pragma unroll
    for (int v = 0; v < V; ++v) {
        const int64_t off = (int64_t)node * W + col0 + 4 * v;
        const float4 hn = ld_stream4(h + off);
        st_stream4(Z + off, make_float4(fmaf(acc[v].x, inv, hn.x), fmaf(acc[v].y, inv, hn.y), fmaf(acc[v].z, inv, hn.z), fmaf(acc[v].w, inv, hn.w)));
    }
    if (lane16 == 0) norm[node] = rs;
}

// Pruned last stage (FusedTrainer): only the tasks of the rows marked active are run (list built by ngacf_active_plan) -- the
// step reads nothing else of the last stage's output (the pair scores gather the batch rows, every other row has a zero
// gradient).  Persistent grid over the compacted list: the working groups are dense however few rows are active.
template <int H, bool DROP>
__global__ void __launch_bounds__(256) aggregate_fwd_list_kernel(const int4* __restrict__ tasks, int T, const int* __restrict__ task_list,
                                                                 const int* __restrict__ task_count, const int* __restrict__ adj_ptr,
                                                                 const int* __restrict__ adj_idx, const int* __restrict__ adj_eid,
                                                                 const int* __restrict__ long_first_slot, int* long_counter, float* scratch,
                                                                 const float* __restrict__ h, const float* __restrict__ s,
                                                                 const uint8_t* __restrict__ edgemask, float scale,
                                                                 float* __restrict__ Z, float* __restrict__ norm) {
    // two lists in one buffer (ngacf_active_plan): user tasks from the front, item tasks from the back
    const int nu = __ldg(task_count), n = nu + __ldg(task_count + 1);
    const int stride = (gridDim.x * blockDim.x) >> 4;
    for (int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 4; g < n; g += stride)
        aggregate_task<H, DROP, false, true>(__ldg(task_list + (g < nu ? g : T - 1 - (g - nu))), tasks, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, h, s,
                                       edgemask, scale, Z, norm, 0x7fffffff);
}

// Z[n] = h[n] + P[n] / norm[n] for rows whose partial sums P (stored in Z) were reduced across ranks
template <int H>
__global__ void __launch_bounds__(256) aggregate_finalize_kernel(float* __restrict__ Z, const float* __restrict__ h,
                                                                 const float* __restrict__ norm, int64_t n_rows) {
    const int64_t n = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    if (n >= n_rows) return;
    const int lane16 = threadIdx.x & 15;
    const int head = H == 8 ? (lane16 >> 1) : 0;
    const float rs = norm[n * H + head];
    const float inv = rs != 0.f ? 1.0f / rs : 0.f;
    const float4 p = ld_stream4(Z + n * D + lane16 * 4), hn = ld_stream4(h + n * D + lane16 * 4);
    st_stream4(Z + n * D + lane16 * 4, make_float4(fmaf(p.x, inv, hn.x), fmaf(p.y, inv, hn.y), fmaf(p.z, inv, hn.z), fmaf(p.w, inv, hn.w)));
}

}  // namespace ngacf

using namespace ngacf;

extern "C" int ngacf_aggregate_finalize(float* Z, const float* h, const float* norm, int32_t H, int64_t n_rows, void* stream) {
    NGACF_REQUIRE(Z && h && norm && n_rows >= 0 && (H == 1 || H == 8), "aggregate_finalize: bad argument");
    if (n_rows == 0) return NGACF_OK;
    const int blocks = ceil_div(n_rows * 16, 256);
    if (H == 8) aggregate_finalize_kernel<8><<<blocks, 256, 0, (cudaStream_t)stream>>>(Z, h, norm, n_rows);
    else        aggregate_finalize_kernel<1><<<blocks, 256, 0, (cudaStream_t)stream>>>(Z, h, norm, n_rows);
    return check_launch("aggregate_finalize");
}

extern "C" int ngacf_feature_mask(uint64_t* feat, int64_t N, uint64_t seed, uint32_t call, const int64_t* call_dev, uint32_t stage,
                                  float droprate, void* stream) {
    NGACF_REQUIRE(feat && N >= 0, "feature_mask: bad args");
    if (N == 0) return NGACF_OK;
    uint32_t thr = keep_threshold(droprate);
    feature_mask_kernel<<<ceil_div(N * 8, 256), 256, 0, (cudaStream_t)stream>>>(feat, N, (uint32_t)seed, (uint32_t)(seed >> 32), call,
                                                                                 call_dev, stage * 2 + 0, thr);
    return check_launch("feature_mask");
}

extern "C" int ngacf_edge_mask(uint8_t* edge, int64_t E, int32_t H, uint64_t seed, uint32_t call, const int64_t* call_dev, uint32_t stage,
                               float droprate, void* stream) {
    NGACF_REQUIRE(edge && E >= 0 && (H == 1 || H == 8), "edge_mask: bad args");
    if (E == 0) return NGACF_OK;
    uint32_t thr = keep_threshold(droprate);
    edge_mask_kernel<<<ceil_div(E, 256), 256, 0, (cudaStream_t)stream>>>(edge, E, H, (uint32_t)seed, (uint32_t)(seed >> 32), call,
                                                                          call_dev, stage * 2 + 1, thr);
    return check_launch("edge_mask");
}

extern "C" int ngacf_dropout_masks_w(uint64_t* const* feat, uint8_t* const* edge, const int32_t* heads, const int32_t* widths, int32_t S,
                                     int64_t N, int64_t E, uint64_t seed, uint32_t call, const int64_t* call_dev, float droprate,
                                     void* stream) {
    NGACF_REQUIRE(feat && edge && heads && S >= 1 && S <= MASK_MAX_STAGES && N >= 0 && E >= 0, "dropout_masks: bad args");
    MaskPlan plan;
    int max_shift = 0;
    for (int k = 0; k < S; ++k) {
        NGACF_REQUIRE(feat[k] && (edge[k] || E == 0) && (heads[k] == 1 || heads[k] == 8), "dropout_masks: bad stage %d", k);
        const int wd = widths ? widths[k] : 64;
        if (!width_supported(wd)) {
            set_error("dropout_masks_w: stage %d input width %d is not built (supported: 64, 128)", k, wd);
            return NGACF_ERR_UNSUPPORTED;
        }
        plan.feat[k] = feat[k]; plan.edge[k] = edge[k]; plan.heads[k] = heads[k];
        plan.wshift[k] = wd == 128 ? 1 : 0;
        if (plan.wshift[k] > max_shift) max_shift = plan.wshift[k];
    }
    plan.S = S;
    plan.feat_blocks = ceil_div((N * 8) << max_shift, 256);
    plan.edge_blocks = ceil_div(E, 256);
    const int64_t blocks = (int64_t)S * (plan.feat_blocks + plan.edge_blocks);
    if (blocks == 0) return NGACF_OK;
    dropout_masks_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(plan, N, E, (uint32_t)seed, (uint32_t)(seed >> 32), call,
                                                                             call_dev, keep_threshold(droprate));
    return check_launch("dropout_masks");
}

extern "C" int ngacf_dropout_masks(uint64_t* const* feat, uint8_t* const* edge, const int32_t* heads, int32_t S, int64_t N, int64_t E,
                                   uint64_t seed, uint32_t call, const int64_t* call_dev, float droprate, void* stream) {
    return ngacf_dropout_masks_w(feat, edge, heads, nullptr, S, N, E, seed, call, call_dev, droprate, stream);
}

extern "C" int ngacf_dropout_masks_ranges(uint64_t* const* feat, uint8_t* const* edge, const int32_t* heads, int32_t S, int64_t fa0, int64_t fb0,
                                          int64_t fa1, int64_t fb1, int64_t e0, int64_t e1, uint64_t seed, uint32_t call, const int64_t* call_dev,
                                          float droprate, void* stream) {
    NGACF_REQUIRE(feat && edge && heads && S >= 1 && S <= MASK_MAX_STAGES && fa0 >= 0 && fb0 >= fa0 && fa1 >= 0 && fb1 >= fa1 && e0 >= 0 && e1 >= e0,
                  "dropout_masks_ranges: bad args");
    MaskPlan plan;
    for (int k = 0; k < S; ++k) {
        NGACF_REQUIRE(feat[k] && (edge[k] || e1 == e0) && (heads[k] == 1 || heads[k] == 8), "dropout_masks_ranges: bad stage %d", k);
        plan.feat[k] = feat[k]; plan.edge[k] = edge[k]; plan.heads[k] = heads[k]; plan.wshift[k] = 0;
    }
    plan.S = S;
    plan.feat_blocks = plan.edge_blocks = 0;
    MaskRanges r;
    r.fa0 = fa0; r.fb0 = fb0; r.fa1 = fa1; r.fb1 = fb1; r.e0 = e0; r.e1 = e1;
    r.fb_blocks0 = ceil_div((fb0 - fa0) * 8, 256);
    r.fb_blocks1 = ceil_div((fb1 - fa1) * 8, 256);
    r.e_blocks = ceil_div(e1 - e0, 256);
    const int64_t blocks = (int64_t)S * (r.fb_blocks0 + r.fb_blocks1 + r.e_blocks);
    if (blocks == 0) return NGACF_OK;
    dropout_masks_ranges_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(plan, r, (uint32_t)seed, (uint32_t)(seed >> 32), call, call_dev,
                                                                                    keep_threshold(droprate));
    return check_launch("dropout_masks_ranges");
}

extern "C" int ngacf_transform_fwd(const float* Xu, const float* Xi, int32_t apply_elu, const uint64_t* featmask, float scale,
                                   const float* const* wtab, int32_t H, int32_t U, int32_t I, float* h, float* s, void* stream) {
    NGACF_REQUIRE(wtab && h && s && U >= 0 && I >= 0 && (U == 0 || Xu) && (I == 0 || Xi), "transform_fwd: null argument");
    if (U + I == 0) return NGACF_OK;
    NGACF_REQUIRE(H == 1 || H == 8, "transform_fwd: H must be 1 or 8 (got %d)", H);
    if (dense_on_tensor_cores()) {
        transform_fwd_tc(Xu, Xi, apply_elu, featmask, scale, wtab, H, U, I, h, s, (cudaStream_t)stream);
        return check_launch("transform_fwd(tc)");
    }
    const int tiles_u = ceil_div(U, TF_TM), tiles_i = ceil_div(I, TF_TM);
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(transform_fwd_kernel<8, 64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TF_SMEM);
        cudaFuncSetAttribute(transform_fwd_kernel<1, 64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TF_SMEM);
    });
    if (H == 8)
        transform_fwd_kernel<8, 64, 64><<<tiles_u + tiles_i, 256, TF_SMEM, (cudaStream_t)stream>>>(Xu, Xi, apply_elu, featmask, scale, wtab, U, I, tiles_u, h, s);
    else
        transform_fwd_kernel<1, 64, 64><<<tiles_u + tiles_i, 256, TF_SMEM, (cudaStream_t)stream>>>(Xu, Xi, apply_elu, featmask, scale, wtab, U, I, tiles_u, h, s);
    return check_launch("transform_fwd");
}

// (d_in, d_out) = (64, 64): ngacf_transform_fwd (tensor cores or NGACF_DENSE=ffma).  The embedSize-128 shapes run on the CUDA-core
// kernel: (128, 64) with 8 heads (first stage) and (64, 128) with one head (last stage).
template <int H, int DIN, int DOUT>
static int launch_transform_fwd_wide(const float* Xu, const float* Xi, int apply_elu, const uint64_t* featmask, float scale,
                                     const float* const* wtab, int U, int I, float* h, float* s, cudaStream_t st) {
    constexpr int TM = tf_tm<DOUT>();
    constexpr size_t SMEM = tf_smem<DIN, DOUT>();
    static PerDeviceOnce once;
    once.run([] { cudaFuncSetAttribute(transform_fwd_kernel<H, DIN, DOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM); });
    const int tiles_u = ceil_div(U, TM), tiles_i = ceil_div(I, TM);
    transform_fwd_kernel<H, DIN, DOUT><<<tiles_u + tiles_i, 256, SMEM, st>>>(Xu, Xi, apply_elu, featmask, scale, wtab, U, I, tiles_u, h, s);
    return check_launch("transform_fwd_w");
}

extern "C" int ngacf_transform_fwd_w(const float* Xu, const float* Xi, int32_t apply_elu, const uint64_t* featmask, float scale,
                                     const float* const* wtab, int32_t H, int32_t d_in, int32_t d_out, int32_t U, int32_t I, float* h,
                                     float* s, void* stream) {
    if (d_in == 64 && d_out == 64) return ngacf_transform_fwd(Xu, Xi, apply_elu, featmask, scale, wtab, H, U, I, h, s, stream);
    const bool first = H == 8 && d_in == 128 && d_out == 64, last = H == 1 && d_in == 64 && d_out == 128;
    if (!first && !last) {
        set_error("transform_fwd_w: (H, d_in, d_out) = (%d, %d, %d) is not built; supported: (1|8, 64, 64), (8, 128, 64), (1, 64, 128)", H,
                  d_in, d_out);
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(wtab && h && s && U >= 0 && I >= 0 && (U == 0 || Xu) && (I == 0 || Xi), "transform_fwd_w: null argument");
    if (U + I == 0) return NGACF_OK;
    if (first) return launch_transform_fwd_wide<8, 128, 64>(Xu, Xi, apply_elu, featmask, scale, wtab, U, I, h, s, (cudaStream_t)stream);
    return launch_transform_fwd_wide<1, 64, 128>(Xu, Xi, apply_elu, featmask, scale, wtab, U, I, h, s, (cudaStream_t)stream);
}

extern "C" int ngacf_aggregate_fwd(const int32_t* tasks, int32_t T, const int32_t* adj_ptr, const int32_t* adj_idx, const int32_t* adj_eid,
                                   const int32_t* long_first_slot, int32_t* long_counter, float* scratch, const float* h, const float* s,
                                   int32_t H, const uint8_t* edgemask, float scale, float* Z, float* norm, int32_t partial_from,
                                   void* stream) {
    NGACF_REQUIRE(tasks && adj_ptr && adj_idx && h && s && Z && norm && T > 0, "aggregate_fwd: null/empty argument");
    if (partial_from < 0) partial_from = T;
    NGACF_REQUIRE(H == 1 || H == 8, "aggregate_fwd: H must be 1 or 8 (got %d)", H);
    NGACF_REQUIRE(!edgemask || adj_eid, "aggregate_fwd: edge dropout needs adj_eid");
    const int blocks = ceil_div((int64_t)T * 16, 256);
    cudaStream_t st = (cudaStream_t)stream;
    const int4* tk = reinterpret_cast<const int4*>(tasks);
    static PerDeviceOnce once;
    once.run([] {     // gather kernels use no shared memory: ask for the whole unified array as L1
#define CARVE(HH, DR, PA) cudaFuncSetAttribute(aggregate_fwd_kernel<HH, DR, PA>, cudaFuncAttributePreferredSharedMemoryCarveout, 0)
        CARVE(8, true, false); CARVE(8, false, false); CARVE(1, true, false); CARVE(1, false, false);
#undef CARVE
    });
#define LAUNCH(HH, DR, PA) aggregate_fwd_kernel<HH, DR, PA><<<blocks, 256, 0, st>>>(tk, T, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, h, s, edgemask, scale, Z, norm, partial_from)
    if (partial_from < T) {
        if (H == 8) { if (edgemask) LAUNCH(8, true, true); else LAUNCH(8, false, true); }
        else        { if (edgemask) LAUNCH(1, true, true); else LAUNCH(1, false, true); }
    } else {
        if (H == 8) { if (edgemask) LAUNCH(8, true, false); else LAUNCH(8, false, false); }
        else        { if (edgemask) LAUNCH(1, true, false); else LAUNCH(1, false, false); }
    }
#undef LAUNCH
    return check_launch("aggregate_fwd");
}

extern "C" int ngacf_aggregate_fwd_w(const int32_t* tasks, int32_t T, const int32_t* adj_ptr, const int32_t* adj_idx, const int32_t* adj_eid,
                                     const int32_t* long_first_slot, int32_t* long_counter, float* scratch, const float* h, const float* s,
                                     int32_t H, int32_t width, const uint8_t* edgemask, float scale, float* Z, float* norm,
                                     int32_t partial_from, void* stream) {
    if (width == 64)
        return ngacf_aggregate_fwd(tasks, T, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, h, s, H, edgemask, scale, Z,
                                   norm, partial_from, stream);
    if (width != 128 || H != 1 || (partial_from >= 0 && partial_from < T)) {
        set_error("aggregate_fwd_w: (H, width) = (%d, %d)%s is not built; 128-wide rows: H = 1, full rows", H, width,
                  (partial_from >= 0 && partial_from < T) ? " with partial rows" : "");
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(tasks && adj_ptr && adj_idx && h && s && Z && norm && T > 0, "aggregate_fwd_w: null/empty argument");
    NGACF_REQUIRE(!edgemask || adj_eid, "aggregate_fwd_w: edge dropout needs adj_eid");
    const int blocks = ceil_div((int64_t)T * 16, 256);
    cudaStream_t st = (cudaStream_t)stream;
    const int4* tk = reinterpret_cast<const int4*>(tasks);
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(aggregate_fwd_wide_kernel<true, 128>, cudaFuncAttributePreferredSharedMemoryCarveout, 0);
        cudaFuncSetAttribute(aggregate_fwd_wide_kernel<false, 128>, cudaFuncAttributePreferredSharedMemoryCarveout, 0);
    });
    if (edgemask)
        aggregate_fwd_wide_kernel<true, 128><<<blocks, 256, 0, st>>>(tk, T, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, h,
                                                                     s, edgemask, scale, Z, norm);
    else
        aggregate_fwd_wide_kernel<false, 128><<<blocks, 256, 0, st>>>(tk, T, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, h,
                                                                      s, edgemask, scale, Z, norm);
    return check_launch("aggregate_fwd_w");
}

int ngacf_launch_aggregate_fwd_cta(const int32_t* tasks, int32_t T, const int32_t* task_list, const int32_t* task_count, const int32_t* adj_ptr,
                                   const int32_t* adj_idx, const int32_t* adj_eid, const int32_t* long_first_slot, int32_t* long_counter,
                                   float* scratch, const float* h, const float* s, const uint8_t* edgemask, float scale, float* Z, float* norm,
                                   cudaStream_t st);      // csrc/pruned_stage.cu

extern "C" int ngacf_aggregate_fwd_active(const int32_t* tasks, int32_t T, const int32_t* task_list, const int32_t* task_count,
                                          const int32_t* adj_ptr, const int32_t* adj_idx, const int32_t* adj_eid,
                                          const int32_t* long_first_slot, int32_t* long_counter, float* scratch, const float* h,
                                          const float* s, int32_t H, const uint8_t* edgemask, float scale, float* Z, float* norm,
                                          void* stream) {
    NGACF_REQUIRE(tasks && task_list && task_count && adj_ptr && adj_idx && h && s && Z && norm && T > 0, "aggregate_fwd_active: null/empty argument");
    NGACF_REQUIRE(H == 1 || H == 8, "aggregate_fwd_active: H must be 1 or 8 (got %d)", H);
    NGACF_REQUIRE(!edgemask || adj_eid, "aggregate_fwd_active: edge dropout needs adj_eid");
    cudaStream_t st = (cudaStream_t)stream;
    if (H == 1)
        return ngacf_launch_aggregate_fwd_cta(tasks, T, task_list, task_count, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, h,
                                              s, edgemask, scale, Z, norm, st);
    int blocks = ceil_div((int64_t)T * 16, 256);
    if (blocks > 148 * 8) blocks = 148 * 8;              // persistent: the list length lives on the device
    const int4* tk = reinterpret_cast<const int4*>(tasks);
#define LAUNCH(HH, DR) aggregate_fwd_list_kernel<HH, DR><<<blocks, 256, 0, st>>>(tk, T, task_list, task_count, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, h, s, edgemask, scale, Z, norm)
    if (H == 8) { if (edgemask) LAUNCH(8, true); else LAUNCH(8, false); }
    else        { if (edgemask) LAUNCH(1, true); else LAUNCH(1, false); }
#undef LAUNCH
    return check_launch("aggregate_fwd_active");
}
