// Backward of one SpUIGAT stage in closed form (SURVEY.md 3.4; the reference relies on autograd through
// graphattention/SPUIGACF.py:340-400).  Unified-node formulation, G = dL/dZ:
//   Ghat[n] = G[n]/norm[n]                      dN[n] = -(G[n].(Z[n]-h[n]))/norm[n]            (per head)
//   d e~(n,m) = Ghat[n].h[m] + Ghat[m].h[n]     d e = keep*scale*d e~ + dN[n] + dN[m]
//   d s = d e * (-e) * LeakyReLU'(s[n]+s[m])    dS[n] = sum_m d s(n,m)
//   dh[n] = G[n] + sum_m drop(e) Ghat[m] + dS[n] (x) a_side
//   dW = Xd^T dh,  da = sum_n dS[n] (x) h[n],  dX = dh W^T (then dropout mask and ELU' of the producer)
// User rows walk the CSR half and store d s per edge; item rows walk the CSC half and read it back
// through adj_eid, so neither side needs atomics.
#include "common.cuh"

namespace ngacf {

template <int H>
__device__ __forceinline__ int lane_head_b(int lane16) { return H == 8 ? (lane16 >> 1) : 0; }
template <int H>
__device__ __forceinline__ bool head_writer(int lane16) { return H == 8 ? ((lane16 & 1) == 0) : (lane16 == 0); }

// ------------------------------------------------------------------------------------------------
template <int H>
__global__ void __launch_bounds__(256) stage_bwd_prep_kernel(const float* __restrict__ G, const float* __restrict__ Z,
                                                             const float* __restrict__ h, const float* __restrict__ norm, int64_t N,
                                                             float* __restrict__ Ghat, float* __restrict__ dN) {
    const int64_t n = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const int lane16 = threadIdx.x & 15;
    const unsigned gm = group_mask();
    if (n >= N) return;
    const int head = lane_head_b<H>(lane16);
    const float4 g = ld_stream4(G + n * D + lane16 * 4);
    const float4 z = ld_stream4(Z + n * D + lane16 * 4);
    const float4 hh = ld_stream4(h + n * D + lane16 * 4);
    const float nr = __ldg(norm + n * H + head);
    const float inv = nr != 0.f ? 1.0f / nr : 0.f;
    float part = g.x * (z.x - hh.x) + g.y * (z.y - hh.y) + g.z * (z.z - hh.z) + g.w * (z.w - hh.w);
    part = head_reduce<H>(part, gm);
    st_stream4(Ghat + n * D + lane16 * 4, make_float4(g.x * inv, g.y * inv, g.z * inv, g.w * inv));
    if (head_writer<H>(lane16)) dN[n * H + head] = -part * inv;
}


// the same for single-head W-wide rows (W = 128): lane l owns columns W/16*l ..
template <int W>
__global__ void __launch_bounds__(256) stage_bwd_prep_wide_kernel(const float* __restrict__ G, const float* __restrict__ Z,
                                                             const float* __restrict__ h, const float* __restrict__ norm, int64_t N,
                                                             float* __restrict__ Ghat, float* __restrict__ dN) {
    constexpr int H = 1, V = W / 64;
    const int64_t n = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const int lane16 = threadIdx.x & 15;
    const unsigned gm = group_mask();
    if (n >= N) return;
    const int head = lane_head_b<H>(lane16);
    float4 g[V], z[V], hh[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
        const int64_t off = n * W + lane16 * 4 * V + 4 * v;
        g[v] = ld_stream4(G + off);
        z[v] = ld_stream4(Z + off);
        hh[v] = ld_stream4(h + off);
    }
    const float nr = __ldg(norm + n * H + head);
    const float inv = nr != 0.f ? 1.0f / nr : 0.f;
    float part = g[0].x * (z[0].x - hh[0].x) + g[0].y * (z[0].y - hh[0].y) + g[0].z * (z[0].z - hh[0].z) + g[0].w * (z[0].w - hh[0].w);
#pragma unroll
    for (int v = 1; v < V; ++v)
        part += g[v].x * (z[v].x - hh[v].x) + g[v].y * (z[v].y - hh[v].y) + g[v].z * (z[v].z - hh[v].z) + g[v].w * (z[v].w - hh[v].w);
    part = head_reduce<H>(part, gm);
#pragma unroll
    for (int v = 0; v < V; ++v)
        st_stream4(Ghat + n * W + lane16 * 4 * V + 4 * v, make_float4(g[v].x * inv, g[v].y * inv, g[v].z * inv, g[v].w * inv));
    if (head_writer<H>(lane16)) dN[n * H + head] = -part * inv;
}

// ------------------------------------------------------------------------------------------------
template <int H, int MODE, bool DROP, bool PARTIAL>
__global__ void __launch_bounds__(256, (MODE == 1 && H == 1) ? 5 : 0) stage_bwd_edges_kernel(const int4* __restrict__ tasks, int T_begin, int T_end,
                                                              const int* __restrict__ adj_ptr, const int* __restrict__ adj_idx,
                                                              const int* __restrict__ adj_eid, const int* __restrict__ long_first_slot,
                                                              int* long_counter, float* scratch, const float* __restrict__ G,
                                                              const float* __restrict__ Ghat, const float* __restrict__ dN,
                                                              const float* __restrict__ h, const float* __restrict__ s,
                                                              const uint8_t* __restrict__ edgemask, float scale,
                                                              const float* const* __restrict__ wtab, int U,
                                                              float* ds_store, float* __restrict__ dh, float* __restrict__ dS) {
    constexpr int DH = D / H;
    const int t = T_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 4);
    if (t >= T_end) return;
    const int lane16 = threadIdx.x & 15;
    const unsigned gm = group_mask();
    const int head = lane_head_b<H>(lane16);
    const int4 tk = __ldg(tasks + t);
    const int node = tk.x, beg = tk.y, end = tk.z, lid = tk.w;
    // H = 1: the user pass stores (d s_e, e*keep) per edge and the item pass reads the pair -- no logit gather, exp or mask byte
    // there (in-box A/B: 60 -> 47 us per launch; for H = 8 the 64-byte pairs cost more than they save, profiles/r1e_ab_prefetch.txt)
    constexpr bool PAIR = (H == 1);
    constexpr bool NEED_MASK = DROP && !(PAIR && MODE == 1);
    const float sn = (PAIR && MODE == 1) ? 0.f : __ldg(s + (int64_t)node * H + head);
    const float sc = DROP ? scale : 1.f;
    float4 ghn = make_float4(0.f, 0.f, 0.f, 0.f), hn = ghn;
    float dNn = 0.f;
    if (MODE == 0) {
        ghn = ld_stream4(Ghat + (int64_t)node * D + lane16 * 4);
        hn = ld_stream4(h + (int64_t)node * D + lane16 * 4);
        dNn = __ldg(dN + (int64_t)node * H + head);
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float dSacc = 0.f;
    // software-pipelined adjacency: batch b+1's neighbour/edge ids are requested before batch b's gathers, its mask bytes
    // right after them (same scheme as aggregate_fwd_kernel)
    int m_l = 0, eid_l = 0;
    unsigned mk_l = 0xFFu;
    if (beg + lane16 < end) {
        m_l = ld_stream_i32(adj_idx + beg + lane16);
        eid_l = ld_stream_i32(adj_eid + beg + lane16);
        if (NEED_MASK) mk_l = edgemask[eid_l];
    }
    for (int base = beg; base < end; base += 16) {
        const int nidx = base + 16 + lane16;
        int m_n = 0, eid_n = 0;
        unsigned mk_n = 0xFFu;
        if (nidx < end) {
            m_n = ld_stream_i32(adj_idx + nidx);
            eid_n = ld_stream_i32(adj_eid + nidx);
        }
        const int cnt = min(16, end - base);
#pragma unroll (MODE == 0 ? 4 : 8)
        for (int j = 0; j < cnt; ++j) {
            const int m = __shfl_sync(gm, m_l, j, 16);
            const int eid = __shfl_sync(gm, eid_l, j, 16);
            if (PAIR && MODE == 1) {
                const float4 g4 = ld_gather4(Ghat + (int64_t)m * D + lane16 * 4);
                const float2 pr = __ldg(reinterpret_cast<const float2*>(ds_store) + eid);
                acc.x = fmaf(pr.y, g4.x, acc.x); acc.y = fmaf(pr.y, g4.y, acc.y);
                acc.z = fmaf(pr.y, g4.z, acc.z); acc.w = fmaf(pr.y, g4.w, acc.w);
                dSacc += pr.x;
                continue;
            }
            const float sm = __ldg(s + (int64_t)m * H + head);
            const float4 gm4 = ld_gather4(Ghat + (int64_t)m * D + lane16 * 4);
            const float x = sn + sm;
            const float e = edge_weight(x);
            float keepsc = sc;
            if (DROP) {
                const unsigned mk = __shfl_sync(gm, mk_l, j, 16);
                keepsc = ((mk >> head) & 1u) ? sc : 0.f;
            }
            const float et = e * keepsc;
            acc.x = fmaf(et, gm4.x, acc.x); acc.y = fmaf(et, gm4.y, acc.y);
            acc.z = fmaf(et, gm4.z, acc.z); acc.w = fmaf(et, gm4.w, acc.w);
            float ds;
            if (MODE == 0) {
                const float4 hm = ld_gather4(h + (int64_t)m * D + lane16 * 4);
                float part = ghn.x * hm.x + ghn.y * hm.y + ghn.z * hm.z + ghn.w * hm.w
                           + gm4.x * hn.x + gm4.y * hn.y + gm4.z * hn.z + gm4.w * hn.w;
                const float det = head_reduce<H>(part, gm);
                const float de = fmaf(det, keepsc, dNn + __ldg(dN + (int64_t)m * H + head));
                ds = de * (-e) * (x > 0.f ? 1.f : LRELU_ALPHA);
                if (head_writer<H>(lane16)) {
                    if (PAIR) reinterpret_cast<float2*>(ds_store)[eid] = make_float2(ds, et);
                    else ds_store[(int64_t)eid * H + head] = ds;
                }
            } else {
                ds = __ldg(ds_store + (int64_t)eid * H + head);
            }
            dSacc += ds;
        }
        if (NEED_MASK && nidx < end) mk_n = edgemask[eid_n];
        m_l = m_n; eid_l = eid_n; mk_l = mk_n;
    }
    if (lid >= 0) {
        float sums[1] = {dSacc};
        const int chunk = (beg - __ldg(adj_ptr + node)) / CHUNK;
        if (!long_row_combine<H, 1>(lid, chunk, long_first_slot, long_counter, scratch, lane16, gm, acc, sums)) return;
        dSacc = sums[0];
    }
    if (PARTIAL) {     // multi-GPU: raw partial sums over this rank's slice of the row; reduced across ranks, then stage_bwd_finalize
        st_stream4(dh + (int64_t)node * D + lane16 * 4, acc);
        if (head_writer<H>(lane16)) dS[(int64_t)node * H + head] = dSacc;
        return;
    }
    const float4 gn = ld_stream4(G + (int64_t)node * D + lane16 * 4);
    const float* ap = wtab[2 * H + head] + (node >= U ? DH : 0) + ((lane16 * 4) % DH);
    const float4 a4 = make_float4(__ldg(ap), __ldg(ap + 1), __ldg(ap + 2), __ldg(ap + 3));
    st_stream4(dh + (int64_t)node * D + lane16 * 4,
               make_float4(gn.x + acc.x + dSacc * a4.x, gn.y + acc.y + dSacc * a4.y, gn.z + acc.z + dSacc * a4.z, gn.w + acc.w + dSacc * a4.w));
    if (head_writer<H>(lane16)) dS[(int64_t)node * H + head] = dSacc;
}

// the single-head pair of edge passes on W-wide rows (W = 128: the last stage at embedSize 128); the same algorithm as
// stage_bwd_edges_kernel<1, MODE, DROP, false>, lane l owns the W/16 columns W/16*l ..
template <int MODE, bool DROP, int W>
__global__ void __launch_bounds__(256) stage_bwd_edges_wide_kernel(const int4* __restrict__ tasks, int T_begin, int T_end,
                                                              const int* __restrict__ adj_ptr, const int* __restrict__ adj_idx,
                                                              const int* __restrict__ adj_eid, const int* __restrict__ long_first_slot,
                                                              int* long_counter, float* scratch, const float* __restrict__ G,
                                                              const float* __restrict__ Ghat, const float* __restrict__ dN,
                                                              const float* __restrict__ h, const float* __restrict__ s,
                                                              const uint8_t* __restrict__ edgemask, float scale,
                                                              const float* const* __restrict__ wtab, int U,
                                                              float* ds_store, float* __restrict__ dh, float* __restrict__ dS) {
    constexpr int H = 1, DH = W;
    constexpr int V = W / 64;          // float4 per lane: lane l owns columns 4V*l .. 4V*l + 4V-1
    const int t = T_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 4);
    if (t >= T_end) return;
    const int lane16 = threadIdx.x & 15;
    const unsigned gm = group_mask();
    const int head = lane_head_b<H>(lane16);
    const int col0 = lane16 * 4 * V;
    const int4 tk = __ldg(tasks + t);
    const int node = tk.x, beg = tk.y, end = tk.z, lid = tk.w;
    constexpr bool PAIR = true;       // the user pass stores (d s_e, e*keep) per edge, the item pass reads the pair
    constexpr bool NEED_MASK = DROP && !(PAIR && MODE == 1);
    const float sn = (PAIR && MODE == 1) ? 0.f : __ldg(s + (int64_t)node * H + head);
    const float sc = DROP ? scale : 1.f;
    float4 ghn[V], hn[V], acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) ghn[v] = hn[v] = acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    float dNn = 0.f;
    if (MODE == 0) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
            ghn[v] = ld_stream4(Ghat + (int64_t)node * W + col0 + 4 * v);
            hn[v] = ld_stream4(h + (int64_t)node * W + col0 + 4 * v);
        }
        dNn = __ldg(dN + (int64_t)node * H + head);
    }
    float dSacc = 0.f;
    // software-pipelined adjacency: batch b+1's neighbour/edge ids are requested before batch b's gathers, its mask bytes
    // right after them (same scheme as aggregate_fwd_kernel)
    int m_l = 0, eid_l = 0;
    unsigned mk_l = 0xFFu;
    if (beg + lane16 < end) {
        m_l = ld_stream_i32(adj_idx + beg + lane16);
        eid_l = ld_stream_i32(adj_eid + beg + lane16);
        if (NEED_MASK) mk_l = edgemask[eid_l];
    }
    for (int base = beg; base < end; base += 16) {
        const int nidx = base + 16 + lane16;
        int m_n = 0, eid_n = 0;
        unsigned mk_n = 0xFFu;
        if (nidx < end) {
            m_n = ld_stream_i32(adj_idx + nidx);
            eid_n = ld_stream_i32(adj_eid + nidx);
        }
        const int cnt = min(16, end - base);
#pragma unroll (MODE == 0 ? 4 : 8)
        for (int j = 0; j < cnt; ++j) {
            const int m = __shfl_sync(gm, m_l, j, 16);
            const int eid = __shfl_sync(gm, eid_l, j, 16);
            if (PAIR && MODE == 1) {
                float4 g4[V];
#pragma unroll
                for (int v = 0; v < V; ++v) g4[v] = ld_gather4(Ghat + (int64_t)m * W + col0 + 4 * v);
                const float2 pr = __ldg(reinterpret_cast<const float2*>(ds_store) + eid);
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    acc[v].x = fmaf(pr.y, g4[v].x, acc[v].x); acc[v].y = fmaf(pr.y, g4[v].y, acc[v].y);
                    acc[v].z = fmaf(pr.y, g4[v].z, acc[v].z); acc[v].w = fmaf(pr.y, g4[v].w, acc[v].w);
                }
                dSacc += pr.x;
                continue;
            }
            const float sm = __ldg(s + (int64_t)m * H + head);
            float4 gm4[V];
#pragma unroll
            for (int v = 0; v < V; ++v) gm4[v] = ld_gather4(Ghat + (int64_t)m * W + col0 + 4 * v);
            const float x = sn + sm;
            const float e = edge_weight(x);
            float keepsc = sc;
            if (DROP) {
                const unsigned mk = __shfl_sync(gm, mk_l, j, 16);
                keepsc = ((mk >> head) & 1u) ? sc : 0.f;
            }
            const float et = e * keepsc;
#pragma unroll
            for (int v = 0; v < V; ++v) {
                acc[v].x = fmaf(et, gm4[v].x, acc[v].x); acc[v].y = fmaf(et, gm4[v].y, acc[v].y);
                acc[v].z = fmaf(et, gm4[v].z, acc[v].z); acc[v].w = fmaf(et, gm4[v].w, acc[v].w);
            }
            float ds;
            if (MODE == 0) {
                float4 hm[V];
#pragma unroll
                for (int v = 0; v < V; ++v) hm[v] = ld_gather4(h + (int64_t)m * W + col0 + 4 * v);
                float part = ghn[0].x * hm[0].x + ghn[0].y * hm[0].y + ghn[0].z * hm[0].z + ghn[0].w * hm[0].w
                           + gm4[0].x * hn[0].x + gm4[0].y * hn[0].y + gm4[0].z * hn[0].z + gm4[0].w * hn[0].w;
#pragma unroll
                for (int v = 1; v < V; ++v)
                    part += ghn[v].x * hm[v].x + ghn[v].y * hm[v].y + ghn[v].z * hm[v].z + ghn[v].w * hm[v].w
                          + gm4[v].x * hn[v].x + gm4[v].y * hn[v].y + gm4[v].z * hn[v].z + gm4[v].w * hn[v].w;
                const float det = head_reduce<H>(part, gm);
                const float de = fmaf(det, keepsc, dNn + __ldg(dN + (int64_t)m * H + head));
                ds = de * (-e) * (x > 0.f ? 1.f : LRELU_ALPHA);
                if (head_writer<H>(lane16)) {
                    if (PAIR) reinterpret_cast<float2*>(ds_store)[eid] = make_float2(ds, et);
                    else ds_store[(int64_t)eid * H + head] = ds;
                }
            } else {
                ds = __ldg(ds_store + (int64_t)eid * H + head);
            }
            dSacc += ds;
        }
        if (NEED_MASK && nidx < end) mk_n = edgemask[eid_n];
        m_l = m_n; eid_l = eid_n; mk_l = mk_n;
    }
    if (lid >= 0) {
        float sums[1] = {dSacc};
        const int chunk = (beg - __ldg(adj_ptr + node)) / CHUNK;
        if (!long_row_combine_wide<W, 1>(lid, chunk, long_first_slot, long_counter, scratch, lane16, gm, acc, sums)) return;
        dSacc = sums[0];
    }
#pragma unroll
    for (int v = 0; v < V; ++v) {
        const int64_t off = (int64_t)node * W + col0 + 4 * v;
        const float4 gn = ld_stream4(G + off);
        const float* ap = wtab[2 * H + head] + (node >= U ? DH : 0) + ((col0 + 4 * v) % DH);
        const float4 a4 = make_float4(__ldg(ap), __ldg(ap + 1), __ldg(ap + 2), __ldg(ap + 3));
        st_stream4(dh + off, make_float4(gn.x + acc[v].x + dSacc * a4.x, gn.y + acc[v].y + dSacc * a4.y, gn.z + acc[v].z + dSacc * a4.z,
                                         gn.w + acc[v].w + dSacc * a4.w));
    }
    if (head_writer<H>(lane16)) dS[(int64_t)node * H + head] = dSacc;
}

// dh[n] = G[n] + P[n] + dS[n] (x) a_side for rows whose partials (P in dh, dS) were reduced across ranks
template <int H>
__global__ void __launch_bounds__(256) stage_bwd_finalize_kernel(float* __restrict__ dh, const float* __restrict__ dS,
                                                                 const float* __restrict__ G, const float* const* __restrict__ wtab,
                                                                 int item_side, int64_t n_rows) {
    constexpr int DH = D / H;
    const int64_t n = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    if (n >= n_rows) return;
    const int lane16 = threadIdx.x & 15;
    const int head = lane_head_b<H>(lane16);
    const float d = dS[n * H + head];
    const float* ap = wtab[2 * H + head] + (item_side ? DH : 0) + ((lane16 * 4) % DH);
    const float4 p = ld_stream4(dh + n * D + lane16 * 4), g = ld_stream4(G + n * D + lane16 * 4);
    st_stream4(dh + n * D + lane16 * 4, make_float4(g.x + p.x + d * __ldg(ap), g.y + p.y + d * __ldg(ap + 1), g.z + p.z + d * __ldg(ap + 2),
                                                    g.w + p.w + d * __ldg(ap + 3)));
}

// ------------------------------------------------------------------------------------------------
// dense backward: dX = dh W^T (+ mask/ELU'), partial dW = Xd^T dh, partial da = W^T-contracted Q = Xd^T dS
// persistent blocks per side, 64-row tiles, three CTAs per SM; deterministic two-pass reduction of the partials.
//   * h = Xd W, hence da[c] = sum_r dS[r,head(c)] h[r,c] = sum_k W[k,c] Q[k,head(c)]: the h tile is never read
//   * ELU'(z) is recovered from the recomputed stage input e = ELU(z) already in shared memory (1 for e > 0, e + 1 otherwise)
//   * lane = (8 row/k groups) x (4 column groups): both GEMMs read 8 + 4 distinct 16-byte words per warp and step,
//     conflict-free with the 68-float row stride
// ------------------------------------------------------------------------------------------------
constexpr int TB_TM = 64;
constexpr int TB_XS = 68;
// (DIN, DOUT) = (64, 64) for every stage of the 64-wide models; embedSize 128 adds (128, 64) (first stage) and (64, 128) (last)
template <int DIN, int DOUT> __host__ __device__ constexpr int tb_smem_floats() {
    return DOUT * DIN + TB_TM * (DOUT + 4) + TB_TM * (DIN + 4) + TB_TM * 8 + 2 * TB_TM * (DIN / 64);   // W^T, dh, Xd, dS, mask words
}
template <int DIN, int DOUT> __host__ __device__ constexpr int tb_part() { return DIN * DOUT + DOUT; }   // floats per block partial
constexpr int TB_SMEM_FLOATS = tb_smem_floats<64, 64>();
constexpr size_t TB_SMEM = (size_t)TB_SMEM_FLOATS * sizeof(float);
constexpr int TB_PART = tb_part<64, 64>();
constexpr int TB_CTAS_PER_SM = 3;     // in-box A/B: 3 CTAs (85 registers, no spills) beat 4 (64 registers, spills)

template <int H>
__global__ void __launch_bounds__(256, TB_CTAS_PER_SM) transform_bwd_kernel(const float* __restrict__ dh, const float* __restrict__ dS,
                                                            const float* __restrict__ Xu,
                                                            const float* __restrict__ Xi, int apply_elu,
                                                            const uint64_t* __restrict__ featmask, float scale,
                                                            const float* const* __restrict__ wtab, int U, int I, int nb_u,
                                                            float* __restrict__ dXu, float* __restrict__ dXi, int accumulate_dx,
                                                            float* __restrict__ partials) {
    extern __shared__ __align__(16) float smem[];
    float* WTs = smem;                       // [c][k] = W[k][c]
    float* dhs = smem + 64 * 64;             // [64][68]
    float* Xds = dhs + TB_TM * TB_XS;        // [64][68]
    float* dSs = Xds + TB_TM * TB_XS;        // [64][H]
    uint64_t* msk = reinterpret_cast<uint64_t*>(dSs + TB_TM * 8);   // [64]
    constexpr int DH = D / H;
    const bool item_side = (int)blockIdx.x >= nb_u;
    const int bs = item_side ? blockIdx.x - nb_u : blockIdx.x;
    const int nbs = item_side ? gridDim.x - nb_u : nb_u;
    const int rows_side = item_side ? I : U;
    const float* X = item_side ? Xi : Xu;
    float* dX = item_side ? dXi : dXu;
    const int64_t node_off = item_side ? U : 0;
    const int tiles = (rows_side + TB_TM - 1) / TB_TM;
    const float inv_scale = featmask ? 1.f / scale : 1.f;

    // WTs[c*64+k] = W[k][c]
    {
        const float* const* wptr = wtab + (item_side ? H : 0);
        for (int idx = threadIdx.x; idx < 64 * 16; idx += blockDim.x) {
            const int k = idx >> 4, c = (idx & 15) * 4;
            const float4 v = __ldg(reinterpret_cast<const float4*>(wptr[c / DH] + k * DH + (c % DH)));
            WTs[(c + 0) * 64 + k] = v.x; WTs[(c + 1) * 64 + k] = v.y; WTs[(c + 2) * 64 + k] = v.z; WTs[(c + 3) * 64 + k] = v.w;
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g8 = (warp & 1) * 8 + (lane >> 2);      // 0..15: row group of GEMM (a), k group of GEMM (b)
    const int c4 = (warp >> 1) * 4 + (lane & 3);      // 0..15: output column group (4 columns) of both GEMMs
    float accW[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) accW[i][0] = accW[i][1] = accW[i][2] = accW[i][3] = 0.f;
    const int qh = c4 & 7;
    const bool qhi = (c4 >> 3) != 0;
    float q[4] = {0.f, 0.f, 0.f, 0.f};   // H=1: Q[4*g8 + j]; H=8: q[0..1] = Q[4*g8 + 2*(c4>>3) + j][c4 & 7]

    for (int tile = bs; tile < tiles; tile += nbs) {
        const int row0 = tile * TB_TM;
        const int nrows = min(TB_TM, rows_side - row0);
        __syncthreads();
        for (int idx = threadIdx.x; idx < TB_TM * 16; idx += 256) {
            const int r = idx >> 4, qd = idx & 15;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f), x = v;
            if (r < nrows) {
                v = ld_stream4(dh + (node_off + row0 + r) * D + qd * 4);
                // same expression as transform_fwd: recomputes the dropped, activated stage input
                x = ld_stream4(X + (int64_t)(row0 + r) * D + qd * 4);
                if (apply_elu) { x.x = elu(x.x); x.y = elu(x.y); x.z = elu(x.z); x.w = elu(x.w); }
                if (featmask) {
                    uint32_t m = (uint32_t)(featmask[node_off + row0 + r] >> (qd * 4)) & 0xFu;
                    x.x = (m & 1u) ? x.x * scale : 0.f; x.y = (m & 2u) ? x.y * scale : 0.f;
                    x.z = (m & 4u) ? x.z * scale : 0.f; x.w = (m & 8u) ? x.w * scale : 0.f;
                }
            }
            *reinterpret_cast<float4*>(dhs + r * TB_XS + qd * 4) = v;
            *reinterpret_cast<float4*>(Xds + r * TB_XS + qd * 4) = x;
        }
        for (int idx = threadIdx.x; idx < TB_TM * H; idx += 256)
            dSs[idx] = idx < nrows * H ? __ldg(dS + (node_off + row0) * H + idx) : 0.f;
        if (threadIdx.x < TB_TM)
            msk[threadIdx.x] = (featmask && (int)threadIdx.x < nrows) ? featmask[node_off + row0 + threadIdx.x] : ~0ull;
        __syncthreads();

        // (a) dXd[r][k] = sum_c dh[r][c] * W[k][c]; thread = rows g8 + 16i, k = 4*c4 .. 4*c4+3
        {
            float acc[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
#pragma unroll 4
            for (int cc = 0; cc < 16; ++cc) {
                const float4 w0 = *reinterpret_cast<const float4*>(WTs + (cc * 4 + 0) * 64 + c4 * 4);
                const float4 w1 = *reinterpret_cast<const float4*>(WTs + (cc * 4 + 1) * 64 + c4 * 4);
                const float4 w2 = *reinterpret_cast<const float4*>(WTs + (cc * 4 + 2) * 64 + c4 * 4);
                const float4 w3 = *reinterpret_cast<const float4*>(WTs + (cc * 4 + 3) * 64 + c4 * 4);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 x = *reinterpret_cast<const float4*>(dhs + (g8 + 16 * i) * TB_XS + cc * 4);
                    acc[i][0] = fmaf(x.x, w0.x, acc[i][0]); acc[i][1] = fmaf(x.x, w0.y, acc[i][1]);
                    acc[i][2] = fmaf(x.x, w0.z, acc[i][2]); acc[i][3] = fmaf(x.x, w0.w, acc[i][3]);
                    acc[i][0] = fmaf(x.y, w1.x, acc[i][0]); acc[i][1] = fmaf(x.y, w1.y, acc[i][1]);
                    acc[i][2] = fmaf(x.y, w1.z, acc[i][2]); acc[i][3] = fmaf(x.y, w1.w, acc[i][3]);
                    acc[i][0] = fmaf(x.z, w2.x, acc[i][0]); acc[i][1] = fmaf(x.z, w2.y, acc[i][1]);
                    acc[i][2] = fmaf(x.z, w2.z, acc[i][2]); acc[i][3] = fmaf(x.z, w2.w, acc[i][3]);
                    acc[i][0] = fmaf(x.w, w3.x, acc[i][0]); acc[i][1] = fmaf(x.w, w3.y, acc[i][1]);
                    acc[i][2] = fmaf(x.w, w3.z, acc[i][2]); acc[i][3] = fmaf(x.w, w3.w, acc[i][3]);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = g8 + 16 * i;
                if (r >= nrows) continue;
                float4 v = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
                if (featmask) {
                    const uint32_t m = (uint32_t)(msk[r] >> (c4 * 4)) & 0xFu;
                    v.x = (m & 1u) ? v.x * scale : 0.f; v.y = (m & 2u) ? v.y * scale : 0.f;
                    v.z = (m & 4u) ? v.z * scale : 0.f; v.w = (m & 8u) ? v.w * scale : 0.f;
                }
                if (apply_elu) {   // the stage input was ELU(Zprev): chain through ELU' = 1 (e > 0) or e + 1 = exp(z)
                    const float4 e = *reinterpret_cast<const float4*>(Xds + r * TB_XS + c4 * 4);
                    const float ex = e.x * inv_scale, ey = e.y * inv_scale, ez = e.z * inv_scale, ew = e.w * inv_scale;
                    v.x *= ex > 0.f ? 1.f : ex + 1.f; v.y *= ey > 0.f ? 1.f : ey + 1.f;
                    v.z *= ez > 0.f ? 1.f : ez + 1.f; v.w *= ew > 0.f ? 1.f : ew + 1.f;
                }
                float* dst = dX + (int64_t)(row0 + r) * D + c4 * 4;
                if (accumulate_dx) {
                    const float4 o = *reinterpret_cast<const float4*>(dst);
                    v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                }
                *reinterpret_cast<float4*>(dst) = v;
            }
        }
        // (b) dW[k][c] += sum_r Xd[r][k] * dh[r][c], Q[k][hd] += sum_r Xd[r][k] * dS[r][hd]; thread = k 4*g8.., c 4*c4..
        //     (rows >= nrows are zero in all three tiles)
#pragma unroll 4
        for (int r = 0; r < TB_TM; ++r) {
            const float4 xs = *reinterpret_cast<const float4*>(Xds + r * TB_XS + g8 * 4);
            const float4 ds = *reinterpret_cast<const float4*>(dhs + r * TB_XS + c4 * 4);
            accW[0][0] = fmaf(xs.x, ds.x, accW[0][0]); accW[0][1] = fmaf(xs.x, ds.y, accW[0][1]);
            accW[0][2] = fmaf(xs.x, ds.z, accW[0][2]); accW[0][3] = fmaf(xs.x, ds.w, accW[0][3]);
            accW[1][0] = fmaf(xs.y, ds.x, accW[1][0]); accW[1][1] = fmaf(xs.y, ds.y, accW[1][1]);
            accW[1][2] = fmaf(xs.y, ds.z, accW[1][2]); accW[1][3] = fmaf(xs.y, ds.w, accW[1][3]);
            accW[2][0] = fmaf(xs.z, ds.x, accW[2][0]); accW[2][1] = fmaf(xs.z, ds.y, accW[2][1]);
            accW[2][2] = fmaf(xs.z, ds.z, accW[2][2]); accW[2][3] = fmaf(xs.z, ds.w, accW[2][3]);
            accW[3][0] = fmaf(xs.w, ds.x, accW[3][0]); accW[3][1] = fmaf(xs.w, ds.y, accW[3][1]);
            accW[3][2] = fmaf(xs.w, ds.z, accW[3][2]); accW[3][3] = fmaf(xs.w, ds.w, accW[3][3]);
            if (H == 1) {
                const float d = dSs[r];
                q[0] = fmaf(xs.x, d, q[0]); q[1] = fmaf(xs.y, d, q[1]); q[2] = fmaf(xs.z, d, q[2]); q[3] = fmaf(xs.w, d, q[3]);
            } else {
                const float d = dSs[r * 8 + qh];
                q[0] = fmaf(qhi ? xs.z : xs.x, d, q[0]);
                q[1] = fmaf(qhi ? xs.w : xs.y, d, q[1]);
            }
        }
    }
    float* part = partials + (size_t)blockIdx.x * TB_PART;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(part + (g8 * 4 + i) * 64 + c4 * 4) = make_float4(accW[i][0], accW[i][1], accW[i][2], accW[i][3]);
    // da partial of this block: da[c] = sum_k W[k][c] * Q[k][head(c)]
    __syncthreads();
    float* Qs = dhs;     // [64][H]
    if (H == 1) {
        if (c4 == 0) { Qs[g8 * 4 + 0] = q[0]; Qs[g8 * 4 + 1] = q[1]; Qs[g8 * 4 + 2] = q[2]; Qs[g8 * 4 + 3] = q[3]; }
    } else {
        const int k0 = g8 * 4 + (qhi ? 2 : 0);
        Qs[(k0 + 0) * 8 + qh] = q[0];
        Qs[(k0 + 1) * 8 + qh] = q[1];
    }
    __syncthreads();
    if (threadIdx.x < 64) {
        const int c = threadIdx.x, hd = c / DH;
        float a = 0.f;
#pragma unroll 8
        for (int k = 0; k < 64; ++k) a = fmaf(WTs[c * 64 + k], Qs[k * H + hd], a);
        part[64 * 64 + c] = a;
    }
}

// the fused dense backward for the two shapes of embedSize 128 (the same algorithm as transform_bwd_kernel above, whose 64 x 64 code
// is kept as tuned): (DIN, DOUT) = (128, 64) (first stage, 8 heads) and (64, 128) (last stage, 1 head); two CTAs per SM
template <int H, int DIN, int DOUT>
__global__ void __launch_bounds__(256, 2) transform_bwd_wide_kernel(const float* __restrict__ dh, const float* __restrict__ dS,
                                                            const float* __restrict__ Xu,
                                                            const float* __restrict__ Xi, int apply_elu,
                                                            const uint64_t* __restrict__ featmask, float scale,
                                                            const float* const* __restrict__ wtab, int U, int I, int nb_u,
                                                            float* __restrict__ dXu, float* __restrict__ dXi, int accumulate_dx,
                                                            float* __restrict__ partials) {
    constexpr int NK = DIN / 64, NC = DOUT / 64, MW = DIN / 64;     // 64-column groups of the input / output; mask words per row
    constexpr int XS_H = DOUT + 4, XS_X = DIN + 4;
    static_assert(NK + NC == 3, "(128, 64) or (64, 128)");
    extern __shared__ __align__(16) float smem[];
    float* WTs = smem;                       // [c][k] = W[k][c]
    float* dhs = smem + DOUT * DIN;          // [64][DOUT+4]
    float* Xds = dhs + TB_TM * XS_H;         // [64][DIN+4]
    float* dSs = Xds + TB_TM * XS_X;         // [64][H]
    uint64_t* msk = reinterpret_cast<uint64_t*>(dSs + TB_TM * 8);   // [64][MW]
    constexpr int DH = DOUT / H;
    const bool item_side = (int)blockIdx.x >= nb_u;
    const int bs = item_side ? blockIdx.x - nb_u : blockIdx.x;
    const int nbs = item_side ? gridDim.x - nb_u : nb_u;
    const int rows_side = item_side ? I : U;
    const float* X = item_side ? Xi : Xu;
    float* dX = item_side ? dXi : dXu;
    const int64_t node_off = item_side ? U : 0;
    const int tiles = (rows_side + TB_TM - 1) / TB_TM;
    const float inv_scale = featmask ? 1.f / scale : 1.f;

    // WTs[c*DIN+k] = W[k][c]
    {
        const float* const* wptr = wtab + (item_side ? H : 0);
        for (int idx = threadIdx.x; idx < DIN * DOUT / 4; idx += blockDim.x) {
            const int k = idx / (DOUT / 4), c = (idx % (DOUT / 4)) * 4;
            const float4 v = __ldg(reinterpret_cast<const float4*>(wptr[c / DH] + k * DH + (c % DH)));
            WTs[(c + 0) * DIN + k] = v.x; WTs[(c + 1) * DIN + k] = v.y; WTs[(c + 2) * DIN + k] = v.z; WTs[(c + 3) * DIN + k] = v.w;
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g8 = (warp & 1) * 8 + (lane >> 2);      // 0..15: row group of GEMM (a), k group of GEMM (b)
    const int c4 = (warp >> 1) * 4 + (lane & 3);      // 0..15: output column group (4 columns) of both GEMMs
    float accW[NK][NC][4][4];
#pragma unroll
    for (int a = 0; a < NK; ++a)
#pragma unroll
        for (int b = 0; b < NC; ++b)
#pragma unroll
            for (int i = 0; i < 4; ++i) accW[a][b][i][0] = accW[a][b][i][1] = accW[a][b][i][2] = accW[a][b][i][3] = 0.f;
    const int qh = c4 & 7;
    const bool qhi = (c4 >> 3) != 0;
    float q[NK][4];   // H=1: Q[64*a + 4*g8 + j]; H=8: q[a][0..1] = Q[64*a + 4*g8 + 2*(c4>>3) + j][c4 & 7]
#pragma unroll
    for (int a = 0; a < NK; ++a) q[a][0] = q[a][1] = q[a][2] = q[a][3] = 0.f;

    for (int tile = bs; tile < tiles; tile += nbs) {
        const int row0 = tile * TB_TM;
        const int nrows = min(TB_TM, rows_side - row0);
        __syncthreads();
        // dh tile (DOUT wide) and the recomputed stage input (DIN wide) -- the same expression as transform_fwd: the dropped,
        // activated input
        auto load_x = [&](int r, int qd) {
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < nrows) {
                x = ld_stream4(X + (int64_t)(row0 + r) * DIN + qd * 4);
                if (apply_elu) { x.x = elu(x.x); x.y = elu(x.y); x.z = elu(x.z); x.w = elu(x.w); }
                if (featmask) {
                    uint32_t m = (uint32_t)(featmask[(node_off + row0 + r) * MW + (qd >> 4)] >> ((qd & 15) * 4)) & 0xFu;
                    x.x = (m & 1u) ? x.x * scale : 0.f; x.y = (m & 2u) ? x.y * scale : 0.f;
                    x.z = (m & 4u) ? x.z * scale : 0.f; x.w = (m & 8u) ? x.w * scale : 0.f;
                }
            }
            *reinterpret_cast<float4*>(Xds + r * XS_X + qd * 4) = x;
        };
        for (int idx = threadIdx.x; idx < TB_TM * (DOUT / 4); idx += 256) {
            const int r = idx / (DOUT / 4), qd = idx % (DOUT / 4);
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < nrows) v = ld_stream4(dh + (node_off + row0 + r) * DOUT + qd * 4);
            *reinterpret_cast<float4*>(dhs + r * XS_H + qd * 4) = v;
        }
        for (int idx = threadIdx.x; idx < TB_TM * (DIN / 4); idx += 256) load_x(idx / (DIN / 4), idx % (DIN / 4));
        for (int idx = threadIdx.x; idx < TB_TM * H; idx += 256)
            dSs[idx] = idx < nrows * H ? __ldg(dS + (node_off + row0) * H + idx) : 0.f;
        for (int idx = threadIdx.x; idx < TB_TM * MW; idx += 256)
            msk[idx] = (featmask && idx / MW < nrows) ? featmask[(node_off + row0) * MW + idx] : ~0ull;
        __syncthreads();

        // (a) dXd[r][k] = sum_c dh[r][c] * W[k][c]; thread = rows g8 + 16i, k = 64*a + 4*c4 .. +3
        {
            float acc[4][NK][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int a = 0; a < NK; ++a) acc[i][a][0] = acc[i][a][1] = acc[i][a][2] = acc[i][a][3] = 0.f;
#pragma unroll 4
            for (int cc = 0; cc < DOUT / 4; ++cc) {
                float4 w0[NK], w1[NK], w2[NK], w3[NK];
#pragma unroll
                for (int a = 0; a < NK; ++a) {
                    w0[a] = *reinterpret_cast<const float4*>(WTs + (cc * 4 + 0) * DIN + 64 * a + c4 * 4);
                    w1[a] = *reinterpret_cast<const float4*>(WTs + (cc * 4 + 1) * DIN + 64 * a + c4 * 4);
                    w2[a] = *reinterpret_cast<const float4*>(WTs + (cc * 4 + 2) * DIN + 64 * a + c4 * 4);
                    w3[a] = *reinterpret_cast<const float4*>(WTs + (cc * 4 + 3) * DIN + 64 * a + c4 * 4);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 x = *reinterpret_cast<const float4*>(dhs + (g8 + 16 * i) * XS_H + cc * 4);
#pragma unroll
                    for (int a = 0; a < NK; ++a) {
                        float* ac = acc[i][a];
                        ac[0] = fmaf(x.x, w0[a].x, ac[0]); ac[1] = fmaf(x.x, w0[a].y, ac[1]);
                        ac[2] = fmaf(x.x, w0[a].z, ac[2]); ac[3] = fmaf(x.x, w0[a].w, ac[3]);
                        ac[0] = fmaf(x.y, w1[a].x, ac[0]); ac[1] = fmaf(x.y, w1[a].y, ac[1]);
                        ac[2] = fmaf(x.y, w1[a].z, ac[2]); ac[3] = fmaf(x.y, w1[a].w, ac[3]);
                        ac[0] = fmaf(x.z, w2[a].x, ac[0]); ac[1] = fmaf(x.z, w2[a].y, ac[1]);
                        ac[2] = fmaf(x.z, w2[a].z, ac[2]); ac[3] = fmaf(x.z, w2[a].w, ac[3]);
                        ac[0] = fmaf(x.w, w3[a].x, ac[0]); ac[1] = fmaf(x.w, w3[a].y, ac[1]);
                        ac[2] = fmaf(x.w, w3[a].z, ac[2]); ac[3] = fmaf(x.w, w3[a].w, ac[3]);
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = g8 + 16 * i;
                if (r >= nrows) continue;
#pragma unroll
                for (int a = 0; a < NK; ++a) {
                    const int k0 = 64 * a + c4 * 4;
                    float4 v = make_float4(acc[i][a][0], acc[i][a][1], acc[i][a][2], acc[i][a][3]);
                    if (featmask) {
                        const uint32_t m = (uint32_t)(msk[r * MW + a] >> (c4 * 4)) & 0xFu;
                        v.x = (m & 1u) ? v.x * scale : 0.f; v.y = (m & 2u) ? v.y * scale : 0.f;
                        v.z = (m & 4u) ? v.z * scale : 0.f; v.w = (m & 8u) ? v.w * scale : 0.f;
                    }
                    if (apply_elu) {   // the stage input was ELU(Zprev): chain through ELU' = 1 (e > 0) or e + 1 = exp(z)
                        const float4 e = *reinterpret_cast<const float4*>(Xds + r * XS_X + k0);
                        const float ex = e.x * inv_scale, ey = e.y * inv_scale, ez = e.z * inv_scale, ew = e.w * inv_scale;
                        v.x *= ex > 0.f ? 1.f : ex + 1.f; v.y *= ey > 0.f ? 1.f : ey + 1.f;
                        v.z *= ez > 0.f ? 1.f : ez + 1.f; v.w *= ew > 0.f ? 1.f : ew + 1.f;
                    }
                    float* dst = dX + (int64_t)(row0 + r) * DIN + k0;
                    if (accumulate_dx) {
                        const float4 o = *reinterpret_cast<const float4*>(dst);
                        v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                    }
                    *reinterpret_cast<float4*>(dst) = v;
                }
            }
        }
        // (b) dW[k][c] += sum_r Xd[r][k] * dh[r][c], Q[k][hd] += sum_r Xd[r][k] * dS[r][hd]; thread = k 64a+4*g8.., c 64b+4*c4..
        //     (rows >= nrows are zero in all three tiles)
#pragma unroll 4
        for (int r = 0; r < TB_TM; ++r) {
            float4 xs[NK], ds[NC];
#pragma unroll
            for (int a = 0; a < NK; ++a) xs[a] = *reinterpret_cast<const float4*>(Xds + r * XS_X + 64 * a + g8 * 4);
#pragma unroll
            for (int b = 0; b < NC; ++b) ds[b] = *reinterpret_cast<const float4*>(dhs + r * XS_H + 64 * b + c4 * 4);
#pragma unroll
            for (int a = 0; a < NK; ++a)
#pragma unroll
                for (int b = 0; b < NC; ++b) {
                    float (&w)[4][4] = accW[a][b];
                    w[0][0] = fmaf(xs[a].x, ds[b].x, w[0][0]); w[0][1] = fmaf(xs[a].x, ds[b].y, w[0][1]);
                    w[0][2] = fmaf(xs[a].x, ds[b].z, w[0][2]); w[0][3] = fmaf(xs[a].x, ds[b].w, w[0][3]);
                    w[1][0] = fmaf(xs[a].y, ds[b].x, w[1][0]); w[1][1] = fmaf(xs[a].y, ds[b].y, w[1][1]);
                    w[1][2] = fmaf(xs[a].y, ds[b].z, w[1][2]); w[1][3] = fmaf(xs[a].y, ds[b].w, w[1][3]);
                    w[2][0] = fmaf(xs[a].z, ds[b].x, w[2][0]); w[2][1] = fmaf(xs[a].z, ds[b].y, w[2][1]);
                    w[2][2] = fmaf(xs[a].z, ds[b].z, w[2][2]); w[2][3] = fmaf(xs[a].z, ds[b].w, w[2][3]);
                    w[3][0] = fmaf(xs[a].w, ds[b].x, w[3][0]); w[3][1] = fmaf(xs[a].w, ds[b].y, w[3][1]);
                    w[3][2] = fmaf(xs[a].w, ds[b].z, w[3][2]); w[3][3] = fmaf(xs[a].w, ds[b].w, w[3][3]);
                }
            if (H == 1) {
                const float d = dSs[r];
#pragma unroll
                for (int a = 0; a < NK; ++a) {
                    q[a][0] = fmaf(xs[a].x, d, q[a][0]); q[a][1] = fmaf(xs[a].y, d, q[a][1]);
                    q[a][2] = fmaf(xs[a].z, d, q[a][2]); q[a][3] = fmaf(xs[a].w, d, q[a][3]);
                }
            } else {
                const float d = dSs[r * 8 + qh];
#pragma unroll
                for (int a = 0; a < NK; ++a) {
                    q[a][0] = fmaf(qhi ? xs[a].z : xs[a].x, d, q[a][0]);
                    q[a][1] = fmaf(qhi ? xs[a].w : xs[a].y, d, q[a][1]);
                }
            }
        }
    }
    constexpr int PART = tb_part<DIN, DOUT>();
    float* part = partials + (size_t)blockIdx.x * PART;
#pragma unroll
    for (int a = 0; a < NK; ++a)
#pragma unroll
        for (int b = 0; b < NC; ++b)
#pragma unroll
            for (int i = 0; i < 4; ++i)
                *reinterpret_cast<float4*>(part + (64 * a + g8 * 4 + i) * DOUT + 64 * b + c4 * 4) =
                    make_float4(accW[a][b][i][0], accW[a][b][i][1], accW[a][b][i][2], accW[a][b][i][3]);
    // da partial of this block: da[c] = sum_k W[k][c] * Q[k][head(c)]
    __syncthreads();
    float* Qs = dhs;     // [DIN][H]
#pragma unroll
    for (int a = 0; a < NK; ++a) {
        if (H == 1) {
            if (c4 == 0) { Qs[64 * a + g8 * 4 + 0] = q[a][0]; Qs[64 * a + g8 * 4 + 1] = q[a][1]; Qs[64 * a + g8 * 4 + 2] = q[a][2]; Qs[64 * a + g8 * 4 + 3] = q[a][3]; }
        } else {
            const int k0 = 64 * a + g8 * 4 + (qhi ? 2 : 0);
            Qs[(k0 + 0) * 8 + qh] = q[a][0];
            Qs[(k0 + 1) * 8 + qh] = q[a][1];
        }
    }
    __syncthreads();
    if (threadIdx.x < DOUT) {
        const int c = threadIdx.x, hd = c / DH;
        float a = 0.f;
#pragma unroll 8
        for (int k = 0; k < DIN; ++k) a = fmaf(WTs[c * DIN + k], Qs[k * H + hd], a);
        part[DIN * DOUT + c] = a;
    }
}

// sums the block partials of each side and writes the per-head gradient tensors.  One CTA = 32 consecutive outputs x 8
// groups of partials (coalesced 128-byte loads, fixed summation order -> deterministic)
template <int H, int DIN = 64, int DOUT = 64>
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ partials, int nb_u, int nb_total,
                                                              float* const* __restrict__ gtab, int accumulate) {
    constexpr int DH = DOUT / H;
    constexpr int PART = tb_part<DIN, DOUT>();
    static_assert(PART % 32 == 0, "a CTA reduces 32 outputs of one side");
    __shared__ float red[8][33];
    const int og = threadIdx.x & 31, pg = threadIdx.x >> 5;
    const int idx = blockIdx.x * 32 + og;
    const int side = idx / PART, o = idx % PART;
    const int b0 = side ? nb_u : 0, b1 = side ? nb_total : nb_u;
    float sum = 0.f;
    for (int b = b0 + pg; b < b1; b += 8) sum += partials[(size_t)b * PART + o];
    red[pg][og] = sum;
    __syncthreads();
    if (pg != 0 || b1 <= b0) return;      // b1 <= b0: this call covered one side only (multi-GPU row sharding)
    sum = ((red[0][og] + red[1][og]) + (red[2][og] + red[3][og])) + ((red[4][og] + red[5][og]) + (red[6][og] + red[7][og]));
    float* dst;
    if (o < DIN * DOUT) {
        const int k = o / DOUT, c = o % DOUT;
        dst = gtab[side * H + c / DH] + k * DH + (c % DH);
    } else {
        const int c = o - DIN * DOUT;
        dst = gtab[2 * H + c / DH] + side * DH + (c % DH);
    }
    *dst = accumulate ? *dst + sum : sum;
}

}  // namespace ngacf

using namespace ngacf;

extern "C" int ngacf_stage_bwd_prep(const float* G, const float* Z, const float* h, const float* norm, int32_t H, int64_t N, float* Ghat,
                                    float* dN, void* stream) {
    NGACF_REQUIRE(G && Z && h && norm && Ghat && dN && N >= 0, "stage_bwd_prep: null argument");
    if (N == 0) return NGACF_OK;
    NGACF_REQUIRE(H == 1 || H == 8, "stage_bwd_prep: H must be 1 or 8");
    const int blocks = ceil_div(N * 16, 256);
    if (H == 8) stage_bwd_prep_kernel<8><<<blocks, 256, 0, (cudaStream_t)stream>>>(G, Z, h, norm, N, Ghat, dN);
    else        stage_bwd_prep_kernel<1><<<blocks, 256, 0, (cudaStream_t)stream>>>(G, Z, h, norm, N, Ghat, dN);
    return check_launch("stage_bwd_prep");
}

extern "C" int ngacf_stage_bwd_finalize(float* dh, const float* dS, const float* G, const float* const* wtab, int32_t H, int32_t item_side,
                                        int64_t n_rows, void* stream) {
    NGACF_REQUIRE(dh && dS && G && wtab && n_rows >= 0 && (H == 1 || H == 8), "stage_bwd_finalize: bad argument");
    if (n_rows == 0) return NGACF_OK;
    const int blocks = ceil_div(n_rows * 16, 256);
    if (H == 8) stage_bwd_finalize_kernel<8><<<blocks, 256, 0, (cudaStream_t)stream>>>(dh, dS, G, wtab, item_side, n_rows);
    else        stage_bwd_finalize_kernel<1><<<blocks, 256, 0, (cudaStream_t)stream>>>(dh, dS, G, wtab, item_side, n_rows);
    return check_launch("stage_bwd_finalize");
}

extern "C" int ngacf_stage_bwd_edges(int32_t mode, const int32_t* tasks, int32_t T_begin, int32_t T_end, const int32_t* adj_ptr,
                                     const int32_t* adj_idx, const int32_t* adj_eid, const int32_t* long_first_slot,
                                     int32_t* long_counter, float* scratch, const float* G, const float* Ghat, const float* dN,
                                     const float* h, const float* s, int32_t H, const uint8_t* edgemask, float scale,
                                     const float* const* wtab, int32_t U, float* ds_store, float* dh, float* dS, int32_t partial,
                                     void* stream) {
    NGACF_REQUIRE(tasks && adj_ptr && adj_idx && adj_eid && G && Ghat && dN && h && s && wtab && ds_store && dh && dS,
                  "stage_bwd_edges: null argument");
    NGACF_REQUIRE((mode == 0 || mode == 1) && (H == 1 || H == 8) && T_end >= T_begin, "stage_bwd_edges: bad mode/H/range");
    if (T_end == T_begin) return NGACF_OK;
    const int blocks = ceil_div((int64_t)(T_end - T_begin) * 16, 256);
    cudaStream_t st = (cudaStream_t)stream;
    const int4* tk = reinterpret_cast<const int4*>(tasks);
    static PerDeviceOnce once;
    once.run([] {
#define CARVE(HH, MM, DR) cudaFuncSetAttribute(stage_bwd_edges_kernel<HH, MM, DR, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 0)
        CARVE(8, 0, true); CARVE(8, 0, false); CARVE(8, 1, true); CARVE(8, 1, false);
        CARVE(1, 0, true); CARVE(1, 0, false); CARVE(1, 1, true); CARVE(1, 1, false);
#undef CARVE
    });
#define LAUNCH(HH, MM, DR, PA)                                                                                                              \
    stage_bwd_edges_kernel<HH, MM, DR, PA><<<blocks, 256, 0, st>>>(tk, T_begin, T_end, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, \
                                                                   scratch, G, Ghat, dN, h, s, edgemask, scale, wtab, U, ds_store, dh, dS)
    const bool dr = edgemask != nullptr;
    NGACF_REQUIRE(!(partial && mode == 0), "stage_bwd_edges: partial sums are produced by the item pass (mode 1) only");
    if (H == 8) {
        if (mode == 0) { if (dr) LAUNCH(8, 0, true, false); else LAUNCH(8, 0, false, false); }
        else if (partial) { if (dr) LAUNCH(8, 1, true, true); else LAUNCH(8, 1, false, true); }
        else           { if (dr) LAUNCH(8, 1, true, false); else LAUNCH(8, 1, false, false); }
    } else {
        if (mode == 0) { if (dr) LAUNCH(1, 0, true, false); else LAUNCH(1, 0, false, false); }
        else if (partial) { if (dr) LAUNCH(1, 1, true, true); else LAUNCH(1, 1, false, true); }
        else           { if (dr) LAUNCH(1, 1, true, false); else LAUNCH(1, 1, false, false); }
    }
#undef LAUNCH
    return check_launch("stage_bwd_edges");
}

static void transform_bwd_grid(int U, int I, int* nb_u, int* nb_i) {
    const int tiles_u = ceil_div(U, TB_TM), tiles_i = ceil_div(I, TB_TM);
    const int budget = TB_CTAS_PER_SM * 148;   // resident CTAs (54 KB of shared memory each; register-limited)
    int bu = (int)((int64_t)budget * tiles_u / (tiles_u + tiles_i > 0 ? tiles_u + tiles_i : 1));
    if (bu < 1) bu = 1;
    if (bu > tiles_u) bu = tiles_u;      // 0 when this call has no user rows
    int bi = budget - bu;
    if (bi < 1) bi = 1;
    if (bi > tiles_i) bi = tiles_i;
    *nb_u = bu;
    *nb_i = bi;
}

extern "C" size_t ngacf_transform_bwd_workspace_bytes(int32_t U, int32_t I) {
    int bu, bi;
    transform_bwd_grid(U, I, &bu, &bi);
    return (size_t)(bu + bi) * TB_PART * sizeof(float);
}

extern "C" int ngacf_transform_bwd(const float* dh, const float* dS, const float* h, const float* Xu, const float* Xi, int32_t apply_elu,
                                   const uint64_t* featmask, float scale, const float* const* wtab, float* const* gtab, int32_t H,
                                   int32_t U, int32_t I, float* dXu, float* dXi, int32_t accumulate_dx, int32_t accumulate_dw,
                                   void* workspace, size_t workspace_bytes, void* stream) {
    NGACF_REQUIRE(dh && dS && wtab && gtab && workspace && U >= 0 && I >= 0 && (U == 0 || (Xu && dXu)) && (I == 0 || (Xi && dXi)),
                  "transform_bwd: null argument");
    if (U + I == 0) return NGACF_OK;
    NGACF_REQUIRE(H == 1 || H == 8, "transform_bwd: H must be 1 or 8");
    if (workspace_bytes < ngacf_transform_bwd_workspace_bytes(U, I)) {
        set_error("transform_bwd: workspace too small");
        return NGACF_ERR_WORKSPACE;
    }
    int bu, bi;
    if (dense_on_tensor_cores()) {
        cudaStream_t st = (cudaStream_t)stream;
        transform_bwd_tc(dh, dS, Xu, Xi, apply_elu, featmask, scale, wtab, H, U, I, dXu, dXi, accumulate_dx, (float*)workspace, &bu, &bi, st);
        if (H == 8) reduce_partials_kernel<8><<<2 * TB_PART / 32, 256, 0, st>>>((float*)workspace, bu, bu + bi, gtab, accumulate_dw);
        else        reduce_partials_kernel<1><<<2 * TB_PART / 32, 256, 0, st>>>((float*)workspace, bu, bu + bi, gtab, accumulate_dw);
        return check_launch("transform_bwd(tc)");
    }
    transform_bwd_grid(U, I, &bu, &bi);
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(transform_bwd_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TB_SMEM);
        cudaFuncSetAttribute(transform_bwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TB_SMEM);
    });
    cudaStream_t st = (cudaStream_t)stream;
    float* partials = (float*)workspace;
    if (H == 8) {
        transform_bwd_kernel<8><<<bu + bi, 256, TB_SMEM, st>>>(dh, dS, Xu, Xi, apply_elu, featmask, scale, wtab, U, I, bu, dXu, dXi, accumulate_dx, partials);
        reduce_partials_kernel<8><<<2 * TB_PART / 32, 256, 0, st>>>(partials, bu, bu + bi, gtab, accumulate_dw);
    } else {
        transform_bwd_kernel<1><<<bu + bi, 256, TB_SMEM, st>>>(dh, dS, Xu, Xi, apply_elu, featmask, scale, wtab, U, I, bu, dXu, dXi, accumulate_dx, partials);
        reduce_partials_kernel<1><<<2 * TB_PART / 32, 256, 0, st>>>(partials, bu, bu + bi, gtab, accumulate_dw);
    }
    return check_launch("transform_bwd");
}

// ------------------------------------------------------------------------------------------------
// width-carrying entry points: width / (d_in, d_out) = 64 reach the calls above (the same kernels); 128-wide single-head rows and
// the two dense shapes of embedSize 128 run the W = 128 instantiations (dense: CUDA-core kernels).
// ------------------------------------------------------------------------------------------------
extern "C" int ngacf_stage_bwd_prep_w(const float* G, const float* Z, const float* h, const float* norm, int32_t H, int32_t width, int64_t N,
                                      float* Ghat, float* dN, void* stream) {
    if (width == 64) return ngacf_stage_bwd_prep(G, Z, h, norm, H, N, Ghat, dN, stream);
    if (width != 128 || H != 1) {
        set_error("stage_bwd_prep_w: (H, width) = (%d, %d) is not built; 128-wide rows: H = 1", H, width);
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(G && Z && h && norm && Ghat && dN && N >= 0, "stage_bwd_prep_w: null argument");
    if (N == 0) return NGACF_OK;
    stage_bwd_prep_wide_kernel<128><<<ceil_div(N * 16, 256), 256, 0, (cudaStream_t)stream>>>(G, Z, h, norm, N, Ghat, dN);
    return check_launch("stage_bwd_prep_w");
}

extern "C" int ngacf_stage_bwd_edges_w(int32_t mode, const int32_t* tasks, int32_t T_begin, int32_t T_end, const int32_t* adj_ptr,
                                       const int32_t* adj_idx, const int32_t* adj_eid, const int32_t* long_first_slot,
                                       int32_t* long_counter, float* scratch, const float* G, const float* Ghat, const float* dN,
                                       const float* h, const float* s, int32_t H, int32_t width, const uint8_t* edgemask, float scale,
                                       const float* const* wtab, int32_t U, float* ds_store, float* dh, float* dS, int32_t partial,
                                       void* stream) {
    if (width == 64)
        return ngacf_stage_bwd_edges(mode, tasks, T_begin, T_end, adj_ptr, adj_idx, adj_eid, long_first_slot, long_counter, scratch, G, Ghat,
                                     dN, h, s, H, edgemask, scale, wtab, U, ds_store, dh, dS, partial, stream);
    if (width != 128 || H != 1 || partial) {
        set_error("stage_bwd_edges_w: (H, width) = (%d, %d)%s is not built; 128-wide rows: H = 1, full rows", H, width,
                  partial ? " with partial rows" : "");
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(tasks && adj_ptr && adj_idx && adj_eid && G && Ghat && dN && h && s && wtab && ds_store && dh && dS,
                  "stage_bwd_edges_w: null argument");
    NGACF_REQUIRE((mode == 0 || mode == 1) && T_end >= T_begin, "stage_bwd_edges_w: bad mode/range");
    if (T_end == T_begin) return NGACF_OK;
    const int blocks = ceil_div((int64_t)(T_end - T_begin) * 16, 256);
    cudaStream_t st = (cudaStream_t)stream;
    const int4* tk = reinterpret_cast<const int4*>(tasks);
    static PerDeviceOnce once;
    once.run([] {
#define CARVE(MM, DR) cudaFuncSetAttribute(stage_bwd_edges_wide_kernel<MM, DR, 128>, cudaFuncAttributePreferredSharedMemoryCarveout, 0)
        CARVE(0, true); CARVE(0, false); CARVE(1, true); CARVE(1, false);
#undef CARVE
    });
#define LAUNCH(MM, DR)                                                                                                                      \
    stage_bwd_edges_wide_kernel<MM, DR, 128><<<blocks, 256, 0, st>>>(tk, T_begin, T_end, adj_ptr, adj_idx, adj_eid, long_first_slot,      \
                                                                          long_counter, scratch, G, Ghat, dN, h, s, edgemask, scale, wtab, U, \
                                                                          ds_store, dh, dS)
    const bool dr = edgemask != nullptr;
    if (mode == 0) { if (dr) LAUNCH(0, true); else LAUNCH(0, false); }
    else           { if (dr) LAUNCH(1, true); else LAUNCH(1, false); }
#undef LAUNCH
    return check_launch("stage_bwd_edges_w");
}

static bool dense_shape_wide(int H, int d_in, int d_out) { return (H == 8 && d_in == 128 && d_out == 64) || (H == 1 && d_in == 64 && d_out == 128); }

static void transform_bwd_grid_wide(int U, int I, int* nb_u, int* nb_i) {
    const int tiles_u = ceil_div(U, TB_TM), tiles_i = ceil_div(I, TB_TM);
    const int budget = 2 * 148;      // transform_bwd_wide_kernel: two resident CTAs per SM (87 KB of shared memory, 128 registers)
    int bu = (int)((int64_t)budget * tiles_u / (tiles_u + tiles_i > 0 ? tiles_u + tiles_i : 1));
    if (bu < 1) bu = 1;
    if (bu > tiles_u) bu = tiles_u;
    int bi = budget - bu;
    if (bi < 1) bi = 1;
    if (bi > tiles_i) bi = tiles_i;
    *nb_u = bu;
    *nb_i = bi;
}

extern "C" size_t ngacf_transform_bwd_workspace_bytes_w(int32_t d_in, int32_t d_out, int32_t U, int32_t I) {
    if (d_in == 64 && d_out == 64) return ngacf_transform_bwd_workspace_bytes(U, I);
    // one partial of d_in * d_out + d_out floats per block: (128, 64) -> 8256, (64, 128) -> 8320
    size_t part;
    if (d_in == 128 && d_out == 64) part = tb_part<128, 64>();
    else if (d_in == 64 && d_out == 128) part = tb_part<64, 128>();
    else return 0;                                                   // not built: ngacf_transform_bwd_w refuses the shape
    int bu, bi;
    transform_bwd_grid_wide(U, I, &bu, &bi);
    return (size_t)(bu + bi) * part * sizeof(float);
}

template <int H, int DIN, int DOUT>
static void launch_transform_bwd_wide(const float* dh, const float* dS, const float* Xu, const float* Xi, int apply_elu, const uint64_t* featmask,
                                      float scale, const float* const* wtab, float* const* gtab, int U, int I, float* dXu, float* dXi,
                                      int accumulate_dx, int accumulate_dw, float* partials, cudaStream_t st) {
    constexpr size_t SMEM = (size_t)tb_smem_floats<DIN, DOUT>() * sizeof(float);
    static PerDeviceOnce once;
    once.run([] { cudaFuncSetAttribute(transform_bwd_wide_kernel<H, DIN, DOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM); });
    int bu, bi;
    transform_bwd_grid_wide(U, I, &bu, &bi);
    transform_bwd_wide_kernel<H, DIN, DOUT><<<bu + bi, 256, SMEM, st>>>(dh, dS, Xu, Xi, apply_elu, featmask, scale, wtab, U, I, bu, dXu, dXi,
                                                                   accumulate_dx, partials);
    reduce_partials_kernel<H, DIN, DOUT><<<2 * tb_part<DIN, DOUT>() / 32, 256, 0, st>>>(partials, bu, bu + bi, gtab, accumulate_dw);
}

extern "C" int ngacf_transform_bwd_w(const float* dh, const float* dS, const float* h, const float* Xu, const float* Xi, int32_t apply_elu,
                                     const uint64_t* featmask, float scale, const float* const* wtab, float* const* gtab, int32_t H,
                                     int32_t d_in, int32_t d_out, int32_t U, int32_t I, float* dXu, float* dXi, int32_t accumulate_dx,
                                     int32_t accumulate_dw, void* workspace, size_t workspace_bytes, void* stream) {
    if (d_in == 64 && d_out == 64)
        return ngacf_transform_bwd(dh, dS, h, Xu, Xi, apply_elu, featmask, scale, wtab, gtab, H, U, I, dXu, dXi, accumulate_dx, accumulate_dw,
                                   workspace, workspace_bytes, stream);
    if (!dense_shape_wide(H, d_in, d_out)) {
        set_error("transform_bwd_w: (H, d_in, d_out) = (%d, %d, %d) is not built; supported: (1|8, 64, 64), (8, 128, 64), (1, 64, 128)", H,
                  d_in, d_out);
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(dh && dS && wtab && gtab && workspace && U >= 0 && I >= 0 && (U == 0 || (Xu && dXu)) && (I == 0 || (Xi && dXi)),
                  "transform_bwd_w: null argument");
    if (U + I == 0) return NGACF_OK;
    if (workspace_bytes < ngacf_transform_bwd_workspace_bytes_w(d_in, d_out, U, I)) {
        set_error("transform_bwd_w: workspace too small");
        return NGACF_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (H == 8)
        launch_transform_bwd_wide<8, 128, 64>(dh, dS, Xu, Xi, apply_elu, featmask, scale, wtab, gtab, U, I, dXu, dXi, accumulate_dx, accumulate_dw,
                                              (float*)workspace, st);
    else
        launch_transform_bwd_wide<1, 64, 128>(dh, dS, Xu, Xi, apply_elu, featmask, scale, wtab, gtab, U, I, dXu, dXi, accumulate_dx, accumulate_dw,
                                              (float*)workspace, st);
    return check_launch("transform_bwd_w");
}
