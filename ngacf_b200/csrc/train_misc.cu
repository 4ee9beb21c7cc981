// Pair scoring + BPR loss + gradient scatter, table-driven Adam, PairSampling sampler.
// Reference: graphattention/SPUIGACF.py:49-52, graphattention/BPRLoss.py:8-9,
// train_eval_Gowalla.py:117-138, data/loadGowalla.py:63-77, run_Gowalla.py:114.
#include "common.cuh"

namespace ngacf {

// fixed summation tree of the 64-wide dot product (oracle/port.py:dot64_tree): products rounded to
// fp32 (no FMA contraction), adjacent pairs first, then lanes 1,2,4,8.
__device__ __forceinline__ float dot64_tree(float4 a, float4 b, unsigned gm) {
    float p0 = __fmul_rn(a.x, b.x), p1 = __fmul_rn(a.y, b.y), p2 = __fmul_rn(a.z, b.z), p3 = __fmul_rn(a.w, b.w);
    float v = __fadd_rn(__fadd_rn(p0, p1), __fadd_rn(p2, p3));
    v = __fadd_rn(v, __shfl_xor_sync(gm, v, 1, 16));
    v = __fadd_rn(v, __shfl_xor_sync(gm, v, 2, 16));
    v = __fadd_rn(v, __shfl_xor_sync(gm, v, 4, 16));
    v = __fadd_rn(v, __shfl_xor_sync(gm, v, 8, 16));
    return v;
}

// the same adjacent-pair tree over 128 products (oracle/port.py:dot64_tree, whose tree is generic over the length): lane l holds
// columns 8l .. 8l+7 as two float4, levels 1-3 in the lane, levels 4-7 across the lanes
__device__ __forceinline__ float dot128_tree(const float4 (&a)[2], const float4 (&b)[2], unsigned gm) {
    float q[2];
#pragma unroll
    for (int v = 0; v < 2; ++v) {
        const float p0 = __fmul_rn(a[v].x, b[v].x), p1 = __fmul_rn(a[v].y, b[v].y), p2 = __fmul_rn(a[v].z, b[v].z), p3 = __fmul_rn(a[v].w, b[v].w);
        q[v] = __fadd_rn(__fadd_rn(p0, p1), __fadd_rn(p2, p3));
    }
    float v = __fadd_rn(q[0], q[1]);
    v = __fadd_rn(v, __shfl_xor_sync(gm, v, 1, 16));
    v = __fadd_rn(v, __shfl_xor_sync(gm, v, 2, 16));
    v = __fadd_rn(v, __shfl_xor_sync(gm, v, 4, 16));
    v = __fadd_rn(v, __shfl_xor_sync(gm, v, 8, 16));
    return v;
}

__device__ __forceinline__ float4 elu4(float4 z) { return make_float4(elu(z.x), elu(z.y), elu(z.z), elu(z.w)); }

__global__ void __launch_bounds__(256) score_pairs_kernel(const float* __restrict__ Z, int U, const int64_t* __restrict__ users,
                                                          const int64_t* __restrict__ items, int B, float* __restrict__ scores) {
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    if (b >= B) return;
    const int lane16 = threadIdx.x & 15;
    const unsigned gm = group_mask();
    const int64_t u = users[b], it = items[b] + U;
    const float4 fu = elu4(ld_gather4(Z + u * D + lane16 * 4));
    const float4 fi = elu4(ld_gather4(Z + it * D + lane16 * 4));
    const float sc = dot64_tree(fu, fi, gm);
    if (lane16 == 0) scores[b] = sc;
}

__global__ void __launch_bounds__(256) score_pairs128_kernel(const float* __restrict__ Z, int U, const int64_t* __restrict__ users,
                                                             const int64_t* __restrict__ items, int B, float* __restrict__ scores) {
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    if (b >= B) return;
    const int lane16 = threadIdx.x & 15;
    const unsigned gm = group_mask();
    const int64_t u = users[b], it = items[b] + U;
    float4 fu[2], fi[2];
#pragma unroll
    for (int v = 0; v < 2; ++v) {
        fu[v] = elu4(ld_gather4(Z + u * 128 + lane16 * 8 + 4 * v));
        fi[v] = elu4(ld_gather4(Z + it * 128 + lane16 * 8 + 4 * v));
    }
    const float sc = dot128_tree(fu, fi, gm);
    if (lane16 == 0) scores[b] = sc;
}

__global__ void final_features_kernel(const float* __restrict__ Z, int64_t n4, float* __restrict__ F) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    st_stream4(F + i * 4, elu4(ld_stream4(Z + i * 4)));
}

// Gradient scatter of the pair scores, deterministic and atomic-free.
// entry e in [0,2B): e<B -> (row = users[e], other = U+items[e]); else (row = U+items[e-B], other = users[e-B]).
// One CTA per entry; only the CTA of the FIRST entry of each distinct row survives.  It reads 2048 keys of the batch at once
// (eight independent loads per thread: one memory round trip), leaves if an earlier entry owns the row, compacts the matching
// entries in batch order, and its 16 lane-groups gather the matching rows in parallel (4 loads in flight each); the 16 partial
// sums are combined in a fixed order.  A PairSampling batch is user-sorted, so a heavy user can own a whole batch: this keeps
// that case parallel.
// W: row width (64, or 128 at embedSize 128: lane l owns columns 8l .. 8l+7)
constexpr int SPB_SUPER = 2048;
template <int W = 64>
__global__ void __launch_bounds__(256) score_pairs_bwd_kernel(const float* __restrict__ Z, int U, const int64_t* __restrict__ users,
                                                              const int64_t* __restrict__ items, const float* __restrict__ dscore, int B,
                                                              float* __restrict__ G, int accumulate) {
    __shared__ int list[SPB_SUPER];
    __shared__ int warp_cnt[8][8];
    constexpr int V = W / 64;
    __shared__ float part[16][W];
    const int e = blockIdx.x;
    const bool user_row = e < B;
    const int eb = user_row ? e : e - B;
    const int64_t* keys = user_row ? users : items;      // only entries of the same kind can match
    const int64_t* others = user_row ? items : users;
    const int64_t key = keys[eb];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int grp = tid >> 4, lane16 = tid & 15;
    float4 acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int sbase = 0; sbase < B; sbase += SPB_SUPER) {
        int64_t kreg[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int j = sbase + c * 256 + tid;
            kreg[c] = j < B ? keys[j] : (int64_t)-1;
        }
        unsigned mbits = 0;
        bool earlier = false;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int j = sbase + c * 256 + tid;
            const bool m = kreg[c] == key;                   // ids are non-negative: the -1 padding never matches
            mbits |= (unsigned)m << c;
            earlier |= m && j < eb;
        }
        if (__syncthreads_or(earlier)) return;               // an earlier entry owns this row (block-uniform)
        unsigned bal[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            bal[c] = __ballot_sync(0xffffffffu, (mbits >> c) & 1u);
            if (lane == 0) warp_cnt[c][warp] = __popc(bal[c]);
        }
        __syncthreads();
        int total = 0;
#pragma unroll
        for (int c = 0; c < 8; ++c) {                        // batch order: chunk, warp, lane
            int off = total;
#pragma unroll
            for (int w = 0; w < 8; ++w) { const int cw = warp_cnt[c][w]; if (w < warp) off += cw; total += cw; }
            if ((mbits >> c) & 1u) list[off + __popc(bal[c] & ((1u << lane) - 1u))] = sbase + c * 256 + tid;
        }
        __syncthreads();
        for (int q0 = grp; q0 < total; q0 += 64) {           // group g takes matches g, g+16, g+32, g+48 per round
            int jj[4]; float c[4]; float4 f[4][V];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int qi = q0 + 16 * q;
                jj[q] = qi < total ? list[qi] : -1;
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (jj[q] >= 0) {
                    const int64_t other = others[jj[q]] + (user_row ? U : 0);
                    c[q] = dscore[jj[q]];
#pragma unroll
                    for (int v = 0; v < V; ++v) f[q][v] = ld_gather4(Z + other * W + lane16 * 4 * V + 4 * v);
                } else {
                    c[q] = 0.f;
#pragma unroll
                    for (int v = 0; v < V; ++v) f[q][v] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const float4 fo = elu4(f[q][v]);
                    float4& a = acc[v];
                    a.x = fmaf(c[q], fo.x, a.x); a.y = fmaf(c[q], fo.y, a.y); a.z = fmaf(c[q], fo.z, a.z); a.w = fmaf(c[q], fo.w, a.w);
                }
            }
        }
        __syncthreads();                                      // list is rewritten by the next 2048 keys
    }
#pragma unroll
    for (int v = 0; v < V; ++v) *reinterpret_cast<float4*>(&part[grp][lane16 * 4 * V + 4 * v]) = acc[v];
    __syncthreads();
    if (tid < W) {
        float sum = 0.f;
#pragma unroll
        for (int g = 0; g < 16; ++g) sum += part[g][tid];
        const int64_t row = user_row ? key : key + U;
        const float gnew = sum * elu_grad(Z[row * W + tid]);
        G[row * W + tid] = accumulate ? G[row * W + tid] + gnew : gnew;
    }
}

// single-block loss: deterministic tree reduction
__global__ void __launch_bounds__(1024) bpr_loss_kernel(const float* __restrict__ pos, const float* __restrict__ neg, int B, float gscale,
                                                        float* __restrict__ loss, float* __restrict__ dpos, float* __restrict__ dneg,
                                                        const int64_t* __restrict__ users, int64_t u_lo, int64_t u_hi) {
    __shared__ float red[32];
    float local = 0.f;
    const float invB = 1.0f / (float)B;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        if (users && (users[b] < u_lo || users[b] >= u_hi)) {      // multi-GPU: the pair belongs to another rank's users
            if (dpos) dpos[b] = 0.f;
            if (dneg) dneg[b] = 0.f;
            continue;
        }
        const float x = pos[b] - neg[b];
        // -log(sigmoid(x)) = softplus(-x), stable form (BPRLoss.py:9 is the naive form)
        local += fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));
        const float sg = 1.0f / (1.0f + expf(x));          // sigmoid(-x)
        const float d = -sg * invB * gscale;
        if (dpos) dpos[b] = d;
        if (dneg) dneg[b] = -d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0 && loss) *loss = v * invB;
    }
}

// ------------------------------------------------------------------------------------------------
// Adam
// ------------------------------------------------------------------------------------------------
struct AdamEntry { float* p; const float* g; float* m; float* v; int64_t numel; };
constexpr int ADAM_MAX_TENSORS = 64;

__global__ void __launch_bounds__(256, 4) adam_kernel(const AdamEntry* __restrict__ tab, int n_tensors, float lr_over_bc1, float inv_sqrt_bc2,
                                                   const double* __restrict__ state, float beta1, float beta2, float eps, float wd) {
    if (state) { lr_over_bc1 = (float)state[1]; inv_sqrt_bc2 = (float)state[2]; }
    __shared__ AdamEntry ent[ADAM_MAX_TENSORS];
    __shared__ int64_t pref[ADAM_MAX_TENSORS + 1];   // prefix in float4 chunks
    if (threadIdx.x < n_tensors) ent[threadIdx.x] = tab[threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t run = 0;
        for (int t = 0; t < n_tensors; ++t) { pref[t] = run; run += (ent[t].numel + 3) / 4; }
        pref[n_tensors] = run;
    }
    __syncthreads();
    const int64_t total = pref[n_tensors];
    // a thread's chunk index only grows: one binary search, then a forward scan (almost always zero steps -- two tensors hold
    // 99.8 % of the chunks); the search per chunk was a third of the kernel's instruction stream (ncu: 350 instructions per
    // warp and chunk, issue-bound at 4 CTAs/SM)
    int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int lo = 0;
    {
        int hi = n_tensors - 1;
        while (lo < hi) {
            int mid = (lo + hi + 1) >> 1;
            if (pref[mid] <= c) lo = mid; else hi = mid - 1;
        }
    }
    for (; c < total; c += (int64_t)gridDim.x * blockDim.x) {
        while (c >= pref[lo + 1]) ++lo;
        const AdamEntry& en = ent[lo];
        const int64_t off = (c - pref[lo]) * 4;
        const int cnt = (int)min((int64_t)4, en.numel - off);
        float pv[4], gv[4], mv[4], vv[4];
        if (cnt == 4) {
            float4 a = *reinterpret_cast<const float4*>(en.p + off), b = *reinterpret_cast<const float4*>(en.g + off);
            float4 mm = *reinterpret_cast<const float4*>(en.m + off), v2 = *reinterpret_cast<const float4*>(en.v + off);
            pv[0] = a.x; pv[1] = a.y; pv[2] = a.z; pv[3] = a.w; gv[0] = b.x; gv[1] = b.y; gv[2] = b.z; gv[3] = b.w;
            mv[0] = mm.x; mv[1] = mm.y; mv[2] = mm.z; mv[3] = mm.w; vv[0] = v2.x; vv[1] = v2.y; vv[2] = v2.z; vv[3] = v2.w;
        } else {
            for (int k = 0; k < cnt; ++k) { pv[k] = en.p[off + k]; gv[k] = en.g[off + k]; mv[k] = en.m[off + k]; vv[k] = en.v[off + k]; }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (k < cnt) {
                const float g = fmaf(wd, pv[k], gv[k]);                 // L2 weight decay added to the gradient
                mv[k] = fmaf(beta1, mv[k], (1.f - beta1) * g);
                vv[k] = fmaf(beta2, vv[k], (1.f - beta2) * g * g);
                const float denom = sqrtf(vv[k]) * inv_sqrt_bc2 + eps;
                pv[k] = pv[k] - lr_over_bc1 * (mv[k] / denom);
            }
        }
        if (cnt == 4) {
            *reinterpret_cast<float4*>(en.p + off) = make_float4(pv[0], pv[1], pv[2], pv[3]);
            *reinterpret_cast<float4*>(en.m + off) = make_float4(mv[0], mv[1], mv[2], mv[3]);
            *reinterpret_cast<float4*>(en.v + off) = make_float4(vv[0], vv[1], vv[2], vv[3]);
        } else {
            for (int k = 0; k < cnt; ++k) { en.p[off + k] = pv[k]; en.m[off + k] = mv[k]; en.v[off + k] = vv[k]; }
        }
    }
}

// device-resident step counter variant (CUDA-graph replayable): state = double[4] {step, lr/bc1, 1/sqrt(bc2), -}
__global__ void adam_tick_kernel(double* state, double lr, double beta1, double beta2) {
    const double t = state[0] + 1.0;
    state[0] = t;
    state[1] = lr / (1.0 - pow(beta1, t));
    state[2] = 1.0 / sqrt(1.0 - pow(beta2, t));
}

// ------------------------------------------------------------------------------------------------
// PairSampling sampler (oracle/port.py:sample_pairs)
// ------------------------------------------------------------------------------------------------
constexpr uint32_t SAMPLER_TAG = 0x5A17u;

__global__ void sample_pairs_kernel(const int* __restrict__ rows_user, const int* __restrict__ train_ptr, const int* __restrict__ train_items,
                                    const int* __restrict__ train_rank, const int* __restrict__ pool, int P, int64_t row_begin, int64_t n,
                                    const int64_t* __restrict__ row_dev, uint32_t k0, uint32_t k1, uint32_t epoch, int64_t* __restrict__ users, int64_t* __restrict__ pos,
                                    int64_t* __restrict__ neg) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    if (row_dev) { row_begin += row_dev[0]; epoch += (uint32_t)row_dev[1]; }
    const uint64_t r = (uint64_t)(row_begin + b);
    uint32_t w[4];
    philox4x32_10((uint32_t)r, (uint32_t)(r >> 32), epoch, SAMPLER_TAG, k0, k1, w);
    const int u = rows_user[row_begin + b];
    const int beg = train_ptr[u], deg = train_ptr[u + 1] - beg;
    users[b] = u;
    const uint32_t pidx = __umulhi(w[0], (uint32_t)deg);
    pos[b] = train_items[beg + (int)pidx];
    const int nneg = P - deg;
    if (nneg <= 0) { neg[b] = -1; return; }
    const int k = (int)__umulhi(w[1], (uint32_t)nneg);
    int lo = 0, hi = deg;                      // smallest j with rank[j]-j > k
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (train_rank[beg + mid] - mid <= k) lo = mid + 1; else hi = mid;
    }
    neg[b] = pool[k + lo];
}

__global__ void counter_add_kernel(int64_t* c, int64_t d) { *c += d; }

// Multi-GPU pair scoring: the rows of the batch live on their owners.  gather: Zb[b] = Z[users[b]] / Zb[B+b] = Z[U+items[b]] if this
// rank owns the row (users [u_lo,u_hi), items [i_lo,i_hi)), zeros otherwise -- summing Zb over the ranks (one all-reduce) yields
// every batch row exactly (a row has one owner).  scatter: the summed rows are written back into a table at their global positions
// so that ngacf_score_pairs(_bwd) run unchanged on every rank.
__global__ void __launch_bounds__(256) batch_rows_gather_kernel(const float* __restrict__ Z, int U, const int64_t* __restrict__ users,
                                                                const int64_t* __restrict__ items, int B, int64_t u_lo, int64_t u_hi,
                                                                int64_t i_lo, int64_t i_hi, float* __restrict__ Zb) {
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    if (e >= 2 * B) return;
    const int lane16 = threadIdx.x & 15;
    const bool user_row = e < B;
    const int64_t id = user_row ? users[e] : items[e - B];
    const bool own = user_row ? (id >= u_lo && id < u_hi) : (id >= i_lo && id < i_hi);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (own) v = ld_gather4(Z + (user_row ? id : id + U) * D + lane16 * 4);
    *reinterpret_cast<float4*>(Zb + (int64_t)e * D + lane16 * 4) = v;
}

__global__ void __launch_bounds__(256) batch_rows_scatter_kernel(const float* __restrict__ Zb, int U, const int64_t* __restrict__ users,
                                                                 const int64_t* __restrict__ items, int B, float* __restrict__ Z) {
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    if (e >= 2 * B) return;
    const int lane16 = threadIdx.x & 15;
    const bool user_row = e < B;
    const int64_t row = user_row ? users[e] : items[e - B] + U;
    *reinterpret_cast<float4*>(Z + row * D + lane16 * 4) = *reinterpret_cast<const float4*>(Zb + (int64_t)e * D + lane16 * 4);   // duplicates write the same row
}

// end-of-step bookkeeping of a captured step in one launch: epoch loss accumulator and train-row cursor
__global__ void step_counters_kernel(double* total, const float* __restrict__ loss, int64_t* row_dev, int64_t row_stride) {
    if (total && loss) *total += (double)*loss;
    if (row_dev) row_dev[0] += row_stride;
}


}  // namespace ngacf

using namespace ngacf;

extern "C" int ngacf_counter_add(int64_t* counter, int64_t delta, void* stream) {
    NGACF_REQUIRE(counter, "counter_add: null argument");
    counter_add_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter, delta);
    return check_launch("counter_add");
}

extern "C" int ngacf_batch_rows_gather(const float* Z, int32_t U, const int64_t* users, const int64_t* items, int32_t B, int64_t u_lo, int64_t u_hi,
                                       int64_t i_lo, int64_t i_hi, float* Zb, void* stream) {
    NGACF_REQUIRE(Z && users && items && Zb && B >= 0, "batch_rows_gather: bad argument");
    if (B == 0) return NGACF_OK;
    batch_rows_gather_kernel<<<ceil_div((int64_t)2 * B * 16, 256), 256, 0, (cudaStream_t)stream>>>(Z, U, users, items, B, u_lo, u_hi, i_lo, i_hi, Zb);
    return check_launch("batch_rows_gather");
}

extern "C" int ngacf_batch_rows_scatter(const float* Zb, int32_t U, const int64_t* users, const int64_t* items, int32_t B, float* Z, void* stream) {
    NGACF_REQUIRE(Z && users && items && Zb && B >= 0, "batch_rows_scatter: bad argument");
    if (B == 0) return NGACF_OK;
    batch_rows_scatter_kernel<<<ceil_div((int64_t)2 * B * 16, 256), 256, 0, (cudaStream_t)stream>>>(Zb, U, users, items, B, Z);
    return check_launch("batch_rows_scatter");
}

extern "C" int ngacf_memset_zero(void* p, size_t bytes, void* stream) {
    NGACF_REQUIRE(p || bytes == 0, "memset_zero: null pointer");
    if (bytes == 0) return NGACF_OK;
    cudaMemsetAsync(p, 0, bytes, (cudaStream_t)stream);
    return check_launch("memset_zero");
}

extern "C" int ngacf_step_counters(double* total, const float* loss, int64_t* row_dev, int64_t row_stride, void* stream) {
    NGACF_REQUIRE((total && loss) || row_dev, "step_counters: nothing to do");
    step_counters_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(total, loss, row_dev, row_stride);
    return check_launch("step_counters");
}

extern "C" int ngacf_score_pairs(const float* Z, int32_t U, const int64_t* users, const int64_t* items, int32_t B, float* scores, void* stream) {
    NGACF_REQUIRE(Z && users && items && scores && B >= 0, "score_pairs: null argument");
    if (B == 0) return NGACF_OK;
    score_pairs_kernel<<<ceil_div((int64_t)B * 16, 256), 256, 0, (cudaStream_t)stream>>>(Z, U, users, items, B, scores);
    return check_launch("score_pairs");
}

extern "C" int ngacf_final_features(const float* Z, int64_t N, float* F, void* stream) {
    NGACF_REQUIRE(Z && F && N >= 0, "final_features: null argument");
    if (N == 0) return NGACF_OK;
    final_features_kernel<<<ceil_div(N * 16, 256), 256, 0, (cudaStream_t)stream>>>(Z, N * 16, F);
    return check_launch("final_features");
}

extern "C" int ngacf_score_pairs_bwd(const float* Z, int32_t U, const int64_t* users, const int64_t* items, const float* dscore, int32_t B,
                                     float* G, int32_t accumulate, void* stream) {
    NGACF_REQUIRE(Z && users && items && dscore && G && B >= 0, "score_pairs_bwd: null argument");
    if (B == 0) return NGACF_OK;
    score_pairs_bwd_kernel<<<2 * B, 256, 0, (cudaStream_t)stream>>>(Z, U, users, items, dscore, B, G, accumulate);
    return check_launch("score_pairs_bwd");
}

extern "C" int ngacf_bpr_loss(const float* pos, const float* neg, int32_t B, float gscale, float* loss, float* dpos, float* dneg, void* stream) {
    NGACF_REQUIRE(pos && neg && B > 0, "bpr_loss: null/empty argument");
    bpr_loss_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(pos, neg, B, gscale, loss, dpos, dneg, nullptr, 0, 0);
    return check_launch("bpr_loss");
}

extern "C" int ngacf_bpr_loss_owned(const float* pos, const float* neg, int32_t B, float gscale, float* loss, float* dpos, float* dneg,
                                    const int64_t* users, int64_t u_lo, int64_t u_hi, void* stream) {
    NGACF_REQUIRE(pos && neg && users && B > 0, "bpr_loss_owned: null/empty argument");
    bpr_loss_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(pos, neg, B, gscale, loss, dpos, dneg, users, u_lo, u_hi);
    return check_launch("bpr_loss_owned");
}

extern "C" int ngacf_adam_step(const uint64_t* tab, int32_t n_tensors, int64_t total_numel, float lr, float beta1, float beta2, float eps,
                               float weight_decay, int64_t step_host, void* stream) {
    NGACF_REQUIRE(tab && n_tensors > 0 && n_tensors <= ADAM_MAX_TENSORS && step_host >= 1, "adam_step: bad table/step");
    const double bc1 = 1.0 - pow((double)beta1, (double)step_host);
    const double bc2 = 1.0 - pow((double)beta2, (double)step_host);
    const float lr_over_bc1 = (float)((double)lr / bc1);
    const float inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    int64_t chunks = total_numel / 4 + n_tensors;
    int blocks = ceil_div(chunks, 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    adam_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const AdamEntry*>(tab), n_tensors, lr_over_bc1, inv_sqrt_bc2,
                                                          nullptr, beta1, beta2, eps, weight_decay);
    return check_launch("adam_step");
}

extern "C" int ngacf_adam_step_dev(const uint64_t* tab, int32_t n_tensors, int64_t total_numel, float lr, float beta1, float beta2, float eps,
                                   float weight_decay, double* state, void* stream) {
    NGACF_REQUIRE(tab && state && n_tensors > 0 && n_tensors <= ADAM_MAX_TENSORS, "adam_step_dev: bad table/state");
    int64_t chunks = total_numel / 4 + n_tensors;
    int blocks = ceil_div(chunks, 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    adam_tick_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(state, (double)lr, (double)beta1, (double)beta2);
    adam_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const AdamEntry*>(tab), n_tensors, 0.f, 0.f, state, beta1, beta2,
                                                          eps, weight_decay);
    return check_launch("adam_step_dev");
}

extern "C" int ngacf_sample_pairs(const int32_t* train_rows_user, const int32_t* train_ptr, const int32_t* train_items,
                                  const int32_t* train_rank, const int32_t* pool, int32_t P, int64_t row_begin, int64_t row_end,
                                  const int64_t* row_dev, uint64_t seed, uint32_t epoch, int64_t* users, int64_t* pos, int64_t* neg, void* stream) {
    NGACF_REQUIRE(train_rows_user && train_ptr && train_items && train_rank && pool && users && pos && neg, "sample_pairs: null argument");
    NGACF_REQUIRE(row_end >= row_begin && P > 0, "sample_pairs: bad range");
    const int64_t n = row_end - row_begin;
    if (n == 0) return NGACF_OK;
    sample_pairs_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(train_rows_user, train_ptr, train_items, train_rank, pool, P,
                                                                             row_begin, n, row_dev, (uint32_t)seed, (uint32_t)(seed >> 32), epoch,
                                                                             users, pos, neg);
    return check_launch("sample_pairs");
}

// width-carrying entry points: width 64 reaches the calls above (the same kernels)
extern "C" int ngacf_score_pairs_w(const float* Z, int32_t width, int32_t U, const int64_t* users, const int64_t* items, int32_t B, float* scores,
                                   void* stream) {
    if (width == 64) return ngacf_score_pairs(Z, U, users, items, B, scores, stream);
    if (width != 128) { set_error("score_pairs_w: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    NGACF_REQUIRE(Z && users && items && scores && B >= 0, "score_pairs_w: null argument");
    if (B == 0) return NGACF_OK;
    score_pairs128_kernel<<<ceil_div((int64_t)B * 16, 256), 256, 0, (cudaStream_t)stream>>>(Z, U, users, items, B, scores);
    return check_launch("score_pairs_w");
}

extern "C" int ngacf_score_pairs_bwd_w(const float* Z, int32_t width, int32_t U, const int64_t* users, const int64_t* items, const float* dscore,
                                       int32_t B, float* G, int32_t accumulate, void* stream) {
    if (width == 64) return ngacf_score_pairs_bwd(Z, U, users, items, dscore, B, G, accumulate, stream);
    if (width != 128) { set_error("score_pairs_bwd_w: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    NGACF_REQUIRE(Z && users && items && dscore && G && B >= 0, "score_pairs_bwd_w: null argument");
    if (B == 0) return NGACF_OK;
    score_pairs_bwd_kernel<128><<<2 * B, 256, 0, (cudaStream_t)stream>>>(Z, U, users, items, dscore, B, G, accumulate);
    return check_launch("score_pairs_bwd_w");
}

extern "C" int ngacf_final_features_w(const float* Z, int64_t N, int32_t width, float* F, void* stream) {
    if (width == 64) return ngacf_final_features(Z, N, F, stream);
    if (width != 128) { set_error("final_features_w: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    NGACF_REQUIRE(Z && F && N >= 0, "final_features_w: null argument");
    if (N == 0) return NGACF_OK;
    final_features_kernel<<<ceil_div(N * 32, 256), 256, 0, (cudaStream_t)stream>>>(Z, N * 32, F);    // elementwise: N*128/4 float4
    return check_launch("final_features_w");
}
