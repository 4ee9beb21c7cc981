// AllNeg evaluation, exact path: fp32 CUDA-core user x item scores with the specified summation tree
// (bit-reproducible), train-positive / item-pool masking and a per-user top-20 fused in the same
// kernel -- the (users x items) score matrix never exists in HBM.  Plus hit lists and metric sums.
// Replaces train_eval_Gowalla.py:300-341 (64x2048 tiles through model(), D2H per tile),
// :370-385 (heapq.nlargest over a dict per user), :419-429 + metrics.py:10-86.
#include <cmath>
#include "topk_common.cuh"

namespace ngacf {

constexpr int K = NGACF_TOPK;
constexpr int EX_USERS = 16;          // users per CTA
constexpr int EX_ITEMS = 64;          // items per tile
constexpr int EX_THREADS = 256;       // 16 users x 16 item lanes, 4 items per thread per tile
template <int W> __host__ __device__ constexpr size_t ex_smem() {
    return (size_t)(W * EX_ITEMS + EX_USERS * W) * 4 + (size_t)EX_THREADS * K * 8 + EX_USERS * 8 + EX_ITEMS + 64;
}
constexpr size_t EX_SMEM = ex_smem<64>();

template <int W = 64>
__global__ void __launch_bounds__(EX_THREADS) score_topk_exact_kernel(const float* __restrict__ F, int U, int I, const int* __restrict__ users,
                                                                      int n_users, const int* __restrict__ train_ptr,
                                                                      const int* __restrict__ train_items, const uint8_t* __restrict__ in_pool,
                                                                      int* __restrict__ top_ids, float* __restrict__ top_scores) {
    // gridDim.y > 1 (few users, ngacf_score_topk_exact_split): CTA (x, y) ranks its 16 users on item slice y only and writes the
    // slice's top-K to row (uslot * gridDim.y + y) of the outputs, which then are partial lists merged by merge_partial_topk_kernel
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int L = W == 64 ? 6 : 7;
    float* It = reinterpret_cast<float*>(smem_raw);                 // [W d][64 items]
    float* Us = It + W * EX_ITEMS;                                  // [16 users][W]
    float* Ls = Us + EX_USERS * W;                                  // [K][256] scores (thread-interleaved)
    int* Li = reinterpret_cast<int*>(Ls + EX_THREADS * K);          // [K][256] ids
    unsigned long long* Mk = reinterpret_cast<unsigned long long*>(Li + EX_THREADS * K);   // [16] train-positive bits of the tile
    uint8_t* Pool = reinterpret_cast<uint8_t*>(Mk + EX_USERS);      // [64]
    __shared__ int cursor[EX_USERS];

    const int tid = threadIdx.x, ul = tid >> 4, il = tid & 15;
    const int uslot = blockIdx.x * EX_USERS + ul;
    const int user = uslot < n_users ? users[uslot] : -1;
    for (int idx = tid; idx < EX_USERS * W; idx += EX_THREADS) {
        int us = blockIdx.x * EX_USERS + idx / W;
        Us[idx] = us < n_users ? F[(int64_t)users[us] * W + (idx % W)] : 0.f;
    }
    for (int k = 0; k < K; ++k) { Ls[k * EX_THREADS + tid] = -INFINITY; Li[k * EX_THREADS + tid] = -1; }
    const int tiles_all = (I + EX_ITEMS - 1) / EX_ITEMS;
    const int i_begin = (int)((int64_t)blockIdx.y * tiles_all / gridDim.y) * EX_ITEMS;
    const int i_end = min(I, (int)((int64_t)(blockIdx.y + 1) * tiles_all / gridDim.y) * EX_ITEMS);
    if (il == 0) {            // first train item of the user inside the slice (sorted list)
        int lo = user >= 0 ? train_ptr[user] : 0, hi = user >= 0 ? train_ptr[user + 1] : 0;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (train_items[mid] < i_begin) lo = mid + 1; else hi = mid;
        }
        cursor[ul] = lo;
    }
    float thr = -INFINITY;    // score of this thread's current K-th entry
    int cnt = 0;
    __syncthreads();
    const int tend = user >= 0 ? train_ptr[user + 1] : 0;

    for (int i0 = i_begin; i0 < i_end; i0 += EX_ITEMS) {
        __syncthreads();
        NGACF_LOAD_ITEM_TILE(W, EX_ITEMS, EX_THREADS, It, F, U, I, i0, tid);     // It[d][j] = F[U+i0+j][d]
        if (tid < EX_ITEMS) Pool[tid] = (i0 + tid < I) ? in_pool[i0 + tid] : 0;
        if (il == 0) {      // train positives of this user inside the tile (sorted list, monotone cursor)
            unsigned long long m = 0ull;
            int c = cursor[ul];
            while (c < tend) {
                int it = train_items[c];
                if (it >= i0 + EX_ITEMS) break;
                if (it >= i0) m |= 1ull << (it - i0);
                ++c;
            }
            cursor[ul] = c;
            Mk[ul] = m;
        }
        __syncthreads();
        TreeN<L> t0, t1, t2, t3;
        const float* up = Us + ul * W;
#pragma unroll
        for (int d = 0; d < W; ++d) {
            const float u = up[d];
            const float* row = It + d * EX_ITEMS + il;
            t0.add(d, __fmul_rn(u, row[0]));
            t1.add(d, __fmul_rn(u, row[16]));
            t2.add(d, __fmul_rn(u, row[32]));
            t3.add(d, __fmul_rn(u, row[48]));
        }
        const unsigned long long mk = Mk[ul];
        const float sc[4] = {t0.st[L - 1], t1.st[L - 1], t2.st[L - 1], t3.st[L - 1]};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int jj = il + 16 * j;
            const int item = i0 + jj;
            const bool cand = user >= 0 && item < I && Pool[jj] && !((mk >> jj) & 1ull);
            const float s = sc[j];
            // strict '>' : an equal score with a larger id never displaces (ids ascend within a thread)
            if (cand && (cnt < K || s > thr)) {
                int pos = cnt < K ? cnt : K - 1;
                while (pos > 0 && Ls[(pos - 1) * EX_THREADS + tid] < s) {
                    Ls[pos * EX_THREADS + tid] = Ls[(pos - 1) * EX_THREADS + tid];
                    Li[pos * EX_THREADS + tid] = Li[(pos - 1) * EX_THREADS + tid];
                    --pos;
                }
                Ls[pos * EX_THREADS + tid] = s;
                Li[pos * EX_THREADS + tid] = item;
                if (cnt < K) ++cnt;
                if (cnt == K) thr = Ls[(K - 1) * EX_THREADS + tid];
            }
        }
    }
    __syncthreads();
    // 16-way merge of the sorted per-thread lists of a user
    if (il == 0 && user >= 0) {
        int head[16];
#pragma unroll
        for (int l = 0; l < 16; ++l) head[l] = 0;
        for (int k = 0; k < K; ++k) {
            float bs = -INFINITY; int bi = -1, bl = -1;
#pragma unroll
            for (int l = 0; l < 16; ++l) {
                if (head[l] < K) {
                    const int t = ul * 16 + l;
                    const int id = Li[head[l] * EX_THREADS + t];
                    const float s = Ls[head[l] * EX_THREADS + t];
                    if (id >= 0 && (bi < 0 || better(s, id, bs, bi))) { bs = s; bi = id; bl = l; }
                }
            }
            const int64_t orow = (int64_t)uslot * gridDim.y + blockIdx.y;
            top_ids[orow * K + k] = bi;
            top_scores[orow * K + k] = bi >= 0 ? bs : 0.f;
            if (bl >= 0) {
#pragma unroll
                for (int l = 0; l < 16; ++l) if (l == bl) ++head[l];
            }
        }
    }
}

// P partial lists of a user (disjoint item slices) -> its top-K under (score desc, id asc).  One CTA per user: the P*K entries go to
// shared memory, every thread ranks its entries against all of them (ids are distinct, so the ranks are a permutation) and the
// entries of rank < K land at their rank.  (A single thread walking the lists K times took 2.5 ms at P = 64.)
constexpr int MERGE_MAX_P = 64;
__global__ void __launch_bounds__(256) merge_partial_topk_kernel(const int* __restrict__ part_ids, const float* __restrict__ part_scores, int n_users, int P,
                                                                int* __restrict__ top_ids, float* __restrict__ top_scores) {
    __shared__ int ids[MERGE_MAX_P * K];
    __shared__ float scs[MERGE_MAX_P * K];
    __shared__ int n_valid;
    const int j = blockIdx.x;
    const int n = P * K;
    if (threadIdx.x == 0) n_valid = 0;
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
        ids[e] = part_ids[(int64_t)j * n + e];
        scs[e] = part_scores[(int64_t)j * n + e];
    }
    __syncthreads();
    int mine = 0;
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
        const int id = ids[e];
        if (id < 0) continue;
        ++mine;
        const float sv = scs[e];
        int rank = 0;
        for (int o = 0; o < n; ++o) {
            const int io = ids[o];
            rank += (io >= 0 && better(scs[o], io, sv, id)) ? 1 : 0;
        }
        if (rank < K) { top_ids[(int64_t)j * K + rank] = id; top_scores[(int64_t)j * K + rank] = sv; }
    }
    atomicAdd(&n_valid, mine);
    __syncthreads();
    for (int k = n_valid + threadIdx.x; k < K; k += blockDim.x) { top_ids[(int64_t)j * K + k] = -1; top_scores[(int64_t)j * K + k] = 0.f; }
}

// ------------------------------------------------------------------------------------------------
// hit lists + metrics (metrics.py:10-86 through get_performance, train_eval_Gowalla.py:419-429)
// ------------------------------------------------------------------------------------------------
// 1 / log2(k + 2), k = 0..19, in double (metrics.py:52-53: np.log2(np.arange(2, size + 2))); evaluated once on the host -- fp64
// transcendental code was most of this kernel's time
__constant__ double c_disc[K];

__global__ void __launch_bounds__(128) eval_metrics_kernel(const int* __restrict__ top_ids, const int* __restrict__ users, int n_users,
                                                           const int* __restrict__ test_ptr, const int* __restrict__ test_items,
                                                           uint8_t* __restrict__ hits, double* __restrict__ partial /* [gridDim.x][16] */) {
    __shared__ double red[128][17];
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    double val[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) val[q] = 0.0;
    if (j < n_users) {
        const int u = users[j];
        const int beg = test_ptr[u], end = test_ptr[u + 1];
        unsigned r = 0;                                   // bit k = hit at rank k
        for (int k = 0; k < K; ++k) {
            const int id = top_ids[(int64_t)j * K + k];
            int lo = beg, hi = end;
            bool hit = false;
            while (id >= 0 && lo < hi) {
                const int mid = (lo + hi) >> 1;
                const int v = test_items[mid];
                if (v == id) { hit = true; break; }
                if (v < id) lo = mid + 1; else hi = mid;
            }
            r |= (hit ? 1u : 0u) << k;
            hits[(int64_t)j * K + k] = hit ? 1 : 0;
        }
        const int Ks[4] = {1, 5, 10, 20};
        const int total_hits = __popc(r);
        const double npos = (double)(end - beg);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int KK = Ks[q];
            int h = 0;
            double dcg = 0.0, idcg = 0.0;
            for (int k = 0; k < KK; ++k) {
                const double disc = c_disc[k];
                if ((r >> k) & 1u) { ++h; dcg += disc; }
                if (k < total_hits) idcg += disc;        // ideal = the top-20 hit list itself, sorted (metrics.py:69-73)
            }
            val[0 + q] = (double)h / (double)KK;                 // precision_at_k
            val[4 + q] = npos > 0 ? (double)h / npos : 0.0;      // recall_at_k
            val[8 + q] = idcg > 0 ? dcg / idcg : 0.0;            // ndcg_at_k
            val[12 + q] = h > 0 ? 1.0 : 0.0;                     // hit_at_k
        }
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) red[threadIdx.x][q] = val[q];
    __syncthreads();
    if (threadIdx.x < 16) {                                // fixed-order sum over the block's users
        double acc = 0.0;
        for (int t = 0; t < 128; ++t) acc += red[t][threadIdx.x];
        partial[(int64_t)blockIdx.x * 16 + threadIdx.x] = acc;
    }
}

// fixed-order sum of the block partials
// 16 warps, one per metric column: lane l sums blocks l, l+32, ... in order, then a fixed shuffle tree (deterministic)
__global__ void __launch_bounds__(512) eval_metrics_reduce_kernel(const double* __restrict__ partial, int nblocks, double* __restrict__ sums) {
    const int c = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double acc = 0.0;
    for (int b = lane; b < nblocks; b += 32) acc += partial[(int64_t)b * 16 + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) sums[c] = acc;
}

}  // namespace ngacf

using namespace ngacf;

extern "C" int ngacf_score_topk_exact(const float* F, int32_t U, int32_t I, const int32_t* users, int32_t n_users, const int32_t* train_ptr,
                                      const int32_t* train_items, const uint8_t* in_pool, int32_t* top_ids, float* top_scores, void* stream) {
    NGACF_REQUIRE(F && users && train_ptr && train_items && in_pool && top_ids && top_scores && U > 0 && I > 0 && n_users >= 0,
                  "score_topk_exact: null/empty argument");
    if (n_users == 0) return NGACF_OK;
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(score_topk_exact_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EX_SMEM);
    });
    score_topk_exact_kernel<64><<<ceil_div(n_users, EX_USERS), EX_THREADS, EX_SMEM, (cudaStream_t)stream>>>(F, U, I, users, n_users, train_ptr,
                                                                                                         train_items, in_pool, top_ids, top_scores);
    return check_launch("score_topk_exact");
}

// few users (the rows the tensor-core path flags): one CTA per 16 users would walk all items alone (6 ms at 92 K items for a single
// row); the item range is split over P CTAs per user group and the P partial lists are merged
static int exact_split_parts(int n_users, int I) {
    const int groups = (n_users + EX_USERS - 1) / EX_USERS;
    int P = groups > 0 ? (2 * 148) / groups : 1;
    const int tiles = (I + EX_ITEMS - 1) / EX_ITEMS;
    if (P > tiles / 8) P = tiles / 8;
    if (P > MERGE_MAX_P) P = MERGE_MAX_P;
    if (P < 1) P = 1;
    return P;
}

extern "C" size_t ngacf_score_topk_exact_split_workspace_bytes(int32_t I, int32_t n_users) {
    return (size_t)(n_users > 0 ? n_users : 1) * exact_split_parts(n_users, I) * K * 8 + 256;
}

extern "C" int ngacf_score_topk_exact_split(const float* F, int32_t U, int32_t I, const int32_t* users, int32_t n_users, const int32_t* train_ptr,
                                            const int32_t* train_items, const uint8_t* in_pool, int32_t* top_ids, float* top_scores,
                                            void* workspace, size_t workspace_bytes, void* stream) {
    NGACF_REQUIRE(F && users && train_ptr && train_items && in_pool && top_ids && top_scores && workspace && U > 0 && I > 0 && n_users >= 0,
                  "score_topk_exact_split: null/empty argument");
    if (workspace_bytes < ngacf_score_topk_exact_split_workspace_bytes(I, n_users)) { set_error("score_topk_exact_split: workspace too small"); return NGACF_ERR_WORKSPACE; }
    if (n_users == 0) return NGACF_OK;
    const int P = exact_split_parts(n_users, I);
    if (P == 1) return ngacf_score_topk_exact(F, U, I, users, n_users, train_ptr, train_items, in_pool, top_ids, top_scores, stream);
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(score_topk_exact_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EX_SMEM);
    });
    cudaStream_t st = (cudaStream_t)stream;
    char* w = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    int* part_ids = (int*)w;
    float* part_scores = (float*)(w + (size_t)n_users * P * K * 4);
    score_topk_exact_kernel<64><<<dim3(ceil_div(n_users, EX_USERS), P), EX_THREADS, EX_SMEM, st>>>(F, U, I, users, n_users, train_ptr, train_items, in_pool,
                                                                                              part_ids, part_scores);
    merge_partial_topk_kernel<<<n_users, 256, 0, st>>>(part_ids, part_scores, n_users, P, top_ids, top_scores);
    return check_launch("score_topk_exact_split");
}

// width-carrying entry points: width 64 reaches the calls above (the same kernel); 128-wide features run the W = 128 instantiation
// (seven-level tree, twice the user / item tiles in shared memory)
static int launch_topk_exact128(const float* F, int U, int I, const int* users, int n_users, const int* train_ptr, const int* train_items,
                                const uint8_t* in_pool, int* top_ids, float* top_scores, int P, cudaStream_t st) {
    static PerDeviceOnce once;
    once.run([] { cudaFuncSetAttribute(score_topk_exact_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ex_smem<128>()); });
    score_topk_exact_kernel<128><<<dim3(ceil_div(n_users, EX_USERS), P), EX_THREADS, ex_smem<128>(), st>>>(F, U, I, users, n_users, train_ptr,
                                                                                                           train_items, in_pool, top_ids, top_scores);
    return check_launch("score_topk_exact_w");
}

extern "C" int ngacf_score_topk_exact_w(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* users, int32_t n_users,
                                        const int32_t* train_ptr, const int32_t* train_items, const uint8_t* in_pool, int32_t* top_ids,
                                        float* top_scores, void* stream) {
    if (width == 64) return ngacf_score_topk_exact(F, U, I, users, n_users, train_ptr, train_items, in_pool, top_ids, top_scores, stream);
    if (width != 128) { set_error("score_topk_exact_w: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    NGACF_REQUIRE(F && users && train_ptr && train_items && in_pool && top_ids && top_scores && U > 0 && I > 0 && n_users >= 0,
                  "score_topk_exact_w: null/empty argument");
    if (n_users == 0) return NGACF_OK;
    return launch_topk_exact128(F, U, I, users, n_users, train_ptr, train_items, in_pool, top_ids, top_scores, 1, (cudaStream_t)stream);
}

extern "C" int ngacf_score_topk_exact_split_w(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* users, int32_t n_users,
                                              const int32_t* train_ptr, const int32_t* train_items, const uint8_t* in_pool, int32_t* top_ids,
                                              float* top_scores, void* workspace, size_t workspace_bytes, void* stream) {
    if (width == 64)
        return ngacf_score_topk_exact_split(F, U, I, users, n_users, train_ptr, train_items, in_pool, top_ids, top_scores, workspace,
                                            workspace_bytes, stream);
    if (width != 128) { set_error("score_topk_exact_split_w: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    NGACF_REQUIRE(F && users && train_ptr && train_items && in_pool && top_ids && top_scores && workspace && U > 0 && I > 0 && n_users >= 0,
                  "score_topk_exact_split_w: null/empty argument");
    if (workspace_bytes < ngacf_score_topk_exact_split_workspace_bytes(I, n_users)) { set_error("score_topk_exact_split_w: workspace too small"); return NGACF_ERR_WORKSPACE; }
    if (n_users == 0) return NGACF_OK;
    const int P = exact_split_parts(n_users, I);
    cudaStream_t st = (cudaStream_t)stream;
    if (P == 1) return launch_topk_exact128(F, U, I, users, n_users, train_ptr, train_items, in_pool, top_ids, top_scores, 1, st);
    char* w = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    int* part_ids = (int*)w;
    float* part_scores = (float*)(w + (size_t)n_users * P * K * 4);
    const int rc = launch_topk_exact128(F, U, I, users, n_users, train_ptr, train_items, in_pool, part_ids, part_scores, P, st);
    if (rc != NGACF_OK) return rc;
    merge_partial_topk_kernel<<<n_users, 256, 0, st>>>(part_ids, part_scores, n_users, P, top_ids, top_scores);
    return check_launch("score_topk_exact_split_w");
}

extern "C" size_t ngacf_eval_metrics_workspace_bytes(int32_t n_users) { return (size_t)(n_users > 0 ? n_users : 1) * 16 * sizeof(double); }

extern "C" int ngacf_eval_metrics(const int32_t* top_ids, const int32_t* users, int32_t n_users, const int32_t* test_ptr,
                                  const int32_t* test_items, uint8_t* hits, double* sums, void* workspace, size_t workspace_bytes, void* stream) {
    NGACF_REQUIRE(top_ids && users && test_ptr && test_items && hits && sums && workspace, "eval_metrics: null argument");
    if (workspace_bytes < ngacf_eval_metrics_workspace_bytes(n_users)) { set_error("eval_metrics: workspace too small"); return NGACF_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    if (n_users == 0) { cudaMemsetAsync(sums, 0, 16 * sizeof(double), st); return NGACF_OK; }
    static PerDeviceOnce once;
    once.run([] {
        double disc[K];
        for (int k = 0; k < K; ++k) disc[k] = 1.0 / std::log2((double)(k + 2));
        cudaMemcpyToSymbol(c_disc, disc, sizeof(disc));
    });
    eval_metrics_kernel<<<ceil_div(n_users, 128), 128, 0, st>>>(top_ids, users, n_users, test_ptr, test_items, hits, (double*)workspace);
    eval_metrics_reduce_kernel<<<1, 512, 0, st>>>((const double*)workspace, ceil_div(n_users, 128), sums);
    return check_launch("eval_metrics");
}
