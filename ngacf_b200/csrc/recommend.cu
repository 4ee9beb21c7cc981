// Top-K recommendation lists (K <= NGACF_RECOMMEND_MAX_K) for any users: the fp32 CUDA-core scores of eval_topk.cu (same item tile,
// same adjacent-pair tree, so the same bits) with a selection that does not keep a K-long list per thread.  Each of the 16 users of a
// CTA owns a candidate buffer of RC_CAP (score, id) entries in shared memory and a threshold (the K-th best entry kept so far); an
// item enters the buffer only if it beats the threshold.  Before a tile, a user whose buffer cannot take another 64 items is
// compacted: all 256 threads rank its entries by counting (ids are distinct, so the ranks are a permutation), the entries of rank
// < K move to their rank and the threshold rises to the K-th.  The same ranking writes the final list.  Every step keeps the exact
// top-K of the items seen, so a row does not depend on which users share the CTA, on when a compaction ran or on the item slicing.
// The same kernel, instantiated with ITEMQ = true, ranks items for query items (similar-item lists): the query row is F[U+q], each
// score is the cosine dot * rn(q) * rn(j) with inverse norms from item_rnorm_kernel, and the only excluded item is q itself.
#include "topk_common.cuh"

namespace ngacf {

constexpr int RC_USERS = 16;          // users per CTA
constexpr int RC_ITEMS = 64;          // items per tile
constexpr int RC_THREADS = 256;       // 16 users x 16 item lanes, 4 items per thread per tile
constexpr int RC_CAP = 256;           // candidate buffer entries per user (= threads: one entry per thread when ranking)
constexpr int RC_MERGE_MAX_P = 64;    // item slices per user
// P * K partial entries per user at most: the merge's binary searches are a dependent chain of shared-memory loads per entry, and at
// P = 64, K = 100 they made a one-user call take 1.1 ms (a 2048-entry merge with 1024 threads is short next to the slices' scoring)
constexpr int RC_MERGE_MAX_ENTRIES = 2048;
constexpr int RC_MERGE_THREADS = 1024;
static_assert(RC_CAP == RC_THREADS && RC_CAP >= NGACF_RECOMMEND_MAX_K + RC_ITEMS, "buffer layout");

template <int W, bool ITEMQ = false> __host__ __device__ constexpr size_t rc_smem() {
    return (size_t)(W * RC_ITEMS + RC_USERS * W) * 4 + (size_t)RC_USERS * RC_CAP * 8 + RC_USERS * 8 + RC_ITEMS + 64 + (ITEMQ ? RC_ITEMS * 4 : 0);
}

// all threads of the CTA: ranks the n = cnt[v] buffered entries of user slot v.  out == nullptr: the entries of rank < K move to
// the front of the buffer and the threshold becomes the K-th; otherwise the K best are written to out_ids/out_scores (row of K,
// padded with -1 / 0.0).
__device__ __forceinline__ void rc_rank_user(int v, int K, float* Bs, int* Bi, int* cnt, float* tau_s, int* tau_i, int* out_ids,
                                             float* out_scores) {
    const int tid = threadIdx.x;
    const int n = cnt[v];
    const float* bs = Bs + v * RC_CAP;
    const int* bi = Bi + v * RC_CAP;
    float s = 0.f;
    int id = -1, rank = RC_CAP;
    if (tid < n) {
        s = bs[tid];
        id = bi[tid];
        rank = 0;
        for (int o = 0; o < n; ++o) rank += better(bs[o], bi[o], s, id) ? 1 : 0;
    }
    if (out_ids) {
        if (rank < K) { out_ids[rank] = id; out_scores[rank] = s; }
        for (int k = n + tid; k < K; k += RC_THREADS) { out_ids[k] = -1; out_scores[k] = 0.f; }
        return;
    }
    __syncthreads();
    if (rank < K) { Bs[v * RC_CAP + rank] = s; Bi[v * RC_CAP + rank] = id; }
    __syncthreads();
    if (tid == 0) {
        cnt[v] = min(n, K);
        if (n >= K) { tau_s[v] = Bs[v * RC_CAP + K - 1]; tau_i[v] = Bi[v * RC_CAP + K - 1]; }
    }
}

// ITEMQ = false: `users` are user ids (rows F[u]), excl_ptr / excl_items the excluded items, rnorm unused.  ITEMQ = true: `users` are
// query item ids (rows F[U+q], ids outside [0, I) rank nothing), excl_ptr / excl_items unused, rnorm[I] the items' inverse norms.
// rnorm is the last parameter so that the user form keeps its parameter offsets (and its SASS).
template <int W, bool ITEMQ = false>
__global__ void __launch_bounds__(RC_THREADS) recommend_topk_kernel(const float* __restrict__ F, int U, int I, const int* __restrict__ users,
                                                                    int n_users, int K, const int* __restrict__ excl_ptr,
                                                                    const int* __restrict__ excl_items, const uint8_t* __restrict__ in_pool,
                                                                    int* __restrict__ top_ids, float* __restrict__ top_scores,
                                                                    const float* __restrict__ rnorm) {
    // gridDim.y > 1 (few users): CTA (x, y) ranks its users on item slice y and writes the slice's list to row (uslot * gridDim.y + y)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int L = W == 64 ? 6 : 7;
    float* It = reinterpret_cast<float*>(smem_raw);                 // [W d][64 items]
    float* Us = It + W * RC_ITEMS;                                  // [16 users][W]
    float* Bs = Us + RC_USERS * W;                                  // [16 users][RC_CAP] buffered scores
    int* Bi = reinterpret_cast<int*>(Bs + RC_USERS * RC_CAP);       // [16 users][RC_CAP] buffered ids
    unsigned long long* Mk = reinterpret_cast<unsigned long long*>(Bi + RC_USERS * RC_CAP);   // [16] excluded items of the tile
    uint8_t* Pool = reinterpret_cast<uint8_t*>(Mk + RC_USERS);      // [64]
    float* Rn = reinterpret_cast<float*>(Pool + RC_ITEMS);          // [64] inverse norms of the tile's items (ITEMQ only)
    __shared__ int cursor[RC_USERS], cnt[RC_USERS], tau_i[RC_USERS], row_user[RC_USERS];
    __shared__ float tau_s[RC_USERS];

    const int tid = threadIdx.x, ul = tid >> 4, il = tid & 15;
    if (tid < RC_USERS) {
        const int us = blockIdx.x * RC_USERS + tid;
        int u = us < n_users ? users[us] : -1;
        row_user[tid] = (u >= 0 && u < (ITEMQ ? I : U)) ? u : -1;   // an id outside [0, U) ([0, I)) ranks nothing and reads nothing
        cnt[tid] = 0;
        tau_s[tid] = -INFINITY;                                     // every item beats (-inf, INT_MAX) until K are kept
        tau_i[tid] = 0x7fffffff;
    }
    __syncthreads();
    const int user = row_user[ul];
    for (int idx = tid; idx < RC_USERS * W; idx += RC_THREADS) {
        const int u = row_user[idx / W];
        Us[idx] = u >= 0 ? F[((ITEMQ ? (int64_t)U : 0) + u) * W + (idx % W)] : 0.f;
    }
    const float qrn = ITEMQ && user >= 0 ? rnorm[user] : 0.f;
    const int tiles_all = (I + RC_ITEMS - 1) / RC_ITEMS;
    const int i_begin = (int)((int64_t)blockIdx.y * tiles_all / gridDim.y) * RC_ITEMS;
    const int i_end = min(I, (int)((int64_t)(blockIdx.y + 1) * tiles_all / gridDim.y) * RC_ITEMS);
    const bool excl = !ITEMQ && excl_ptr != nullptr && user >= 0;
    if (il == 0) {            // first excluded item of the user inside the slice (sorted list)
        int lo = excl ? excl_ptr[user] : 0, hi = excl ? excl_ptr[user + 1] : 0;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (excl_items[mid] < i_begin) lo = mid + 1; else hi = mid;
        }
        cursor[ul] = lo;
    }
    const int tend = excl ? excl_ptr[user + 1] : 0;

    for (int i0 = i_begin; i0 < i_end; i0 += RC_ITEMS) {
        __syncthreads();
        for (int v = 0; v < RC_USERS; ++v)              // cnt[] is stable here: the same decision in every thread
            if (cnt[v] > RC_CAP - RC_ITEMS) rc_rank_user(v, K, Bs, Bi, cnt, tau_s, tau_i, nullptr, nullptr);
        NGACF_LOAD_ITEM_TILE(W, RC_ITEMS, RC_THREADS, It, F, U, I, i0, tid);     // It[d][j] = F[U+i0+j][d]
        if (tid < RC_ITEMS) Pool[tid] = (i0 + tid < I) ? (in_pool ? in_pool[i0 + tid] : 1) : 0;
        if (ITEMQ && tid < RC_ITEMS) Rn[tid] = (i0 + tid < I) ? rnorm[i0 + tid] : 0.f;
        if (!ITEMQ && il == 0) {      // excluded items of this user inside the tile (sorted list, monotone cursor)
            unsigned long long m = 0ull;
            int c = cursor[ul];
            while (c < tend) {
                int it = excl_items[c];
                if (it >= i0 + RC_ITEMS) break;
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
            const float* row = It + d * RC_ITEMS + il;
            t0.add(d, __fmul_rn(u, row[0]));
            t1.add(d, __fmul_rn(u, row[16]));
            t2.add(d, __fmul_rn(u, row[32]));
            t3.add(d, __fmul_rn(u, row[48]));
        }
        const unsigned long long mk = ITEMQ ? 0ull : Mk[ul];
        float sc[4] = {t0.st[L - 1], t1.st[L - 1], t2.st[L - 1], t3.st[L - 1]};
        const float ts = tau_s[ul];
        const int ti = tau_i[ul];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int jj = il + 16 * j;
            const int item = i0 + jj;
            if (ITEMQ) sc[j] = __fmul_rn(__fmul_rn(sc[j], qrn), Rn[jj]);     // cosine: (dot * rn(q)) * rn(j), in this order
            const bool cand = user >= 0 && item < I && Pool[jj] && (ITEMQ ? item != user : !((mk >> jj) & 1ull));
            if (cand && better(sc[j], item, ts, ti)) {
                const int p = atomicAdd(&cnt[ul], 1);    // < RC_CAP: at most 64 entries per tile after the check above
                Bs[ul * RC_CAP + p] = sc[j];
                Bi[ul * RC_CAP + p] = item;
            }
        }
    }
    __syncthreads();
    for (int v = 0; v < RC_USERS; ++v) {
        const int us = blockIdx.x * RC_USERS + v;
        if (us >= n_users) break;
        const int64_t orow = (int64_t)us * gridDim.y + blockIdx.y;
        rc_rank_user(v, K, Bs, Bi, cnt, tau_s, tau_i, top_ids + orow * K, top_scores + orow * K);
    }
}

// P sorted partial lists of K per user (disjoint item slices, padded with -1) -> the user's top-K.  One CTA per user; the entry at
// position k of list p has rank k + (number of entries of every other list that beat it), found by binary search in each sorted list.
__global__ void __launch_bounds__(RC_MERGE_THREADS) recommend_merge_kernel(const int* __restrict__ part_ids, const float* __restrict__ part_scores, int P,
                                                              int K, int* __restrict__ top_ids, float* __restrict__ top_scores) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int* ids = reinterpret_cast<int*>(smem_raw);
    float* scs = reinterpret_cast<float*>(ids + P * K);
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
        const int p = e / K;
        int rank = e - p * K;
        for (int q = 0; q < P; ++q) {
            if (q == p) continue;
            int lo = 0, hi = K;          // entries of list q that beat (sv, id): a prefix (valid entries first, sorted)
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                const int io = ids[q * K + mid];
                if (io >= 0 && better(scs[q * K + mid], io, sv, id)) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < K) { top_ids[(int64_t)j * K + rank] = id; top_scores[(int64_t)j * K + rank] = sv; }
    }
    atomicAdd(&n_valid, mine);
    __syncthreads();
    for (int k = n_valid + threadIdx.x; k < K; k += blockDim.x) { top_ids[(int64_t)j * K + k] = -1; top_scores[(int64_t)j * K + k] = 0.f; }
}

// rnorm[j] = 1 / sqrt(F[U+j] . F[U+j]) (0 when the sum is not > 0), the sum by the scoring tree: one warp per item, lane l holds the
// W/32 consecutive terms from l * W/32, sums them pairwise, then xor-shuffles 1..16 (a + b == b + a in IEEE, so every lane of a pair
// holds the same bits and the shuffles are the tree's upper levels)
constexpr int RN_THREADS = 256;
template <int W>
__global__ void __launch_bounds__(RN_THREADS) item_rnorm_kernel(const float* __restrict__ F, int U, int I, float* __restrict__ rnorm) {
    constexpr int PER = W / 32;
    const int j = blockIdx.x * (RN_THREADS / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (j >= I) return;
    const float* row = F + ((int64_t)U + j) * W + lane * PER;
    float v[PER];
#pragma unroll
    for (int k = 0; k < PER; ++k) v[k] = __fmul_rn(row[k], row[k]);
#pragma unroll
    for (int n = PER; n > 1; n >>= 1)
#pragma unroll
        for (int k = 0; k < n / 2; ++k) v[k] = __fadd_rn(v[2 * k], v[2 * k + 1]);
    float s = v[0];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
    if (lane == 0) rnorm[j] = s > 0.f ? __fdiv_rn(1.f, __fsqrt_rn(s)) : 0.f;
}

}  // namespace ngacf

using namespace ngacf;

// item slices per user: 1 (lists written directly, no workspace) once there are enough 16-user CTAs to fill the SMs twice, else
// the item range is split so that about two CTAs per SM run, each slice keeping at least 8 tiles
static int recommend_parts(int n_users, int I, int K) {
    const int groups = (n_users + RC_USERS - 1) / RC_USERS;
    int P = groups > 0 ? (2 * 148) / groups : 1;
    const int tiles = (I + RC_ITEMS - 1) / RC_ITEMS;
    if (P > tiles / 8) P = tiles / 8;
    if (P > RC_MERGE_MAX_P) P = RC_MERGE_MAX_P;
    if (P > RC_MERGE_MAX_ENTRIES / K) P = RC_MERGE_MAX_ENTRIES / K;
    if (P < 1) P = 1;
    return P;
}

static bool recommend_shape_ok(int width, int K) { return width_supported(width) && K >= 1 && K <= NGACF_RECOMMEND_MAX_K; }

extern "C" size_t ngacf_recommend_topk_workspace_bytes(int32_t width, int32_t I, int32_t n_users, int32_t K) {
    if (!recommend_shape_ok(width, K) || I <= 0 || n_users <= 0) return 0;
    const int P = recommend_parts(n_users, I, K);
    return P == 1 ? 0 : (size_t)n_users * P * K * 8 + 256;
}

template <int W, bool ITEMQ>
static int launch_recommend(const float* F, int U, int I, const int* users, int n_users, int K, const int* excl_ptr, const int* excl_items,
                            const uint8_t* in_pool, int* top_ids, float* top_scores, const float* rnorm, int P, cudaStream_t st) {
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(recommend_topk_kernel<W, ITEMQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rc_smem<W, ITEMQ>());
    });
    recommend_topk_kernel<W, ITEMQ><<<dim3(ceil_div(n_users, RC_USERS), P), RC_THREADS, rc_smem<W, ITEMQ>(), st>>>(
        F, U, I, users, n_users, K, excl_ptr, excl_items, in_pool, top_ids, top_scores, rnorm);
    return check_launch(ITEMQ ? "similar_items_topk" : "recommend_topk");
}

// one ranking pass (P == 1: straight into the outputs) or P item slices into the partial lists at `part` and their merge
template <bool ITEMQ>
static int rank_and_merge(const float* F, int width, int U, int I, const int* queries, int n, int K, const int* excl_ptr,
                          const int* excl_items, const uint8_t* in_pool, int* top_ids, float* top_scores, const float* rnorm, int P,
                          char* part, cudaStream_t st) {
    auto launch = width == 64 ? launch_recommend<64, ITEMQ> : launch_recommend<128, ITEMQ>;
    if (P == 1) return launch(F, U, I, queries, n, K, excl_ptr, excl_items, in_pool, top_ids, top_scores, rnorm, 1, st);
    int* part_ids = (int*)part;
    float* part_scores = (float*)(part + (size_t)n * P * K * 4);
    const int rc = launch(F, U, I, queries, n, K, excl_ptr, excl_items, in_pool, part_ids, part_scores, rnorm, P, st);
    if (rc != NGACF_OK) return rc;
    recommend_merge_kernel<<<n, RC_MERGE_THREADS, (size_t)P * K * 8, st>>>(part_ids, part_scores, P, K, top_ids, top_scores);
    return check_launch(ITEMQ ? "similar_items_topk merge" : "recommend_topk merge");
}

static char* align256(void* p) { return (char*)(((uintptr_t)p + 255) & ~(uintptr_t)255); }

extern "C" int ngacf_recommend_topk(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* users, int32_t n_users, int32_t K,
                                    const int32_t* excl_ptr, const int32_t* excl_items, const uint8_t* in_pool, int32_t* top_ids,
                                    float* top_scores, void* workspace, size_t workspace_bytes, void* stream) {
    if (!width_supported(width)) { set_error("recommend_topk: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    if (K < 1 || K > NGACF_RECOMMEND_MAX_K) { set_error("recommend_topk: K = %d is outside 1..%d", K, NGACF_RECOMMEND_MAX_K); return NGACF_ERR_UNSUPPORTED; }
    NGACF_REQUIRE(F && users && top_ids && top_scores && U > 0 && I > 0 && n_users >= 0 && (excl_ptr == nullptr) == (excl_items == nullptr),
                  "recommend_topk: null/empty argument (excl_ptr and excl_items are both given or both NULL)");
    const size_t need = ngacf_recommend_topk_workspace_bytes(width, I, n_users, K);
    if (workspace_bytes < need || (need > 0 && workspace == nullptr)) {
        set_error("recommend_topk: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return NGACF_ERR_WORKSPACE;
    }
    if (n_users == 0) return NGACF_OK;
    const int P = recommend_parts(n_users, I, K);
    return rank_and_merge<false>(F, width, U, I, users, n_users, K, excl_ptr, excl_items, in_pool, top_ids, top_scores, nullptr, P,
                                 P == 1 ? nullptr : align256(workspace), (cudaStream_t)stream);
}

// the I inverse norms (256-byte aligned block), then the partial lists when the item range is split
static size_t rnorm_bytes(int I) { return ((size_t)I * 4 + 255) & ~(size_t)255; }

extern "C" size_t ngacf_similar_items_topk_workspace_bytes(int32_t width, int32_t I, int32_t n_items, int32_t K) {
    if (!recommend_shape_ok(width, K) || I <= 0 || n_items <= 0) return 0;
    const int P = recommend_parts(n_items, I, K);
    return rnorm_bytes(I) + (P == 1 ? 0 : (size_t)n_items * P * K * 8) + 256;
}

extern "C" int ngacf_similar_items_topk(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* items, int32_t n_items, int32_t K,
                                        const uint8_t* in_pool, int32_t* top_ids, float* top_scores, void* workspace, size_t workspace_bytes,
                                        void* stream) {
    if (!width_supported(width)) { set_error("similar_items_topk: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    if (K < 1 || K > NGACF_RECOMMEND_MAX_K) { set_error("similar_items_topk: K = %d is outside 1..%d", K, NGACF_RECOMMEND_MAX_K); return NGACF_ERR_UNSUPPORTED; }
    NGACF_REQUIRE(F && items && top_ids && top_scores && U >= 0 && I > 0 && n_items >= 0, "similar_items_topk: null/empty argument");
    const size_t need = ngacf_similar_items_topk_workspace_bytes(width, I, n_items, K);
    if (workspace_bytes < need || (need > 0 && workspace == nullptr)) {
        set_error("similar_items_topk: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return NGACF_ERR_WORKSPACE;
    }
    if (n_items == 0) return NGACF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    char* w = align256(workspace);
    float* rnorm = (float*)w;
    if (width == 64) item_rnorm_kernel<64><<<ceil_div(I, RN_THREADS / 32), RN_THREADS, 0, st>>>(F, U, I, rnorm);
    else item_rnorm_kernel<128><<<ceil_div(I, RN_THREADS / 32), RN_THREADS, 0, st>>>(F, U, I, rnorm);
    const int rc = check_launch("similar_items_topk norms");
    if (rc != NGACF_OK) return rc;
    const int P = recommend_parts(n_items, I, K);
    return rank_and_merge<true>(F, width, U, I, items, n_items, K, nullptr, nullptr, in_pool, top_ids, top_scores, rnorm, P,
                                w + rnorm_bytes(I), st);
}
