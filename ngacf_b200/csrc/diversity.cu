// Intra-list diversity (ILD) and MMR re-ranking of lists of up to 100 entries, from the cosine of the items' final features.
//   Both kernels run one CTA per list and share dv_stage_sims: warp 0 compacts the list's valid entries (ids in [0, I)) into slots
//   0..m-1 in rank order; the slots' rows are staged in shared memory transposed, It[d][slot] (the layout of NGACF_LOAD_ITEM_TILE,
//   so a column read is conflict-free); thread s computes rn(s) with the scoring tree; then every thread takes 2 x 4 blocks of
//   slot pairs (a, b) (two rows a, four columns b: one 8-byte and one 16-byte shared load per d for eight TreeN dots) and writes
//   sim(a, b) = (dot * rn(a)) * rn(b), the entry of lower rank first, to both halves of an m x m matrix S.  Nothing of size I x I.
//   list_diversity_kernel: thread b sums r_b = sum_{a<b} (1 - sim(a, b)) in fp64 in a ascending, then thread q sums r_1..r_{m_q - 1}
//     in b ascending for cut-off q (m_q: valid entries among its first k) and divides once by m_q (m_q - 1) / 2.
//   mmr_rerank_kernel: one warp runs the greedy loop with no block barriers; lane l owns candidates l, l+32, l+64, l+96 and keeps
//     their relevance and their max similarity to the picks in registers; the argmax is an xor-shuffle reduction in the `better`
//     order on (mmr, slot), NaN values ranking below every number, and m(c) is updated from row `pick` of S.
#include "topk_common.cuh"

namespace ngacf {

constexpr int DV_THREADS = 256;
constexpr int DV_MAX = NGACF_RECOMMEND_MAX_K;   // entries per list

struct DivKs {                         // by value in the kernel parameters: CUDA-graph replay safe
    int32_t n;
    int32_t k[NGACF_CUTOFF_MAX_KS];
};

// P = the slot count rounded up to a multiple of 4: It [W][P], S [P][P], rn / slot ids / slot positions [P]; ILD adds its fp64 r_b [P]
// in front (16-byte multiples throughout, so every array stays aligned)
__host__ __device__ constexpr int dv_slots(int n) { return (n + 3) & ~3; }
__host__ __device__ constexpr size_t dv_smem(int W, int P, bool ild) { return (size_t)(W * P + P * P + 3 * P) * 4 + (ild ? (size_t)P * 8 : 0); }

// all threads of the CTA: the first n entries of `row` -> m valid slots (returned), It / rn / S filled; ends in a block barrier
template <int W>
__device__ __forceinline__ int dv_stage_sims(const float* __restrict__ F, int U, int I, const int* __restrict__ row, int n, int P,
                                             float* It, float* S, float* rn, int* sid, int* spos) {
    constexpr int L = W == 64 ? 6 : 7;
    __shared__ int s_m;
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid < 32) {
        int base = 0;
        for (int r0 = 0; r0 < n; r0 += 32) {
            const int r = r0 + lane;
            const int id = r < n ? row[r] : -1;
            const bool ok = id >= 0 && id < I;
            const unsigned b = __ballot_sync(0xffffffffu, ok);
            if (ok) {
                const int s = base + __popc(b & ((1u << lane) - 1u));
                sid[s] = id;
                spos[s] = r;
            }
            base += __popc(b);
        }
        if (lane == 0) s_m = base;
    }
    __syncthreads();
    const int m = s_m;
    // slot-fastest: consecutive lanes write consecutive words of It; a row's 16-byte pieces come from L1 after its first one
    for (int idx = tid; idx < P * (W / 4); idx += DV_THREADS) {
        const int s = idx % P, q = idx / P;
        const float4 v = s < m ? ld_gather4(F + ((int64_t)U + sid[s]) * W + q * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        It[(q * 4 + 0) * P + s] = v.x; It[(q * 4 + 1) * P + s] = v.y;
        It[(q * 4 + 2) * P + s] = v.z; It[(q * 4 + 3) * P + s] = v.w;
    }
    __syncthreads();
    if (tid < m) {       // the tree of item_rnorm_kernel, so the bits of the similar-item lists' norms
        TreeN<L> t;
#pragma unroll
        for (int d = 0; d < W; ++d) {
            const float x = It[d * P + tid];
            t.add(d, __fmul_rn(x, x));
        }
        const float sum = t.st[L - 1];
        rn[tid] = sum > 0.f ? __fdiv_rn(1.f, __fsqrt_rn(sum)) : 0.f;
    }
    __syncthreads();
    // blocks (A, B): rows 2A, 2A+1, columns 4B..4B+3; row block A needs the column blocks B >= A/2 (some b > a), so the blocks are
    // enumerated row block by row block, nB - A/2 of them each
    const int nA = (m + 1) >> 1, nB = (m + 3) >> 2;
    int total = 0;
    for (int A = 0; A < nA; ++A) total += nB - (A >> 1);
    int A = 0, c0 = 0;
    for (int t = tid; t < total; t += DV_THREADS) {
        while (t >= c0 + nB - (A >> 1)) { c0 += nB - (A >> 1); ++A; }
        const int B = (A >> 1) + (t - c0);
        TreeN<L> tr[2][4];
#pragma unroll
        for (int d = 0; d < W; ++d) {
            const float2 x = *reinterpret_cast<const float2*>(It + d * P + 2 * A);
            const float4 y = *reinterpret_cast<const float4*>(It + d * P + 4 * B);
            tr[0][0].add(d, __fmul_rn(x.x, y.x)); tr[0][1].add(d, __fmul_rn(x.x, y.y));
            tr[0][2].add(d, __fmul_rn(x.x, y.z)); tr[0][3].add(d, __fmul_rn(x.x, y.w));
            tr[1][0].add(d, __fmul_rn(x.y, y.x)); tr[1][1].add(d, __fmul_rn(x.y, y.y));
            tr[1][2].add(d, __fmul_rn(x.y, y.z)); tr[1][3].add(d, __fmul_rn(x.y, y.w));
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int a = 2 * A + i;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int b = 4 * B + j;
                if (a < b && b < m) {
                    const float s = __fmul_rn(__fmul_rn(tr[i][j].st[L - 1], rn[a]), rn[b]);   // the lower slot (rank) first
                    S[a * P + b] = s;
                    S[b * P + a] = s;
                }
            }
        }
    }
    __syncthreads();
    return m;
}

template <int W>
__global__ void __launch_bounds__(DV_THREADS) list_diversity_kernel(const float* __restrict__ F, int U, int I, const int* __restrict__ top_ids,
                                                                    int K_list, DivKs ks, double* __restrict__ rows) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int j = blockIdx.x, tid = threadIdx.x;
    const int nk = ks.n, kmax = ks.k[nk - 1];
    const int P = dv_slots(kmax);
    double* R = reinterpret_cast<double*>(smem_raw);             // [P] r_b
    float* It = reinterpret_cast<float*>(R + P);                 // [W][P]
    float* S = It + W * P;                                       // [P][P]
    float* rn = S + P * P;
    int* sid = reinterpret_cast<int*>(rn + P);
    int* spos = sid + P;
    const int m = dv_stage_sims<W>(F, U, I, top_ids + (int64_t)j * K_list, kmax, P, It, S, rn, sid, spos);
    for (int b = tid; b < m; b += DV_THREADS) {
        double r = 0.0;
        for (int a = 0; a < b; ++a) r = __dadd_rn(r, __dsub_rn(1.0, (double)S[a * P + b]));
        R[b] = r;
    }
    __syncthreads();
    if (tid < nk) {
        const int k = ks.k[tid];
        int mq = 0;                    // slots are in rank order: the valid entries among the first k are slots 0..mq-1
        while (mq < m && spos[mq] < k) ++mq;
        double num = 0.0;
        for (int b = 1; b < mq; ++b) num = __dadd_rn(num, R[b]);
        rows[(int64_t)j * nk + tid] = mq < 2 ? 0.0 : __ddiv_rn(num, (double)(mq * (mq - 1) / 2));
    }
}

template <int W>
__global__ void __launch_bounds__(DV_THREADS) mmr_rerank_kernel(const float* __restrict__ F, int U, int I, const int* __restrict__ cand_ids,
                                                                const float* __restrict__ cand_scores, int N, int K, float lam,
                                                                int* __restrict__ out_ids, float* __restrict__ out_scores) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int j = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int P = dv_slots(N);
    float* It = reinterpret_cast<float*>(smem_raw);
    float* S = It + W * P;
    float* rn = S + P * P;
    int* sid = reinterpret_cast<int*>(rn + P);
    int* spos = sid + P;
    const int m = dv_stage_sims<W>(F, U, I, cand_ids + (int64_t)j * N, N, P, It, S, rn, sid, spos);
    if (tid >= 32) return;
    const float* sc_row = cand_scores + (int64_t)j * N;
    float sc[4], rel[4], mx[4];
    bool open[4];
    float smax = -INFINITY, smin = INFINITY;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int c = lane + 32 * q;
        open[q] = c < m;
        sc[q] = open[q] ? sc_row[spos[c]] : 0.f;
        mx[q] = 0.f;
        if (open[q]) { smax = fmaxf(smax, sc[q]); smin = fminf(smin, sc[q]); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        smax = fmaxf(smax, __shfl_xor_sync(0xffffffffu, smax, o));
        smin = fminf(smin, __shfl_xor_sync(0xffffffffu, smin, o));
    }
    const bool spread = smax > smin;
    const float range = spread ? __fsub_rn(smax, smin) : 1.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) rel[q] = open[q] && spread ? __fdiv_rn(__fsub_rn(sc[q], smin), range) : 0.f;
    const float oml = __fsub_rn(1.f, lam);
    int* oi = out_ids + (int64_t)j * K;
    float* os = out_scores + (int64_t)j * K;
    const int picks = min(K, m);
    for (int step = 0; step < picks; ++step) {
        float bv = -INFINITY;
        int bp = 0x7fffffff;
#pragma unroll
        for (int q = 0; q < 4; ++q) {           // ascending slots, so a lane's ties keep the lower one
            const float v = __fsub_rn(__fmul_rn(lam, rel[q]), __fmul_rn(oml, mx[q]));
            if (open[q] && better(v, lane + 32 * q, bv, bp)) { bv = v; bp = lane + 32 * q; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int op = __shfl_xor_sync(0xffffffffu, bp, o);
            if (better(ov, op, bv, bp)) { bv = ov; bp = op; }
        }
        // NaN values (non-finite scores or features) rank below every number: `better` takes none of them, and when every open
        // value is NaN the lowest open slot is the pick (bp is warp-uniform here; finite values are never -inf, lam * rel being in
        // [0, 1] and m(c) a finite cosine or NaN)
        if (bp == 0x7fffffff) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const unsigned b = __ballot_sync(0xffffffffu, open[q]);
                if (b) { bp = 32 * q + __ffs(b) - 1; break; }
            }
        }
        if (lane == (bp & 31)) {
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (bp == lane + 32 * q) { open[q] = false; oi[step] = sid[bp]; os[step] = sc[q]; }
        }
        const float* srow = S + bp * P;         // sim(c, pick) with the lower slot first: both halves of S hold it
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int c = lane + 32 * q;
            if (open[q]) mx[q] = step == 0 ? srow[c] : fmaxf(mx[q], srow[c]);
        }
    }
    for (int k = picks + lane; k < K; k += 32) { oi[k] = -1; os[k] = 0.f; }
}

}  // namespace ngacf

using namespace ngacf;

template <int W>
static void launch_list_diversity(const float* F, int U, int I, const int* top_ids, int K_list, int n_rows, const DivKs& ks, double* rows,
                                  cudaStream_t st) {
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(list_diversity_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dv_smem(W, DV_MAX, true));
    });
    list_diversity_kernel<W><<<n_rows, DV_THREADS, dv_smem(W, dv_slots(ks.k[ks.n - 1]), true), st>>>(F, U, I, top_ids, K_list, ks, rows);
}

template <int W>
static void launch_mmr(const float* F, int U, int I, const int* cand_ids, const float* cand_scores, int n_rows, int N, int K, float lam,
                       int* out_ids, float* out_scores, cudaStream_t st) {
    static PerDeviceOnce once;
    once.run([] {
        cudaFuncSetAttribute(mmr_rerank_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dv_smem(W, DV_MAX, false));
    });
    mmr_rerank_kernel<W><<<n_rows, DV_THREADS, dv_smem(W, dv_slots(N), false), st>>>(F, U, I, cand_ids, cand_scores, N, K, lam, out_ids,
                                                                                     out_scores);
}

extern "C" int ngacf_list_diversity(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* top_ids, int32_t K_list,
                                    int32_t n_rows, const int32_t* ks, int32_t n_ks, double* rows, void* stream) {
    if (!width_supported(width)) { set_error("list_diversity: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    if (K_list < 1 || K_list > NGACF_RECOMMEND_MAX_K) {
        set_error("list_diversity: list length %d is outside 1..%d", K_list, NGACF_RECOMMEND_MAX_K);
        return NGACF_ERR_UNSUPPORTED;
    }
    if (n_ks < 1 || n_ks > NGACF_CUTOFF_MAX_KS) {
        set_error("list_diversity: %d cut-offs, 1..%d are supported", n_ks, NGACF_CUTOFF_MAX_KS);
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(ks, "list_diversity: null cut-off array");
    DivKs kp{};
    kp.n = n_ks;
    for (int q = 0; q < n_ks; ++q) {
        if (ks[q] < 1 || ks[q] > K_list || (q > 0 && ks[q] <= ks[q - 1])) {
            set_error("list_diversity: cut-offs must be strictly increasing in 1..%d (the list length); cut-off %d is %d", K_list, q, ks[q]);
            return NGACF_ERR_UNSUPPORTED;
        }
        kp.k[q] = ks[q];
    }
    NGACF_REQUIRE(F && top_ids && rows, "list_diversity: null features, lists or rows");
    NGACF_REQUIRE(n_rows >= 0 && U >= 0 && I >= 0, "list_diversity: negative row, user or item count");
    if (n_rows == 0) return NGACF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (width == 64) launch_list_diversity<64>(F, U, I, top_ids, K_list, n_rows, kp, rows, st);
    else launch_list_diversity<128>(F, U, I, top_ids, K_list, n_rows, kp, rows, st);
    return check_launch("list_diversity");
}

extern "C" int ngacf_mmr_rerank(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* cand_ids, const float* cand_scores,
                                int32_t n_rows, int32_t N, int32_t K, float lam, int32_t* out_ids, float* out_scores, void* stream) {
    if (!width_supported(width)) { set_error("mmr_rerank: width %d is not built (supported: 64, 128)", width); return NGACF_ERR_UNSUPPORTED; }
    if (N < 1 || N > NGACF_RECOMMEND_MAX_K) { set_error("mmr_rerank: N = %d candidates is outside 1..%d", N, NGACF_RECOMMEND_MAX_K); return NGACF_ERR_UNSUPPORTED; }
    if (K < 1 || K > N) { set_error("mmr_rerank: K = %d is outside 1..%d (the candidates)", K, N); return NGACF_ERR_UNSUPPORTED; }
    NGACF_REQUIRE(F && cand_ids && cand_scores && out_ids && out_scores, "mmr_rerank: null features, candidates or outputs");
    NGACF_REQUIRE(lam >= 0.f && lam <= 1.f, "mmr_rerank: lambda %g is not in [0, 1]", (double)lam);
    NGACF_REQUIRE(n_rows >= 0 && U >= 0 && I >= 0, "mmr_rerank: negative row, user or item count");
    if (n_rows == 0) return NGACF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (width == 64) launch_mmr<64>(F, U, I, cand_ids, cand_scores, n_rows, N, K, lam, out_ids, out_scores, st);
    else launch_mmr<128>(F, U, I, cand_ids, cand_scores, n_rows, N, K, lam, out_ids, out_scores, st);
    return check_launch("mmr_rerank");
}
