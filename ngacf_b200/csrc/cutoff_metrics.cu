// Full-ranking metrics at up to NGACF_CUTOFF_MAX_KS cut-offs over ranked lists of any length up to NGACF_RECOMMEND_MAX_K, with the
// standard ideal DCG (min(|test|, k) hits).  One warp per user: lanes test list positions r, r+32, r+64, r+96 against the user's
// sorted test items, __ballot_sync gathers a 128-bit hit mask, and lane q evaluates cut-off q from popcounts of that mask.  Per-user
// rows, then fixed-order sums (block partials, then one warp per column), so two runs give the same bits.
#include "common.cuh"

namespace ngacf {

constexpr int CM_WARPS = 8;            // users per CTA
constexpr int CM_COLS = 5 * NGACF_CUTOFF_MAX_KS;

struct CutoffKs {                      // by value in the kernel parameters: no symbol copy per call, CUDA-graph replay safe
    int32_t n;
    int32_t k[NGACF_CUTOFF_MAX_KS];
};

// 1 / log2(r + 2), r = 0..99: the bits of numpy's 1.0 / np.log2(np.arange(2, 102)) (hex literals, exact)
__constant__ double c_cut_disc[NGACF_RECOMMEND_MAX_K] = {
    0x1.0000000000000p+0, 0x1.430939835353ep-1, 0x1.0000000000000p-1, 0x1.b903469050f73p-2,
    0x1.8c23246dc0aa0p-2, 0x1.6cc193acea9b5p-2, 0x1.5555555555555p-2, 0x1.430939835353ep-2,
    0x1.34413509f79ffp-2, 0x1.28009c1dd6454p-2, 0x1.1da3383416064p-2, 0x1.14b94f8d9641fp-2,
    0x1.0cf3ffed2d6acp-2, 0x1.0619dc46d3e15p-2, 0x1.0000000000000p-2, 0x1.f50b57eac5885p-3,
    0x1.eb22cc68aa6e3p-3, 0x1.e21e1180c5dabp-3, 0x1.d9dcd21439834p-3, 0x1.d244c78367a0dp-3,
    0x1.cb40589ac173ep-3, 0x1.c4bd95ba8d72bp-3, 0x1.bead76898f8cep-3, 0x1.b903469050f73p-3,
    0x1.b3b433f2eb070p-3, 0x1.aeb6f759c46fdp-3, 0x1.aa038eb0e3bfep-3, 0x1.a593062b38d8dp-3,
    0x1.a15f4c32b95a3p-3, 0x1.9d630dccc7ddfp-3, 0x1.999999999999ap-3, 0x1.95fec808a6094p-3,
    0x1.928ee7b0b4f23p-3, 0x1.8f46acf8c06e3p-3, 0x1.8c23246dc0aa0p-3, 0x1.8921a744e1aedp-3,
    0x1.863fd1a4a3053p-3, 0x1.837b7a642195ep-3, 0x1.80d2abffdfee9p-3, 0x1.7e439e8fed2b0p-3,
    0x1.7bccb2952736ep-3, 0x1.796c6c7b22305p-3, 0x1.772170b2747aap-3, 0x1.74ea804c2020fp-3,
    0x1.72c67602d3540p-3, 0x1.70b443a1f7c88p-3, 0x1.6eb2efbd2c1adp-3, 0x1.6cc193acea9b5p-3,
    0x1.6adf59c6e689dp-3, 0x1.690b7bca1f15ep-3, 0x1.67454177dda00p-3, 0x1.658bff53d6bf2p-3,
    0x1.63df15867d0dep-3, 0x1.623deedd496bap-3, 0x1.60a7ffe55458ap-3, 0x1.5f1cc61d1c5f1p-3,
    0x1.5d9bc73ac2288p-3, 0x1.5c2490845f2f3p-3, 0x1.5ab6b6386aaa4p-3, 0x1.5951d3046396fp-3,
    0x1.57f587883063fp-3, 0x1.56a179e4d652cp-3, 0x1.5555555555555p-3, 0x1.5410c9d09a12cp-3,
    0x1.52d38bb397b32p-3, 0x1.519d5372b6ce4p-3, 0x1.506ddd51defe8p-3, 0x1.4f44e92275a60p-3,
    0x1.4e223a06beda9p-3, 0x1.4d05963a1d8a7p-3, 0x1.4beec6ddbe115p-3, 0x1.4add97c942e46p-3,
    0x1.49d1d75f15f0ep-3, 0x1.48cb56640af5fp-3, 0x1.47c9e7da07ae1p-3, 0x1.46cd60dd6e321p-3,
    0x1.45d598850cb5ap-3, 0x1.44e267c45bba2p-3, 0x1.43f3a94fd9227p-3, 0x1.430939835353ep-3,
    0x1.4222f649fbc95p-3, 0x1.4140bf081c4a9p-3, 0x1.406274864d58fp-3, 0x1.3f87f8de0f744p-3,
    0x1.3eb12f67ab8e2p-3, 0x1.3dddfca9417e7p-3, 0x1.3d0e4646ed7c2p-3, 0x1.3c41f2f3ef9fbp-3,
    0x1.3b78ea64c23f4p-3, 0x1.3ab315420d981p-3, 0x1.39f05d1c68ad2p-3, 0x1.3930ac60d89e8p-3,
    0x1.3873ee4e00ec7p-3, 0x1.37ba0ee9f8387p-3, 0x1.3702faf8b610bp-3, 0x1.364e9ff30f403p-3,
    0x1.359cebfe36ed5p-3, 0x1.34edcde3bb953p-3, 0x1.34413509f79ffp-3, 0x1.3397116cededfp-3,
};

__global__ void __launch_bounds__(CM_WARPS * 32) cutoff_metrics_kernel(const int* __restrict__ top_ids, int K_list, const int* __restrict__ users,
                                                                      int n_users, const int* __restrict__ test_ptr,
                                                                      const int* __restrict__ test_items, CutoffKs ks,
                                                                      double* __restrict__ per_user, double* __restrict__ partial) {
    __shared__ double rows[CM_WARPS][CM_COLS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * CM_WARPS + warp;
    const int nk = ks.n, nc = 5 * nk;
    if (j < n_users) {                 // warp-uniform
        const int u = users[j];
        const int beg = test_ptr[u], end = test_ptr[u + 1];
        unsigned m[4];                 // bit b of m[w]: list position 32 w + b is a test item
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int r = 32 * w + lane;
            bool hit = false;
            if (r < K_list) {
                const int id = top_ids[(int64_t)j * K_list + r];
                int lo = beg, hi = end;
                while (id >= 0 && lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    const int v = test_items[mid];
                    if (v == id) { hit = true; break; }
                    if (v < id) lo = mid + 1; else hi = mid;
                }
            }
            m[w] = __ballot_sync(0xffffffffu, hit);
        }
        if (lane < nk) {
            const int k = ks.k[lane];
            const int nt = end - beg;
            const unsigned long long m0 = m[0] | (unsigned long long)m[1] << 32, m1 = m[2] | (unsigned long long)m[3] << 32;
            const unsigned long long a = k >= 64 ? m0 : m0 & ((1ull << k) - 1);            // hits among the first k positions
            const unsigned long long b = k <= 64 ? 0ull : m1 & ((1ull << (k - 64)) - 1);   // k <= 100: shift < 64
            const int h = __popcll(a) + __popcll(b);
            const int first = a ? __ffsll(a) - 1 : (b ? 63 + __ffsll(b) : -1);
            double* row = per_user ? per_user + (int64_t)j * nc + lane : nullptr;
            auto put = [&](int q, double v) {
                rows[warp][q * nk + lane] = v;
                if (row) row[q * nk] = v;
            };
            put(0, (double)h / (double)k);
            put(1, nt > 0 ? (double)h / (double)nt : 0.0);
            put(3, h > 0 ? 1.0 : 0.0);
            put(4, first >= 0 ? 1.0 / (double)(first + 1) : 0.0);
            double dcg = 0.0, idcg = 0.0;   // both summed in rank order
            for (unsigned long long t = a; t; t &= t - 1) dcg += c_cut_disc[__ffsll(t) - 1];
            for (unsigned long long t = b; t; t &= t - 1) dcg += c_cut_disc[63 + __ffsll(t)];
            const int ideal = min(nt, k);
            for (int r = 0; r < ideal; ++r) idcg += c_cut_disc[r];
            put(2, idcg > 0.0 ? dcg / idcg : 0.0);
        }
    } else if (lane < nk) {
#pragma unroll
        for (int q = 0; q < 5; ++q) rows[warp][q * nk + lane] = 0.0;
    }
    __syncthreads();
    if (threadIdx.x < nc) {            // fixed-order sum over the block's users
        double acc = 0.0;
#pragma unroll
        for (int w = 0; w < CM_WARPS; ++w) acc += rows[w][threadIdx.x];
        partial[(int64_t)blockIdx.x * nc + threadIdx.x] = acc;
    }
}

// one warp per column: lane l sums blocks l, l+32, ... in order, then a fixed shuffle tree
__global__ void __launch_bounds__(32) cutoff_metrics_reduce_kernel(const double* __restrict__ partial, int nblocks, int nc, double* __restrict__ sums) {
    const int c = blockIdx.x, lane = threadIdx.x;
    double acc = 0.0;
    for (int b = lane; b < nblocks; b += 32) acc += partial[(int64_t)b * nc + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) sums[c] = acc;
}

}  // namespace ngacf

using namespace ngacf;

extern "C" size_t ngacf_cutoff_metrics_workspace_bytes(int32_t n_users, int32_t n_ks) {
    if (n_ks < 1 || n_ks > NGACF_CUTOFF_MAX_KS) return 0;
    return (size_t)ceil_div(n_users > 0 ? n_users : 1, CM_WARPS) * 5 * n_ks * sizeof(double);
}

extern "C" int ngacf_cutoff_metrics(const int32_t* top_ids, int32_t K_list, const int32_t* users, int32_t n_users, const int32_t* test_ptr,
                                    const int32_t* test_items, const int32_t* ks, int32_t n_ks, double* sums, double* per_user,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    if (K_list < 1 || K_list > NGACF_RECOMMEND_MAX_K) {
        set_error("cutoff_metrics: list length %d is outside 1..%d", K_list, NGACF_RECOMMEND_MAX_K);
        return NGACF_ERR_UNSUPPORTED;
    }
    if (n_ks < 1 || n_ks > NGACF_CUTOFF_MAX_KS) {
        set_error("cutoff_metrics: %d cut-offs, 1..%d are supported", n_ks, NGACF_CUTOFF_MAX_KS);
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(ks, "cutoff_metrics: null cut-off array");
    CutoffKs kp{};
    kp.n = n_ks;
    for (int q = 0; q < n_ks; ++q) {
        if (ks[q] < 1 || ks[q] > K_list || (q > 0 && ks[q] <= ks[q - 1])) {
            set_error("cutoff_metrics: cut-offs must be strictly increasing in 1..%d (the list length); cut-off %d is %d", K_list, q, ks[q]);
            return NGACF_ERR_UNSUPPORTED;
        }
        kp.k[q] = ks[q];
    }
    NGACF_REQUIRE(sums && workspace && n_users >= 0, "cutoff_metrics: null sums / workspace or negative user count");
    const size_t need = ngacf_cutoff_metrics_workspace_bytes(n_users, n_ks);
    if (workspace_bytes < need) {
        set_error("cutoff_metrics: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return NGACF_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (n_users == 0) { cudaMemsetAsync(sums, 0, 5 * n_ks * sizeof(double), st); return check_launch("cutoff_metrics"); }
    NGACF_REQUIRE(top_ids && users && test_ptr && test_items, "cutoff_metrics: null argument");
    const int nblocks = ceil_div(n_users, CM_WARPS);
    cutoff_metrics_kernel<<<nblocks, CM_WARPS * 32, 0, st>>>(top_ids, K_list, users, n_users, test_ptr, test_items, kp, per_user,
                                                             (double*)workspace);
    cutoff_metrics_reduce_kernel<<<5 * n_ks, 32, 0, st>>>((const double*)workspace, nblocks, 5 * n_ks, sums);
    return check_launch("cutoff_metrics");
}
