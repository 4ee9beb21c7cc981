// Beyond-accuracy statistics of ranked lists and per-group column sums.
//   ngacf_list_stats: one warp per list row.  Exposure: each valid entry at rank r adds 1 (integer atomics: deterministic) to the
//     bucket of the first cut-off k > r, and a second kernel turns the buckets into the counts at each cut-off by a prefix over the
//     cut-offs.  Per-row means of fp64 item tables: each lane gathers the values of its list positions, then the whole warp walks the
//     positions in rank order through shuffles, so the sum at each cut-off is the sequential fp64 sum a numpy loop gives.
//   ngacf_group_sums: fp64 column sums of rows per group, block partials in a fixed order, then one warp per (group, column) as in
//     cutoff_metrics_reduce_kernel: two runs give the same bits.
#include "common.cuh"

namespace ngacf {

constexpr int LS_WARPS = 8;            // list rows per CTA
constexpr int GS_ROWS = 256;           // rows per CTA of the group sums
constexpr int GS_SLICES = 4;           // row slices per CTA (256 threads = 4 slices x 64 columns)
constexpr int GS_COLS = 64;

struct ListKs {                        // by value in the kernel parameters: CUDA-graph replay safe
    int32_t n;
    int32_t k[NGACF_CUTOFF_MAX_KS];
};

__global__ void __launch_bounds__(LS_WARPS * 32) list_stats_kernel(const int* __restrict__ top_ids, int K_list, int n_rows, int I,
                                                                  ListKs ks, const double* __restrict__ item_vals, int n_vals,
                                                                  int* __restrict__ counts, double* __restrict__ rows) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * LS_WARPS + warp;
    if (j >= n_rows) return;           // warp-uniform
    const int nk = ks.n, kmax = ks.k[nk - 1];
    int id[4];
    unsigned m[4];                     // bit b of m[w]: list position 32 w + b holds a valid id
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const int r = 32 * w + lane;
        id[w] = r < kmax ? top_ids[(int64_t)j * K_list + r] : -1;
        const bool ok = id[w] >= 0 && id[w] < I;
        m[w] = __ballot_sync(0xffffffffu, ok);
        if (counts && ok) {
            int q = 0;
            while (ks.k[q] <= r) ++q;  // first cut-off that includes rank r (r < kmax)
            atomicAdd(counts + (int64_t)q * I + id[w], 1);
        }
    }
    if (!rows || n_vals == 0) return;
    int cnt = 0;                       // lane q < nk: valid entries among the first k_q
    if (lane < nk) {
        const int k = ks.k[lane];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int lo = 32 * w;
            const unsigned mask = k >= lo + 32 ? 0xffffffffu : (k <= lo ? 0u : (1u << (k - lo)) - 1u);
            cnt += __popc(m[w] & mask);
        }
    }
    for (int v = 0; v < n_vals; ++v) {
        const double* tab = item_vals + (int64_t)v * I;
        double x[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) x[w] = (m[w] >> lane) & 1u ? tab[id[w]] : 0.0;
        double acc = 0.0, mine = 0.0;  // acc: the same rank-order sum on every lane; mine: lane q's snapshot at cut-off q
        int q = 0;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            if (32 * w >= kmax) break;
#pragma unroll 8
            for (int b = 0; b < 32; ++b) {
                const int r = 32 * w + b;
                if (r >= kmax) break;
                const double y = __shfl_sync(0xffffffffu, x[w], b);
                if ((m[w] >> b) & 1u) acc += y;
                if (r + 1 == ks.k[q]) {
                    if (lane == q) mine = acc;
                    ++q;
                }
            }
        }
        if (lane < nk) rows[(int64_t)j * n_vals * nk + v * nk + lane] = cnt > 0 ? mine / (double)cnt : 0.0;
    }
}

// counts[q][i] held the entries whose first including cut-off is q; make them the counts of the first k_q entries
__global__ void list_stats_prefix_kernel(int* __restrict__ counts, int I, int nk) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= I) return;
    int c = 0;
    for (int q = 0; q < nk; ++q) {
        c += counts[(int64_t)q * I + i];
        counts[(int64_t)q * I + i] = c;
    }
}

// thread (s, c) sums column c of rows b*GS_ROWS + s, + 4, + 8, ... of its CTA into its own shared slot per group, in row order;
// the 4 slices are then added in order into the CTA's partial [G][n_cols]
__global__ void __launch_bounds__(GS_SLICES * GS_COLS) group_sums_kernel(const double* __restrict__ rows, int n_rows, int n_cols,
                                                                        const int* __restrict__ group, int G, double* __restrict__ partial) {
    __shared__ double acc[GS_SLICES][NGACF_GROUP_MAX][GS_COLS];
    const int c = threadIdx.x % GS_COLS, s = threadIdx.x / GS_COLS;
    for (int g = 0; g < G; ++g) acc[s][g][c] = 0.0;
    const int r0 = blockIdx.x * GS_ROWS, r1 = min(n_rows, r0 + GS_ROWS);
    if (c < n_cols) {
        for (int r = r0 + s; r < r1; r += GS_SLICES) {
            const int g = group[r];
            if (g < 0 || g >= G) continue;
            acc[s][g][c] += rows[(int64_t)r * n_cols + c];
        }
    }
    __syncthreads();
    if (s == 0 && c < n_cols) {
        for (int g = 0; g < G; ++g) {
            double t = acc[0][g][c];
#pragma unroll
            for (int q = 1; q < GS_SLICES; ++q) t += acc[q][g][c];
            partial[((int64_t)blockIdx.x * G + g) * n_cols + c] = t;
        }
    }
}

// one warp per (group, column): lane l sums blocks l, l+32, ... in order, then a fixed shuffle tree
__global__ void __launch_bounds__(32) group_sums_reduce_kernel(const double* __restrict__ partial, int nblocks, int nv, double* __restrict__ sums) {
    const int c = blockIdx.x, lane = threadIdx.x;
    double acc = 0.0;
    for (int b = lane; b < nblocks; b += 32) acc += partial[(int64_t)b * nv + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) sums[c] = acc;
}

}  // namespace ngacf

using namespace ngacf;

extern "C" int ngacf_list_stats(const int32_t* top_ids, int32_t K_list, int32_t n_rows, int32_t I, const int32_t* ks, int32_t n_ks,
                                const double* item_vals, int32_t n_vals, int32_t* counts, double* rows, void* stream) {
    if (K_list < 1 || K_list > NGACF_RECOMMEND_MAX_K) {
        set_error("list_stats: list length %d is outside 1..%d", K_list, NGACF_RECOMMEND_MAX_K);
        return NGACF_ERR_UNSUPPORTED;
    }
    if (n_ks < 1 || n_ks > NGACF_CUTOFF_MAX_KS) {
        set_error("list_stats: %d cut-offs, 1..%d are supported", n_ks, NGACF_CUTOFF_MAX_KS);
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(ks, "list_stats: null cut-off array");
    ListKs kp{};
    kp.n = n_ks;
    for (int q = 0; q < n_ks; ++q) {
        if (ks[q] < 1 || ks[q] > K_list || (q > 0 && ks[q] <= ks[q - 1])) {
            set_error("list_stats: cut-offs must be strictly increasing in 1..%d (the list length); cut-off %d is %d", K_list, q, ks[q]);
            return NGACF_ERR_UNSUPPORTED;
        }
        kp.k[q] = ks[q];
    }
    if (n_vals < 0 || n_vals > NGACF_LIST_MAX_VALS) {
        set_error("list_stats: %d item tables, 0..%d are supported", n_vals, NGACF_LIST_MAX_VALS);
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(n_rows >= 0 && I >= 0, "list_stats: negative row or item count");
    NGACF_REQUIRE(n_rows == 0 || top_ids, "list_stats: null lists");
    NGACF_REQUIRE(!rows || n_vals == 0 || item_vals, "list_stats: null item tables");
    cudaStream_t st = (cudaStream_t)stream;
    if (counts && I > 0) {
        const cudaError_t e = cudaMemsetAsync(counts, 0, (size_t)n_ks * I * sizeof(int32_t), st);
        if (e != cudaSuccess) {
            set_error("list_stats: zeroing the counts: CUDA error %d (%s)", (int)e, cudaGetErrorString(e));
            return NGACF_ERR_CUDA;
        }
    }
    if (n_rows > 0 && (counts || (rows && n_vals > 0)))
        list_stats_kernel<<<ceil_div(n_rows, LS_WARPS), LS_WARPS * 32, 0, st>>>(top_ids, K_list, n_rows, I, kp, item_vals, n_vals, counts, rows);
    if (counts && I > 0 && n_rows > 0 && n_ks > 1) list_stats_prefix_kernel<<<ceil_div(I, 256), 256, 0, st>>>(counts, I, n_ks);
    return check_launch("list_stats");
}

extern "C" size_t ngacf_group_sums_workspace_bytes(int32_t n_rows, int32_t n_cols, int32_t G) {
    if (n_cols < 1 || n_cols > NGACF_GROUP_MAX_COLS || G < 1 || G > NGACF_GROUP_MAX) return 0;
    return (size_t)ceil_div(n_rows > 0 ? n_rows : 1, GS_ROWS) * G * n_cols * sizeof(double);
}

extern "C" int ngacf_group_sums(const double* rows, int32_t n_rows, int32_t n_cols, const int32_t* group, int32_t G, double* sums,
                                void* workspace, size_t workspace_bytes, void* stream) {
    if (n_cols < 1 || n_cols > NGACF_GROUP_MAX_COLS) {
        set_error("group_sums: %d columns, 1..%d are supported", n_cols, NGACF_GROUP_MAX_COLS);
        return NGACF_ERR_UNSUPPORTED;
    }
    if (G < 1 || G > NGACF_GROUP_MAX) {
        set_error("group_sums: %d groups, 1..%d are supported", G, NGACF_GROUP_MAX);
        return NGACF_ERR_UNSUPPORTED;
    }
    NGACF_REQUIRE(sums && workspace && n_rows >= 0, "group_sums: null sums / workspace or negative row count");
    const size_t need = ngacf_group_sums_workspace_bytes(n_rows, n_cols, G);
    if (workspace_bytes < need) {
        set_error("group_sums: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return NGACF_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (n_rows == 0) {
        const cudaError_t e = cudaMemsetAsync(sums, 0, (size_t)G * n_cols * sizeof(double), st);
        if (e != cudaSuccess) {
            set_error("group_sums: zeroing the sums: CUDA error %d (%s)", (int)e, cudaGetErrorString(e));
            return NGACF_ERR_CUDA;
        }
        return NGACF_OK;
    }
    NGACF_REQUIRE(rows && group, "group_sums: null argument");
    const int nblocks = ceil_div(n_rows, GS_ROWS);
    group_sums_kernel<<<nblocks, GS_SLICES * GS_COLS, 0, st>>>(rows, n_rows, n_cols, group, G, (double*)workspace);
    group_sums_reduce_kernel<<<G * n_cols, 32, 0, st>>>((const double*)workspace, nblocks, G * n_cols, sums);
    return check_launch("group_sums");
}
