/*
 * ngacf_b200 -- C-ABI of the B200-native SPUIGACF propagation-and-scoring hot path.
 *
 * The reference (cleverer123/NGACF) has no FFI: its boundary for this path is the Python call surface
 * of graphattention/SPUIGACF.py, graphattention/BPRLoss.py and train_eval_Gowalla.py (SURVEY.md 8b).
 * Every entry point below replaces one or more reference call sites and says which (file:line relative
 * to the reference root).  INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is DEVICE memory unless the name ends in _host;
 *   - the caller owns every buffer; nothing is allocated, freed or synchronised here, so every call
 *     is CUDA-graph capturable (ngacf_graph_build is the one documented exception: it is a build-time
 *     call, still async, and reports its data-dependent sizes through a device counter array);
 *   - `stream` is a cudaStream_t passed as void*;
 *   - return value: NGACF_OK or a negative NGACF_ERR_* code; ngacf_last_error() gives the text;
 *   - all float tensors are fp32 row-major with 64 columns (embedSize 64 of every BASELINE config); the `_w` variants at the
 *     end take other row widths (embedSize 128);
 *   - node numbering: users 0..U-1 then items U..U+I-1 ("features" layout of SPUIGACF.py:38);
 *   - H = heads of a stage: 8 (eight 64->8 heads, SPUIGACF.py:191-198) or 1 (out_att 64->64, :200-205).
 */
#ifndef NGACF_B200_H
#define NGACF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NGACF_OK 0
#define NGACF_ERR_INVALID_ARG (-1)
#define NGACF_ERR_CUDA (-2)
#define NGACF_ERR_WORKSPACE (-3)
#define NGACF_ERR_UNSUPPORTED (-4)

#define NGACF_D 64            /* embedding width */
#define NGACF_CHUNK 128       /* max edges per aggregation task (degree bucketing granularity) */
#define NGACF_TOPK 20         /* K_max of eval_neg_all (train_eval_Gowalla.py:276,375) */

const char* ngacf_last_error(void);
int ngacf_version(void);

/* ---------------------------------------------------------------------------------------------
 * (a1) graph builder.  Replaces get_adj_mat/buildLaplacianMat('ui_mat')/scipySP_torchSP/.coalesce()
 * (data/loadGowalla.py:179-186,218-219,229-253) and the per-call COO rebuild + coalesce sort of
 * SPUIGACF.py:365,377.  Input: COO (u,i) int64, any order, duplicates allowed.  Output: coalesced CSR,
 * CSC, CSC->CSR edge permutation, the unified node adjacency used by the aggregation kernels and the
 * degree-bucketed task list.
 *
 * counts[0]=E (unique edges) counts[1]=T (tasks) counts[2]=L (long rows, >NGACF_CHUNK edges)
 * counts[3]=S (scratch slots) counts[4]=#users with zero edges (reference asserts 0, SPUIGACF.py:368)
 * counts[5]=#out-of-range input edges  counts[6]=T_u: tasks [0,T_u) are user rows, [T_u,T) item rows;
 * inside a side the tasks are ordered longest first (the degree buckets).  Buffer capacities: *_idx/perm/adj_* for E_in edges,
 * tasks for (U+I)+2*E_in/NGACF_CHUNK entries of 4 ints, long_* for 2*E_in/NGACF_CHUNK+1 ints.
 * ------------------------------------------------------------------------------------------- */
size_t ngacf_graph_build_workspace_bytes(int64_t E_in, int32_t U, int32_t I);
int ngacf_graph_build(const int64_t* coo_u, const int64_t* coo_i, int64_t E_in, int32_t U, int32_t I,
                      int32_t* rowptr, int32_t* colidx, int32_t* colptr, int32_t* rowidx, int32_t* perm,
                      int32_t* adj_ptr, int32_t* adj_idx, int32_t* adj_eid,
                      int32_t* tasks /* [cap][4] = node,beg,end,long_id|-1 */,
                      int32_t* long_first_slot, int32_t* long_counter,
                      int32_t* counts /* [8] */, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * dropout keep masks (specified Philox4x32-10 streams; the reference draws from torch's global
 * generator at SPUIGACF.py:208,213 (features) and :375 (edges), which no custom kernel can replay).
 * feat: uint64[N], bit d = keep (n,d).  edge: uint8[E], bit k = keep (edge e, head k).
 * ------------------------------------------------------------------------------------------- */
int ngacf_feature_mask(uint64_t* feat, int64_t N, uint64_t seed, uint32_t call, const int64_t* call_dev, uint32_t stage, float droprate, void* stream);
int ngacf_edge_mask(uint8_t* edge, int64_t E, int32_t H, uint64_t seed, uint32_t call, const int64_t* call_dev, uint32_t stage, float droprate, void* stream);
/* all S stages of one propagation in ONE launch: feat/edge/heads are HOST arrays of S entries (device pointers / head counts);
 * stage k uses Philox sites 2k / 2k+1 -- identical bits to S pairs of the two calls above. */
int ngacf_dropout_masks(uint64_t* const* feat, uint8_t* const* edge, const int32_t* heads, int32_t S, int64_t N, int64_t E,
                        uint64_t seed, uint32_t call, const int64_t* call_dev, float droprate, void* stream);
/* the same streams restricted to the node ranges [fa0,fb0) and [fa1,fb1) and the edge range [e0,e1), written at their global
 * positions (multi-GPU user sharding: a rank needs the masks of the rows it transforms and of the edges it owns only) */
int ngacf_dropout_masks_ranges(uint64_t* const* feat, uint8_t* const* edge, const int32_t* heads, int32_t S, int64_t fa0, int64_t fb0,
                               int64_t fa1, int64_t fb1, int64_t e0, int64_t e1, uint64_t seed, uint32_t call, const int64_t* call_dev,
                               float droprate, void* stream);
/* call_dev (may be NULL): device-resident int64 added to `call` at run time; likewise ngacf_sample_pairs'
 * row_dev = int64[2] {added to row_begin, added to epoch}.  A CUDA graph captured once then replays with
 * advancing dropout streams, train rows and epochs. */
int ngacf_counter_add(int64_t* counter, int64_t delta, void* stream);

/* ---------------------------------------------------------------------------------------------
 * (a3,a5,a6) dense transform: h = dropout(act(X)) @ [W_0..W_{H-1}],  s[n,k] = a_k . h[n, head k].
 * Replaces getFeatureMat (SPUIGACF.py:30-39), F.dropout (:208,213), the 2x torch.mm of every head
 * (:356-357) and the `a.mm(edge_h)` logit (:359-361, which is rank-1: s[u]+s[i]).
 * Xu/Xi: stage input rows of users/items (embedding tables for stage 0; Z_prev, Z_prev+64*U after).
 * apply_elu: input is a pre-activation (ELU applied on load, SPUIGACF.py:397-398).
 * wtab: device array of 3*H pointers [W_u heads | W_i heads | a heads], the reference's own
 * parameter tensors (64,DH) and (1,2*DH).  U or I may be 0 (row-sharded multi-GPU calls process one side,
 * with every pointer pre-offset to the first row; ngacf_transform_bwd then leaves the absent side's gradients untouched).
 * Implementation: tcgen05 tensor cores with fp32-class operand splits (3xTF32 forward and dX; three-term bf16 for the fused
 * backward, whose dW product needs MN-major operands) -- csrc/transform_tc.cu; the environment variable NGACF_DENSE=ffma,
 * read once per process, selects the CUDA-core kernels instead (parity triage).  Errors vs an fp64 product: 2-7e-7 either way.
 * ------------------------------------------------------------------------------------------- */
int ngacf_transform_fwd(const float* Xu, const float* Xi, int32_t apply_elu, const uint64_t* featmask, float scale,
                        const float* const* wtab, int32_t H, int32_t U, int32_t I, float* h, float* s, void* stream);

/* ---------------------------------------------------------------------------------------------
 * (a6-a9) fused edge softmax + neighbour aggregation, both sides in one launch:
 *   e = exp(-LeakyReLU_0.2(s[n]+s[m])), norm[n] = sum_m e, Z[n] = h[n] + sum_m drop(e) h[m] / norm[n]
 * Replaces SPUIGACF.py:359-391 (2 sparse_coo_tensor + 2 coalesce + 4 sparse.mm + div + NaN->0).
 * Z is PRE-ELU; the consumer applies ELU (:397-398, :214).  scratch: S*(64+8) floats.
 * ------------------------------------------------------------------------------------------- */
int ngacf_aggregate_fwd(const int32_t* tasks, int32_t T, const int32_t* adj_ptr, const int32_t* adj_idx, const int32_t* adj_eid,
                        const int32_t* long_first_slot, int32_t* long_counter, float* scratch,
                        const float* h, const float* s, int32_t H, const uint8_t* edgemask, float scale,
                        float* Z, float* norm, int32_t partial_from, void* stream);
/* Multi-GPU user sharding: tasks with index >= partial_from (pass T_u; -1 = none) hold only this rank's slice of
 * a row's edges and write raw partials (sum in Z, weight sum in norm); after the cross-rank sum (NCCL all-reduce)
 * ngacf_aggregate_finalize computes Z = h + P/norm for those n_rows rows (pointers pre-offset to the first row). */
int ngacf_aggregate_finalize(float* Z, const float* h, const float* norm, int32_t H, int64_t n_rows, void* stream);

/* ---------------------------------------------------------------------------------------------
 * (a10) pair scoring: score[b] = ELU(Z[u_b]) . ELU(Z[U+i_b])   (SPUIGACF.py:49-52), fixed summation
 * tree (see DESIGN.md), and its backward G[row] += dscore * ELU(Z[other]) * ELU'(Z[row]),
 * deterministic (no atomics).  Only the batch's distinct rows of G are written: the caller zero-fills G, or treats every
 * other row as zero (ngacf_stage_bwd_prep_active).
 * ------------------------------------------------------------------------------------------- */
int ngacf_score_pairs(const float* Z, int32_t U, const int64_t* users, const int64_t* items, int32_t B, float* scores, void* stream);
int ngacf_score_pairs_bwd(const float* Z, int32_t U, const int64_t* users, const int64_t* items, const float* dscore,
                          int32_t B, float* G, int32_t accumulate, void* stream);
/* accumulate != 0: G[row] += ... for the batch's distinct rows (NegSampling scatters its B*(K+1) pairs one column of B pairs at a
 * time: the kernel's cost grows with the square of the pairs per call) */

/* ---------------------------------------------------------------------------------------------
 * Pruned output stage of a TRAINING step (exact; csrc/pruned_stage.cu; used by the fused trainer, the semantics of
 * train_eval_Gowalla.py:131-137 are kept).  The loss reads the last stage's output only at the batch rows
 * (SPUIGACF.py:49-52), so that stage's aggregation is computed for those rows only, its gradient G is defined on those
 * rows only, and d s_e vanishes on every edge without such an endpoint.  Results equal the full computation up to the
 * order of additions (everything skipped is an exact zero).
 *   mark_active : stamp[users[b]] = stamp[U+items[b]] = val (+ *val_dev); a node is active for a propagation iff its stamp
 *                 equals that propagation's value (the trainer uses the dropout call index: no clearing is ever needed).
 *                 task_count (int32[2], may be NULL) is reset to 0 for the plan call that follows.
 *   active_plan : task_list int32[T] / task_count int32[2] = the tasks (ngacf_graph_build) whose row is active: user tasks from the
 *                 front of the list (count[0]), item tasks from its back (count[1]: list[T-1], list[T-2], ...);
 *                 edge_bits uint32[(n_adj+31)/32]: bit p = neighbour adj_idx[p] is active (n_adj = 2E positions).
 *   aggregate_fwd_active     : ngacf_aggregate_fwd over the listed tasks only (Z/norm of every other row keep stale data).
 *   stage_bwd_prep_active    : Ghat/dN of the listed rows only (H = 1).
 *   stage_bwd_edges_active   : the pruned pair of edge passes (H = 1): mode 0 = user rows (stores (d s_e, e*keep) of the
 *                 visited edges; the rows of ACTIVE users are walked by one CTA per listed task), mode 1 = item rows.  G / Ghat / dN are read at active rows only; dh / dS are written for
 *                 every row of the side.
 * ------------------------------------------------------------------------------------------- */
int ngacf_mark_active(int32_t* stamp, const int64_t* users, const int64_t* items, int32_t B, int32_t U, int32_t val,
                      const int64_t* val_dev, int32_t* task_count, void* stream);
int ngacf_active_plan(const int32_t* stamp, int32_t val, const int64_t* val_dev, const int32_t* tasks, int32_t T, int32_t T_users,
                      const int32_t* adj_idx, int64_t n_adj, int32_t* task_list, int32_t* task_count, uint32_t* edge_bits,
                      void* stream);
int ngacf_aggregate_fwd_active(const int32_t* tasks, int32_t T, const int32_t* task_list, const int32_t* task_count,
                               const int32_t* adj_ptr, const int32_t* adj_idx, const int32_t* adj_eid,
                               const int32_t* long_first_slot, int32_t* long_counter, float* scratch,
                               const float* h, const float* s, int32_t H, const uint8_t* edgemask, float scale,
                               float* Z, float* norm, void* stream);
int ngacf_stage_bwd_prep_active(const int32_t* tasks, int32_t T, const int32_t* task_list, const int32_t* task_count,
                                const float* G, const float* Z, const float* h, const float* norm, int32_t H,
                                float* Ghat, float* dN, void* stream);
int ngacf_stage_bwd_edges_active(int32_t mode, const int32_t* tasks, int32_t T_begin, int32_t T_end,
                                 const int32_t* task_list, const int32_t* task_count, const int32_t* adj_ptr,
                                 const int32_t* adj_idx, const int32_t* adj_eid,
                                 const int32_t* long_first_slot, int32_t* long_counter, float* scratch,
                                 const float* G, const float* Ghat, const float* dN, const float* h, const float* s, int32_t H,
                                 const uint8_t* edgemask, float scale, const float* const* wtab, int32_t U,
                                 const int32_t* stamp, int32_t stamp_val, const int64_t* stamp_dev, const uint32_t* edge_bits,
                                 float* ds_store, float* dh, float* dS, void* stream);
/* end-of-step bookkeeping of a captured step (train_eval_Gowalla.py:139 `total_loss += loss`, :111-115 row cursor):
 * *total += *loss (either may be NULL together), row_dev[0] += row_stride (row_dev may be NULL) */
int ngacf_step_counters(double* total, const float* loss, int64_t* row_dev, int64_t row_stride, void* stream);

/* Multi-GPU pair scoring (users range-partitioned, item rows owned by range; replaces the thread-per-GPU scatter/gather of
 * parallel.py:94-130,165-196): gather writes the batch's rows this rank owns (zeros for the others) into the compact table
 * Zb[2B][64] = {user rows | item rows}; after an all-reduce of Zb, scatter writes the rows back at their global positions of a
 * table on which ngacf_score_pairs(_bwd) run unchanged.  memset_zero: cudaMemsetAsync behind the same ABI. */
int ngacf_batch_rows_gather(const float* Z, int32_t U, const int64_t* users, const int64_t* items, int32_t B, int64_t u_lo, int64_t u_hi,
                            int64_t i_lo, int64_t i_hi, float* Zb, void* stream);
int ngacf_batch_rows_scatter(const float* Zb, int32_t U, const int64_t* users, const int64_t* items, int32_t B, float* Z, void* stream);
int ngacf_memset_zero(void* p, size_t bytes, void* stream);

/* F = ELU(Z) materialised for evaluation (SPUIGACF.py:214) */
int ngacf_final_features(const float* Z, int64_t N, float* F, void* stream);

/* (a11) BPRLoss (BPRLoss.py:8-9): loss = mean softplus(-(pos-neg)); dpos = -sigmoid(-(pos-neg))*gscale/B, dneg = -dpos */
int ngacf_bpr_loss(const float* pos, const float* neg, int32_t B, float gscale, float* loss, float* dpos, float* dneg, void* stream);
/* multi-GPU: only pairs whose user lies in [u_lo,u_hi) count (loss is still divided by the global B); others get zero gradient */
int ngacf_bpr_loss_owned(const float* pos, const float* neg, int32_t B, float gscale, float* loss, float* dpos, float* dneg,
                         const int64_t* users, int64_t u_lo, int64_t u_hi, void* stream);

/* ---------------------------------------------------------------------------------------------
 * (a12) backward of one stage (closed form of SURVEY.md 3.4; the reference uses autograd).
 * prep:   Ghat = G/norm, dN = -(G . (Z-h))/norm per head.
 * edges:  mode 0 = user rows (CSR walk): computes d s_e per edge, stores it in ds_store (float[E*8]; H = 1 stores (d s_e, e*keep) pairs);
 *         mode 1 = item rows (CSC walk): reads d s_e through adj_eid -- no atomics on either side.
 *         dh[n] = G[n] + sum_m drop(e) Ghat[m] + dS[n] (x) a_side,  dS[n] = sum_m ds.
 * transform_bwd: dW/da (accumulated into gtab, same layout as wtab), dX -> Gprev = dX*mask*scale*ELU'(Zprev)
 *         (stage > 0) or accumulated into the embedding gradients (stage 0).  da is formed as W^T-contracted
 *         Xd^T dS, so the `h` argument is not read any more (kept in the signature; may be NULL).
 * ------------------------------------------------------------------------------------------- */
int ngacf_stage_bwd_prep(const float* G, const float* Z, const float* h, const float* norm, int32_t H, int64_t N,
                         float* Ghat, float* dN, void* stream);
int ngacf_stage_bwd_edges(int32_t mode, const int32_t* tasks, int32_t T_begin, int32_t T_end, const int32_t* adj_ptr,
                          const int32_t* adj_idx, const int32_t* adj_eid,
                          const int32_t* long_first_slot, int32_t* long_counter, float* scratch,
                          const float* G, const float* Ghat, const float* dN, const float* h, const float* s, int32_t H,
                          const uint8_t* edgemask, float scale, const float* const* wtab, int32_t U,
                          float* ds_store, float* dh, float* dS, int32_t partial, void* stream);
/* partial != 0 (multi-GPU, item rows): dh/dS receive raw partial sums; after the cross-rank sum
 * ngacf_stage_bwd_finalize computes dh = G + P + dS (x) a_side for n_rows rows of one side (pointers pre-offset). */
int ngacf_stage_bwd_finalize(float* dh, const float* dS, const float* G, const float* const* wtab, int32_t H, int32_t item_side,
                             int64_t n_rows, void* stream);
size_t ngacf_transform_bwd_workspace_bytes(int32_t U, int32_t I);
int ngacf_transform_bwd(const float* dh, const float* dS, const float* h, const float* Xu, const float* Xi, int32_t apply_elu,
                        const uint64_t* featmask, float scale, const float* const* wtab, float* const* gtab, int32_t H,
                        int32_t U, int32_t I, float* dXu, float* dXi, int32_t accumulate_dx, int32_t accumulate_dw,
                        void* workspace, size_t workspace_bytes, void* stream);

/* The same dense backward split in two, so that only dX sits on the backward dependency chain:
 *   ngacf_transform_bwd_dx: dX = dh W^T (+ dropout mask, ELU' of the producer) -> G of the previous stage / embedding grads;
 *   ngacf_transform_bwd_dw: dW = Xd^T dh and da (through V = Xd^T dS, so h is not re-read), accumulated into gtab; it is only
 *   needed by the optimizer and is launched on a separate stream, overlapping the next stage's gather kernels. */
int ngacf_transform_bwd_dx(const float* dh, const float* Xu, const float* Xi, int32_t apply_elu, const uint64_t* featmask, float scale,
                           const float* const* wtab, int32_t H, int32_t U, int32_t I, float* dXu, float* dXi, int32_t accumulate,
                           void* stream);
size_t ngacf_transform_bwd_dw_workspace_bytes(int32_t U, int32_t I);
int ngacf_transform_bwd_dw(const float* dh, const float* dS, const float* Xu, const float* Xi, int32_t apply_elu,
                           const uint64_t* featmask, float scale, const float* const* wtab, float* const* gtab, int32_t H, int32_t U,
                           int32_t I, int32_t accumulate, void* workspace, size_t workspace_bytes, void* stream);

/* (a13) Adam with L2 weight decay over a table of tensors (torch.optim.Adam semantics, run_Gowalla.py:114).
 * tab: device array of n entries {param, grad, exp_avg, exp_avg_sq, numel} (5 x 64-bit words each).
 * step_host is the 1-based step count (bias corrections computed on the host in double). */
int ngacf_adam_step(const uint64_t* tab, int32_t n_tensors, int64_t total_numel, float lr, float beta1, float beta2, float eps,
                    float weight_decay, int64_t step_host, void* stream);
/* same, with the step counter resident on the device so a captured CUDA graph can be replayed:
 * state = double[4] {step, lr/(1-beta1^step), 1/sqrt(1-beta2^step), unused}; the call increments step first. */
int ngacf_adam_step_dev(const uint64_t* tab, int32_t n_tensors, int64_t total_numel, float lr, float beta1, float beta2, float eps,
                        float weight_decay, double* state, void* stream);

/* ---------------------------------------------------------------------------------------------
 * (a14) PairSampling sampler.  Replaces train_pos_neg_exclude_test + train_pair_sampling
 * (data/loadGowalla.py:63-77): per train row, one positive uniform from the user's train items and one
 * negative uniform from item_pool minus train items (rank-select; negatives are never materialised).
 * Specified stream: Philox counter (row, epoch, TAG), key = seed.  neg = -1 if the user has no negative.
 * ------------------------------------------------------------------------------------------- */
int ngacf_sample_pairs(const int32_t* train_rows_user, const int32_t* train_ptr, const int32_t* train_items,
                       const int32_t* train_rank, const int32_t* pool, int32_t P, int64_t row_begin, int64_t row_end,
                       const int64_t* row_dev, uint64_t seed, uint32_t epoch, int64_t* users, int64_t* pos, int64_t* neg, void* stream);

/* ---------------------------------------------------------------------------------------------
 * (a16,a17) AllNeg evaluation.  Replaces the 64x2048 score tiles + D2H + heapq.nlargest of
 * train_eval_Gowalla.py:300-341,370-385: for every listed user the top-20 candidate items
 * (candidates = item_pool - train items; order = score desc, item id asc) straight from the
 * propagated features; the dense score matrix never exists in HBM.
 *   exact: fp32 CUDA-core scores with the fixed summation tree (bit-reproducible).
 *   tc:    tcgen05 bf16x3 user x item GEMM (fp32 accumulators in TMEM) with a top-32 candidate selection fused on
 *          the accumulators, then exact re-scoring + ordering of the candidates and an error-bound proof that no
 *          other item can enter the top-20; rows whose proof fails are flagged in `fallback` (the caller recomputes
 *          them through the exact entry point), so the returned ids are always the exact ones.
 * F = ELU(Z_last) (N,64) final features (ngacf_final_features).  in_pool: uint8[I].
 * top_ids int32 [n_users][20] (-1 padded), top_scores fp32 likewise.  fallback (tc only): int32[n_users + 1], flag per user and, in
 * the last element, the number of flagged users.
 * ------------------------------------------------------------------------------------------- */
int ngacf_score_topk_exact(const float* F, int32_t U, int32_t I, const int32_t* users, int32_t n_users,
                           const int32_t* train_ptr, const int32_t* train_items, const uint8_t* in_pool,
                           int32_t* top_ids, float* top_scores, void* stream);
/* the same result for FEW users (the rows the tc path flags): the item range is split over several CTAs per 16 users and the
 * partial lists are merged -- one CTA walking all items alone takes 6 ms at 92 K items, whatever the user count. */
size_t ngacf_score_topk_exact_split_workspace_bytes(int32_t I, int32_t n_users);
int ngacf_score_topk_exact_split(const float* F, int32_t U, int32_t I, const int32_t* users, int32_t n_users,
                                 const int32_t* train_ptr, const int32_t* train_items, const uint8_t* in_pool,
                                 int32_t* top_ids, float* top_scores, void* workspace, size_t workspace_bytes, void* stream);
size_t ngacf_score_topk_tc_workspace_bytes(int32_t I, int32_t n_users);
int ngacf_score_topk_tc(const float* F, int32_t U, int32_t I, const int32_t* users, int32_t n_users,
                        const int32_t* train_ptr, const int32_t* train_items, const uint8_t* in_pool,
                        int32_t* top_ids, float* top_scores, int32_t* fallback, int32_t reuse_mask, void* workspace,
                        size_t workspace_bytes, void* stream);
/* reuse_mask: the tc path keeps, inside the workspace, a bit matrix [item tile][user][128] of the columns a user may be ranked on
 * (item pool minus the user's train positives, train_eval_Gowalla.py:305-318,374-378).  It depends on (users, train_ptr,
 * train_items, in_pool) only.  0: build it in this call; 1: the caller asserts that this workspace already holds the matrix built
 * by an earlier call with the same four arrays (every evaluation after the first one of a run). */
/* hits + metric sums (metrics.py:10-86 via get_performance, train_eval_Gowalla.py:419-429):
 * hits uint8 [n_users][20]; sums double[16] = {precision,recall,ndcg,hit}@{1,5,10,20} summed over users
 * (the caller divides by the reference's divisor, the number of users with train data, :283). */
size_t ngacf_eval_metrics_workspace_bytes(int32_t n_users);
int ngacf_eval_metrics(const int32_t* top_ids, const int32_t* users, int32_t n_users, const int32_t* test_ptr,
                       const int32_t* test_items, uint8_t* hits, double* sums, void* workspace, size_t workspace_bytes,
                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * NegSampling training / SampledNeg evaluation (SURVEY 8f-3; the CLI's default modes, run_Gowalla.py:179-180).
 * Replaces loadGowalla.py:56-60,80-83,101-105 (negative sets + random.sample), the tensor building of
 * train_eval_Gowalla.py:58-77,226-243, BCEWithLogitsLoss (run_Gowalla.py:110) and torch.topk + hit/ndcg
 * (train_eval_Gowalla.py:251-270, graphattention/evaluation.py).  Propagation, ngacf_score_pairs(_bwd) and Adam are shared.
 *   sample_negs: rows [row_begin,row_end) of (rows_user, rows_item); all_ptr/all_rank = CSR of every user's train+test items as
 *     ranks in the sorted pool; writes users/items int64[(n)(K+1)]: column 0 the row's positive, then K distinct negatives
 *     (specified Philox stream, oracle/port.py:sample_negs); tag = 0x4E54 train / 0x4E45 eval; row_dev as in ngacf_sample_pairs;
 *     col_stride = 0: row-major (n, K+1); > 0: column-major, element (row b, column j) at j*col_stride + b.
 *   bce_logits_loss: mean over n scores of softplus(x) - y x; y = 1 at every `group`-th element (group > 0) or for the first
 *     -group elements (group < 0, column-major pairs); dscore may be NULL.
 *   rank_metrics: per row of `group` scores, rank of column 0 (strictly larger scores); sums[0] += [rank < top_k],
 *     sums[1] += 1/log2(rank+2) for hits (caller zero-fills sums; HR/NDCG = sums / n_rows).
 * ------------------------------------------------------------------------------------------- */
int ngacf_sample_negs(const int32_t* rows_user, const int32_t* rows_item, const int32_t* all_ptr, const int32_t* all_rank,
                      const int32_t* pool, int32_t P, int64_t row_begin, int64_t row_end, const int64_t* row_dev, uint64_t seed,
                      uint32_t epoch, int32_t K, uint32_t tag, int64_t col_stride, int64_t* users, int64_t* items, void* stream);
int ngacf_bce_logits_loss(const float* scores, int64_t n, int32_t group, float* loss, float* dscore, void* stream);
int ngacf_rank_metrics(const float* scores, int64_t n_rows, int32_t group, int32_t top_k, double* sums, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SPUIGAGPCF (SURVEY 8f-1): GPLayer.forward = torch.sparse.mm(laplacianMat + selfLoop, features) (SPUIGACF.py:174-185) with the
 * normalised adjacency of buildLaplacianMat (data/loadGowalla.py:197-227).  The Laplacian of the bipartite graph is symmetric and
 * has the pattern of the unified adjacency plus a diagonal: val[E] holds one value per undirected edge (CSR edge id), diag[N]
 * one per node (self loop included).  Y = diag (.) X + A_val X over the task list of ngacf_graph_build; the transpose (backward)
 * is the same call.  X != Y.
 * ------------------------------------------------------------------------------------------- */
int ngacf_spmm_sym(const int32_t* tasks, int32_t T, const int32_t* adj_ptr, const int32_t* adj_idx, const int32_t* adj_eid,
                   const int32_t* long_first_slot, int32_t* long_counter, float* scratch, const float* val, const float* diag,
                   const float* X, float* Y, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SpGraphAttentionLayer / SpGAT (SURVEY 8f-4; graphattention/SPGA.py:330-421): one W for every node, directed logit
 * e(n->m) = exp(-LeakyReLU(a[:out].h[n] + a[out:].h[m])), row-normalised, no residual: out[n] = sum_m drop(e) h[m] / sum_m e.
 * The adjacency is the unified adjacency of ngacf_graph_build (symmetric bipartite pattern) plus, if self_loops, one edge n->n per
 * node.  Directed edges are identified by adjacency position (0..n_adj-1, n_adj = 2E; self edge of n: n_adj + n): emask
 * (uint8[n_adj (+N)], bit k = head k kept; NULL = no dropout) and pairs (float2[(n_adj (+N)) * H]) use that index; rev[p] is the
 * position of the reverse edge.  h is produced by ngacf_transform_fwd with W_u = W_i = W in wtab ([W x H | W x H | a x H]).
 *   node_logits:      p[n,k] = a_k[:DH].h[n,head k], q[n,k] = a_k[DH:].h[n,head k]
 *   spgat_aggregate_fwd: Z = out (pre-ELU), norm = row sums.
 *   spgat_bwd:        from G = dL/dZ: Ghat, pairs, dP, dQ (scratch outputs) and dh = dL/dh complete (attention terms included),
 *                     which ngacf_transform_bwd turns into dW / dX.
 *   node_logits_bwd:  partials[b][0:64] = sum_n dP[n,head(c)] h[n,c], partials[b][64:128] the same with dQ, over the rows block b
 *                     owns (n_blocks blocks, fixed order); da_k = [sum_b partials[b][cols of head k] | ... dQ part].
 * ------------------------------------------------------------------------------------------- */
int ngacf_node_logits(const float* h, const float* const* wtab, int32_t H, int64_t N, float* p, float* q, void* stream);
int ngacf_node_logits_bwd(const float* h, const float* dP, const float* dQ, int32_t H, int64_t N, float* partials, int32_t n_blocks,
                          void* stream);
int ngacf_spgat_aggregate_fwd(const int32_t* tasks, int32_t T, const int32_t* adj_ptr, const int32_t* adj_idx,
                              const int32_t* long_first_slot, int32_t* long_counter, float* scratch, const float* h, const float* p,
                              const float* q, int32_t H, const uint8_t* emask, float scale, int32_t self_loops, int32_t n_adj,
                              float* Z, float* norm, void* stream);
int ngacf_spgat_bwd(const int32_t* tasks, int32_t T, const int32_t* adj_ptr, const int32_t* adj_idx, const int32_t* rev,
                    const int32_t* long_first_slot, int32_t* long_counter, float* scratch, const float* G, const float* Z,
                    const float* norm, const float* h, const float* p, const float* q, int32_t H, const uint8_t* emask, float scale,
                    int32_t self_loops, int32_t n_adj, const float* const* wtab, float* Ghat, float* pairs, float* dP, float* dQ,
                    float* dh, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Row widths other than 64 (embedSize 128).  Every entry point above is the 64-wide case and keeps its signature; the `_w`
 * variants carry the widths.  Width 64 in a `_w` call reaches exactly the kernels of the unsuffixed call (tensor-core dense
 * transforms and NGACF_DENSE included).  The SPUIGACF stage shapes at embedSize d = 128: the first stage (8 heads) reads d-wide
 * rows and writes 64, a middle stage (SPUIMultiGACF) is 64 -> 64, the last stage (1 head) writes d-wide rows; the scores read
 * d-wide rows.  Built: width 128 for single-head rows, the dense shapes (H, d_in, d_out) = (8, 128, 64) and (1, 64, 128) (CUDA-core
 * kernels), the 128-wide scores and the exact AllNeg top-K.  Anything else returns NGACF_ERR_UNSUPPORTED with a message (not
 * built at 128: partial-row multi-GPU calls, the pruned output stage, the tcgen05 dense kernels and AllNeg scorer).
 * Buffer sizes at width w: rows (N, w) fp32; feature masks w/64 uint64 words per row (word j = columns 64j .. 64j+63; row n draws
 * Philox counters n*(w/8) + c, c = 0 .. w/8-1, eight columns each); long-row scratch S*(w+8) floats.
 * ------------------------------------------------------------------------------------------- */
/* widths: HOST array of S per-stage INPUT widths (NULL = all 64) */
int ngacf_dropout_masks_w(uint64_t* const* feat, uint8_t* const* edge, const int32_t* heads, const int32_t* widths, int32_t S, int64_t N,
                          int64_t E, uint64_t seed, uint32_t call, const int64_t* call_dev, float droprate, void* stream);
int ngacf_transform_fwd_w(const float* Xu, const float* Xi, int32_t apply_elu, const uint64_t* featmask, float scale,
                          const float* const* wtab, int32_t H, int32_t d_in, int32_t d_out, int32_t U, int32_t I, float* h, float* s,
                          void* stream);
/* workspace of ngacf_transform_bwd_w for that shape (one d_in*d_out + d_out float partial per block); 0 for a shape that is not built */
size_t ngacf_transform_bwd_workspace_bytes_w(int32_t d_in, int32_t d_out, int32_t U, int32_t I);
int ngacf_transform_bwd_w(const float* dh, const float* dS, const float* h, const float* Xu, const float* Xi, int32_t apply_elu,
                          const uint64_t* featmask, float scale, const float* const* wtab, float* const* gtab, int32_t H, int32_t d_in,
                          int32_t d_out, int32_t U, int32_t I, float* dXu, float* dXi, int32_t accumulate_dx, int32_t accumulate_dw,
                          void* workspace, size_t workspace_bytes, void* stream);
int ngacf_aggregate_fwd_w(const int32_t* tasks, int32_t T, const int32_t* adj_ptr, const int32_t* adj_idx, const int32_t* adj_eid,
                          const int32_t* long_first_slot, int32_t* long_counter, float* scratch, const float* h, const float* s, int32_t H,
                          int32_t width, const uint8_t* edgemask, float scale, float* Z, float* norm, int32_t partial_from, void* stream);
int ngacf_stage_bwd_prep_w(const float* G, const float* Z, const float* h, const float* norm, int32_t H, int32_t width, int64_t N,
                           float* Ghat, float* dN, void* stream);
int ngacf_stage_bwd_edges_w(int32_t mode, const int32_t* tasks, int32_t T_begin, int32_t T_end, const int32_t* adj_ptr,
                            const int32_t* adj_idx, const int32_t* adj_eid, const int32_t* long_first_slot, int32_t* long_counter,
                            float* scratch, const float* G, const float* Ghat, const float* dN, const float* h, const float* s, int32_t H,
                            int32_t width, const uint8_t* edgemask, float scale, const float* const* wtab, int32_t U, float* ds_store,
                            float* dh, float* dS, int32_t partial, void* stream);
int ngacf_score_pairs_w(const float* Z, int32_t width, int32_t U, const int64_t* users, const int64_t* items, int32_t B, float* scores,
                        void* stream);
int ngacf_score_pairs_bwd_w(const float* Z, int32_t width, int32_t U, const int64_t* users, const int64_t* items, const float* dscore,
                            int32_t B, float* G, int32_t accumulate, void* stream);
int ngacf_final_features_w(const float* Z, int64_t N, int32_t width, float* F, void* stream);
/* scores of 128-wide rows: the same adjacent-pair tree over 128 products (7 levels); the split variant uses the workspace size of
 * ngacf_score_topk_exact_split_workspace_bytes */
int ngacf_score_topk_exact_w(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* users, int32_t n_users,
                             const int32_t* train_ptr, const int32_t* train_items, const uint8_t* in_pool, int32_t* top_ids,
                             float* top_scores, void* stream);
int ngacf_score_topk_exact_split_w(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* users, int32_t n_users,
                                   const int32_t* train_ptr, const int32_t* train_items, const uint8_t* in_pool, int32_t* top_ids,
                                   float* top_scores, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Top-K recommendation lists for any users (K = 1 .. NGACF_RECOMMEND_MAX_K).  F: (U+I, width) final features (ELU applied, as
 * ngacf_final_features(_w) writes them), width 64 or 128.  The score of (u, i) is F[u] . F[U+i] with products rounded to fp32 and
 * summed by the adjacent-pair tree of ngacf_score_topk_exact(_w), so the scores are the bits of the AllNeg ranking.
 *   candidates: items with in_pool[i] != 0 (in_pool NULL: every item) minus the user's excluded items, given as a CSR over users
 *               (excl_ptr[U+1], excl_items ascending per user; both NULL: nothing is excluded).
 *   order:      score descending, then item id ascending.  Row r of top_ids / top_scores ([n_users][K]) is users[r]'s list; a row
 *               with fewer than K candidates is padded with id -1 / score 0.0, and so is the whole row of a user id outside [0, U)
 *               (nothing of it is read).  Duplicated users get identical rows; a row does not depend on the other users of the call.
 *   workspace:  ngacf_recommend_topk_workspace_bytes(width, I, n_users, K) bytes (0 when there are enough users to rank every item
 *               range in one pass; few users split the item range and merge partial lists there).  A smaller workspace returns
 *               NGACF_ERR_WORKSPACE; nothing beyond the reported size is written.
 * Width other than 64 / 128 or K outside 1 .. NGACF_RECOMMEND_MAX_K returns NGACF_ERR_UNSUPPORTED.  Deterministic; no allocation, no
 * synchronisation (CUDA-graph capturable).  n_users == 0 is a no-op.
 * ------------------------------------------------------------------------------------------- */
#define NGACF_RECOMMEND_MAX_K 100
size_t ngacf_recommend_topk_workspace_bytes(int32_t width, int32_t I, int32_t n_users, int32_t K);
int ngacf_recommend_topk(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* users, int32_t n_users, int32_t K,
                         const int32_t* excl_ptr, const int32_t* excl_items, const uint8_t* in_pool, int32_t* top_ids,
                         float* top_scores, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Similar-item lists for any query items (K = 1 .. NGACF_RECOMMEND_MAX_K), by cosine similarity of the items' final features.  F as
 * for ngacf_recommend_topk; item j's row is F[U+j].  With dot(a, b) the adjacent-pair tree of ngacf_recommend_topk over products
 * rounded to fp32:
 *   rn(j)      = 1 / sqrt(dot(F[U+j], F[U+j])) (correctly rounded division and square root), 0 when that sum is not > 0;
 *   sim(q, j)  = (dot(F[U+q], F[U+j]) * rn(q)) * rn(j), each product rounded to fp32, in this order.  An all-zero row has
 *                similarity 0 to every item.
 *   candidates: items with in_pool[j] != 0 (in_pool NULL: every item) minus the query item itself.
 *   order:      similarity descending, then item id ascending.  Row r of top_ids / top_scores ([n_items][K]) is items[r]'s list,
 *               padded with id -1 / score 0.0 past the candidates; a query id outside [0, I) gives a padded row and reads nothing.
 *               Duplicated queries get identical rows; a row does not depend on the other queries of the call.
 *   workspace:  ngacf_similar_items_topk_workspace_bytes(width, I, n_items, K) bytes: the I inverse norms (the call computes them
 *               itself), plus the partial lists when few queries split the item range.  Never 0 for n_items > 0.  A smaller
 *               workspace returns NGACF_ERR_WORKSPACE and writes nothing; nothing beyond the reported size is written.
 * Width other than 64 / 128 or K outside 1 .. NGACF_RECOMMEND_MAX_K returns NGACF_ERR_UNSUPPORTED.  Deterministic; no allocation, no
 * synchronisation (CUDA-graph capturable).  n_items == 0 is a no-op.
 * ------------------------------------------------------------------------------------------- */
size_t ngacf_similar_items_topk_workspace_bytes(int32_t width, int32_t I, int32_t n_items, int32_t K);
int ngacf_similar_items_topk(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* items, int32_t n_items, int32_t K,
                             const uint8_t* in_pool, int32_t* top_ids, float* top_scores, void* workspace, size_t workspace_bytes,
                             void* stream);

/* ---------------------------------------------------------------------------------------------
 * Audience lists: the users to show each query item to (K = 1 .. NGACF_RECOMMEND_MAX_K).  F as for ngacf_recommend_topk.  The score
 * of (item q, user u) is dot(F[U+q], F[u]) by the tree of ngacf_recommend_topk; the products commute exactly in IEEE fp32, so it has
 * the bits of the recommend score of (u, q).
 *   candidates: users with user_pool[u] != 0 (user_pool NULL: every user) minus the item's excluded users, given as a CSR over items
 *               (excl_ptr[I+1], excl_users ascending per item; both NULL: nothing is excluded).
 *   order:      score descending, then user id ascending.  Row r of top_ids / top_scores ([n_items][K]) is items[r]'s list, padded
 *               with id -1 / score 0.0 past the candidates; a query id outside [0, I) gives a padded row and reads nothing.
 *               Duplicated queries get identical rows; a row does not depend on the other queries of the call.
 *   workspace:  ngacf_audience_topk_workspace_bytes(width, U, n_items, K) bytes (0 when there are enough queries to rank every user
 *               range in one pass; few queries split the user range and merge partial lists there).  A smaller workspace returns
 *               NGACF_ERR_WORKSPACE and writes nothing; nothing beyond the reported size is written.
 * Width other than 64 / 128 or K outside 1 .. NGACF_RECOMMEND_MAX_K returns NGACF_ERR_UNSUPPORTED.  Deterministic; no allocation, no
 * synchronisation (CUDA-graph capturable).  n_items == 0 is a no-op.
 * ------------------------------------------------------------------------------------------- */
size_t ngacf_audience_topk_workspace_bytes(int32_t width, int32_t U, int32_t n_items, int32_t K);
int ngacf_audience_topk(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* items, int32_t n_items, int32_t K,
                        const int32_t* excl_ptr, const int32_t* excl_users, const uint8_t* user_pool, int32_t* top_ids,
                        float* top_scores, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Similar-user lists for any query users (K = 1 .. NGACF_RECOMMEND_MAX_K): ngacf_similar_items_topk with the users' rows F[u] in
 * place of the items' rows.
 *   rn(u)      = 1 / sqrt(dot(F[u], F[u])), 0 when that sum is not > 0;  sim(q, u) = (dot(F[q], F[u]) * rn(q)) * rn(u).
 *   candidates: users with user_pool[u] != 0 (user_pool NULL: every user) minus the query user itself.
 *   order:      similarity descending, then user id ascending.  Rows as for ngacf_similar_items_topk; a query id outside [0, U) gives
 *               a padded row and reads nothing.
 *   workspace:  ngacf_similar_users_topk_workspace_bytes(width, U, n_users, K) bytes: the U inverse norms (256-byte aligned), plus
 *               the partial lists when few queries split the user range.  Never 0 for n_users > 0.  A smaller workspace returns
 *               NGACF_ERR_WORKSPACE and writes nothing; nothing beyond the reported size is written.
 * Width other than 64 / 128 or K outside 1 .. NGACF_RECOMMEND_MAX_K returns NGACF_ERR_UNSUPPORTED.  Deterministic; no allocation, no
 * synchronisation (CUDA-graph capturable).  n_users == 0 is a no-op.
 * ------------------------------------------------------------------------------------------- */
size_t ngacf_similar_users_topk_workspace_bytes(int32_t width, int32_t U, int32_t n_users, int32_t K);
int ngacf_similar_users_topk(const float* F, int32_t width, int32_t U, int32_t I, const int32_t* users, int32_t n_users, int32_t K,
                             const uint8_t* user_pool, int32_t* top_ids, float* top_scores, void* workspace, size_t workspace_bytes,
                             void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NGACF_B200_H */
