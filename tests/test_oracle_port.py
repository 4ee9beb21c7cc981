"""CPU tests: pin oracle/port.py (the CPU restatement) against the committed golden fixtures that
oracle/make_golden.py produced by running the UNMODIFIED reference.  These are the "oracle against the
golden vectors" tests."""
import numpy as np
import pytest
import torch

from oracle import port


def sd_from(gz, prefix):
    return {k[len(prefix):]: torch.from_numpy(gz[k]) for k in gz.files if k.startswith(prefix)}


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-300))


@pytest.mark.parametrize("name", ["fwd_bwd_small", "fwd_bwd_medium"])
def test_forward_backward_fp64_matches_reference(golden, name):
    gz = golden(name)
    U, I = int(gz["U"]), int(gz["I"])
    g = port.build_graph(np.stack([gz["edge_u"], gz["edge_i"]]), U, I)
    p = port.params_from_state_dict(sd_from(gz, "sd/"), torch.float64)
    F, caches = port.propagate(p, g)
    users, items, w = gz["users"], gz["items"], torch.from_numpy(gz["w"])
    sc = port.scores(F, U, users, items)
    assert rel_err(sc.numpy(), gz["scores_f64"]) < 1e-12
    ut = torch.from_numpy(users)
    itt = torch.from_numpy(items) + U
    dF = torch.zeros_like(F)
    dF.index_add_(0, ut, w[:, None] * F[itt])
    dF.index_add_(0, itt, w[:, None] * F[ut])
    grads = port.state_dict_from_params(port.propagate_backward(dF, p, g, caches))
    for k, v in grads.items():
        assert rel_err(v.numpy(), gz["grad_f64/" + k]) < 1e-11, k


@pytest.mark.parametrize("name", ["fwd_bwd_small", "fwd_bwd_medium"])
def test_forward_backward_fp32_within_tolerance(golden, name):
    """fp32 port vs fp32 reference AND vs fp64 reference: the 1e-4 relative bar of north_star."""
    gz = golden(name)
    U, I = int(gz["U"]), int(gz["I"])
    g = port.build_graph(np.stack([gz["edge_u"], gz["edge_i"]]), U, I)
    p = port.params_from_state_dict(sd_from(gz, "sd/"), torch.float32)
    F, caches = port.propagate(p, g)
    sc = port.scores(F, U, gz["users"], gz["items"])
    assert rel_err(sc.numpy(), gz["scores_f32"]) < 1e-4
    assert rel_err(sc.numpy(), gz["scores_f64"]) < 1e-4


@pytest.mark.parametrize("name", ["fwd_bwd_small", "fwd_bwd_medium"])
def test_injected_dropout_matches_reference(golden, name):
    """Philox keep masks injected into the reference's F.dropout/nn.Dropout (SPUIGACF.py:208,213,375):
    port(masks) == reference(masks) in fp64, and the masks regenerate from (seed, call)."""
    gz = golden(name)
    U, I = int(gz["U"]), int(gz["I"])
    g = port.build_graph(np.stack([gz["edge_u"], gz["edge_i"]]), U, I)
    pdrop = float(gz["drop_p"])
    masks = port.dropout_masks(g, int(gz["drop_seed"]), int(gz["drop_call"]), pdrop)
    assert np.array_equal(masks["feat"][0], gz["drop_feat0"]) and np.array_equal(masks["feat"][1], gz["drop_feat1"])
    assert np.array_equal(masks["edge"][0], gz["drop_edge0"]) and np.array_equal(masks["edge"][1], gz["drop_edge1"])
    keep_frac = port.unpack_feature_mask(masks["feat"][0]).mean()
    assert abs(keep_frac - (1 - pdrop)) < 0.02
    p = port.params_from_state_dict(sd_from(gz, "sd/"), torch.float64)
    F, caches = port.propagate(p, g, masks, pdrop)
    users, items, w = gz["users"], gz["items"], torch.from_numpy(gz["w"])
    sc = port.scores(F, U, users, items)
    assert rel_err(sc.numpy(), gz["scores_drop_f64"]) < 1e-12
    ut = torch.from_numpy(users)
    itt = torch.from_numpy(items) + U
    dF = torch.zeros_like(F)
    dF.index_add_(0, ut, w[:, None] * F[itt])
    dF.index_add_(0, itt, w[:, None] * F[ut])
    grads = port.state_dict_from_params(port.propagate_backward(dF, p, g, caches))
    for k, v in grads.items():
        assert rel_err(v.numpy(), gz["grad_drop_f64/" + k]) < 1e-11, k


def test_train_epochs_match_reference(golden):
    """Two reference train_bpr epochs (dropout 0.2, Adam) with injected samples and masks."""
    gz = golden("train_eval_small")
    U, I = int(gz["U"]), int(gz["I"])
    it = port.build_interactions(U, I, gz["train_u"], gz["train_i"], gz["test_u"], gz["test_i"])
    eu = np.concatenate([gz["train_u"], gz["test_u"]])
    ei = np.concatenate([gz["train_i"], gz["test_i"]])
    g = port.build_graph(np.stack([eu, ei]), U, I)          # graph = train + test (run_Gowalla.py:82)
    p = port.params_from_state_dict(sd_from(gz, "sd0/"), torch.float32)
    st = port.adam_init(p)
    call = 0
    losses = []
    for ep in range(int(gz["epochs"])):
        loss, call = port.train_bpr(p, g, it, int(gz["batch"]), st, float(gz["lr"]), float(gz["wd"]), ep,
                                    int(gz["sample_seed"]), float(gz["droprate"]), int(gz["drop_seed"]), call)
        losses.append(loss)
    assert rel_err(np.array(losses), gz["epoch_losses"]) < 1e-4
    sd1 = port.state_dict_from_params(p)
    for k, v in sd1.items():
        assert rel_err(v.numpy(), gz["sd1/" + k]) < 2e-3, k     # 16 Adam steps amplify fp32 rounding via sign-like m/sqrt(v)


def test_eval_top20_and_metrics_match_reference(golden):
    gz = golden("train_eval_small")
    U, I = int(gz["U"]), int(gz["I"])
    it = port.build_interactions(U, I, gz["train_u"], gz["train_i"], gz["test_u"], gz["test_i"])
    users, divisor = port.eval_users(it)
    assert np.array_equal(users, gz["eval/users"])
    res = {k: np.zeros(4) for k in ("precision", "recall", "ndcg", "hit_ratio")}
    for j, u in enumerate(users):
        top = port.topk_allneg(gz["eval/scores"][j], it, int(u))
        assert np.array_equal(top, gz["eval/top20"][j][:top.shape[0]]), u    # ids bit-exact on identical scores
        m = port.metrics_from_hits(port.hits_for(top, it, int(u)), int(it.test_ptr[u + 1] - it.test_ptr[u]))
        for k in res:
            res[k] += m[k] / divisor
    for k in res:
        assert np.allclose(res[k], gz["eval/" + k], rtol=1e-12, atol=1e-15), k


def test_eval_from_features_close_to_reference(golden):
    """Full port pipeline (propagate -> dot64_tree -> topk) on the trained reference weights."""
    gz = golden("train_eval_small")
    U, I = int(gz["U"]), int(gz["I"])
    it = port.build_interactions(U, I, gz["train_u"], gz["train_i"], gz["test_u"], gz["test_i"])
    g = port.build_graph(np.stack([np.concatenate([gz["train_u"], gz["test_u"]]),
                                   np.concatenate([gz["train_i"], gz["test_i"]])]), U, I)
    p = port.params_from_state_dict(sd_from(gz, "sd1/"), torch.float32)
    F, _ = port.propagate(p, g)
    res, tops, users = port.eval_neg_all(F.numpy(), it)
    for k in ("precision", "recall", "ndcg", "hit_ratio"):
        assert np.allclose(res[k], gz["eval/" + k], rtol=1e-4, atol=1e-6), k
    assert (tops == gz["eval/top20"]).mean() > 0.999


def test_metrics_known_answers(golden):
    gz = golden("metrics_kat")
    for r, n, vals in zip(gz["r"], gz["npos"], gz["vals"]):
        m = port.metrics_from_hits(r, int(n))
        got = np.stack([m["precision"], m["recall"], m["ndcg"], m["hit_ratio"]])
        assert np.allclose(got, vals, rtol=1e-13, atol=0)


def test_graph_matches_torch_coalesce():
    """Bit-exact CSR/CSC vs torch's own coalesce / to_sparse_csr / to_sparse_csc, with duplicates and
    shuffled input (SURVEY.md section 4 test plan item 1)."""
    rng = np.random.default_rng(0)
    U, I = 50, 70
    u = rng.integers(0, U, 900)
    i = rng.integers(0, I, 900)
    g = port.build_graph(np.stack([u, i]), U, I)
    sp = torch.sparse_coo_tensor(torch.from_numpy(np.stack([u, i])), torch.ones(900), (U, I)).coalesce()
    assert np.array_equal(sp.indices()[0].numpy(), g.eu) and np.array_equal(sp.indices()[1].numpy(), g.ei)
    csr = sp.to_sparse_csr()
    assert np.array_equal(csr.crow_indices().numpy(), g.rowptr) and np.array_equal(csr.col_indices().numpy(), g.colidx)
    csc = sp.to_sparse_csc()
    assert np.array_equal(csc.ccol_indices().numpy(), g.colptr) and np.array_equal(csc.row_indices().numpy(), g.rowidx)
    assert np.array_equal(g.eu[g.perm], g.rowidx)
    assert np.array_equal(np.sort(g.perm), np.arange(g.E))
    perm = rng.permutation(900)
    g2 = port.build_graph(np.stack([u[perm], i[perm]]), U, I)
    assert np.array_equal(g2.colidx, g.colidx) and np.array_equal(g2.perm, g.perm)


def test_zero_degree_user_is_an_error():
    g = port.build_graph(np.array([[0, 2], [1, 1]]), 3, 2)
    with pytest.raises(ValueError):
        port.check_every_user_has_edge(g)


def test_philox_known_answer():
    """Random123 known-answer vectors for philox4x32-10."""
    out = port.philox4x32_10(0, 0, 0, 0, 0, 0)
    assert [int(x) for x in out] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    out = port.philox4x32_10(0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff)
    assert [int(x) for x in out] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    out = port.philox4x32_10(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0xa4093822, 0x299f31d0)
    assert [int(x) for x in out] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_sampler_properties():
    """Never a train positive as negative, test positives allowed, positives uniform (chi^2),
    negatives uniform over pool - train (chi^2)  (SURVEY.md section 4 item 5)."""
    U, I = 6, 40
    rng = np.random.default_rng(1)
    tu = np.repeat(np.arange(U), 5)
    ti = np.concatenate([rng.choice(I - 4, 5, replace=False) for _ in range(U)])   # items 36..39 never in rt
    su = np.arange(U)
    si = np.array([int(np.setdiff1d(np.arange(I - 4), ti[tu == u])[0]) for u in range(U)])
    it = port.build_interactions(U, I, tu, ti, su, si)
    reps = 4000
    big = port.Interactions(U, I, it.train_ptr, it.train_items, it.train_rank, it.pool, it.test_ptr, it.test_items,
                            np.tile(it.train_rows_user, reps))
    users, pos, neg = port.sample_pairs(big, 0, big.train_rows_user.shape[0], 123, 0)
    pool = set(it.pool.tolist())
    seen_test_as_neg = False
    for u in range(U):
        tr = set(it.train_items[it.train_ptr[u]:it.train_ptr[u + 1]].tolist())
        m = users == u
        assert set(pos[m].tolist()) <= tr
        assert not (set(neg[m].tolist()) & tr)
        assert set(neg[m].tolist()) <= pool
        seen_test_as_neg |= int(si[u]) in set(neg[m].tolist())
        cnt = np.array([np.sum(pos[m] == x) for x in sorted(tr)])
        chi = ((cnt - cnt.mean()) ** 2 / cnt.mean()).sum()
        assert chi < 30, chi           # 4 dof, p ~ 1e-5
        cand = sorted(pool - tr)
        cn = np.array([np.sum(neg[m] == x) for x in cand])
        chi = ((cn - cn.mean()) ** 2 / cn.mean()).sum()
        assert chi < 90, chi           # ~30 dof
    assert seen_test_as_neg
    # determinism and row addressing: a sub-range equals the slice of the full range
    u2, p2, n2 = port.sample_pairs(big, 100, 200, 123, 0)
    assert np.array_equal(p2, pos[100:200]) and np.array_equal(n2, neg[100:200])
    _, p3, _ = port.sample_pairs(big, 100, 200, 123, 1)
    assert not np.array_equal(p3, p2)


def test_dot64_tree_is_fp32_close_to_exact():
    rng = np.random.default_rng(2)
    a = rng.standard_normal((100, 64)).astype(np.float32)
    b = rng.standard_normal((100, 64)).astype(np.float32)
    ex = (a.astype(np.float64) * b.astype(np.float64)).sum(1)
    assert np.abs(port.dot64_tree(a, b) - ex).max() < 1e-5


def test_config1_ml100k_first_epoch_matches_reference(golden):
    """BASELINE config 1 on the real ml100k split: one epoch (40 steps, dropout 0.2, Adam) of the port vs the reference."""
    gz = golden("ml100k_2epochs")
    U, I = int(gz["U"]), int(gz["I"])
    it = port.build_interactions(U, I, gz["train_u"], gz["train_i"], gz["test_u"], gz["test_i"])
    g = port.build_graph(np.stack([np.concatenate([gz["train_u"], gz["test_u"]]), np.concatenate([gz["train_i"], gz["test_i"]])]), U, I)
    assert g.E == 100000 and it.train_rows_user.shape[0] == 80000
    p = port.params_from_state_dict(sd_from(gz, "sd0/"), torch.float32)
    st = port.adam_init(p)
    loss, _ = port.train_bpr(p, g, it, int(gz["batch"]), st, float(gz["lr"]), float(gz["wd"]), 0, int(gz["sample_seed"]),
                             float(gz["droprate"]), int(gz["drop_seed"]), 0)
    assert abs(loss - gz["epoch_losses"][0]) < 1e-4 * gz["epoch_losses"][0]


def test_multi_gacf_three_stage_matches_reference(golden):
    """SPUIMultiGACF (SURVEY.md 8f-1): the port's generic stage list vs the reference's 3-stage model, fp64, injected dropout."""
    gz = golden("multi_fwd_bwd_small")
    U, I = int(gz["U"]), int(gz["I"])
    g = port.build_graph(np.stack([gz["edge_u"], gz["edge_i"]]), U, I)
    p = port.params_from_state_dict(sd_from(gz, "sd/"), torch.float64)
    assert len(p["stages"]) == 3
    stages = [(8, 8), (8, 8), (1, 64)]
    masks = port.dropout_masks(g, int(gz["drop_seed"]), int(gz["drop_call"]), float(gz["drop_p"]), stages)
    F, caches = port.propagate(p, g, masks, float(gz["drop_p"]))
    users, items, w = gz["users"], gz["items"], torch.from_numpy(gz["w"])
    assert rel_err(port.scores(F, U, users, items).numpy(), gz["scores_drop_f64"]) < 1e-12
    ut, itt = torch.from_numpy(users), torch.from_numpy(items) + U
    dF = torch.zeros_like(F)
    dF.index_add_(0, ut, w[:, None] * F[itt])
    dF.index_add_(0, itt, w[:, None] * F[ut])
    grads = port.state_dict_from_params(port.propagate_backward(dF, p, g, caches))
    for k, v in grads.items():
        assert rel_err(v.numpy(), gz["grad_drop_f64/" + k]) < 1e-11, k


# ----------------------------------------------------------------------------------------------
# NegSampling / SampledNeg (SURVEY 8f-3)
# ----------------------------------------------------------------------------------------------
def _neg_case(gz):
    U, I = int(gz["U"]), int(gz["I"])
    it = port.build_interactions(U, I, gz["train_u"], gz["train_i"], gz["test_u"], gz["test_i"])
    g = port.build_graph(np.stack([np.concatenate([gz["train_u"], gz["test_u"]]),
                                   np.concatenate([gz["train_i"], gz["test_i"]])]), U, I)
    return U, I, it, g, port.AllPositives(it)


def test_neg_sampling_epochs_match_reference(golden):
    """Two reference train_neg_sample epochs (BCE-with-logits on 1 positive + 4 sampled negatives, dropout 0.2, Adam) with the
    specified negatives and dropout masks injected, then the reference's eval_neg_sample (HR/NDCG@10 over 1 + 99 candidates)."""
    gz = golden("neg_sampling_small")
    U, I, it, g, allpos = _neg_case(gz)
    p = port.params_from_state_dict(sd_from(gz, "sd0/"), torch.float32)
    st = port.adam_init(p)
    call, losses = 0, []
    for ep in range(int(gz["epochs"])):
        loss, call = port.train_neg_sample(p, g, it, allpos, gz["train_i"].astype(np.int32), int(gz["batch"]), st, float(gz["lr"]),
                                           float(gz["wd"]), ep, int(gz["sample_seed"]), float(gz["droprate"]), int(gz["drop_seed"]), call)
        losses.append(loss)
    assert rel_err(np.array(losses), gz["epoch_losses"]) < 1e-4
    sd1 = port.state_dict_from_params(p)
    for k, v in sd1.items():
        assert rel_err(v.numpy(), gz["sd1/" + k]) < 2e-3, k
    # evaluation on the reference's trained weights
    p1 = port.params_from_state_dict(sd_from(gz, "sd1/"), torch.float32)
    F, _ = port.propagate(p1, g)
    hr, nd, _ = port.eval_sampled_neg(F.numpy(), it, allpos, gz["test_u"].astype(np.int32), gz["test_i"].astype(np.int32),
                                      int(gz["eval_seed"]), int(gz["top_k"]))
    assert abs(hr - float(gz["eval/hr"])) < 1e-12 and abs(nd - float(gz["eval/ndcg"])) < 1e-9


def test_sample_negs_properties():
    """K distinct negatives, none of them a positive of the user, column 0 = the row's own item; deterministic in (seed, epoch)."""
    U, I, E = 80, 150, 1500
    u, i = port.synth_bipartite(U, I, E, 3)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 4)
    it = port.build_interactions(U, I, tu, ti, su, si)
    ap = port.AllPositives(it)
    a = port.sample_negs(it, ap, it.train_rows_user, ti.astype(np.int32), 5, 70, 9, 2, 4, port.NEG_TAG_TRAIN)
    b = port.sample_negs(it, ap, it.train_rows_user, ti.astype(np.int32), 5, 70, 9, 2, 4, port.NEG_TAG_TRAIN)
    c = port.sample_negs(it, ap, it.train_rows_user, ti.astype(np.int32), 5, 70, 9, 3, 4, port.NEG_TAG_TRAIN)
    assert np.array_equal(a[1], b[1]) and not np.array_equal(a[1], c[1])
    users, items = a
    assert np.array_equal(items[:, 0], ti[5:70]) and np.array_equal(users[:, 0], tu[5:70])
    for r in range(users.shape[0]):
        pos = set(ap.items[ap.ptr[users[r, 0]]:ap.ptr[users[r, 0] + 1]].tolist())
        negs = items[r, 1:].tolist()
        assert len(set(negs)) == 4 and not (set(negs) & pos) and set(negs) <= set(it.pool.tolist())


# ----------------------------------------------------------------------------------------------
# property tests (hypothesis): invariants of the specified generators and metrics on random shapes
# ----------------------------------------------------------------------------------------------
from hypothesis import given, settings, strategies as st  # noqa: E402


@settings(max_examples=25, deadline=None)
@given(U=st.integers(3, 40), I=st.integers(12, 60), density=st.floats(0.05, 0.5), seed=st.integers(0, 10 ** 6), K=st.integers(1, 6))
def test_sample_negs_invariants(U, I, density, seed, K):
    """For any graph / split / seed: K distinct negatives, none a positive of the user, all from the pool; the positive column and
    the user column echo the rows; rows are independent of the requested window (row r gets the same draw in any batch)."""
    E = max(U, int(U * I * density))
    u, i = port.synth_bipartite(U, I, min(E, U * I), seed % 97)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, seed % 89)
    it = port.build_interactions(U, I, tu, ti, su, si)
    ap = port.AllPositives(it)
    if it.pool.shape[0] - int(np.diff(ap.ptr).max()) < K:
        return
    n = tu.shape[0]
    users, items = port.sample_negs(it, ap, it.train_rows_user, ti.astype(np.int32), 0, n, seed, 1, K, port.NEG_TAG_TRAIN)
    assert np.array_equal(users[:, 0], tu) and np.array_equal(items[:, 0], ti)
    pool = set(it.pool.tolist())
    for r in range(n):
        pos = set(ap.items[ap.ptr[tu[r]]:ap.ptr[tu[r] + 1]].tolist())
        negs = items[r, 1:].tolist()
        assert len(set(negs)) == K and not (set(negs) & pos) and set(negs) <= pool
    lo = n // 3
    _, part = port.sample_negs(it, ap, it.train_rows_user, ti.astype(np.int32), lo, n, seed, 1, K, port.NEG_TAG_TRAIN)
    assert np.array_equal(part, items[lo:])


@settings(max_examples=50, deadline=None)
@given(rows=st.integers(1, 30), cands=st.integers(2, 40), top_k=st.integers(1, 12), seed=st.integers(0, 10 ** 6))
def test_rank_metrics_properties(rows, cands, top_k, seed):
    """HR is the fraction of rows whose positive has fewer than top_k strictly better candidates; NDCG <= HR; raising the positive's
    score never lowers either; a positive that beats everything gives 1 / 1."""
    rng = np.random.default_rng(seed)
    sc = rng.standard_normal((rows, cands)).astype(np.float32)
    hr, nd = port.rank_metrics(sc, top_k)
    rank = (sc[:, 1:] > sc[:, :1]).sum(1)
    assert abs(hr - float((rank < top_k).mean())) < 1e-12 and nd <= hr + 1e-12 and 0.0 <= nd
    better = sc.copy()
    better[:, 0] += 1.0
    hr2, nd2 = port.rank_metrics(better, top_k)
    assert hr2 >= hr - 1e-12 and nd2 >= nd - 1e-12
    best = sc.copy()
    best[:, 0] = sc.max() + 1
    assert port.rank_metrics(best, top_k) == (1.0, 1.0)


@settings(max_examples=20, deadline=None)
@given(U=st.integers(2, 30), I=st.integers(2, 40), E=st.integers(1, 300), seed=st.integers(0, 10 ** 6))
def test_build_graph_invariants(U, I, E, seed):
    """CSR and CSC describe the same coalesced edge set; perm maps CSC positions to CSR edge ids; duplicates collapse."""
    rng = np.random.default_rng(seed)
    u = np.concatenate([np.arange(U), rng.integers(0, U, E)])       # every user has an edge (the reference asserts it)
    i = np.concatenate([rng.integers(0, I, U), rng.integers(0, I, E)])
    g = port.build_graph(np.stack([u, i]), U, I)
    key = np.unique(u.astype(np.int64) * I + i)
    assert g.E == key.shape[0]
    assert np.array_equal(g.eu.astype(np.int64) * I + g.ei, key)                       # coalesced row-major, like adj.indices()
    assert np.array_equal(np.repeat(np.arange(U), np.diff(g.rowptr)), g.eu) and np.array_equal(g.colidx, g.ei)
    cols = np.repeat(np.arange(I), np.diff(g.colptr))
    assert np.array_equal(g.eu[g.perm], g.rowidx) and np.array_equal(g.ei[g.perm], cols)
    assert np.array_equal(np.sort(g.perm), np.arange(g.E))


def test_port_embeddings_match_reference_fixture(golden):
    """The oracle port's propagation against the reference's own fp64 features (embeddings_medium.npz): 1e-12."""
    gz = golden("embeddings_medium")
    U, I = int(gz["U"]), int(gz["I"])
    g = port.build_graph(np.stack([gz["edge_u"], gz["edge_i"]]), U, I)
    sd = {k[3:]: torch.from_numpy(gz[k]) for k in gz.files if k.startswith("sd/")}
    p = port.params_from_state_dict(sd, torch.float64)
    F, _ = port.propagate(p, g)
    ref = gz["features_f64"]
    assert np.abs(F.numpy() - ref).max() <= 1e-12 * np.abs(ref).max()


@pytest.mark.parametrize("name", ["spgacf_small", "spgacf_selfloops_small"])
def test_port_spgat_matches_reference_fixture(golden, name):
    """The SpGAT restatement (forward and closed-form backward) against the reference's own fp64 SPGACF run -- without dropout and
    with the fixture's injected keep masks: scores, features and every gradient to 1e-12."""
    gz = golden(name)
    U = int(gz["U"])
    g = port.build_graph(np.stack([gz["edge_u"], gz["edge_i"]]), U, int(gz["I"]))
    row, col = port.homo_edges(g, bool(gz["self_loops"]))
    assert (row == gz["row"]).all() and (col == gz["col"]).all()
    p = port.spgat_params_from_state_dict({k[3:]: torch.from_numpy(gz[k]) for k in gz.files if k.startswith("sd/")}, torch.float64)
    users, items, w = (torch.from_numpy(gz[k]) for k in ("users", "items", "w"))
    fk = [torch.from_numpy(port.unpack_feature_mask(gz["drop_feat%d" % k])) for k in (0, 1)]
    ek = [torch.from_numpy(port.unpack_edge_mask(gz["drop_edge%d_nz" % k], H)) for k, H in ((0, 8), (1, 1))]
    for tag, masks, dr in (("f64", (None, None), 0.0), ("drop_f64", (fk, ek), float(gz["drop_p"]))):
        F, caches = port.spgat_propagate(p, row, col, masks[0], masks[1], dr)
        sc = (F[users] * F[items + U]).sum(1)
        assert np.abs(sc.numpy() - gz["scores_" + tag]).max() <= 1e-12 * np.abs(gz["scores_" + tag]).max()
        dF = torch.zeros_like(F).index_add_(0, users, w[:, None] * F[items + U]).index_add_(0, items + U, w[:, None] * F[users])
        gr = port.spgat_propagate_backward(dF, p, row, col, caches)
        got = {"uEmbd.weight": gr["uEmbd"], "iEmbd.weight": gr["iEmbd"], "gat.out_att.W": gr["stages"][1]["W"][0], "gat.out_att.a": gr["stages"][1]["a"]}
        for k in range(8):
            got["gat.attention_%d.W" % k] = gr["stages"][0]["W"][k]
            got["gat.attention_%d.a" % k] = gr["stages"][0]["a"][k:k + 1]
        for k, v in got.items():
            ref = gz["grad_%s/%s" % (tag, k)]
            assert np.abs(v.numpy() - ref).max() <= 1e-11 * max(np.abs(ref).max(), 1e-30), (tag, k)
    F, _ = port.spgat_propagate(p, row, col)
    assert np.abs(F.numpy() - gz["features_f64"]).max() <= 1e-12 * np.abs(gz["features_f64"]).max()
