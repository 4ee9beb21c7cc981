"""User-side lists: ngacf_audience_topk / ngacf_similar_users_topk, Recommender.audience / Recommender.similar_users and recommend.py
--audience / --similar-users.

The oracle computes the specified fp32 values with dot = port.dot64_tree.  Audience of item q: score(q, u) = dot(F[U+q], F[u]), the
recommend score of (u, q) with the product operands swapped (IEEE multiplication commutes, so the same bits).  Similar users of user q:
rn(u) = 1 / sqrt(dot(F[u], F[u])) (0 when that sum is not > 0), sim(q, u) = (dot(F[q], F[u]) * rn(q)) * rn(u), each operation rounded
to fp32 as numpy float32 does it.  Both rank the user pool minus the excluded users (audience: a CSR over items; similar users: the
query itself), score descending then user id ascending."""
import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------
# oracle
# ------------------------------------------------------------------------------------------------
def rnorms(X):
    """rn of every row of X (n, W) float32"""
    s = port.dot64_tree(X, X)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = (np.float32(1) / np.sqrt(s)).astype(np.float32)
    return np.where(s > 0, r, np.float32(0)).astype(np.float32)


def recommend_matrix(F, U, users):
    """(n, I) recommend scores of the users' rows against every item row of F (U+I, W)"""
    F = np.asarray(F, np.float32)
    return np.stack([port.dot64_tree(np.broadcast_to(F[u], F[U:].shape), F[U:]) for u in users])


def audience_matrix(F, U, items):
    """(n, U) audience scores of the items (ids in [0, I)) against every user row of F"""
    F = np.asarray(F, np.float32)
    return np.stack([port.dot64_tree(np.broadcast_to(F[U + q], F[:U].shape), F[:U]) for q in items])


def user_sim_matrix(F, U, users):
    """(n, U) cosine similarities of the query users (ids in [0, U)) against every user row of F"""
    X = np.asarray(F, np.float32)[:U]
    rn = rnorms(X)
    rows = [((port.dot64_tree(np.broadcast_to(X[q], X.shape), X) * rn[q]).astype(np.float32) * rn).astype(np.float32) for q in users]
    return np.stack(rows) if rows else np.zeros((0, U), np.float32)


def oracle_rank(S_of, queries, bound, n_cand, K, excl=None, pool=None, self_excl=False):
    """S_of(valid queries) -> (m, n_cand) scores; excl: dict query -> excluded candidate ids; pool: bool[n_cand] (None: all).
    -> ids int64 (n, K) (-1 padded), scores float32 (n, K) (0.0 padded); queries outside [0, bound) give padded rows"""
    queries = np.asarray(queries, np.int64)
    valid = (queries >= 0) & (queries < bound)
    S = S_of(queries[valid]) if valid.any() else np.zeros((0, n_cand), np.float32)
    ids = np.full((queries.size, K), -1, np.int64)
    sc = np.zeros((queries.size, K), np.float32)
    for r, srow in zip(np.nonzero(valid)[0], S):
        q = int(queries[r])
        cand = np.ones(n_cand, bool) if pool is None else np.asarray(pool, bool).copy()
        if excl is not None:
            cand[np.asarray(sorted(excl.get(q, ())), np.int64)] = False
        if self_excl:
            cand[q] = False
        c = np.nonzero(cand)[0]
        s = srow[c]
        order = np.lexsort((c, -s.astype(np.float64)))[:K]
        ids[r, :order.size] = c[order]
        sc[r, :order.size] = s[order]
    return ids, sc


def oracle_audience(F, U, items, K, excl=None, pool=None):
    I = np.asarray(F).shape[0] - U
    return oracle_rank(lambda q: audience_matrix(F, U, q), items, I, U, K, excl, pool)


def oracle_similar_users(F, U, users, K, pool=None):
    return oracle_rank(lambda q: user_sim_matrix(F, U, q), users, U, U, K, None, pool, self_excl=True)


def item_user_sets(I, pairs):
    """item -> set of users over the (u, i) arrays of `pairs`"""
    out = {i: set() for i in range(I)}
    for uu, ii in pairs:
        for u, i in zip(np.asarray(uu).tolist(), np.asarray(ii).tolist()):
            out[i].add(u)
    return out


def csr(n, sets):
    ptr = np.zeros(n + 1, np.int64)
    vals = []
    for r in range(n):
        s = sorted(sets.get(r, ()))
        ptr[r + 1] = ptr[r] + len(s)
        vals += s
    return ptr, np.asarray(vals, np.int64)


def bits(t):
    return np.asarray(t.cpu().numpy() if torch.is_tensor(t) else t, np.float32).view(np.int32)


def assert_lists(ids, sc, ref_ids, ref_sc):
    ids = ids.cpu().numpy() if torch.is_tensor(ids) else np.asarray(ids)
    assert np.array_equal(ids.astype(np.int64), ref_ids)
    assert np.array_equal(bits(sc), bits(ref_sc))


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("width", [64, 128])
def test_oracle_similarity_is_the_cosine(width):
    rng = np.random.default_rng(width)
    U, I = 40, 3
    F = rng.standard_normal((U + I, width)).astype(np.float32) * rng.uniform(0.01, 30, (U + I, 1)).astype(np.float32)
    F[7] = 0.0
    X = F[:U].astype(np.float64)
    n = np.linalg.norm(X, axis=1)
    rn = rnorms(F[:U])
    ok = n > 0
    assert np.allclose(rn[ok], 1.0 / n[ok], rtol=1e-6, atol=0) and rn[7] == 0
    S = user_sim_matrix(F, U, np.arange(U))
    with np.errstate(divide="ignore", invalid="ignore"):
        ref = (X @ X.T) / np.outer(n, n)
    ref[~ok, :] = 0
    ref[:, ~ok] = 0
    assert S.dtype == np.float32 and np.abs(S - ref).max() < 1e-6
    assert (S[7] == 0).all() and (S[:, 7] == 0).all()


@pytest.mark.parametrize("width", [64, 128])
def test_audience_scores_are_the_transposed_recommend_scores(width):
    rng = np.random.default_rng(width + 3)
    U, I = 37, 29
    F = rng.standard_normal((U + I, width)).astype(np.float32) * rng.uniform(0.01, 30, (U + I, 1)).astype(np.float32)
    A = audience_matrix(F, U, np.arange(I))
    R = recommend_matrix(F, U, np.arange(U))
    assert A.shape == (I, U) and np.array_equal(bits(A), bits(R.T))


def test_user_side_csr_is_the_transposed_exclusion():
    """Recommender's host-side item -> users CSR and user pool (no propagation involved)"""
    from ngacf_b200.data import Interactions
    from ngacf_b200.recommend import Recommender
    U, I, E = 50, 70, 600
    u, i = port.synth_bipartite(U, I - 4, E, 31)
    (tu, ti), (su, si) = port.split_train_test(u, i, U + 3, 32)
    inter = Interactions(U + 3, I, tu, ti, su, si, "cpu")            # users U..U+2 have no interaction
    for exclude, pairs in (("none", None), ("train", [(tu, ti)]), ("all", [(tu, ti), (su, si)])):
        rec = Recommender.__new__(Recommender)
        rec.U, rec.I, rec.inter, rec.exclude, rec.F, rec._user_side = U + 3, I, inter, exclude, torch.zeros(1), None
        ptr, users, pool = rec.user_candidates()
        assert pool.dtype == torch.uint8 and pool.tolist() == [1] * U + [0] * 3
        if pairs is None:
            assert ptr is None and users is None
            continue
        ref_ptr, ref_users = csr(I, item_user_sets(I, pairs))
        assert ptr.dtype == torch.int32 and users.dtype == torch.int32
        assert ptr.tolist() == ref_ptr.tolist() and users.tolist() == ref_users.tolist()
        assert rec.user_candidates()[0] is ptr                       # built once


def test_cli_user_lists_parsing_without_cuda(monkeypatch, tmp_path):
    import recommend as RC
    import torch.distributed as dist
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: pytest.fail("process group created"))
    base = ["--resume_from", "7"]
    a = RC.parse_args(base + ["--audience", "3, 17,42"])
    assert a.audience_ids.tolist() == [3, 17, 42] and a.out == "recs/SPUIGACF_ml100k_007_audience20.tsv"
    assert a.item_ids is None and a.similar_user_ids is None
    for ex in ("none", "all"):           # --exclude applies to the audience
        assert RC.parse_args(base + ["--audience", "all", "--exclude", ex]).exclude == ex
    f = tmp_path / "ids.txt"
    f.write_text("5\n\n 9\n")
    a = RC.parse_args(base + ["--similar-users", "@%s" % f, "--topk", "100", "--dataset", "synth-tiny"])
    assert a.similar_user_ids.tolist() == [5, 9] and a.out == "recs/SPUIGACF_synth-tiny_007_similarusers100.tsv"
    assert a.audience_ids is None and a.item_ids is None
    assert RC.parse_args(base + ["--similar-users", "all"]).similar_user_ids == "all"
    assert RC.parse_args(base + ["--audience", "all", "--out", "s.tsv"]).out == "s.tsv"
    assert RC.parse_args(base + ["--similar-items", "1"]).out == "recs/SPUIGACF_ml100k_007_similar20.tsv"
    a = RC.parse_args(base)              # without the flags: the user lists, as before
    assert a.audience_ids is None and a.similar_user_ids is None and a.out == "recs/SPUIGACF_ml100k_007_top20.tsv"
    # at most one of the query-list flags
    for pair in ((["--similar-items", "1"], ["--audience", "1"]), (["--similar-items", "1"], ["--similar-users", "1"]),
                 (["--audience", "1"], ["--similar-users", "1"])):
        with pytest.raises(ValueError, match="at most one"):
            RC.parse_args(base + pair[0] + pair[1])
    for flag, bad, match in (("--audience", ["--users", "all"], "--users"), ("--audience", ["--users", "3"], "--users"),
                             ("--similar-users", ["--users", "all"], "--users"), ("--similar-users", ["--exclude", "none"], "--exclude"),
                             ("--similar-users", ["--exclude", "all"], "--exclude"), ("--audience", ["--exclude", "test"], "--exclude"),
                             ("--audience", ["--topk", "0"], "--topk"), ("--similar-users", ["--topk", "101"], "--topk")):
        with pytest.raises(ValueError, match=match):
            RC.parse_args(base + [flag, "1,2"] + bad)
    for flag in ("--audience", "--similar-users"):
        for spec in ("1,x", "eval", "", "1;2"):
            with pytest.raises(ValueError, match=flag):
                RC.parse_args(base + [flag, spec])
    assert not dist.is_initialized()


def test_cli_refuses_out_of_range_ids_before_the_checkpoint(monkeypatch, tmp_path):
    import recommend as RC
    import run_Gowalla as R
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(R, "prepareData", lambda args: (None, None, None, None, 50, 40, None))   # 50 users, 40 items
    monkeypatch.setattr(R, "createModels", lambda *a: pytest.fail("model created"))
    base = ["--dataset", "synth-tiny", "--resume_from", "4"]
    for flag, spec in (("--audience", "3,40"), ("--audience", "-1"), ("--similar-users", "0,50")):
        with pytest.raises(ValueError, match="%s: ids must lie in" % flag):
            RC.main(RC.parse_args(base + [flag, spec]))
    for flag, spec in (("--audience", "39"), ("--similar-users", "49"), ("--audience", "all"), ("--similar-users", "all")):
        with pytest.raises(FileNotFoundError, match="ckpts/SPUIGACF_synth-tiny_004.pkl"):
            RC.main(RC.parse_args(base + [flag, spec]))


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _dev_i32(a):
    return None if a is None else torch.as_tensor(np.asarray(a), dtype=torch.int32).to(DEV)


def _dev_pool(p):
    return None if p is None else torch.as_tensor(np.asarray(p, np.uint8)).to(DEV)


def _audience(F, U, I, items, K, excl_ptr=None, excl_users=None, pool=None):
    from ngacf_b200 import ops
    q = _dev_i32(items)
    n = q.numel()
    ids = torch.empty((n, K), dtype=torch.int32, device=DEV)
    sc = torch.empty((n, K), dtype=torch.float32, device=DEV)
    ws = torch.empty(ops.audience_topk_workspace_bytes(F.shape[-1], U, n, K), dtype=torch.uint8, device=DEV)
    ops.audience_topk(F, U, I, q, K, _dev_i32(excl_ptr), _dev_i32(excl_users), _dev_pool(pool), ids, sc, ws)
    return ids, sc


def _similar_users(F, U, I, users, K, pool=None):
    from ngacf_b200 import ops
    q = _dev_i32(users)
    n = q.numel()
    ids = torch.empty((n, K), dtype=torch.int32, device=DEV)
    sc = torch.empty((n, K), dtype=torch.float32, device=DEV)
    ws = torch.empty(ops.similar_users_topk_workspace_bytes(F.shape[-1], U, n, K), dtype=torch.uint8, device=DEV)
    ops.similar_users_topk(F, U, I, q, K, _dev_pool(pool), ids, sc, ws)
    return ids, sc


def _recommend(F, U, I, users, K):
    from ngacf_b200 import ops
    q = _dev_i32(users)
    n = q.numel()
    ids = torch.empty((n, K), dtype=torch.int32, device=DEV)
    sc = torch.empty((n, K), dtype=torch.float32, device=DEV)
    ws = torch.empty(ops.recommend_topk_workspace_bytes(F.shape[-1], I, n, K), dtype=torch.uint8, device=DEV)
    ops.recommend_topk(F, U, I, q, K, None, None, None, ids, sc, ws)
    return ids, sc


def _seeded_model(cls, U, I, width, seed=5):
    torch.manual_seed(seed)
    m = cls(U, I, width, [64, 64], 0.1).to(DEV)
    with torch.no_grad():            # larger embeddings than the N(0, 0.01) init, so that the scores spread
        m.uEmbd.weight.mul_(30)
        m.iEmbd.weight.mul_(30)
    return m


@gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("exclude", ["none", "train", "all"])
@pytest.mark.parametrize("pooled", [False, True])
def test_audience_oracle_match_across_k(width, exclude, pooled):
    U, I, E = 1250, 60, 9000                     # 20 user tiles, the last one partial
    rng = np.random.default_rng(width + 7 * pooled)
    F = rng.standard_normal((U + I, width)).astype(np.float32) * rng.uniform(0.1, 3, (U + I, 1)).astype(np.float32)
    Ft = torch.from_numpy(F).to(DEV)
    u, i = port.synth_bipartite(U, I - 5, E, 11)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 12)
    excl = {"none": None, "train": item_user_sets(I, [(tu, ti)]), "all": item_user_sets(I, [(tu, ti), (su, si)])}[exclude]
    ptr, users = csr(I, excl) if excl is not None else (None, None)
    pool = None
    if pooled:
        pool = np.ones(U, bool)
        pool[rng.choice(U, 150, replace=False)] = False
    queries = np.concatenate([rng.choice(I, 40, replace=False), [0, I - 1, 7, 7]])
    for K in (1, 20, 37, 100):
        ids, sc = _audience(Ft, U, I, queries, K, ptr, users, pool)
        assert_lists(ids, sc, *oracle_audience(F, U, queries, K, excl, pool))


@gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("pooled", [False, True])
def test_similar_users_oracle_match_across_k(width, pooled):
    U, I = 1250, 60
    rng = np.random.default_rng(width + 5 * pooled)
    F = rng.standard_normal((U + I, width)).astype(np.float32) * rng.uniform(0.1, 3, (U + I, 1)).astype(np.float32)
    Ft = torch.from_numpy(F).to(DEV)
    pool = None
    if pooled:
        pool = np.ones(U, bool)
        pool[rng.choice(U, 150, replace=False)] = False
    queries = np.concatenate([rng.choice(U, 40, replace=False), [0, U - 1, 7, 7]])
    for K in (1, 20, 37, 100):
        ids, sc = _similar_users(Ft, U, I, queries, K, pool)
        assert_lists(ids, sc, *oracle_similar_users(F, U, queries, K, pool))
        assert not (ids.cpu().numpy() == queries[:, None]).any(), "a query user in its own list"


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_audience_and_recommend_lists_give_the_same_pair_scores(width):
    U, I = 90, 80                                # K = 100 >= U and >= I: every (user, item) pair is in both sets of lists
    rng = np.random.default_rng(width)
    F = rng.standard_normal((U + I, width)).astype(np.float32)
    Ft = torch.from_numpy(F).to(DEV)
    a_ids, a_sc = (t.cpu().numpy() for t in _audience(Ft, U, I, np.arange(I), 100))
    r_ids, r_sc = (t.cpu().numpy() for t in _recommend(Ft, U, I, np.arange(U), 100))
    assert (a_ids[:, :U] >= 0).all() and (a_ids[:, U:] == -1).all() and (r_ids[:, :I] >= 0).all() and (r_ids[:, I:] == -1).all()
    A = np.zeros((U, I), np.int32)               # score bits by (user, item) from the audience lists
    R = np.zeros((U, I), np.int32)
    A[a_ids[:, :U], np.arange(I)[:, None]] = bits(a_sc[:, :U])
    R[np.arange(U)[:, None], r_ids[:, :I]] = bits(r_sc[:, :I])
    assert np.array_equal(A, R)
    assert np.array_equal(A, bits(recommend_matrix(F, U, np.arange(U))))


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_similar_users_exclude_themselves(width):
    U, I = 700, 5
    rng = np.random.default_rng(3)
    F = rng.standard_normal((U + I, width)).astype(np.float32)
    ids, sc = _similar_users(torch.from_numpy(F).to(DEV), U, I, np.arange(U), 10)
    ids = ids.cpu().numpy()
    assert not (ids == np.arange(U)[:, None]).any() and (ids >= 0).all()
    sel = np.array([0, 350, U - 1])
    assert_lists(ids[sel], sc[sel], *oracle_similar_users(F, U, sel, 10))


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_ties_zero_rows_short_pools_and_odd_queries(width):
    U, I = 1500, 20
    rng = np.random.default_rng(width)
    base = rng.standard_normal((U // 6 + 1, width)).astype(np.float32)
    F = np.concatenate([base[np.arange(U) // 6], rng.standard_normal((I, width)).astype(np.float32)])   # users equal in groups of 6
    F[100] = 0.0                                                                                        # an all-zero user row
    Ft = torch.from_numpy(F).to(DEV)
    items, users = np.array([0, 3, 11, I - 1]), np.array([0, 3, 100, 101, 777, U - 1])
    for K in (37, 100):
        assert_lists(*_audience(Ft, U, I, items, K), *oracle_audience(F, U, items, K))
        assert_lists(*_similar_users(Ft, U, I, users, K), *oracle_similar_users(F, U, users, K))
    # ties come in id order: the group of user 0 for user 0, and each group of 6 in the audience
    ids, sc = _similar_users(Ft, U, I, [0], 5)
    assert ids[0].tolist() == [1, 2, 3, 4, 5] and len(set(bits(sc[0]).tolist())) == 1
    ids, sc = _audience(Ft, U, I, [3], 6)
    top = int(ids[0, 0])
    assert ids[0].tolist() == list(range(top, top + 6)) and top % 6 == 0 and len(set(bits(sc[0]).tolist())) == 1
    # the zero row: similarity 0 to every user (ids ascend around the query), audience score 0 for every item
    ids, sc = _similar_users(Ft, U, I, [100], 100)
    assert ids[0].tolist() == [x for x in range(101) if x != 100] and (sc == 0).all()
    assert (audience_matrix(F, U, np.arange(I))[:, 100] == 0).all()
    # a pool of 12 users: a query user in the pool gets 11 entries, one outside it 12; an audience row 12 minus the excluded
    pool = np.zeros(U, bool)
    pool[rng.choice(U, 12, replace=False)] = True
    inside, outside = int(np.nonzero(pool)[0][0]), int(np.nonzero(~pool)[0][0])
    ids, sc = _similar_users(Ft, U, I, [inside, outside], 20, pool)
    assert_lists(ids, sc, *oracle_similar_users(F, U, [inside, outside], 20, pool))
    assert (ids[0, :11] >= 0).all() and (ids[0, 11:] == -1).all() and (sc[0, 11:] == 0).all()
    assert (ids[1, :12] >= 0).all() and (ids[1, 12:] == -1).all()
    sets = {0: set(range(U)), 1: set(np.nonzero(pool)[0][:5].tolist())}
    ptr, ex = csr(I, sets)
    ids, sc = _audience(Ft, U, I, [0, 1, 2], 20, ptr, ex, pool)
    assert_lists(ids, sc, *oracle_audience(F, U, [0, 1, 2], 20, sets, pool))
    assert (ids[0] == -1).all() and (sc[0] == 0).all() and (ids[1, 7:] == -1).all() and (ids[1, :7] >= 0).all()
    assert (ids[2, :12] >= 0).all() and (ids[2, 12:] == -1).all()
    # query ids outside their range: padded rows; duplicate queries: identical rows
    for rank, bound, oracle in ((_audience, I, oracle_audience), (_similar_users, U, oracle_similar_users)):
        ids, sc = rank(Ft, U, I, [-1, bound, 9, 1 << 30, 9], 30)
        assert (ids[[0, 1, 3]] == -1).all() and (sc[[0, 1, 3]] == 0).all()
        assert torch.equal(ids[2], ids[4]) and torch.equal(sc[2].view(torch.int32), sc[4].view(torch.int32))
        assert_lists(ids[2:3], sc[2:3], *oracle(F, U, [9], 30))


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_rows_independent_of_the_batch(width):
    from ngacf_b200 import ops
    U, I = 3000, 2600                            # all items (163 blocks of 16) or all users (188): one pass; a few queries: P >= 2
    rng = np.random.default_rng(width + 1)
    F = rng.standard_normal((U + I, width)).astype(np.float32)
    F[1000:1100] = F[5]
    Ft = torch.from_numpy(F).to(DEV)
    sets = {i: set(rng.choice(U, 30, replace=False).tolist()) for i in range(I)}
    ptr, ex = csr(I, sets)
    pool = rng.random(U) < 0.9
    for K in (20, 100):
        assert ops.audience_topk_workspace_bytes(width, U, I, K) == 0 and ops.audience_topk_workspace_bytes(width, U, 1, K) > 0
        rn_only = ops.similar_users_topk_workspace_bytes(width, U, U, K)
        assert rn_only == 4 * U + 256 + (-4 * U) % 256 and ops.similar_users_topk_workspace_bytes(width, U, 1, K) > rn_only
        for rank, n_q, picks, oracle in (
                (lambda q, K: _audience(Ft, U, I, q, K, ptr, ex, pool), I, (0, 5, 1050, I - 1),
                 lambda q, K: oracle_audience(F, U, q, K, sets, pool)),
                (lambda q, K: _similar_users(Ft, U, I, q, K, pool), U, (0, 5, 1050, U - 1),
                 lambda q, K: oracle_similar_users(F, U, q, K, pool))):
            full_ids, full_sc = rank(np.arange(n_q), K)
            for q in picks:
                for batch in ([q], [3, q, 1900], [q, q, q], [q] * 40):
                    ids, sc = rank(batch, K)
                    for r, b in enumerate(batch):
                        if b == q:
                            assert torch.equal(ids[r], full_ids[q]) and torch.equal(sc[r].view(torch.int32), full_sc[q].view(torch.int32))
            sel = np.array(picks)
            assert_lists(full_ids[sel], full_sc[sel], *oracle(sel, K))


@gpu
def test_c_abi_edges():
    from ngacf_b200 import _lib, ops
    lib = _lib.load()
    U, I, W = 2500, 40, 64
    rng = np.random.default_rng(9)
    F = rng.standard_normal((U + I, W)).astype(np.float32)
    Ft = torch.from_numpy(F).to(DEV)
    q = torch.tensor([4, 8], dtype=torch.int32, device=DEV)
    sets = {4: {1, 2, 3}, 8: {0}}
    ptr, ex = (_dev_i32(a) for a in csr(I, sets))
    out_i = torch.full((2, 100), 7, dtype=torch.int32, device=DEV)
    out_s = torch.full((2, 100), 3.0, dtype=torch.float32, device=DEV)

    def audience(width, K, nbytes, n=2, p=ptr, e=ex, out=(out_i, out_s)):
        return lib.ngacf_audience_topk(Ft.data_ptr(), width, U, I, q.data_ptr(), n, K, p.data_ptr() if p is not None else None,
                                       e.data_ptr() if e is not None else None, None, out[0].data_ptr() if out else None,
                                       out[1].data_ptr() if out else None, buf.data_ptr(), nbytes, ops._s())

    def similar(width, K, nbytes, n=2, out=(out_i, out_s)):
        return lib.ngacf_similar_users_topk(Ft.data_ptr(), width, U, I, q.data_ptr(), n, K, None, out[0].data_ptr() if out else None,
                                            out[1].data_ptr() if out else None, buf.data_ptr(), nbytes, ops._s())
    cases = ((audience, ops.audience_topk_workspace_bytes, oracle_audience(F, U, [4, 8], 100, sets),
              lambda ws, oi, os_, K=100: ops.audience_topk(Ft, U, I, q, K, ptr, ex, None, oi, os_, ws)),
             (similar, ops.similar_users_topk_workspace_bytes, oracle_similar_users(F, U, [4, 8], 100),
              lambda ws, oi, os_, K=100: ops.similar_users_topk(Ft, U, I, q, K, None, oi, os_, ws)))
    for call, ws_bytes, ref, op in cases:
        out_i.fill_(7)
        out_s.fill_(3.0)
        need = ws_bytes(W, U, 2, 100)
        assert need > 0
        buf = torch.full((need + 4096,), 0xAB, dtype=torch.uint8, device=DEV)
        for width, K, what in ((W, 0, b"K = 0"), (W, 101, b"K = 101"), (96, 20, b"width 96")):
            assert call(width, K, need) == -4 and what in lib.ngacf_last_error()
        assert call(W, 100, need, out=None) == -1 and b"null" in lib.ngacf_last_error()
        assert call(W, 100, need - 1) == -3 and b"workspace" in lib.ngacf_last_error()
        assert call(W, 100, 0, n=0) == 0                             # n = 0: nothing to do, no workspace needed
        if call is audience:                                         # excl_ptr and excl_users are both given or both NULL
            assert audience(W, 100, need, p=None) == -1 and audience(W, 100, need, e=None) == -1
            assert b"both" in lib.ngacf_last_error()
        torch.cuda.synchronize()
        assert bool((out_i == 7).all()) and bool((out_s == 3.0).all()) and bool((buf == 0xAB).all()), "a refused call wrote"
        assert call(W, 100, need) == 0
        torch.cuda.synchronize()
        assert bool((buf[need:] == 0xAB).all()), "wrote past the reported workspace"
        assert_lists(out_i, out_s, *ref)
        with pytest.raises(_lib.NgacfError, match="K = 101"):
            op(buf, out_i, out_s, 101)
        # captured in a CUDA graph and replayed twice: the eager call's bits
        ws = torch.empty(need, dtype=torch.uint8, device=DEV)
        gi, gs = torch.full_like(out_i, 7), torch.zeros_like(out_s)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            op(ws, gi, gs)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            op(ws, gi, gs)
        for _ in range(2):
            gi.fill_(7)
            gs.zero_()
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(gi, out_i) and torch.equal(gs.view(torch.int32), out_s.view(torch.int32))
        assert ws_bytes(96, U, 2, 20) == 0 and ws_bytes(W, U, 1, 0) == 0 and ws_bytes(W, U, 0, 20) == 0
    assert lib.ngacf_audience_topk(Ft.data_ptr(), W, U, I, q.data_ptr(), 0, 20, None, None, None, None, None, None, 0,
                                   ops._s()) == -1     # null outputs are refused even for n = 0
    assert lib.ngacf_similar_users_topk(Ft.data_ptr(), W, U, I, q.data_ptr(), 0, 20, None, None, None, None, 0, ops._s()) == -1


@gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("multi", [False, True])
def test_recommender_user_lists(width, multi, monkeypatch):
    from ngacf_b200 import ops
    from ngacf_b200.data import Interactions
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    from ngacf_b200.recommend import Recommender
    U, I, E = 300, 900, 9000
    u, i = port.synth_bipartite(U, I, E, 21)
    keep = u < U - 20                                            # users U-20.. are in the graph but have no interaction: outside the pool
    (tu, ti), (su, si) = port.split_train_test(u[keep], i[keep], U, 22)
    dit = Interactions(U, I, tu, ti, su, si, DEV)
    adj = torch.from_numpy(np.stack([u, i])).to(DEV)
    model = _seeded_model(SPUIMultiGACF if multi else SPUIGACF, U, I, width)
    items, users = np.array([0, 17, 450, I - 1, 17]), np.array([0, 17, 150, U - 1, 17])
    rec = Recommender(model, adj, exclude="none")
    F = rec.F.cpu().numpy()
    # without interactions every user is a candidate
    ids, sc = rec.audience(items, 50)
    assert ids.dtype == torch.int64 and sc.dtype == torch.float32 and ids.is_cuda and ids.shape == (5, 50)
    assert_lists(ids, sc, *oracle_audience(F, U, items, 50))
    s_ids, s_sc = rec.similar_users(users, 50)
    assert s_ids.dtype == torch.int64 and s_sc.dtype == torch.float32 and s_ids.is_cuda and s_ids.shape == (5, 50)
    assert_lists(s_ids, s_sc, *oracle_similar_users(F, U, users, 50))
    # with interactions: the users with a train or test item, minus (audience) the users the exclusion rule names for the item
    pool = np.diff(dit.host["all_ptr"]) > 0
    assert not pool[U - 20:].any() and pool[:U - 20].all()
    ref_sim = oracle_similar_users(F, U, users, 50, pool)
    for exclude, pairs in (("none", None), ("train", [(tu, ti)]), ("all", [(tu, ti), (su, si)])):
        r = Recommender(model, adj, dit, exclude)
        excl = None if pairs is None else item_user_sets(I, pairs)
        assert_lists(*r.audience(torch.from_numpy(items).to(DEV), 100), *oracle_audience(F, U, items, 100, excl, pool))
        assert_lists(*r.similar_users(users, 50), *ref_sim)
    assert rec.audience([], 5)[0].shape == (0, 5) and rec.similar_users([], 5)[0].shape == (0, 5)
    # refresh() follows the parameters
    with torch.no_grad():
        model.uEmbd.weight[: U // 2].mul_(-1)
    rec.refresh()
    assert not torch.equal(rec.audience(items, 50)[0], ids) and not torch.equal(rec.similar_users(users, 50)[0], s_ids)
    # invalid input raises before any launch
    monkeypatch.setattr(ops, "audience_topk", lambda *a, **k: pytest.fail("ranking launched"))
    monkeypatch.setattr(ops, "similar_users_topk", lambda *a, **k: pytest.fail("ranking launched"))
    for method, bound, what in ((rec.audience, I, "item"), (rec.similar_users, U, "user")):
        for bad in ([0, bound], [-1], np.zeros((2, 2), np.int64), [0.5], torch.tensor([1.0])):
            with pytest.raises(ValueError, match=what):
                method(bad, 20)
        for K in (0, 101, 2.0, True):
            with pytest.raises(ValueError, match="K"):
                method([0], K)


@gpu
def test_cli_end_to_end(tmp_path, monkeypatch, capsys):
    import recommend as RC
    import run_Gowalla as R
    from ngacf_b200.recommend import Recommender
    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--lr", "0.002",
            "--droprate", "0.2", "--batch_size", "2048", "--parallel", "False"]
    monkeypatch.chdir(tmp_path)
    args = R.parse_args(base + ["--epochs", "1", "--eval_every", "1", "--save_every", "1"])
    RC.seed_all(args.seed)
    R.main(args)

    def read(path, n, K):
        rows = [line.rstrip("\n").split("\t") for line in open(path)]
        return rows, (np.array([int(r[2]) for r in rows]).reshape(n, K),
                      np.array([np.float32(float(r[3])) for r in rows], np.float32).reshape(n, K))

    a = R.parse_args(base)
    RC.seed_all(a.seed)
    inter, _, _, _, U, I, adj = R.prepareData(a)
    model, _, _ = R.createModels(a, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    # --audience: the API's lists with the train users excluded
    items, ids, scores = RC.main(RC.parse_args(base + ["--resume_from", "1", "--audience", "0,5,7", "--topk", "10"]))
    assert "recommend: 3 items, audience of 10" in capsys.readouterr().out
    rows, (got, got_sc) = read("recs/SPUIGACF_synth-tiny_001_audience10.tsv", 3, 10)
    assert [int(r[0]) for r in rows[::10]] == [0, 5, 7] and [int(r[1]) for r in rows[:10]] == list(range(1, 11))
    api_ids, api_sc = Recommender(model, adj, inter, "train").audience([0, 5, 7], 10)
    assert np.array_equal(got, api_ids.cpu().numpy()) and np.array_equal(bits(got_sc), bits(api_sc))
    assert np.array_equal(ids, api_ids.cpu().numpy()) and np.array_equal(items, [0, 5, 7])
    # --similar-users all: every user, K = 5
    users, ids, scores = RC.main(RC.parse_args(base + ["--resume_from", "1", "--similar-users", "all", "--topk", "5"]))
    assert "recommend: %d users, 5 most similar" % U in capsys.readouterr().out
    assert np.array_equal(users, np.arange(U)) and (ids >= 0).all()
    rows, (got, got_sc) = read("recs/SPUIGACF_synth-tiny_001_similarusers5.tsv", U, 5)
    api_ids, api_sc = Recommender(model, adj, inter, "none").similar_users(np.arange(U), 5)
    assert np.array_equal(got, api_ids.cpu().numpy()) and np.array_equal(bits(got_sc), bits(api_sc))
