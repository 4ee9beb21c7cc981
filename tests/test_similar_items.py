"""Similar-item lists: ngacf_similar_items_topk, Recommender.similar_items and recommend.py --similar-items.

The oracle computes the specified fp32 cosine: dot = port.dot64_tree, rn(j) = 1 / sqrt(dot(F[U+j], F[U+j])) (0 when that sum is not
> 0), sim(q, j) = (dot(F[U+q], F[U+j]) * rn(q)) * rn(j), each operation rounded to fp32 as numpy float32 does it.  It ranks the pool
minus the query item, similarity descending then id ascending."""
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


def sim_matrix(F, U, queries):
    """(n, I) float32 similarities of the query items (ids in [0, I)) against every item of F (U+I, W)"""
    items = np.asarray(F, np.float32)[U:]
    rn = rnorms(items)
    rows = []
    for q in queries:
        d = port.dot64_tree(np.broadcast_to(items[q], items.shape), items)
        rows.append(((d * rn[q]).astype(np.float32) * rn).astype(np.float32))
    return np.stack(rows) if rows else np.zeros((0, items.shape[0]), np.float32)


def oracle_similar(F, U, queries, K, in_pool=None):
    """-> ids int64 (n, K) (-1 padded), scores float32 (n, K) (0.0 padded); queries outside [0, I) give padded rows"""
    I = np.asarray(F).shape[0] - U
    queries = np.asarray(queries, np.int64)
    valid = (queries >= 0) & (queries < I)
    S = sim_matrix(F, U, queries[valid])
    ids = np.full((queries.size, K), -1, np.int64)
    sc = np.zeros((queries.size, K), np.float32)
    for r, srow in zip(np.nonzero(valid)[0], S):
        cand = np.ones(I, bool) if in_pool is None else np.asarray(in_pool, bool).copy()
        cand[queries[r]] = False
        c = np.nonzero(cand)[0]
        s = srow[c]
        order = np.lexsort((c, -s.astype(np.float64)))[:K]
        ids[r, :order.size] = c[order]
        sc[r, :order.size] = s[order]
    return ids, sc


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
def test_oracle_is_the_cosine(width):
    rng = np.random.default_rng(width)
    U, I = 3, 40
    F = rng.standard_normal((U + I, width)).astype(np.float32) * rng.uniform(0.01, 30, (U + I, 1)).astype(np.float32)
    F[U + 7] = 0.0
    X = F[U:].astype(np.float64)
    n = np.linalg.norm(X, axis=1)
    rn = rnorms(F[U:])
    ok = n > 0
    assert np.allclose(rn[ok], 1.0 / n[ok], rtol=1e-6, atol=0) and rn[7] == 0
    S = sim_matrix(F, U, np.arange(I))
    with np.errstate(divide="ignore", invalid="ignore"):
        ref = (X @ X.T) / np.outer(n, n)
    ref[~ok, :] = 0
    ref[:, ~ok] = 0
    assert S.dtype == np.float32 and np.abs(S - ref).max() < 1e-6
    assert (S[7] == 0).all() and (S[:, 7] == 0).all()


def test_cli_similar_items_parsing_without_cuda(monkeypatch, tmp_path):
    import recommend as RC
    import torch.distributed as dist
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: pytest.fail("process group created"))
    base = ["--resume_from", "7"]
    a = RC.parse_args(base + ["--similar-items", "3, 17,42"])
    assert a.item_ids.tolist() == [3, 17, 42] and a.out == "recs/SPUIGACF_ml100k_007_similar20.tsv"
    f = tmp_path / "items.txt"
    f.write_text("5\n\n 9\n")
    a = RC.parse_args(base + ["--similar-items", "@%s" % f, "--topk", "100", "--dataset", "synth-tiny"])
    assert a.item_ids.tolist() == [5, 9] and a.out == "recs/SPUIGACF_synth-tiny_007_similar100.tsv"
    assert RC.parse_args(base + ["--similar-items", "all"]).item_ids == "all"
    assert RC.parse_args(base + ["--similar-items", "all", "--out", "s.tsv"]).out == "s.tsv"
    a = RC.parse_args(base)          # without the flag: the user lists, as before
    assert a.item_ids is None and a.out == "recs/SPUIGACF_ml100k_007_top20.tsv"
    for bad, match in ((["--users", "all"], "--users"), (["--users", "3"], "--users"), (["--exclude", "none"], "--exclude"),
                       (["--topk", "0"], "--topk"), (["--topk", "101"], "--topk")):
        with pytest.raises(ValueError, match=match):
            RC.parse_args(base + ["--similar-items", "1,2"] + bad)
    for spec in ("1,x", "eval", "", "1;2"):
        with pytest.raises(ValueError, match="--similar-items"):
            RC.parse_args(base + ["--similar-items", spec])
    assert not dist.is_initialized()


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _ranker(F, U, I, items, K, in_pool=None):
    from ngacf_b200 import ops
    q = torch.as_tensor(np.asarray(items), dtype=torch.int32).to(DEV)
    n = q.numel()
    ids = torch.empty((n, K), dtype=torch.int32, device=DEV)
    sc = torch.empty((n, K), dtype=torch.float32, device=DEV)
    ws = torch.empty(ops.similar_items_topk_workspace_bytes(F.shape[-1], I, n, K), dtype=torch.uint8, device=DEV)
    pool = None if in_pool is None else torch.as_tensor(np.asarray(in_pool, np.uint8)).to(DEV)
    ops.similar_items_topk(F, U, I, q, K, pool, ids, sc, ws)
    return ids, sc


def _seeded_model(cls, U, I, width, seed=5):
    torch.manual_seed(seed)
    m = cls(U, I, width, [64, 64], 0.1).to(DEV)
    with torch.no_grad():            # larger embeddings than the N(0, 0.01) init, so that the similarities spread
        m.uEmbd.weight.mul_(30)
        m.iEmbd.weight.mul_(30)
    return m


@gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("pooled", [False, True])
def test_oracle_match_across_k(width, pooled):
    from ngacf_b200.data import Interactions
    U, I, E = 60, 1250, 8000                     # 20 item tiles, the last one partial
    rng = np.random.default_rng(width + pooled)
    F = rng.standard_normal((U + I, width)).astype(np.float32) * rng.uniform(0.1, 3, (U + I, 1)).astype(np.float32)
    Ft = torch.from_numpy(F).to(DEV)
    in_pool = None
    if pooled:                                   # the pool of an Interactions that leaves items out
        u, i = port.synth_bipartite(U, I - 10, E, 11)
        (tu, ti), (su, si) = port.split_train_test(u, i, U, 12)
        pool = np.setdiff1d(np.arange(I), rng.choice(I, 150, replace=False))
        in_pool = Interactions(U, I, tu, ti, su, si, DEV, pool=pool).in_pool.cpu().numpy()
        assert in_pool.sum() == pool.size
    queries = np.concatenate([rng.choice(I, 40, replace=False), [0, I - 1, 7, 7]])
    for K in (1, 20, 37, 100):
        ids, sc = _ranker(Ft, U, I, queries, K, in_pool)
        assert_lists(ids, sc, *oracle_similar(F, U, queries, K, in_pool))
        assert not (ids.cpu().numpy() == queries[:, None]).any(), "a query item in its own list"


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_self_exclusion_for_every_item(width):
    U, I = 5, 700
    rng = np.random.default_rng(3)
    F = rng.standard_normal((U + I, width)).astype(np.float32)
    ids, sc = _ranker(torch.from_numpy(F).to(DEV), U, I, np.arange(I), 10)
    ids = ids.cpu().numpy()
    assert not (ids == np.arange(I)[:, None]).any() and (ids >= 0).all()
    sel = np.array([0, 350, I - 1])
    assert_lists(ids[sel], sc[sel], *oracle_similar(F, U, sel, 10))


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_ties_degenerate_rows_and_padding(width):
    U, I = 20, 1500
    rng = np.random.default_rng(width)
    base = rng.standard_normal((I // 6 + 1, width)).astype(np.float32)
    F = np.concatenate([rng.standard_normal((U, width)).astype(np.float32), base[np.arange(I) // 6]])   # items equal in groups of 6
    F[U + 100] = 0.0                                                                                    # an all-zero item row
    Ft = torch.from_numpy(F).to(DEV)
    queries = np.array([0, 3, 100, 101, 777, 1499])
    for K in (37, 100):
        ids, sc = _ranker(Ft, U, I, queries, K)
        ref_ids, ref_sc = oracle_similar(F, U, queries, K)
        assert_lists(ids, sc, ref_ids, ref_sc)
    # the group of 0 (items 1..5) ties at the top and comes in id order
    ids, sc = _ranker(Ft, U, I, [0], 5)
    assert ids[0].tolist() == [1, 2, 3, 4, 5] and len(set(bits(sc[0]).tolist())) == 1
    # the zero row scores 0 against everything: every candidate ties, ids ascend around the query
    ids, sc = _ranker(Ft, U, I, [100], 100)
    assert ids[0].tolist() == [x for x in range(101) if x != 100] and (sc == 0).all()
    full = torch.from_numpy(sim_matrix(F, U, [3])).to(DEV)
    assert float(full[0, 100]) == 0.0
    # a pool of 12: a query in the pool gets 11 entries, one outside it 12, then -1 / 0.0
    pool = np.zeros(I, bool)
    pool[rng.choice(I, 12, replace=False)] = True
    inside, outside = int(np.nonzero(pool)[0][0]), int(np.nonzero(~pool)[0][0])
    ids, sc = _ranker(Ft, U, I, [inside, outside], 20, pool)
    assert_lists(ids, sc, *oracle_similar(F, U, [inside, outside], 20, pool))
    assert (ids[0, :11] >= 0).all() and (ids[0, 11:] == -1).all() and (sc[0, 11:] == 0).all()
    assert (ids[1, :12] >= 0).all() and (ids[1, 12:] == -1).all()
    # query ids outside [0, I): padded rows; duplicate queries: identical rows
    ids, sc = _ranker(Ft, U, I, [-1, I, 9, 1 << 30, 9], 30)
    assert (ids[[0, 1, 3]] == -1).all() and (sc[[0, 1, 3]] == 0).all()
    assert torch.equal(ids[2], ids[4]) and torch.equal(sc[2].view(torch.int32), sc[4].view(torch.int32))
    assert_lists(ids[2:3], sc[2:3], *oracle_similar(F, U, [9], 30))


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_rows_independent_of_the_batch(width):
    from ngacf_b200 import ops
    U, I = 30, 2600
    rng = np.random.default_rng(width + 1)
    F = rng.standard_normal((U + I, width)).astype(np.float32)
    F[U + 1000:U + 1100] = F[U + 5]
    Ft = torch.from_numpy(F).to(DEV)
    pool = rng.random(I) < 0.9
    allq = np.arange(I)                          # 163 blocks of 16 queries: one pass, no partial lists
    for K in (20, 100):
        rn_only = ops.similar_items_topk_workspace_bytes(width, I, I, K)
        assert rn_only == 4 * I + 256 + (-4 * I) % 256 and ops.similar_items_topk_workspace_bytes(width, I, 1, K) > rn_only
        full_ids, full_sc = _ranker(Ft, U, I, allq, K, pool)
        for q in (0, 5, 1050, I - 1):
            for batch in ([q], [3, q, 1900], [q, q, q], [q] * 40):
                ids, sc = _ranker(Ft, U, I, batch, K, pool)
                for r, b in enumerate(batch):
                    if b == q:
                        assert torch.equal(ids[r], full_ids[q]) and torch.equal(sc[r].view(torch.int32), full_sc[q].view(torch.int32))
        sel = np.array([0, 5, 1050, I - 1])
        assert_lists(full_ids[sel], full_sc[sel], *oracle_similar(F, U, sel, K, pool))


@gpu
def test_c_abi_edges():
    from ngacf_b200 import _lib, ops
    lib = _lib.load()
    U, I, W = 40, 2500, 64
    rng = np.random.default_rng(9)
    F = rng.standard_normal((U + I, W)).astype(np.float32)
    Ft = torch.from_numpy(F).to(DEV)
    items = torch.tensor([4, 8], dtype=torch.int32, device=DEV)
    out_i = torch.full((2, 100), 7, dtype=torch.int32, device=DEV)
    out_s = torch.full((2, 100), 3.0, dtype=torch.float32, device=DEV)
    need = ops.similar_items_topk_workspace_bytes(W, I, 2, 100)
    assert need > 4 * I
    buf = torch.full((need + 4096,), 0xAB, dtype=torch.uint8, device=DEV)

    def call(width, K, nbytes, n=2):
        return lib.ngacf_similar_items_topk(Ft.data_ptr(), width, U, I, items.data_ptr(), n, K, None, out_i.data_ptr(),
                                            out_s.data_ptr(), buf.data_ptr(), nbytes, ops._s())
    for width, K, what in ((W, 0, b"K = 0"), (W, 101, b"K = 101"), (96, 20, b"width 96")):
        assert call(width, K, need) == -4 and what in lib.ngacf_last_error()
    with pytest.raises(_lib.NgacfError, match="K = 101"):
        ops.similar_items_topk(Ft, U, I, items, 101, None, out_i, out_s, buf)
    assert call(W, 100, need - 1) == -3 and b"workspace" in lib.ngacf_last_error()
    assert call(W, 100, 0, n=0) == 0          # n_items = 0: nothing to do, no workspace needed
    torch.cuda.synchronize()
    assert bool((out_i == 7).all()) and bool((out_s == 3.0).all()) and bool((buf == 0xAB).all()), "a refused call wrote"
    assert call(W, 100, need) == 0
    torch.cuda.synchronize()
    assert bool((buf[need:] == 0xAB).all()), "ngacf_similar_items_topk wrote past its reported workspace"
    ref = oracle_similar(F, U, [4, 8], 100)
    assert_lists(out_i, out_s, *ref)
    # captured in a CUDA graph and replayed twice: the eager call's bits
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    gi, gs = torch.full_like(out_i, 7), torch.zeros_like(out_s)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.similar_items_topk(Ft, U, I, items, 100, None, gi, gs, ws)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.similar_items_topk(Ft, U, I, items, 100, None, gi, gs, ws)
    for _ in range(2):
        gi.fill_(7)
        gs.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(gi, out_i) and torch.equal(gs.view(torch.int32), out_s.view(torch.int32))
    assert lib.ngacf_similar_items_topk_workspace_bytes(96, I, 2, 20) == 0 and lib.ngacf_similar_items_topk_workspace_bytes(W, I, 1, 0) == 0
    assert lib.ngacf_similar_items_topk(Ft.data_ptr(), W, U, I, items.data_ptr(), 0, 20, None, None, None, None, 0,
                                        ops._s()) == -1     # null outputs are refused even for n_items == 0


@gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("multi", [False, True])
def test_recommender_similar_items(width, multi, monkeypatch):
    from ngacf_b200 import ops
    from ngacf_b200.data import Interactions
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    from ngacf_b200.recommend import Recommender
    U, I, E = 300, 900, 9000
    u, i = port.synth_bipartite(U, I, E, 21)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 22)
    rng = np.random.default_rng(4)
    dit = Interactions(U, I, tu, ti, su, si, DEV, pool=np.setdiff1d(np.arange(I), rng.choice(I, 90, replace=False)))
    adj = torch.from_numpy(np.stack([u, i])).to(DEV)
    model = _seeded_model(SPUIMultiGACF if multi else SPUIGACF, U, I, width)
    queries = np.array([0, 17, 450, I - 1, 17])
    rec = Recommender(model, adj, exclude="none")
    F = rec.F.cpu().numpy()
    ids, sc = rec.similar_items(queries, 50)
    assert ids.dtype == torch.int64 and sc.dtype == torch.float32 and ids.is_cuda and ids.shape == (5, 50)
    assert_lists(ids, sc, *oracle_similar(F, U, queries, 50))
    # with interactions the item pool restricts the candidates; the user exclusion rule does not apply to item queries
    in_pool = dit.in_pool.cpu().numpy()
    ref = oracle_similar(F, U, queries, 50, in_pool)
    for exclude in ("train", "all", "none"):
        assert_lists(*Recommender(model, adj, dit, exclude).similar_items(torch.from_numpy(queries).to(DEV), 50), *ref)
    assert rec.similar_items([], 5)[0].shape == (0, 5)
    # refresh() follows the parameters
    with torch.no_grad():
        model.iEmbd.weight[: I // 2].mul_(-1)
    rec.refresh()
    assert not torch.equal(rec.similar_items(queries, 50)[0], ids)
    # invalid input raises before any launch
    monkeypatch.setattr(ops, "similar_items_topk", lambda *a, **k: pytest.fail("ranking launched"))
    for bad in ([0, I], [-1], np.zeros((2, 2), np.int64), [0.5], torch.tensor([1.0])):
        with pytest.raises(ValueError, match="item"):
            rec.similar_items(bad, 20)
    for K in (0, 101, 2.0, True):
        with pytest.raises(ValueError, match="K"):
            rec.similar_items([0], K)


@gpu
def test_cli_end_to_end(tmp_path, monkeypatch, capsys):
    import recommend as RC
    import run_Gowalla as R
    from ngacf_b200 import ops
    from ngacf_b200.recommend import Recommender
    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--lr", "0.002",
            "--droprate", "0.2", "--batch_size", "2048", "--parallel", "False"]
    monkeypatch.chdir(tmp_path)
    args = R.parse_args(base + ["--epochs", "1", "--eval_every", "1", "--save_every", "1"])
    RC.seed_all(args.seed)
    R.main(args)
    items, ids, scores = RC.main(RC.parse_args(base + ["--resume_from", "1", "--similar-items", "0,5,7", "--topk", "10"]))
    assert "recommend: 3 items, 10 most similar" in capsys.readouterr().out
    rows = [line.rstrip("\n").split("\t") for line in open("recs/SPUIGACF_synth-tiny_001_similar10.tsv")]
    assert len(rows) == 30 and [int(r[0]) for r in rows[::10]] == [0, 5, 7] and [int(r[1]) for r in rows[:10]] == list(range(1, 11))
    got = np.array([int(r[2]) for r in rows]).reshape(3, 10)
    got_sc = np.array([np.float32(float(r[3])) for r in rows], np.float32).reshape(3, 10)
    # the API's lists for the same checkpoint
    a = R.parse_args(base)
    RC.seed_all(a.seed)
    inter, _, _, _, U, I, adj = R.prepareData(a)
    model, _, _ = R.createModels(a, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    api_ids, api_sc = Recommender(model, adj, inter, "none").similar_items([0, 5, 7], 10)
    assert np.array_equal(got, api_ids.cpu().numpy()) and np.array_equal(bits(got_sc), bits(api_sc))
    assert np.array_equal(ids, api_ids.cpu().numpy()) and np.array_equal(items, [0, 5, 7])
    # item ids outside [0, itemNum) are refused before the checkpoint loads (--resume_from 4 does not exist)
    monkeypatch.setattr(ops, "similar_items_topk", lambda *a, **k: pytest.fail("ranking launched"))
    with pytest.raises(ValueError, match="--similar-items"):
        RC.main(RC.parse_args(base + ["--resume_from", "4", "--similar-items", "3,%d" % I]))
    with pytest.raises(FileNotFoundError, match="ckpts/SPUIGACF_synth-tiny_004.pkl"):
        RC.main(RC.parse_args(base + ["--resume_from", "4", "--similar-items", "3"]))
