"""Top-K recommendation lists: ngacf_recommend_topk, ngacf_b200.recommend.Recommender and the recommend.py CLI.

The oracle ranks every candidate (in_pool minus the excluded items) by port.dot64_tree scores, score descending then id ascending,
for any width, K, exclusion and pool; at K = 20 with the train items excluded it is port.topk_allneg."""
import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------
# oracle and fixtures
# ------------------------------------------------------------------------------------------------
def score_matrix(F, U, users):
    """dot64_tree scores (n, I) of the users' rows against every item row of F (U+I, W)"""
    F = np.asarray(F, np.float32)
    items = F[U:]
    return np.stack([port.dot64_tree(np.broadcast_to(F[u], items.shape), items) for u in users])


def oracle_topk(S, users, U, K, excl=None, in_pool=None):
    """S: (n, I) scores of `users`; excl: dict user -> excluded item ids (None: nothing); in_pool: bool[I] (None: every item).
    -> ids int64 (n, K) (-1 padded), scores float32 (n, K) (0.0 padded)"""
    n, I = S.shape
    ids = np.full((n, K), -1, np.int64)
    sc = np.zeros((n, K), np.float32)
    for r, u in enumerate(users):
        if not 0 <= u < U:
            continue
        cand = np.ones(I, bool) if in_pool is None else np.asarray(in_pool, bool).copy()
        if excl is not None:
            cand[np.asarray(list(excl.get(int(u), ())), np.int64)] = False
        c = np.nonzero(cand)[0]
        s = S[r, c]
        order = np.lexsort((c, -s.astype(np.float64)))[:K]
        ids[r, :order.size] = c[order]
        sc[r, :order.size] = s[order]
    return ids, sc


def excl_sets(U, pairs):
    out = {u: set() for u in range(U)}
    for uu, ii in pairs:
        for u, i in zip(np.asarray(uu).tolist(), np.asarray(ii).tolist()):
            out[u].add(i)
    return out


def excl_csr(U, sets):
    ptr = np.zeros(U + 1, np.int64)
    items = []
    for u in range(U):
        s = sorted(sets.get(u, ()))
        ptr[u + 1] = ptr[u] + len(s)
        items += s
    return ptr, np.asarray(items, np.int64)


def bits(t):
    return np.asarray(t.cpu().numpy() if torch.is_tensor(t) else t, np.float32).view(np.int32)


def assert_lists(ids, sc, ref_ids, ref_sc):
    ids = ids.cpu().numpy() if torch.is_tensor(ids) else np.asarray(ids)
    assert np.array_equal(ids.astype(np.int64), ref_ids)
    assert np.array_equal(bits(sc), bits(ref_sc))


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_oracle_equals_port_topk_allneg():
    U, I, E = 40, 300, 2500
    u, i = port.synth_bipartite(U, I, E, 3)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 4)
    it = port.build_interactions(U, I, tu, ti, su, si)
    rng = np.random.default_rng(0)
    F = rng.standard_normal((U + I, 64)).astype(np.float32)
    F[U + 10:U + 40] = F[U + 200]                       # exact ties across ids
    users = np.arange(U)
    S = score_matrix(F, U, users)
    in_pool = np.zeros(I, bool)
    in_pool[it.pool] = True
    ids, _ = oracle_topk(S, users, U, 20, excl_sets(U, [(tu, ti)]), in_pool)
    for r, uu in enumerate(users):
        ref = port.topk_allneg(S[r], it, int(uu), 20)
        assert np.array_equal(ids[r, :ref.size], ref) and (ids[r, ref.size:] == -1).all()


def test_cli_refusals_without_cuda(monkeypatch, tmp_path):
    import recommend as RC
    import torch.distributed as dist
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: pytest.fail("process group created"))
    base = ["--resume_from", "7"]
    for bad, match in ((["--topk", "0"], "--topk"), (["--topk", "101"], "--topk"), (["--users", "5,x"], "--users"),
                       (["--parallel", "True"], "one GPU"), (["--exclude", "test"], "--exclude"), ([], "--resume_from")):
        with pytest.raises(ValueError, match=match):
            RC.parse_args((base if bad else []) + bad)
    assert not dist.is_initialized()
    f = tmp_path / "users.txt"
    f.write_text("3\n17\n\n 42\n")
    a = RC.parse_args(base + ["--users", "@%s" % f])
    assert a.user_ids.tolist() == [3, 17, 42]
    assert RC.parse_args(base + ["--users", "3, 17,42"]).user_ids.tolist() == [3, 17, 42]
    assert RC.parse_args(base).user_ids == "eval" and RC.parse_args(base + ["--users", "all"]).user_ids == "all"
    assert a.out == "recs/SPUIGACF_ml100k_007_top20.tsv"
    a = RC.parse_args(base + ["--model", "SPUIMultiGACF", "--dataset", "synth-tiny", "--topk", "100"])
    assert a.out == "recs/SPUIMultiGACF_synth-tiny_007_top100.tsv"
    assert RC.parse_args(base + ["--out", "x.tsv"]).out == "x.tsv"


def test_recommender_refuses_other_models_and_options():
    from ngacf_b200.gp import SPUIGAGPCF
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.recommend import Recommender
    with pytest.raises(NotImplementedError):
        Recommender(SPUIGAGPCF(4, 5, None, 64, [64, 64], 0.1), None, None, "none")
    with pytest.raises(ValueError, match="exclude"):
        Recommender(SPUIGACF(4, 5, 64, [64, 64], 0.1), None, None, "train")
    with pytest.raises(ValueError, match="exclude"):
        Recommender(SPUIGACF(4, 5, 64, [64, 64], 0.1), None, None, "test")


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _long_graph():
    """the shape of test_embed_width._long_graph: rows longer than one chunk, items without edges"""
    U, I, E = 400, 600, 30000
    u, i = port.synth_bipartite(U, I - 5, E, 6)
    g = port.build_graph(np.stack([u, i]), U, I)
    assert (np.diff(g.rowptr) > 128).any() and (np.diff(g.colptr) > 128).any() and (np.diff(g.colptr) == 0).any()
    return U, I, u, i


def _seeded_model(cls, U, I, width, seed=5):
    torch.manual_seed(seed)
    m = cls(U, I, width, [64, 64], 0.1).to(DEV)
    with torch.no_grad():            # larger embeddings than the N(0, 0.01) init, so that the scores spread
        m.uEmbd.weight.mul_(30)
        m.iEmbd.weight.mul_(30)
    return m


def _ranker(F, U, I, users, K, excl_ptr=None, excl_items=None, in_pool=None):
    from ngacf_b200 import ops
    dev_i32 = lambda a: None if a is None else torch.as_tensor(np.asarray(a), dtype=torch.int32).to(DEV)
    u = dev_i32(users)
    n = u.numel()
    ids = torch.empty((n, K), dtype=torch.int32, device=DEV)
    sc = torch.empty((n, K), dtype=torch.float32, device=DEV)
    ws = torch.empty(ops.recommend_topk_workspace_bytes(F.shape[-1], I, n, K), dtype=torch.uint8, device=DEV)
    pool = None if in_pool is None else torch.as_tensor(np.asarray(in_pool, np.uint8)).to(DEV)
    ops.recommend_topk(F, U, I, u, K, dev_i32(excl_ptr), dev_i32(excl_items), pool, ids, sc, ws)
    return ids, sc


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_bit_identical_to_exact_allneg_path(width):
    from ngacf_b200 import ops
    from ngacf_b200.data import Interactions
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.recommend import Recommender
    U, I, u, i = _long_graph()
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 2)
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    model = _seeded_model(SPUIGACF, U, I, width)
    rec = Recommender(model, torch.from_numpy(np.stack([u, i])), dit, "train")
    ids, sc = rec(dit.eval_users, 20)
    n = dit.eval_users.numel()
    ref_ids = torch.empty((n, 20), dtype=torch.int32, device=DEV)
    ref_sc = torch.empty((n, 20), dtype=torch.float32, device=DEV)
    ops.score_topk_exact(rec.F, U, I, dit.eval_users, dit, ref_ids, ref_sc)
    assert torch.equal(ids, ref_ids.long())
    assert np.array_equal(bits(sc), bits(ref_sc))
    assert ids.dtype == torch.int64 and sc.dtype == torch.float32 and ids.is_cuda


@pytest.fixture(scope="module")
def seeded_setup():
    """propagated features of seeded models at both widths, a split and a pool that leaves items out"""
    from ngacf_b200.data import Interactions
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.recommend import Recommender
    U, I, E = 120, 1300, 9000
    u, i = port.synth_bipartite(U, I - 10, E, 11)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 12)
    rng = np.random.default_rng(5)
    pool = np.setdiff1d(np.arange(I), rng.choice(I, 150, replace=False))
    dit = Interactions(U, I, tu, ti, su, si, DEV, pool=pool)
    in_pool = np.zeros(I, bool)
    in_pool[pool] = True
    adj = torch.from_numpy(np.stack([u, i]))
    out = dict(U=U, I=I, dit=dit, in_pool=in_pool, adj=adj,
               excl={"none": None, "train": excl_sets(U, [(tu, ti)]), "all": excl_sets(U, [(tu, ti), (su, si)])})
    users = np.concatenate([np.arange(U), [7, 7, 0, U - 1]])
    for width in (64, 128):
        model = _seeded_model(SPUIGACF, U, I, width, seed=width)
        recs = {ex: Recommender(model, adj, dit, ex) for ex in ("none", "train", "all")}
        F = recs["none"].F.cpu().numpy()
        out[width] = dict(recs=recs, S=score_matrix(F, U, users), users=users)
    return out


@gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("exclude", ["none", "train", "all"])
def test_oracle_match_across_k_and_options(seeded_setup, width, exclude):
    st = seeded_setup
    w = st[width]
    for K in (1, 5, 20, 37, 64, 100):
        ids, sc = w["recs"][exclude](w["users"], K)
        ref_ids, ref_sc = oracle_topk(w["S"], w["users"], st["U"], K, st["excl"][exclude], st["in_pool"])
        assert_lists(ids, sc, ref_ids, ref_sc)


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_ties_and_short_rows(width):
    U, I = 50, 1500
    rng = np.random.default_rng(width)
    base = rng.standard_normal((I // 6 + 1, width)).astype(np.float32)
    F = np.concatenate([rng.standard_normal((U, width)).astype(np.float32), base[np.arange(I) // 6]])   # items tie in groups of 6
    Ft = torch.from_numpy(F).to(DEV)
    users = np.arange(U)
    S = score_matrix(F, U, users)
    for K in (37, 100):
        ids, sc = _ranker(Ft, U, I, users, K)
        assert_lists(ids, sc, *oracle_topk(S, users, U, K))
    # equal features: every score ties, ids ascend (around the excluded ones)
    Fe = torch.full((U + I, width), 0.125, device=DEV)
    sets = {u: {u, u + 3} for u in range(U)}
    ptr, items = excl_csr(U, sets)
    ids, sc = _ranker(Fe, U, I, users, 100, ptr, items)
    for u in range(U):
        assert ids[u].tolist() == [x for x in range(102) if x not in sets[u]][:100]
    # fewer candidates than K: -1 / 0.0 padding; a user with every item excluded: an all -1 row
    pool = np.zeros(I, bool)
    pool[rng.choice(I, 12, replace=False)] = True
    sets = {0: set(range(I)), 1: set(np.nonzero(pool)[0][:5].tolist())}
    ptr, items = excl_csr(U, sets)
    ids, sc = _ranker(Ft, U, I, users, 20, ptr, items, pool)
    ref_ids, ref_sc = oracle_topk(S, users, U, 20, sets, pool)
    assert_lists(ids, sc, ref_ids, ref_sc)
    assert (ids[0] == -1).all() and (sc[0] == 0).all()
    assert (ids[1, 7:] == -1).all() and (ids[1, :7] >= 0).all() and (ids[2:, 12:] == -1).all() and (sc[2:, 12:] == 0).all()


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_rows_independent_of_the_batch(width):
    from ngacf_b200 import ops
    U, I = 2500, 2000
    rng = np.random.default_rng(width + 1)
    F = rng.standard_normal((U + I, width)).astype(np.float32)
    F[U + 1000:U + 1100] = F[U + 5]
    Ft = torch.from_numpy(F).to(DEV)
    sets = {u: set(rng.choice(I, 30, replace=False).tolist()) for u in range(U)}
    ptr, items = excl_csr(U, sets)
    pool = rng.random(I) < 0.9
    for K in (20, 100):
        # both sides of the switch between the item-sliced launch (few users, workspace) and the unsliced one (no workspace)
        assert ops.recommend_topk_workspace_bytes(width, I, 1, K) > 0 and ops.recommend_topk_workspace_bytes(width, I, U, K) == 0
        full_ids, full_sc = _ranker(Ft, U, I, np.arange(U), K, ptr, items, pool)
        for u in (0, 77, U - 1):
            for batch in ([u], [3, u, 1900], [u, u, u], [u] * 40):
                ids, sc = _ranker(Ft, U, I, batch, K, ptr, items, pool)
                for r, b in enumerate(batch):
                    if b == u:
                        assert torch.equal(ids[r], full_ids[u]) and torch.equal(sc[r].view(torch.int32), full_sc[u].view(torch.int32))
        sel = np.array([0, 77, U - 1])
        assert_lists(full_ids[sel], full_sc[sel], *oracle_topk(score_matrix(F, U, sel), sel, U, K, sets, pool))


@gpu
def test_c_abi_edges():
    from ngacf_b200 import _lib, ops
    lib = _lib.load()
    U, I, W = 300, 2500, 64
    rng = np.random.default_rng(9)
    F = rng.standard_normal((U + I, W)).astype(np.float32)
    Ft = torch.from_numpy(F).to(DEV)
    # user ids outside [0, U): -1 rows
    ids, sc = _ranker(Ft, U, I, [-1, U, 5, 1 << 30], 30)
    assert (ids[[0, 1, 3]] == -1).all() and (sc[[0, 1, 3]] == 0).all()
    assert_lists(ids[2:3], sc[2:3], *oracle_topk(score_matrix(F, U, [5]), [5], U, 30))
    users = torch.tensor([4, 8], dtype=torch.int32, device=DEV)
    out_i = torch.empty((2, 100), dtype=torch.int32, device=DEV)
    out_s = torch.empty((2, 100), dtype=torch.float32, device=DEV)
    need = ops.recommend_topk_workspace_bytes(W, I, 2, 100)
    assert need > 0
    buf = torch.full((need + 4096,), 0xAB, dtype=torch.uint8, device=DEV)

    def call(width, K, nbytes):
        return lib.ngacf_recommend_topk(Ft.data_ptr(), width, U, I, users.data_ptr(), 2, K, None, None, None, out_i.data_ptr(),
                                        out_s.data_ptr(), buf.data_ptr(), nbytes, ops._s())
    for width, K, what in ((W, 0, b"K = 0"), (W, 101, b"K = 101"), (96, 20, b"width 96")):
        assert call(width, K, need) == -4 and what in lib.ngacf_last_error()
    with pytest.raises(_lib.NgacfError, match="K = 101"):
        ops.recommend_topk(Ft, U, I, users, 101, None, None, None, out_i, out_s, buf)
    assert call(W, 100, need - 1) == -3 and b"workspace" in lib.ngacf_last_error()
    assert call(W, 100, need) == 0
    torch.cuda.synchronize()
    assert bool((buf[need:] == 0xAB).all()), "ngacf_recommend_topk wrote past its reported workspace"
    assert bool((buf[:need] != 0xAB).any())
    ref = oracle_topk(score_matrix(F, U, [4, 8]), [4, 8], U, 100)
    assert_lists(out_i, out_s, *ref)
    # captured in a CUDA graph and replayed
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    gi, gs = torch.full_like(out_i, 7), torch.zeros_like(out_s)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.recommend_topk(Ft, U, I, users, 100, None, None, None, gi, gs, ws)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.recommend_topk(Ft, U, I, users, 100, None, None, None, gi, gs, ws)
    gi.fill_(7)
    gs.zero_()
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    assert_lists(gi, gs, *ref)
    assert lib.ngacf_recommend_topk_workspace_bytes(96, I, 2, 20) == 0 and lib.ngacf_recommend_topk_workspace_bytes(W, I, 1, 0) == 0
    assert lib.ngacf_recommend_topk(Ft.data_ptr(), W, U, I, users.data_ptr(), 0, 20, None, None, None, None, None, None, 0,
                                    ops._s()) == -1     # null outputs are refused even for n_users == 0


@gpu
def test_prefix_property_at_synth_tiny_shape():
    from ngacf_b200.data import Interactions
    U, I, E = 2000, 3000, 60000
    u, i = port.synth_bipartite(U, I, E, 0)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 1)
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    rng = np.random.default_rng(2)
    Ft = torch.from_numpy(rng.standard_normal((U + I, 64)).astype(np.float32)).to(DEV)
    allu = np.arange(U)
    ptr, items = dit.train_ptr.cpu().numpy(), dit.train_items.cpu().numpy()
    pool = dit.in_pool.cpu().numpy()
    i100, s100 = _ranker(Ft, U, I, allu, 100, ptr, items, pool)
    i20, s20 = _ranker(Ft, U, I, allu, 20, ptr, items, pool)
    assert torch.equal(i100[:, :20], i20) and torch.equal(s100[:, :20], s20)
    assert (i100 >= 0).all()


@gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("multi", [False, True])
def test_recommender_matches_exact_evaluator(width, multi):
    from ngacf_b200.data import Interactions
    from ngacf_b200.evaluate import AllNegEvaluator
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    from ngacf_b200.recommend import Recommender, recommend
    U, I, E = 300, 900, 9000
    u, i = port.synth_bipartite(U, I, E, 21)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 22)
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    adj = torch.from_numpy(np.stack([u, i])).to(DEV)
    model = _seeded_model(SPUIMultiGACF if multi else SPUIGACF, U, I, width)
    for training in (True, False):
        model.train(training)
        rec = Recommender(model, adj, dit)
        assert model.training == training
    ids, sc = rec(dit.eval_users.cpu().numpy(), 20)
    with torch.no_grad():
        Z = model.propagate(adj)
    ev = AllNegEvaluator(dit, mode="exact")
    ev.rank(Z)
    assert torch.equal(ids, ev.top_ids.long()) and torch.equal(sc, ev.top_scores)
    ids2, _ = recommend(model, adj, dit.eval_users, 20, inter=dit)
    assert torch.equal(ids2, ids)
    # refresh() follows the parameters
    with torch.no_grad():
        model.iEmbd.weight.mul_(-1)
    rec.refresh()
    ids3, _ = rec(dit.eval_users, 20)
    assert not torch.equal(ids3, ids)
    for bad in ([0, U], [-1], np.zeros((2, 2), np.int64), [0.5]):
        with pytest.raises(ValueError):
            rec(bad, 20)
    for K in (0, 101, 2.0):
        with pytest.raises(ValueError):
            rec([0], K)
    assert rec([], 5)[0].shape == (0, 5)


@gpu
def test_cli_end_to_end(tmp_path, monkeypatch, capsys):
    import recommend as RC
    import run_Gowalla as R
    from ngacf_b200 import ops
    from ngacf_b200.evaluate import AllNegEvaluator
    from ngacf_b200.recommend import Recommender

    def train(sub, extra):
        d = tmp_path / sub
        d.mkdir()
        monkeypatch.chdir(d)
        args = R.parse_args(base + extra + ["--epochs", "1", "--eval_every", "1", "--save_every", "1"])
        RC.seed_all(args.seed)
        R.main(args)

    def read_tsv(path):
        rows = [line.rstrip("\n").split("\t") for line in open(path)]
        return [(int(a), int(b), int(c), np.float32(float(d))) for a, b, c, d in rows]

    def as_lists(rows, users, K):
        pos = {u: r for r, u in enumerate(users.tolist())}
        ids = np.full((len(users), K), -1, np.int64)
        sc = np.zeros((len(users), K), np.float32)
        for u, rank, item, s in rows:
            ids[pos[u], rank - 1] = item
            sc[pos[u], rank - 1] = s
        return ids, sc

    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--lr", "0.002",
            "--droprate", "0.2", "--batch_size", "2048", "--parallel", "False"]
    train("d64", [])
    users, ids, scores = RC.main(RC.parse_args(base + ["--resume_from", "1", "--users", "eval", "--topk", "20"]))
    out = capsys.readouterr().out
    assert "recommend: %d users, top-20" % users.size in out
    # the exact evaluator's lists for the loaded model
    args = R.parse_args(base)
    RC.seed_all(args.seed)
    inter, _, _, _, U, I, adj = R.prepareData(args)
    model, _, _ = R.createModels(args, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    model.eval()
    with torch.no_grad():
        Z = model.propagate(adj.to(DEV))
    ev = AllNegEvaluator(inter, mode="exact")
    ev.rank(Z)
    assert np.array_equal(users, inter.eval_users.cpu().numpy())
    t_ids, t_sc = as_lists(read_tsv("recs/SPUIGACF_synth-tiny_001_top20.tsv"), users, 20)
    assert np.array_equal(t_ids, ev.top_ids.cpu().numpy().astype(np.int64))
    assert np.array_equal(bits(t_sc), bits(ev.top_scores))
    # K = 100, nothing excluded, explicit users: the TSV parses back to the API's lists
    sel = np.array([5, 0, 1999, 5])
    RC.main(RC.parse_args(base + ["--resume_from", "1", "--users", "5,0,1999,5", "--topk", "100", "--exclude", "none", "--out", "r.tsv"]))
    api_ids, api_sc = Recommender(model, adj, inter, "none")(sel, 100)
    rows = read_tsv("r.tsv")
    assert len(rows) == 400 and [r[0] for r in rows[::100]] == sel.tolist()
    got = np.array([r[2] for r in rows]).reshape(4, 100)
    got_sc = np.array([r[3] for r in rows], np.float32).reshape(4, 100)
    assert np.array_equal(got, api_ids.cpu().numpy()) and np.array_equal(bits(got_sc), bits(api_sc))
    # ids outside [0, userNum) are refused before any ranking launch; a missing checkpoint names its path
    monkeypatch.setattr(ops, "recommend_topk", lambda *a, **k: pytest.fail("ranking launched"))
    with pytest.raises(ValueError, match="--users"):
        RC.main(RC.parse_args(base + ["--resume_from", "1", "--users", "3,2000"]))
    with pytest.raises(FileNotFoundError, match="ckpts/SPUIGACF_synth-tiny_004.pkl"):
        RC.main(RC.parse_args(base + ["--resume_from", "4"]))
    monkeypatch.undo()
    # embedSize 128
    train("d128", ["--embedSize", "128"])
    users, ids, scores = RC.main(RC.parse_args(base + ["--embedSize", "128", "--resume_from", "1", "--users", "all", "--topk", "50"]))
    assert ids.shape == (2000, 50) and (ids[:, 0] >= 0).all()
    assert len(read_tsv("recs/SPUIGACF_synth-tiny_001_top50.tsv")) == int((ids >= 0).sum())
