"""Beyond-accuracy metrics of ranked lists and metrics per user-activity group: ngacf_list_stats, ngacf_group_sums,
FullRankingEvaluator.list_metrics / group_metrics, train_eval_Gowalla.list_reports and run_Gowalla.py --eval_beyond / --eval_groups.

The oracle evaluates the definitions of ngacf_b200/cutoff_eval.py in numpy and plain Python floats: exposure counts, coverage, the
Gini index in int64 with one fp64 division, and per-user novelty / ARP summed in rank order and divided once, which reproduces the
kernel's per-user values bit for bit."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
gpu = pytest.mark.gpu
METRICS = ("precision", "recall", "ndcg", "hit_ratio", "mrr")


# ------------------------------------------------------------------------------------------------
# oracle
# ------------------------------------------------------------------------------------------------
def item_tables(train_items, I, n_tr):
    """(2, I) float64: nov(i) = -log2((d_i + 1) / (n_tr + 1)) and d_i, d_i = distinct train users of item i"""
    d = np.bincount(np.asarray(train_items, np.int64), minlength=I).astype(np.float64)
    return np.stack([-np.log2((d + 1.0) / (n_tr + 1.0)), d])


def exposure(lists, I, ks):
    """(len(ks), I) int64: counts[q][i] = rows whose first ks[q] entries contain item i (ids outside [0, I) skipped)"""
    lists = np.asarray(lists, np.int64)
    out = np.zeros((len(ks), I), np.int64)
    for q, k in enumerate(ks):
        ids = lists[:, :k].ravel()
        np.add.at(out[q], ids[(ids >= 0) & (ids < I)], 1)
    return out


def list_rows(lists, I, ks, tables):
    """(n, n_vals len(ks)) float64, table-major: the mean of each table over the valid entries among the first k, summed in rank
    order with Python floats (IEEE fp64) and divided once"""
    lists = np.asarray(lists, np.int64)
    nv, nk = len(tables), len(ks)
    out = np.zeros((lists.shape[0], nv * nk))
    for j, row in enumerate(lists.tolist()):
        for v in range(nv):
            tab = tables[v]
            s, c, q = 0.0, 0, 0
            for r in range(ks[-1]):
                i = row[r]
                if 0 <= i < I:
                    s += float(tab[i])
                    c += 1
                if r + 1 == ks[q]:
                    out[j, v * nk + q] = s / c if c else 0.0
                    q += 1
    return out


def coverage_gini(counts, pool):
    c = np.asarray(counts, np.int64)[:, pool]
    n = c.shape[1]
    cov = np.array([np.count_nonzero(x) / n for x in c])
    gini = []
    for x in c:
        x = np.sort(x)
        num = int(sum((2 * (j + 1) - n - 1) * int(v) for j, v in enumerate(x)))
        den = n * int(x.sum())
        gini.append(np.float64(num) / np.float64(den) if den else 0.0)
    return cov, np.array(gini)


def group_sums(rows, group, G):
    out = np.zeros((G, rows.shape[1]))
    for r, g in zip(rows, group):
        if 0 <= g < G:
            out[g] += r
    return out


def synthetic_lists(rng, n, K_list, I=2000):
    """distinct-id lists with -1 padding, a few ids outside [0, I) and one all-padding row"""
    lists = np.full((n, K_list), -1, np.int64)
    pop = rng.zipf(1.3, 20 * I) % I              # skewed popularity, so that exposure and the Gini index spread
    for j in range(n):
        length = K_list if j % 3 else int(rng.integers(0, K_list + 1))
        if j == 5:
            length = 0
        ids = np.unique(rng.choice(pop, 3 * K_list + 10))
        ids = rng.permutation(ids)[:length]
        lists[j, :ids.size] = ids
        if j % 7 == 1 and ids.size:
            lists[j, int(rng.integers(0, ids.size))] = I + int(rng.integers(0, 5))
        if j % 11 == 2 and ids.size:
            lists[j, int(rng.integers(0, ids.size))] = -3
    return lists


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_oracle_equals_brute_force():
    from ngacf_b200.cutoff_eval import coverage_gini as host_coverage_gini
    rng = np.random.default_rng(0)
    I = 300
    lists = synthetic_lists(rng, 120, 37, I)
    ks = [1, 5, 20, 37]
    tables = item_tables(rng.integers(0, I, 5000), I, 900)
    counts = exposure(lists, I, ks)
    rows = list_rows(lists, I, ks, tables)
    pool = np.sort(rng.choice(I, 250, replace=False))
    for q, k in enumerate(ks):
        bf = {}
        for row in lists.tolist():
            for i in row[:k]:
                if 0 <= i < I:
                    bf[i] = bf.get(i, 0) + 1
        assert all(counts[q, i] == bf.get(i, 0) for i in range(I))
        for j, row in enumerate(lists.tolist()):
            vals = [i for i in row[:k] if 0 <= i < I]
            for v in range(2):
                ref = float(np.mean([tables[v][i] for i in vals])) if vals else 0.0
                assert abs(rows[j, v * len(ks) + q] - ref) <= 1e-12 * max(abs(ref), 1.0)
    cov, gini = coverage_gini(counts, pool)
    for q in range(len(ks)):
        x = counts[q, pool].astype(np.float64)
        assert cov[q] == np.count_nonzero(x) / pool.size
        mad = np.abs(x[:, None] - x[None, :]).sum() / (2 * x.size ** 2 * x.mean())
        assert abs(gini[q] - mad) <= 1e-12
    # the evaluator's host formula gives the same bits
    hc, hg = host_coverage_gini(counts, pool)
    assert np.array_equal(hc, cov) and np.array_equal(hg, gini)
    assert np.array_equal(host_coverage_gini(np.zeros((2, I), np.int64), pool)[1], [0.0, 0.0])
    # a novelty table with the +1: items that appear only in test stay finite
    assert np.isfinite(tables).all() and (tables[0] > 0).all()


def test_item_tables_come_from_the_train_split():
    from ngacf_b200.cutoff_eval import item_degrees
    from ngacf_b200.data import Interactions
    U, I = 50, 80
    rng = np.random.default_rng(3)
    tu, ti = rng.integers(0, U, 600), rng.integers(0, I, 600)
    su, si = rng.integers(0, U, 200), rng.integers(0, I, 200)
    it = Interactions.from_arrays(U, I, tu, ti, su, si, device="cpu")
    d = item_degrees(it)
    pairs = set(zip(tu.tolist(), ti.tolist()))
    assert d.tolist() == [sum(1 for (_, i) in pairs if i == x) for x in range(I)]
    tab = item_tables(it.host["train_items"], I, it.n_train_users)
    assert np.array_equal(tab[1], d.astype(np.float64))


def test_group_split():
    from ngacf_b200.cutoff_eval import split_groups
    rng = np.random.default_rng(4)
    users = rng.permutation(5000)[:1200]
    deg = rng.zipf(1.8, users.size) % 700 + 1
    for G in range(1, 9):
        su, sd, g = split_groups(users, deg, G)
        assert sorted(su.tolist()) == sorted(users.tolist())               # every user once
        key = list(zip(sd.tolist(), su.tolist()))
        assert key == sorted(key)                                          # (degree, id) order
        assert (np.diff(g) >= 0).all() and g.min() >= 0 and g.max() <= G - 1   # contiguous groups
        T = sd.sum()
        for x in range(G):
            tot = sd[g == x].sum()
            if (g == x).any():
                assert abs(tot - T / G) <= sd.max()
        if G == 1:
            assert (g == 0).all()
    # one user holds most of the interactions: every user starts in the first quarter of the total, the other groups are empty
    su, sd, g = split_groups(np.arange(10), [1] * 9 + [1000], 4)
    assert np.bincount(g, minlength=4).tolist() == [10, 0, 0, 0]
    su, sd, g = split_groups(np.arange(10), [1000] + [1] * 9, 4)
    assert su[-1] == 0 and np.bincount(g, minlength=4).tolist() == [10, 0, 0, 0]
    su, sd, g = split_groups(np.arange(11), [5] * 10 + [100], 4)
    counts = np.bincount(g, minlength=4)
    assert (counts == 0).any() and counts.sum() == 11
    for bad in (0, 9, 2.0, True, "3"):
        with pytest.raises(ValueError):
            split_groups(np.arange(3), [1, 2, 3], bad)


def test_cli_parsing(monkeypatch):
    import run_Gowalla as R
    import torch.distributed as dist
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: pytest.fail("process group created"))
    a = R.parse_args([])
    assert a.eval_beyond is False and a.eval_groups is None
    a = R.parse_args(["--eval_ks", "20", "--eval_beyond", "True", "--eval_groups", "4"])
    assert a.eval_beyond is True and a.eval_groups == 4
    assert R.parse_args(["--eval_ks", "20", "--eval_groups", "1"]).eval_groups == 1
    assert R.parse_args(["--eval_ks", "20", "--eval_groups", "8", "--eval_beyond", "False"]).eval_groups == 8
    for bad in (["--eval_beyond", "True"], ["--eval_groups", "4"], ["--eval_ks", "20", "--eval_groups", "0"],
                ["--eval_ks", "20", "--eval_groups", "9"], ["--eval_ks", "20", "--eval_groups", "x"],
                ["--eval_ks", "20", "--eval_groups", "2.5"], ["--eval_ks", "20", "--eval_beyond", "yes"],
                ["--eval_ks", "20", "--eval_beyond", "1"]):
        with pytest.raises(ValueError):
            R.parse_args(["--parallel", "True"] + bad)
    assert not dist.is_initialized()


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _t(a, dt=torch.int32):
    return torch.as_tensor(np.asarray(a)).to(dt).to(DEV).contiguous()


def _list_stats(ids, I, ks, tables, counts=True, rows=True):
    from ngacf_b200 import ops
    n = ids.shape[0]
    nv = 0 if tables is None else tables.shape[0]
    c = torch.full((len(ks), I), 12345, dtype=torch.int32, device=DEV) if counts else None
    r = torch.full((n, nv * len(ks)), -7.0, dtype=torch.float64, device=DEV) if rows else None
    ops.list_stats(ids, I, ks, tables, c, r)
    return c, r


@gpu
@pytest.mark.parametrize("K_list", [1, 20, 37, 100])
def test_list_stats_matches_oracle(K_list):
    rng = np.random.default_rng(K_list)
    I = 2000
    lists = synthetic_lists(rng, 700, K_list, I)
    tab = item_tables(rng.integers(0, I, 30000), I, 1500)
    ids, tables = _t(lists), _t(tab, torch.float64)
    for n_ks in range(1, 9):
        ks = sorted(rng.choice(np.arange(1, K_list + 1), min(n_ks, K_list), replace=False).tolist())
        if n_ks == 1:
            ks = [K_list]
        ref_c = exposure(lists, I, ks)
        for nv in (0, 1, 2):
            c, r = _list_stats(ids, I, ks, tables[:nv] if nv else None)
            assert np.array_equal(c.cpu().numpy(), ref_c)
            assert np.array_equal(r.cpu().numpy(), list_rows(lists, I, ks, tab[:nv])), (ks, nv)   # bit for bit
        if K_list == 1:
            break


def _group_case(rng, n, n_cols, G):
    rows = rng.standard_normal((n, n_cols)) * rng.choice([1e-3, 1.0, 1e3], (n, 1))
    group = rng.integers(0, G, n)
    if G > 2:
        group[group == 1] = 0                 # group 1 empty
    group[rng.random(n) < 0.05] = -1          # outside [0, G): skipped
    group[rng.random(n) < 0.05] = G
    group[rng.random(n) < 0.01] = 1 << 20
    return rows, group


def _gsums(rows, group, G):
    from ngacf_b200 import ops
    s = torch.full((G, rows.shape[1]), -7.0, dtype=torch.float64, device=DEV)
    ws = torch.empty(ops.group_sums_workspace_bytes(rows.shape[0], rows.shape[1], G), dtype=torch.uint8, device=DEV)
    ops.group_sums(rows, group, G, s, ws)
    return s


@gpu
def test_group_sums_match_a_sequential_oracle():
    rng = np.random.default_rng(11)
    for G in range(1, 9):
        for n, n_cols in ((1, 1), (255, 7), (257, 40), (30000, 56), (4097, 14)):
            rows, group = _group_case(rng, n, n_cols, G)
            got = _gsums(_t(rows, torch.float64), _t(group), G).cpu().numpy()
            ref = group_sums(rows, group, G)
            np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-12 * np.abs(rows).sum(0).max())
            if G > 2 and n > 300:
                assert (got[1] == 0).all()


@gpu
def test_c_abi_edges():
    from ngacf_b200 import _lib, ops
    lib = _lib.load()
    rng = np.random.default_rng(7)
    I = 1500
    lists = synthetic_lists(rng, 333, 100, I)
    tab = item_tables(rng.integers(0, I, 20000), I, 900)
    ids, tables = _t(lists), _t(tab, torch.float64)
    n = ids.shape[0]
    ks = [1, 10, 20, 50, 100]
    counts = torch.full((len(ks), I), 0x5A5A, dtype=torch.int32, device=DEV)
    rows = torch.full((n, 2 * len(ks)), -7.0, dtype=torch.float64, device=DEV)

    def ls(K_list=100, k=ks, nv=2, c=counts.data_ptr(), r=rows.data_ptr()):
        ka = (ctypes.c_int32 * max(len(k), 1))(*k)
        return lib.ngacf_list_stats(ids.data_ptr(), K_list, n, I, ka, len(k), tables.data_ptr(), nv, c, r, ops._s())
    for kw, what in (({"K_list": 0}, b"list length 0"), ({"K_list": 101}, b"list length 101"), ({"k": []}, b"0 cut-offs"),
                     ({"k": list(range(1, 10))}, b"9 cut-offs"), ({"k": [5, 5]}, b"strictly increasing"),
                     ({"k": [10, 5]}, b"strictly increasing"), ({"k": [0, 5]}, b"strictly increasing"),
                     ({"K_list": 50, "k": [20, 100]}, b"1..50"), ({"nv": 3}, b"3 item tables"), ({"nv": -1}, b"-1 item tables")):
        assert ls(**kw) == -4 and what in lib.ngacf_last_error(), kw
    with pytest.raises(_lib.NgacfError, match="strictly increasing"):
        ops.list_stats(ids, I, [20, 10], tables, counts, rows)
    # group sums refusals and a short workspace
    grp = _t(rng.integers(-1, 5, n))
    need = ops.group_sums_workspace_bytes(n, 10, 4)
    assert need > 0 and ops.group_sums_workspace_bytes(n, 57, 4) == 0 and ops.group_sums_workspace_bytes(n, 10, 9) == 0
    ws = torch.full((need + 4096,), 0xAB, dtype=torch.uint8, device=DEV)
    sums = torch.full((8, 57), -7.0, dtype=torch.float64, device=DEV)

    def gs(n_cols=10, G=4, nbytes=need, s=sums.data_ptr(), n_rows=n):
        return lib.ngacf_group_sums(rows.data_ptr(), n_rows, n_cols, grp.data_ptr(), G, s, ws.data_ptr(), nbytes, ops._s())
    for kw, what in (({"n_cols": 0}, b"0 columns"), ({"n_cols": 57}, b"57 columns"), ({"G": 0}, b"0 groups"), ({"G": 9}, b"9 groups")):
        assert gs(**kw) == -4 and what in lib.ngacf_last_error(), kw
    assert gs(s=None) == -1
    assert gs(nbytes=need - 1) == -3 and b"workspace" in lib.ngacf_last_error()
    torch.cuda.synchronize()
    assert bool((counts == 0x5A5A).all()) and bool((rows == -7.0).all()), "a refused ngacf_list_stats call wrote"
    assert bool((ws == 0xAB).all()) and bool((sums == -7.0).all()), "a refused ngacf_group_sums call wrote"
    # NULL optional outputs
    ref_c, ref_r = exposure(lists, I, ks), list_rows(lists, I, ks, tab)
    assert ls(r=None) == 0
    torch.cuda.synchronize()
    assert np.array_equal(counts.cpu().numpy(), ref_c) and bool((rows == -7.0).all())
    counts.fill_(0x5A5A)
    assert ls(c=None) == 0
    torch.cuda.synchronize()
    assert np.array_equal(rows.cpu().numpy(), ref_r) and bool((counts == 0x5A5A).all())
    assert ls(c=None, r=None) == 0
    # group sums within the reported workspace, twice the same bits
    s10 = sums[:4, :10]
    s_ok = torch.empty((4, 10), dtype=torch.float64, device=DEV)
    assert gs(s=s_ok.data_ptr()) == 0
    torch.cuda.synchronize()
    assert bool((ws[need:] == 0xAB).all()), "ngacf_group_sums wrote past its reported workspace"
    np.testing.assert_allclose(s_ok.cpu().numpy(), group_sums(ref_r, grp.cpu().numpy(), 4), rtol=1e-12, atol=1e-12)
    del s10
    c1, r1 = _list_stats(ids, I, ks, tables)
    c2, r2 = _list_stats(ids, I, ks, tables)
    g1, g2 = _gsums(r1, grp, 4), _gsums(r1, grp, 4)
    assert torch.equal(c1, c2) and torch.equal(r1, r2) and torch.equal(g1, g2) and torch.equal(g1, s_ok)
    # n_rows = 0: the counts are zeroed, the sums are zeros
    empty = ids[:0]
    c0, r0 = _list_stats(empty, I, ks, tables)
    assert bool((c0 == 0).all()) and r0.numel() == 0
    z = torch.full((3, 10), -7.0, dtype=torch.float64, device=DEV)
    assert gs(n_rows=0, G=3, s=z.data_ptr(), nbytes=ops.group_sums_workspace_bytes(0, 10, 3)) == 0
    torch.cuda.synchronize()
    assert bool((z == 0).all())
    # captured in a CUDA graph, replayed twice over garbage counts: the eager call's bits
    gc = torch.zeros_like(c1)
    gr = torch.zeros_like(r1)
    gsum = torch.zeros((4, 10), dtype=torch.float64, device=DEV)
    gws = torch.empty(need, dtype=torch.uint8, device=DEV)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        ops.list_stats(ids, I, ks, tables, gc, gr)
        ops.group_sums(gr, grp, 4, gsum, gws)
    torch.cuda.current_stream().wait_stream(st)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.list_stats(ids, I, ks, tables, gc, gr)
        ops.group_sums(gr, grp, 4, gsum, gws)
    for fill in (77, -1):
        gc.fill_(fill)
        gr.fill_(float(fill))
        gsum.fill_(float(fill))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(gc, c1) and torch.equal(gr, r1) and torch.equal(gsum, g1)


def _seeded_model(cls, U, I, width, seed=5):
    torch.manual_seed(seed)
    m = cls(U, I, width, [64, 64], 0.1).to(DEV)
    with torch.no_grad():            # larger embeddings than the N(0, 0.01) init, so that the scores spread
        m.uEmbd.weight.mul_(30)
        m.iEmbd.weight.mul_(30)
    return m


@pytest.fixture(scope="module")
def trained_case():
    """a split of a synthetic graph with skewed degrees, its interactions and seeded models' pre-ELU outputs at both widths"""
    from ngacf_b200.data import Interactions
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    U, I, E = 400, 900, 12000
    u, i = port.synth_bipartite(U, I, E, 31)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 32)
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    adj = torch.from_numpy(np.stack([u, i])).to(DEV)
    Z = {}
    for key, cls, width in (("64", SPUIGACF, 64), ("128", SPUIGACF, 128), ("multi64", SPUIMultiGACF, 64)):
        model = _seeded_model(cls, U, I, width).eval()
        with torch.no_grad():
            Z[key] = model.propagate(adj).clone()
    return SimpleNamespace(U=U, I=I, dit=dit, Z=Z, split=(tu, ti, su, si))


def _oracle_reports(ev, G):
    """list_metrics / group_metrics from the oracle applied to the evaluator's own lists and per-user rows"""
    it = ev.inter
    ks, nk = ev.ks, len(ev.ks)
    n = ev.users.numel()
    lists = ev.top_ids[:n].cpu().numpy()
    tab = item_tables(it.host["train_items"], it.I, it.n_train_users)
    counts = exposure(lists, it.I, ks)
    lrows = list_rows(lists, it.I, ks, tab)
    cov, gini = coverage_gini(counts, it.host["pool"])
    beyond = {"coverage": cov, "gini": gini, "novelty": lrows[:, :nk].sum(0) / n, "arp": lrows[:, nk:].sum(0) / n}
    # groups: users in (degree, id) order over the whole evaluation set
    users = it.eval_users.cpu().numpy()
    deg = np.diff(it.host["train_ptr"])[users]
    order = sorted(range(users.size), key=lambda j: (deg[j], users[j]))
    T = int(deg.sum())
    gid, C = {}, 0
    for j in order:
        gid[int(users[j])] = min(G - 1, (G * C) // T)
        C += int(deg[j])
    mine = ev.users.cpu().numpy()
    grp = np.array([gid[int(u)] for u in mine])
    acc = ev.per_user().cpu().numpy()
    groups = {"n_users": np.bincount(grp, minlength=G)}
    cnt = np.maximum(groups["n_users"], 1)[:, None]
    sa, sl = group_sums(acc, grp, G) / cnt, group_sums(lrows, grp, G) / cnt
    for q, name in enumerate(METRICS):
        groups[name] = sa[:, q * nk:(q + 1) * nk]
    groups["novelty"], groups["arp"] = sl[:, :nk], sl[:, nk:]
    gd = np.array([deg[j] for j in range(users.size)])
    ga = np.array([gid[int(u)] for u in users])
    groups["degree"] = np.array([[gd[ga == g].min(), gd[ga == g].max()] if (ga == g).any() else [0, 0] for g in range(G)])
    groups["interactions"] = np.array([gd[ga == g].sum() for g in range(G)])
    return beyond, groups, counts


def _close(got, ref):
    np.testing.assert_allclose(np.asarray(got, np.float64), np.asarray(ref, np.float64), rtol=1e-12, atol=1e-300)


def _check(ev, G):
    beyond, groups, counts = _oracle_reports(ev, G)
    b = ev.list_metrics()
    assert np.array_equal(ev._counts.cpu().numpy(), counts)
    assert np.array_equal(b["coverage"], beyond["coverage"]) and np.array_equal(b["gini"], beyond["gini"])
    _close(b["novelty"], beyond["novelty"])
    _close(b["arp"], beyond["arp"])
    assert b["ks"] == ev.ks and b["n_users"] == ev.users.numel() and b["n_items"] == ev.inter.host["pool"].size
    g = ev.group_metrics(G)
    assert g["groups"] == G and g["ks"] == ev.ks
    assert np.array_equal(g["n_users"], groups["n_users"])
    assert np.array_equal(g["degree"], groups["degree"]) and np.array_equal(g["interactions"], groups["interactions"])
    for name in METRICS + ("novelty", "arp"):
        assert g[name].shape == (G, len(ev.ks))
        _close(g[name], groups[name])
    return b, g


@gpu
@pytest.mark.parametrize("key,ks", [("64", [10, 20]), ("64", [5, 50, 100]), ("128", [20]), ("128", [1, 37, 100]), ("multi64", [3, 10, 37])])
def test_evaluator_matches_oracle(trained_case, key, ks):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    ev = FullRankingEvaluator(trained_case.dit, ks)
    m = ev(trained_case.Z[key])
    for G in (1, 3, 4, 8):
        _check(ev, G)
    one = ev.group_metrics(1)
    assert one["n_users"].tolist() == [m["n_users"]]
    for name in METRICS:
        _close(one[name][0], m[name])
    b = ev.list_metrics()
    _close(one["novelty"][0], b["novelty"])
    _close(one["arp"][0], b["arp"])


@gpu
def test_both_sources_give_the_same_reports(trained_case):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    for ks in ([1, 5, 10, 20], [3, 7]):
        a = FullRankingEvaluator(trained_case.dit, ks, "auto")
        b = FullRankingEvaluator(trained_case.dit, ks, "exact")
        a.rank(trained_case.Z["64"])
        b.rank(trained_case.Z["64"])
        assert a.source == "tc" and b.source == "list"
        for x, y in ((a.list_metrics(), b.list_metrics()), (a.group_metrics(5), b.group_metrics(5))):
            assert x.keys() == y.keys()
            for k in x:
                assert np.array_equal(np.asarray(x[k]), np.asarray(y[k])), k


@gpu
def test_refusals(trained_case):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    it = trained_case.dit
    ev = FullRankingEvaluator(it, [20])
    with pytest.raises(RuntimeError):
        ev.list_metrics()
    ev.rank(trained_case.Z["64"])
    for bad in (0, 9, 2.5, True, None):
        with pytest.raises(ValueError):
            ev.group_metrics(bad)
    # the same split without the test items of users 0..9: those users are no evaluation users there
    from ngacf_b200.data import Interactions
    tu, ti, su, si = trained_case.split
    keep = su >= 10
    it2 = Interactions.from_arrays(it.U, it.I, tu, ti, su[keep], si[keep], device=DEV)
    assert not bool((it2.eval_users < 10).any())
    users = torch.cat([it2.eval_users[:5], _t([3])])
    ev2 = FullRankingEvaluator(it2, [20], users=users)
    ev2.rank(trained_case.Z["64"])
    with pytest.raises(ValueError, match="evaluation users"):
        ev2.group_metrics(2)
    ev2.list_metrics()      # any users are fine for the list metrics


@gpu
def test_shards_equal_the_whole(trained_case, monkeypatch):
    """world 1..4: the shards' counts add up to the whole exactly, and with the all-reduce played back over the shards' own buffers
    every rank's dicts equal the unsharded ones (coverage and Gini exactly, the rest to 1e-12)"""
    import ngacf_b200.dist as D
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    it = trained_case.dit
    for ks in ([5, 20], [5, 50, 100]):
        whole = FullRankingEvaluator(it, ks)
        whole.rank(trained_case.Z["64"])
        wb, wg = whole.list_metrics(), whole.group_metrics(4)
        wcounts = whole._counts.clone()
        for world in range(1, 5):
            evs = [FullRankingEvaluator(it, ks, users=D.shard_eval_users(it.eval_users, r, world)) for r in range(world)]
            for ev in evs:
                ev.rank(trained_case.Z["64"])
            total = torch.zeros_like(wcounts)
            for ev in evs:
                ev._list_stats(True)
                total += ev._counts
            assert torch.equal(total, wcounts)
            for method, arg, ref in (("list_metrics", (), wb), ("group_metrics", (4,), wg)):
                recorded = [[] for _ in evs]             # phase 1: each rank's buffers before the all-reduce
                for r, ev in enumerate(evs):
                    monkeypatch.setattr(D, "allreduce_sums", lambda t, r=r: recorded[r].append(t.clone()) or t)
                    getattr(ev, method)(*arg)
                for r, ev in enumerate(evs):             # phase 2: the all-reduce returns the sum over the ranks
                    calls = iter(range(len(recorded[0])))

                    def merged(t):
                        c = next(calls)
                        return t.copy_(sum(rec[c] for rec in recorded))
                    monkeypatch.setattr(D, "allreduce_sums", merged)
                    got = getattr(ev, method)(*arg)
                    for k in ref:
                        if k in ("coverage", "gini", "ks", "groups", "n_users", "n_items", "degree", "interactions"):
                            assert np.array_equal(np.asarray(got[k]), np.asarray(ref[k])), (world, method, k)
                        else:
                            _close(got[k], ref[k])
            monkeypatch.undo()


def _cli_lines(R, flags, capsys):
    args = R.parse_args(flags)
    torch.manual_seed(args.seed)
    torch.cuda.manual_seed_all(args.seed)
    np.random.seed(args.seed)
    R.main(args)
    out = capsys.readouterr().out
    # wall-clock times vary between runs
    return [l.split(", time")[0] for l in out.splitlines() if "time of evaluate" not in l and "timeStamp" not in l]


NEW_LINES = ("beyond-accuracy metrics:", "user-group metrics:")


def _check_against_checkpoint(R, flags, lines, ks, G, capsys):
    """the printed beyond-accuracy and user-group lines of a run equal the Python API on the checkpoint that run saved"""
    import ast
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    i = [j for j, l in enumerate(lines) if "full-ranking" in l]
    assert len(i) == 1 and lines[i[0] + 1].startswith("epoch:0 beyond-accuracy metrics:")
    assert lines[i[0] + 2].startswith("epoch:0 user-group metrics:")
    assert not any("full-ranking" in l for l in lines[i[0] + 1:])
    beyond = ast.literal_eval(lines[i[0] + 1].split("beyond-accuracy metrics:", 1)[1])
    groups = ast.literal_eval(lines[i[0] + 2].split("user-group metrics:", 1)[1])
    args = R.parse_args(flags)
    inter, _, _, _, U, I, adj = R.prepareData(args)
    capsys.readouterr()          # prepareData's own lines
    model, _, _ = R.createModels(args, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    model.eval()
    ev = FullRankingEvaluator(inter, ks)
    with torch.no_grad():
        ev.rank(model.propagate(adj.to(DEV)))
    b, g = ev.list_metrics(), ev.group_metrics(G)
    for k in b:
        if k in ("coverage", "gini", "ks", "n_users", "n_items"):
            assert beyond[k] == (b[k].tolist() if hasattr(b[k], "tolist") else b[k]), k
        else:
            _close(beyond[k], b[k])
    for k in g:
        if k in ("ks", "groups", "n_users", "degree", "interactions"):
            assert groups[k] == (g[k].tolist() if hasattr(g[k], "tolist") else g[k]), k
        else:
            _close(groups[k], g[k])
    return i[0]


@gpu
def test_cli(tmp_path, monkeypatch, capsys):
    import run_Gowalla as R
    monkeypatch.chdir(tmp_path)
    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--epochs", "1", "--eval_every", "1", "--save_every", "1",
            "--droprate", "0.2", "--batch_size", "2048", "--eval_ks", "100,5,50"]
    flags = ["--eval_beyond", "True", "--eval_groups", "3"]
    allneg = base + ["--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--lr", "0.002", "--parallel", "False"]
    plain = _cli_lines(R, allneg, capsys)
    assert not any(s in l for l in plain for s in NEW_LINES)
    both = _cli_lines(R, allneg + flags, capsys)
    assert [l for l in both if not any(s in l for s in NEW_LINES)] == plain
    i = _check_against_checkpoint(R, allneg, both, [5, 50, 100], 3, capsys)
    assert len(both) == i + 3                # AllNeg: the full-ranking line ends the epoch's evaluation
    # the default modes (NegSampling / SampledNeg): the lines follow the full-ranking line with the values of the Python API,
    # --parallel True in one process prints the same, and the other lines are those of a run without the flags
    neg = base[:-2] + ["--eval_ks", "20"]
    plain = _cli_lines(R, neg + ["--parallel", "False"], capsys)
    a = _cli_lines(R, neg + flags + ["--parallel", "False"], capsys)
    c = _cli_lines(R, neg + flags + ["--parallel", "True"], capsys)
    assert a == c
    assert [l for l in a if not any(s in l for s in NEW_LINES)] == plain
    i = _check_against_checkpoint(R, neg + ["--parallel", "False"], a, [20], 3, capsys)
    assert "HR:" in a[i - 1]
