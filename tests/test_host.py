"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/ngacf_b200.h
declares (no compute call is made without a GPU), the drop-in module mirrors the reference's
constructor / parameter names / init, and the product refuses to run without CUDA."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    txt = open(os.path.join(ROOT, "include", "ngacf_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(ngacf_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    from ngacf_b200 import _lib
    ge.build()
    lib = _lib.load()
    names = header_functions()
    assert len(names) >= 20
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    assert set(names) == set(_lib.SIGNATURES), set(names) ^ set(_lib.SIGNATURES)
    assert lib.ngacf_version() >= 100
    # argument validation happens before any CUDA call
    assert lib.ngacf_transform_fwd(None, None, 0, None, 1.0, None, 8, 10, 10, None, None, None) == -1
    assert b"transform_fwd" in lib.ngacf_last_error()


def test_only_sm100a_code_in_the_library():
    import subprocess
    from ngacf_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.STDOUT).stdout.decode()
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_dense_and_eval_kernels_use_the_tensor_cores():
    """tcgen05 in the SASS: UTCHMMA (MMA), LDTM (TMEM loads) for the dense transforms and the AllNeg scorer."""
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from ngacf_b200 import _lib
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=600).stdout
    per_kernel = {}
    name = None
    for line in sass.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
        elif name and "UTCHMMA" in line:
            per_kernel[name] = per_kernel.get(name, 0) + 1
    assert any("transform_tc_kernel" in k for k in per_kernel), sorted(per_kernel)
    assert any("transform_bwd_tc_kernel" in k for k in per_kernel), sorted(per_kernel)
    assert any("score_topk_tc_kernel" in k for k in per_kernel), sorted(per_kernel)
    assert "LDTM" in sass


def test_model_mirrors_reference_names_and_shapes():
    from graphattention.BPRLoss import BPRLoss  # noqa: F401  (re-export import path of the reference)
    from graphattention.SPUIGACF import SPUIGACF
    m = SPUIGACF(30, 40, 64, [64, 64], 0.1)
    sd = m.state_dict()
    want = {"uEmbd.weight": (30, 64), "iEmbd.weight": (40, 64), "gat.out_att.W_u": (64, 64), "gat.out_att.W_i": (64, 64), "gat.out_att.a": (1, 128)}
    for k in range(8):
        want.update({f"gat.attention_{k}.W_u": (64, 8), f"gat.attention_{k}.W_i": (64, 8), f"gat.attention_{k}.a": (1, 16)})
    assert {k: tuple(v.shape) for k, v in sd.items()} == want
    assert len(list(m.parameters())) == 29


def test_same_seed_same_init_and_checkpoint_interchange(golden):
    """torch.manual_seed(s) -> the drop-in module draws exactly the reference's initial parameters, and the
    state_dicts load into each other (SURVEY.md 5.4 checkpoint contract).  The reference's draws are the sd0/ arrays of
    tests/golden/ml100k_2epochs.npz: its state_dict, in its key order, right after torch.manual_seed(2019) and
    SPUIGACF(943, 1682, 64, [64, 64], 0.2) (oracle/make_golden.py:case_ml100k)."""
    from ngacf_b200.model import SPUIGACF
    gz = golden("ml100k_2epochs")
    sr = {k[len("sd0/"):]: torch.from_numpy(gz[k]) for k in gz.files if k.startswith("sd0/")}
    torch.manual_seed(2019)
    mine = SPUIGACF(int(gz["U"]), int(gz["I"]), 64, [64, 64], 0.2)
    sm = mine.state_dict()
    assert list(sr.keys()) == list(sm.keys())
    for k in sr:
        assert torch.equal(sr[k], sm[k]), k
    assert [n for n, _ in mine.named_parameters()] == list(sr.keys())      # parameters only: nothing else to carry over
    mine.load_state_dict(sr)


def test_no_cpu_fallback():
    from ngacf_b200 import NgacfError
    from ngacf_b200.model import SPUIGACF
    m = SPUIGACF(5, 6, 64, [64, 64], 0.0)
    with pytest.raises(NgacfError):
        m(torch.tensor([0]), torch.tensor([1]), torch.tensor([[0, 1, 2, 3, 4], [0, 1, 2, 3, 4]]))


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under ngacf_b200/ or the drop-in entry modules may import it."""
    bad = []
    files = [os.path.join(dp, f) for dp, _, fs in os.walk(os.path.join(ROOT, "ngacf_b200")) for f in fs if f.endswith(".py")]
    files += [os.path.join(ROOT, f) for f in ("train_eval_Gowalla.py", "run_Gowalla.py") if os.path.exists(os.path.join(ROOT, f))]
    files += [os.path.join(ROOT, "graphattention", f) for f in os.listdir(os.path.join(ROOT, "graphattention")) if f.endswith(".py")]
    for f in files:
        src = open(f).read()
        if re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M):
            bad.append(f)
    assert not bad, bad


def test_interactions_from_reference_frames_matches_arrays():
    """The pandas-sets structures of the reference (loadGowalla.py:63-67,86-88) convert to the same CSR."""
    import pandas as pd
    from ngacf_b200.data import Interactions
    U, I = 40, 60
    u, i = port.synth_bipartite(U, I, 500, 9)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 10)
    a = Interactions.from_arrays(U, I, tu, ti, su, si, device="cpu")
    rt_items = set(np.concatenate([ti, si]).tolist())
    train_df = pd.DataFrame(dict(userId=tu, itemId=ti, rating=1))
    tpn = train_df.groupby("userId")["itemId"].apply(set).reset_index().rename(columns={"itemId": "positive_items"})
    tpn["negative_items"] = tpn["positive_items"].apply(lambda x: rt_items - x)
    test_pos = pd.DataFrame(dict(userId=su, itemId=si)).groupby("userId")["itemId"].apply(set).reset_index().rename(columns={"itemId": "positive_items"})
    b = Interactions.from_reference_frames(U, I, train_df, tpn, test_pos, device="cpu")
    c = Interactions.from_reference_frames(U, I, None, tpn, test_pos, device="cpu")
    for name in ("train_ptr", "train_items", "train_rank", "pool", "in_pool", "test_ptr", "test_items", "eval_users"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
        assert torch.equal(getattr(a, name), getattr(c, name)), name
    assert torch.equal(a.train_rows_user, b.train_rows_user)
    assert a.n_train_users == b.n_train_users == c.n_train_users
    ref = port.build_interactions(U, I, tu, ti, su, si)
    assert np.array_equal(a.train_ptr.numpy(), ref.train_ptr) and np.array_equal(a.train_rank.numpy(), ref.train_rank)
    users, div = port.eval_users(ref)
    assert np.array_equal(a.eval_users.numpy(), users) and a.n_train_users == div


def test_interactions_negsampling_views_on_cpu():
    """Row-order item columns, test rows and the train+test union used by the NegSampling / SampledNeg kernels (host logic only)."""
    from ngacf_b200.data import Interactions
    U, I, E = 40, 60, 500
    u, i = port.synth_bipartite(U, I, E, 1)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 2)
    it = port.build_interactions(U, I, tu, ti, su, si)
    ap = port.AllPositives(it)
    d = Interactions.from_arrays(U, I, tu, ti, su, si, device="cpu")
    assert np.array_equal(d.train_rows_item.numpy(), ti) and np.array_equal(d.test_rows_user.numpy(), su) and np.array_equal(d.test_rows_item.numpy(), si)
    assert np.array_equal(d.all_ptr.numpy(), ap.ptr) and np.array_equal(d.all_rank.numpy(), ap.rank)
    assert d.n_test_rows == su.shape[0]
    assert d.min_negatives() == it.pool.shape[0] - int(np.diff(ap.ptr).max())


def test_host_data_layer_csv_and_splits(tmp_path):
    """run_Gowalla.py's prepareData without python sets (SURVEY 8f-2): the Gowalla/Yelp CSV layout, the synthetic shapes and both
    split rules (80/20 per user for PairSampling, leave-one-out for NegSampling)."""
    from ngacf_b200 import hostdata
    rng = np.random.default_rng(0)
    U, I = 30, 50
    rows = np.unique(np.stack([rng.integers(0, U, 600), rng.integers(0, I, 600)], 1), axis=0)
    rows = np.concatenate([rows, np.stack([np.arange(U), np.arange(U) % I], 1)])          # every user present
    rows = np.unique(rows, axis=0)
    is_test = np.zeros(len(rows), bool)
    is_test[::5] = True
    te, tr = rows[is_test], rows[~is_test]
    os.makedirs(tmp_path / "Gowalla")
    np.savetxt(tmp_path / "Gowalla" / "g_train.csv", np.c_[tr, np.ones(len(tr), int)], fmt="%d", delimiter=",")
    np.savetxt(tmp_path / "Gowalla" / "g_test.csv", np.c_[te, np.ones(len(te), int)], fmt="%d", delimiter=",")
    d = hostdata.load_dataset("Gowalla", str(tmp_path))
    assert d["userNum"] == rows[:, 0].max() + 1 and d["itemNum"] == rows[:, 1].max() + 1
    assert np.array_equal(d["train_u"], tr[:, 0]) and np.array_equal(d["train_i"], tr[:, 1])
    assert np.array_equal(d["test_u"], te[:, 0]) and np.array_equal(d["test_i"], te[:, 1])
    assert np.array_equal(np.sort(d["rt_u"] * 1000 + d["rt_i"]), np.sort(rows[:, 0] * 1000 + rows[:, 1]))
    with pytest.raises(FileNotFoundError):
        hostdata.load_dataset("Yelp", str(tmp_path))
    # synthetic shapes: PairSampling keeps >= 1 train edge per user; NegSampling holds out exactly one row per user
    a = hostdata.load_dataset("synth-tiny", None, "PairSampling")
    b = hostdata.load_dataset("synth-tiny", None, "NegSampling")
    Ut = a["userNum"]
    assert np.bincount(a["train_u"], minlength=Ut).min() >= 1 and len(a["train_u"]) + len(a["test_u"]) == 60000
    assert np.array_equal(np.bincount(b["test_u"], minlength=Ut), np.ones(Ut, np.int64)) and len(b["train_u"]) + Ut == 60000
    assert np.array_equal(np.sort(a["rt_u"] * 10000 + a["rt_i"]), np.sort(b["rt_u"] * 10000 + b["rt_i"]))


def test_integration_stub_matches_the_abi():
    """The ctypes stub shown in INTEGRATION.md binds ngacf_aggregate_fwd with as many arguments as the library's signature table."""
    from ngacf_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "INTEGRATION.md")).read()
    m = re.search(r"lib\.ngacf_aggregate_fwd\.argtypes = \[(.*?)\]", text)
    assert m, "stub not found"
    shown = [a.strip() for a in m.group(1).split(",")]
    sig = _lib.SIGNATURES["ngacf_aggregate_fwd"][1]
    assert len(shown) == len(sig), (len(shown), len(sig))
    for name in re.findall(r"`(ngacf_[a-z_0-9]+)`", text):       # every entry point the document names exists
        base = name
        assert base in _lib.SIGNATURES or any(k.startswith(base) for k in _lib.SIGNATURES), name


def test_normalized_laplacian_matches_reference_fixture():
    """ngacf_b200.gp.normalized_laplacian (host side of SPUIGAGPCF, SURVEY 8f-1) == the reference's buildLaplacianMat(..., 'norm_adj')
    + scipySP_torchSP + coalesce, whose output is stored in tests/golden/gagpcf_small.npz."""
    from ngacf_b200.gp import normalized_laplacian
    gz = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gagpcf_small.npz"))
    U, I = int(gz["U"]), int(gz["I"])
    L = normalized_laplacian(U, I, gz["edge_u"], gz["edge_i"], gz["rating"], "norm_adj")
    assert np.array_equal(L.indices()[0].numpy(), gz["lap_row"]) and np.array_equal(L.indices()[1].numpy(), gz["lap_col"])
    assert np.allclose(L.values().numpy(), gz["lap_val"], rtol=1e-6, atol=0)
    M = normalized_laplacian(U, I, gz["edge_u"], gz["edge_i"], None, "mean_adj").to_dense().numpy()
    assert np.allclose(M, M.T) and np.allclose(np.diag(M), 0)


def test_fused_paths_take_exact_model_types_only():
    """A subclass with layers behind the propagation (SPUIGAGPCF) is an SPUIGACF instance, but the captured training steps and the
    evaluators work on the 64-wide SpUIGAT features alone: they must refuse it instead of silently training / ranking its base."""
    import torch
    import train_eval_Gowalla as te
    from graphattention.BPRLoss import BPRLoss
    from graphattention.SPUIGACF import SPUIGACF, SPUIGAGPCF, SPUIMultiGACF
    U, I = 12, 15
    L = torch.sparse_coo_tensor(torch.tensor([[0, U], [U, 0]]), torch.tensor([0.5, 0.5]), (U + I, U + I))
    for cls, ok in ((SPUIGACF, True), (SPUIMultiGACF, True)):
        m = cls(U, I, 64, [64, 64], 0.1, useCuda=False)
        opt = torch.optim.Adam(m.parameters(), lr=0.01)
        assert te._fused_ok(m, opt, BPRLoss()) is ok
        assert te._plain_gat_model(m)
    m = SPUIGAGPCF(U, I, L, 64, [64, 64], 0.1, useCuda=False)
    opt = torch.optim.Adam(m.parameters(), lr=0.01)
    assert isinstance(m, SPUIGACF) and not te._fused_ok(m, opt, BPRLoss()) and not te._plain_gat_model(m)
    with pytest.raises(NotImplementedError):
        te._require_plain(m, "eval_neg_all")


def test_homograph_nonzero_index_matches_adj_nonzero_order():
    """HomoGraph.nonzero_index (kernel order of the directed edges -> index into adj.nonzero(), the order in which the reference
    draws its edge dropout, SPGA.py:379,398) against the dense adjacency, with and without the diagonal.  Runs on CPU tensors: the
    method is pure index arithmetic over the unified adjacency."""
    import types
    import torch
    from oracle import port
    from ngacf_b200.spgat import HomoGraph
    U, I = 17, 23
    u, i = port.synth_bipartite(U, I, 160, 3)
    g = port.build_graph(np.stack([u, i]), U, I)
    N, E = U + I, g.E
    adj_ptr = np.concatenate([g.rowptr.astype(np.int64), E + g.colptr[1:].astype(np.int64)])
    adj_idx = np.concatenate([g.colidx.astype(np.int64) + U, g.rowidx.astype(np.int64)])        # neighbour node of every position
    node = np.repeat(np.arange(N), np.diff(adj_ptr))
    fake = types.SimpleNamespace(adj_ptr=torch.from_numpy(adj_ptr), N=N, U=U, E=E, device=torch.device("cpu"))
    for self_loops in (False, True):
        row, col = port.homo_edges(g, self_loops)
        dense = torch.zeros(N, N)
        dense[torch.from_numpy(row), torch.from_numpy(col)] = 1
        nz = dense.nonzero().numpy()
        assert (nz[:, 0] == row).all() and (nz[:, 1] == col).all()          # the port's edge order IS adj.nonzero()
        idx = HomoGraph.nonzero_index(types.SimpleNamespace(g=fake, self_loops=self_loops)).numpy()
        assert idx.shape[0] == 2 * E + (N if self_loops else 0) and len(set(idx.tolist())) == idx.shape[0]
        assert (row[idx[:2 * E]] == node).all() and (col[idx[:2 * E]] == adj_idx).all()
        if self_loops:
            assert (row[idx[2 * E:]] == np.arange(N)).all() and (col[idx[2 * E:]] == np.arange(N)).all()
