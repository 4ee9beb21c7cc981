"""embedSize 128: the width-carrying (`_w`) entry points, the models, trainers, evaluators and the CLI at d = 128.

The oracle at d = 128 is the CPU port (oracle/port.py) with the width taken from the parameters: its stage forward, Philox and
summation tree (dot64_tree is generic over the length) are width-generic; the helpers below restate the two places where it names
64 (the per-row mask stream and the dW reshape of the closed-form backward) for any width.  At width 64 they equal the port's
functions, which are pinned against the reference fixtures (test_feature_mask_stream_widths, test_stage_backward_at_64_equals_port)."""
import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------
# width-generic oracle helpers
# ------------------------------------------------------------------------------------------------
def feature_mask_bits(N, seed, call, stage, droprate, width=64):
    """uint64[N * width/64]: row n draws Philox counters (n*(width/8) + c, 0, site, call), c = 0 .. width/8-1, eight decisions each
    for columns 8c .. 8c+7; word w of the row holds columns 64w .. 64w+63."""
    thr = port.keep_threshold(droprate)
    site = stage * 2 + port.SITE_FEAT
    C = width // 8
    n = np.arange(N, dtype=np.uint64)
    out = np.zeros((N, width // 64), dtype=np.uint64)
    for c in range(C):
        idx = n * np.uint64(C) + np.uint64(c)
        w = port.philox4x32_10((idx & port._MASK32).astype(np.uint32), (idx >> np.uint64(32)).astype(np.uint32), np.uint32(site),
                               np.uint32(call), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
        for j in range(8):
            out[:, c // 8] |= port._decisions(w, j, thr).astype(np.uint64) << np.uint64(8 * (c % 8) + j)
    return out.reshape(-1)


def unpack_feature_mask(bits, width=64):
    words = np.asarray(bits, np.uint64).reshape(-1, width // 64)
    return ((words[:, :, None] >> np.arange(64, dtype=np.uint64)[None, None, :]) & np.uint64(1)).astype(bool).reshape(-1, width)


def stages_of(width, multi=False):
    return [(8, 8)] * (2 if multi else 1) + [(1, width)]


def init_params(U, I, width, seed=3, dtype=torch.float64, multi=False):
    """the port's initialisation with stage input widths (width, 64, ...)"""
    gen = torch.Generator().manual_seed(seed)

    def xavier(shape, fan_in, fan_out):
        std = 1.414 * np.sqrt(2.0 / (fan_in + fan_out))
        return (torch.randn(shape, generator=gen, dtype=torch.float64) * std).to(dtype)
    p = dict(uEmbd=(torch.randn((U, width), generator=gen, dtype=torch.float64) * 0.2).to(dtype),
             iEmbd=(torch.randn((I, width), generator=gen, dtype=torch.float64) * 0.2).to(dtype), stages=[])
    din = width
    for H, DH in stages_of(width, multi):
        p["stages"].append(dict(Wu=xavier((H, din, DH), DH, din), Wi=xavier((H, din, DH), DH, din), a=xavier((H, 2 * DH), 2 * DH, 1)))
        din = H * DH
    return p


def propagate(p, g, keeps=None, droprate=0.0):
    """port.propagate with explicit (feature keep (N, d_in) bool, edge keep (E, H) bool) per stage"""
    X = torch.cat([p["uEmbd"], p["iEmbd"]], 0)
    caches = []
    for k, st in enumerate(p["stages"]):
        fk, ek = (None, None) if keeps is None else keeps[k]
        c = port.stage_forward(X, st, g, fk, ek, droprate)
        caches.append(c)
        X = port._elu(c["Z"])
    return X, caches


def stage_backward(G, c, st, g):
    """port.stage_backward (the closed form of SURVEY.md 3.4) with dW shaped from the stage input width instead of port.D"""
    U, N = g.U, g.N
    H, DH = c["H"], c["DH"]
    Din = c["Xd"].shape[1]
    eu = torch.from_numpy(g.eu)
    ei = torch.from_numpy(g.ei) + U
    Gv = G.view(N, H, DH)
    hv = c["h"].view(N, H, DH)
    Ghat = Gv * c["inv"][:, :, None]
    dN = -(Gv * c["A"].view(N, H, DH)).sum(-1) * c["inv"]
    det = (Ghat[eu] * hv[ei]).sum(-1) + (Ghat[ei] * hv[eu]).sum(-1)
    m = 1.0 if c["edge_keep"] is None else c["edge_keep"].to(G.dtype) * c["scale"]
    de = det * m + dN[eu] + dN[ei]
    x = c["s"][eu] + c["s"][ei]
    ds = de * (-c["e"]) * torch.where(x > 0, torch.ones_like(x), torch.full_like(x, port.ALPHA))
    dS = torch.zeros(N, H, dtype=G.dtype).index_add_(0, eu, ds).index_add_(0, ei, ds)
    dh = Gv.clone()
    dh.index_add_(0, eu, c["et"][:, :, None] * Ghat[ei])
    dh.index_add_(0, ei, c["et"][:, :, None] * Ghat[eu])
    a_u, a_i = st["a"][:, :DH], st["a"][:, DH:]
    dh[:U] += dS[:U, :, None] * a_u[None]
    dh[U:] += dS[U:, :, None] * a_i[None]
    da = torch.cat([(dS[:U, :, None] * hv[:U]).sum(0), (dS[U:, :, None] * hv[U:]).sum(0)], 1)
    dh2 = dh.reshape(N, H * DH)
    dWu = (c["Xd"][:U].t() @ dh2[:U]).view(Din, H, DH).permute(1, 0, 2).contiguous()
    dWi = (c["Xd"][U:].t() @ dh2[U:]).view(Din, H, DH).permute(1, 0, 2).contiguous()
    dXd = torch.cat([dh2[:U] @ port._wcat(st["Wu"]).t(), dh2[U:] @ port._wcat(st["Wi"]).t()], 0)
    dX = dXd if c["feat_keep"] is None else dXd * c["feat_keep"].to(G.dtype) * c["scale"]
    return dX, dict(Wu=dWu, Wi=dWi, a=da)


def propagate_backward(dF, p, g, caches):
    grads = dict(stages=[None] * len(caches))
    dX = dF
    for k in range(len(caches) - 1, -1, -1):
        G = dX * port._elu_grad(caches[k]["Z"])
        dX, gs = stage_backward(G, caches[k], p["stages"][k], g)
        grads["stages"][k] = gs
    grads["uEmbd"], grads["iEmbd"] = dX[:g.U].clone(), dX[g.U:].clone()
    return grads


def port_keeps(g, seed, call, droprate, width, multi=False):
    st = stages_of(width, multi)
    w_in = [width] + [H * DH for H, DH in st[:-1]]
    feat = [feature_mask_bits(g.N, seed, call, k, droprate, w) for k, w in enumerate(w_in)]
    edge = [port.edge_mask_bits(g.E, H, seed, call, k, droprate) for k, (H, _) in enumerate(st)]
    keeps = [(torch.from_numpy(unpack_feature_mask(f, w)), torch.from_numpy(port.unpack_edge_mask(e, H)))
             for f, e, w, (H, _) in zip(feat, edge, w_in, st)]
    return feat, edge, keeps


def small_graph(U=60, I=90, E=900, seed=4):
    u, i = port.synth_bipartite(U, I - 3, E, seed)       # the last items have no edge
    return u, i, port.build_graph(np.stack([u, i]), U, I)


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-300))


# ------------------------------------------------------------------------------------------------
# CPU: the specification at d = 128
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("multi", [False, True])
@pytest.mark.parametrize("droprate", [0.0, 0.3])
def test_port_backward_equals_autograd_at_128(multi, droprate):
    u, i, g = small_graph()
    p = init_params(g.U, g.I, 128, multi=multi)
    keeps = port_keeps(g, 11, 2, droprate, 128, multi)[2] if droprate > 0 else None
    leaves = [p["uEmbd"], p["iEmbd"]] + [st[k] for st in p["stages"] for k in ("Wu", "Wi", "a")]
    for t in leaves:
        t.requires_grad_(True)
    F, caches = propagate(p, g, keeps, droprate)
    assert F.shape == (g.N, 128)
    dF = torch.randn(F.shape, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    (F * dF).sum().backward()
    with torch.no_grad():
        grads = propagate_backward(dF, p, g, caches)
    assert torch.allclose(grads["uEmbd"], p["uEmbd"].grad, rtol=0, atol=1e-10 * p["uEmbd"].grad.abs().max())
    assert torch.allclose(grads["iEmbd"], p["iEmbd"].grad, rtol=0, atol=1e-10 * p["iEmbd"].grad.abs().max())
    for gs, st in zip(grads["stages"], p["stages"]):
        for k in ("Wu", "Wi", "a"):
            assert gs[k].shape == st[k].shape
            assert (gs[k] - st[k].grad).abs().max() <= 1e-10 * st[k].grad.abs().max(), k


def test_stage_backward_at_64_equals_port():
    u, i, g = small_graph()
    p = port.init_params(g.U, g.I, 3, torch.float64)
    masks = port.dropout_masks(g, 8, 1, 0.3)
    F, caches = port.propagate(p, g, masks, 0.3)
    dF = torch.randn(F.shape, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    ref = port.propagate_backward(dF, p, g, caches)
    ours = propagate_backward(dF, p, g, caches)
    assert torch.equal(ours["uEmbd"], ref["uEmbd"]) and torch.equal(ours["iEmbd"], ref["iEmbd"])
    for a, b in zip(ours["stages"], ref["stages"]):
        for k in ("Wu", "Wi", "a"):
            assert torch.equal(a[k], b[k]), k


def test_feature_mask_stream_widths():
    N = 300
    bits64 = feature_mask_bits(N, 0x1234567890ABCDEF, 7, 1, 0.3, 64)
    assert np.array_equal(bits64, port.feature_mask_bits(N, 0x1234567890ABCDEF, 7, 1, 0.3))
    bits = feature_mask_bits(N, 0x1234567890ABCDEF, 7, 0, 0.3, 128)
    assert bits.shape == (2 * N,)
    # layout: decision (n, col) comes from counter n*16 + col//8, 16-bit field col%8, in word 2n + col//64 at bit col%64
    thr = port.keep_threshold(0.3)
    for n, col in ((0, 0), (0, 127), (5, 64), (N - 1, 71), (17, 9)):
        ctr = n * 16 + col // 8
        w = port.philox4x32_10(np.uint32(ctr), np.uint32(0), np.uint32(0), np.uint32(7), 0x90ABCDEF, 0x12345678)
        dec = bool(port._decisions(w, col % 8, thr))
        assert bool((int(bits[2 * n + col // 64]) >> (col % 64)) & 1) == dec
    keep = unpack_feature_mask(bits, 128).mean()
    sd = np.sqrt(0.7 * 0.3 / (N * 128))
    assert abs(keep - 0.7) < 5 * sd


def test_models_at_128_on_cpu():
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    torch.manual_seed(0)
    m = SPUIGACF(30, 40, 128, [64, 64], 0.1)
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert shapes["uEmbd.weight"] == (30, 128) and shapes["iEmbd.weight"] == (40, 128)
    for k in range(8):
        assert shapes["gat.attention_%d.W_u" % k] == (128, 8) and shapes["gat.attention_%d.W_i" % k] == (128, 8)
        assert shapes["gat.attention_%d.a" % k] == (1, 16)
    assert shapes["gat.out_att.W_u"] == (64, 128) and shapes["gat.out_att.W_i"] == (64, 128) and shapes["gat.out_att.a"] == (1, 256)
    assert m.stages == ((8, 8), (1, 128))
    m2 = SPUIGACF(30, 40, 128, [64, 64], 0.1)
    m2.load_state_dict(m.state_dict())
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    mm = SPUIMultiGACF(30, 40, 128, [64, 64], 0.1)
    sh = {k: tuple(v.shape) for k, v in mm.state_dict().items()}
    assert sh["gat.attention1_0.W_u"] == (128, 8) and sh["gat.attention2_0.W_u"] == (64, 8) and sh["gat.out_att.W_u"] == (64, 128)
    assert mm.stages == ((8, 8), (8, 8), (1, 128))
    p = port.params_from_state_dict(mm.state_dict(), torch.float64)
    assert p["stages"][0]["Wu"].shape == (8, 128, 8) and p["stages"][2]["Wu"].shape == (1, 64, 128)
    # at 64 the construction (and so the RNG draw order) is unchanged
    torch.manual_seed(0)
    a = SPUIMultiGACF(30, 40, 64, [64, 64], 0.1).state_dict()
    assert {k: tuple(v.shape) for k, v in a.items()}["gat.attention2_3.W_u"] == (64, 8)


@pytest.mark.parametrize("bad", [32, 96, 256])
def test_unsupported_widths_refuse(bad):
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    for cls in (SPUIGACF, SPUIMultiGACF):
        with pytest.raises(ValueError, match="64 and 128"):
            cls(10, 10, bad, [64, 64], 0.1)


def test_refusals_at_128():
    from ngacf_b200.dist import require_width_64
    from ngacf_b200.gp import SPUIGAGPCF
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.spgat import SPGACF
    adj = torch.tensor([[0, 1], [0, 1]])
    with pytest.raises(ValueError, match="embedSize 64"):
        SPUIGAGPCF(2, 2, adj, 128, [64, 64], 0.1)
    with pytest.raises(ValueError, match="embedSize 64"):
        SPGACF(2, 2, adj, 128, [64, 64], 0.1)
    with pytest.raises(ValueError, match="multi-GPU"):
        require_width_64(SPUIGACF(2, 2, 128, [64, 64], 0.1))
    require_width_64(SPUIGACF(2, 2, 64, [64, 64], 0.1))


def test_cli_refuses_parallel_128_before_process_group(monkeypatch):
    import run_Gowalla as R
    import torch.distributed as dist
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: pytest.fail("process group created"))
    with pytest.raises(ValueError, match="--parallel True"):
        R.parse_args(["--parallel", "True", "--embedSize", "128"])
    with pytest.raises(ValueError, match="64 and 128"):
        R.parse_args(["--embedSize", "96"])
    assert not dist.is_initialized()
    assert R.parse_args(["--embedSize", "128"]).embedSize == 128


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _cuda_graph(u, i, U, I):
    from ngacf_b200.graph import BipartiteGraph
    return BipartiteGraph(torch.from_numpy(np.stack([u, i]).astype(np.int64)).to(DEV), U, I)


def _long_graph():
    U, I, E = 400, 600, 30000
    u, i = port.synth_bipartite(U, I - 5, E, 6)
    g = port.build_graph(np.stack([u, i]), U, I)
    assert (np.diff(g.rowptr) > 128).any() and (np.diff(g.colptr) > 128).any() and (np.diff(g.colptr) == 0).any()
    return u, i, g


@gpu
def test_w_entry_points_at_64_equal_unsuffixed():
    """width 64 in every `_w` entry point gives the bits of the unsuffixed call"""
    from ngacf_b200 import _lib, ops
    from ngacf_b200.propagation import Propagation
    u, i, ref = _long_graph()
    g = _cuda_graph(u, i, ref.U, ref.I)
    N = g.N
    gen = torch.Generator(device=DEV).manual_seed(1)
    f32 = dict(dtype=torch.float32, device=DEV)
    p = init_params(ref.U, ref.I, 64, dtype=torch.float32)
    st = [[t.to(DEV).contiguous() for t in list(s["Wu"]) + list(s["Wi"]) + [s["a"][k:k + 1] for k in range(s["a"].shape[0])]] for s in p["stages"]]
    wt = [ops.pointer_table(s) for s in st]
    uE, iE = p["uEmbd"].to(DEV), p["iEmbd"].to(DEV)
    prop = Propagation(g)
    prop.set_dropout(0.2, 5, 1)
    fm = [torch.empty(N, dtype=torch.int64, device=DEV) for _ in range(2)]
    em = [torch.empty(max(g.E, 1), dtype=torch.uint8, device=DEV) for _ in range(2)]
    import ctypes
    fa = (ctypes.c_void_p * 2)(*[f.data_ptr() for f in fm])
    ea = (ctypes.c_void_p * 2)(*[e.data_ptr() for e in em])
    _lib.call("ngacf_dropout_masks_w", fa, ea, (ctypes.c_int32 * 2)(8, 1), (ctypes.c_int32 * 2)(64, 64), 2, N, g.E, 5, 1, None, 0.2, ops._s())
    for k in range(2):
        assert torch.equal(fm[k], prop.featmask[k]) and torch.equal(em[k][:g.E], prop.edgemask[k])
    for H, k in ((8, 0), (1, 1)):
        outs = []
        for name in ("ngacf_transform_fwd", "ngacf_transform_fwd_w"):
            h, s = torch.empty((N, 64), **f32), torch.empty((N, H), **f32)
            extra = (64, 64) if name.endswith("_w") else ()
            _lib.call(name, ops._p(uE), ops._p(iE), 0, ops._p(prop.featmask[k]), 1.25, ops._p(wt[k]), H, *extra, g.U, g.I, ops._p(h), ops._p(s), ops._s())
            outs.append((h, s))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
        h, s = outs[0]
        Zs, ns = [], []
        for w in (None, 64):
            Z, nrm = torch.empty((N, 64), **f32), torch.empty((N, H), **f32)
            if w is None:
                ops.aggregate_fwd(g, prop.scratch, prop.counter, h, s, H, prop.edgemask[k], 1.25, Z, nrm)
            else:
                _lib.call("ngacf_aggregate_fwd_w", ops._p(g.tasks), g.T, ops._p(g.adj_ptr), ops._p(g.adj_idx), ops._p(g.adj_eid),
                          ops._p(g.long_first_slot), ops._p(prop.counter), ops._p(prop.scratch), ops._p(h), ops._p(s), H, 64,
                          ops._p(prop.edgemask[k]), 1.25, ops._p(Z), ops._p(nrm), -1, ops._s())
            Zs.append(Z)
            ns.append(nrm)
        assert torch.equal(Zs[0], Zs[1]) and torch.equal(ns[0], ns[1])
        Z, nrm = Zs[0], ns[0]
        G = torch.randn((N, 64), generator=gen, **f32)
        res = []
        for w in (None, 64):
            Ghat, dN, dh, dS = torch.zeros((N, 64), **f32), torch.zeros((N, 8), **f32), torch.zeros((N, 64), **f32), torch.zeros((N, 8), **f32)
            ds = torch.zeros(g.E * 8, **f32)
            kw = {} if w is None else dict(width=64)
            if w is None:
                ops.stage_bwd_prep(G, Z, h, nrm, H, Ghat, dN)
            else:
                _lib.call("ngacf_stage_bwd_prep_w", ops._p(G), ops._p(Z), ops._p(h), ops._p(nrm), H, 64, N, ops._p(Ghat), ops._p(dN), ops._s())
            for mode in (0, 1):
                if w is None:
                    ops.stage_bwd_edges(mode, g, prop.scratch, prop.counter, G, Ghat, dN, h, s, H, prop.edgemask[k], 1.25, wt[k], ds, dh, dS)
                else:
                    t0, t1 = (0, g.T_users) if mode == 0 else (g.T_users, g.T)
                    _lib.call("ngacf_stage_bwd_edges_w", mode, ops._p(g.tasks), t0, t1, ops._p(g.adj_ptr), ops._p(g.adj_idx), ops._p(g.adj_eid),
                              ops._p(g.long_first_slot), ops._p(prop.counter), ops._p(prop.scratch), ops._p(G), ops._p(Ghat), ops._p(dN),
                              ops._p(h), ops._p(s), H, 64, ops._p(prop.edgemask[k]), 1.25, ops._p(wt[k]), g.U, ops._p(ds), ops._p(dh), ops._p(dS),
                              0, ops._s())
            grads = [torch.zeros_like(t) for t in st[k]]
            gt = ops.pointer_table(grads)
            dU, dI = torch.zeros_like(uE), torch.zeros_like(iE)
            nb = ops.transform_bwd_workspace_bytes(g.U, g.I)
            assert nb == int(_lib.load().ngacf_transform_bwd_workspace_bytes_w(64, 64, g.U, g.I))
            ws = torch.empty(nb // 4, **f32)
            if w is None:
                ops.transform_bwd(dh, dS, h, uE, iE, 0, prop.featmask[k], 1.25, wt[k], gt, H, g.U, g.I, dU, dI, 0, 0, ws)
            else:
                _lib.call("ngacf_transform_bwd_w", ops._p(dh), ops._p(dS), ops._p(h), ops._p(uE), ops._p(iE), 0, ops._p(prop.featmask[k]), 1.25,
                          ops._p(wt[k]), ops._p(gt), H, 64, 64, g.U, g.I, ops._p(dU), ops._p(dI), 0, 0, ops._p(ws), nb, ops._s())
            res.append([Ghat, dN, dh, dS, dU, dI] + grads)
        for a, b in zip(*res):
            assert torch.equal(a, b)
    # scores, features, exact top-K (both variants)
    from ngacf_b200.data import Interactions
    (tu, ti), (su, si) = port.split_train_test(u, i, ref.U, 2)
    dit = Interactions.from_arrays(ref.U, ref.I, tu, ti, su, si, device=DEV)
    Z = torch.randn((N, 64), generator=gen, **f32)
    users = torch.randint(0, g.U, (700,), generator=gen, device=DEV)
    items = torch.randint(0, g.I, (700,), generator=gen, device=DEV)
    a, b = torch.empty(700, **f32), torch.empty(700, **f32)
    ops.score_pairs(Z, g.U, users, items, a)
    _lib.call("ngacf_score_pairs_w", ops._p(Z), 64, g.U, ops._p(users), ops._p(items), 700, ops._p(b), ops._s())
    assert torch.equal(a, b)
    dsc = torch.randn(700, generator=gen, **f32)
    G1, G2 = torch.zeros_like(Z), torch.zeros_like(Z)
    ops.score_pairs_bwd(Z, g.U, users, items, dsc, G1)
    _lib.call("ngacf_score_pairs_bwd_w", ops._p(Z), 64, g.U, ops._p(users), ops._p(items), ops._p(dsc), 700, ops._p(G2), 0, ops._s())
    assert torch.equal(G1, G2)
    F1, F2 = torch.empty_like(Z), torch.empty_like(Z)
    ops.final_features(Z, F1)
    _lib.call("ngacf_final_features_w", ops._p(Z), N, 64, ops._p(F2), ops._s())
    assert torch.equal(F1, F2)
    ev_users = dit.eval_users
    n = ev_users.numel()
    for name, extra in (("ngacf_score_topk_exact", ()), ("ngacf_score_topk_exact_split", ())):
        ids = [torch.empty((n, 20), dtype=torch.int32, device=DEV) for _ in range(2)]
        scs = [torch.empty((n, 20), **f32) for _ in range(2)]
        ws = torch.empty(int(_lib.load().ngacf_score_topk_exact_split_workspace_bytes(g.I, n)), dtype=torch.uint8, device=DEV)
        wargs = (ops._p(ws), ws.numel()) if "split" in name else ()
        common = (g.U, g.I, ops._p(ev_users), n, ops._p(dit.train_ptr), ops._p(dit.train_items), ops._p(dit.in_pool))
        _lib.call(name, ops._p(F1), *common, ops._p(ids[0]), ops._p(scs[0]), *wargs, ops._s())
        _lib.call(name + "_w", ops._p(F1), 64, *common, ops._p(ids[1]), ops._p(scs[1]), *wargs, ops._s())
        assert torch.equal(ids[0], ids[1]) and torch.equal(scs[0], scs[1])


@gpu
def test_unbuilt_shapes_return_unsupported():
    from ngacf_b200 import _lib
    lib = _lib.load()
    assert lib.ngacf_transform_fwd_w(None, None, 0, None, 1.0, None, 8, 64, 128, 1, 1, None, None, None) == -4
    assert b"not built" in lib.ngacf_last_error()
    assert lib.ngacf_score_pairs_w(None, 96, 1, None, None, 1, None, None) == -4
    assert lib.ngacf_aggregate_fwd_w(None, 1, None, None, None, None, None, None, None, None, 8, 128, None, 1.0, None, None, -1, None) == -4


@gpu
def test_masks_at_128_bit_exact():
    from ngacf_b200.propagation import Propagation
    u, i, ref = small_graph()
    g = _cuda_graph(u, i, ref.U, ref.I)
    for multi in (False, True):
        prop = Propagation(g, stages_of(128, multi))
        prop.set_dropout(0.3, 0xABCDEF0123, 9)
        feat, edge, _ = port_keeps(ref, 0xABCDEF0123, 9, 0.3, 128, multi)
        for k in range(len(feat)):
            assert np.array_equal(prop.featmask[k].cpu().numpy().view(np.uint64), feat[k]), k
            assert np.array_equal(prop.edgemask[k].cpu().numpy(), edge[k]), k


@gpu
@pytest.mark.parametrize("H,d_in,d_out", [(8, 128, 64), (1, 64, 128)])
def test_dense_transforms_at_128_vs_fp64(H, d_in, d_out):
    from ngacf_b200 import ops
    U, I = 700, 900
    gen = torch.Generator().manual_seed(H)
    DH = d_out // H
    Wu, Wi = torch.randn(H, d_in, DH, generator=gen) * 0.2, torch.randn(H, d_in, DH, generator=gen) * 0.2
    a = torch.randn(H, 2 * DH, generator=gen) * 0.3
    X = torch.randn(U + I, d_in, generator=gen)
    keep = torch.from_numpy(unpack_feature_mask(feature_mask_bits(U + I, 3, 1, 0, 0.25, d_in), d_in))
    mask = torch.from_numpy(feature_mask_bits(U + I, 3, 1, 0, 0.25, d_in).view(np.int64)).to(DEV)
    tabs = [t.contiguous().to(DEV) for t in list(Wu) + list(Wi) + [a[k:k + 1] for k in range(H)]]
    wt = ops.pointer_table(tabs)
    Xd = X.to(DEV)
    scale = 1 / 0.75
    for elu in (0, 1):
        h = torch.empty(U + I, d_out, device=DEV)
        s = torch.empty(U + I, H, device=DEV)
        ops.transform_fwd(Xd[:U], Xd[U:], elu, mask, scale, wt, H, U, I, h, s, d_in=d_in, d_out=d_out)
        X64 = X.double()
        Xa = port._elu(X64) if elu else X64
        Xk = Xa * keep * scale
        st = dict(Wu=Wu.double(), Wi=Wi.double(), a=a.double())
        href = torch.cat([Xk[:U] @ port._wcat(st["Wu"]), Xk[U:] @ port._wcat(st["Wi"])], 0)
        sref = torch.cat([(href[:U].view(U, H, DH) * st["a"][:, :DH]).sum(-1), (href[U:].view(I, H, DH) * st["a"][:, DH:]).sum(-1)], 0)
        assert rel_err(h.cpu(), href) < 1e-6
        assert rel_err(s.cpu(), sref) < 1e-6
        # backward: dX (mask, ELU'), dW, da against fp64
        dh = torch.randn(U + I, d_out, generator=gen)
        dS = torch.randn(U + I, H, generator=gen)
        grads = [torch.zeros_like(t) for t in tabs]
        gt = ops.pointer_table(grads)
        dX = torch.zeros(U + I, d_in, device=DEV)
        ws = torch.empty(ops.transform_bwd_workspace_bytes(U, I, d_in, d_out) // 4, device=DEV)
        ops.transform_bwd(dh.to(DEV), dS.to(DEV), h, Xd[:U], Xd[U:], elu, mask, scale, wt, gt, H, U, I, dX[:U], dX[U:], 0, 0, ws,
                          d_in=d_in, d_out=d_out)
        dh64, dS64 = dh.double(), dS.double()
        dXref = torch.cat([dh64[:U] @ port._wcat(st["Wu"]).t(), dh64[U:] @ port._wcat(st["Wi"]).t()], 0) * keep * scale
        if elu:
            dXref = dXref * port._elu_grad(X64)
        assert rel_err(dX.cpu(), dXref) < 1e-6
        dWu = (Xk[:U].t() @ dh64[:U]).view(d_in, H, DH).permute(1, 0, 2)
        hv = href.view(U + I, H, DH)
        da_u = (dS64[:U, :, None] * hv[:U]).sum(0)
        assert rel_err(torch.stack(grads[:H]).cpu(), dWu) < 1e-6
        assert rel_err(torch.cat(grads[2 * H:], 0)[:, :DH].cpu(), da_u) < 1e-6


def _model_vs_port(cls, multi, droprate):
    u, i, ref = _long_graph()
    U, I = ref.U, ref.I
    p64 = init_params(U, I, 128, multi=multi)
    model = cls(U, I, 128, [64, 64], droprate)
    model.load_state_dict({k: v.float() for k, v in port.state_dict_from_params(p64).items()})
    model = model.to(DEV).train()
    model.drop_seed, model._call = 99, 3
    keeps = port_keeps(ref, 99, 3, droprate, 128, multi)[2] if droprate > 0 else None
    F, caches = propagate(p64, ref, keeps, droprate)
    rng = np.random.default_rng(0)
    users, items, w = rng.integers(0, U, 512), rng.integers(0, I, 512), rng.standard_normal(512)
    sc_ref = port.scores(F, U, users, items)
    ut, itt, wt = torch.from_numpy(users), torch.from_numpy(items) + U, torch.from_numpy(w)
    dF = torch.zeros_like(F)
    dF.index_add_(0, ut, wt[:, None] * F[itt])
    dF.index_add_(0, itt, wt[:, None] * F[ut])
    gref = port.state_dict_from_params(propagate_backward(dF, p64, ref, caches))
    adj = torch.from_numpy(np.stack([u, i])).to(DEV)
    sc = model(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), adj)
    assert rel_err(sc.detach().cpu().numpy(), sc_ref.numpy()) < 1e-4
    model._call = 3                                  # the same dropout stream as the scored call
    Zl = model.propagate(adj)
    assert rel_err(port._elu(Zl.detach().double().cpu()), F) < 1e-4
    (sc * wt.float().to(DEV)).sum().backward()
    for k, v in model.named_parameters():
        assert v.grad.shape == v.shape
        assert rel_err(v.grad.cpu().numpy(), gref[k].numpy()) < 1e-4, k
    model._call = 3
    sc2 = model(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), adj)
    assert torch.equal(sc, sc2)


@gpu
@pytest.mark.parametrize("multi", [False, True])
@pytest.mark.parametrize("droprate", [0.0, 0.25])
def test_models_at_128_forward_backward_vs_port(multi, droprate):
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    _model_vs_port(SPUIMultiGACF if multi else SPUIGACF, multi, droprate)


@gpu
def test_scores_topk_and_allneg_at_128():
    from ngacf_b200 import _lib, ops
    from ngacf_b200.data import Interactions
    from ngacf_b200.evaluate import AllNegEvaluator
    U, I, E = 300, 1000, 9000
    u, i = port.synth_bipartite(U, I, E, 2)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 3)
    it = port.build_interactions(U, I, tu, ti, su, si)
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    rng = np.random.default_rng(1)
    Z = rng.standard_normal((U + I, 128)).astype(np.float32) * 0.5
    src, dst = rng.integers(0, I, 100), rng.integers(0, I, 100)
    Z[U + dst] = Z[U + src]                      # ties: the lowest id wins
    Zt = torch.from_numpy(Z).to(DEV)
    F = torch.empty_like(Zt)
    ops.final_features(Zt, F)
    Fn = F.cpu().numpy()
    assert np.array_equal(Fn, port._elu(torch.from_numpy(Z).double()).float().numpy()) or rel_err(Fn, port._elu(torch.from_numpy(Z).double())) < 1e-6
    users = torch.from_numpy(rng.integers(0, U, 4000)).to(DEV)
    items = torch.from_numpy(rng.integers(0, I, 4000)).to(DEV)
    sc = torch.empty(4000, device=DEV)
    ops.score_pairs(Zt, U, users, items, sc)
    ref = port.dot64_tree(Fn[users.cpu().numpy()], Fn[U + items.cpu().numpy()])
    assert np.array_equal(sc.cpu().numpy(), ref)
    ev = AllNegEvaluator(dit, "auto")
    ev.rank(Zt)
    res = ev.metrics()
    pres, ptop, _ = port.eval_neg_all(Fn, it)
    assert np.array_equal(ev.top_ids.cpu().numpy().astype(np.int64), ptop)
    for k in ("precision", "recall", "ndcg", "hit_ratio"):
        assert np.allclose(res[k], pres[k], rtol=1e-9, atol=1e-12), k
    ids2 = torch.empty_like(ev.top_ids)
    sc2 = torch.empty((ids2.shape[0], 20), device=DEV)
    ops.score_topk_exact_split(F, U, I, dit.eval_users, dit, ids2, sc2)
    assert torch.equal(ids2, ev.top_ids)
    with pytest.raises(_lib.NgacfError, match="64-wide"):
        AllNegEvaluator(dit, "tc").rank(Zt)


def _trainer_setup(kind, droprate=0.2):
    from ngacf_b200.data import Interactions
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.optim import FusedAdam
    U, I, E = 300, 500, 8000
    u, i = port.synth_bipartite(U, I, E, 7)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 8)
    torch.manual_seed(1)
    model = SPUIGACF(U, I, 128, [64, 64], droprate).to(DEV)
    model.drop_seed = 55
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    adj = torch.from_numpy(np.stack([np.concatenate([tu, su]), np.concatenate([ti, si])]))
    optim = FusedAdam(model.parameters(), lr=0.005, weight_decay=1e-6)
    return model, dit, adj, optim, (U, I, tu, ti, su, si)


@gpu
def test_fused_trainer_at_128_equals_eager():
    import train_eval_Gowalla as T
    from ngacf_b200.loss import BPRLoss
    from ngacf_b200.optim import FusedAdam
    runs = []
    for fused in (True, False):
        model, dit, adj, optim, _ = _trainer_setup("pair")
        losses = [T.train_bpr(model, 256, dit, dit, adj, optim, BPRLoss(), False, epoch=ep, sample_seed=3, fused=fused) for ep in range(2)]
        runs.append((np.array(losses), {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}))
    assert rel_err(runs[0][0], runs[1][0]) < 1e-4
    for k in runs[0][1]:
        assert rel_err(runs[0][1][k], runs[1][1][k]) < 5e-3, k
    # captured steps replayed twice from the same state are bit-identical; the full output stage runs at 128
    from ngacf_b200.train import FusedTrainer
    outs = []
    for _ in range(2):
        model, dit, adj, optim, _ = _trainer_setup("pair")
        tr = FusedTrainer(model, dit, model.graph_for(adj.to(DEV)), 256, optim, sample_seed=3)
        assert not tr.prune_last_stage
        tr.run_steps(3)
        torch.cuda.synchronize()
        outs.append([p.detach().clone() for p in model.parameters()])
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    model, dit, adj, _, _ = _trainer_setup("pair")
    with pytest.raises(NotImplementedError):
        FusedTrainer(model, dit, model.graph_for(adj.to(DEV)), 256, FusedAdam(model.parameters()), sample_seed=3, split_dense_backward=True)


@gpu
def test_negsampling_and_sampled_eval_at_128():
    import train_eval_Gowalla as T
    from ngacf_b200.negsampling import SampledNegEvaluator
    runs = []
    for fused in (True, False):
        model, dit, adj, optim, _ = _trainer_setup("neg")
        lossfn = torch.nn.BCEWithLogitsLoss()
        kw = {} if fused else dict(fused=False)
        losses = [T.train_neg_sample(model, 256, dit, dit, adj, optim, lossfn, False, epoch=ep, sample_seed=3, **kw) for ep in range(2)]
        runs.append((np.array(losses), {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}))
    assert rel_err(runs[0][0], runs[1][0]) < 1e-4
    for k in runs[0][1]:
        assert rel_err(runs[0][1][k], runs[1][1][k]) < 5e-3, k
    model.eval()
    Z = model.propagate(adj.to(DEV))
    ev = SampledNegEvaluator(dit, top_k=10, K=99, seed=4)
    hr, ndcg = ev(Z)
    # the same sampled rows ranked on the CPU from the GPU features
    F = port._elu(Z.detach().double().cpu()).float().numpy()
    pu, pi = ev.pu.cpu().numpy(), ev.pi.cpu().numpy()
    sc = port.dot64_tree(F[pu], F[model.userNum + pi]).reshape(-1, 100)
    rank = (sc[:, 1:] > sc[:, :1]).sum(1)
    assert abs(hr - float((rank < 10).mean())) < 1e-12
    assert abs(ndcg - float(np.where(rank < 10, 1.0 / np.log2(rank + 2), 0.0).mean())) < 1e-9


@gpu
def test_cli_at_128(tmp_path, monkeypatch, capsys):
    import run_Gowalla as R
    monkeypatch.chdir(tmp_path)
    base = ["--dataset", "synth-tiny", "--embedSize", "128", "--lr", "0.002", "--droprate", "0.2", "--batch_size", "2048",
            "--eval_every", "1", "--save_every", "1", "--parallel", "False"]

    def run(extra):
        args = R.parse_args(base + extra)
        torch.manual_seed(args.seed)
        torch.cuda.manual_seed_all(args.seed)
        np.random.seed(args.seed)
        R.main(args)
        return capsys.readouterr().out
    for model in ("SPUIGACF", "SPUIMultiGACF"):
        out = run(["--model", model, "--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--epochs", "2"])
        assert "------epoch:1, train_loss:" in out and "metrics:" in out
        ck = torch.load(tmp_path / "ckpts" / ("%s_synth-tiny_002.pkl" % model), map_location="cpu", weights_only=False)
        assert tuple(ck["model"]["uEmbd.weight"].shape)[1] == 128 and tuple(ck["model"]["gat.out_att.W_u"].shape) == (64, 128)
    out = run(["--model", "SPUIGACF", "--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--epochs", "3", "--resume_from", "2"])
    assert "=> loaded checkpoint" in out and "------epoch:2, train_loss:" in out
    out = run(["--model", "SPUIGACF", "--train_mode", "NegSampling", "--eval_mode", "SampledNeg", "--epochs", "1"])
    assert "------epoch:0, train_loss:" in out


@gpu
@pytest.mark.parametrize("H,d_in,d_out", [(8, 64, 64), (8, 128, 64), (1, 64, 128)])
def test_transform_bwd_stays_inside_reported_workspace(H, d_in, d_out):
    """ngacf_transform_bwd(_w) writes nothing past ngacf_transform_bwd_workspace_bytes(_w) of its shape: the workspace is allocated
    at the reported size followed by a canary tail, and the tail is checked after the call"""
    from ngacf_b200 import ops
    U, I = 3000, 5000                    # enough row tiles that every resident block of the grid writes a partial
    gen = torch.Generator().manual_seed(d_out)
    DH = d_out // H
    tabs = [(torch.randn(d_in, DH, generator=gen) * 0.2).to(DEV) for _ in range(2 * H)] + \
        [(torch.randn(1, 2 * DH, generator=gen) * 0.2).to(DEV) for _ in range(H)]
    grads = [torch.zeros_like(t) for t in tabs]
    wt, gt = ops.pointer_table(tabs), ops.pointer_table(grads)
    X = torch.randn(U + I, d_in, generator=gen).to(DEV)
    h = torch.randn(U + I, d_out, generator=gen).to(DEV)
    dh = torch.randn(U + I, d_out, generator=gen).to(DEV)
    dS = torch.randn(U + I, H, generator=gen).to(DEV)
    dX = torch.zeros(U + I, d_in, device=DEV)
    nb = ops.transform_bwd_workspace_bytes(U, I, d_in, d_out)
    assert nb > 0 and nb % 4 == 0
    canary = 1 << 16
    buf = torch.full((nb // 4 + canary,), 1234.5, device=DEV)
    ws = buf[:nb // 4]
    ops.transform_bwd(dh, dS, h, X[:U], X[U:], 0, None, 1.0, wt, gt, H, U, I, dX[:U], dX[U:], 0, 0, ws, d_in=d_in, d_out=d_out)
    torch.cuda.synchronize()
    assert bool((buf[nb // 4:] == 1234.5).all()), "transform_bwd wrote past its reported workspace"
    assert bool((ws != 1234.5).any())
