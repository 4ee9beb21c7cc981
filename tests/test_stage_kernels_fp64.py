"""The stage gather kernels element by element against float64 references, on a graph built around the chunk boundaries.

Every kernel is compared with the same operation written in float64 (a few lines of ``index_add_``) from the fp32 inputs the
kernel receives (h, s, the unpacked edge masks, scale, G, the attention vectors a, and Ghat / dN / Z / norm where the kernel reads
them).  The references are pinned to ``oracle.port`` (stage_forward / stage_backward, spgat_stage_forward / spgat_stage_backward)
and to the Laplacian of ``ngacf_b200.gp`` on the CPU, so they compute the operations the port specifies.

Per-element bound.  Every output element must satisfy

    |gpu - ref| <= u * (c * M + Mx) + TINY,        u = 2^-24,

with M the reference evaluated on absolute values (the sums of |terms| of the running-error analysis) and Mx the same sums
weighted by each term's own relative error, in units of u, where a term carries more than one rounding:

  * the edge weight: the kernels evaluate e = __expf(-l), l = LeakyReLU(fl(s_n + s_m)) with the fp32 constant 0.2f.  The CUDA C
    Programming Guide bounds __expf(y) by 2 + floor(1.173 |y|) ulp, i.e. (4 + 2.346 |l|) u relative; the rounding of the logit sum,
    of 0.2f * x and the difference 0.2f - 0.2 add 2.25 |l| u.  So a weight carries EXP_ERR = 4 + 4.6 |l| units, explicitly per
    edge (one more with the dropout product w * scale);
  * a summed scalar of a row of degree d is formed in at most depth(d) = min(d, 128) + slots(d) dependent additions: one
    CHUNK = 128-edge task accumulates at most 128 terms (fma chains, lane trees or the eight 16-edge groups of the CTA kernels, all
    of them no deeper than the number of terms), and a row longer than a chunk adds its slots(d) = ceil(d / 128) partial sums;
  * a per-head dot product (det, dN, the node logits) has at most DOT = 20 roundings: 16 products of a 128-wide lane slice in
    sequence and a 4-level lane tree (the 64-wide and 8-head forms are shallower);
  * the division by norm is 1 / rs, correctly rounded, followed by a product: 2 roundings on top of the relative error of rs.

From these, Z = h + acc / norm gets c = 2 depth + 2 (acc and rs each contribute depth, the reciprocal, the product and the final
fma one each), norm gets c = depth, dN gets c = DOT + 4 (the difference Z - h, the product, the dot, the reciprocal and the
product), Ghat c = 2, d s_e propagates the bound of de plus three roundings, and the row sums of d s_e and of e~ Ghat add
depth.  Multi-GPU partial rows add one addition per rank to depth.  c is derived, not fitted: the measured error / bound ratios are
printed by every GPU test (RATIO lines) and appear in its failure message.

The CPU tests show that each bound bites: the fp64 reference after a single wrong term (an edge left out of a degree-1 row, the last
slot of a 257-edge row dropped, an edge-mask bit flipped, two heads of dS swapped, norm taken after the mask, the keep * scale
factor left out of one d s_e) fails it, while several of those wrong results pass the max-normalised ``rel_err < 1e-4``.
"""
from __future__ import annotations

import functools
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
gpu = pytest.mark.gpu

u = 2.0 ** -24
TINY = 1e-38                  # subnormal results: the kernels keep denormals, each rounding there is below 2^-149
ALPHA = port.ALPHA
CHUNK = 128
DOT = 20
DEGREES = (1, 2, 15, 16, 17, 127, 128, 129, 255, 256, 257, 1000)
N_EMPTY = 5                   # items without an edge (the NaN -> 0 path); they are the last N_EMPTY item ids
DROP = 0.2
SCALE = 1.0 / (1.0 - DROP)    # 1.25, exact in fp32
f64 = torch.float64


# ------------------------------------------------------------------------------------------------
# the boundary graph
# ------------------------------------------------------------------------------------------------
def depth_of(deg):
    deg = np.asarray(deg, np.int64)
    slots = np.where(deg > CHUNK, -(-deg // CHUNK), 0)
    return torch.from_numpy((np.minimum(deg, CHUNK) + slots).astype(np.float64))


@functools.lru_cache(maxsize=None)
def boundary():
    """power-law base graph + one user and one item of every degree in DEGREES (their edges go to base rows only, so the degrees
    are exact on both sides) + N_EMPTY isolated items; U = 1112 and I = 1318 are multiples of neither 16 nor 128"""
    rng = np.random.default_rng(2026)
    nd = len(DEGREES)
    U0, I0 = 1100, 1301
    U, I = U0 + nd, I0 + nd + N_EMPTY
    bu, bi = port.synth_bipartite(U0, I0, 20000, seed=4)
    lone = np.setdiff1d(np.arange(I0), bi)             # base items the power law left without an edge get one
    bu, bi = np.concatenate([bu, rng.choice(U0, lone.shape[0])]), np.concatenate([bi, lone])
    pu, pi = rng.permutation(U), rng.permutation(I - N_EMPTY)
    ou, su = pu[:U0], pu[U0:]
    oi, si = pi[:I0], pi[I0:]
    us, its = [ou[bu]], [oi[bi]]
    for k, d in enumerate(DEGREES):
        us += [np.full(d, su[k]), rng.choice(ou, d, replace=False)]
        its += [rng.choice(oi, d, replace=False), np.full(d, si[k])]
    uu, ii = np.concatenate(us), np.concatenate(its)
    g = port.build_graph(np.stack([uu, ii]), U, I)
    deg = np.concatenate([np.diff(g.rowptr), np.diff(g.colptr)])
    eu = torch.from_numpy(g.eu)
    ei = torch.from_numpy(g.ei) + U
    return SimpleNamespace(U=U, I=I, N=U + I, E=g.E, g=g, u=uu, i=ii, eu=eu, ei=ei, deg=deg, depth=depth_of(deg),
                           spec_u={d: int(su[k]) for k, d in enumerate(DEGREES)}, spec_i={d: int(U + si[k]) for k, d in enumerate(DEGREES)})


def rows_scaled(N, W, gen, lo, hi):
    """rows of N(0,1) entries scaled by a log-uniform factor in [lo, hi]: magnitudes differ by orders between rows"""
    x = torch.randn((N, W), generator=gen, dtype=f64)
    sc = torch.empty((N, 1), dtype=f64).uniform_(np.log(lo), np.log(hi), generator=gen).exp()
    return (x * sc).float()


def stage_inputs(N, H, W, seed):
    gen = torch.Generator().manual_seed(seed)
    return SimpleNamespace(h=rows_scaled(N, W, gen, 1e-2, 1.0), s=(torch.randn((N, H), generator=gen, dtype=f64) * 1.5).float(),
                           G=rows_scaled(N, W, gen, 1e-3, 1.0), a=(torch.randn((H, 2 * W // H), generator=gen, dtype=f64) * 0.5).float())


def edge_keep(E, H, drop, stage=0):
    """Philox edge masks of the port (uint8 bits in CSR edge order) and the unpacked keep decisions, or (None, None)"""
    if drop == 0:
        return None, None
    bits = port.edge_mask_bits(E, H, 5, 3, stage, drop)
    return bits, torch.from_numpy(port.unpack_edge_mask(bits, H))


# ------------------------------------------------------------------------------------------------
# float64 references (inputs: the fp32 tensors the kernels read)
# ------------------------------------------------------------------------------------------------
def weights(x):
    """e = exp(-LeakyReLU(x)) and its relative error in units of u (EXP_ERR of the module docstring)"""
    l = torch.where(x > 0, x, ALPHA * x)
    return torch.exp(-l), 4.0 + 4.6 * l.abs()


def ref_aggregate(h, x, H, keep, scale, r, m, N, depth, residual=True):
    """Z[n] = (h[n] if residual) + sum_{(n,m)} drop(e) h[m] / sum e over the directed pairs (r, m) with logits x (one row per r),
    the raw sums acc / norm and the bounds of all three"""
    h = h.double()
    W = h.shape[1]
    DH = W // H
    e, ee = weights(x)
    wd, eed = (e, ee) if keep is None else (e * keep * scale, ee + 1)
    hv = h.view(N, H, DH)
    norm, normX = torch.zeros((N, H), dtype=f64), torch.zeros((N, H), dtype=f64)
    acc, accM, accX = (torch.zeros((N, H, DH), dtype=f64) for _ in range(3))
    t = wd[:, :, None] * hv[m]
    norm.index_add_(0, r, e)
    normX.index_add_(0, r, ee * e)
    acc.index_add_(0, r, t)
    accM.index_add_(0, r, t.abs())
    accX.index_add_(0, r, eed[:, :, None] * t.abs())
    inv = torch.where(norm > 0, 1.0 / norm, torch.zeros_like(norm))[:, :, None]
    d = depth.view(N, 1, 1)
    base = hv if residual else torch.zeros_like(hv)
    M = base.abs() + accM * inv
    Mx = (accX + accM * normX[:, :, None] * inv) * inv
    return dict(Z=(base + acc * inv).reshape(N, W), Z_bound=(u * ((2 * d + 2) * M + Mx) + TINY).reshape(N, W),
                norm=norm, norm_bound=u * (depth.view(N, 1) * norm + normX) + TINY,
                acc=acc.reshape(N, W), acc_bound=(u * (d * accM + accX) + TINY).reshape(N, W))


def bip_pairs(eu, ei):
    """directed pairs of the unified adjacency: user rows (CSR order), then item rows (users ascending, the CSC order)"""
    return torch.cat([eu, ei]), torch.cat([ei, eu])


def ref_stage_fwd(h, s, H, keep, scale, eu, ei, N, depth):
    s = s.double()
    x = s[eu] + s[ei]
    r, m = bip_pairs(eu, ei)
    k2 = None if keep is None else torch.cat([keep, keep]).double()
    return ref_aggregate(h, torch.cat([x, x]), H, k2, scale, r, m, N, depth)


def ref_prep(G, Z, h, norm, H):
    N, W = G.shape
    DH = W // H
    G, Z, h, norm = (t.double() for t in (G, Z, h, norm))
    inv = torch.where(norm != 0, 1.0 / norm, torch.zeros_like(norm))
    Gv = G.view(N, H, DH)
    t = Gv * (Z - h).view(N, H, DH)
    Ghat = Gv * inv[:, :, None]
    return dict(Ghat=Ghat.reshape(N, W), Ghat_bound=(2 * u * Ghat.abs() + TINY).reshape(N, W),
                dN=-t.sum(-1) * inv, dN_bound=u * (DOT + 4) * t.abs().sum(-1) * inv + TINY)


def ref_stage_bwd(G, Ghat, dN, h, s, a, H, keep, scale, eu, ei, U, N, depth):
    """the edge passes of the bipartite stage backward (csrc/propagate_bwd.cu header): per undirected edge d s and e~, per row the
    raw sums acc = sum e~ Ghat[m] and dS = sum d s, and dh = G + acc + dS (x) a_side"""
    G, Ghat, dN, h, s, a = (t.double() for t in (G, Ghat, dN, h, s, a))
    W = h.shape[1]
    DH = W // H
    x = s[eu] + s[ei]
    e, ee = weights(x)
    ksc = torch.ones_like(e) if keep is None else keep.double() * scale
    et = e * ksc
    Gh, hv, Gv = Ghat.view(N, H, DH), h.view(N, H, DH), G.view(N, H, DH)
    t1, t2 = Gh[eu] * hv[ei], Gh[ei] * hv[eu]
    det = (t1 + t2).sum(-1)
    detM = (t1.abs() + t2.abs()).sum(-1)
    dsum = dN[eu] + dN[ei]
    de = det * ksc + dsum
    deB = u * (DOT * detM * ksc + dsum.abs() + de.abs())
    slope = torch.where(x > 0, torch.ones_like(x), torch.full_like(x, ALPHA))
    ds = -de * e * slope
    dsB = (deB + de.abs() * u * (ee + 3)) * e * slope + TINY
    acc, accM, accX = (torch.zeros((N, H, DH), dtype=f64) for _ in range(3))
    dS, dSM, dSB = (torch.zeros((N, H), dtype=f64) for _ in range(3))
    for r, m in ((eu, ei), (ei, eu)):
        tt = et[:, :, None] * Gh[m]
        acc.index_add_(0, r, tt)
        accM.index_add_(0, r, tt.abs())
        accX.index_add_(0, r, (ee + 1)[:, :, None] * tt.abs())
        dS.index_add_(0, r, ds)
        dSM.index_add_(0, r, ds.abs())
        dSB.index_add_(0, r, dsB)
    d = depth.view(N, 1)
    accB = u * (d[:, :, None] * accM + accX)
    dSB = dSB + u * d * dSM
    side = torch.cat([a[:, :DH].expand(U, H, DH), a[:, DH:].expand(N - U, H, DH)])
    dh = Gv + acc + dS[:, :, None] * side
    dhB = accB + dSB[:, :, None] * side.abs() + 3 * u * (Gv.abs() + accM + dSM[:, :, None] * side.abs()) + TINY
    return dict(ds=ds, ds_bound=dsB, et=et, et_bound=u * (ee + 1) * et + TINY, x=x, e=e, det=det, dsum=dsum, ksc=ksc,
                acc=acc.reshape(N, W), acc_bound=(accB + TINY).reshape(N, W), dS=dS, dS_bound=dSB + TINY,
                dh=dh.reshape(N, W), dh_bound=dhB.reshape(N, W))


def ref_spmm(X, val, diag, eu, ei, N, depth):
    """Y = diag (.) X + sum val[e] X[m] over the unified adjacency (csrc/laplacian.cu)"""
    X, val, diag = X.double(), val.double(), diag.double()
    r, m = bip_pairs(eu, ei)
    t = torch.cat([val, val])[:, None] * X[m]
    Y = diag[:, None] * X
    YM = Y.abs().clone()
    Y.index_add_(0, r, t)
    YM.index_add_(0, r, t.abs())
    return Y, u * (depth.view(N, 1) + 1) * YM + TINY


def ref_spgat_bwd(G, Z, norm, h, p, q, a, H, keep, scale, r, c, N, depth):
    """SpGAT backward (csrc/spgat.cu header) over the directed edges (r -> c): Ghat, the per-edge (d s, e~) pairs, dP (row sums),
    dQ (column sums) and dh = sum_in e~ Ghat[n] + dP a_src + dQ a_dst"""
    G, Z, norm, h, p, q, a = (t.double() for t in (G, Z, norm, h, p, q, a))
    W = h.shape[1]
    DH = W // H
    Gv, Zv, hv = G.view(N, H, DH), Z.view(N, H, DH), h.view(N, H, DH)
    inv = torch.where(norm != 0, 1.0 / norm, torch.zeros_like(norm))
    Ghat = Gv * inv[:, :, None]
    tz = Gv * Zv
    dN = -tz.sum(-1) * inv
    dNB = u * (DOT + 2) * tz.abs().sum(-1) * inv
    x = p[r] + q[c]
    e, ee = weights(x)
    ksc = torch.ones_like(e) if keep is None else keep.double() * scale
    t = Ghat[r] * hv[c]
    det = t.sum(-1)
    de = det * ksc + dN[r]
    deB = u * (DOT + 2) * t.abs().sum(-1) * ksc + dNB[r] + u * de.abs()
    slope = torch.where(x > 0, torch.ones_like(x), torch.full_like(x, ALPHA))
    ds = -de * e * slope
    dsB = (deB + de.abs() * u * (ee + 3)) * e * slope + TINY
    et = e * ksc
    d = depth.view(N, 1)
    sums = {}
    for name, idx in (("dP", r), ("dQ", c)):
        v, vM, vB = (torch.zeros((N, H), dtype=f64) for _ in range(3))
        v.index_add_(0, idx, ds)
        vM.index_add_(0, idx, ds.abs())
        vB.index_add_(0, idx, dsB)
        sums[name] = (v, vM, vB + u * d * vM + TINY)
    acc, accM, accX = (torch.zeros((N, H, DH), dtype=f64) for _ in range(3))
    tt = et[:, :, None] * Ghat[r]
    acc.index_add_(0, c, tt)
    accM.index_add_(0, c, tt.abs())
    accX.index_add_(0, c, (ee + 3)[:, :, None] * tt.abs())
    (dP, dPM, dPB), (dQ, dQM, dQB) = sums["dP"], sums["dQ"]
    a_src, a_dst = a[None, :, :DH], a[None, :, DH:]
    dh = acc + dP[:, :, None] * a_src + dQ[:, :, None] * a_dst
    dhB = (u * (d[:, :, None] * accM + accX) + dPB[:, :, None] * a_src.abs() + dQB[:, :, None] * a_dst.abs()
           + 3 * u * (accM + dPM[:, :, None] * a_src.abs() + dQM[:, :, None] * a_dst.abs()) + TINY)
    return dict(Ghat=Ghat.reshape(N, W), Ghat_bound=(2 * u * Ghat.abs() + TINY).reshape(N, W), ds=ds, ds_bound=dsB, et=et,
                et_bound=u * (ee + 1) * et + TINY, dP=dP, dP_bound=dPB, dQ=dQ, dQ_bound=dQB, dh=dh.reshape(N, W), dh_bound=dhB.reshape(N, W))


def node_logits_ref(h, a, H):
    N, W = h.shape
    DH = W // H
    hv, a = h.double().view(N, H, DH), a.double()
    tp, tq = hv * a[None, :, :DH], hv * a[None, :, DH:]
    return tp.sum(-1), u * DOT * tp.abs().sum(-1) + TINY, tq.sum(-1), u * DOT * tq.abs().sum(-1) + TINY


def laplacian_values(bg, L):
    """LaplacianOp's {value per CSR edge, diagonal} of an (N,N) Laplacian, on the host: diag32 as LaplacianOp forms it in fp32,
    diag64 the exact 1 + L[n,n]"""
    L = L.coalesce()
    r, c = L.indices()
    v = L.values().to(torch.float32)
    on = r == c
    diag32 = torch.ones(bg.N, dtype=torch.float32).index_add_(0, r[on], v[on])
    diag64 = torch.ones(bg.N, dtype=f64).index_add_(0, r[on], v[on].double())
    up = (r < bg.U) & (c >= bg.U)
    keys = torch.from_numpy(bg.g.eu * bg.I + bg.g.ei)
    val = torch.zeros(bg.E, dtype=torch.float32)
    val[torch.searchsorted(keys, r[up] * bg.I + (c[up] - bg.U))] = v[up]
    return val, diag32, diag64


def rel_err(a, b):
    return float((a - b).abs().max() / b.abs().max())


def violations(got, ref, bound):
    return ~((got.double() - ref).abs() <= bound)


# ------------------------------------------------------------------------------------------------
# CPU: the graph covers the boundaries; the references are the port's operations; the bounds bite
# ------------------------------------------------------------------------------------------------
def test_boundary_graph_covers_every_degree():
    bg = boundary()
    du, di = np.diff(bg.g.rowptr), np.diff(bg.g.colptr)
    for d in DEGREES:
        assert (du == d).any() and (di == d).any(), d
        assert du[bg.spec_u[d]] == d and di[bg.spec_i[d] - bg.U] == d
    assert (di == 0).sum() == N_EMPTY and (di[-N_EMPTY:] == 0).all() and (du > 0).all()
    for n in (bg.U, bg.I, bg.I - N_EMPTY):
        assert n % 16 and n % 128
    assert 10_000 < bg.E < 60_000
    # every long-row shape: 2, 3 and 8 slots
    assert {2, 3, 8} <= set((-(-bg.deg[bg.deg > CHUNK] // CHUNK)).tolist())


@pytest.mark.parametrize("drop", [0.0, DROP])
@pytest.mark.parametrize("k", [0, 1])
def test_bipartite_references_equal_port(k, drop):
    """ref_stage_fwd / ref_prep / ref_stage_bwd compute port.stage_forward / stage_backward: Z and norm directly, dh and dS through
    the parameter and input gradients the port returns"""
    bg = boundary()
    g, U, N = bg.g, bg.U, bg.N
    p = port.init_params(U, bg.I, 11, dtype=f64)
    st = p["stages"][k]
    H, _, DH = st["Wu"].shape
    gen = torch.Generator().manual_seed(k)
    X = torch.randn((N, 64), generator=gen, dtype=f64)
    fk = ek = None
    if drop:
        fk = torch.from_numpy(port.unpack_feature_mask(port.feature_mask_bits(N, 5, 3, k, drop)))
        ek = edge_keep(bg.E, H, drop, k)[1]
    c = port.stage_forward(X, st, g, fk, ek, drop)
    f = ref_stage_fwd(c["h"], c["s"], H, ek, SCALE, bg.eu, bg.ei, N, bg.depth)
    assert torch.allclose(f["Z"], c["Z"], rtol=1e-12, atol=1e-14)
    assert torch.allclose(f["norm"], c["norm"], rtol=1e-12, atol=0)
    G = torch.randn((N, 64), generator=gen, dtype=f64)
    dX, grads = port.stage_backward(G, c, st, g)
    pr = ref_prep(G, c["Z"], c["h"], c["norm"], H)
    b = ref_stage_bwd(G, pr["Ghat"], pr["dN"], c["h"], c["s"], st["a"], H, ek, SCALE, bg.eu, bg.ei, U, N, bg.depth)
    hv = c["h"].view(N, H, DH)
    da = torch.cat([(b["dS"][:U, :, None] * hv[:U]).sum(0), (b["dS"][U:, :, None] * hv[U:]).sum(0)], 1)
    dh = b["dh"]
    dWu = (c["Xd"][:U].t() @ dh[:U]).view(64, H, DH).permute(1, 0, 2)
    dWi = (c["Xd"][U:].t() @ dh[U:]).view(64, H, DH).permute(1, 0, 2)
    dXd = torch.cat([dh[:U] @ port._wcat(st["Wu"]).t(), dh[U:] @ port._wcat(st["Wi"]).t()])
    dX_ref = dXd if fk is None else dXd * fk.double() * SCALE
    for ours, theirs in ((da, grads["a"]), (dWu, grads["Wu"]), (dWi, grads["Wi"]), (dX_ref, dX)):
        assert rel_err(ours, theirs) < 1e-12


@pytest.mark.parametrize("self_loops", [True, False])
def test_spgat_references_equal_port(self_loops):
    bg = boundary()
    U, I = bg.U, bg.I if self_loops else bg.I - N_EMPTY          # without self loops an isolated item has no attention row
    g = port.build_graph(np.stack([bg.u, bg.i]), U, I)
    N = U + I
    row, col = port.homo_edges(g, self_loops)
    gen = torch.Generator().manual_seed(3)
    for H, DH in ((8, 8), (1, 64)):
        st = dict(W=torch.randn((H, 64, DH), generator=gen, dtype=f64) * 0.2, a=torch.randn((H, 2 * DH), generator=gen, dtype=f64))
        X = torch.randn((N, 64), generator=gen, dtype=f64)
        ek = torch.rand((row.shape[0], H), generator=gen, dtype=f64) < 0.8
        c = port.spgat_stage_forward(X, st, row, col, None, ek, DROP)
        r, cc = torch.from_numpy(row), torch.from_numpy(col)
        deg = np.bincount(row, minlength=N)
        f = ref_aggregate(c["h"], c["p"][r] + c["q"][cc], H, ek.double(), SCALE, r, cc, N, depth_of(deg), residual=False)
        assert torch.allclose(f["Z"], c["Z"], rtol=1e-12, atol=1e-14)
        assert torch.allclose(f["norm"], 1.0 / c["inv"], rtol=1e-12, atol=0)
        p_, _, q_, _ = node_logits_ref(c["h"], st["a"], H)
        assert torch.allclose(p_, c["p"], rtol=1e-12, atol=1e-14) and torch.allclose(q_, c["q"], rtol=1e-12, atol=1e-14)
        G = torch.randn((N, 64), generator=gen, dtype=f64)
        dX, grads = port.spgat_stage_backward(G, c, st, row, col)
        b = ref_spgat_bwd(G, c["Z"], f["norm"], c["h"], c["p"], c["q"], st["a"], H, ek, SCALE, r, cc, N, depth_of(deg))
        hv = c["h"].view(N, H, DH)
        da = torch.cat([(b["dP"][:, :, None] * hv).sum(0), (b["dQ"][:, :, None] * hv).sum(0)], 1)
        dW = (c["Xd"].t() @ b["dh"]).view(64, H, DH).permute(1, 0, 2)
        assert rel_err(da, grads["a"]) < 1e-12 and rel_err(dW, grads["W"]) < 1e-12
        assert rel_err(b["dh"] @ port._wcat(st["W"]).t(), dX) < 1e-12


@pytest.mark.parametrize("kind", ["norm_adj", "mean_adj"])
def test_spmm_reference_equals_laplacian(kind):
    from ngacf_b200.gp import normalized_laplacian
    bg = boundary()
    L = normalized_laplacian(bg.U, bg.I, bg.u, bg.i, kind=kind)
    val, _, diag64 = laplacian_values(bg, L)
    X = torch.randn((bg.N, 64), generator=torch.Generator().manual_seed(1), dtype=f64)
    Y, _ = ref_spmm(X, val, diag64, bg.eu, bg.ei, bg.N, bg.depth)
    Y_lap = torch.sparse.mm(L.double(), X) + X                    # (L + I) X, GPLayer.forward
    assert rel_err(Y, Y_lap) < 1e-12


def test_bounds_fail_on_single_wrong_terms():
    """each mutation stands for a kernel that gets one term wrong: the element-wise bound fails at that row (or edge); the
    max-normalised rel_err < 1e-4 of the model-level tests passes several of them"""
    bg = boundary()
    U, N, E, H = bg.U, bg.N, bg.E, 8
    inp = stage_inputs(N, H, 64, 21)
    _, keep = edge_keep(E, H, DROP)
    h, s = inp.h, inp.s
    f = ref_stage_fwd(h, s, H, keep, SCALE, bg.eu, bg.ei, N, bg.depth)
    x = s.double()[bg.eu] + s.double()[bg.ei]
    r, m = bip_pairs(bg.eu, bg.ei)
    k2 = torch.cat([keep, keep]).double()
    x2 = torch.cat([x, x])

    def fwd_without(drop_pair):
        sel = torch.ones(r.shape[0], dtype=torch.bool)
        sel[drop_pair] = False
        return ref_aggregate(h, x2[sel], H, k2[sel], SCALE, r[sel], m[sel], N, bg.depth)

    results = {}

    def expect_fail(name, got, ref, bound, where):
        bad = violations(got, ref, bound)
        assert bad[where].any(), "%s: the bound does not catch it" % name
        results[name] = rel_err(got, ref)

    # (1) the only edge of a degree-1 user left out of its row
    n1 = bg.spec_u[1]
    p1 = int(torch.nonzero(r == n1)[0, 0])
    expect_fail("degree-1 row misses its edge", fwd_without(p1)["Z"], f["Z"], f["Z_bound"], n1)
    # (2) the last slot of a 257-edge item row (its 257th edge, alone in slot 3) dropped
    n257 = bg.spec_i[257]
    p257 = torch.nonzero(r == n257)[:, 0]
    assert p257.numel() == 257
    expect_fail("257-edge row drops its last slot", fwd_without(int(p257[-1]))["Z"], f["Z"], f["Z_bound"], n257)
    # (3) one edge-mask bit flipped on an edge of the 1000-edge user (one term of a thousand)
    n1000 = bg.spec_u[1000]
    e0 = int(torch.nonzero(bg.eu == n1000)[500, 0])
    kf = keep.clone()
    kf[e0, 3] = ~kf[e0, 3]
    expect_fail("edge-mask bit flipped", ref_stage_fwd(h, s, H, kf, SCALE, bg.eu, bg.ei, N, bg.depth)["Z"], f["Z"], f["Z_bound"], n1000)
    # (4) norm taken after the mask (the kernels sum the unmasked weights, as the reference does)
    e, _ = weights(x2)
    norm_after = torch.zeros((N, H), dtype=f64).index_add_(0, r, e * k2 * SCALE)
    A = (f["Z"] - h.double()).view(N, H, 8) * f["norm"][:, :, None]
    inv_after = torch.where(norm_after > 0, 1 / norm_after, torch.zeros_like(norm_after))
    Z_after = (h.double().view(N, H, 8) + A * inv_after[:, :, None]).reshape(N, 64)
    expect_fail("norm after the mask", Z_after, f["Z"], f["Z_bound"], slice(None))

    # backward: Ghat / dN rounded to fp32 are the kernel inputs
    pr = ref_prep(inp.G, f["Z"].float(), h, f["norm"].float(), H)
    b = ref_stage_bwd(inp.G, pr["Ghat"].float(), pr["dN"].float(), h, s, inp.a, H, keep, SCALE, bg.eu, bg.ei, U, N, bg.depth)
    # (5) heads 2 and 5 of dS swapped
    perm = [0, 1, 5, 3, 4, 2, 6, 7]
    expect_fail("dS heads swapped", b["dS"][:, perm], b["dS"], b["dS_bound"], slice(None))
    # (6) the keep * scale factor left out of one d s (a dropped head of an edge: keep = 0): the smallest such change that the
    # bounds of the stored d s and of the dS of both endpoints resolve by a factor 100
    ds_wrong = -(b["det"] + b["dsum"]) * b["e"] * torch.where(b["x"] > 0, 1.0, ALPHA)
    delta = torch.where(b["ksc"] == 0, (ds_wrong - b["ds"]).abs(), torch.zeros_like(ds_wrong))
    resolved = torch.maximum(b["ds_bound"], torch.maximum(b["dS_bound"][bg.eu], b["dS_bound"][bg.ei]))
    delta = torch.where(delta > 100 * resolved, delta, torch.full_like(delta, float("inf")))
    ei0, k0 = divmod(int(delta.argmin()), H)
    ds_mut = b["ds"].clone()
    ds_mut[ei0, k0] = ds_wrong[ei0, k0]
    expect_fail("keep*scale missing in one d s", ds_mut, b["ds"], b["ds_bound"], ei0)
    dS_mut = b["dS"].clone()
    for n in (int(bg.eu[ei0]), int(bg.ei[ei0])):
        dS_mut[n, k0] += ds_wrong[ei0, k0] - b["ds"][ei0, k0]
    expect_fail("keep*scale missing in one d s -> dS", dS_mut, b["dS"], b["dS_bound"], int(bg.eu[ei0]))
    print("\nmax-normalised error of each mutation (the model-level bar is 1e-4):")
    for name, v in results.items():
        print("  %-40s %.3e" % (name, v))
    assert sum(v < 1e-4 for v in results.values()) >= 2, results


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
RATIOS = {}


def check(name, got, ref, bound):
    """|got - ref| <= bound element-wise (NaN fails); records and prints the largest error / bound"""
    got = got.detach().double().cpu()
    err = (got - ref).abs()
    bad = ~(err <= bound)
    ratio = float((err / bound).nan_to_num(float("inf")).max()) if err.numel() else 0.0
    RATIOS[name] = max(RATIOS.get(name, 0.0), ratio)
    print("RATIO %-48s %.3f" % (name, ratio))
    if bad.any():
        i = tuple(int(v) for v in torch.nonzero(bad)[0])
        raise AssertionError("%s: %d of %d elements exceed the bound (max error/bound %.3g); first at %s: got %r, ref %r, bound %.3g"
                             % (name, int(bad.sum()), bad.numel(), ratio, i, float(got[i]), float(ref[i]), float(bound[i])))


def nan_like(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device=DEV)


def bits_of(t):
    return t.detach().contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def run_twice(fn):
    """runs fn twice (fresh NaN-filled outputs each time) and requires bit-identical results: long rows combine in slot order"""
    a = fn()
    b = fn()
    for x, y in zip(a, b):
        assert torch.equal(bits_of(x), bits_of(y)), "second run differs"
    return a


def cuda_graph(u_, i_, U, I):
    from ngacf_b200.graph import BipartiteGraph
    return BipartiteGraph(torch.from_numpy(np.stack([u_, i_])).to(DEV), U, I, check_users=False)


@functools.lru_cache(maxsize=None)
def gpu_graph():
    bg = boundary()
    g = cuda_graph(bg.u, bg.i, bg.U, bg.I)
    assert g.E == bg.E and np.array_equal(g.colidx.cpu().numpy(), bg.g.colidx) and np.array_equal(g.perm.cpu().numpy(), bg.g.perm)
    return g


def scratch_for(g, W=64):
    return (torch.empty(max(g.S, 1) * (W + 8), dtype=torch.float32, device=DEV), torch.zeros(max(g.L, 1), dtype=torch.int32, device=DEV))


def wtab_for(a, W, H):
    """pointer table [W_u x H | W_i x H | a x H]; the gather kernels read the attention rows a only"""
    from ngacf_b200 import ops
    DH = W // H
    ts = [torch.zeros((64, DH), dtype=torch.float32, device=DEV) for _ in range(2 * H)]
    ts += [a[k:k + 1].contiguous().to(DEV) for k in range(H)]
    return ops.pointer_table(ts), ts


def dev(*ts):
    return [None if t is None else torch.as_tensor(t).to(DEV) for t in ts]


@gpu
@pytest.mark.parametrize("drop", [0.0, DROP])
@pytest.mark.parametrize("H,W", [(8, 64), (1, 64), (1, 128)])
def test_stage_kernels_vs_fp64(H, W, drop):
    """aggregate_fwd -> Z, norm; stage_bwd_prep -> Ghat, dN; stage_bwd_edges mode 0 -> d s of every edge and head, user rows of
    dh / dS; mode 1 -> item rows of dh / dS.  `_w` entry points at W = 128."""
    from ngacf_b200 import ops
    bg, g = boundary(), gpu_graph()
    N, U, E = bg.N, bg.U, bg.E
    inp = stage_inputs(N, H, W, 100 + H + W)
    bits, keep = edge_keep(E, H, drop)
    scale = SCALE if drop else 1.0
    h, s, G = dev(inp.h, inp.s, inp.G)
    em, = dev(bits)
    wt, _keep_alive = wtab_for(inp.a, W, H)
    tag = "H=%d W=%d drop=%g" % (H, W, drop)

    def fwd():
        scratch, counter = scratch_for(g, W)
        Z, norm = nan_like(N, W), nan_like(N, H)
        ops.aggregate_fwd(g, scratch, counter, h, s, H, em, scale, Z, norm, width=W)
        return Z, norm
    Z, norm = run_twice(fwd)
    f = ref_stage_fwd(inp.h, inp.s, H, keep, scale, bg.eu, bg.ei, N, bg.depth)
    check("aggregate_fwd Z " + tag, Z, f["Z"], f["Z_bound"])
    check("aggregate_fwd norm " + tag, norm, f["norm"], f["norm_bound"])

    def bwd():
        scratch, counter = scratch_for(g, W)
        Ghat, dN = nan_like(N, W), nan_like(N, H)
        ds_store, dh, dS = nan_like(E * 8), nan_like(N, W), nan_like(N, H)
        ops.stage_bwd_prep(G, Z, h, norm, H, Ghat, dN, width=W)
        for mode in (0, 1):
            ops.stage_bwd_edges(mode, g, scratch, counter, G, Ghat, dN, h, s, H, em, scale, wt, ds_store, dh, dS, width=W)
        return Ghat, dN, ds_store, dh, dS
    Ghat, dN, ds_store, dh, dS = run_twice(bwd)
    pr = ref_prep(inp.G, Z.cpu(), inp.h, norm.cpu(), H)
    check("stage_bwd_prep Ghat " + tag, Ghat, pr["Ghat"], pr["Ghat_bound"])
    check("stage_bwd_prep dN " + tag, dN, pr["dN"], pr["dN_bound"])
    b = ref_stage_bwd(inp.G, Ghat.cpu(), dN.cpu(), inp.h, inp.s, inp.a, H, keep, scale, bg.eu, bg.ei, U, N, bg.depth)
    # ds_store layout (csrc/propagate_bwd.cu, stage_bwd_edges_kernel): H = 8 stores d s at [eid * 8 + head]; H = 1 stores the pair
    # (d s, e * keep * scale) as a float2 at [eid] -- the item pass reads the pair instead of recomputing the weight
    if H == 8:
        check("stage_bwd_edges ds " + tag, ds_store.view(E, 8), b["ds"], b["ds_bound"])
    else:
        pairs = ds_store[:2 * E].view(E, 2)
        check("stage_bwd_edges ds " + tag, pairs[:, :1], b["ds"], b["ds_bound"])
        check("stage_bwd_edges e*keep " + tag, pairs[:, 1:], b["et"], b["et_bound"])
    for side, rows in (("users (mode 0)", slice(0, U)), ("items (mode 1)", slice(U, N))):
        check("stage_bwd_edges dh %s %s" % (side, tag), dh[rows], b["dh"][rows], b["dh_bound"][rows])
        check("stage_bwd_edges dS %s %s" % (side, tag), dS[rows], b["dS"][rows], b["dS_bound"][rows])


@gpu
@pytest.mark.parametrize("drop", [0.0, DROP])
@pytest.mark.parametrize("H", [8, 1])
def test_pruned_stage_vs_fp64(H, drop):
    """aggregate_fwd_active (H = 8, 1), stage_bwd_prep_active and stage_bwd_edges_active (H = 1) against the full fp64 stage whose
    G is zero outside the active rows.  What csrc/pruned_stage.cu promises for the rest: the forward and the prep write the
    active rows only; the user pass writes dh / dS of every user and the item pass of every item (G = 0 on inactive rows), and d s
    is stored for the visited edges only -- those with an active endpoint."""
    from ngacf_b200 import ops
    bg, g = boundary(), gpu_graph()
    N, U, E, W = bg.N, bg.U, bg.E, 64
    inp = stage_inputs(N, H, W, 300 + H)
    bits, keep = edge_keep(E, H, drop)
    scale = SCALE if drop else 1.0
    rng = np.random.default_rng(7)
    su, si = bg.spec_u, bg.spec_i
    users = [su[1000], su[257], su[1], su[1], su[129], su[1000]] + rng.choice(U, 40).tolist()
    items = [si[1000] - U, si[257] - U, si[1] - U, si[1000] - U, si[256] - U, N - U - 1] + rng.choice(bg.I, 40).tolist()
    active = torch.zeros(N, dtype=torch.bool)
    active[torch.tensor(users)] = True
    active[U + torch.tensor(items)] = True
    h, s = dev(inp.h, inp.s)
    em, = dev(bits)
    ut, it = dev(np.array(users, np.int64), np.array(items, np.int64))
    act = ops.ActiveRows(g, val=7)
    act.mark(ut, it)
    tag = "H=%d drop=%g" % (H, drop)

    def fwd():
        scratch, counter = scratch_for(g)
        Z, norm = nan_like(N, W), nan_like(N, H)
        ops.aggregate_fwd_active(g, scratch, counter, h, s, H, em, scale, Z, norm, act)
        return Z, norm
    Z, norm = run_twice(fwd)
    f = ref_stage_fwd(inp.h, inp.s, H, keep, scale, bg.eu, bg.ei, N, bg.depth)
    check("aggregate_fwd_active Z " + tag, Z[active.to(DEV)], f["Z"][active], f["Z_bound"][active])
    check("aggregate_fwd_active norm " + tag, norm[active.to(DEV)], f["norm"][active], f["norm_bound"][active])
    assert Z.cpu()[~active].isnan().all() and norm.cpu()[~active].isnan().all(), "rows outside the batch were written"
    if H != 1:
        return
    G32 = torch.where(active[:, None], inp.G, torch.zeros_like(inp.G))
    G, = dev(G32)
    wt, _keep_alive = wtab_for(inp.a, W, H)

    def bwd():
        scratch, counter = scratch_for(g)
        Ghat, dN = nan_like(N, W), nan_like(N, H)
        ds_store, dh, dS = nan_like(2 * E), nan_like(N, W), nan_like(N, H)
        ops.stage_bwd_prep_active(g, G, Z, h, norm, H, Ghat, dN, act)
        for mode in (0, 1):
            ops.stage_bwd_edges_active(mode, g, scratch, counter, G, Ghat, dN, h, s, H, em, scale, wt, ds_store, dh, dS, act)
        return Ghat, dN, ds_store, dh, dS
    Ghat, dN, ds_store, dh, dS = (t.cpu() for t in run_twice(bwd))
    pr = ref_prep(G32, Z.cpu(), inp.h, norm.cpu(), H)
    check("stage_bwd_prep_active Ghat " + tag, Ghat[active], pr["Ghat"][active], pr["Ghat_bound"][active])
    check("stage_bwd_prep_active dN " + tag, dN[active], pr["dN"][active], pr["dN_bound"][active])
    assert Ghat[~active].isnan().all() and dN[~active].isnan().all(), "prep wrote rows outside the batch"
    Ghat_in = torch.where(active[:, None], Ghat, torch.zeros_like(Ghat))
    dN_in = torch.where(active[:, None], dN, torch.zeros_like(dN))
    b = ref_stage_bwd(G32, Ghat_in, dN_in, inp.h, inp.s, inp.a, H, keep, scale, bg.eu, bg.ei, U, N, bg.depth)
    visited = active[bg.eu] | active[bg.ei]
    pairs = ds_store.view(E, 2)
    check("stage_bwd_edges_active ds " + tag, pairs[visited, :1], b["ds"][visited], b["ds_bound"][visited])
    check("stage_bwd_edges_active e*keep " + tag, pairs[visited, 1:], b["et"][visited], b["et_bound"][visited])
    assert pairs[~visited].isnan().all(), "d s stored for an edge without an active endpoint"
    for side, rows in (("users", slice(0, U)), ("items", slice(U, N))):
        check("stage_bwd_edges_active dh %s %s" % (side, tag), dh[rows], b["dh"][rows], b["dh_bound"][rows])
        check("stage_bwd_edges_active dS %s %s" % (side, tag), dS[rows], b["dS"][rows], b["dS_bound"][rows])


@gpu
@pytest.mark.parametrize("H", [8, 1])
@pytest.mark.parametrize("world", [2, 3])
def test_partial_rows_vs_fp64(world, H):
    """each rank's local graph as ShardedTrainer builds it (ShardPlan, local_edges): aggregate_fwd(partial_from = T_users) and
    stage_bwd_edges(mode 1, partial = 1) emit raw item-row sums over the rank's edges; summed over the ranks in rank order (the
    reduce-scatter), aggregate_finalize / stage_bwd_finalize give the full stage"""
    from ngacf_b200 import ops
    from ngacf_b200.dist import ShardPlan
    bg = boundary()
    N, U, E, W = bg.N, bg.U, bg.E, 64
    inp = stage_inputs(N, H, W, 500 + H)
    bits, keep = edge_keep(E, H, DROP)
    h, s, G = dev(inp.h, inp.s, inp.G)
    em, = dev(bits)
    wt, _keep_alive = wtab_for(inp.a, W, H)
    plan = ShardPlan(bg.u, bg.i, U, bg.I, world)
    assert np.array_equal(plan.eu, bg.g.eu) and np.array_equal(plan.ei, bg.g.ei)
    f = ref_stage_fwd(inp.h, inp.s, H, keep, SCALE, bg.eu, bg.ei, N, bg.depth + world)
    # backward inputs: the fp32 Ghat / dN of the full stage (all-gathered on every rank)
    pr = ref_prep(inp.G, f["Z"].float(), inp.h, f["norm"].float(), H)
    Ghat32, dN32 = pr["Ghat"].float(), pr["dN"].float()
    Ghat, dN = dev(Ghat32, dN32)
    b = ref_stage_bwd(inp.G, Ghat32, dN32, inp.h, inp.s, inp.a, H, keep, SCALE, bg.eu, bg.ei, U, N, bg.depth + world)
    tag = "world=%d H=%d" % (world, H)
    Zp, normp, dhp, dSp = [], [], [], []
    for rank in range(world):
        lu, li = plan.local_edges(rank)
        (e0, e1), (u0, u1) = plan.edges(rank), plan.users(rank)
        gl = cuda_graph(lu, li, U, bg.I)
        el = em[e0:]
        eu_l, ei_l = torch.from_numpy(lu), torch.from_numpy(li) + U
        deg_l = np.concatenate([np.bincount(lu, minlength=U), np.bincount(li, minlength=bg.I)])
        kl = keep[e0:e1]
        fl = ref_stage_fwd(inp.h, inp.s, H, kl, SCALE, eu_l, ei_l, N, depth_of(deg_l))

        def fwd():
            scratch, counter = scratch_for(gl)
            Z, norm = nan_like(N, W), nan_like(N, H)
            ops.aggregate_fwd(gl, scratch, counter, h, s, H, el, SCALE, Z, norm, partial_from=gl.T_users)
            return Z, norm
        Z, norm = run_twice(fwd)
        own = slice(u0, u1)
        check("aggregate_fwd own users " + tag, Z[own], fl["Z"][own], fl["Z_bound"][own])
        check("aggregate_fwd partial item sums " + tag, Z[U:], fl["acc"][U:], fl["acc_bound"][U:])
        check("aggregate_fwd partial item norm " + tag, norm[U:], fl["norm"][U:], fl["norm_bound"][U:])
        Zp.append(Z[U:])
        normp.append(norm[U:])

        def bwd():
            scratch, counter = scratch_for(gl)
            ds_store, dh, dS = nan_like(max(gl.E, 1) * 8), nan_like(N, W), nan_like(N, H)
            for mode in (0, 1):
                ops.stage_bwd_edges(mode, gl, scratch, counter, G, Ghat, dN, h, s, H, el, SCALE, wt, ds_store, dh, dS, partial=mode)
            return ds_store, dh, dS
        ds_store, dh, dS = run_twice(bwd)
        bl = ref_stage_bwd(inp.G, Ghat32, dN32, inp.h, inp.s, inp.a, H, kl, SCALE, eu_l, ei_l, U, N, depth_of(deg_l))
        El = e1 - e0
        ds_l = ds_store.view(-1, 8)[:El] if H == 8 else ds_store[:2 * El].view(El, 2)[:, :1]
        check("stage_bwd_edges ds (rank-local) " + tag, ds_l, bl["ds"], bl["ds_bound"])
        check("stage_bwd_edges own users dh " + tag, dh[own], bl["dh"][own], bl["dh_bound"][own])
        check("stage_bwd_edges own users dS " + tag, dS[own], bl["dS"][own], bl["dS_bound"][own])
        check("stage_bwd_edges partial item dh " + tag, dh[U:], bl["acc"][U:], bl["acc_bound"][U:])
        check("stage_bwd_edges partial item dS " + tag, dS[U:], bl["dS"][U:], bl["dS_bound"][U:])
        dhp.append(dh[U:])
        dSp.append(dS[U:])
    P, nrm, dhs, dSs = Zp[0].clone(), normp[0].clone(), dhp[0].clone(), dSp[0].clone()
    for r in range(1, world):
        P += Zp[r]
        nrm += normp[r]
        dhs += dhp[r]
        dSs += dSp[r]
    ops.aggregate_finalize(P, h[U:], nrm, H)
    check("aggregate_finalize Z items " + tag, P, f["Z"][U:], f["Z_bound"][U:])
    ops.stage_bwd_finalize(dhs, dSs, G[U:], wt, H, 1)
    check("stage_bwd_finalize dh items " + tag, dhs, b["dh"][U:], b["dh_bound"][U:])


@gpu
@pytest.mark.parametrize("kind", ["norm_adj", "mean_adj"])
def test_spmm_sym_vs_fp64(kind):
    """SPUIGAGPCF's Laplacian product (its backward is the same call)"""
    from ngacf_b200.gp import LaplacianOp, normalized_laplacian
    bg, g = boundary(), gpu_graph()
    L = normalized_laplacian(bg.U, bg.I, bg.u, bg.i, kind=kind)
    op = LaplacianOp(g, L)
    val, diag32, _ = laplacian_values(bg, L)
    assert torch.equal(op.val[:bg.E].cpu(), val) and torch.equal(op.diag.cpu(), diag32)
    X32 = rows_scaled(bg.N, 64, torch.Generator().manual_seed(9), 1e-2, 1.0)
    X, = dev(X32)
    Y = run_twice(lambda: (op(X),))[0]
    Y_ref, bound = ref_spmm(X32, val, diag32, bg.eu, bg.ei, bg.N, bg.depth)
    check("spmm_sym " + kind, Y, Y_ref, bound)


@gpu
@pytest.mark.parametrize("drop", [0.0, DROP])
@pytest.mark.parametrize("H", [8, 1])
@pytest.mark.parametrize("self_loops", [True, False])
def test_spgat_kernels_vs_fp64(self_loops, H, drop):
    """node_logits, spgat_aggregate_fwd, spgat_bwd (Ghat, the stored pairs, dP, dQ, dh) and node_logits_bwd on the boundary graph
    (without self loops: without its isolated items, which have no attention row)"""
    from ngacf_b200 import ops
    from ngacf_b200.spgat import HomoGraph
    bg = boundary()
    U, I = bg.U, bg.I if self_loops else bg.I - N_EMPTY
    N, W = U + I, 64
    DH = W // H
    hg = HomoGraph.from_pairs(torch.from_numpy(np.stack([bg.u, bg.i])).to(DEV), U, I, self_loops)
    g = hg.g
    ptr = g.adj_ptr.cpu().to(torch.int64)
    r = torch.repeat_interleave(torch.arange(N), torch.diff(ptr))
    c = g.adj_idx.cpu().to(torch.int64)
    deg = torch.diff(ptr).numpy()
    depth = depth_of(deg) + (1 if self_loops else 0)
    if self_loops:
        r, c = torch.cat([r, torch.arange(N)]), torch.cat([c, torch.arange(N)])
    n_edges = r.numel()
    assert n_edges == hg.n_edges
    inp = stage_inputs(N, H, W, 700 + H)
    rng = np.random.default_rng(8)
    keep = None if drop == 0 else torch.from_numpy(rng.random((n_edges, H)) >= drop)
    scale = SCALE if drop else 1.0
    em = None if keep is None else torch.from_numpy(port.pack_edge_mask(keep.numpy())).to(DEV)
    h, G = dev(inp.h, inp.G)
    wt, _keep_alive = wtab_for(inp.a, W, H)
    nb = 64
    tag = "self_loops=%d H=%d drop=%g" % (self_loops, H, drop)

    def run():
        scratch, counter = scratch_for(g)
        p, q, Z, norm = nan_like(N, H), nan_like(N, H), nan_like(N, W), nan_like(N, H)
        Ghat, pairs, dP, dQ, dh = nan_like(N, W), nan_like(n_edges * H * 2), nan_like(N, H), nan_like(N, H), nan_like(N, W)
        part = nan_like(nb, 2 * W)
        ops.node_logits(h, wt, H, N, p, q)
        ops.spgat_aggregate_fwd(hg, scratch, counter, h, p, q, H, em, scale, Z, norm)
        ops.spgat_bwd(hg, scratch, counter, G, Z, norm, h, p, q, H, em, scale, wt, Ghat, pairs, dP, dQ, dh)
        ops.node_logits_bwd(h, dP, dQ, H, N, part)
        return p, q, Z, norm, Ghat, pairs, dP, dQ, dh, part
    p, q, Z, norm, Ghat, pairs, dP, dQ, dh, part = (t.cpu() for t in run_twice(run))
    p_ref, p_b, q_ref, q_b = node_logits_ref(inp.h, inp.a, H)
    check("node_logits p " + tag, p, p_ref, p_b)
    check("node_logits q " + tag, q, q_ref, q_b)
    f = ref_aggregate(inp.h, p.double()[r] + q.double()[c], H, None if keep is None else keep.double(), scale, r, c, N, depth,
                      residual=False)
    check("spgat_aggregate_fwd Z " + tag, Z, f["Z"], f["Z_bound"])
    check("spgat_aggregate_fwd norm " + tag, norm, f["norm"], f["norm_bound"])
    b = ref_spgat_bwd(inp.G, Z, norm, inp.h, p, q, inp.a, H, keep, scale, r, c, N, depth)
    check("spgat_bwd Ghat " + tag, Ghat, b["Ghat"], b["Ghat_bound"])
    pv = pairs.view(n_edges, H, 2)
    check("spgat_bwd pair ds " + tag, pv[..., 0], b["ds"], b["ds_bound"])
    check("spgat_bwd pair e*keep " + tag, pv[..., 1], b["et"], b["et_bound"])
    check("spgat_bwd dP " + tag, dP, b["dP"], b["dP_bound"])
    check("spgat_bwd dQ " + tag, dQ, b["dQ"], b["dQ_bound"])
    check("spgat_bwd dh " + tag, dh, b["dh"], b["dh_bound"])
    # da = sum_n [dP h | dQ h] from the kernel's own dP / dQ: grid-stride rows per lane, 16 groups, then the block partials
    hv = inp.h.double().view(N, H, DH)
    ts = torch.cat([(dP.double()[:, :, None] * hv).reshape(N, W), (dQ.double()[:, :, None] * hv).reshape(N, W)], 1)
    da_depth = -(-N // (nb * 16)) + 16 + 1
    check("node_logits_bwd da " + tag, part.double().sum(0), ts.sum(0), u * da_depth * ts.abs().sum(0) + TINY)
