"""SPUIGAGPCF (SURVEY.md 8f-1; graphattention/SPUIGACF.py:103-185 of the reference): the SpUIGAT propagation of SPUIGACF followed by
Laplacian-propagation layers

    features <- ReLU(Linear((L + I) features))        (GPLayer :174-185, Affinelayers :129-132)

whose outputs are concatenated to the attention output; the score is the dot product of the concatenated user / item rows.

The sparse parts run on this repo's kernels: the attention propagation is the SPUIGACF path, the Laplacian product is
``ngacf_spmm_sym`` over the same adjacency and task list (the Laplacian of a bipartite interaction graph is symmetric and has the
adjacency's pattern plus a diagonal, so one value per undirected edge and one per node describe it, and the backward is the same
call).  The 64x64 affine layers, the ReLU, the concatenation and the 192-wide pair dot product are plain torch ops
(library GEMM): this model is a widening row, not the measured hot path.

Note: the reference's ``createModels`` branch for this model reads an undefined ``adj`` (run_Gowalla.py:102) -- it crashes as
written; the constructor signature below is the class's own (``SPUIGAGPCF(userNum, itemNum, adj, embedSize, layers, droprate)``).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn

from . import _lib, ops
from .graph import BipartiteGraph
from .model import ALPHA, SPUIGACF, SpUIGAT


def normalized_laplacian(userNum, itemNum, users, items, ratings=None, kind="norm_adj"):
    """buildLaplacianMat (data/loadGowalla.py:184-227) for 'norm_adj' (D^-1/2 (A + I) D^-1/2, degrees of A + I) and 'mean_adj'
    (D^-1/2 A D^-1/2), as a coalesced torch sparse COO tensor (N x N) like scipySP_torchSP + coalesce (:179-182,253).
    A = [[0, R], [R^T, 0]] with R the (summed) rating matrix."""
    import scipy.sparse as sp
    N = userNum + itemNum
    r = np.ones(len(users), np.float64) if ratings is None else np.asarray(ratings, np.float64)
    R = sp.coo_matrix((r, (np.asarray(users), np.asarray(items))), shape=(userNum, itemNum)).tocsr()
    A = sp.bmat([[None, R], [R.T, None]], format="csr")
    if kind == "norm_adj":
        A = A + sp.eye(N, format="csr")
    elif kind != "mean_adj":
        raise ValueError("kind must be norm_adj or mean_adj")
    deg = np.asarray(A.sum(axis=1)).reshape(-1)
    with np.errstate(divide="ignore"):
        d = np.power(deg, -0.5)
    L = sp.diags(d).dot(A).dot(sp.diags(d)).tocoo()
    idx = torch.from_numpy(np.stack([L.row, L.col]).astype(np.int64))
    return torch.sparse_coo_tensor(idx, torch.from_numpy(L.data.astype(np.float32)), (N, N)).coalesce()


class LaplacianOp:
    """(L + I) as {one value per undirected edge of the graph, one per node}.  `L` is the constructor's `adj`: a (N,N) torch sparse
    tensor, symmetric, whose off-diagonal pattern lies inside the interaction graph's."""

    def __init__(self, graph: BipartiteGraph, L: torch.Tensor):
        g = graph
        dev = g.device
        L = L.coalesce().to(dev)
        r, c = L.indices()
        v = L.values().to(torch.float32)
        N, U, I = g.N, g.U, g.I
        if tuple(L.shape) != (N, N):
            raise ValueError("the Laplacian must be (%d,%d)" % (N, N))
        self.diag = torch.ones(N, dtype=torch.float32, device=dev)          # the `+ selfLoop` of GPLayer.forward (:179)
        on = r == c
        self.diag.index_add_(0, r[on], v[on])
        # CSR edge id of every (user, item) entry: position of its key among the graph's sorted unique keys
        rows = torch.repeat_interleave(torch.arange(U, device=dev), torch.diff(g.rowptr.to(torch.int64)))
        keys = rows * I + g.colidx.to(torch.int64)

        def edge_ids(uu, ii):
            k = uu * I + ii
            pos = torch.searchsorted(keys, k)
            ok = (pos < keys.numel()) & (keys[pos.clamp(max=max(keys.numel() - 1, 0))] == k)
            if not bool(ok.all()):
                raise ValueError("the Laplacian has an off-diagonal entry outside the interaction graph")
            return pos
        up = (r < U) & (c >= U)
        lo = (r >= U) & (c < U)
        if bool((~(up | lo | on)).any()):
            raise ValueError("the Laplacian has user-user or item-item entries: not a bipartite interaction graph")
        self.val = torch.zeros(max(g.E, 1), dtype=torch.float32, device=dev)
        self.val[edge_ids(r[up], c[up] - U)] = v[up]
        low = torch.zeros_like(self.val)
        low[edge_ids(c[lo], r[lo] - U)] = v[lo]
        if not torch.allclose(self.val, low, rtol=1e-6, atol=1e-12):
            raise NotImplementedError("the Laplacian is not symmetric (ngacf_spmm_sym stores one value per undirected edge)")
        self.g = g
        self.scratch, self.counter = g.scratch("laplacian")

    def __call__(self, X: torch.Tensor) -> torch.Tensor:
        Y = torch.empty_like(X)
        ops.spmm_sym(self.g, self.scratch, self.counter, self.val, self.diag, X.contiguous(), Y)
        return Y


class _SpmmSymFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, op, X):
        ctx.op = op
        return op(X.detach())

    @staticmethod
    def backward(ctx, dY):
        return None, ctx.op(dY.contiguous())        # symmetric operator: the transpose is the same product


class GPLayer(nn.Module):
    """features <- (laplacianMat + selfLoop) features  (SPUIGACF.py:174-185); the operator is prepared once per graph."""

    def forward(self, features, laplacian: LaplacianOp, selfLoop=None):
        return _SpmmSymFn.apply(laplacian, features)


class SPUIGAGPCF(SPUIGACF):
    def __init__(self, userNum, itemNum, adj, embedSize, layers, droprate, useCuda=True):
        if embedSize != 64:
            raise ValueError("SPUIGAGPCF is built for embedSize 64 only (its GP layers and stage kernels are 64 wide)")
        super().__init__(userNum, itemNum, embedSize, list(layers), droprate, useCuda)
        self.LaplacianMat = adj
        self._lap_key, self._lap = None, None

    def _extra_modules(self, embedSize, layers):
        # same construction order as the reference (:123-129): the GP / affine layers exist before the embeddings are initialised
        self.GPlayers = nn.ModuleList()
        self.Affinelayers = nn.ModuleList()
        dims = [embedSize] + list(layers)              # `layers.insert(0, embedSize)` (:125)
        for From, To in zip(dims[:-1], dims[1:]):
            if From != 64:
                raise ValueError("the Laplacian product is specialised for 64-wide features (layers must be [64, ...])")
            self.GPlayers.append(GPLayer())
            self.Affinelayers.append(nn.Linear(From, To))

    def _laplacian_for(self, graph):
        key = id(graph)
        if key != self._lap_key:
            self._lap = LaplacianOp(graph, self.LaplacianMat)
            self._lap_key = key
        return self._lap

    def final_embeddings(self, mask):
        """(N, 64 * (1 + number of GP layers)): [ELU(Z_gat) | GP layer outputs]  (SPUIGACF.py:159-166)"""
        graph = self.graph_for(mask)
        features = torch.nn.functional.elu(self.propagate(graph))
        lap = self._laplacian_for(graph)
        final = [features]
        for gp, aff in zip(self.GPlayers, self.Affinelayers):
            features = torch.relu(aff(gp(features, lap)))
            final.append(features)
        return torch.cat(final, dim=1)

    def forward(self, userIdx, itemIdx, mask):
        F = self.final_embeddings(mask)
        dev = F.device
        return torch.sum(F[userIdx.to(dev)] * F[itemIdx.to(dev) + self.userNum], dim=1)
