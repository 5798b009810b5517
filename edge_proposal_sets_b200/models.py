"""Scoring models of the filter / rank path, same names, call signature and state-dict keys as the
reference's ``models.py`` so its checkpoints load unchanged and its callers
(``model(x, edges, adj_t)`` at /root/reference/filter.py:118 and train_and_eval.py:111) keep working:

  GCN / SAGE           /root/reference/models.py:163-187, 417-440   (GCNConv / SAGEConv, PyG 1.7)
  LinkPredictor        /root/reference/models.py:461-485
  LinkGNN              /root/reference/models.py:487-506
  CommonNeighborsPredictor ('simple' | 'adamic' | 'adamic_ogb' | 'resource_allocation')
                       /root/reference/models.py:508-554, plus the degree-normalised similarities of
                       SIMILARITY_MODELS (no reference counterpart; include/eps.h EPS_SCORE_*) and the
                       Local Path index 'local_path' (no reference counterpart; include/eps.h eps_local_path_*)
  build_model          /root/reference/models.py:578-670
  default_model_configs/root/reference/models.py:673-790

What is different is where the arithmetic runs: neighbour aggregation is the K1 SpMM kernel,
the (u,v) MLP is the fused K2 kernel, CN/AA is the K3 intersection kernel.  The node embeddings
``h`` are computed ONCE per (graph, weights) and cached — the reference recomputes the whole GNN
for every batch of candidates (models.py:505 inside the loop at filter.py:116-118).

Two modes, selected like the reference does with ``model.train()`` / ``model.eval()``:
  * eval (scoring path): fused kernels under ``torch.no_grad`` — K1 with bias/ReLU folded in, K2 with
    the gather folded in, embeddings cached;
  * train (SURVEY §8f row 4): the same K1 aggregation kernel behind ``autograd.spmm`` (backward = K1 on
    the transposed matrix), dropout active, dense layers as torch / cuBLAS ops so that
    ``loss.backward()`` of /root/reference/train_and_eval.py:31-96 works unchanged.
Checkpoints in the PyG-2.x GCNConv layout (``convs.i.lin.weight [out,in]``) are accepted on load.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn.functional as F
from torch import nn

from . import autograd, ops, parallel
from .graph import SparseAdj

GNN_MODELS = ("gcn", "sage")
# c / f(deg u, deg v) scores of the classic local-similarity table (Zhou, Lue & Zhang 2009) and a * b; structural and
# symmetric, computed from the exact common-neighbour count by the same kernels (``ops.cn_aa(kind=...)``)
SIMILARITY_MODELS = ("jaccard", "sorensen", "salton", "hub_promoted", "hub_depressed", "leicht_holme_newman",
                     "preferential_attachment")
# the Local Path index (Lue, Jin & Zhou 2009): (A^2)_uv + 1e-3 (A^3)_uv, structural and symmetric
# (``candidates.two_hop_local_path`` on the filter side, ``ops.local_path`` on pair lists)
LOCAL_PATH = "local_path"
HEURISTIC_MODELS = ("simple", "adamic", "adamic_ogb", "resource_allocation") + SIMILARITY_MODELS + (LOCAL_PATH,)
SUPPORTED_MODELS = GNN_MODELS + HEURISTIC_MODELS


class GCNConv(nn.Module):
    """PyG-1.7 parameter layout: ``weight [in,out]`` (glorot), ``bias [out]`` (zeros)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(in_channels, out_channels))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        a = math.sqrt(6.0 / (self.weight.shape[0] + self.weight.shape[1]))
        nn.init.uniform_(self.weight, -a, a)
        nn.init.zeros_(self.bias)

    def forward(self, x: torch.Tensor, adj: SparseAdj, relu: bool = False) -> torch.Tensor:
        rowptr, col, val = adj.gcn_norm()
        xw = x @ self.weight                       # dense GEMM stays in the library (cuBLAS fp32)
        if torch.is_grad_enabled() and (xw.requires_grad or self.bias.requires_grad):
            out = autograd.spmm(xw, rowptr, col, val, "sum", val_t=adj.gcn_norm_transposed_values()) + self.bias
            return torch.relu(out) if relu else out
        return ops.spmm_csr(rowptr, col, val, xw, "sum", self.bias, relu)

    @torch.no_grad()
    def forward_rows(self, x_rows: torch.Tensor, adj: SparseAdj, bounds, rank: int, relu: bool) -> torch.Tensor:
        """Rows [bounds[rank], bounds[rank+1]) of the layer output from the same rows of its input (scoring
        path): x·W for the local row blocks (cuBLAS fp32), all-gather of the ``n/G x H`` slabs, K1 over the
        local rows of the normalised matrix with bias / ReLU fused."""
        lo, hi = bounds[rank], bounds[rank + 1]
        rowptr, col, val = adj.gcn_norm()
        xw = parallel.allgather_row_slabs(parallel.block_matmul(x_rows, self.weight, lo, hi, adj.n), bounds)
        return ops.spmm_csr(rowptr[lo:hi + 1], col, val, xw, "sum", self.bias, relu)

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        # PyG >= 2.0 stores GCNConv's weight as ``lin.weight [out,in]`` (SURVEY §8f row 4)
        k2 = prefix + "lin.weight"
        if k2 in state_dict and prefix + "weight" not in state_dict:
            state_dict[prefix + "weight"] = state_dict.pop(k2).t().contiguous()
        return super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)


class SAGEConv(nn.Module):
    """PyG-1.7 ``SAGEConv``: ``lin_l`` (bias) on the neighbour mean, ``lin_r`` (no bias) on the root."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.lin_l = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_r = nn.Linear(in_channels, out_channels, bias=False)

    def reset_parameters(self):
        self.lin_l.reset_parameters()
        self.lin_r.reset_parameters()

    def forward(self, x: torch.Tensor, adj: SparseAdj, relu: bool = False) -> torch.Tensor:
        if torch.is_grad_enabled() and x.requires_grad:
            agg = autograd.spmm(x, adj.rowptr, adj.col, None, "mean", inv_deg=adj.inv_degree())
        else:
            agg = ops.spmm_csr(adj.rowptr, adj.col, None, x, "mean")   # edge values dropped (A.4)
        out = self.lin_l(agg) + self.lin_r(x)
        return torch.relu(out) if relu else out

    @torch.no_grad()
    def forward_rows(self, x_rows: torch.Tensor, adj: SparseAdj, bounds, rank: int, relu: bool) -> torch.Tensor:
        """Row-sharded scoring-path forward (see GCNConv.forward_rows): the layer INPUT is all-gathered, the
        neighbour mean (K1) and the two dense products run on the local rows only."""
        lo, hi = bounds[rank], bounds[rank + 1]
        x_full = parallel.allgather_row_slabs(x_rows, bounds)
        agg = ops.spmm_csr(adj.rowptr[lo:hi + 1], adj.col, None, x_full, "mean")
        out = parallel.block_matmul(agg, self.lin_l.weight.t(), lo, hi, adj.n)
        out += self.lin_l.bias
        out += parallel.block_matmul(x_rows.contiguous(), self.lin_r.weight.t(), lo, hi, adj.n)
        return torch.relu_(out) if relu else out


class _ConvStack(nn.Module):
    conv_cls = None

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__()
        dims = [in_channels] + [hidden_channels] * (num_layers - 1) + [out_channels]
        self.convs = nn.ModuleList(self.conv_cls(dims[i], dims[i + 1]) for i in range(num_layers))
        self.dropout = dropout

    def reset_parameters(self):
        for c in self.convs:
            c.reset_parameters()

    def forward(self, x, adj_t):
        last = len(self.convs) - 1
        for i, conv in enumerate(self.convs):
            x = conv(x, adj_t, relu=i != last)    # ReLU fused; dropout is identity in eval
            if i != last and self.training and self.dropout > 0:
                x = F.dropout(x, p=self.dropout, training=True)       # models.py:184-185 / 437-438
        return x


    @torch.no_grad()
    def embed_rows(self, x: torch.Tensor, adj: SparseAdj, rank: int = 0, world: int = 1) -> torch.Tensor:
        """Scoring-path forward, row-sharded over ``world`` ranks (world == 1: the same code on one GPU).
        Rank r owns a block-aligned row range of near-equal nnz (parallel.row_partition); per layer one
        all-gather of ``n/G x H`` fp32 slabs; the result is the full ``h`` on every rank, bit-identical
        for every world size (same row blocks in the dense products, same per-row order in K1)."""
        rowptr = adj.gcn_norm()[0] if self.conv_cls is GCNConv else adj.rowptr
        bounds = parallel.row_partition(rowptr, adj.n, world)
        lo, hi = bounds[rank], bounds[rank + 1]
        xr = x[lo:hi].contiguous().float()
        last = len(self.convs) - 1
        for i, conv in enumerate(self.convs):
            xr = conv.forward_rows(xr, adj, bounds, rank, relu=i != last)
        return parallel.allgather_row_slabs(xr, bounds).contiguous()


class GCN(_ConvStack):
    conv_cls = GCNConv


class SAGE(_ConvStack):
    conv_cls = SAGEConv


class LinkPredictor(nn.Module):
    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__()
        dims = [in_channels] + [hidden_channels] * (num_layers - 1) + [out_channels]
        self.lins = nn.ModuleList(nn.Linear(dims[i], dims[i + 1]) for i in range(num_layers))
        self.dropout = dropout
        # K2 arm: "prefilter" (default) = fp32 results everywhere; the filter step additionally uses the tcgen05
        # arm to preselect the band around its top-k (filter_step.FilterJob); "fp32" / "f16" force one arm
        self.precision = "prefilter"

    def reset_parameters(self):
        for lin in self.lins:
            lin.reset_parameters()

    def score_pairs(self, h: torch.Tensor, edges: torch.Tensor, precision: Optional[str] = None) -> torch.Tensor:
        """sigmoid(MLP(h[u]*h[v])) for edges [2,B] -> [B]; gather fused into the kernel.  ``precision``:
        "fp32" (FFMA, reference arithmetic) or "f16" (tcgen05, fp16 operands; alias "bf16"); default ``self.precision`` ("prefilter", the
        filter step's two-stage mode, scores a plain pair list in fp32)."""
        prec = precision or self.precision
        return ops.linkpred_mlp(h, edges, [l.weight for l in self.lins], [l.bias for l in self.lins],
                                precision="fp32" if prec == "prefilter" else prec, sigmoid=True)

    def tc_context(self, h: torch.Tensor) -> "ops.LinkpredTC":
        """The tcgen05 arm bound to ``h`` and the current weights for a series of slabs (fp16 table and weight
        images built once): ``ctx.score(edges)`` == ``score_pairs(h, edges, "f16")``."""
        return ops.LinkpredTC(h, [l.weight for l in self.lins], [l.bias for l in self.lins])

    def forward_pairs(self, h: torch.Tensor, edges: torch.Tensor) -> torch.Tensor:
        """Training-mode forward from the embedding table (models.py:478-485 after models.py:506): z0 by K7
        (``autograd.pair_hadamard``: one fused gather-multiply, scatter-add backward), then the Linear layers."""
        from . import autograd
        x = autograd.pair_hadamard(h, edges)
        for lin in self.lins[:-1]:
            x = F.dropout(F.relu(lin(x)), p=self.dropout, training=self.training)
        return torch.sigmoid(self.lins[-1](x))

    def forward(self, x_i, x_j):
        """Reference signature (two gathered [B,H] blocks) kept for callers that use it."""
        if torch.is_grad_enabled() and (self.training or x_i.requires_grad or x_j.requires_grad):
            x = x_i * x_j                                             # models.py:478-485, autograd ops
            for lin in self.lins[:-1]:
                x = F.dropout(F.relu(lin(x)), p=self.dropout, training=self.training)
            return torch.sigmoid(self.lins[-1](x))
        B = x_i.shape[0]
        h = torch.cat([x_i, x_j], 0).contiguous()
        ar = torch.arange(B, device=h.device, dtype=torch.int32)
        return self.score_pairs(h, torch.stack([ar, ar + B])).unsqueeze(1)


class LinkGNN(nn.Module):
    def __init__(self, emb, gnn, linkpred):
        super().__init__()
        self.gnn = gnn
        self.linkpred = linkpred
        self.emb = emb
        self._h_key = None
        self._h = None

    def reset_parameters(self):
        self.gnn.reset_parameters()
        self.linkpred.reset_parameters()
        if self.emb is not None:
            self.emb.reset_parameters()
        self._h_key = None

    def _input(self, x):
        if x is None:
            return self.emb.weight
        if self.emb is not None:
            return torch.cat([self.emb.weight, x], dim=1)
        return x

    @torch.no_grad()
    def embed(self, x, adj: SparseAdj, distributed: bool = False) -> torch.Tensor:
        """h = gnn(input, adj) in eval arithmetic (dropout off), cached on (graph uid, input identity,
        parameter versions).  ``distributed``: row-sharded over the ranks of the default process group and
        all-gathered (every rank ends up with the full h, the same bits as on one GPU).  While the module
        is in training mode nothing is cached (a later eval call must not see dropout-perturbed h)."""
        rank, world = parallel.world_info() if distributed else (0, 1)
        key = (adj.uid, None if x is None else (x.data_ptr(), x._version),
               tuple((p.data_ptr(), p._version) for p in self.parameters()))
        if self.training:
            return self.gnn(self._input(x), adj).contiguous()
        if key != self._h_key:
            self._h = self.gnn.embed_rows(self._input(x), adj, rank, world)
            self._h_key = key
        return self._h

    def forward(self, x, edges, adj):
        if self.training and torch.is_grad_enabled():
            # train_and_eval.py:60: the whole GNN runs per batch, with autograd (models.py:500-506)
            h = self.gnn(self._input(x), adj)
            return self.linkpred.forward_pairs(h, edges)
        with torch.no_grad():
            h = self.embed(x, adj)
            return self.linkpred.score_pairs(h, edges).unsqueeze(1)   # [B,1] like the reference


class CommonNeighborsPredictor(nn.Module):
    def __init__(self, emb, in_channels, hidden_channels, out_channels, num_layers, dropout,
                 model_type="simple"):
        super().__init__()
        if model_type not in HEURISTIC_MODELS + ("katz",):
            raise ValueError(f"model_type {model_type!r} is outside the scoring path "
                             f"(supported: {HEURISTIC_MODELS})")
        self.type = model_type
        self.emb = emb
        self.mlp = nn.Identity()
        self.grouped_by_v = False   # set by the filter driver for column-major candidate lists

    def reset_parameters(self):
        if self.emb is not None:
            self.emb.reset_parameters()

    @torch.no_grad()
    def forward(self, x, edges, adj: SparseAdj):
        if self.type in ("adamic_ogb", "resource_allocation", "katz"):
            return None                            # reference behaviour (models.py:534-535)
        if self.type in SIMILARITY_MODELS:
            return ops.cn_aa(adj, edges, kind=self.type, grouped_by_v=self.grouped_by_v)
        if self.type == LOCAL_PATH:
            return ops.local_path(adj, edges)
        if self.type == "simple":
            # sum_k adj[u,k]*adj[v,k]; raw value, no sigmoid (models.py:539-542)
            return ops.cn_aa(adj, edges, None, use_values=True, grouped_by_v=self.grouped_by_v)
        # 'adamic': sigmoid(sum_{k in CN} 1/log(deg_k + 1e-6)), indices only (models.py:544-554)
        return ops.cn_aa(adj, edges, adj.adamic_weights(), use_values=False, sigmoid=True,
                         grouped_by_v=self.grouped_by_v)


def build_model(args, data, device):
    """models.build_model for the models on the scoring path."""
    if args.model not in SUPPORTED_MODELS:
        raise ValueError(f"model {args.model!r} is outside the scoring path (supported: {SUPPORTED_MODELS})")
    emb = None
    input_dim = 0
    if args.use_learnable_embedding:
        emb = nn.Embedding(data.num_nodes, args.hidden_channels, device=device)
        input_dim += args.hidden_channels
    if args.use_feature:
        input_dim += data.x.shape[1]
    if args.model in GNN_MODELS:
        cls = GCN if args.model == "gcn" else SAGE
        gnn = cls(input_dim, args.hidden_channels, args.hidden_channels, args.num_layers, args.dropout).to(device)
        linkpred = LinkPredictor(args.hidden_channels, args.hidden_channels, 1, args.num_layers,
                                 args.dropout).to(device)
        linkpred.precision = getattr(args, "mlp_precision", None) or "prefilter"
        return LinkGNN(emb, gnn, linkpred)
    return CommonNeighborsPredictor(emb, input_dim, args.hidden_channels, args.hidden_channels,
                                    args.num_layers, args.dropout, model_type=args.model).to(device)


# (dataset family) -> shared settings, then per-model-family GNN settings; values are the
# reference's table (/root/reference/models.py:685-771).  'ppa' has no entry in the reference
# (SURVEY A.8); the row here is this build's choice and only fills values the CLI left unset.
_GNN = ("sage", "gcn")
_DATASET_DEFAULTS = {
    "ddi": dict(use_feature=False, use_learnable_embedding=True, batch_size=64 * 1024,
                gnn=dict(num_layers=2, hidden_channels=256, dropout=0.5, lr=0.005, epochs=200)),
    "collab": dict(use_feature=True, use_learnable_embedding=True, batch_size=16 * 1024,
                   gnn=dict(num_layers=3, hidden_channels=256, dropout=0.0, lr=0.001, epochs=200)),
    "reddit": dict(use_feature=True, use_learnable_embedding=True, batch_size=64 * 1024,
                   gnn=dict(num_layers=3, hidden_channels=256, dropout=0.0, lr=0.005, epochs=200)),
    "email": dict(use_feature=False, use_learnable_embedding=True, batch_size=16 * 1024,
                  gnn=dict(num_layers=3, hidden_channels=300, dropout=0.0, lr=0.001, epochs=200)),
    "ppa": dict(use_feature=True, use_learnable_embedding=True, batch_size=64 * 1024,
                gnn=dict(num_layers=3, hidden_channels=256, dropout=0.0, lr=0.001, epochs=200)),
}
_DATASET_DEFAULTS["twitch"] = _DATASET_DEFAULTS["reddit"]
_DATASET_DEFAULTS["fb"] = _DATASET_DEFAULTS["reddit"]
_OVERRIDABLE = ("num_layers", "hidden_channels", "dropout", "batch_size", "lr", "epochs",
                "use_feature", "use_learnable_embedding")


def default_model_configs(args):
    """Fill every model argument the CLI left as ``None`` from the per-(dataset, model) table."""
    base = args.dataset.split("-shape")[0]
    table = _DATASET_DEFAULTS.get(base, {})
    d = {k: None for k in _OVERRIDABLE}
    for k in ("use_feature", "use_learnable_embedding", "batch_size"):
        d[k] = table.get(k)
    if args.model in _GNN:
        d.update(table.get("gnn", {}))
    if base == "ddi" and args.model == "simple":
        d["batch_size"] = 1024                     # models.py:706-707
    for k in _OVERRIDABLE:
        if getattr(args, k, None) is None:
            setattr(args, k, d[k])
    if args.model in HEURISTIC_MODELS + ("katz",):
        args.use_feature = False                   # models.py:783-785
        args.use_learnable_embedding = False
    return args
