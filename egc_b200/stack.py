"""`EGC` - the layer stack the reference trains on the full-graph workloads, on the sm_100a kernels.

Mirrors /root/reference/experiments/mag/models.py:16-69: `num_layers` EGConv layers (IN_FEATURES -> hidden -> ... ->
OUT_ROUNDED), ReLU + dropout between them, the last layer's output truncated to OUT_TRUE columns, `log_softmax`.
Same constructor arguments, `convs` ModuleList (so `state_dict` keys match: `convs.{i}.bases_weight`, ...),
`reset_parameters()` and `forward(x, adj_t)`.

Differences in execution only:
  * the ReLU after every hidden layer (ref :63) runs inside the layer: `max(., 0)` in the aggregation kernel's epilogue,
    `grad * (out > 0)` while the backward's first pass stages the gradient row - no separate elementwise kernels, no
    extra [N, F] round trips;
  * every layer of the stack uses the same aggregator list, so the prepared graph (CSR, CSC, symnorm weights, plans)
    is built ONCE and shared by the layers (the reference caches one copy per layer, `cached=True`);
  * `forward` also accepts a `PartitionedGraph` (row-partitioned multi-GPU run, `egc_b200.dist`): `x` then holds
    this rank's rows and the result is this rank's rows of the single-GPU result;
  * opt-in (`fused_dropout=True`): in training mode the dropout after every hidden layer runs in the same epilogue, after
    the ReLU, and its backward is the ReLU's mask scaled by 1 / (1 - p) - no separate kernels, no stored mask.  Its random
    stream is a counter-based one (`egc_b200.functional.egconv`), not torch's F.dropout stream, so it is not the default.
"""
from typing import Iterable

import torch
import torch.nn.functional as F
from torch import Tensor

from .conv import EGConv
from .functional import draw_dropout_seed
from .graph import GraphStructure

IN_FEATURES = 128        # ref mag/models.py:8-10
OUT_ROUNDED = 352
OUT_TRUE = 349


class EGC(torch.nn.Module):
    def __init__(self, hidden_channels: int, num_layers: int, dropout: float, num_heads: int, num_bases: int,
                 aggrs: Iterable[str], in_features: int = IN_FEATURES, out_rounded: int = OUT_ROUNDED,
                 out_true: int = OUT_TRUE, *, fused_dropout: bool = False, **conv_kwargs):
        super().__init__()
        if num_layers < 2:
            raise ValueError("EGC needs at least two layers (ref mag/models.py:22-54)")
        aggrs = list(aggrs)
        dims = [in_features] + [hidden_channels] * (num_layers - 1) + [out_rounded]
        self.convs = torch.nn.ModuleList(
            EGConv(dims[i], dims[i + 1], aggrs=aggrs, num_heads=num_heads, num_bases=num_bases, cached=True, **conv_kwargs)
            for i in range(num_layers))
        self.dropout = dropout
        self.out_true = out_true
        self.fused_dropout = bool(fused_dropout)
        # seed tensors of the fused dropout drawn by the last forward, in layer order (inside a captured CUDA graph: the
        # graph's buffers, which hold each replay's seeds) - enough to rebuild the masks exactly
        self.last_dropout_seeds = []

    def reset_parameters(self):
        for conv in self.convs:
            conv.reset_parameters()

    def prepare(self, x: Tensor, adj_t):
        """The prepared graph shared by the layers: built and cached by the first layer's rules (`cached=True`,
        ref optimized_layers.py:126-175), so - as in the reference - later calls reuse the first call's graph."""
        from .dist import PartitionedGraph
        if isinstance(adj_t, (GraphStructure, PartitionedGraph)):
            return adj_t
        return self.convs[0]._prepare(x, adj_t)

    def forward(self, x: Tensor, adj_t) -> Tensor:
        from .dist import PartitionedGraph, partitioned_egconv
        g = self.prepare(x, adj_t)
        seeds = []

        def run(conv, h, relu, dropout=0.0):
            seed = None
            if dropout > 0.0:                                          # one seed per layer call, in layer order
                seed = draw_dropout_seed(h.device)
                seeds.append(seed)
            if isinstance(g, PartitionedGraph):
                return partitioned_egconv(h, g, conv, relu=relu, dropout=dropout, dropout_seed=seed)
            return conv(h, g, relu=relu, dropout=dropout, dropout_seed=seed)
        fused = self.fused_dropout and self.training and self.dropout > 0
        for conv in self.convs[:-1]:                                   # ref :61-65
            if fused:                                                  # conv + ReLU + dropout: one epilogue
                x = run(conv, x, True, self.dropout)
            else:
                x = run(conv, x, True)                                 # conv + ReLU: fused epilogue / backward mask
                x = F.dropout(x, p=self.dropout, training=self.training)
        self.last_dropout_seeds = seeds
        x = run(self.convs[-1], x, False)[:, :self.out_true]            # ref :68
        return x.log_softmax(dim=-1)                                   # ref :69


def fold_batchnorm(bn: torch.nn.BatchNorm1d):
    """(scale, shift) of an eval-mode BatchNorm1d:  bn(y) = y * scale + shift  with scale = gamma / sqrt(running_var +
    eps), shift = beta - running_mean * scale (gamma = 1, beta = 0 without affine).  Constants: detached."""
    if bn.running_mean is None or bn.running_var is None:
        raise ValueError("fold_batchnorm needs running statistics (track_running_stats=True)")
    with torch.no_grad():
        scale = torch.rsqrt(bn.running_var + bn.eps)
        if bn.weight is not None:
            scale = scale * bn.weight
        shift = -bn.running_mean * scale
        if bn.bias is not None:
            shift = shift + bn.bias
    return scale.float().contiguous(), shift.float().contiguous()


class EGCBlock(torch.nn.Module):
    """One block of the reference's normalised stacks (/root/reference/experiments/arxiv/norm_models.py:33-40, the same
    pattern in zinc/models.py:60-74):  conv -> BatchNorm -> ReLU -> dropout -> (+ identity).

    In eval mode (inference, or fine-tuning with frozen statistics) the whole tail runs inside the layer's aggregation
    kernel: the BatchNorm folded to an affine map, the ReLU and the residual add are its epilogue - one kernel, no extra
    [N, F] round trips.  In training mode BatchNorm needs the batch statistics of the layer's complete output first, so the
    tail stays ordinary torch ops after the layer (the ReLU cannot be fused either: it follows the normalisation)."""

    def __init__(self, conv: EGConv, dropout: float = 0.0, residual: bool = False):
        super().__init__()
        if residual and conv.in_channels != conv.out_channels:
            raise ValueError("a residual block needs in_channels == out_channels")
        self.conv = conv
        self.bn = torch.nn.BatchNorm1d(conv.out_channels)
        self.dropout, self.residual = dropout, residual
        self._folded = None                        # (versions of the BatchNorm tensors, scale, shift)

    def forward(self, x: Tensor, edge_index) -> Tensor:
        if self.training:
            y = F.relu(self.bn(self.conv(x, edge_index)))
            y = F.dropout(y, p=self.dropout, training=True)
            return y + x if self.residual else y
        bn = self.bn
        key = tuple((t.data_ptr(), t._version) for t in (bn.running_mean, bn.running_var, bn.weight, bn.bias) if t is not None)
        if self._folded is None or self._folded[0] != key:      # refolded only when the statistics / affine parameters change
            self._folded = (key,) + fold_batchnorm(bn)
        _, scale, shift = self._folded
        return self.conv(x, edge_index, relu=True, scale=scale, shift=shift, residual=x if self.residual else None)


class EgcArxivNet(torch.nn.Module):
    """The reference's normalised full-graph model (/root/reference/experiments/arxiv/norm_models.py:14-46 `ArxivNet` +
    :96-127 `EgcArxivNet`): Linear embed -> num_graph_layers x [EfficientGraphConv -> BatchNorm1d -> ReLU -> dropout ->
    (+ identity)] -> Linear -> log_softmax.  Same constructor arguments, submodule names and `state_dict` keys
    (`embed.0.*`, `convs.{i}.comb_weights.*`, `convs.{i}.bases_weight.{b}`, `convs.{i}.bias`, `bns.{i}.*`, `out.*`), so
    the reference's checkpoints load.

    Execution: the prepared graph is built once per forward and shared by the layers.  In eval mode, for the EGC-S
    configuration (`aggrs=["symadd"]`, the reference's arxiv / egc_s setting, no softmax weights) every block is ONE
    aggregation kernel: the folded BatchNorm, the ReLU and the residual add are its epilogue (the BatchNorm's own affine
    parameters are constants there: no gradient for them).  Everything else - training mode (batch statistics), mixed
    aggregators (the paper variant adds self-loops for `symadd` only: two graphs) - runs the layer followed by torch ops."""

    def __init__(self, hidden_dim: int, num_graph_layers: int, dropout: float, residual: bool, heads: int = 8, bases: int = 8,
                 softmax: bool = False, aggrs=None, num_features: int = 128, num_classes: int = 40):
        super().__init__()
        from .compat import EfficientGraphConv
        assert aggrs is not None                                                       # ref :108
        self.num_graph_layers = num_graph_layers
        self.embed = torch.nn.Sequential(torch.nn.Linear(num_features, hidden_dim))    # mlp([F, hidden]) (utils.py:33-43)
        self.convs = torch.nn.ModuleList(
            EfficientGraphConv(hidden_dim, hidden_dim, num_heads=heads, num_bases=bases, softmax_weights=softmax,
                               aggrs=list(aggrs)) for _ in range(num_graph_layers))
        self.bns = torch.nn.ModuleList(torch.nn.BatchNorm1d(hidden_dim) for _ in range(num_graph_layers))
        self.out = torch.nn.Linear(hidden_dim, num_classes)
        self.dropout, self.residual = dropout, residual
        self.heads, self.bases, self.softmax, self.aggrs = heads, bases, softmax, list(aggrs)

    def _fusable(self) -> bool:
        return not self.training and self.aggrs == ["symadd"] and not self.softmax

    def forward(self, x: Tensor, edge_index) -> Tensor:
        from .functional import egconv
        x = self.embed(x)
        if self._fusable():
            graph = self.convs[0]._graph(edge_index, x.size(0), True)                  # gcn_norm + self-loops, once
            for conv, bn in zip(self.convs, self.bns):
                scale, shift = fold_batchnorm(bn)
                # one aggregator: the paper's comb-weight order h * (B * A) + b * A + a is EGConv's h * (A * B) + a * B + b
                x = egconv(x, graph, torch.cat(list(conv.bases_weight), dim=1), conv.comb_weights.weight,
                           conv.comb_weights.bias, conv.bias, conv.num_heads, conv.num_bases, ["symnorm"], False,
                           conv.gemm_algo, 0, True, scale, shift, x if self.residual else None)
        else:
            for conv, bn in zip(self.convs, self.bns):                                 # ref :31-40
                identity = x
                x = F.relu(bn(conv(x, edge_index)))
                x = F.dropout(x, p=self.dropout, training=self.training)
                if self.residual:
                    x = x + identity
        return self.out(x).log_softmax(dim=-1)                                         # ref :42-43
