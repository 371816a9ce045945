"""`EfficientGraphConv` - the paper variant of the layer (/root/reference/experiments/layers.py:11-228), as a
thin adapter over the same kernels as `EGConv`, plus the checkpoint converter between the two layouts
(SURVEY.md App. B).

Differences to `EGConv` that the adapter carries (not re-layouts):
  * aggregator names `symadd / add / mean / min / max / var / std`                      (ref layers.py:153-160)
  * self-loops (and `gcn_norm`) apply to `symadd` ONLY; every other aggregator sees the graph as
    given                                                                               (ref layers.py:167-188)
    -> with add_self_loops=True and mixed aggregators the layer runs the fused kernel once per graph and adds
       the two partial outputs (the combination is linear in the aggregates);
  * B separate basis matrices in a ParameterList, concatenated column-wise              (ref layers.py:56-65, 97-101)
  * comb-weight column order h * (B * A) + b * A + a (basis-major)                      (ref layers.py:106-129)
  * weight post-processing: softmax over B * A per head, sigmoid or hardtanh            (ref layers.py:112-125)
  * var / std on a SparseTensor input raise NotImplementedError                         (ref layers.py:222-224)
State-dict keys match the reference (`comb_weights.*`, `bases_weight.<b>`, `bias`), so its checkpoints load.
"""
from typing import Dict, Iterable, List, Optional

import torch
import torch.nn.functional as F
from torch import Tensor
from torch.nn import Linear, Parameter, ParameterList

from . import _lib
from .functional import aggregate_combine_autograd, project_autograd
from .graph import GraphStructure, adjacency_to_csr

_NAME_MAP = {"symadd": "symnorm", "add": "sum", "mean": "mean", "min": "min", "max": "max", "var": "var", "std": "std"}


def paper_to_egconv_perm(num_heads: int, num_bases: int, num_aggrs: int) -> Tensor:
    """perm with  egconv_cols = paper_cols[:, perm]:  EGConv column h*(A*B) + a*B + b  <-  paper column h*(B*A) + b*A + a."""
    h, b, a = num_heads, num_bases, num_aggrs
    idx = torch.arange(h * b * a).view(h, b, a)            # paper order
    return idx.permute(0, 2, 1).reshape(-1)                # read in (h, a, b) order


class EfficientGraphConv(torch.nn.Module):
    def __init__(self, in_channels: int, out_channels: int, num_heads: int, num_bases: int, softmax_weights: bool,
                 add_self_loops: bool = True, bias: bool = True, aggrs: Optional[Iterable[str]] = None,
                 cache: bool = False, sigmoid_weights: bool = False, hardtanh_weights: bool = False, **kwargs):
        super().__init__()
        assert aggrs is not None                                                              # ref layers.py:29
        self.in_channels, self.out_channels = in_channels, out_channels
        self.num_heads, self.num_bases = num_heads, num_bases
        self.softmax_weights, self.add_self_loops = softmax_weights, add_self_loops
        self.sigmoid_weights, self.hardtanh_weights = sigmoid_weights, hardtanh_weights
        if softmax_weights:                                                                   # ref layers.py:40-45
            assert not sigmoid_weights and not hardtanh_weights
        elif sigmoid_weights:
            assert not softmax_weights and not hardtanh_weights
        elif hardtanh_weights:
            assert not softmax_weights and not sigmoid_weights
        assert out_channels % num_heads == 0                                                  # ref layers.py:47
        self.aggregators: List[str] = list(aggrs)
        for a in self.aggregators:
            if a not in _NAME_MAP:
                raise ValueError(f'Unknown aggregator "{a}".')
        self.cache = cache
        self.gemm_algo = kwargs.pop("gemm_algo", _lib.GEMM_AUTO)
        if kwargs.pop("storage_dtype", torch.float32) != torch.float32:
            raise NotImplementedError("EfficientGraphConv: bf16 storage is not supported; use egc_b200.EGConv(..., "
                                      "storage_dtype=torch.bfloat16)")
        self.comb_weights = Linear(in_channels, num_heads * num_bases * len(self.aggregators))
        self.bases_weight = ParameterList([Parameter(torch.empty(in_channels, out_channels // num_heads))
                                           for _ in range(num_bases)])
        if bias:
            self.bias = Parameter(torch.zeros(out_channels))
        else:
            self.register_parameter("bias", None)
        self._cached = {}
        self.reset_parameters()

    def reset_parameters(self):                                                               # ref layers.py:83-88
        self.comb_weights.reset_parameters()
        for w in self.bases_weight:
            a = (6.0 / (w.size(-2) + w.size(-1))) ** 0.5
            with torch.no_grad():
                w.uniform_(-a, a)
        if self.bias is not None:
            with torch.no_grad():
                self.bias.zero_()
        self._cached = {}

    # ------------------------------------------------------------------------------------------
    def _graph(self, edge_index, num_nodes: int, symnorm: bool) -> GraphStructure:
        """symadd: gcn_norm(add_self_loops=self.add_self_loops); everything else: the graph untouched."""
        key = "sym" if symnorm else "raw"
        if self.cache and key in self._cached:
            return self._cached[key]
        loops = bool(self.add_self_loops) and symnorm
        if isinstance(edge_index, Tensor) and edge_index.layout == torch.strided:
            g = GraphStructure.from_edge_index(edge_index, num_nodes, symnorm, loops)
        else:
            rowptr, col, value, n_src = adjacency_to_csr(edge_index)
            g = GraphStructure.from_csr(rowptr, col, value, n_src, symnorm, loops)
        if self.cache:
            self._cached[key] = g
        return g

    def forward(self, x: Tensor, edge_index) -> Tensor:
        if not x.is_cuda:
            raise RuntimeError("egc_b200.EfficientGraphConv runs on CUDA (sm_100a) only")
        is_tensor = isinstance(edge_index, Tensor) and edge_index.layout == torch.strided
        if not is_tensor and any(a in ("var", "std") for a in self.aggregators):
            raise NotImplementedError                                                         # ref layers.py:222-224
        h, b, n_a = self.num_heads, self.num_bases, len(self.aggregators)
        bases_weight = torch.cat(list(self.bases_weight), dim=1)                              # [F_in, B*D], ref :97-101
        bases, lin = project_autograd(x, bases_weight, self.comb_weights.weight, self.comb_weights.bias, self.gemm_algo)
        if self.softmax_weights:                                                              # ref layers.py:112-120
            w = lin.view(-1, h, b * n_a).softmax(dim=-1).reshape(-1, h * b * n_a)
        elif self.sigmoid_weights:
            w = torch.sigmoid(lin)
        elif self.hardtanh_weights:
            w = F.hardtanh(lin)
        else:
            w = lin
        w = w.view(-1, h, b, n_a)                                                             # paper order [N, H, B, A]
        names = [_NAME_MAP[a] for a in self.aggregators]
        n = x.size(0)
        sym_idx = [i for i, a in enumerate(names) if a == "symnorm"]
        other_idx = [i for i, a in enumerate(names) if a != "symnorm"]
        # one fused call per distinct graph: symadd on the normalised (self-looped) graph, the rest on the raw graph
        groups = []
        # A valued adjacency also needs the split without self-loops: the symnorm graph carries D^-1/2 A D^-1/2 only,
        # while add / mean / max / min multiply by the adjacency values (ref layers.py:225 `matmul(adj_t, x, reduce=)`)
        valued = (not is_tensor) and (edge_index.has_value() if hasattr(edge_index, "has_value") else
                                      getattr(edge_index, "layout", None) == torch.sparse_csr)
        if sym_idx and other_idx and (self.add_self_loops or valued):
            groups = [(sym_idx, True), (other_idx, False)]
        else:
            groups = [(list(range(n_a)), bool(sym_idx))]
        out = None
        for k, (idx, symnorm) in enumerate(groups):
            g = self._graph(edge_index, n, symnorm)
            sel = w[:, :, :, idx].permute(0, 1, 3, 2).reshape(n, -1).contiguous()            # -> h*(A'*B) + a*B + b
            part = aggregate_combine_autograd(bases, sel, self.bias if k == 0 else None, g, h, b,
                                              [names[i] for i in idx])
            out = part if out is None else out + part
        return out

    def extra_repr(self):                                                                     # ref layers.py:141-146
        return (f"(In={self.in_channels}, Out={self.out_channels}, H={self.num_heads}, "
                + f"B={self.num_bases}, SL={self.add_self_loops}, SM={self.softmax_weights}, "
                + f"Bias={self.bias is not None})")


def convert_paper_state_dict(state: Dict[str, Tensor], num_heads: int, num_bases: int, num_aggrs: int) -> Dict[str, Tensor]:
    """`EfficientGraphConv.state_dict()` -> `EGConv.state_dict()` (SURVEY.md App. B): bases concatenated block-wise,
    comb-weight rows permuted from basis-major to aggregator-major.  The two layers compute the same function only
    where their self-loop rules coincide (add_self_loops=False, or `symadd` as the only aggregator) and without
    softmax / hardtanh weights - the caller is responsible for that."""
    perm = paper_to_egconv_perm(num_heads, num_bases, num_aggrs)
    out = {"bases_weight": torch.cat([state[f"bases_weight.{i}"] for i in range(num_bases)], dim=1),
           "comb_weight.weight": state["comb_weights.weight"][perm],
           "comb_weight.bias": state["comb_weights.bias"][perm]}
    if "bias" in state:
        out["bias"] = state["bias"]
    return out
