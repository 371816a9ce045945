"""`EGConv` - drop-in for the reference operator, running on the sm_100a kernels.

Mirrors /root/reference/experiments/optimized_layers.py:19-286: same constructor, attributes,
parameters / `state_dict` keys (`bases_weight`, `comb_weight.weight`, `comb_weight.bias`, `bias`),
initialisation, caching behaviour, error messages and `__repr__`; `forward(x, edge_index)` accepts
a LongTensor `[2, E]` (row 0 = source, row 1 = target) or a SparseTensor-like `adj_t` whose rows are
targets.  Everything after argument checking happens on the GPU; there is no CPU fallback.
"""
import math
from typing import Iterable, Optional

import torch
from torch import Tensor
from torch.nn import Linear, Parameter

from . import _lib
from .functional import check_storage_dtype, egconv
from .graph import GraphStructure, adjacency_to_csr

_AGGREGATORS = {"sum", "mean", "symnorm", "min", "max", "var", "std"}


class EGConv(torch.nn.Module):
    r"""Efficient Graph Convolution (`x_i' = ||_h sum_{agg} sum_b w_{i,h,agg,b} AGG_{j in N(i) u {i}} Theta_b x_j`).

    Args match the reference (optimized_layers.py:74-86): in_channels, out_channels,
    aggrs=("symnorm",), num_heads=8, num_bases=4, cached=False, add_self_loops=True, bias=True,
    sigmoid=False.  Extra keyword-only knobs of this implementation:
      gemm_algo: one of egc_b200.GEMM_* (projection kernels; default AUTO)
      deterministic: route min/max gradients without fp32 atomics
      storage_dtype: torch.float32 (default) or torch.bfloat16 - bf16 storage (round to nearest even) of the two gathered
        tensors, the basis rows and the backward's target-side streams; x, parameters, out, all accumulation and every
        gradient stay fp32.  Covers num_bases * out_channels / num_heads of 40..128, a multiple of 8; other shapes raise
        ValueError at the first forward.
    """

    def __init__(self, in_channels: int, out_channels: int, aggrs: Iterable[str] = ("symnorm",),
                 num_heads: int = 8, num_bases: int = 4, cached: bool = False, add_self_loops: bool = True,
                 bias: bool = True, sigmoid: bool = False, *, gemm_algo: int = _lib.GEMM_AUTO,
                 deterministic: bool = False, storage_dtype: torch.dtype = torch.float32, **kwargs):
        super().__init__()
        if out_channels % num_heads != 0:
            raise ValueError("out_channels must be divisible by the number of heads")          # ref :89-90
        aggrs = list(aggrs)
        for a in aggrs:
            if a not in _AGGREGATORS:
                raise ValueError("Unsupported aggregator: {}".format(a))                         # ref :92-94

        self.in_channels = in_channels
        self.out_channels = out_channels
        self.num_heads = num_heads
        self.num_bases = num_bases
        self.cached = cached
        self.add_self_loops = add_self_loops
        self.aggregators = aggrs
        self.sigmoid = sigmoid
        self.gemm_algo = gemm_algo
        self.deterministic = deterministic
        self.storage_dtype = check_storage_dtype(storage_dtype)
        self.node_dim = 0                                                                        # ref :87

        self.bases_weight = Parameter(torch.empty(in_channels, (out_channels // num_heads) * num_bases))
        self.comb_weight = Linear(in_channels, num_heads * num_bases * len(aggrs))
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):                                                                  # ref :117-122
        a = math.sqrt(6.0 / (self.bases_weight.size(-2) + self.bases_weight.size(-1)))           # PyG glorot
        with torch.no_grad():
            self.bases_weight.uniform_(-a, a)
            if self.bias is not None:
                self.bias.zero_()
        self.comb_weight.reset_parameters()
        self._cached_adj_t = None
        self._cached_edge_index = None

    # ------------------------------------------------------------------------------------------
    def _prepare(self, x: Tensor, edge_index) -> GraphStructure:
        """Graph preparation + caching with the reference's rules (ref :126-175)."""
        if isinstance(edge_index, GraphStructure):
            return edge_index
        symnorm = "symnorm" in self.aggregators
        is_tensor = isinstance(edge_index, Tensor) and edge_index.layout == torch.strided
        cache_attr = "_cached_edge_index" if is_tensor else "_cached_adj_t"
        cache = getattr(self, cache_attr)
        # symnorm branch consults the cache whenever it is filled (ref :129-130,144-145); the self-loop
        # branch only when `cached` (ref :161,170).  The cache is only ever filled when `cached`.  With
        # add_self_loops=False the reference has nothing to cache; here the CSR build itself is cached.
        if cache is not None and (symnorm or self.cached):
            return cache
        num_nodes = x.size(self.node_dim)
        if is_tensor:
            g = GraphStructure.from_edge_index(edge_index, num_nodes, symnorm, self.add_self_loops)
        else:
            rowptr, col, value, n_src = adjacency_to_csr(edge_index)
            g = GraphStructure.from_csr(rowptr, col, value, n_src, symnorm, self.add_self_loops)
        if self.cached:
            setattr(self, cache_attr, g)
        return g

    def forward(self, x: Tensor, edge_index, relu: bool = False, scale: Optional[Tensor] = None,
                shift: Optional[Tensor] = None, residual: Optional[Tensor] = None, dropout: float = 0.0,
                dropout_seed: Optional[Tensor] = None) -> Tensor:
        """Extensions (keyword arguments the reference does not have; used by `egc_b200.EGC` / `egc_b200.EGCBlock`): the
        stack around the layer fused into the aggregation kernel's epilogue -
        `relu(layer(x) * scale + shift) + residual`, with `scale` / `shift` an eval-mode BatchNorm folded to constants
        (`egc_b200.fold_batchnorm`).  Same values as the separate torch ops; the backward masks / scales the incoming
        gradient inside its first pass.  `dropout` = p > 0 (with relu=True): dropout after the ReLU in the same epilogue,
        applied whenever p > 0 - the caller decides on training mode, as with F.dropout(training=...); its mask is the
        counter-based one of `egc_b200.functional.egconv` (`dropout_seed`: see there), not torch's random stream."""
        if not x.is_cuda:
            raise RuntimeError("egc_b200.EGConv runs on CUDA (sm_100a) only; move the module and inputs to the GPU")
        if x.size(self.node_dim) == 0:                         # zero-node batch: empty output, zero parameter gradients
            keep = sum(p.sum() for p in self.parameters()) * 0.0
            return x.new_zeros((0, self.out_channels)) + keep + x.sum() * 0.0     # every epilogue of nothing is nothing
        graph = self._prepare(x, edge_index)
        flags = (_lib.BWD_DETERMINISTIC if self.deterministic else 0) | int(getattr(self, "bwd_flags", 0))
        return egconv(x, graph, self.bases_weight, self.comb_weight.weight, self.comb_weight.bias, self.bias,
                      self.num_heads, self.num_bases, self.aggregators, self.sigmoid, self.gemm_algo, flags, relu,
                      scale, shift, residual, self.storage_dtype, dropout, dropout_seed)

    def __repr__(self):                                                                          # ref :280-286
        return "{}({}, {}, {})".format(self.__class__.__name__, self.in_channels, self.out_channels,
                                       self.aggregators)
