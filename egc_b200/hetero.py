"""Heterogeneous EGC layer (SURVEY.md section 8 f-2): drop-in for the reference's `REGConv`
(/root/reference/experiments/rmag/models.py:75-148) on the same CUDA kernels as `EGConv`.

Per node type t:       bases[t] = x[t] . bases_weight                       (shared basis weights, ref :116-118)
root term:             out[t]  = combine(root_combs[t](x[t]), bases[t])     (ref :120-132)
per relation (s,r,t):  out[t] += combine(rel_combs[s_r_t](x[t]), [mean | max over adj_t[(s,r,t)] of bases[s]])   (ref :134-146)

B200 execution: ONE tensor-core projection per node type produces bases[t] together with the combination weights of
the root term and of EVERY relation that targets t (their Linear layers are concatenated row-wise); the root term is
the fused aggregate+combine kernel on the identity graph; each relation is one launch of the same kernel on its
rectangular CSR (n_dst x n_src, aggregators mean + max, no self-loops) whose epilogue adds the running sum of the
previous terms (accumulate-into-output, no separate elementwise add), with the usual CSC backward.
State-dict keys, parameter shapes and initialisation follow the reference.
"""
from typing import Dict, Optional, Sequence, Tuple

import torch
from torch import Tensor
from torch.nn import Linear, ModuleDict, Parameter

from . import _lib
from .functional import aggregate_combine_autograd, project_autograd
from .graph import GraphStructure, adjacency_to_csr

# ogbn-mag schema of the reference (rmag/models.py:17-26)
NODE_TYPES = ("author", "field_of_study", "institution", "paper")
EDGE_TYPES = (
    ("author", "affiliated_with", "institution"),
    ("institution", "to", "author"),
    ("author", "writes", "paper"),
    ("paper", "to", "author"),
    ("paper", "cites", "paper"),
    ("paper", "has_topic", "field_of_study"),
    ("field_of_study", "to", "paper"),
)
EdgeType = Tuple[str, str, str]


class REGConv(torch.nn.Module):
    def __init__(self, in_channels: int, out_channels: int, num_heads: int, num_bases: int,
                 node_types: Sequence[str] = NODE_TYPES, edge_types: Sequence[EdgeType] = EDGE_TYPES,
                 cached: bool = True, gemm_algo: int = _lib.GEMM_AUTO, *, storage_dtype: torch.dtype = torch.float32,
                 deterministic: bool = False):
        """deterministic: route the max gradients of the relations without fp32 atomics, so the backward gives the same
        bits on every run (as `EGConv(..., deterministic=True)`)."""
        super().__init__()
        if storage_dtype != torch.float32:
            raise NotImplementedError("REGConv: bf16 storage is not supported; use storage_dtype=torch.float32")
        if out_channels % num_heads != 0:
            raise ValueError("out_channels must be divisible by the number of heads")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.num_heads, self.num_bases = num_heads, num_bases
        self.node_types, self.edge_types = tuple(node_types), tuple(tuple(k) for k in edge_types)
        self.cached, self.gemm_algo = cached, gemm_algo
        self.deterministic = deterministic
        self.bases_weight = Parameter(torch.empty(in_channels, (out_channels // num_heads) * num_bases))
        self.rel_combs = ModuleDict({f"{k[0]}_{k[1]}_{k[2]}": Linear(in_channels, 2 * num_heads * num_bases)
                                     for k in self.edge_types})                                  # ref :89-97
        self.root_combs = ModuleDict({k: Linear(in_channels, num_heads * num_bases) for k in self.node_types})
        self._graphs: Dict[object, GraphStructure] = {}
        self.reset_parameters()

    def reset_parameters(self):                                                                  # ref :105-110
        a = (6.0 / (self.bases_weight.size(-2) + self.bases_weight.size(-1))) ** 0.5             # PyG glorot
        with torch.no_grad():
            self.bases_weight.uniform_(-a, a)
        for lin in list(self.rel_combs.values()) + list(self.root_combs.values()):
            lin.reset_parameters()
        self._graphs = {}

    # ------------------------------------------------------------------------------------------
    def _identity(self, n: int, device) -> GraphStructure:
        key = ("identity", n, str(device))
        g = self._graphs.get(key)
        if g is None:
            g = GraphStructure.from_prepared(torch.arange(n + 1, device=device), torch.arange(n, device=device), n)
            self._graphs[key] = g
        return g

    def _relation(self, key: EdgeType, adj_t, device) -> GraphStructure:
        if isinstance(adj_t, GraphStructure):
            return adj_t
        # the reference does no caching (rmag/models.py:134); here the CSR -> device structure build is cached per edge
        # type AND per adjacency object, so a different adjacency passed under the same key is rebuilt, never reused
        hit = self._graphs.get(key) if self.cached else None
        if hit is not None and hit[0] is adj_t:
            return hit[1]
        rowptr, col, value, n_src = adjacency_to_csr(adj_t)
        g = GraphStructure.from_csr(rowptr.to(device), col.to(device), value.to(device) if value is not None else None,
                                    n_src, False, False)
        if self.cached:
            self._graphs[key] = (adj_t, g)
        return g

    def forward(self, x_dict: Dict[str, Tensor], adj_t_dict) -> Dict[str, Tensor]:
        """`adj_t_dict`: {(src, rel, dst): adj_t} over whole node sets, or an `egc_b200.dist.PartitionedHeteroGraph` with
        `x_dict` holding this rank's rows of every type (`row_range`): the result is then this rank's rows of the
        single-GPU layer's output, and the parameter gradients are summed over the ranks."""
        from .dist import PartitionedHeteroGraph
        phg = adj_t_dict if isinstance(adj_t_dict, PartitionedHeteroGraph) else None
        keys = phg.edge_types if phg is not None else list(adj_t_dict)
        h, b = self.num_heads, self.num_bases
        hb = h * b
        bwd_flags = _lib.BWD_DETERMINISTIC if self.deterministic else 0
        names, params = map(list, zip(*self.named_parameters()))
        if phg is not None:
            unknown = [k for k in keys if k not in self.edge_types]
            if unknown:
                raise ValueError(f"REGConv: relations {unknown} of the partitioned graph are not among the layer's edge types")
            if set(x_dict) != set(phg.types):
                raise ValueError(f"REGConv: x_dict has node types {sorted(x_dict)}, the partitioned graph {sorted(phg.types)}")
            key, n_flat = id(self), sum(p.numel() for p in params)
            params = phg.replicated(key, params)        # gradients summed over the ranks
        P = dict(zip(names, params))
        # relations grouped by the node type they write to, in adj_t_dict order (the reference's accumulation order)
        incoming = {t: [k for k in keys if k[2] == t] for t in x_dict}
        bases, weights = {}, {}
        for t, x in x_dict.items():
            if not x.is_cuda:
                raise RuntimeError("egc_b200.REGConv runs on CUDA (sm_100a) only; move the module and inputs to the GPU")
            lins = [f"root_combs.{t}"] + [f"rel_combs.{k[0]}_{k[1]}_{k[2]}" for k in incoming[t]]
            w_cat = torch.cat([P[n + ".weight"] for n in lins], 0) if len(lins) > 1 else P[lins[0] + ".weight"]
            b_cat = torch.cat([P[n + ".bias"] for n in lins], 0) if len(lins) > 1 else P[lins[0] + ".bias"]
            bases[t], weights[t] = project_autograd(x, P["bases_weight"], w_cat, b_cat, self.gemm_algo)
        # source tables: the own rows, or [own | halo] rows of every type after the halo exchange
        src = phg.exchange(key, n_flat, bases) if phg is not None else bases
        out = {}
        for t, x in x_dict.items():
            w_root = weights[t][:, :hb].contiguous()
            if x.size(0) == 0:                                  # a node type without nodes (ref handles empty tensors)
                out[t] = x.new_zeros((0, self.out_channels)) + weights[t].sum() * 0.0
                continue
            own = src[t] if src[t].size(0) == x.size(0) else src[t][:x.size(0)]
            out[t] = aggregate_combine_autograd(own, w_root, None, self._identity(x.size(0), x.device), h, b, ("sum",))
            for i, k in enumerate(incoming[t]):
                if src[k[0]].size(0) == 0:                      # relation from an empty node type: contributes nothing
                    continue
                g = phg.graphs[k] if phg is not None else self._relation(k, adj_t_dict[k], x.device)
                if g.n_dst != x.size(0) or g.n_src != src[k[0]].size(0):
                    raise ValueError(f"adjacency of {k} is {g.n_dst} x {g.n_src}, expected {x.size(0)} x {src[k[0]].size(0)}")
                w_rel = weights[t][:, hb + 2 * hb * i: hb + 2 * hb * (i + 1)].contiguous()
                # root_combined[t] += ... (ref :146): the running sum is the `add` input of the kernel's epilogue
                out[t] = aggregate_combine_autograd(src[k[0]], w_rel, None, g, h, b, ("mean", "max"), bwd_flags,
                                                    add=out[t])
        if phg is not None:
            phg.end_forward(key, bases[phg.types[0]].size(1), n_flat)
        return out

    def __repr__(self):
        return f"{self.__class__.__name__}({self.in_channels}, {self.out_channels}, heads={self.num_heads}, bases={self.num_bases})"
