"""Autograd boundary between PyTorch and the C-ABI kernels of `libegc_b200.so`.

`egconv(x, graph, bases_weight, comb_weight, comb_bias, bias, ...)` computes what
/root/reference/experiments/optimized_layers.py:177-210 computes after graph preparation
(projections -> multi-aggregator message passing -> per-head combination -> bias) and its backward is
the hand-written one (CSR pass, atomic-free CSC pass, projection gradients).  PyTorch only owns
the memory and the stream.
"""
import ctypes
from typing import Optional, Sequence

import torch
from torch import Tensor

from . import _lib
from ._lib import LayerDesc, check, ptr
from .graph import GraphStructure, _stream, _ws


def make_desc(graph: GraphStructure, heads: int, bases: int, dim: int, aggrs: Sequence[str], sigmoid: bool,
              relu: bool = False) -> LayerDesc:
    if len(aggrs) < 1 or len(aggrs) > _lib.EGC_MAX_AGGR:
        raise ValueError(f"between 1 and {_lib.EGC_MAX_AGGR} aggregators are supported, got {len(aggrs)}")
    d = LayerDesc()
    d.n_dst, d.n_src = graph.n_dst, graph.n_src
    d.heads, d.bases, d.dim = heads, bases, dim
    d.n_aggr = len(aggrs)
    for i, a in enumerate(aggrs):
        if a not in _lib.AGGR_CODES:
            raise ValueError(f'Unknown aggregator "{a}".')           # ref :246
        d.aggr[i] = _lib.AGGR_CODES[a]
    d.sigmoid = int(bool(sigmoid))
    d.relu = int(bool(relu))
    return d


def _require_cuda_f32(name: str, t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError(f"egc_b200: `{name}` must be a CUDA tensor - this library has no CPU path")
    if t.dtype != torch.float32:
        raise TypeError(f"egc_b200: `{name}` must be float32 (got {t.dtype})")
    return t.contiguous()


STORAGE_DTYPES = (torch.float32, torch.bfloat16)


def check_storage_dtype(storage_dtype) -> torch.dtype:
    if storage_dtype not in STORAGE_DTYPES:
        raise ValueError(f"storage_dtype must be torch.float32 or torch.bfloat16 (got {storage_dtype})")
    return storage_dtype


def check_bf16_layer(desc: LayerDesc, graph: GraphStructure) -> None:
    """Raises ValueError for the layers the bf16-storage kernels do not cover (include/egc_b200.h, the *_bf16 entry points)."""
    bd, hd = desc.bases * desc.dim, desc.heads * desc.dim
    hab = desc.heads * desc.n_aggr * desc.bases
    if bd % 8 != 0 or not 40 <= bd <= 128:
        raise ValueError(f"storage_dtype=torch.bfloat16 needs num_bases * out_channels / num_heads between 40 and 128 and a "
                         f"multiple of 8 (got {bd})")
    if hd > (512 if desc.dim % 4 == 0 else 128):
        raise ValueError(f"storage_dtype=torch.bfloat16: out_channels={hd} is too wide for one pass of the bf16 kernels")
    # per-warp staging of the row-block kernel: aggregates, 8 rows of weights, column ids and weights of 384 nnz (floats)
    if (desc.n_aggr * bd + 3) // 4 * 4 + (8 * hab + 3) // 4 * 4 + 768 > 72 * 1024 // 32:
        raise ValueError(f"storage_dtype=torch.bfloat16: {desc.n_aggr} aggregators x {bd} basis values and {hab} weights per "
                         "row are too wide for one pass of the bf16 kernels")
    if graph.val_lin is not None:
        raise ValueError("storage_dtype=torch.bfloat16 does not support an adjacency with edge values (without symnorm)")


def check_dropout(p) -> float:
    """The drop probability of the fused dropout: 0 <= p < 1 (0 = no dropout), else ValueError."""
    p = float(p)
    if not 0.0 <= p < 1.0:
        raise ValueError(f"dropout probability has to be in [0, 1), got {p}")
    return p


def dropout_constants(p: float):
    """(threshold, scale) of the fused dropout (include/egc_b200.h, egc_dropout): p is rounded to fp32 first, as the C
    call receives it; keep iff the Philox word < threshold = floor((1 - p) * 2^32), kept values times scale = fp32(1 / (1 - p))."""
    keep = 1.0 - float(ctypes.c_float(p).value)
    return min(int(keep * 4294967296.0), 0xFFFFFFFF), float(ctypes.c_float(1.0 / keep).value)


def check_dropout_seed(seed: Tensor, device) -> Tensor:
    """A caller-supplied seed of the fused dropout: one int64 word on `device` (the kernel reads it from there)."""
    if not (isinstance(seed, Tensor) and seed.is_cuda and seed.dtype == torch.int64 and seed.numel() == 1 and
            seed.device == torch.device(device)):
        raise ValueError("dropout_seed must be a one-element int64 tensor on the device of x")
    return seed.contiguous()


def draw_dropout_seed(device) -> Tensor:
    """The per-call seed of the fused dropout: one draw from the default CUDA generator of `device`, so it follows
    torch.manual_seed and - inside a CUDA graph - is drawn afresh at every replay.  Every layer call that applies dropout
    draws exactly one seed, in layer order."""
    return torch.randint(0, 2 ** 63 - 1, (1,), dtype=torch.int64, device=device)


def project(x: Tensor, bases_weight: Tensor, comb_weight: Tensor, comb_bias: Optional[Tensor], sigmoid: bool,
            algo: int = _lib.GEMM_AUTO, bases_out: Optional[Tensor] = None, storage_dtype: torch.dtype = torch.float32):
    """bases = x @ W_b ; weightings = act(x @ W_c^T + b_c)   (ref :180-184).  `bases_out` lets a caller
    provide the (row-prefix of a larger) buffer the basis rows are written to.  storage_dtype=torch.bfloat16: `bases` is
    stored as bf16 (round to nearest even from the fp32 product); the weightings stay fp32."""
    lib = _lib.load()
    n, f_in = x.shape
    bd, hab = bases_weight.shape[1], comb_weight.shape[0]
    bases = bases_out if bases_out is not None else torch.empty((n, bd), dtype=storage_dtype, device=x.device)
    weightings = torch.empty((n, hab), dtype=torch.float32, device=x.device)
    fn = lib.egc_project_fwd_bf16 if bases.dtype == torch.bfloat16 else lib.egc_project_fwd
    if n > 0:
        check(fn(ptr(x), ptr(bases_weight), ptr(comb_weight), ptr(comb_bias), n, f_in, bd, hab,
                 int(sigmoid), ptr(bases), ptr(weightings), algo, _stream()), fn.__name__)
    return bases, weightings


def alloc_aggregate_outputs(desc: LayerDesc, device, want_out=True, want_agg=False, want_arg=False, want_saved=False):
    lib = _lib.load()
    n, bd, hd = desc.n_dst, desc.bases * desc.dim, desc.heads * desc.dim
    out = torch.empty((n, hd), dtype=torch.float32, device=device) if want_out else None
    agg = torch.empty((n, desc.n_aggr, bd), dtype=torch.float32, device=device) if want_agg else None
    arg = torch.empty((n, desc.n_aggr, bd), dtype=torch.int32, device=device) if want_arg else None
    saved = saved_arg = None
    if want_saved:
        saved = torch.empty((n, lib.egc_saved_slots(desc), bd), dtype=torch.float32, device=device)
        n_arg = lib.egc_saved_arg_slots(desc)
        saved_arg = torch.empty((n, n_arg, bd), dtype=torch.int32, device=device) if n_arg else None
    return out, agg, arg, saved, saved_arg


def aggregate_combine(desc: LayerDesc, graph: GraphStructure, bases: Tensor, weightings: Optional[Tensor],
                      bias: Optional[Tensor], want_out: bool = True, want_agg: bool = False, want_arg: bool = False,
                      want_saved: bool = False, row_subset: Optional[Tensor] = None, use_plan: bool = True,
                      outputs=None, epilogue=None, dropout=None):
    """Fused SpMM + combination (ref :191-208).  Returns (out, agg, arg, saved, saved_arg); unrequested ones
    are None.  `saved` / `saved_arg` are what the backward pass consumes (see include/egc_b200.h).
    `row_subset` (int32 device tensor) restricts the row tasks; `outputs` reuses buffers of a previous call.
    `epilogue` = (scale, shift, add[, agg_init]) tensors or None each: the fused tail  y*scale+shift -> relu (desc.relu) ->
    +add; agg_init [n_dst, A, B*D] = partial aggregates of an earlier call over another entry subset (sum / symnorm only).
    `dropout` = (seed [1] int64 CUDA tensor, p, global id of row 0) or None: dropout after the ReLU (egc_dropout)."""
    lib = _lib.load()
    dev = bases.device
    bf16 = bases.dtype == torch.bfloat16
    if bf16:
        check_bf16_layer(desc, graph)
        if row_subset is not None or not use_plan or (epilogue is not None and len(epilogue) > 3 and epilogue[3] is not None):
            raise NotImplementedError("bf16 basis rows: row subsets, plan-less calls and agg_init are not supported")
    if outputs is None:
        outputs = alloc_aggregate_outputs(desc, dev, want_out, want_agg, want_arg, want_saved)
    out, agg, arg, saved, saved_arg = outputs
    if desc.n_dst == 0:                                   # no target rows: empty outputs (the reference returns [0, F])
        return outputs
    if desc.n_src == 0:
        raise ValueError("egc_b200: aggregation over a graph with target rows but no source nodes")
    plan = graph.plan.struct if use_plan else None
    nbytes = lib.egc_aggregate_fwd_workspace_bytes(desc, plan)
    ws = _ws(nbytes, dev)
    drop = None
    if dropout is not None:
        seed, p, row_offset = dropout
        drop = _lib.Dropout(seed.data_ptr(), p, int(row_offset))
    if bf16:
        epi = None
        if epilogue is not None and any(t is not None for t in epilogue):
            epi = _lib.Epilogue(*(t.data_ptr() if t is not None else None for t in tuple(epilogue)[:3]), None)
        check(lib.egc_aggregate_fwd_bf16_dropout(desc, ptr(graph.rowptr), ptr(graph.col), ptr(graph.val_sym), plan,
                                                 ptr(bases), ptr(weightings), ptr(bias), epi, drop, ptr(out), ptr(agg),
                                                 ptr(arg), ptr(saved), ptr(saved_arg), ptr(ws), nbytes, _stream()),
              "egc_aggregate_fwd_bf16")
        return outputs
    n_subset = int(row_subset.numel()) if row_subset is not None else 0
    if row_subset is not None and n_subset == 0 and not (use_plan and graph.plan.n_long):
        return outputs
    epi = None
    if epilogue is not None and any(t is not None for t in epilogue):
        scale, shift, add, agg_init = tuple(epilogue) + (None,) * (4 - len(epilogue))
        epi = _lib.Epilogue(*(t.data_ptr() if t is not None else None for t in (scale, shift, add, agg_init)))
    check(lib.egc_aggregate_fwd_dropout(desc, ptr(graph.rowptr), ptr(graph.col), ptr(graph.val_sym), ptr(graph.val_lin),
                                        plan, ptr(bases), ptr(weightings), ptr(bias), epi, drop,
                                        ptr(row_subset) if n_subset else None, n_subset, ptr(out), ptr(agg), ptr(arg),
                                        ptr(saved), ptr(saved_arg), ptr(ws), nbytes, _stream()),
          "egc_aggregate_fwd")
    return outputs


def aggregate_backward(desc: LayerDesc, graph: GraphStructure, bases: Tensor, weightings: Tensor, saved: Tensor,
                       saved_arg: Optional[Tensor], grad_out: Tensor, want_bias: bool, flags: int = 0,
                       want_lin_colsum: bool = False, out_bias: Optional[Tensor] = None,
                       out_lin_colsum: Optional[Tensor] = None, col_split: Optional[int] = None, between_phases=None,
                       out_act: Optional[Tensor] = None, epi_scale: Optional[Tensor] = None,
                       tstreams_out: Optional[Tensor] = None):
    """Backward of `aggregate_combine`: returns (d_weightings [n_dst, HAB], d_bases [n_src, BD], d_bias|None) and,
    with `want_lin_colsum`, a 4th item: the column sums of d_weightings (= gradient of the comb-weight bias).
    `col_split` (row-partitioned callers): run the source columns >= col_split first (EGC_BWD_COLS_HEAD), call
    `between_phases(d_bases)` - typically the NVLink push of those rows on a side stream - then the rest (COLS_TAIL).
    `out_act`: the forward's post-activation output (before an epilogue `add`) when the layer carries the fused ReLU
    (desc.relu): grad_out is masked with it; `epi_scale`: the fused affine epilogue's scale (multiplies the gradient).
    `tstreams_out` [>= n_dst rows, L * B * D] (row-partitioned callers that exchange the target-side streams): pass 1 only
    (EGC_BWD_PASS1_ONLY) - the streams of the n_dst targets are written to its first rows, d_bases is returned as None
    and comes from `aggregate_backward_cols` once the peers' rows have arrived."""
    lib = _lib.load()
    dev = bases.device
    bd, hab = desc.bases * desc.dim, desc.heads * desc.n_aggr * desc.bases
    pass1_only = tstreams_out is not None
    if pass1_only:
        flags |= _lib.BWD_PASS1_ONLY
    if desc.n_dst == 0:                                   # no target rows: every gradient is zero
        d_w = torch.zeros((0, hab), dtype=torch.float32, device=dev)
        d_bases = torch.zeros((desc.n_src, bd), dtype=torch.float32, device=dev)
        d_bias = (out_bias.zero_() if out_bias is not None else
                  torch.zeros(desc.heads * desc.dim, dtype=torch.float32, device=dev)) if want_bias else None
        if want_lin_colsum:
            return d_w, d_bases, d_bias, (out_lin_colsum.zero_() if out_lin_colsum is not None else
                                          torch.zeros(hab, dtype=torch.float32, device=dev))
        return d_w, d_bases, d_bias
    bf16 = bases.dtype == torch.bfloat16
    if pass1_only and tstreams_out.dtype != bases.dtype:
        raise TypeError(f"tstreams_out must have the dtype of bases ({bases.dtype}, got {tstreams_out.dtype})")
    if not pass1_only:
        graph.ensure_csc()
    d_w = torch.empty((desc.n_dst, hab), dtype=torch.float32, device=dev)
    d_bases = torch.empty((desc.n_src, bd), dtype=torch.float32, device=dev) if not pass1_only else None
    d_bias = (out_bias if out_bias is not None else
              torch.empty(desc.heads * desc.dim, dtype=torch.float32, device=dev)) if want_bias else None
    d_lin_sum = (out_lin_colsum if out_lin_colsum is not None else
                 torch.empty(hab, dtype=torch.float32, device=dev)) if want_lin_colsum else None
    csc_plan = graph.csc_plan.struct if not pass1_only else None
    if bf16:
        nbytes = lib.egc_aggregate_bwd_bf16_workspace_bytes(desc, csc_plan, flags)
    else:
        nbytes = lib.egc_aggregate_bwd_workspace_bytes(desc, csc_plan, flags)
    ws = _ws(nbytes, dev)
    def call(phase_flags):
        if bf16:
            csc = (None,) * 4 if pass1_only else (ptr(graph.colptr), ptr(graph.rowidx), ptr(graph.csr2csc), ptr(graph.csc_val_sym))
            check(lib.egc_aggregate_bwd_bf16_partitioned(desc, ptr(graph.rowptr), ptr(graph.col), *csc, csc_plan, ptr(bases),
                                                         ptr(weightings), ptr(saved), ptr(saved_arg), ptr(grad_out),
                                                         ptr(out_act), ptr(epi_scale), ptr(d_w), ptr(d_bases), ptr(d_bias),
                                                         ptr(d_lin_sum), ptr(tstreams_out), flags | phase_flags,
                                                         int(col_split or 0), ptr(ws), nbytes, _stream()),
                  "egc_aggregate_bwd_bf16_partitioned")
            return
        check(lib.egc_aggregate_bwd(desc, ptr(graph.rowptr), ptr(graph.col), ptr(graph.val_lin),
                                    *((None,) * 5 if pass1_only else (ptr(graph.colptr), ptr(graph.rowidx), ptr(graph.csr2csc),
                                                                      ptr(graph.csc_val_sym), ptr(graph.csc_val_lin))),
                                    csc_plan, ptr(bases), ptr(weightings), ptr(saved), ptr(saved_arg),
                                    ptr(grad_out), ptr(out_act), ptr(epi_scale), ptr(d_w), ptr(d_bases), ptr(d_bias), ptr(d_lin_sum),
                                    ptr(tstreams_out), flags | phase_flags,
                                    int(col_split or 0), ptr(ws), nbytes, _stream()),
              "egc_aggregate_bwd")

    if col_split is None:
        call(0)
    else:
        call(_lib.BWD_COLS_HEAD)
        if between_phases is not None:
            between_phases(d_bases)
        call(_lib.BWD_COLS_TAIL)
    if want_lin_colsum:
        return d_w, d_bases, d_bias, d_lin_sum
    return d_w, d_bases, d_bias



def aggregate_backward_cols(desc_t: LayerDesc, graph_t: GraphStructure, tstreams: Tensor, bases: Optional[Tensor],
                            d_bases: Optional[Tensor] = None, accumulate: bool = False) -> Tensor:
    """Pass 2 of the backward alone (`egc_aggregate_bwd_cols`): `graph_t` is the TRANSPOSED local adjacency in CSR form
    (rows = own source columns, column ids = rows of `tstreams`, values = the entries' weights), `desc_t` its descriptor
    (n_dst of the descriptor = rows of `tstreams`, n_src = rows of `graph_t`).  Returns d_bases [n_src, B * D].
    A bf16 `tstreams` (from a bf16 pass 1) runs `egc_aggregate_bwd_cols_bf16`: `bases` are then the bf16 basis rows and
    d_bases stays fp32."""
    lib = _lib.load()
    dev = tstreams.device
    bd = desc_t.bases * desc_t.dim
    bf16 = tstreams.dtype == torch.bfloat16
    if bf16 and bases is not None and bases.dtype != torch.bfloat16:
        raise TypeError(f"bf16 target-side streams need bf16 basis rows (got {bases.dtype})")
    if d_bases is None:
        d_bases = torch.empty((desc_t.n_src, bd), dtype=torch.float32, device=dev)
    if desc_t.n_src == 0:
        return d_bases
    plan = graph_t.plan.struct
    nbytes = lib.egc_aggregate_bwd_cols_workspace_bytes(desc_t, plan)
    ws = _ws(nbytes, dev)
    flags = _lib.BWD_ACCUMULATE if accumulate else 0
    if bf16:
        check(lib.egc_aggregate_bwd_cols_bf16(desc_t, ptr(graph_t.rowptr), ptr(graph_t.col), ptr(graph_t.val_sym), plan,
                                              ptr(tstreams), ptr(bases), ptr(d_bases), flags, ptr(ws), nbytes, _stream()),
              "egc_aggregate_bwd_cols_bf16")
        return d_bases
    check(lib.egc_aggregate_bwd_cols(desc_t, ptr(graph_t.rowptr), ptr(graph_t.col), ptr(graph_t.val_sym), ptr(graph_t.val_lin),
                                     plan, ptr(tstreams), ptr(bases), ptr(d_bases), flags, ptr(ws), nbytes, _stream()),
          "egc_aggregate_bwd_cols")
    return d_bases

def project_backward(x: Tensor, bases_weight: Tensor, comb_weight: Tensor, d_bases: Tensor, d_lin: Tensor,
                     need_x: bool, need_wb: bool, need_wc: bool, need_bc: bool, algo: int = _lib.GEMM_AUTO,
                     out_wb: Optional[Tensor] = None, out_wc: Optional[Tensor] = None):
    """Autograd of `project`: returns (d_x, d_bases_weight, d_comb_weight, d_comb_bias), None where not needed."""
    lib = _lib.load()
    dev = x.device
    n, f_in = x.shape
    bd, hab = bases_weight.shape[1], comb_weight.shape[0]
    d_x = torch.empty_like(x) if need_x else None
    d_wb = (out_wb if out_wb is not None else torch.empty_like(bases_weight)) if need_wb else None
    d_wc = (out_wc if out_wc is not None else torch.empty_like(comb_weight)) if need_wc else None
    d_bc = torch.empty(hab, dtype=torch.float32, device=dev) if need_bc else None
    if n == 0:                                            # no rows: the parameter gradients are zero
        for t in (d_wb, d_wc, d_bc):
            if t is not None:
                t.zero_()
        return d_x, d_wb, d_wc, d_bc
    nbytes = lib.egc_project_bwd_workspace_bytes(n, f_in, bd, hab)
    ws = _ws(nbytes, dev)
    check(lib.egc_project_bwd(ptr(x), ptr(bases_weight), ptr(comb_weight), ptr(d_bases), ptr(d_lin), n, f_in, bd, hab,
                              ptr(d_x), ptr(d_wb), ptr(d_wc), ptr(d_bc), algo, ptr(ws), nbytes, _stream()),
          "egc_project_bwd")
    return d_x, d_wb, d_wc, d_bc


class _EGConvFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, bases_weight, comb_weight, comb_bias, bias, graph, heads, num_bases, aggrs, sigmoid, algo,
                bwd_flags, grad_mode=True, relu=False, epi_scale=None, epi_shift=None, epi_add=None,
                storage_dtype=torch.float32, dropout=0.0, dropout_seed=None):
        x = _require_cuda_f32("x", x)
        dropout = check_dropout(dropout)
        if dropout > 0.0:
            if not relu:
                raise ValueError("the fused dropout follows the fused ReLU: dropout > 0 needs relu=True")
            if epi_scale is not None or epi_shift is not None or epi_add is not None:
                raise ValueError("the fused dropout cannot be combined with `scale`, `shift` or `residual`")
        epi_scale, epi_shift = _require_cuda_f32("scale", epi_scale), _require_cuda_f32("shift", epi_shift)
        epi_add = _require_cuda_f32("residual", epi_add)
        if (epi_scale is None) != (epi_shift is None):
            raise ValueError("the fused affine epilogue needs both `scale` and `shift`")
        if (epi_scale is not None and epi_scale.requires_grad) or (epi_shift is not None and epi_shift.requires_grad):
            raise ValueError("`scale` / `shift` of the fused epilogue are constants (a folded eval-mode BatchNorm): detach them")
        bases_weight = _require_cuda_f32("bases_weight", bases_weight)
        comb_weight = _require_cuda_f32("comb_weight.weight", comb_weight)
        comb_bias = _require_cuda_f32("comb_weight.bias", comb_bias)
        bias = _require_cuda_f32("bias", bias)
        if x.dim() != 2 or x.size(0) != graph.n_src or graph.n_src != graph.n_dst:
            raise ValueError(f"x must be [num_nodes, in_channels] with num_nodes == {graph.n_src}")
        dim = bases_weight.size(1) // num_bases
        desc = make_desc(graph, heads, num_bases, dim, aggrs, sigmoid, relu)
        if storage_dtype == torch.bfloat16:
            check_bf16_layer(desc, graph)
        # needs_input_grad ignores torch.no_grad(); the caller samples the grad mode before apply()
        needs_grad = grad_mode and any(ctx.needs_input_grad[:5])
        with torch.cuda.device(x.device):
            bases, weightings = project(x, bases_weight, comb_weight, comb_bias, sigmoid, algo, storage_dtype=storage_dtype)
            hd = heads * dim
            for name, t, shape in (("scale", epi_scale, (hd,)), ("shift", epi_shift, (hd,)), ("residual", epi_add, (graph.n_dst, hd))):
                if t is not None and tuple(t.shape) != shape:
                    raise ValueError(f"`{name}` of the fused epilogue must have shape {shape} (got {tuple(t.shape)})")
            drop = None
            if dropout > 0.0:
                seed = check_dropout_seed(dropout_seed, x.device) if dropout_seed is not None else draw_dropout_seed(x.device)
                drop = (seed, dropout, 0)
            out, _, _, saved, saved_arg = aggregate_combine(desc, graph, bases, weightings, bias, want_saved=needs_grad,
                                                            epilogue=(epi_scale, epi_shift, epi_add), dropout=drop)
        if needs_grad or (epi_add is not None and ctx.needs_input_grad[16] and grad_mode):
            # the fused ReLU's backward needs the sign of the post-activation value: `out` itself (the next layer's input
            # anyway, nothing extra is written) - or out - add when a residual was added after the activation
            act = None
            if relu:
                act = out if epi_add is None else out - epi_add
            if dropout > 0.0:
                # out > 0 exactly where the ReLU was open and the element kept: pass 1's mask-and-scale with scale = k is
                # the exact ReLU + dropout backward, and no mask is stored
                epi_scale = torch.full((heads * dim,), dropout_constants(dropout)[1], dtype=torch.float32, device=x.device)
            ctx.save_for_backward(x, bases_weight, comb_weight, bases, weightings, saved, saved_arg, act, epi_scale)
        ctx.graph, ctx.desc, ctx.algo, ctx.bwd_flags = graph, desc, algo, bwd_flags
        ctx.has_bias, ctx.has_comb_bias = bias is not None, comb_bias is not None
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, bases_weight, comb_weight, bases, weightings, saved, saved_arg, out_act, epi_scale = ctx.saved_tensors
        grad_out = _require_cuda_f32("grad_out", grad_out)
        need_x, need_wb, need_wc, need_bc, need_b = ctx.needs_input_grad[:5]
        d_add = grad_out if ctx.needs_input_grad[16] else None      # the residual is added after the activation
        if saved is None:                                           # only the residual needed a gradient
            return (None,) * 16 + (d_add, None, None, None)
        with torch.cuda.device(x.device):
            want_bc = bool(need_bc and ctx.has_comb_bias)
            d_w, d_bases, d_bias, d_bc = aggregate_backward(ctx.desc, ctx.graph, bases, weightings, saved, saved_arg,
                                                            grad_out, need_b and ctx.has_bias, ctx.bwd_flags,
                                                            want_lin_colsum=True, out_act=out_act, epi_scale=epi_scale)
            d_x, d_wb, d_wc, _ = project_backward(x, bases_weight, comb_weight, d_bases, d_w, need_x, need_wb,
                                                  need_wc, False, ctx.algo)
            if not want_bc:
                d_bc = None
        return (d_x, d_wb, d_wc, d_bc, d_bias) + (None,) * 11 + (d_add, None, None, None)


def egconv(x: Tensor, graph: GraphStructure, bases_weight: Tensor, comb_weight: Tensor, comb_bias: Optional[Tensor],
           bias: Optional[Tensor], num_heads: int, num_bases: int, aggrs: Sequence[str], sigmoid: bool = False,
           algo: int = _lib.GEMM_AUTO, bwd_flags: int = 0, relu: bool = False, scale: Optional[Tensor] = None,
           shift: Optional[Tensor] = None, residual: Optional[Tensor] = None,
           storage_dtype: torch.dtype = torch.float32, dropout: float = 0.0,
           dropout_seed: Optional[Tensor] = None) -> Tensor:
    """Differentiable EGConv layer body on a prepared graph.  storage_dtype=torch.bfloat16 stores the basis rows and the
    backward's target-side streams as bf16 (half the gathered bytes); x, parameters, weightings, out, the saved aggregates,
    all accumulation and every gradient stay fp32.  Fused epilogue of the stack around the layer (SURVEY 8 f-1):
    `scale` / `shift` [F_out] = an eval-mode BatchNorm folded to an affine map (constants), `relu=True` the ReLU that
    follows (mag/models.py:63, arxiv/norm_models.py:35-36), `residual` [N, F_out] added after the activation (:38-39):
    out = relu(layer(x) * scale + shift) + residual, all inside the aggregation kernel's epilogue; the backward masks and
    scales grad_out while its first pass stages the row.
    `dropout` = p > 0 (with relu=True, without scale / shift / residual): training-mode dropout after the ReLU in the same
    epilogue, out = keep ? relu(y) / (1 - p) : 0, with the counter-based mask of include/egc_b200.h (egc_dropout) keyed by
    `dropout_seed` (a one-element int64 CUDA tensor; drawn by `draw_dropout_seed` when None).  The caller decides on training
    mode, as with F.dropout(training=...).  The random stream is not torch's F.dropout stream."""
    return _EGConvFunction.apply(x, bases_weight, comb_weight, comb_bias, bias, graph, num_heads, num_bases,
                                 tuple(aggrs), bool(sigmoid), int(algo), int(bwd_flags), torch.is_grad_enabled(), bool(relu),
                                 scale, shift, residual, check_storage_dtype(storage_dtype), float(dropout), dropout_seed)


class _ProjectFunction(torch.autograd.Function):
    """bases, pre-activation weightings = project(x)  (ref :180-182) as its own autograd node - used by callers
    that post-process the weightings with ordinary torch ops (the paper-variant layer, `compat.py`)."""

    @staticmethod
    def forward(ctx, x, bases_weight, comb_weight, comb_bias, algo):
        x = _require_cuda_f32("x", x)
        bases_weight = _require_cuda_f32("bases_weight", bases_weight)
        comb_weight = _require_cuda_f32("comb_weight", comb_weight)
        comb_bias = _require_cuda_f32("comb_bias", comb_bias)
        with torch.cuda.device(x.device):
            bases, lin = project(x, bases_weight, comb_weight, comb_bias, False, algo)
        ctx.save_for_backward(x, bases_weight, comb_weight)
        ctx.algo, ctx.has_comb_bias = algo, comb_bias is not None
        return bases, lin

    @staticmethod
    def backward(ctx, d_bases, d_lin):
        x, bases_weight, comb_weight = ctx.saved_tensors
        need_x, need_wb, need_wc, need_bc = ctx.needs_input_grad[:4]
        d_bases = _require_cuda_f32("d_bases", d_bases)
        d_lin = _require_cuda_f32("d_lin", d_lin)
        with torch.cuda.device(x.device):
            d_x, d_wb, d_wc, d_bc = project_backward(x, bases_weight, comb_weight, d_bases, d_lin, need_x, need_wb,
                                                     need_wc, need_bc and ctx.has_comb_bias, ctx.algo)
        return d_x, d_wb, d_wc, d_bc, None


class _AggregateCombineFunction(torch.autograd.Function):
    """out = combine(aggregate(bases), weightings) + bias  (ref :191-208) as its own autograd node; `weightings`
    is whatever the caller made of the comb-weight projection (column order h * (A * B) + a * B + b)."""

    @staticmethod
    def forward(ctx, bases, weightings, bias, graph, heads, num_bases, aggrs, bwd_flags, grad_mode=True, add=None):
        if bases is not None and bases.dtype == torch.bfloat16:
            raise NotImplementedError("aggregate_combine_autograd: bf16 `bases` are not supported (use EGConv(..., "
                                      "storage_dtype=torch.bfloat16))")
        bases = _require_cuda_f32("bases", bases)
        add = _require_cuda_f32("add", add)
        weightings = _require_cuda_f32("weightings", weightings)
        bias = _require_cuda_f32("bias", bias)
        if bases.dim() != 2 or bases.size(0) != graph.n_src:
            raise ValueError(f"bases must be [n_src, B * D] with n_src == {graph.n_src} (got {tuple(bases.shape)})")
        if bases.size(1) % num_bases != 0:
            raise ValueError(f"bases width {bases.size(1)} is not divisible by num_bases={num_bases}")
        dim = bases.size(1) // num_bases
        hab = heads * len(aggrs) * num_bases
        if weightings.dim() != 2 or weightings.size(0) != graph.n_dst or weightings.size(1) != hab:
            raise ValueError(f"weightings must be [n_dst, H * A * B] = [{graph.n_dst}, {hab}] (got {tuple(weightings.shape)})")
        if bias is not None and bias.numel() != heads * dim:
            raise ValueError(f"bias must have H * D = {heads * dim} entries (got {bias.numel()})")
        desc = make_desc(graph, heads, num_bases, dim, aggrs, False)
        needs_grad = grad_mode and any(ctx.needs_input_grad[:3])
        if add is not None and tuple(add.shape) != (graph.n_dst, heads * dim):
            raise ValueError(f"`add` must be [n_dst, H * D] = [{graph.n_dst}, {heads * dim}] (got {tuple(add.shape)})")
        with torch.cuda.device(bases.device):
            out, _, _, saved, saved_arg = aggregate_combine(desc, graph, bases, weightings, bias, want_saved=needs_grad,
                                                            epilogue=(None, None, add))
        if needs_grad:
            ctx.save_for_backward(bases, weightings, saved, saved_arg)
        ctx.graph, ctx.desc, ctx.bwd_flags, ctx.has_bias = graph, desc, bwd_flags, bias is not None
        return out

    @staticmethod
    def backward(ctx, grad_out):
        grad_out = _require_cuda_f32("grad_out", grad_out)
        d_add = grad_out if ctx.needs_input_grad[9] else None        # out = f(bases, weightings) + add
        if not ctx.saved_tensors:
            return (None,) * 9 + (d_add,)
        bases, weightings, saved, saved_arg = ctx.saved_tensors
        with torch.cuda.device(bases.device):
            d_w, d_bases, d_bias = aggregate_backward(ctx.desc, ctx.graph, bases, weightings, saved, saved_arg, grad_out,
                                                      ctx.needs_input_grad[2] and ctx.has_bias, ctx.bwd_flags)
        return d_bases, d_w, d_bias, None, None, None, None, None, None, d_add


def project_autograd(x: Tensor, bases_weight: Tensor, comb_weight: Tensor, comb_bias: Optional[Tensor],
                     algo: int = _lib.GEMM_AUTO):
    """Differentiable (bases, comb-weight pre-activations)."""
    return _ProjectFunction.apply(x, bases_weight, comb_weight, comb_bias, int(algo))


def aggregate_combine_autograd(bases: Tensor, weightings: Tensor, bias: Optional[Tensor], graph: GraphStructure,
                               num_heads: int, num_bases: int, aggrs: Sequence[str], bwd_flags: int = 0,
                               add: Optional[Tensor] = None) -> Tensor:
    """Differentiable fused aggregation + combination on a prepared graph; `add` [n_dst, H * D] is added in the kernel's
    epilogue (accumulate-into-output: REGConv's running sum over relations, ref rmag/models.py:146)."""
    return _AggregateCombineFunction.apply(bases, weightings, bias, graph, num_heads, num_bases, tuple(aggrs),
                                           int(bwd_flags), torch.is_grad_enabled(), add)
