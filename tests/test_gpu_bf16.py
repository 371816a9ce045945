"""Opt-in bf16 storage of the gathered tensors (EGConv(..., storage_dtype=torch.bfloat16)).

Each stage is pinned on its own, so that no tolerance hides a bug: the projection against the bf16 rounding of the fp64
product; the aggregation + combination against the fp64 oracle fed with the device's OWN bf16 basis rows (argmax ids
bit-exact); the backward against the fp64 oracle with a bound derived from one bf16 rounding of the target-side streams."""
import os
import re
import types

import pytest
import torch

import egc_b200
from egc_b200 import _lib
from egc_b200.functional import (aggregate_backward, aggregate_combine, aggregate_combine_autograd, check_bf16_layer,
                                 make_desc, project)
from oracle import restatement as R
from tests.util import random_graph, rel_err, to_adj_csr

DEV = "cuda:0"
TOL = 1e-5
gpu = pytest.mark.gpu
NEW_SYMBOLS = ["egc_project_fwd_bf16", "egc_aggregate_fwd_bf16", "egc_aggregate_bwd_bf16_workspace_bytes",
               "egc_aggregate_bwd_bf16"]


# ------------------------------------------------------------------------------------------------
# CPU: interface and guards
# ------------------------------------------------------------------------------------------------
def test_bf16_symbols_declared_and_signed():
    header = open(os.path.join(os.path.dirname(__file__), "..", "include", "egc_b200.h")).read()
    for name in NEW_SYMBOLS:
        assert re.search(rf"\b{name}\(", header), name
        assert name in _lib.SIGNATURES, name
    assert "#define EGC_ABI_VERSION 5" in header


def test_storage_dtype_argument():
    ref = egc_b200.EGConv(16, 32, aggrs=["symnorm"], num_heads=4, num_bases=4)
    c = egc_b200.EGConv(16, 32, aggrs=["symnorm"], num_heads=4, num_bases=4, storage_dtype=torch.bfloat16)
    assert c.storage_dtype == torch.bfloat16 and ref.storage_dtype == torch.float32
    assert list(c.state_dict()) == list(ref.state_dict()) and repr(c) == repr(ref)
    assert len(list(c.buffers())) == len(list(ref.buffers()))
    for bad in (torch.float16, torch.float64, "bf16"):
        with pytest.raises(ValueError):
            egc_b200.EGConv(16, 32, storage_dtype=bad)
    stack = egc_b200.EGC(32, 3, 0.0, 4, 4, ["symnorm"], in_features=16, out_rounded=40, out_true=40,
                         storage_dtype=torch.bfloat16)
    assert all(conv.storage_dtype == torch.bfloat16 for conv in stack.convs)


def test_unsupported_paths_raise_not_implemented():
    with pytest.raises(NotImplementedError):
        egc_b200.REGConv(16, 32, 4, 4, storage_dtype=torch.bfloat16)
    with pytest.raises(NotImplementedError):
        egc_b200.EfficientGraphConv(16, 32, 4, 4, False, aggrs=["add"], storage_dtype=torch.bfloat16)
    conv = egc_b200.EGConv(16, 32, storage_dtype=torch.bfloat16)
    with pytest.raises(NotImplementedError):
        egc_b200.dist.partitioned_egconv(torch.zeros(4, 16), None, conv)
    with pytest.raises(NotImplementedError):
        aggregate_combine_autograd(torch.zeros(4, 32, dtype=torch.bfloat16), torch.zeros(4, 8), None, None, 4, 4, ["sum"])


@pytest.mark.parametrize("heads,bases,dim,aggrs,ok", [
    (4, 4, 32, ["symnorm", "max", "std"], True),     # cfg2 / CIFAR: B*D = 128
    (8, 4, 16, ["symnorm"], True),                   # cfg4: B*D = 64
    (4, 4, 10, ["symnorm", "max", "std"], True),     # the 40-class output layer of cfg3: B*D = 40
    (8, 4, 13, ["sum"], False),                      # ZINC: B*D = 52, not a multiple of 8
    (4, 4, 88, ["symnorm"], False),                  # B*D = 352: wider than one pass
    (4, 2, 16, ["sum"], False),                      # B*D = 32: narrower than the kernels cover
    (4, 4, 32, ["sum", "mean", "symnorm", "min", "max", "var", "std"], False),   # 7 x 128 values: staging too wide
])
def test_bf16_shape_rules(heads, bases, dim, aggrs, ok):
    g = types.SimpleNamespace(n_dst=10, n_src=10, val_lin=None)
    desc = make_desc(g, heads, bases, dim, aggrs, False)
    if ok:
        check_bf16_layer(desc, g)
    else:
        with pytest.raises(ValueError):
            check_bf16_layer(desc, g)


# ------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------
def _bf16_ulp(ref: torch.Tensor) -> torch.Tensor:
    _, e = torch.frexp(ref.double())
    return torch.ldexp(torch.ones_like(ref, dtype=torch.float64), e - 8)


def _graphs(n, e, seed, hub, kind, symnorm, multi_aggr, loops=True):
    ei = random_graph(n, e, seed=seed, hub=hub)
    if kind == "edge_index":
        return ei.to(DEV), R.graph_from_edge_index(ei, n, symnorm, loops), egc_b200.GraphStructure.from_edge_index(
            ei.to(DEV), n, symnorm, loops)
    rowptr, col, _ = to_adj_csr(ei, n)
    st = egc_b200.SparseTensor(rowptr=rowptr.to(DEV), col=col.to(DEV), sparse_sizes=(n, n), is_sorted=True)
    return st, R.graph_from_csr(rowptr, col, None, n, symnorm, loops, multi_aggr), egc_b200.GraphStructure.from_csr(
        rowptr.to(DEV), col.to(DEV), None, n, symnorm, loops)


def _src_ids(col, pos):
    nnz = col.numel()
    return torch.where((pos >= 0) & (pos < nnz), col[pos.clamp(0, nnz - 1)], torch.full_like(pos, -1))


def _layer_from_bases(g, bases, weightings, bias, aggrs, num_heads, grad_out=None):
    """The oracle's aggregation + combination (R.aggregate / R.combine) from GIVEN basis rows - the device's own bf16
    rows, widened - so that the stages after the projection are checked on their own.  Returns {"out", "args"} and, with
    `grad_out`, {"d_bases", "d_bases_mag", "d_weightings"}.  d_bases_mag[j] = sum over the entries e of column j and over
    the target-side streams of |stream term of e|: each aggregator gets its own copy of the gathered rows, var / std one
    for the mean and one for the square, so terms that cancel inside an entry are counted by magnitude - that is what
    a per-value relative rounding of each stored stream is relative to."""
    ge = R.OracleGraph(g.rowptr, torch.arange(g.nnz), g.n_dst, g.nnz, g.val_sym, g.val_lin, g.deg, g.dis)
    grad = grad_out is not None
    xe = bases.index_select(0, g.col).detach().requires_grad_(grad)       # one leaf row per entry
    w = weightings.detach().requires_grad_(grad)
    with torch.set_grad_enabled(grad):
        agg, args = R.aggregate(ge, xe, aggrs)
        out = R.combine(w, agg, bias, num_heads)
    res = {"out": out.detach(), "args": args}
    if not grad:
        return res
    d_xe, d_w = torch.autograd.grad(out, [xe, w], grad_out)
    zeros = bases.new_zeros(bases.shape)
    res["d_bases"], res["d_weightings"] = zeros.index_add(0, g.col, d_xe), d_w
    # per-stream magnitudes (no edge values: the bf16 path rejects them)
    row, n = ge.row, g.n_dst
    cnt = (g.rowptr[1:] - g.rowptr[:-1]).clamp(min=1).to(xe.dtype).view(-1, 1)
    rz = xe.new_zeros((n, xe.shape[1]))
    leaves, parts = [], []
    with torch.enable_grad():
        for a in aggrs:
            if a in ("var", "std"):
                xl, xs = xe.detach().clone().requires_grad_(True), xe.detach().clone().requires_grad_(True)
                mean = rz.index_add(0, row, xl) / cnt
                r = rz.index_add(0, row, xs * xs) / cnt - mean * mean
                if a == "std":
                    r = torch.sqrt(torch.relu(r) + R.STD_EPS)
                leaves += [xl, xs]
            else:
                xa = xe.detach().clone().requires_grad_(True)
                r = R.aggregate(ge, xa, [a])[0][:, 0]
                leaves.append(xa)
            parts.append(r)
        out_m = R.combine(w.detach(), torch.stack(parts, dim=1), bias, num_heads)
    mags = torch.autograd.grad(out_m, leaves, grad_out)
    res["d_bases_mag"] = zeros.index_add(0, g.col, sum(m.abs() for m in mags))
    return res


def _stage_check(n, e, hub, kind, f_in, heads, bases, dim, aggrs, seed=0, deterministic=False):
    """Projection, forward and backward of one layer in bf16 storage, each against its own fp64 reference."""
    symnorm = "symnorm" in aggrs
    _, og, g = _graphs(n, e, seed + 1, hub, kind, symnorm, len(aggrs) > 1)
    torch.manual_seed(seed)
    bd, hd, hab = bases * dim, heads * dim, heads * len(aggrs) * bases
    x = torch.randn(n, f_in)
    wb, wc, bc, bias = torch.randn(f_in, bd) * 0.1, torch.randn(hab, f_in) * 0.1, torch.randn(hab) * 0.1, torch.randn(hd)
    go = torch.randn(n, hd)
    xd, wbd, wcd, bcd, biasd, god = (t.to(DEV) for t in (x, wb, wc, bc, bias, go))
    # projection: the bf16 rows are the round-to-nearest-even of the layer's own fp32 products (bit-exact), and within one
    # bf16 ulp of the rounded fp64 product, plus the fp32 accumulation error where a row's terms cancel
    bases_bf, w = project(xd, wbd, wcd, bcd, False, storage_dtype=torch.bfloat16)
    assert bases_bf.dtype == torch.bfloat16 and w.dtype == torch.float32
    bases32, _ = project(xd, wbd, wcd, bcd, False)
    assert torch.equal(bases_bf, bases32.to(torch.bfloat16))
    exact = x.double() @ wb.double()
    ref = exact.to(torch.bfloat16)
    acc_err = 1e-6 * (x.double().abs() @ wb.double().abs())
    assert ((bases_bf.cpu().double() - ref.double()).abs() <= _bf16_ulp(ref) + acc_err).all()
    assert rel_err(w, torch.nn.functional.linear(x.double(), wc.double(), bc.double())) < TOL
    # forward from the device's own rows
    desc = make_desc(g, heads, bases, dim, aggrs, False)
    out, _, arg, saved, saved_arg = aggregate_combine(desc, g, bases_bf, w, biasd, want_arg=True, want_saved=True)
    b64 = bases_bf.cpu().double()
    ores = _layer_from_bases(og, b64, w.cpu().double(), bias.double(), aggrs, heads, go.double())
    o32 = _layer_from_bases(og, b64.float(), w.cpu(), bias, aggrs, heads)
    assert rel_err(out, ores["out"]) < max(TOL, 4 * rel_err(o32["out"], ores["out"]))
    for name in ("min", "max"):
        if name in aggrs:
            k = aggrs.index(name)
            assert torch.equal(g.source_ids(arg[:, k]).cpu(), _src_ids(og.col, ores["args"][name])), name
    # backward: each stream value rounded once to bf16 (relative error <= 2^-9) -> |error| <= 2^-8 * (the column pass over
    # the magnitudes of the stream terms) + the fp32 rule
    flags = _lib.BWD_DETERMINISTIC if deterministic else 0
    d_w, d_bases, d_bias, d_bc = aggregate_backward(desc, g, bases_bf, w, saved, saved_arg, god, True, flags,
                                                    want_lin_colsum=True)
    ref_db, ref_abs = ores["d_bases"], ores["d_bases_mag"]
    bound = 2.0 ** -8 * ref_abs + TOL * ref_db.abs().max()
    assert ((d_bases.cpu().double() - ref_db).abs() <= bound).all()
    w_bar = max(TOL, 4 * rel_err(_layer_from_bases(og, b64.float(), w.cpu(), bias, aggrs, heads, go)["d_weightings"],
                                 ores["d_weightings"]))
    assert rel_err(d_w, ores["d_weightings"]) < w_bar
    assert rel_err(d_bias, go.double().sum(0)) < TOL
    assert rel_err(d_bc, ores["d_weightings"].sum(0)) < w_bar
    return g, (desc, bases_bf, w, saved, saved_arg, god, flags)


SHAPES = [  # f_in, heads, bases, dim, aggrs
    (128, 4, 4, 32, ["symnorm", "max", "std"]),       # cfg2 / CIFAR (A = 3, B*D = 128)
    (128, 8, 4, 16, ["symnorm"]),                     # cfg4 (B*D = 64)
    (128, 4, 4, 10, ["symnorm", "max", "std"]),       # cfg3 output layer (B*D = 40, D % 4 != 0)
    (64, 4, 2, 32, ["sum", "mean", "min", "max", "var", "std"]),   # every other aggregator, B*D = 64
] + [(64, 4, 4, 32, [a]) for a in ("sum", "mean", "symnorm", "min", "max", "var", "std")]


@gpu
@pytest.mark.parametrize("kind", ["edge_index", "adj_t"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"h{s[1]}b{s[2]}d{s[3]}-{'+'.join(s[4])}")
def test_stages_against_the_oracle(shape, kind):
    f_in, h, b, d, aggrs = shape
    _stage_check(2000, 16000, 700, kind, f_in, h, b, d, aggrs)     # hub rows / columns of > 256 nnz: the chunk plan


@gpu
def test_deterministic_routing_is_bit_reproducible():
    """Dyadic inputs (test_deterministic_routing_*): x in multiples of 1/4, weights in multiples of 1/16."""
    n, aggrs = 3000, ["max", "min", "std"]
    ei = random_graph(n, 30000, seed=71, hub=900).to(DEV)
    torch.manual_seed(10)
    c = egc_b200.EGConv(128, 128, aggrs=aggrs, num_heads=4, num_bases=4, deterministic=True,
                        storage_dtype=torch.bfloat16).to(DEV)
    with torch.no_grad():
        c.bases_weight.copy_(torch.round(c.bases_weight * 16) / 16)
    x = (torch.round(torch.randn(n, 128) * 4) / 4).to(DEV)
    go = torch.randn(n, 128, device=DEV)
    runs = []
    for _ in range(4):
        xc = x.clone().requires_grad_(True)
        out = c(xc, ei)
        runs.append([out] + list(torch.autograd.grad(out, [xc] + list(c.parameters()), go)))
    for r in runs[1:]:
        for a, bb in zip(r, runs[0]):
            assert torch.equal(a, bb)
    _stage_check(n, 30000, 900, "edge_index", 128, 4, 4, 32, aggrs, seed=71, deterministic=True)


@gpu
def test_layer_gradients_against_the_oracle():
    """d_x of the whole layer: the bound of the column pass carried through W_b, plus the fp32 rule."""
    n, f_in, aggrs = 2000, 96, ["symnorm", "max", "std"]
    ei, og, _ = _graphs(n, 16000, 5, 700, "edge_index", True, True)
    torch.manual_seed(4)
    c = egc_b200.EGConv(f_in, 128, aggrs=aggrs, num_heads=4, num_bases=4, storage_dtype=torch.bfloat16).to(DEV)
    x, go = torch.randn(n, f_in), torch.randn(n, 128)
    xc = x.to(DEV).requires_grad_(True)
    out = c(xc, ei)
    d_x, d_wb, d_wc, d_bc, d_bias = torch.autograd.grad(out, [xc, c.bases_weight, c.comb_weight.weight,
                                                             c.comb_weight.bias, c.bias], go.to(DEV))
    wb, wc = c.bases_weight.detach().cpu().double(), c.comb_weight.weight.detach().cpu().double()
    bases_bf, w = project(xc.detach(), c.bases_weight, c.comb_weight.weight, c.comb_weight.bias, False,
                          storage_dtype=torch.bfloat16)
    ores = _layer_from_bases(og, bases_bf.cpu().double(), w.cpu().double(), c.bias.detach().cpu().double(), aggrs, 4,
                              go.double())
    ref_dx = ores["d_bases"] @ wb.T + ores["d_weightings"] @ wc
    bound = 2.0 ** -8 * (ores["d_bases_mag"] @ wb.abs().T) + TOL * ref_dx.abs().max()
    assert ((d_x.cpu().double() - ref_dx).abs() <= bound).all()
    assert rel_err(d_wc, ores["d_weightings"].T @ x.double()) < 1e-4
    assert rel_err(d_bias, go.double().sum(0)) < TOL
    assert torch.isfinite(d_wb).all() and torch.isfinite(d_bc).all()


@gpu
def test_fused_epilogue_matches_separate_ops():
    n, aggrs = 2000, ["symnorm", "max", "std"]
    ei = random_graph(n, 16000, seed=3, hub=600).to(DEV)
    torch.manual_seed(2)
    c = egc_b200.EGConv(128, 128, aggrs=aggrs, num_heads=4, num_bases=4, storage_dtype=torch.bfloat16).to(DEV)
    x = torch.randn(n, 128, device=DEV)
    scale, shift = torch.rand(128, device=DEV) + 0.5, torch.randn(128, device=DEV)
    res, go = torch.randn(n, 128, device=DEV), torch.randn(n, 128, device=DEV)
    grads = []
    for fused in (True, False):
        xc = x.clone().requires_grad_(True)
        out = c(xc, ei, relu=True, scale=scale, shift=shift, residual=res) if fused else \
            torch.relu(c(xc, ei) * scale + shift) + res
        grads.append([out] + list(torch.autograd.grad(out, [xc] + list(c.parameters()), go)))
    for a, b in zip(*grads):
        assert rel_err(a, b.double()) < 1e-4


@gpu
def test_empty_and_zero_row_inputs():
    c = egc_b200.EGConv(64, 128, aggrs=["symnorm", "max", "std"], num_heads=4, num_bases=4,
                        storage_dtype=torch.bfloat16).to(DEV)
    x0 = torch.zeros(0, 64, device=DEV, requires_grad=True)
    out = c(x0, torch.zeros(2, 0, dtype=torch.long, device=DEV))
    out.sum().backward()
    assert out.shape == (0, 128)
    # isolated nodes (empty rows without self-loops) and a single node (its self-loop only)
    for n, ei, loops in ((50, torch.tensor([[0, 1, 2], [1, 2, 3]]), False), (1, torch.zeros(2, 0, dtype=torch.long), True)):
        c.add_self_loops = loops
        c._cached_edge_index = None
        x = torch.randn(n, 64, device=DEV, requires_grad=True)
        out = c(x, ei.to(DEV))
        out.sum().backward()
        assert torch.isfinite(out).all() and torch.isfinite(x.grad).all()


@gpu
def test_unsupported_shapes_raise_value_error():
    n = 100
    ei = random_graph(n, 800, seed=1).to(DEV)
    x = torch.randn(n, 52, device=DEV)
    with pytest.raises(ValueError):
        egc_b200.EGConv(52, 104, aggrs=["sum"], num_heads=8, num_bases=4, storage_dtype=torch.bfloat16).to(DEV)(x, ei)
    rowptr, col, v = to_adj_csr(ei.cpu(), n, torch.rand(ei.size(1)))
    st = egc_b200.SparseTensor(rowptr=rowptr.to(DEV), col=col.to(DEV), value=v.to(DEV), sparse_sizes=(n, n), is_sorted=True)
    with pytest.raises(ValueError):
        egc_b200.EGConv(52, 128, aggrs=["sum"], num_heads=4, num_bases=4, storage_dtype=torch.bfloat16).to(DEV)(x, st)


@gpu
def test_full_size_cfg2():
    """arxiv-shaped EGC-M at full size (169343 nodes, hub-heavy random graph): the same bars as the stage test."""
    _stage_check(169_343, 1_166_243, 3000, "edge_index", 128, 4, 4, 32, ["symnorm", "max", "std"], seed=11)


@gpu
def test_three_layer_stack_graph_replay_equals_eager():
    n = 5000
    ei = random_graph(n, 40000, seed=8, hub=800).to(DEV)
    torch.manual_seed(0)
    m = egc_b200.EGC(128, 3, 0.0, 4, 4, ["symnorm", "max", "std"], in_features=128, out_rounded=40, out_true=40,
                     storage_dtype=torch.bfloat16, deterministic=True).to(DEV)
    x = torch.randn(n, 128, device=DEV, requires_grad=True)
    go = torch.randn(n, 40, device=DEV)

    def step():
        out = m(x, ei)
        return [out] + list(torch.autograd.grad(out, [x] + list(m.parameters()), go))

    eager = [t.detach().clone() for t in step()]      # no autograd graph of the eager call stays alive
    graphed = egc_b200.GraphedStep(step, warmup=2)
    graphed.replay()
    torch.cuda.synchronize()
    for a, b in zip(graphed.outputs, eager):
        assert torch.equal(a, b)
