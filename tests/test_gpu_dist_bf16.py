"""bf16-storage layers (EGConv(..., storage_dtype=torch.bfloat16)) row-partitioned over ranks: on every rank the result is
this rank's rows of the SINGLE-GPU bf16 layer's results, at the bars that tests/test_gpu_dist.py applies to fp32.  Halo basis
rows and T-exchange stream rows travel as bf16, halo partial sums as fp32.

The one-GPU tests pin the two C entry points the partitioned backward uses (pass 1 into a caller's bf16 stream table + the
column pass over it, and the column phases) against the one-call bf16 backward; the two-rank tests need >= 2 GPUs."""
import os
import re
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from egc_b200 import _lib
from tests.util import random_graph, rel_err

DEV = "cuda:0"
BF16 = torch.bfloat16
gpu = pytest.mark.gpu
two_gpus = pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
NEW_SYMBOLS = ["egc_aggregate_bwd_bf16_partitioned", "egc_aggregate_bwd_cols_bf16"]


def test_partitioned_bf16_symbols_declared_and_signed():
    header = open(os.path.join(os.path.dirname(__file__), "..", "include", "egc_b200.h")).read()
    for name in NEW_SYMBOLS:
        assert re.search(rf"\b{name}\(", header), name
        assert name in _lib.SIGNATURES, name


# ------------------------------------------------------------------------------------------------
# one GPU: the C entry points of the partitioned bf16 backward
# ------------------------------------------------------------------------------------------------
def _bf16_layer_state(aggrs, h, b, d, seed, n=3000):
    """A graph with hub rows / columns (the chunk plans) and the saved state of a bf16 forward over it."""
    import egc_b200
    from egc_b200.functional import aggregate_combine, make_desc, project
    ei = random_graph(n, 30000, seed=seed, hub=700).to(DEV)
    g = egc_b200.GraphStructure.from_edge_index(ei, n, "symnorm" in aggrs, True)
    desc = make_desc(g, h, b, d, aggrs, False)
    torch.manual_seed(seed)
    f_in = 64
    x = torch.randn(n, f_in, device=DEV)
    wb, wc = torch.randn(f_in, b * d, device=DEV) * 0.1, torch.randn(h * len(aggrs) * b, f_in, device=DEV) * 0.1
    bases, w = project(x, wb, wc, None, False, storage_dtype=BF16)
    go = torch.randn(n, h * d, device=DEV)
    _, _, _, saved, saved_arg = aggregate_combine(desc, g, bases, w, None, want_saved=True)
    return g, desc, bases, w, saved, saved_arg, go


@gpu
@pytest.mark.parametrize("aggrs,h,b,d", [(["symnorm"], 8, 4, 16), (["sum"], 8, 4, 16)], ids=["symnorm", "sum"])
def test_bf16_pass1_into_table_then_column_pass_equals_one_call(aggrs, h, b, d):
    """The T-exchange backward on one GPU: bf16 pass 1 into a caller's table, then the column pass over the transposed
    adjacency, runs the same column kernel over the same entries in the same order as the one-call bf16 backward: the same
    bits."""
    import egc_b200
    from egc_b200.dist import n_target_streams, transpose_csr
    from egc_b200.functional import aggregate_backward, aggregate_backward_cols
    g, desc, bases, w, saved, saved_arg, go = _bf16_layer_state(aggrs, h, b, d, seed=31)
    n = g.n_dst
    ref = aggregate_backward(desc, g, bases, w, saved, saved_arg, go, True, want_lin_colsum=True)
    pad = 5                                                     # extra table rows (a partitioned caller's halo rows)
    t_ext = torch.zeros((n + pad, n_target_streams(aggrs) * b * d), dtype=BF16, device=DEV)
    got = aggregate_backward(desc, g, bases, w, saved, saved_arg, go, True, want_lin_colsum=True, tstreams_out=t_ext)
    assert got[1] is None and torch.equal(got[0], ref[0]) and torch.equal(got[2], ref[2]) and torch.equal(got[3], ref[3])
    assert bool((t_ext[:n] != 0).any()) and not bool((t_ext[n:] != 0).any())
    rowptr_t, col_t, *vals = transpose_csr(g.rowptr.cpu(), g.col.cpu(), g.val_sym.cpu() if g.val_sym is not None else None)
    gt = egc_b200.GraphStructure.from_prepared(rowptr_t, col_t, n + pad, val_sym=vals[0], device=DEV)
    desc_t = egc_b200.make_desc(gt, h, b, d, aggrs, False)
    desc_t.n_dst, desc_t.n_src = gt.n_src, gt.n_dst
    d_bases = aggregate_backward_cols(desc_t, gt, t_ext, bases)
    assert d_bases.dtype == torch.float32 and torch.equal(d_bases, ref[1])
    with pytest.raises(TypeError):                              # bf16 bases need a bf16 stream table
        aggregate_backward(desc, g, bases, w, saved, saved_arg, go, True, tstreams_out=t_ext.float())


@gpu
@pytest.mark.parametrize("aggrs", [["sum", "symnorm"], ["symnorm", "std"], ["symnorm", "max", "std"]], ids="+".join)
def test_bf16_column_phases_equal_one_call(aggrs):
    """COLS_HEAD then COLS_TAIL at col_split = n / 2 == the one-call bf16 backward: bit for bit without min / max; with max
    the routed gradients come first and pass 2 accumulates, one more rounding per value."""
    from egc_b200.functional import aggregate_backward
    g, desc, bases, w, saved, saved_arg, go = _bf16_layer_state(aggrs, 4, 4, 32, seed=32)
    n = g.n_dst
    ref = aggregate_backward(desc, g, bases, w, saved, saved_arg, go, True, want_lin_colsum=True)
    seen = {}
    got = aggregate_backward(desc, g, bases, w, saved, saved_arg, go, True, want_lin_colsum=True, col_split=n // 2,
                             between_phases=lambda d_b: seen.setdefault("head", d_b[n // 2:].clone()))
    routed = "max" in aggrs
    for a, r in zip(got, ref):
        if routed:
            assert rel_err(a, r) < 2e-6
        else:
            assert torch.equal(a, r)
    assert rel_err(seen["head"], ref[1][n // 2:]) < 2e-6     # the HEAD columns are final before the TAIL call
    if not routed:
        assert torch.equal(seen["head"], ref[1][n // 2:])


# ------------------------------------------------------------------------------------------------
# ranks: one process per GPU
# ------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    return dev


def _run(fn, world, *args):
    ret = mp.Manager().dict()
    mp.spawn(fn, args=(world, _free_port(), ret) + args, nprocs=world, join=True)
    assert dict(ret) == {r: "ok" for r in range(world)}


def _check(out, grads, out_ref, grads_ref, tag="", bars=(1e-6, 1e-5)):
    """One layer: the bars of tests/test_gpu_dist.py.  Stacks (`bars` of its two-layer check, 1e-5 / 2e-5, and 3e-5 for three
    layers) run with deterministic min / max routing: a lower layer's backward rounds its target-side streams to bf16, so
    an fp32 rounding difference in the gradient it receives (atomic routing order, the order of the halo partial sums) can
    move a stored stream value by one bf16 ulp."""
    e = rel_err(out, out_ref)
    assert e < bars[0], (tag, "out", e)
    for i, (a, r) in enumerate(zip(grads, grads_ref)):
        e = rel_err(a, r)
        assert e < bars[1], (tag, i, e)


def _grads(fn, x, go, params):
    xs = x.requires_grad_(True)
    out = fn(xs)
    return out, torch.autograd.grad(out, [xs] + params, go)


LAYERS = {  # name: (aggrs, heads, bases, dim, expect T exchange on two ranks)
    "egcm": (["symnorm", "max", "std"], 4, 4, 32, False),     # partial-sum exchange, routed
    "egcs": (["symnorm"], 8, 4, 16, True),                    # T exchange
    "sum_symnorm": (["sum", "symnorm"], 4, 4, 32, False),     # column-phase split backward (peer transport)
}


def _edges(n, seed, one_way):
    ei = random_graph(n, 30000, seed=seed, hub=900)
    blk = torch.randint(0, n // 2, (2, 15000), generator=torch.Generator().manual_seed(seed))
    parts = [ei, blk, blk + n // 2]
    if one_way:                # extra one-way edges: the transposed halo differs from the forward one
        g = torch.Generator().manual_seed(seed + 1)
        parts.append(torch.stack([torch.randint(0, n // 3, (4000,), generator=g), torch.randint(n // 2, n, (4000,), generator=g)]))
    return torch.cat(parts, 1)


def _layer_worker(rank, world, port, ret, transport, case):
    import egc_b200
    from egc_b200.dist import GraphedStep, PartitionedGraph, partitioned_egconv
    dev = _init(rank, world, port)
    pg = None
    try:
        aggrs, h, b, d, expect_t = LAYERS[case]
        n = 4000
        eid = _edges(n, 6, one_way=expect_t).to(dev)
        torch.manual_seed(0)
        mk = lambda f_in: egc_b200.EGConv(f_in, h * d, aggrs=aggrs, num_heads=h, num_bases=b, storage_dtype=BF16).to(dev)
        conv, conv2 = mk(64), mk(h * d)
        params, params2 = list(conv.parameters()), list(conv.parameters()) + list(conv2.parameters())
        g = egc_b200.GraphStructure.from_edge_index(eid, n, True, True)
        pg = PartitionedGraph.from_global(g, rank, world, dev, transport=transport, storage_dtype=BF16)
        assert pg.uses_t_exchange(aggrs) == (expect_t and world > 1)
        assert not pg.uses_overlap(aggrs, BF16)
        bb, e = pg.part.row_begin, pg.part.row_end
        gen = torch.Generator().manual_seed(1)
        x, go = torch.randn(n, 64, generator=gen), torch.randn(n, h * d, generator=gen)

        def step(xf, gf, tag):
            ref = _grads(lambda t: conv(t, eid), xf.to(dev), gf.to(dev), params)
            got = _grads(lambda t: partitioned_egconv(t, pg, conv), xf[bb:e].to(dev), gf[bb:e].to(dev), params)
            _check(got[0], got[1], ref[0][bb:e], (ref[1][0][bb:e],) + ref[1][1:], tag)

        for it in range(3):                                     # fresh data: epoch flags and buffer reuse
            gen = torch.Generator().manual_seed(10 + it)
            step(torch.randn(x.shape, generator=gen), torch.randn(go.shape, generator=gen), f"step {it}")
        pg.check()
        with torch.no_grad():                                   # no_grad twice, then a training step
            for _ in range(2):
                assert rel_err(partitioned_egconv(x[bb:e].to(dev), pg, conv), conv(x.to(dev), eid)[bb:e]) < 1e-6
        step(x, go, "after no_grad")
        pg.check()
        # two stacked layers, each with its own exchange buffers
        conv.deterministic = conv2.deterministic = True
        ref = _grads(lambda t: conv2(torch.relu(conv(t, eid)), eid), x.to(dev), go.to(dev), params2)
        got = _grads(lambda t: partitioned_egconv(torch.relu(partitioned_egconv(t, pg, conv)), pg, conv2),
                     x[bb:e].to(dev), go[bb:e].to(dev), params2)
        _check(got[0], got[1], ref[0][bb:e], (ref[1][0][bb:e],) + ref[1][1:], "two layers", (1e-5, 2e-5))
        conv.deterministic = False
        pg.check()
        if transport == "peer" and world > 1:
            ctx = next(c for k, c in pg._peer_ctx.items() if k[0] == id(conv))
            assert ctx.bases_ext.dtype == BF16 and (ctx.t_ext is None or ctx.t_ext.dtype == BF16)
            import gc
            gc.collect()
            x_static, go_static = x[bb:e].to(dev).requires_grad_(True), go[bb:e].to(dev)

            def graphed_step():
                o = partitioned_egconv(x_static, pg, conv)
                return (o,) + torch.autograd.grad(o, [x_static] + params, go_static)

            graphed = GraphedStep(graphed_step, warmup=2)
            for it in range(3):
                gen = torch.Generator().manual_seed(50 + it)
                xf, gf = torch.randn(x.shape, generator=gen), torch.randn(go.shape, generator=gen)
                with torch.no_grad():
                    x_static.copy_(xf[bb:e].to(dev))
                    go_static.copy_(gf[bb:e].to(dev))
                res = graphed.replay()
                ref = _grads(lambda t: conv(t, eid), xf.to(dev), gf.to(dev), params)
                _check(res[0], res[1:], ref[0][bb:e], (ref[1][0][bb:e],) + ref[1][1:], f"replay {it}")
            pg.check()
        torch.cuda.synchronize()
        ret[rank] = "ok"
    finally:
        if pg is not None:
            pg.close()
        dist.destroy_process_group()


@gpu
@pytest.mark.parametrize("case", list(LAYERS))
def test_bf16_layer_on_one_rank_matches_single_gpu(case):
    """One rank (no halo, the NCCL path): the bf16 layer through the partitioned autograd function."""
    _run(_layer_worker, 1, "nccl", case)


@gpu
@two_gpus
@pytest.mark.parametrize("transport", ["peer", "nccl"])
@pytest.mark.parametrize("case", list(LAYERS))
def test_bf16_partitioned_layer_matches_single_gpu_world2(transport, case):
    _run(_layer_worker, 2, transport, case)


def _more_worker(rank, world, port, ret, transport):
    """Interior-heavy graph, 3-layer EGC stack, mixed fp32 / bf16 stack, EGC_DIST_OVERLAP, exchange bytes and guards."""
    import egc_b200
    from egc_b200.dist import PartitionedGraph, partitioned_egconv
    os.environ["EGC_DIST_OVERLAP"] = "1"
    dev = _init(rank, world, port)
    pgs = []
    try:
        n = 4000
        gen = torch.Generator().manual_seed(3)
        x, go = torch.randn(n, 128, generator=gen), torch.randn(n, 128, generator=gen)
        eid = _edges(n, 7, one_way=True).to(dev)
        g = egc_b200.GraphStructure.from_edge_index(eid, n, True, True)
        pg = PartitionedGraph.from_global(g, rank, world, dev, transport=transport, storage_dtype=BF16)
        pgs.append(pg)
        bb, e = pg.part.row_begin, pg.part.row_end
        torch.manual_seed(0)

        def compare(ref_fn, fn, params, x_full, go_full, tag, bars=(1e-6, 1e-5)):
            ref = _grads(ref_fn, x_full.to(dev), go_full.to(dev), params)
            got = _grads(fn, x_full[bb:e].to(dev), go_full[bb:e].to(dev), params)
            _check(got[0], got[1], ref[0][bb:e], (ref[1][0][bb:e],) + ref[1][1:], tag, bars)
            pg.check()

        # a bf16 layer on a graph that did not opt in
        conv = egc_b200.EGConv(128, 128, aggrs=["symnorm"], num_heads=8, num_bases=4, storage_dtype=BF16).to(dev)
        plain = PartitionedGraph.from_global(g, rank, world, dev, transport=transport)
        pgs.append(plain)
        try:
            partitioned_egconv(x[bb:e].to(dev), plain, conv)
            raise AssertionError("a bf16 layer ran on a graph built without storage_dtype=torch.bfloat16")
        except NotImplementedError:
            pass
        # EGC_DIST_OVERLAP=1: the fp32 twin of this layer would overlap, the bf16 layer waits and matches
        assert pg.uses_overlap(["symnorm"]) == (transport == "peer") and not pg.uses_overlap(["symnorm"], BF16)
        compare(lambda t: conv(t, eid), lambda t: partitioned_egconv(t, pg, conv), list(conv.parameters()), x, go, "overlap=1")
        if transport == "peer":
            # halo and stream rows travel as bf16: half the bytes of the fp32 context of the same layer
            k = next(k for k in pg._peer_ctx if k[0] == id(conv))
            c16 = pg._peer_ctx[k]
            c32 = pg.peer_context("fp32 twin", *k[1:4])
            assert c16.t_ext is not None and c16.t_ext.dtype == BF16 and c32.t_ext.dtype == torch.float32
            assert 2 * c16.bases_ext.nbytes == c32.bases_ext.nbytes and 2 * c16.t_ext.nbytes == c32.t_ext.nbytes
            assert 2 * c16.bd_words == c32.bd_words and 2 * c16.t_words == c32.t_words
            assert c16.staging.dtype == torch.float32 and c16.staging.nbytes == c32.staging.nbytes
        # mixed stack on the bf16-enabled graph: an fp32 layer, then a bf16 layer
        kw = dict(aggrs=["symnorm", "max", "std"], num_heads=4, num_bases=4, deterministic=True)
        f32 = egc_b200.EGConv(128, 128, **kw).to(dev)
        b16 = egc_b200.EGConv(128, 128, storage_dtype=BF16, **kw).to(dev)
        params = list(f32.parameters()) + list(b16.parameters())
        compare(lambda t: b16(torch.relu(f32(t, eid)), eid),
                lambda t: partitioned_egconv(partitioned_egconv(t, pg, f32, relu=True), pg, b16), params, x, go, "mixed",
                (1e-5, 2e-5))
        # 3-layer EGC stack (cfg3 shape: 40-value output layer), dropout 0
        m = egc_b200.EGC(128, 3, 0.0, 4, 4, ["symnorm", "max", "std"], in_features=128, out_rounded=40, out_true=40,
                         storage_dtype=BF16, deterministic=True).to(dev)
        compare(lambda t: m(t, eid), lambda t: m(t, pg), list(m.parameters()), x, go[:, :40], "EGC stack", (1e-5, 3e-5))
        # interior-heavy graph (two blocks joined by a few edges): fp32 would aggregate the interior rows while the halo
        # rows travel, the bf16 layer waits and runs one contiguous launch
        blk = torch.randint(0, n // 2, (2, 20000), generator=torch.Generator().manual_seed(9))
        cross = torch.stack([torch.arange(0, 40), torch.arange(n // 2, n // 2 + 40)])
        eid2 = torch.cat([blk, blk + n // 2, cross], 1).to(dev)
        g2 = egc_b200.GraphStructure.from_edge_index(eid2, n, True, True)
        pg2 = PartitionedGraph.from_global(g2, rank, world, dev, transport=transport, storage_dtype=BF16)
        pgs.append(pg2)
        assert pg2.overlap_interior and pg2.part.n_halo > 0
        egcm = egc_b200.EGConv(128, 128, aggrs=["symnorm", "max", "std"], num_heads=4, num_bases=4, storage_dtype=BF16).to(dev)
        b2, e2 = pg2.part.row_begin, pg2.part.row_end
        ref = _grads(lambda t: egcm(t, eid2), x.to(dev), go.to(dev), list(egcm.parameters()))
        got = _grads(lambda t: partitioned_egconv(t, pg2, egcm), x[b2:e2].to(dev), go[b2:e2].to(dev), list(egcm.parameters()))
        _check(got[0], got[1], ref[0][b2:e2], (ref[1][0][b2:e2],) + ref[1][1:], "interior-heavy")
        pg2.check()
        # edge values: ValueError on every rank, before anything collective
        rowptr, col = g.rowptr.long(), g.col.long()
        gv = egc_b200.GraphStructure.from_csr(rowptr, col, torch.rand(col.numel(), device=dev), n, False, False)
        assert gv.val_lin is not None
        try:
            PartitionedGraph.from_global(gv, rank, world, dev, transport=transport, storage_dtype=BF16)
            raise AssertionError("an edge-valued graph was accepted for bf16 storage")
        except ValueError:
            pass
        dist.barrier()
        torch.cuda.synchronize()
        ret[rank] = "ok"
    finally:
        for p in pgs:
            p.close()
        dist.destroy_process_group()


@gpu
@two_gpus
@pytest.mark.parametrize("transport", ["peer", "nccl"])
def test_bf16_partitioned_stacks_and_guards_world2(transport):
    _run(_more_worker, 2, transport)
