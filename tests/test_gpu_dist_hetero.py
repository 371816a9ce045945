"""REGConv row-partitioned over ranks (`egc_b200.dist.PartitionedHeteroGraph`): on every rank the result is this rank's rows
of every node type of the single-GPU REGConv, for both transports (our NVLink peer-memory kernels and the NCCL baseline),
across repeated steps, under no_grad, for a two-layer stack and when the whole step is replayed from a CUDA graph.

One GPU: the one-rank graph (bit for bit, with deterministic max routing), the peer push with more segments than one per
peer, and the guards.  The two- and four-rank tests need >= 2 / >= 4 GPUs."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import hetero as OH
from tests.util import rel_err

pytestmark = pytest.mark.gpu
# the hub graph of tests/test_hetero.py::test_regconv_cuda_vs_oracle_larger_graph_with_hubs
SIZES = {"author": 1500, "field_of_study": 90, "institution": 40, "paper": 1100}
TYPES = list(SIZES)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run(fn, world, *args):
    ret = mp.Manager().dict()
    mp.spawn(fn, args=(world, _free_port(), ret) + args, nprocs=world, join=True)
    assert dict(ret) == {r: "ok" for r in range(world)}


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    return dev


def _adj(dev):
    import egc_b200
    csr = OH.random_hetero_graph(SIZES, 9000, 5)
    return {k: egc_b200.SparseTensor(rowptr=rp.to(dev), col=col.to(dev), sparse_sizes=(rp.numel() - 1, ns), is_sorted=True)
            for k, (rp, col, ns) in csr.items()}


def _data(seed, f_in=64, f_out=128):
    gen = torch.Generator().manual_seed(seed)
    return ({t: torch.randn(n, f_in, generator=gen) for t, n in SIZES.items()},
            {t: torch.randn(n, f_out, generator=gen) for t, n in SIZES.items()})


def _grads(fn, x, go, params, dev):
    xs = {t: v.to(dev).requires_grad_(True) for t, v in x.items()}
    out = fn(xs)
    loss = sum((out[t] * go[t].to(dev)).sum() for t in TYPES)
    return out, torch.autograd.grad(loss, [xs[t] for t in TYPES] + params)


def _local(d, phg):
    return {t: v[slice(*phg.row_range(t))] for t, v in d.items()}


def _check(got, ref, phg, tag, bars):
    out, grads = got
    out_ref, grads_ref = ref
    for i, t in enumerate(TYPES):
        b, e = phg.row_range(t)
        e_out, e_x = rel_err(out[t], out_ref[t][b:e]), rel_err(grads[i], grads_ref[i][b:e])
        assert e_out < bars[0], (tag, t, "out", e_out)
        assert e_x < bars[1], (tag, t, "d_x", e_x)
    for j, (a, r) in enumerate(zip(grads[len(TYPES):], grads_ref[len(TYPES):])):
        assert rel_err(a, r) < bars[1], (tag, "param", j, rel_err(a, r))


# ------------------------------------------------------------------------------------------------
# one GPU
# ------------------------------------------------------------------------------------------------
def _one_rank_worker(rank, world, port, ret, transport):
    import egc_b200
    from egc_b200.dist import PartitionedHeteroGraph
    dev = _init(rank, world, port)
    phg = None
    try:
        adj = _adj(dev)
        torch.manual_seed(0)
        # deterministic max routing: with fp32 atomics the single-GPU layer itself differs from run to run in the last bits
        conv = egc_b200.REGConv(64, 128, 8, 4, deterministic=True).to(dev)
        params = list(conv.parameters())
        phg = PartitionedHeteroGraph.from_global(adj, SIZES, rank, world, dev, transport=transport)
        assert phg.transport == transport and phg.edge_types == list(adj)
        for t, n in SIZES.items():
            assert phg.row_range(t) == (0, n)
        for it in range(2):
            x, go = _data(20 + it)
            ref = _grads(lambda xs: conv(xs, adj), x, go, params, dev)
            got = _grads(lambda xs: conv(xs, phg), x, go, params, dev)
            for t in TYPES:
                assert torch.equal(got[0][t], ref[0][t]), (it, t)
            for a, r in zip(got[1], ref[1]):
                assert torch.equal(a, r), it
        with torch.no_grad():
            x, _ = _data(30)
            xs = {t: v.to(dev) for t, v in x.items()}
            out, out_ref = conv(xs, phg), conv(xs, adj)
            assert all(torch.equal(out[t], out_ref[t]) for t in TYPES)
        phg.check()
        if transport == "peer":
            # a stale backward: the layer ran another forward since the one being differentiated
            xs = {t: v.to(dev).requires_grad_(True) for t, v in x.items()}
            first = conv(xs, phg)
            conv(xs, phg)
            with pytest.raises(RuntimeError):
                sum(v.sum() for v in first.values()).backward()
        torch.cuda.synchronize()
        ret[rank] = "ok"
    finally:
        if phg is not None:
            phg.close()
        dist.destroy_process_group()


@pytest.mark.parametrize("transport", ["peer", "nccl"])
def test_one_rank_partitioned_regconv_is_bit_identical(transport):
    _run(_one_rank_worker, 1, transport)


@pytest.mark.parametrize("width", [64, 5])
def test_peer_push_rows_more_segments_than_peers(width):
    """20 segments (the kernel's binary-search instantiation; 7 peers x 4 types of an 8-rank REGConv is 28), each with its
    own source table and local destination buffer, some empty; no flags.  width 5: the scalar (non-float4) kernel."""
    import ctypes

    from egc_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(3)
    n_seg = 20
    counts = [int(c) for c in torch.randint(0, 300, (n_seg,), generator=gen)]
    counts[3] = counts[11] = 0
    counts[7] = 5000
    srcs = [torch.randn(int(torch.randint(1, 400, (1,), generator=gen)), width, generator=gen).to(dev) for _ in range(n_seg)]
    idx = [torch.randint(0, s.size(0), (c,), generator=gen) for s, c in zip(srcs, counts)]
    dsts = [torch.full((c, width), float("nan"), device=dev) for c in counts]
    index = torch.cat(idx).to(dev, torch.int32)
    seg_ptr = (ctypes.c_int32 * (n_seg + 1))()
    for s, c in enumerate(counts):
        seg_ptr[s + 1] = seg_ptr[s] + c
    src_arr = (ctypes.c_void_p * n_seg)(*[s.data_ptr() for s in srcs])
    dst_arr = (ctypes.c_void_p * n_seg)(*[d.data_ptr() if d.numel() else 0 for d in dsts])
    with torch.cuda.device(dev):
        _lib.check(lib.egc_peer_push_rows(n_seg, src_arr, dst_arr, seg_ptr, index.data_ptr(), width, None, 1, 0, 0, None,
                                          None, torch.cuda.current_stream().cuda_stream), "egc_peer_push_rows")
    torch.cuda.synchronize()
    for s in range(n_seg):
        assert torch.equal(dsts[s], srcs[s].index_select(0, idx[s].to(dev))), s
    too_many = (ctypes.c_int32 * (_lib.MAX_PUSH_SEGMENTS + 2))()
    ptrs = (ctypes.c_void_p * (_lib.MAX_PUSH_SEGMENTS + 1))()
    assert lib.egc_peer_push_rows(_lib.MAX_PUSH_SEGMENTS + 1, ptrs, ptrs, too_many, None, width, None, 1, 0, 0, None, None,
                                  torch.cuda.current_stream().cuda_stream) != 0


def _guards_worker(rank, world, port, ret):
    import egc_b200
    from egc_b200.dist import PartitionedHeteroGraph
    dev = _init(rank, world, port)
    phg = None
    try:
        with pytest.raises(NotImplementedError):
            egc_b200.REGConv(64, 128, 8, 4, storage_dtype=torch.bfloat16)
        adj = _adj(dev)
        adj[("paper", "written_by", "author")] = adj[("paper", "to", "author")]
        phg = PartitionedHeteroGraph.from_global(adj, SIZES, rank, world, dev)
        conv = egc_b200.REGConv(64, 128, 8, 4).to(dev)
        x, _ = _data(1)
        with pytest.raises(ValueError, match="written_by"):
            conv({t: v.to(dev) for t, v in x.items()}, phg)
        with pytest.raises(ValueError):
            PartitionedHeteroGraph.from_global(_adj(dev), {**SIZES, "institution": 0}, rank, world, dev)
        ret[rank] = "ok"
    finally:
        if phg is not None:
            phg.close()
        dist.destroy_process_group()


def test_partitioned_regconv_guards():
    _run(_guards_worker, 1)


# ------------------------------------------------------------------------------------------------
# ranks: one process per GPU
# ------------------------------------------------------------------------------------------------
def _ranks_worker(rank, world, port, ret, transport, full):
    import egc_b200
    from egc_b200.dist import GraphedStep, PartitionedHeteroGraph
    dev = _init(rank, world, port)
    phg = None
    try:
        adj = _adj(dev)
        torch.manual_seed(0)
        conv = egc_b200.REGConv(64, 128, 8, 4).to(dev)
        conv2 = egc_b200.REGConv(128, 128, 8, 4).to(dev)
        params, params2 = list(conv.parameters()), list(conv.parameters()) + list(conv2.parameters())
        phg = PartitionedHeteroGraph.from_global(adj, SIZES, rank, world, dev, transport=transport)
        assert all(phg.part.tables[t].n_halo > 0 for t in TYPES)

        def step(x, go, tag):
            ref = _grads(lambda xs: conv(xs, adj), x, go, params, dev)
            got = _grads(lambda xs: conv(xs, phg), _local(x, phg), _local(go, phg), params, dev)
            _check(got, ref, phg, tag, (1e-6, 1e-5))

        for it in range(3 if full else 1):              # fresh data: epoch flags and buffer reuse
            step(*_data(10 + it), f"step {it}")
        phg.check()
        if full:
            x, go = _data(3)
            with torch.no_grad():                       # no_grad twice, then a training step
                for _ in range(2):
                    out = conv({t: v.to(dev) for t, v in _local(x, phg).items()}, phg)
                    out_ref = conv({t: v.to(dev) for t, v in x.items()}, adj)
                    for t in TYPES:
                        assert rel_err(out[t], out_ref[t][slice(*phg.row_range(t))]) < 1e-6, t
            step(x, go, "after no_grad")
            phg.check()
            relu = lambda d: {t: torch.relu(v) for t, v in d.items()}     # noqa: E731
            ref = _grads(lambda xs: conv2(relu(conv(xs, adj)), adj), x, go, params2, dev)
            got = _grads(lambda xs: conv2(relu(conv(xs, phg)), phg), _local(x, phg), _local(go, phg), params2, dev)
            _check(got, ref, phg, "two layers", (1e-5, 2e-5))
            phg.check()
        if transport == "peer":
            import gc
            gc.collect()
            x, go = _data(40)
            x_static = {t: v.to(dev).requires_grad_(True) for t, v in _local(x, phg).items()}
            go_static = {t: v.to(dev) for t, v in _local(go, phg).items()}

            def graphed_step():
                out = conv(x_static, phg)
                loss = sum((out[t] * go_static[t]).sum() for t in TYPES)
                return (out,) + torch.autograd.grad(loss, [x_static[t] for t in TYPES] + params)

            graphed = GraphedStep(graphed_step, warmup=2)
            phg.check()
            for it in range(3 if full else 1):
                x, go = _data(50 + it)
                with torch.no_grad():
                    for t in TYPES:
                        x_static[t].copy_(_local(x, phg)[t].to(dev))
                        go_static[t].copy_(_local(go, phg)[t].to(dev))
                res = graphed.replay()
                ref = _grads(lambda xs: conv(xs, adj), x, go, params, dev)
                _check((res[0], res[1:]), ref, phg, f"replay {it}", (1e-6, 1e-5))
            phg.check()
        torch.cuda.synchronize()
        ret[rank] = "ok"
    finally:
        if phg is not None:
            phg.close()
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("transport", ["peer", "nccl"])
def test_partitioned_regconv_matches_single_gpu_world2(transport):
    _run(_ranks_worker, 2, transport, True)


@pytest.mark.skipif(torch.cuda.device_count() < 4, reason="needs 4 GPUs")
def test_partitioned_regconv_matches_single_gpu_world4():
    """One step and one replay: the pushes run 12 (peer, type) segments over real peers."""
    _run(_ranks_worker, 4, "peer", False)
