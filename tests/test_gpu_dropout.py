"""Fused dropout after the ReLU (include/egc_b200.h, egc_dropout) on the device.

Forward: for every kernel family the dispatch can select, out == where(keep, out_relu * k, 0) BIT FOR BIT, with out_relu the
same layer without dropout and keep from the host Philox model (tests/dropout_model.py).  Backward: every gradient equals the
unfused composition (fused-ReLU layer, then torch ops with the same mask).  Statistics of the mask, the argument guards (Python
and C), the EGC stack (eval mode unchanged, training = the documented seed order, CUDA-graph replays draw fresh masks) and the
row-partitioned layer (each rank's rows of the single-GPU mask)."""
import os
import socket
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import egc_b200
from egc_b200 import _lib
from egc_b200.functional import draw_dropout_seed, egconv
from tests.dropout_model import dropout_constants, keep_mask
from tests.util import random_graph, rel_err, to_adj_csr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5                   # the fp32 bar of tests/test_gpu_parity.py
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _seed_value(seed: torch.Tensor) -> int:
    return int(seed.item()) & 0xFFFFFFFFFFFFFFFF


def _keep(seed, row0, n, hd, p):
    return torch.from_numpy(keep_mask(_seed_value(seed), row0, n, hd, p)).to(DEV)


class Layer:
    """Parameters + prepared graph of one layer, called through functional.egconv."""

    def __init__(self, n, e, f_in, heads, bases, dim, aggrs, seed=0, hub=0, valued=False, storage=torch.float32,
                 deterministic=True):
        gen = torch.Generator().manual_seed(seed)
        ei = random_graph(n, e, seed=seed, hub=hub)
        symnorm = "symnorm" in aggrs
        if valued:
            rowptr, col, _ = to_adj_csr(ei, n)
            value = torch.rand(col.numel(), generator=gen) + 0.5
            self.graph = egc_b200.GraphStructure.from_csr(rowptr.to(DEV), col.to(DEV), value.to(DEV), n, symnorm, True)
            assert self.graph.val_lin is not None
        else:
            self.graph = egc_b200.GraphStructure.from_edge_index(ei.to(DEV), n, symnorm, True)
        self.heads, self.bases, self.aggrs, self.storage = heads, bases, list(aggrs), storage
        self.hd = heads * dim
        a = (6.0 / (f_in + bases * dim)) ** 0.5
        self.wb = ((torch.rand(f_in, bases * dim, generator=gen) * 2 - 1) * a).to(DEV).requires_grad_(True)
        self.wc = (torch.randn(heads * len(aggrs) * bases, f_in, generator=gen) / f_in ** 0.5).to(DEV).requires_grad_(True)
        self.bc = (torch.randn(heads * len(aggrs) * bases, generator=gen) * 0.1).to(DEV).requires_grad_(True)
        self.b = (torch.randn(self.hd, generator=gen) * 0.1).to(DEV).requires_grad_(True)
        self.x = torch.randn(n, f_in, generator=gen).to(DEV).requires_grad_(True)
        self.go = torch.randn(n, self.hd, generator=gen).to(DEV)
        self.flags = _lib.BWD_DETERMINISTIC if deterministic else 0
        self.n = n

    @property
    def params(self):
        return [self.x, self.wb, self.wc, self.bc, self.b]

    def __call__(self, relu=True, dropout=0.0, seed=None, **kw):
        return egconv(self.x, self.graph, self.wb, self.wc, self.bc, self.b, self.heads, self.bases, self.aggrs, False,
                      bwd_flags=self.flags, relu=relu, storage_dtype=self.storage, dropout=dropout, dropout_seed=seed, **kw)


ARXIV = 169343
FWD_CASES = {
    # name: (n, e, f_in, heads, bases, dim, aggrs, extra)
    "arxiv_rows_static": (ARXIV, 1_166_243, 128, 4, 4, 32, ["symnorm", "max", "std"], {}),
    "static_long_rows": (30000, 240000, 64, 4, 4, 32, ["symnorm", "max", "std"], {"hub": 700}),
    "rows_g16_dynamic": (20000, 150000, 32, 4, 2, 24, ["sum", "max"], {"hub": 700}),
    "scalar_tail_d13": (20000, 150000, 32, 8, 4, 13, ["sum"], {"hub": 700}),
    "general_kernel_bd176": (12000, 90000, 32, 8, 4, 44, ["symnorm", "mean"], {"hub": 700}),
    "valued_adjacency": (12000, 90000, 32, 4, 4, 16, ["sum", "max"], {"valued": True, "hub": 700}),
    "bf16_static": (30000, 240000, 64, 4, 4, 32, ["symnorm", "max", "std"], {"storage": torch.bfloat16, "hub": 700}),
    "bf16_dynamic_g8": (20000, 150000, 32, 4, 4, 10, ["sum", "mean"], {"storage": torch.bfloat16, "hub": 700}),
}


def _check_forward(case, p=0.5):
    n, e, f_in, heads, bases, dim, aggrs, extra = FWD_CASES[case]
    layer = Layer(n, e, f_in, heads, bases, dim, aggrs, **extra)
    with torch.no_grad():
        ref = layer(relu=True)
        seed = draw_dropout_seed(DEV)
        out = layer(relu=True, dropout=p, seed=seed)
        again = layer(relu=True, dropout=p, seed=seed)
    keep = _keep(seed, 0, n, layer.hd, p)
    _, k = dropout_constants(p)
    expect = torch.where(keep, ref * k, torch.zeros_like(ref))
    assert (ref > 0).any() and (ref == 0).any()
    assert torch.equal(out, expect), f"{case}: {(out != expect).sum().item()} outputs differ"
    assert torch.equal(out, again)


@pytest.mark.parametrize("case", list(FWD_CASES))
def test_forward_bit_exact(case):
    _check_forward(case)


def test_forward_bit_exact_warp_per_row_kernel():
    """EGC_FWD_WARP_PER_ROW is read once per process: a fresh interpreter runs the cases on the warp-per-row kernel, its
    statically configured instantiation (the arxiv layer shape) and its dynamic ones."""
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_dropout import _check_forward; "
            "[_check_forward(c) for c in ('static_long_rows', 'rows_g16_dynamic', 'scalar_tail_d13')]; print('ok')" % ROOT)
    env = dict(os.environ, EGC_FWD_WARP_PER_ROW="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-2000:] + r.stderr[-4000:]


BWD_CASES = ["rows_g16_dynamic", "scalar_tail_d13", "general_kernel_bd176", "valued_adjacency", "bf16_static"]


@pytest.mark.parametrize("case", BWD_CASES)
def test_backward_matches_unfused_composition(case):
    n, e, f_in, heads, bases, dim, aggrs, extra = FWD_CASES[case]
    layer = Layer(n, e, f_in, heads, bases, dim, aggrs, **extra)
    p = 0.3
    seed = draw_dropout_seed(DEV)
    keep = _keep(seed, 0, n, layer.hd, p)
    _, k = dropout_constants(p)
    y = layer(relu=True)
    ref = torch.where(keep, y * k, torch.zeros_like(y))
    g_ref = torch.autograd.grad(ref, layer.params, layer.go)
    out = layer(relu=True, dropout=p, seed=seed)
    g = torch.autograd.grad(out, layer.params, layer.go)
    assert torch.equal(out, ref.detach())
    bitwise = [torch.equal(a, b) for a, b in zip(g, g_ref)]
    print(f"{case}: gradients bit-identical to the unfused composition: {bitwise}")
    for name, a, b in zip(("d_x", "d_bases_weight", "d_comb_weight", "d_comb_bias", "d_bias"), g, g_ref):
        assert rel_err(a, b) <= TOL, name


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_mask_statistics(p):
    """A layer whose ReLU output is 1 everywhere (zero weights, bias 1): out = k where kept, 0 where dropped."""
    n, hd = 80000, 128
    ei = random_graph(n, 4 * n, seed=3)
    g = egc_b200.GraphStructure.from_edge_index(ei.to(DEV), n, True, True)
    wb = torch.zeros(32, 4 * 32, device=DEV)
    wc = torch.zeros(4 * 4, 32, device=DEV)
    bias = torch.ones(hd, device=DEV)
    x = torch.randn(n, 32, device=DEV)

    def run(seed):
        with torch.no_grad():
            return egconv(x, g, wb, wc, None, bias, 4, 4, ["symnorm"], relu=True, dropout=p, dropout_seed=seed)

    s1, s2 = draw_dropout_seed(DEV), draw_dropout_seed(DEV)
    o1, o1b, o2 = run(s1), run(s1.clone()), run(s2)
    _, k = dropout_constants(p)
    kept = o1 != 0
    assert torch.equal(o1[kept], torch.full_like(o1[kept], k))
    m = n * hd                                                     # 10.24 M outputs
    frac = kept.double().mean().item()
    assert abs(frac - (1 - p)) <= 5 * (p * (1 - p) / m) ** 0.5, frac
    col = kept.double().mean(0)
    assert ((col - (1 - p)).abs() <= 5 * (p * (1 - p) / n) ** 0.5).all(), (col.min().item(), col.max().item())
    assert torch.equal(o1, o1b)                                    # same seed, same mask
    assert _seed_value(s1) != _seed_value(s2) and not torch.equal(kept, o2 != 0)
    assert torch.equal(kept.cpu(), torch.from_numpy(keep_mask(_seed_value(s1), 0, n, hd, p)))


def test_guards_python():
    layer = Layer(2000, 10000, 16, 4, 4, 8, ["symnorm"])
    seed = draw_dropout_seed(DEV)
    for bad in (-0.1, 1.0, 1.5):
        with pytest.raises(ValueError):
            layer(relu=True, dropout=bad, seed=seed)
    with pytest.raises(ValueError):
        layer(relu=False, dropout=0.5, seed=seed)
    hd = layer.hd
    one = torch.ones(hd, device=DEV)
    for kw in ({"scale": one, "shift": one}, {"residual": torch.zeros(layer.n, hd, device=DEV)}):
        with pytest.raises(ValueError):
            layer(relu=True, dropout=0.5, seed=seed, **kw)
    with pytest.raises(ValueError):                                # a seed that is not one int64 word
        layer(relu=True, dropout=0.5, seed=torch.zeros(2, dtype=torch.int64, device=DEV))
    assert torch.equal(layer(relu=True, dropout=0.0), layer(relu=True))     # p = 0: no dropout


def test_guards_c_abi():
    from egc_b200.functional import alloc_aggregate_outputs, make_desc, project
    from egc_b200.graph import _stream, _ws
    lib = _lib.load()
    layer = Layer(2000, 10000, 16, 4, 4, 16, ["symnorm"])
    g = layer.graph
    with torch.no_grad():
        bases, w = project(layer.x, layer.wb, layer.wc, layer.bc, False)
    seed = draw_dropout_seed(DEV)
    one = torch.ones(layer.hd, device=DEV)

    def call(relu, p, epilogue=None, bf16=False):
        desc = make_desc(g, 4, 4, 16, ["symnorm"], False, relu)
        out = alloc_aggregate_outputs(desc, DEV)[0]
        nbytes = lib.egc_aggregate_fwd_workspace_bytes(desc, g.plan.struct)
        ws = _ws(nbytes, torch.device(DEV))
        drop = _lib.Dropout(seed.data_ptr(), p, 0)
        if bf16:
            b16 = bases.to(torch.bfloat16)
            return lib.egc_aggregate_fwd_bf16_dropout(desc, _lib.ptr(g.rowptr), _lib.ptr(g.col), _lib.ptr(g.val_sym),
                                                      g.plan.struct, _lib.ptr(b16), _lib.ptr(w), None, epilogue, drop,
                                                      _lib.ptr(out), None, None, None, None, _lib.ptr(ws), nbytes, _stream())
        return lib.egc_aggregate_fwd_dropout(desc, _lib.ptr(g.rowptr), _lib.ptr(g.col), _lib.ptr(g.val_sym), None,
                                             g.plan.struct, _lib.ptr(bases), _lib.ptr(w), None, epilogue, drop, None, 0,
                                             _lib.ptr(out), None, None, None, None, _lib.ptr(ws), nbytes, _stream())

    scale = _lib.Epilogue(one.data_ptr(), one.data_ptr(), None, None)
    add = _lib.Epilogue(None, None, torch.zeros(layer.n, layer.hd, device=DEV).data_ptr(), None)
    for bf16 in (False, True):
        assert call(True, 0.5, bf16=bf16) == 0
        assert call(True, 0.0, bf16=bf16) == 0
        for relu, p, epi in ((True, 1.0, None), (True, -0.5, None), (True, float("nan"), None), (False, 0.5, None),
                             (True, 0.5, scale), (True, 0.5, add)):
            assert call(relu, p, epi, bf16) == -1, (relu, p, bf16)     # EGC_ERR_INVALID_ARGUMENT
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------
# the EGC stack
# ------------------------------------------------------------------------------------------------
def _stack(fused, seed=0, storage=torch.float32):
    torch.manual_seed(seed)
    return egc_b200.EGC(64, 3, 0.5, 4, 4, ["symnorm", "max", "std"], in_features=32, out_rounded=40, out_true=37,
                        fused_dropout=fused, storage_dtype=storage, deterministic=True).to(DEV)


def _stack_graph(n=6000):
    ei = random_graph(n, 40000, seed=11, hub=600)
    gen = torch.Generator().manual_seed(12)
    return ei.to(DEV), torch.randn(n, 32, generator=gen).to(DEV), torch.randn(n, 37, generator=gen).to(DEV)


def _compose(model, x, g, seeds):
    """The stack as functional calls with the given dropout seeds (one per hidden layer, in layer order)."""
    h = x
    for i, conv in enumerate(model.convs):
        last = i == len(model.convs) - 1
        h = egconv(h, g, conv.bases_weight, conv.comb_weight.weight, conv.comb_weight.bias, conv.bias, conv.num_heads,
                   conv.num_bases, conv.aggregators, conv.sigmoid, conv.gemm_algo, _lib.BWD_DETERMINISTIC, relu=not last,
                   storage_dtype=conv.storage_dtype, dropout=0.0 if last else model.dropout,
                   dropout_seed=None if last else seeds[i])
    return h[:, :model.out_true].log_softmax(dim=-1)


@pytest.mark.parametrize("storage", [torch.float32, torch.bfloat16])
def test_stack_eval_mode_unchanged(storage):
    ei, x, _ = _stack_graph()
    a, b = _stack(False, storage=storage).eval(), _stack(True, storage=storage).eval()
    with torch.no_grad():
        assert torch.equal(a(x, ei), b(x, ei))
    assert b.last_dropout_seeds == []


@pytest.mark.parametrize("storage", [torch.float32, torch.bfloat16])
def test_stack_training_follows_the_seed_order(storage):
    ei, x, go = _stack_graph()
    model = _stack(True, storage=storage).train()
    g = model.prepare(x, ei)
    torch.manual_seed(123)
    out = model(x, ei)
    grads = torch.autograd.grad(out, list(model.parameters()), go)
    torch.manual_seed(123)
    seeds = [draw_dropout_seed(DEV) for _ in range(len(model.convs) - 1)]      # one per hidden layer, in layer order
    assert [int(s) for s in model.last_dropout_seeds] == [int(s) for s in seeds]
    ref = _compose(model, x, g, seeds)
    grads_ref = torch.autograd.grad(ref, list(model.parameters()), go)
    assert torch.equal(out, ref)
    for a, b in zip(grads, grads_ref):
        assert torch.equal(a, b)
    # the unfused stack (torch's F.dropout) draws other masks: same parameters, different output
    torch.manual_seed(123)
    unfused = _stack(False, storage=storage).train()
    assert not torch.equal(unfused(x, ei), out)


def test_stack_graph_replays_draw_fresh_masks():
    ei, x, go = _stack_graph()
    model = _stack(True).train()
    g = model.prepare(x, ei)
    params = list(model.parameters())

    def step():
        o = model(x, g)
        return [o] + list(torch.autograd.grad(o, params, go))

    graphed = egc_b200.GraphedStep(step, warmup=2)
    seed_bufs = list(model.last_dropout_seeds)                     # the captured seed buffers
    assert len(seed_bufs) == 2
    masks = []
    for _ in range(2):
        res = [t.clone() for t in graphed.replay()]
        torch.cuda.synchronize()
        seeds = [s.clone() for s in seed_bufs]
        ref = _compose(model, x, g, seeds)
        grads_ref = torch.autograd.grad(ref, params, go)
        assert torch.equal(res[0], ref)
        for a, b in zip(res[1:], grads_ref):
            assert rel_err(a, b) <= TOL
        masks.append([int(s) for s in seeds])
    assert masks[0] != masks[1]


# ------------------------------------------------------------------------------------------------
# row-partitioned layer
# ------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dist_worker(rank, world, port, n, ei, x, go, transport, seed_value, ret, aggrs, env):
    os.environ.update(env)
    from egc_b200.dist import PartitionedGraph, partitioned_egconv
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    pg = None
    try:
        torch.manual_seed(0)
        conv = egc_b200.EGConv(64, 128, aggrs=aggrs, num_heads=4, num_bases=4, deterministic=True).to(dev)
        params = list(conv.parameters())
        eid = ei.to(dev)
        g = egc_b200.GraphStructure.from_edge_index(eid, n, True, True)
        pg = PartitionedGraph.from_global(g, rank, world, dev, transport=transport)
        b, e = pg.part.row_begin, pg.part.row_end
        assert pg.overlap_interior or world > 1           # one rank: the interior / boundary row-subset launches
        # the overlapped exchange: own-column launch, then the halo launch continuing its sums (agg_init) with dropout
        assert pg.uses_overlap(aggrs) == (env.get("EGC_DIST_OVERLAP") == "1" and transport == "peer" and world > 1)
        seed = torch.tensor([seed_value], dtype=torch.int64, device=dev)
        p = 0.4
        xs = x.to(dev).requires_grad_(True)
        ref = conv(xs, eid, relu=True, dropout=p, dropout_seed=seed)
        g_ref = torch.autograd.grad(ref, [xs] + params, go.to(dev))
        xl = x[b:e].to(dev).requires_grad_(True)
        out = partitioned_egconv(xl, pg, conv, relu=True, dropout=p, dropout_seed=seed)
        grads = torch.autograd.grad(out, [xl] + params, go[b:e].to(dev))
        assert torch.equal(out, ref[b:e])
        assert rel_err(grads[0], g_ref[0][b:e]) < 1e-5
        for a, r in zip(grads[1:], g_ref[1:]):
            assert rel_err(a, r) < 1e-5
        # without an explicit seed every rank draws it from its own generator: identical seeding -> one global mask
        torch.manual_seed(77)
        out2 = partitioned_egconv(xl, pg, conv, relu=True, dropout=p)
        torch.manual_seed(77)
        ref2 = conv(xs, eid, relu=True, dropout=p)
        assert torch.equal(out2, ref2[b:e])
        torch.cuda.synchronize()
        ret[rank] = "ok"
    finally:
        if pg is not None:
            try:
                pg.close()
            except Exception:
                pass
        dist.destroy_process_group()


def _dist_inputs():
    n = 4000
    ei = random_graph(n, 30000, seed=5, hub=900)
    blk = torch.randint(0, n // 2, (2, 15000), generator=torch.Generator().manual_seed(6))
    ei = torch.cat([ei, blk, blk + n // 2], 1)
    gen = torch.Generator().manual_seed(1)
    return n, ei, torch.randn(n, 64, generator=gen), torch.randn(n, 128, generator=gen)


@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("transport", ["peer", "nccl"])
@pytest.mark.parametrize("aggrs,overlap", [(["symnorm", "max", "std"], "0"), (["symnorm"], "1")],
                         ids=["egc_m", "symnorm_overlap"])
def test_partitioned_rows_match_single_gpu(world, transport, aggrs, overlap):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    n, ei, x, go = _dist_inputs()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_dist_worker, args=(world, _free_port(), n, ei, x, go, transport, 0x5DEECE66D1234567, ret, aggrs,
                                 {"EGC_DIST_OVERLAP": overlap}), nprocs=world, join=True)
    assert dict(ret) == {r: "ok" for r in range(world)}
