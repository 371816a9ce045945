"""Pins the CPU oracle (oracle/restatement.py): against the golden vectors generated from the
UNMODIFIED reference source (tests/golden, made by oracle/make_golden.py) and, where
the reference sources are present (oracle/reference_loader.py), against the reference itself executed through oracle/shims."""
import itertools

import pytest
import torch

from oracle import reference_loader as rl
from oracle import restatement as R
from tests.util import golden_cases, load_golden, random_graph, rel_err, to_adj_csr


def oracle_from_golden(rec, dtype):
    m = R.EGConvOracle(rec["f_in"], rec["f_out"], aggrs=rec["aggrs"], num_heads=rec["heads"], num_bases=rec["bases"],
                       add_self_loops=rec["add_self_loops"], bias="bias" in rec["state_dict"],
                       sigmoid=rec["sigmoid"]).to(dtype)
    m.load_state_dict({k: v.to(dtype) for k, v in rec["state_dict"].items()})
    if rec["kind"] == "edge_index":
        gi = rec["edge_index"]
    else:
        v = rec["adj_value"]
        gi = (rec["adj_rowptr"], rec["adj_col"], v.to(dtype) if v is not None else None)
    return m, gi


@pytest.mark.parametrize("name", golden_cases())
def test_restatement_matches_golden(name):
    rec = load_golden(name)
    for tag, dt, tol in (("f64", torch.float64, 1e-11), ("f32", torch.float32, 2e-5)):
        m, gi = oracle_from_golden(rec, dt)
        x = rec["x"].to(dt).requires_grad_(True)
        out = m(x, gi)
        params = list(m.named_parameters())
        grads = torch.autograd.grad(out, [x] + [p for _, p in params], rec["grad_out"].to(dt))
        assert rel_err(out, rec[f"out_{tag}"]) < tol
        assert rel_err(grads[0], rec[f"grad_x_{tag}"]) < tol
        for (pn, _), g in zip(params, grads[1:]):
            assert rel_err(g, rec[f"grad_{pn}_{tag}"]) < tol, pn


@pytest.mark.parametrize("name", golden_cases())
def test_prepared_graph_matches_golden_bit_exact(name):
    """CSR / self-loops / degree-normalisation exactly as the reference's helpers produce them."""
    rec = load_golden(name)
    sym = "symnorm" in rec["aggrs"]
    n = rec["n"]
    if rec["kind"] == "edge_index":
        g = R.graph_from_edge_index(rec["edge_index"], n, sym, rec["add_self_loops"])
        ei2 = rec["prep_edge_index"]
        order = torch.argsort(ei2[1], stable=True)
        assert torch.equal(g.col, ei2[0][order])
        assert torch.equal(g.row, ei2[1][order])
        if sym:
            assert torch.equal(g.val_sym, rec["prep_weight"][order])
    else:
        g = R.graph_from_csr(rec["adj_rowptr"], rec["adj_col"], rec["adj_value"], n, sym, rec["add_self_loops"], True)
        assert torch.equal(g.rowptr, rec["prep_rowptr"])
        assert torch.equal(g.col, rec["prep_col"])
        if sym:
            assert torch.equal(g.val_sym, rec["prep_value"])
        elif rec["prep_value"] is not None:
            assert torch.equal(g.val_lin, rec["prep_value"])


def test_analytic_backward_matches_autograd():
    torch.manual_seed(0)
    n, f_in, f_out, h, b = 90, 12, 32, 4, 4
    ei = random_graph(n, 500, seed=3)
    for aggrs, sig in itertools.product((["symnorm", "max", "std"], ["sum", "mean", "min", "var"]), (False, True)):
        m = R.EGConvOracle(f_in, f_out, aggrs=aggrs, num_heads=h, num_bases=b, sigmoid=sig).double()
        x = torch.randn(n, f_in, dtype=torch.float64, requires_grad=True)
        go = torch.randn(n, f_out, dtype=torch.float64)
        out = m(x, ei)
        auto = torch.autograd.grad(out, [x, m.bases_weight, m.comb_weight.weight, m.comb_weight.bias, m.bias], go)
        man = R.egconv_backward(x.detach(), m.prepare(x, ei), m.bases_weight.detach(), m.comb_weight.weight.detach(),
                                m.comb_weight.bias.detach(), m.bias.detach(), aggrs, h, go, sig)
        for a, key in zip(auto, ("d_x", "d_bases_weight", "d_comb_weight", "d_comb_bias", "d_bias")):
            assert rel_err(man[key], a) < 1e-12, key


def test_gradcheck_fp64():
    torch.manual_seed(1)
    n = 24
    ei = random_graph(n, 60, seed=5, isolated=1, self_loops=2, dups=4)
    m = R.EGConvOracle(6, 8, aggrs=["symnorm", "mean", "var"], num_heads=2, num_bases=2).double()
    x = torch.randn(n, 6, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda t: m(t, ei), (x,), eps=1e-6, atol=1e-6)


def test_hand_computed_tiny_graph():
    """SURVEY.md App. A-9 consequences on a 4-node graph: 0 <- 1, 0 <- 2 (twice), node 3 isolated."""
    ei = torch.tensor([[1, 2, 2], [0, 0, 0]])
    bases = torch.tensor([[1.0, -1.0], [2.0, 5.0], [4.0, 3.0], [7.0, 7.0]])
    g = R.graph_from_edge_index(ei, 4, symnorm=True, add_self_loops=True)
    assert g.rowptr.tolist() == [0, 4, 5, 6, 7] and g.col.tolist() == [1, 2, 2, 0, 1, 2, 3]
    assert g.deg.tolist() == [4.0, 1.0, 1.0, 1.0]
    agg, arg = R.aggregate(g, bases, ["sum", "mean", "max", "min", "var", "std", "symnorm"])
    assert agg[0, 0].tolist() == [11.0, 10.0]                 # multi-edge counted twice, + self-loop
    assert agg[0, 1].tolist() == [2.75, 2.5]
    assert agg[0, 2].tolist() == [4.0, 5.0] and agg[0, 3].tolist() == [1.0, -1.0]
    assert arg["max"][0].tolist() == [1, 0]                   # first of the duplicated edge wins the tie
    assert agg[3, 4].tolist() == [0.0, 0.0]                   # isolated + loop: var exactly 0
    assert torch.allclose(agg[3, 5], torch.full((2,), 1e-5).sqrt())
    assert torch.allclose(agg[0, 6], (bases[1] + 2 * bases[2]) * 0.5 + bases[0] * 0.25)
    g2 = R.graph_from_edge_index(ei, 4, symnorm=False, add_self_loops=False)
    agg2, _ = R.aggregate(g2, bases, ["max", "std"])
    assert agg2[3, 0].tolist() == [0.0, 0.0]                  # empty row -> 0 for max
    assert torch.allclose(agg2[3, 1], torch.full((2,), 1e-5).sqrt())
    # add_remaining_self_loops without num_nodes: node 3 (> max id 2) gets no loop (ref :164)
    g3 = R.graph_from_edge_index(ei, 4, symnorm=False, add_self_loops=True)
    assert g3.rowptr.tolist() == [0, 4, 5, 6, 6]


@pytest.mark.skipif(not rl.available(), reason="needs the reference sources (oracle/_ref or EGC_REFERENCE_ROOT)")
def test_restatement_matches_reference_source():
    ref = rl.load()
    n = 150
    ei = random_graph(n, 1200, seed=0, isolated=3, self_loops=10, dups=50)
    worst = 0.0
    for aggrs, loops, sig, kind in itertools.product(
            (["symnorm"], ["sum"], ["symnorm", "max", "std"], ["sum", "mean", "min", "var"], ["max", "min", "std", "mean"]),
            (True, False), (False, True), ("ei", "csr", "csrv")):
        torch.manual_seed(1)
        conv = ref.EGConv(16, 32, aggrs=aggrs, num_heads=4, num_bases=4, add_self_loops=loops, sigmoid=sig).double()
        with torch.no_grad():
            conv.bias.normal_()
        o = R.EGConvOracle(16, 32, aggrs=aggrs, num_heads=4, num_bases=4, add_self_loops=loops, sigmoid=sig).double()
        o.load_state_dict(conv.state_dict())
        x = torch.randn(n, 16, dtype=torch.float64, requires_grad=True)
        if kind == "ei":
            a_ref, a_or = ei, ei
        else:
            val = torch.rand(ei.size(1), dtype=torch.float64) + 0.5 if kind == "csrv" else None
            rowptr, col, v = to_adj_csr(ei, n, val)
            a_ref = ref.SparseTensor(rowptr=rowptr, col=col, value=v, sparse_sizes=(n, n), is_sorted=True)
            a_or = (rowptr, col, v)
        go = torch.randn(n, 32, dtype=torch.float64)
        g_ref = torch.autograd.grad(conv(x, a_ref), [x] + list(conv.parameters()), go)
        g_or = torch.autograd.grad(o(x, a_or), [x] + list(o.parameters()), go)
        worst = max(worst, rel_err(o(x, a_or), conv(x, a_ref)), *(rel_err(a, b) for a, b in zip(g_or, g_ref)))
    assert worst < 1e-12


@pytest.mark.skipif(not rl.available(), reason="needs the reference sources (oracle/_ref or EGC_REFERENCE_ROOT)")
def test_paper_layer_agrees_with_fused_layer():
    """Secondary pin (SURVEY.md App. B): EfficientGraphConv == EGConv under the weight permutation when
    add_self_loops=False (the only setting where their self-loop rules coincide)."""
    ref = rl.load()
    torch.manual_seed(0)
    n, f_in, f_out, h, b = 120, 10, 24, 4, 3
    ei = random_graph(n, 700, seed=9)
    for new_aggrs, old_aggrs in ((["symnorm", "max", "std"], ["symadd", "max", "std"]),
                                 (["sum", "mean", "min", "var"], ["add", "mean", "min", "var"])):
        a = len(new_aggrs)
        new = ref.EGConv(f_in, f_out, aggrs=new_aggrs, num_heads=h, num_bases=b, add_self_loops=False).double()
        old = ref.EfficientGraphConv(f_in, f_out, h, b, softmax_weights=False, add_self_loops=False,
                                     aggrs=old_aggrs).double()
        perm = [hh * a * b + aa * b + bb for hh in range(h) for bb in range(b) for aa in range(a)]
        d = f_out // h
        with torch.no_grad():
            old.comb_weights.weight.copy_(new.comb_weight.weight[perm])
            old.comb_weights.bias.copy_(new.comb_weight.bias[perm])
            for k in range(b):
                old.bases_weight[k].copy_(new.bases_weight[:, k * d:(k + 1) * d])
        x = torch.randn(n, f_in, dtype=torch.float64)
        assert rel_err(old(x, ei), new(x, ei)) < 1e-12


@pytest.mark.parametrize("name", golden_cases("paper_"))
def test_paper_restatement_matches_golden(name):
    """The paper-variant fixtures (generated from the unmodified experiments/layers.py) against the CPU
    restatement the adapter `egc_b200.EfficientGraphConv` follows: output and the gradient w.r.t. x."""
    rec = load_golden(name)
    sd = {k: v.double() for k, v in rec["state_dict"].items()}
    x = rec["x"].double().requires_grad_(True)
    gi = rec["edge_index"] if rec["kind"] == "edge_index" else (rec["adj_rowptr"], rec["adj_col"], None)
    out = R.paper_forward(x, gi, [sd[f"bases_weight.{i}"] for i in range(rec["bases"])], sd["comb_weights.weight"],
                          sd["comb_weights.bias"], sd.get("bias"), rec["aggrs"], rec["heads"],
                          add_self_loops=rec["add_self_loops"], post=rec["post"],
                          graph_dtype=torch.float32)      # gcn_norm materialises fp32 ones, as in the reference
    assert rel_err(out, rec["out_f64"]) < 1e-11
    (gx,) = torch.autograd.grad(out, [x], rec["grad_out"].double())
    assert rel_err(gx, rec["grad_x_f64"]) < 1e-10


def test_paper_to_egconv_permutation():
    from egc_b200.compat import paper_to_egconv_perm
    h, b, a = 3, 4, 2
    perm = paper_to_egconv_perm(h, b, a)
    expect = [hh * b * a + bb * a + aa for hh in range(h) for aa in range(a) for bb in range(b)]
    assert perm.tolist() == expect and sorted(perm.tolist()) == list(range(h * b * a))


ADJ_CASES = [n for n in golden_cases() + golden_cases("paper_") if load_golden(n)["kind"] != "edge_index"]


@pytest.mark.parametrize("name", ADJ_CASES)
def test_to_sparse_tensor_matches_the_golden_adjacency_bit_exact(name):
    """egc_b200.to_sparse_tensor against the adj_t the golden generator built from the same edge list with the
    reference's ordering (experiments/utils.py:93; duplicates, self-loops and isolated nodes kept): same rowptr, same
    column order."""
    import egc_b200
    rec = load_golden(name)
    rowptr, col, value = egc_b200.to_sparse_tensor(rec["edge_index"], rec["n"]).csr()
    assert value is None
    assert torch.equal(rowptr, rec["adj_rowptr"]) and torch.equal(col, rec["adj_col"])


@pytest.mark.skipif(not rl.available(), reason="needs the reference sources (oracle/_ref or EGC_REFERENCE_ROOT)")
def test_to_sparse_tensor_matches_the_reference_transform_bit_exact():
    """egc_b200.to_sparse_tensor == experiments/utils.py:82-118 ToSparseTensor (run through the shims) on an edge list
    with duplicates and self-loops: same rowptr, same column order."""
    import importlib
    from types import SimpleNamespace

    import egc_b200
    rl.load()
    try:
        utils = importlib.import_module("experiments.utils")
    except Exception as exc:                                   # the module pulls optional training dependencies
        pytest.skip(f"experiments.utils not importable here: {exc}")
    n = 300
    ei = random_graph(n, 2500, seed=21, hub=120)

    class Data(SimpleNamespace):
        def __iter__(self):
            return iter(list(vars(self).items()))

        def __setitem__(self, k, v):
            setattr(self, k, v)

    data = utils.ToSparseTensor()(Data(edge_index=ei.clone(), num_nodes=n, num_edges=ei.size(1)))
    rowptr_ref, col_ref, _ = data.adj_t.csr()
    mine = egc_b200.to_sparse_tensor(ei, n)
    rowptr, col, value = mine.csr()
    assert value is None and mine.sparse_sizes() == (n, n)
    assert torch.equal(rowptr, rowptr_ref) and torch.equal(col, col_ref)
