"""Heterogeneous layer REGConv (SURVEY.md section 8 f-2; ref experiments/rmag/models.py:75-148).
CPU: the restatement (oracle/hetero.py) against the golden vectors generated from the UNMODIFIED reference class and,
where the reference sources are present, against that class executed through the shims.  GPU: egc_b200.REGConv against the
goldens and the fp64 restatement, through the C ABI."""
import importlib

import pytest
import torch

from oracle import hetero as OH
from oracle import reference_loader as rl
from tests.util import golden_cases, load_golden, rel_err

CASES = golden_cases("regconv_")


def _oracle_from_golden(rec, dtype):
    m = OH.REGConvOracle(rec["f_in"], rec["f_out"], rec["heads"], rec["bases"]).to(dtype)
    m.load_state_dict({k: v.to(dtype) for k, v in rec["state_dict"].items()})
    return m


def _run(model, x, graph, go, types):
    out = model(x, graph)
    params = list(model.named_parameters())
    loss = sum((out[t] * go[t]).sum() for t in types)
    grads = torch.autograd.grad(loss, [x[t] for t in types] + [p for _, p in params])
    return out, dict(zip(types, grads[:len(types)])), {n: g for (n, _), g in zip(params, grads[len(types):])}


@pytest.mark.parametrize("name", CASES)
def test_restatement_matches_reference_golden(name):
    rec = load_golden(name)
    types = list(rec["sizes"])
    for tag, dt, tol in (("f64", torch.float64, 1e-11), ("f32", torch.float32, 2e-5)):
        m = _oracle_from_golden(rec, dt)
        x = {t: rec["x"][t].to(dt).requires_grad_(True) for t in types}
        go = {t: rec["grad_out"][t].to(dt) for t in types}
        out, gx, gp = _run(m, x, rec["csr"], go, types)
        for t in types:
            assert rel_err(out[t], rec[tag]["out"][t]) < tol, t
            assert rel_err(gx[t], rec[tag]["grad_x"][t]) < tol, t
        for n, g in gp.items():
            assert rel_err(g, rec[tag]["grad_p"][n]) < tol, n


@pytest.mark.skipif(not rl.available(), reason="needs the reference sources (oracle/_ref or EGC_REFERENCE_ROOT)")
def test_restatement_matches_reference_source():
    rl.load()
    ref = importlib.import_module("experiments.rmag.models")
    ST = rl.shims().SparseTensor
    sizes = {"author": 33, "field_of_study": 11, "institution": 5, "paper": 21}
    types = list(sizes)
    for seed in range(3):
        torch.manual_seed(seed)
        conv = ref.REGConv(12, 24, 4, 3).double()
        m = OH.REGConvOracle(12, 24, 4, 3).double()
        m.load_state_dict(conv.state_dict())
        csr = OH.random_hetero_graph(sizes, 90, seed)
        adj = {k: ST(rowptr=rp, col=col, sparse_sizes=(rp.numel() - 1, ns), is_sorted=True) for k, (rp, col, ns) in csr.items()}
        x = {t: torch.randn(n, 12, dtype=torch.float64) for t, n in sizes.items()}
        go = {t: torch.randn(n, 24, dtype=torch.float64) for t, n in sizes.items()}
        xa = {t: v.clone().requires_grad_(True) for t, v in x.items()}
        xb = {t: v.clone().requires_grad_(True) for t, v in x.items()}
        oa, gxa, gpa = _run(conv, xa, adj, go, types)
        ob, gxb, gpb = _run(m, xb, csr, go, types)
        for t in types:
            assert rel_err(ob[t], oa[t]) < 1e-12 and rel_err(gxb[t], gxa[t]) < 1e-12
        for n in gpa:
            assert rel_err(gpb[n], gpa[n]) < 1e-12, n


def test_state_dict_layout_matches_reference_names():
    import egc_b200
    rec = load_golden(CASES[0])
    c = egc_b200.REGConv(rec["f_in"], rec["f_out"], rec["heads"], rec["bases"])
    assert set(c.state_dict()) == set(rec["state_dict"])
    for k, v in c.state_dict().items():
        assert tuple(v.shape) == tuple(rec["state_dict"][k].shape), k
    with pytest.raises(ValueError):
        egc_b200.REGConv(16, 30, 4, 2)
    with pytest.raises(RuntimeError):                       # no CPU path
        c(rec["x"], {})


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_regconv_cuda_matches_reference_golden(name):
    import egc_b200
    rec = load_golden(name)
    types = list(rec["sizes"])
    conv = egc_b200.REGConv(rec["f_in"], rec["f_out"], rec["heads"], rec["bases"])
    conv.load_state_dict(rec["state_dict"])
    conv = conv.cuda()
    x = {t: rec["x"][t].cuda().requires_grad_(True) for t in types}
    go = {t: rec["grad_out"][t].cuda() for t in types}
    adj = {k: egc_b200.SparseTensor(rowptr=rp.cuda(), col=col.cuda(), sparse_sizes=(rp.numel() - 1, ns), is_sorted=True)
           for k, (rp, col, ns) in rec["csr"].items()}
    for rep in range(2):                                    # second pass runs on the cached graph structures
        out, gx, gp = _run(conv, x, adj, go, types)
        for t in types:
            tol = max(1e-5, 4.0 * rel_err(rec["f32"]["out"][t], rec["f64"]["out"][t]))
            assert rel_err(out[t], rec["f64"]["out"][t]) < tol, t
            tol = max(1e-5, 4.0 * rel_err(rec["f32"]["grad_x"][t], rec["f64"]["grad_x"][t]))
            assert rel_err(gx[t], rec["f64"]["grad_x"][t]) < tol, t
        for n, g in gp.items():
            tol = max(1e-5, 4.0 * rel_err(rec["f32"]["grad_p"][n], rec["f64"]["grad_p"][n]))
            assert rel_err(g, rec["f64"]["grad_p"][n]) < tol, n


@pytest.mark.gpu
def test_regconv_cuda_vs_oracle_larger_graph_with_hubs():
    """Rectangular relations with long rows / columns (> 256 nnz) and empty rows, fp64 restatement as the checker."""
    import egc_b200
    sizes = {"author": 1500, "field_of_study": 90, "institution": 40, "paper": 1100}
    types = list(sizes)
    torch.manual_seed(3)
    o = OH.REGConvOracle(64, 128, 8, 4).double()
    c = egc_b200.REGConv(64, 128, 8, 4)
    c.load_state_dict({k: v.float() for k, v in o.state_dict().items()})
    c = c.cuda()
    csr = OH.random_hetero_graph(sizes, 9000, 5)            # institution / field_of_study rows get > 256 nnz
    x = {t: torch.randn(n, 64) for t, n in sizes.items()}
    go = {t: torch.randn(n, 128) for t, n in sizes.items()}
    xo = {t: v.double().requires_grad_(True) for t, v in x.items()}
    oo, gxo, gpo = _run(o, xo, csr, {t: v.double() for t, v in go.items()}, types)
    xc = {t: v.cuda().requires_grad_(True) for t, v in x.items()}
    adj = {k: egc_b200.SparseTensor(rowptr=rp.cuda(), col=col.cuda(), sparse_sizes=(rp.numel() - 1, ns), is_sorted=True)
           for k, (rp, col, ns) in csr.items()}
    oc, gxc, gpc = _run(c, xc, adj, {t: v.cuda() for t, v in go.items()}, types)
    for t in types:
        assert rel_err(oc[t], oo[t]) < 1e-5 and rel_err(gxc[t], gxo[t]) < 1e-5, t
    for n in gpo:
        assert rel_err(gpc[n], gpo[n]) < 1e-5, n
