"""Row partition of a heterogeneous graph (`egc_b200.dist.HeteroPartitionPlan`) on CPU: one halo per source type, shared by
every relation that reads it, exchanged by `HaloExchange` over gloo.  The compute on each rank is the CPU restatement of
REGConv (oracle/hetero.py, oracle/restatement.py) on this rank's rows, so what is checked is the product's index and
communication plumbing: partitioned result == single-process `REGConvOracle`, in fp64."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from egc_b200.dist import HaloExchange, HeteroPartitionPlan
from oracle import hetero as OH
from oracle import restatement as R
from tests.util import rel_err

SIZES = {"author": 150, "field_of_study": 12, "institution": 6, "paper": 110}
F_IN, F_OUT, HEADS, BASES = 12, 24, 4, 3


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _graph(seed):
    """Duplicates, empty rows (the last two of every target type) and institution rows / columns with > 256 nnz."""
    return OH.random_hetero_graph(SIZES, 2000, seed)


def _plan(csr, world):
    return HeteroPartitionPlan({k: (rp, col) for k, (rp, col, _) in csr.items()}, SIZES, world)


def _worker(rank, world, port, seed, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        csr = _graph(seed)
        types = list(SIZES)
        torch.manual_seed(seed)
        layer = OH.REGConvOracle(F_IN, F_OUT, HEADS, BASES).double()
        gen = torch.Generator().manual_seed(seed + 100)
        x = {t: torch.randn(n, F_IN, generator=gen, dtype=torch.float64) for t, n in SIZES.items()}
        go = {t: torch.randn(n, F_OUT, generator=gen, dtype=torch.float64) for t, n in SIZES.items()}
        params = list(layer.parameters())
        # single process
        xs = {t: v.clone().requires_grad_(True) for t, v in x.items()}
        out_ref = layer(xs, csr)
        loss = sum((out_ref[t] * go[t]).sum() for t in types)
        grads_ref = torch.autograd.grad(loss, [xs[t] for t in types] + params)

        part = _plan(csr, world).local(rank)
        rng = {t: (part.tables[t].row_begin, part.tables[t].row_end) for t in types}
        ex = {t: HaloExchange(part.tables[t], "cpu") for t in types}
        x_loc = {t: x[t][b:e].clone().requires_grad_(True) for t, (b, e) in rng.items()}
        # forward: local projection, ONE halo exchange per source type, root term + relations over [own | halo]
        bases = {t: x_loc[t] @ layer.bases_weight for t in types}
        halo = {t: ex[t].forward(bases[t].detach()).requires_grad_(True) for t in types}
        for t in types:
            assert rel_err(halo[t], (x[t] @ layer.bases_weight.detach())[part.tables[t].halo_ids]) < 1e-13
        ext = {t: torch.cat([bases[t], halo[t]]) for t in types}
        out = {t: R.combine(layer.root_combs[t](x_loc[t]), bases[t].unsqueeze(1), None, HEADS) for t in types}
        for k, rel in part.relations.items():
            g = R.graph_from_csr(rel.rowptr, rel.col, None, ext[k[0]].size(0), False, False, True, dtype=torch.float64)
            agg, _ = R.aggregate(g, ext[k[0]], ["mean", "max"])
            out[k[2]] = out[k[2]] + R.combine(layer.rel_combs[f"{k[0]}_{k[1]}_{k[2]}"](x_loc[k[2]]), agg, None, HEADS)
        for t, (b, e) in rng.items():
            assert rel_err(out[t], out_ref[t][b:e]) < 1e-12, t
        # backward: local autograd gives partial sums for the halo rows of every type; they travel back to their owners
        loss = sum((out[t] * go[t][b:e]).sum() for t, (b, e) in rng.items())
        grads = torch.autograd.grad(loss, [x_loc[t] for t in types] + [halo[t] for t in types] + params,
                                    retain_graph=True, allow_unused=True)
        d_x = dict(zip(types, grads[:len(types)]))
        d_halo = dict(zip(types, grads[len(types):2 * len(types)]))
        d_par = list(grads[2 * len(types):])
        extra = {t: torch.zeros_like(bases[t]) for t in types}
        for t in types:
            if d_halo[t] is not None:
                ex[t].reverse(d_halo[t], extra[t])
        more = torch.autograd.grad([bases[t] for t in types], [x_loc[t] for t in types] + params,
                                   [extra[t] for t in types], allow_unused=True)
        for i, t in enumerate(types):
            b, e = rng[t]
            assert rel_err(d_x[t] + more[i], grads_ref[i][b:e]) < 1e-11, t
        for gp, ge, gr in zip(d_par, more[len(types):], grads_ref[len(types):]):
            tot = (gp if gp is not None else 0) + (ge if ge is not None else 0)
            tot = tot if torch.is_tensor(tot) else torch.zeros_like(gr)
            dist.all_reduce(tot)
            assert rel_err(tot, gr) < 1e-11
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_partitioned_hetero_layer_matches_single_process_gloo(world):
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), 4, ret), nprocs=world, join=True)
    assert dict(ret) == {r: "ok" for r in range(world)}


@pytest.mark.parametrize("world", [1, 2, 3, 6])
def test_hetero_partition_plan_invariants(world):
    csr = _graph(7)
    plan = _plan(csr, world)
    parts = [plan.local(r) for r in range(world)]
    nnz = {k: int(rp[-1]) for k, (rp, _, _) in csr.items()}
    for t, n in SIZES.items():
        b = plan.bounds[t]
        assert b[0] == 0 and b[-1] == n and all(b[r + 1] > b[r] for r in range(world)), (t, b)
    assert any(int((rp[1:] - rp[:-1]).max()) > 256 for rp, _, _ in csr.values())        # long rows
    assert any(int(torch.bincount(col).max()) > 256 for _, col, _ in csr.values())        # long columns
    for r, part in enumerate(parts):
        assert list(part.relations) == list(csr)
        for s, tab in part.tables.items():
            cb, ce = plan.bounds[s][r], plan.bounds[s][r + 1]
            assert (tab.row_begin, tab.row_end) == (cb, ce) and tab.rowptr is None
            assert sum(tab.recv_counts) == tab.n_halo and tab.recv_counts[r] == 0
            assert torch.equal(tab.halo_ids, torch.unique(tab.halo_ids))                # ascending, no repeats
            owner = torch.searchsorted(torch.tensor(plan.bounds[s]), tab.halo_ids, right=True) - 1
            off = 0
            for q, c in enumerate(tab.recv_counts):                                      # grouped by owner
                assert bool((owner[off:off + c] == q).all())
                off += c
            # the union halo is exactly the set of remote s ids that my target rows reference in every relation (s, r, t)
            want = []
            for k, (rp, col, _) in csr.items():
                if k[0] == s:
                    b, e = plan.bounds[k[2]][r], plan.bounds[k[2]][r + 1]
                    c = col[rp[b]:rp[e]]
                    want.append(c[(c < cb) | (c >= ce)])
            want = torch.unique(torch.cat(want)) if want else torch.zeros(0, dtype=torch.long)
            assert torch.equal(tab.halo_ids, want), (r, s)
            for q in range(world):                                                       # send / receive mirror
                qt = parts[q].tables[s]
                assert tab.send_rows[q].numel() == qt.recv_counts[r]
                qoff = sum(qt.recv_counts[:r])
                assert torch.equal(tab.send_rows[q] + cb, qt.halo_ids[qoff:qoff + qt.recv_counts[r]])
        for k, rel in part.relations.items():                                            # column remap
            rp, col, _ = csr[k]
            tab = part.tables[k[0]]
            b, e = plan.bounds[k[2]][r], plan.bounds[k[2]][r + 1]
            assert (rel.row_begin, rel.row_end) == (b, e) and rel.n_own_cols == tab.n_local
            ext = torch.cat([torch.arange(tab.row_begin, tab.row_end), tab.halo_ids])
            assert torch.equal(rel.rowptr, rp[b:e + 1] - rp[b])
            assert torch.equal(ext[rel.col], col[rp[b]:rp[e]])
            assert rel.halo_ids is tab.halo_ids and rel.send_rows is tab.send_rows
    assert sum(parts[r].relations[k].rowptr[-1] for r in range(world) for k in csr) == sum(nnz.values())


def test_type_with_fewer_rows_than_ranks_is_rejected():
    csr = _graph(1)
    with pytest.raises(ValueError, match="institution"):
        _plan(csr, 8)                                       # 6 institutions over 8 ranks
    with pytest.raises(ValueError):
        HeteroPartitionPlan({("a", "to", "b"): (torch.zeros(4, dtype=torch.long), torch.zeros(0, dtype=torch.long))},
                            {"a": 5, "b": 2}, 2)            # rowptr of 3 rows for a type of 2
