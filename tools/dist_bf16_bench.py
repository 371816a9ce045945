"""fp32 vs bf16 storage (EGConv(..., storage_dtype=torch.bfloat16)) of row-partitioned layers, fwd+bwd per step.

Run one process per GPU:

    torchrun --nproc-per-node 8 tools/dist_bf16_bench.py --steps 50 --rounds 5 --out profiles/r03_dist_bf16_8gpu.json

Workloads and graphs are those of `bench.py --gpus N` (same synthetic graphs, seeds, locality and nnz-balanced row
ranges): cfg2 = arxiv-shaped EGC-M, one layer; cfg3 = the same as a 3-layer EGC stack; cfg4 = mag-shaped EGC-S, one layer.
Both arms run on one PartitionedGraph built with storage_dtype=torch.bfloat16 (fp32 layers run on it unchanged), transport
`--transport`.  Each arm's step is captured into one CUDA graph (peer transport); the timed window replays it `--steps` times
between two CUDA events, the arms alternate over `--rounds` rounds, and the time of a window is the max over ranks.  A
separate eager pass records rank 0's per-kernel table (egc_profile_*) with the exchange kernel `k_peer_push` listed on its
own.  Each arm is checked against the single-GPU layer of the same storage type on the same graph (dropout off).  Rank 0
writes one JSON document to stdout (and to --out)."""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import bench  # noqa: E402  (workload definitions, graph generator, kernel tracing)
from bf16_bench import CONFIGS, gpu_facts, make_model  # noqa: E402

ARMS = (("float32", torch.float32), ("bfloat16", torch.bfloat16))


def build_graph(w, n, ei, dev):
    import egc_b200
    sym = "symnorm" in w["aggrs"]
    if w["kind"] == "edge_index":
        return egc_b200.GraphStructure.from_edge_index(ei.to(dev), n, sym, True)
    rowptr, col = bench.to_adj_t(ei, n)
    return egc_b200.GraphStructure.from_csr(rowptr.to(dev), col.to(dev), None, n, sym, True)


def run(model, layers, x, graph):
    from egc_b200.dist import PartitionedGraph, partitioned_egconv
    if layers == 1 and isinstance(graph, PartitionedGraph):
        return partitioned_egconv(x, graph, model)
    return model(x, graph)                               # EGConv on a prepared graph, or the EGC stack on either kind


def max_over_ranks(values, dev):
    t = torch.tensor(values, device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def parity(model, layers, g, pg, x_full, go_full, dev):
    """out / d_x rows and parameter gradients of the partitioned step against the single-GPU layer of the same storage
    type on the same graph, dropout off, deterministic min / max routing (a lower bf16 layer rounds its streams to bf16, so
    run-to-run atomic noise in the gradient it receives could move a stored value by one ulp); max over ranks.  Bars of
    bench.py: 1e-6 (out) and 1e-5 (gradients) per layer."""
    was = model.training
    model.eval()
    convs = [m for m in model.modules() if hasattr(m, "deterministic")]
    for m in convs:
        m.deterministic = True
    params = list(model.parameters())
    b, e = pg.part.row_begin, pg.part.row_end
    xs = x_full.to(dev).requires_grad_(True)
    ref_out = run(model, layers, xs, g)
    ref = (ref_out,) + torch.autograd.grad(ref_out, [xs] + params, go_full.to(dev))
    xl = x_full[b:e].to(dev).requires_grad_(True)
    out = run(model, layers, xl, pg)
    got = (out,) + torch.autograd.grad(out, [xl] + params, go_full[b:e].to(dev))
    model.train(was)
    for m in convs:
        m.deterministic = False
    errs = [bench.rel_err(got[0], ref[0][b:e]), bench.rel_err(got[1], ref[1][b:e])]
    errs.append(max(bench.rel_err(a, r) for a, r in zip(got[2:], ref[2:])))
    o, dx, dp = max_over_ranks(errs, dev)
    tol_out, tol_grad = 1e-6 * layers, 1e-5 * layers
    return {"out": o, "d_x": dx, "param_grads": dp, "tol": {"out": tol_out, "grads": tol_grad},
            "ok": bool(o < tol_out and dx < tol_grad and dp < tol_grad)}


def main():
    import egc_b200
    from egc_b200.dist import GraphedStep, PartitionedGraph
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--transport", choices=["peer", "nccl"], default="peer")
    ap.add_argument("--configs", default="cfg2,cfg3,cfg4")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/dist_bf16_bench.py measures on GPUs; none is available")
    if "RANK" not in os.environ:
        raise SystemExit("run under torchrun --nproc-per-node N")
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    wanted = args.configs.split(",")
    result = {"what": "ms per fwd+bwd step of the row-partitioned layer, max over ranks of CUDA-event windows; storage = "
                      "dtype of the gathered and exchanged basis / stream rows",
              "gpu": gpu_facts(), "n_gpus": world, "transport": args.transport if world > 1 else "none (one rank)",
              "launch": "CUDA-graph replay" if args.transport == "peer" and world > 1 else "eager",
              "steps_per_window": args.steps, "rounds": args.rounds, "configs": {}}
    for key, name, layers in CONFIGS:
        if key not in wanted:
            continue
        w = bench.WORKLOADS[name]
        n, ei = bench.synth_graph(name, args.seed, p_intra=0.8, blocks=8)        # the graph of bench.py --gpus N
        g = build_graph(w, n, ei, dev)
        pg = PartitionedGraph.from_global(g, rank, world, dev, transport=args.transport, storage_dtype=torch.bfloat16)
        b, e = pg.part.row_begin, pg.part.row_end
        gen = torch.Generator().manual_seed(args.seed + 1)
        x_full, go_full = torch.randn(n, w["f_in"], generator=gen), torch.randn(n, bench.out_width(w, layers), generator=gen)
        x_loc, go_loc = x_full[b:e].to(dev).requires_grad_(True), go_full[b:e].to(dev)
        arms = {}
        for label, storage in ARMS:
            model = make_model(w, layers, storage, seed=args.seed).to(dev)
            params = list(model.parameters())
            check = parity(model, layers, g, pg, x_full, go_full, dev)

            def step(model=model, params=params):
                out = run(model, layers, x_loc, pg)
                return (out,) + torch.autograd.grad(out, [x_loc] + params, go_loc)

            _, kernels = bench.traced_kernels(step, 5)
            replay = GraphedStep(step, warmup=2).replay if pg.transport == "peer" else step
            arms[label] = {"replay": replay, "kernels": kernels, "parity": check}
        times = {k: [] for k in arms}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):                     # alternate the arms: drift of the shared host hits both
            for k, arm in arms.items():
                for _ in range(args.warmup):
                    arm["replay"]()
                torch.cuda.synchronize()
                dist.barrier()
                ev0.record()
                for _ in range(args.steps):
                    arm["replay"]()
                ev1.record()
                torch.cuda.synchronize()
                times[k].append(max_over_ranks([ev0.elapsed_time(ev1) / args.steps], dev)[0])
        pg.check()
        halo = max_over_ranks([pg.part.n_halo], dev)[0]
        entry = {"workload": w["desc"] if layers == 1 else f"{w['desc']} as a {layers}-layer EGC stack", "nodes": n,
                 "edges_directed": int(ei.size(1)), "layers": layers, "max_halo_rows_per_rank": int(halo),
                 "t_exchange": pg.uses_t_exchange(w["aggrs"])}
        for k, arm in arms.items():
            ts = sorted(times[k])
            kern = dict(arm["kernels"])
            push = kern.pop("k_peer_push", {"launches_per_step": 0, "ms_per_step": 0.0})
            entry[k] = {"ms_per_step_median": ts[len(ts) // 2], "ms_per_step_min": ts[0], "ms_per_step_max": ts[-1],
                        "k_peer_push_rank0": push, "kernels_rank0_eager": kern, "parity": arm["parity"]}
        entry["speedup_median"] = entry["float32"]["ms_per_step_median"] / entry["bfloat16"]["ms_per_step_median"]
        result["configs"][key] = entry
        del arms
        pg.close()
        torch.cuda.empty_cache()
    ok = all(c[k]["parity"]["ok"] for c in result["configs"].values() for k, _ in ARMS)
    if rank == 0:
        text = json.dumps(result, indent=1)
        print(text)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")
    dist.destroy_process_group()
    if not ok:
        sys.exit("tools/dist_bf16_bench.py: a partitioned step differs from its single-GPU layer beyond the bar")


if __name__ == "__main__":
    main()
