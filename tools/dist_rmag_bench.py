"""REGConv row-partitioned over the GPUs of one node (`egc_b200.dist.PartitionedHeteroGraph`) against the single-GPU
REGConv, fwd+bwd per step, on the graph of `bench.py --workload rmag`.

Run one process per GPU:

    torchrun --nproc-per-node 8 tools/dist_rmag_bench.py --steps 20 --out profiles/r04_dist_rmag_8gpu.json

The graph is `bench.synth_hetero_csr(1.0, seed)` (ogbn-mag-shaped: 1.94 M nodes of four types, 42.2 M nnz over seven
relations) and the layer `bench.RMAG` (128 -> 128, 8 heads, 4 bases).  Every node type is split into nnz-balanced row
ranges; the endpoints of the generator are random permutations, so most referenced rows of every type are remote.
  * step time, partitioned: the whole step (forward, backward, exchanges, parameter all-reduce) captured once by
    `GraphedStep` (peer transport; the NCCL transport runs eagerly), `--steps` replays between two CUDA events, the max
    over ranks;
  * step time, single GPU: the single-GPU REGConv on the whole graph on each rank's GPU, eagerly as in bench.py (max over
    ranks);
  * rank 0's per-kernel table of a separate eager pass (egc_profile_*), `k_peer_push` on its own line;
  * halo rows per type and rank, and the bytes of one push;
  * parity: out and d_x rows of every type and every parameter gradient against the single-GPU layer (eager step and
    graph replay), max over ranks, bars of bench.py (1e-6 out, 1e-5 gradients);
  * the GPU name and power limit.
Rank 0 prints one JSON document (and writes it to --out)."""
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

import bench  # noqa: E402  (graph generator, layer shape, kernel tracing)
from bf16_bench import gpu_facts  # noqa: E402


def max_over_ranks(values, dev):
    t = torch.tensor(values, device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / steps


def main():
    import egc_b200
    from egc_b200.dist import GraphedStep, PartitionedHeteroGraph
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--transport", choices=["peer", "nccl"], default="peer")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dist_rmag_bench.py measures on GPUs; none is visible")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29531")
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    R = bench.RMAG
    sizes, csr = bench.synth_hetero_csr(1.0, args.seed)
    types = list(sizes)
    nnz = sum(int(v[1].numel()) for v in csr.values())
    adj = {k: egc_b200.SparseTensor(rowptr=rp.to(dev), col=col.to(dev), sparse_sizes=(rp.numel() - 1, ns), is_sorted=True)
           for k, (rp, col, ns) in csr.items()}
    del csr
    torch.manual_seed(0)
    conv = egc_b200.REGConv(R["f_in"], R["f_out"], R["heads"], R["bases"]).to(dev)
    params = list(conv.parameters())
    names = [n for n, _ in conv.named_parameters()]
    phg = PartitionedHeteroGraph.from_global(adj, sizes, rank, world, dev, transport=args.transport)
    rng = {t: phg.row_range(t) for t in types}
    gen = torch.Generator().manual_seed(args.seed + 1)
    x_full = {t: torch.randn(n, R["f_in"], generator=gen).to(dev) for t, n in sizes.items()}
    go_full = {t: torch.randn(n, R["f_out"], generator=gen).to(dev) for t, n in sizes.items()}
    x_loc = {t: x_full[t][b:e].clone().requires_grad_(True) for t, (b, e) in rng.items()}
    go_loc = {t: go_full[t][b:e].clone() for t, (b, e) in rng.items()}
    x_ref = {t: v.clone().requires_grad_(True) for t, v in x_full.items()}

    def step_single():
        out = conv(x_ref, adj)
        loss = sum((out[t] * go_full[t]).sum() for t in types)
        return (out,) + torch.autograd.grad(loss, [x_ref[t] for t in types] + params)

    def step_part():
        out = conv(x_loc, phg)
        loss = sum((out[t] * go_loc[t]).sum() for t in types)
        return (out,) + torch.autograd.grad(loss, [x_loc[t] for t in types] + params)

    def parity(res, ref):
        errs = {}
        for i, t in enumerate(types):
            b, e = rng[t]
            errs[f"out.{t}"] = bench.rel_err(res[0][t], ref[0][t][b:e])
            errs[f"d_x.{t}"] = bench.rel_err(res[1 + i], ref[1 + i][b:e])
        for n, a, r in zip(names, res[1 + len(types):], ref[1 + len(types):]):
            errs[f"d_{n}"] = bench.rel_err(a, r)
        errs = dict(zip(errs, max_over_ranks(list(errs.values()), dev)))
        ok = all(v < (1e-6 if k.startswith("out.") else 1e-5) for k, v in errs.items())
        return {"max_rel_err": errs, "green": ok}

    ref = step_single()
    par_eager = parity(step_part(), ref)
    phg.check()
    ms_single = timed(step_single, args.steps, args.warmup)
    if args.transport == "peer":
        import gc
        gc.collect()
        graphed = GraphedStep(step_part, warmup=2)
        ms_part = timed(graphed.replay, args.steps, args.warmup)
        par_replay = parity(graphed.replay(), ref)
    else:
        ms_part = timed(step_part, args.steps, args.warmup)
        par_replay = None
    phg.check()
    ms_part_max, ms_single_max = max_over_ranks([ms_part, ms_single], dev)
    _, kernels = bench.traced_kernels(step_part, max(3, min(args.steps, 10)))     # every rank steps; rank 0 reports
    phg.check()
    halo = {t: phg.part.tables[t].n_halo for t in types}
    own = {t: e - b for t, (b, e) in rng.items()}
    every = [None] * world
    dist.all_gather_object(every, {"own_rows": own, "halo_rows": halo})
    facts = gpu_facts()
    if rank == 0:
        push = kernels.get("k_peer_push", {"launches_per_step": 0, "ms_per_step": 0.0})
        row_bytes = 4 * (R["f_out"] // R["heads"]) * R["bases"]
        doc = {
            "what": "REGConv fwd+bwd per step, row-partitioned over GPUs vs the single-GPU layer",
            "workload": R["desc"], "graph": f"bench.synth_hetero_csr(1.0, {args.seed}): {sum(sizes.values())} nodes, "
                                             f"{nnz} nnz over 7 relations",
            "gpus": world, "transport": args.transport, "steps": args.steps, "warmup": args.warmup,
            "timing": "CUDA graph replay of the whole step (peer) / eager steps (nccl, single GPU), CUDA events, max "
                      "over ranks",
            "ms_per_step_partitioned": ms_part_max, "ms_per_step_single_gpu": ms_single_max,
            "speedup_vs_single_gpu": ms_single_max / ms_part_max if ms_part_max else None,
            "per_rank_rows": every,
            "max_halo_rows": max(sum(r["halo_rows"].values()) for r in every),
            "push_bytes_max_rank": max(sum(r["halo_rows"].values()) for r in every) * row_bytes,
            "k_peer_push_rank0": push,
            "kernels_rank0": dict(sorted(kernels.items(), key=lambda kv: -kv[1]["ms_per_step"])),
            "parity_eager": par_eager, "parity_replay": par_replay, **facts,
        }
        text = json.dumps(doc, indent=1)
        print(text)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")
    dist.barrier()
    phg.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
