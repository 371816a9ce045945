"""Separate vs fused training-mode dropout of the EGC stack (EGC(..., fused_dropout=True)), fwd+bwd per step.

Workload and inputs are those of `bench.py --layers 3` (cfg3: the arxiv-shaped EGC-M graph and the 3-layer EGC stack, same
synthetic graph, seeds and locality as tools/bf16_bench.py), in training mode with dropout 0.5.  Arm A runs F.dropout after
every hidden layer; arm B runs it inside the aggregation kernel's epilogue.  Each arm's step is captured into one CUDA graph;
the timed window replays it `--steps` times between two CUDA events, and the arms alternate over `--rounds` rounds (medians
and the spread are reported).  Per arm also: the peak of torch.cuda.max_memory_allocated over one eager step, the launches of
libegc_b200 per step (egc_launch_count) and, in a separate eager pass, the per-kernel table of egc_profile_*.  The GPU name,
power limit and max SM clock are read in the same run.  egc_launch_count counts libegc_b200's kernels only, so a
torch.profiler pass of one eager step also counts every CUDA kernel of the step (torch's own, F.dropout's included).
Writes one JSON document to stdout (and to --out when given).

    python tools/dropout_bench.py --steps 50 --rounds 5 --out profiles/r04_fused_dropout.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload definitions, graph generator, kernel tracing)

DROPOUT = 0.5


def gpu_facts():
    facts = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        facts["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        facts["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return facts


def torch_kernel_counts(step):
    """{kernel name: launches} of every CUDA kernel one eager `step()` runs (torch.profiler, a pass of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    counts = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            counts[e.name] = counts.get(e.name, 0) + 1
    return counts


def make_model(w, fused, dev):
    import egc_b200
    torch.manual_seed(0)
    return egc_b200.EGC(w["f_out"], 3, DROPOUT, w["heads"], w["bases"], w["aggrs"], in_features=w["f_in"],
                        out_rounded=w["classes"][0], out_true=w["classes"][1], fused_dropout=fused).to(dev).train()


def main():
    import egc_b200
    from egc_b200 import _lib
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/dropout_bench.py measures on a GPU; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    w = bench.WORKLOADS["arxiv"]
    n, ei = bench.synth_graph("arxiv", seed=0, p_intra=0.8)
    graph_in = bench.device_graph_input(w, n, ei, dev)
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(n, w["f_in"], generator=gen).to(dev).requires_grad_(True)
    go = torch.randn(n, bench.out_width(w, 3), generator=gen).to(dev)
    result = {"what": "ms per fwd+bwd step of the cfg3 stack in training mode (dropout 0.5), CUDA-graph replay, CUDA events; "
                      "A = F.dropout after each hidden layer, B = dropout fused into the aggregation epilogue",
              "gpu": gpu_facts(), "workload": f"{w['desc']} as a 3-layer EGC stack", "nodes": n,
              "edges_directed": int(ei.size(1)), "steps_per_window": args.steps, "rounds": args.rounds, "arms": {}}
    arms = {}
    for key, fused in (("A_separate", False), ("B_fused", True)):
        model = make_model(w, fused, dev)
        params = list(model.parameters())

        def step(model=model, params=params):
            out = model(x, graph_in)
            return [out] + list(torch.autograd.grad(out, [x] + params, go))

        for _ in range(2):                                # warm every shape, build the cached graph
            step()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        l0 = _lib.launch_count()
        res = step()
        torch.cuda.synchronize()
        launches = _lib.launch_count() - l0
        peak = torch.cuda.max_memory_allocated(dev)
        del res
        _, kernels = bench.traced_kernels(step, 5)
        all_kernels = torch_kernel_counts(step)
        graphed = egc_b200.GraphedStep(step, warmup=args.warmup)
        arms[key] = {"graphed": graphed, "entry": {"peak_allocated_bytes_eager_step": peak,
                                                   "allocated_before_step_bytes": base,
                                                   "step_peak_above_resident_bytes": peak - base,
                                                   "libegc_launches_per_step": launches,
                                                   "cuda_kernels_per_step_all": sum(all_kernels.values()),
                                                   "cuda_kernel_counts": all_kernels, "kernels_eager": kernels}}
    times = {k: [] for k in arms}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):                          # alternate the arms: drift of the shared host hits both
        for k, arm in arms.items():
            for _ in range(args.warmup):
                arm["graphed"].replay()
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(args.steps):
                arm["graphed"].replay()
            ev1.record()
            torch.cuda.synchronize()
            times[k].append(ev0.elapsed_time(ev1) / args.steps)
    for k, arm in arms.items():
        ts = sorted(times[k])
        e = arm["entry"]
        e.update(ms_per_step_median=ts[len(ts) // 2], ms_per_step_min=ts[0], ms_per_step_max=ts[-1], ms_per_step_rounds=times[k])
        result["arms"][k] = e
    a, b = result["arms"]["A_separate"], result["arms"]["B_fused"]
    result["speedup_median"] = a["ms_per_step_median"] / b["ms_per_step_median"]
    result["peak_saving_bytes"] = a["peak_allocated_bytes_eager_step"] - b["peak_allocated_bytes_eager_step"]
    ca, cb = a["cuda_kernel_counts"], b["cuda_kernel_counts"]
    result["cuda_kernels_only_in_A_separate"] = {k: v - cb.get(k, 0) for k, v in ca.items() if v != cb.get(k, 0)}
    result["cuda_kernels_only_in_B_fused"] = {k: v - ca.get(k, 0) for k, v in cb.items() if v != ca.get(k, 0)}
    ka, kb = a["kernels_eager"].get("k_aggregate_fwd", {}), b["kernels_eager"].get("k_aggregate_fwd", {})
    result["k_aggregate_fwd_ms_per_step"] = {"A_separate": ka.get("ms_per_step"), "B_fused": kb.get("ms_per_step"),
                                             "note": "all three layers' forward aggregations; only the two hidden ones "
                                                     "apply dropout in B"}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
