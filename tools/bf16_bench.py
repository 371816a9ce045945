"""fp32 vs bf16 storage of the gathered tensors (EGConv(..., storage_dtype=torch.bfloat16)), fwd+bwd per step.

Workloads and inputs are those of bench.py (same synthetic graphs, seeds and locality): cfg2 = arxiv-shaped EGC-M, one
layer; cfg3 = the same as a 3-layer EGC stack; cfg4 = mag-shaped EGC-S, one layer.  Each (workload, storage) step is
captured into one CUDA graph; the timed window replays it `--steps` times between two CUDA events, and the two storage
types alternate over `--rounds` rounds (the spread is reported).  A separate eager pass records the per-kernel table of
egc_profile_*.  Writes one JSON document to stdout (and to --out when given).

    python tools/bf16_bench.py --steps 50 --rounds 5 --out profiles/r03_bf16_storage.json
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

CONFIGS = [("cfg2", "arxiv", 1), ("cfg3", "arxiv", 3), ("cfg4", "mag", 1)]


def make_model(w, layers, storage, seed=0):
    import egc_b200
    torch.manual_seed(seed)
    if layers == 1:
        return egc_b200.EGConv(w["f_in"], w["f_out"], aggrs=w["aggrs"], num_heads=w["heads"], num_bases=w["bases"],
                               cached=True, storage_dtype=storage)
    return egc_b200.EGC(w["f_out"], layers, 0.5, w["heads"], w["bases"], w["aggrs"], in_features=w["f_in"],
                        out_rounded=w["classes"][0], out_true=w["classes"][1], storage_dtype=storage)


def gpu_facts():
    facts = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        facts["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        facts["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return facts


def main():
    import egc_b200
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/bf16_bench.py measures on a GPU; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = {"what": "ms per fwd+bwd step, CUDA-graph replay, CUDA events; storage = dtype of the gathered tensors",
              "gpu": gpu_facts(), "steps_per_window": args.steps, "rounds": args.rounds, "configs": {}}
    for key, name, layers in CONFIGS:
        w = bench.WORKLOADS[name]
        n, ei = bench.synth_graph(name, seed=0, p_intra=0.8)
        graph_in = bench.device_graph_input(w, n, ei, dev)
        gen = torch.Generator().manual_seed(1)
        x = torch.randn(n, w["f_in"], generator=gen).to(dev).requires_grad_(True)
        go = torch.randn(n, bench.out_width(w, layers), generator=gen).to(dev)
        arms = {}
        for storage in (torch.float32, torch.bfloat16):
            model = make_model(w, layers, storage).to(dev)
            params = list(model.parameters())

            def step(model=model, params=params):
                out = model(x, graph_in)
                return [out] + list(torch.autograd.grad(out, [x] + params, go))

            torch.manual_seed(0)                         # the same dropout masks in both arms
            eager = [t.detach().clone() for t in step()]
            _, kernels = bench.traced_kernels(step, 5)
            graphed = egc_b200.GraphedStep(step, warmup=args.warmup)
            arms[str(storage).replace("torch.", "")] = {"graphed": graphed, "kernels": kernels, "eager": eager}
        times = {k: [] for k in arms}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):                     # alternate the arms: drift of the shared host hits both
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
        f32, b16 = arms["float32"]["eager"], arms["bfloat16"]["eager"]
        diffs = [float((b.double() - a.double()).abs().max() / a.double().abs().max().clamp(min=1e-30)) for a, b in zip(f32, b16)]
        entry = {"workload": w["desc"] if layers == 1 else f"{w['desc']} as a {layers}-layer EGC stack", "nodes": n,
                 "edges_directed": int(ei.size(1)), "layers": layers}
        for k in arms:
            ts = sorted(times[k])
            entry[k] = {"ms_per_step_median": ts[len(ts) // 2], "ms_per_step_min": ts[0], "ms_per_step_max": ts[-1],
                        "kernels_eager": arms[k]["kernels"]}
        entry["speedup_median"] = entry["float32"]["ms_per_step_median"] / entry["bfloat16"]["ms_per_step_median"]
        entry["bf16_vs_fp32_max_rel_diff"] = {"out": diffs[0], "d_x": diffs[1], "max_param_grad": max(diffs[2:])}
        result["configs"][key] = entry
        del arms
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
