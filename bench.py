#!/usr/bin/env python
"""Headline benchmark: EGConv forward+backward edges/s on synthetic graphs of the shapes BASELINE.json names.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload arxiv|mag|zinc|cifar|rmag] [--layers L] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

Default (no flags, N = 1): BASELINE.json configs[1] - one EGC-M layer (symnorm+max+std, H4 B4, 128->128) forward +
backward over an ogbn-arxiv-shaped graph, structure cached as in the reference's full-graph training.  `--layers 3`
runs the reference's `EGC` stack (configs[2]); `--workload mag` configs[3].  N > 1 (torchrun): the same layer / stack
row-partitioned over N GPUs with the halo exchange over NVLink peer memory - strong scaling on the SAME graph (one
generator setting, p_intra = 0.8 over 8 id blocks, for every N) in the same launch mode (the whole step replayed from
one CUDA graph), max-over-ranks CUDA-event time, and a `parity_check` of the partitioned step against the single-GPU
layer before anything is timed (non-zero exit above the bar).  The default run also times the other full-graph
configurations of BASELINE.json and puts them under `other_configs` of the same line (3-layer arxiv stack, mag, and at
N = 1 the generator's uniform graph, the round-1 headline graph).  Other workloads: `zinc` / `cifar` (configs[0] / [4]:
128 collated small graphs through a 4-layer stack + readout, structure rebuilt every step), `rmag` (REGConv).

Rank 0 prints ONE JSON line.  `value` = aggregated nnz (after symmetrisation + self-loops) x layers per second with
inputs resident in HBM; `e2e` = the same through the public API with the step's features arriving from pinned host
memory and the loss read back; `roofline` = the dominant kernel's algorithmic bytes / its CUDA-event time against the
measured HBM peak (`traffic` = its DRAM bytes from the committed ncu capture of that workload, else null);
`step_roofline` = the step's unique bytes / step time; `cpu_baseline` = the oracle port of the reference path timed on
this box's host cores, whose results are also the checker of `parity_check` at N = 1 (GPU vs fp64 oracle, full graph);
`gpu_launches` = kernels of libegc_b200 launched in the timed region.  `--impl reference` times the CPU path alone on
the same workload.  `--dump-outputs DIR` (one GPU, full-graph workloads) writes what the last timed step returned as
DIR/<name>.npy (`dump_outputs`); the inputs are seeded (`--seed`), so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: nodes, raw directed edges, F_in, F_out, heads, bases, aggregators, input kind, zipf exponent
    "arxiv": dict(n=169_343, e0=1_166_243, f_in=128, f_out=128, heads=4, bases=4, classes=(40, 40),
                  aggrs=["symnorm", "max", "std"], kind="edge_index", zipf=0.75,
                  desc="EGC-M (symnorm+max+std, H4 B4) 128->128, ogbn-arxiv-shaped, 1 layer fwd+bwd"),
    "mag": dict(n=736_389, e0=5_416_271, f_in=128, f_out=128, heads=8, bases=4, classes=(352, 349),
                aggrs=["symnorm"], kind="adj_t", zipf=0.70,
                desc="EGC-S (symnorm, H8 B4) 128->128, ogbn-mag-shaped paper graph, 1 layer fwd+bwd"),
}
# mini-batch workloads (BASELINE configs 1 / 5): a step = collated batch of 128 small graphs through a 4-layer stack
MINIBATCH = {
    "zinc": dict(graphs=128, f_in=104, hidden=104, heads=8, bases=4, aggrs=["sum"], layers=4,
                 desc="EGC-S (sum, H8 B4, hidden 104, 4 layers + mean readout), 128 ZINC-shaped molecular graphs per step"),
    "cifar": dict(graphs=128, f_in=128, hidden=128, heads=4, bases=4, aggrs=["symnorm", "max", "std"], layers=4,
                  desc="EGC-M (symnorm+max+std, H4 B4, hidden 128, 4 layers + mean readout), 128 CIFAR10-superpixel-shaped graphs per step"),
}
L2_BYTES = 126e6


# ------------------------------------------------------------------------------------------------
# synthetic graphs (seeded; shapes from SURVEY.md section 8)
# ------------------------------------------------------------------------------------------------
def synth_graph(kind: str, seed: int = 0, p_intra: float = 0.0, blocks: int = 8):
    """(num_nodes, edge_index int64 [2, E]) - power-law in-degree (Zipf over a random node order),
    near-uniform out-degree, symmetrised + de-duplicated like `to_undirected` / `to_symmetric`
    (ref experiments/arxiv/configs.py:100, experiments/mag/configs.py:84-85).
    p_intra: probability that an edge stays inside its target's contiguous id block (locality knob
    for row-partitioned runs)."""
    w = WORKLOADS[kind]
    n, e0 = w["n"], w["e0"]
    rng = np.random.default_rng(seed)
    rank = rng.permutation(n)
    p = 1.0 / np.power(np.arange(1, n + 1, dtype=np.float64), w["zipf"])
    p /= p.sum()
    dst = rank[rng.choice(n, size=e0, p=p)]
    src = rng.integers(0, n, size=e0)
    if p_intra > 0:
        bs = (n + blocks - 1) // blocks
        local = rng.random(e0) < p_intra
        lo = (dst // bs) * bs
        src = np.where(local, np.minimum(lo + rng.integers(0, bs, size=e0), n - 1), src)
    key = np.unique(np.concatenate([src * n + dst, dst * n + src]))
    ei = np.stack([key // n, key % n])
    return n, torch.from_numpy(ei.astype(np.int64))


def to_adj_t(edge_index, n):
    """rows = targets, sorted by (target, source) (ref experiments/utils.py:93,107-109)."""
    perm = (edge_index[1] * n + edge_index[0]).argsort(stable=True)
    src, dst = edge_index[0][perm], edge_index[1][perm]
    rowptr = torch.zeros(n + 1, dtype=torch.long)
    rowptr[1:] = torch.cumsum(torch.bincount(dst, minlength=n), 0)
    return rowptr, src


# ------------------------------------------------------------------------------------------------
# algorithmic (unique) bytes - SURVEY.md section 8(d) / BASELINE.md section 2
# ------------------------------------------------------------------------------------------------
def stream_counts(aggrs):
    sym = int("symnorm" in aggrs)
    lin = int(any(a in ("sum", "mean", "var", "std") for a in aggrs))
    sq = int(any(a in ("var", "std") for a in aggrs))
    n_arg = sum(a in ("max", "min") for a in aggrs)
    return sym, lin, sq, n_arg


def algorithmic_bytes(n, e, f_in, heads, bases, dim, aggrs):
    a, bd, f_out = len(aggrs), bases * dim, heads * dim
    hab = heads * a * bases
    sym, lin, sq, n_arg = stream_counts(aggrs)
    L = sym + lin + sq
    bf = 4 * n * (f_in + 2 * bd + 2 * hab + f_out + n_arg * bd) + 4 * (e + n + 1) + 4 * n * sym
    bb = 4 * n * (f_out + hab + bd + n_arg * bd + 2 * hab + 2 * L * bd + 2 * bd + 2 * f_in) + 8 * (e + n + 1) + 4 * n * sym
    return bf, bb


def kernel_algorithmic_bytes(n, e, f_in, heads, bases, dim, aggrs):
    """Unique bytes each kernel of the step must move PER LAUNCH (DESIGN.md 'kernels'); same accounting as above."""
    a, bd, f_out = len(aggrs), bases * dim, heads * dim
    hab = heads * a * bases
    sym, lin, sq, n_arg = stream_counts(aggrs)
    L = sym + lin + sq
    s_saved = a + (1 if sq else 0)
    csr = 4 * (e + n + 1)
    return {
        # x (or [d_bases | d_lin]) in, [bases | weightings] (or d_x) out: both launches move the same bytes
        "k_project_tc": 4 * n * (f_in + bd + hab),
        "k_wgrad_tc": 4 * n * (f_in + bd + hab),
        # training forward: gather table + weightings in, out + saved aggregates + saved argmax out, CSR + symnorm weights
        "k_aggregate_fwd": 4 * n * (bd + hab + f_out + s_saved * bd + n_arg * bd) + csr + 4 * e * sym,
        # per target: grad_out, weightings, saved in; d_weightings, t-streams, routed min/max gradients out
        "k_combine_bwd": 4 * n * (f_out + hab + s_saved * bd + hab + L * bd + n_arg * bd),
        "k_route_minmax": 4 * n * n_arg * bd * 2 + (8 * n * bd if n_arg else 0),
        # per source (CSC): t-streams in, d_bases out (+ bases for the var/std term, + the routed partial), CSC + weights
        "k_scatter_bwd": 4 * n * (L * bd + bd + (bd if sq else 0) + (bd if n_arg else 0)) + csr + 4 * e * sym,
    }


def measured_traffic(workload, kernel):
    """DRAM bytes per launch (dram__bytes_read + dram__bytes_write) of `kernel` on `workload` from the committed
    `ncu --set full` capture of this round (profiles/r02_dram_traffic.json, written by tools/ncu_summary.py), or None
    when that workload / kernel was not captured."""
    path = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
    try:
        return json.load(open(path)).get(workload, {}).get(kernel)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
# clocks sampler (recipe in /opt/skills/guides/B200_PROFILING.md)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            t0 = time.time()                       # nvidia-smi needs a moment to start: a short timed region must not
            while not self.samples and time.time() - t0 < 3.0:      # end before the first sample exists
                time.sleep(0.05)
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None and len(self.samples) < 3:
            time.sleep(0.25)                       # at least a few samples taken right at the end of the timed region
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx.append(float(s[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# models: ONE layer (configs[1] / [3]) or the reference's `EGC` stack (configs[2]: experiments/mag/models.py:16-69)
# ------------------------------------------------------------------------------------------------
def layer_dims(w, layers):
    """[(f_in, f_out)] of the conv layers: a single 128 -> 128 layer, or IN -> hidden ... -> OUT_ROUNDED of the stack."""
    if layers == 1:
        return [(w["f_in"], w["f_out"])]
    return list(zip([w["f_in"]] + [w["f_out"]] * (layers - 1), [w["f_out"]] * (layers - 1) + [w["classes"][0]]))


def make_oracle_model(w, layers, seed=0, dtype=torch.float32, dropout=0.5):
    """CPU restatement with the parameters every arm of the benchmark shares (seeded)."""
    from oracle import restatement as R
    torch.manual_seed(seed)
    if layers == 1:
        m = R.EGConvOracle(w["f_in"], w["f_out"], aggrs=w["aggrs"], num_heads=w["heads"], num_bases=w["bases"], cached=True)
    else:
        m = R.EGCOracle(w["f_out"], layers, dropout, w["heads"], w["bases"], w["aggrs"], in_features=w["f_in"],
                        out_rounded=w["classes"][0], out_true=w["classes"][1])
    return m.to(dtype)


def make_gpu_model(w, layers, dev, state_dict=None, seed=0, dropout=0.5):
    import egc_b200
    torch.manual_seed(seed)
    if layers == 1:
        m = egc_b200.EGConv(w["f_in"], w["f_out"], aggrs=w["aggrs"], num_heads=w["heads"], num_bases=w["bases"], cached=True)
    else:
        m = egc_b200.EGC(w["f_out"], layers, dropout, w["heads"], w["bases"], w["aggrs"], in_features=w["f_in"],
                         out_rounded=w["classes"][0], out_true=w["classes"][1])
    if state_dict is not None:
        m.load_state_dict({k: v.float() for k, v in state_dict.items()})
    return m.to(dev)


def out_width(w, layers):
    return w["f_out"] if layers == 1 else w["classes"][1]


def stack_bytes(w, n, nnz, layers):
    """Unique bytes of one fwd+bwd step: the per-layer model summed over the conv layers (elementwise glue ignored)."""
    total = 0
    for f_in, f_out in layer_dims(w, layers):
        bf, bb = algorithmic_bytes(n, nnz, f_in, w["heads"], w["bases"], f_out // w["heads"], w["aggrs"])
        total += bf + bb
    return total


def workload_config(name, w, n, nnz, layers, p_intra, world):
    """The `config` object BOTH arms print (ours and --impl reference): only what defines the workload."""
    desc = w["desc"] if layers == 1 else w["desc"].replace("1 layer fwd+bwd", f"{layers}-layer EGC stack "
                                                           f"(conv-ReLU-dropout, log_softmax; ref mag/models.py) fwd+bwd")
    return {"workload": desc, "name": name, "layers": layers, "nodes": n, "raw_directed_edges": w["e0"], "nnz": nnz,
            "edges_counted": "aggregated nnz (symmetrised + self-loops) x layers", "input": w["kind"],
            "structure": "cached (graph prepared once, as the reference's cached=True)",
            "generator": {"seed": 0, "p_intra": p_intra, "blocks": 8}, "n_gpus": world,
            "l2": f"no flush: per-step working set {stack_bytes(w, n, nnz, layers) / 1e9:.2f} GB >> {L2_BYTES / 1e6:.0f} MB L2",
            "algorithmic_bytes_per_step": stack_bytes(w, n, nnz, layers)}


def default_locality(args):
    """p_intra of the generator: ONE graph for every GPU count (the scaling curve compares like with like)."""
    return args.locality if args.locality >= 0 else 0.8


# ------------------------------------------------------------------------------------------------
# CPU path of the reference (oracle port), used by --impl reference and by the cpu_baseline leg
# ------------------------------------------------------------------------------------------------
def cpu_reference_job(w, n, edge_index, layers=1, frac=1.0, seed=0, dtype=torch.float32, train=True):
    """One fwd+bwd of the reference path on the host (targets < frac*n when frac < 1).  Returns a dict with the step
    closure (-> out, {name: grad}), the model, the inputs and the aggregated nnz."""
    ei = edge_index
    if frac < 1.0:
        ei = ei[:, ei[1] < int(frac * n)]
    model = make_oracle_model(w, layers, seed, dtype)
    model.train(train)
    gen = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(n, w["f_in"], generator=gen).to(dtype).requires_grad_(True)
    go = torch.randn(n, out_width(w, layers), generator=gen).to(dtype)
    if w["kind"] == "edge_index":
        graph_in = ei
    else:
        rowptr, col = to_adj_t(ei, n)
        graph_in = (rowptr, col, None)
    first = model if layers == 1 else model.convs[0]
    g = first.prepare(x, graph_in)                       # cached structure, like the reference's full-graph runs
    if layers > 1:
        for conv in model.convs[1:]:
            conv._graph = g
    names = [k for k, _ in model.named_parameters()]

    def step():
        out = model(x, graph_in)
        grads = torch.autograd.grad(out, [x] + list(model.parameters()), go)
        return out.detach(), dict(zip(["x"] + names, grads))

    sample = (f"targets < {frac:.3f}*N of the {w['kind']} graph ({g.nnz} nnz incl. self-loops), full x"
              if frac < 1.0 else f"the whole {w['kind']} graph ({g.nnz} nnz incl. self-loops)")
    return {"step": step, "model": model, "x": x, "go": go, "nnz": g.nnz, "sample": sample, "graph_in": graph_in}


def time_cpu(step, steps, warmup):
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / max(steps, 1)


def run_reference_arm(args, name, w):
    """The reference's CPU path alone, on OUR arm's workload (same generator, same graph, same layer count)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    p_intra = default_locality(args)
    n, ei = synth_graph(name, args.seed, p_intra=p_intra, blocks=8)
    job = cpu_reference_job(w, n, ei, args.layers)
    nnz_full = job["nnz"]
    t_full = time_cpu(job["step"], 1, 0)                 # calibration = the first warm-up step
    budget = 300.0
    frac = 1.0
    if t_full * (args.steps + args.warmup) > budget:     # only then: a bounded sample of the same graph
        frac = max(budget / (t_full * (args.steps + args.warmup)), 1 / 64)
        job = cpu_reference_job(w, n, ei, args.layers, frac)
    t = time_cpu(job["step"], args.steps, max(args.warmup - (1 if frac == 1.0 else 0), 0))
    value = job["nnz"] * args.layers / t
    line = {
        "impl": "reference", "metric": "EGConv fwd+bwd edges/s", "value": value, "unit": "edges/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, w, n, nnz_full, args.layers, p_intra, args.gpus),
        "path": "oracle port of the reference's PyG path (pure-torch leaf ops), host CPU, all host threads",
        "cpu_baseline": {"value": value, "unit": "edges/s", "cores": cores, "kind": "port", "sample": job["sample"]},
        "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))


def device_graph_input(w, n, edge_index, dev):
    import egc_b200
    if w["kind"] == "edge_index":
        return edge_index.to(dev)
    rowptr, col = to_adj_t(edge_index, n)
    return egc_b200.SparseTensor(rowptr=rowptr.to(dev), col=col.to(dev), sparse_sizes=(n, n), is_sorted=True)


def cuda_timed(fn, steps, warmup, barrier=None, last=None):
    """CUDA-event time per call of `fn` after `warmup` untimed calls; (ms, kernels launched by libegc_b200).
    `last` (a list), when given, receives what the last timed call returned."""
    from egc_b200 import _lib
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if barrier:
        barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _lib.launch_count()
    ev0.record()
    if last is None:
        for _ in range(steps):
            fn()
    else:
        for _ in range(steps):
            last[:] = [fn()]
    ev1.record()
    torch.cuda.synchronize()
    if barrier:
        barrier()
    return ev0.elapsed_time(ev1) / steps, _lib.launch_count() - l0


DUMP_ROWS = 16_384          # rows kept of each per-node array by --dump-outputs (8 MB for a 128-wide fp32 array)


def dump_outputs(directory, named, n, seed=0):
    """Write the arrays a step returned (`named`: name -> tensor) as `directory`/<name>.npy in float32.  Per-node arrays
    (first dimension `n`: the output, d_x) keep the same DUMP_ROWS rows, drawn with a fixed seed and sorted, so that
    the files of two builds compare row for row and stay far below 64 MB; parameter gradients are written whole."""
    os.makedirs(directory, exist_ok=True)
    rows = None
    if n > DUMP_ROWS:
        rows = torch.from_numpy(np.sort(np.random.default_rng(seed).choice(n, DUMP_ROWS, replace=False)))
    for name, t in named.items():
        t = t.detach()
        if rows is not None and t.dim() > 0 and t.size(0) == n:
            t = t[rows.to(t.device)]
        np.save(os.path.join(directory, f"{name}.npy"), t.float().cpu().numpy())


def traced_kernels(fn, steps):
    """Per-kernel CUDA-event times of libegc_b200's launches over `steps` eager calls (separate pass)."""
    from egc_b200 import _lib
    _lib.profile_enable(True)
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    return prof, {k: {"launches_per_step": c / steps, "ms_per_step": t / steps} for k, (c, t) in prof.items()}


def dominant_roofline(name, prof, kernels, kbytes, peak, peak_src):
    cand = [k for k in kernels if kbytes.get(k)]
    if not cand:
        return None
    dom = max(cand, key=lambda k: kernels[k]["ms_per_step"])
    per_launch_ms = prof[dom][1] / prof[dom][0]
    achieved = kbytes[dom] / (per_launch_ms * 1e-3) / 1e9
    return {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": measured_traffic(name, dom), "peak_source": peak_src,
            "algorithmic_bytes_per_launch": kbytes[dom], "ms_per_launch": per_launch_ms}


class SingleGpuJob:
    """One workload on one GPU: model, resident inputs, the eager step (public API) and its CUDA-graph replay."""

    def __init__(self, name, w, layers, dev, p_intra, seed=0, state_dict=None, x=None, go=None):
        from egc_b200.dist import GraphedStep
        self.name, self.w, self.layers, self.dev = name, w, layers, dev
        self.n, self.ei = synth_graph(name, seed, p_intra=p_intra, blocks=8)
        self.model = make_gpu_model(w, layers, dev, state_dict)
        gen = torch.Generator().manual_seed(seed + 1)
        self.x_host = (x if x is not None else torch.randn(self.n, w["f_in"], generator=gen)).float().pin_memory()
        go = go if go is not None else torch.randn(self.n, out_width(w, layers), generator=gen)
        self.go = go.float().to(dev)
        self.graph_in = device_graph_input(w, self.n, self.ei, dev)
        self.x = self.x_host.to(dev).requires_grad_(True)
        self.params = list(self.model.parameters())
        self.step()                                      # builds + caches the graph structure (CSR, CSC, plans)
        first = self.model if layers == 1 else self.model.convs[0]
        self.graph = first._cached_edge_index if w["kind"] == "edge_index" else first._cached_adj_t
        self.nnz = self.graph.nnz
        self._graphed = None
        self._GraphedStep = GraphedStep

    def step(self):
        out = self.model(self.x, self.graph_in)
        return (out,) + torch.autograd.grad(out, [self.x] + self.params, self.go)

    def replay(self):
        if self._graphed is None:
            self._graphed = self._GraphedStep(self.step, warmup=2)
        return self._graphed.replay()

    def grads_named(self, res):
        names = ["x"] + [k for k, _ in self.model.named_parameters()]
        return res[0], dict(zip(names, res[1:]))


def parity_vs_cpu(job, cpu32, cpu64):
    """GPU step (eval mode: dropout off) against the fp64 CPU oracle on the same inputs and parameters.  Bar: 1e-5, or
    4x the error the reference's own fp32 arithmetic shows against fp64 on this input where that is larger (std)."""
    was = job.model.training
    job.model.eval()
    out, grads = job.grads_named(job.step())
    job.model.train(was)
    out32, g32 = cpu32
    out64, g64 = cpu64
    errs, tols = {"out": rel_err(out, out64)}, {"out": max(1e-5, 4 * rel_err(out32, out64))}
    for k in grads:
        errs[k], tols[k] = rel_err(grads[k], g64[k]), max(1e-5, 4 * rel_err(g32[k], g64[k]))
    ok = all(errs[k] < tols[k] for k in errs)
    return {"against": "CPU oracle in fp64, same inputs and parameters, full graph", "max_rel_err": max(errs.values()),
            "rel_err": errs, "tol": tols, "tol_rule": "max(1e-5, 4 x |oracle fp32 - oracle fp64|)", "ok": ok}


def run_single_gpu(args, name, w):
    from egc_b200 import _lib
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    p_intra = default_locality(args)
    layers = args.layers
    oracle = make_oracle_model(w, layers, args.seed)
    job = SingleGpuJob(name, w, layers, dev, p_intra, args.seed, oracle.state_dict())
    job.model.bwd_flags = args.bwd_flags
    n, nnz, x_host, go, model, params, graph_in = job.n, job.nnz, job.x_host, job.go, job.model, job.params, job.graph_in

    # end-to-end step: the step's features come from pinned host memory, the loss is read back.  The copy of
    # step k+1 is issued on a side stream while step k computes (double-buffered input prefetch, what a
    # training loop does); every timed step still contains exactly one H2D copy and one D2H read.
    copy_stream = torch.cuda.Stream(device=dev)
    x_bufs = [torch.empty((n, w["f_in"]), device=dev) for _ in range(2)]
    ev_ready = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    e2e_state = {"k": 0, "primed": False}

    def issue_copy(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[slot])            # the step that last used this buffer has finished
            x_bufs[slot].copy_(x_host, non_blocking=True)
            ev_ready[slot].record(copy_stream)

    def step_e2e():
        k = e2e_state["k"]
        slot = k & 1
        if not e2e_state["primed"]:
            for e in ev_free:
                e.record()
            issue_copy(slot)
            e2e_state["primed"] = True
        issue_copy(slot ^ 1)                                 # prefetch the next step's features
        torch.cuda.current_stream().wait_event(ev_ready[slot])
        xs = x_bufs[slot].detach().requires_grad_(True)
        out = model(xs, graph_in)
        loss = (out * go).sum()
        torch.autograd.grad(loss, [xs] + params)
        ev_free[slot].record()
        e2e_state["k"] = k + 1
        return float(loss.item())

    l0 = _lib.launch_count()
    job.step()
    launches_per_step = _lib.launch_count() - l0
    last = [] if args.dump_outputs else None
    with ClockSampler(dev.index or 0) as clocks:
        if args.no_graph:
            ms, _ = cuda_timed(job.step, args.steps, args.warmup, last=last)
            ms_eager = ms
        else:
            ms, _ = cuda_timed(job.replay, args.steps, args.warmup, last=last)
        if args.dump_outputs:
            out, grads = job.grads_named(last[0])
            dump_outputs(args.dump_outputs, {"out": out, **{f"grad_{k}": g for k, g in grads.items()}}, n, args.seed)
        if not args.no_graph:
            ms_eager, _ = cuda_timed(job.step, args.steps, args.warmup)
        ms_e2e, _ = cuda_timed(step_e2e, max(3, min(args.steps, 10)), 2)
    prof, kernels = traced_kernels(job.step, args.steps)

    peak, peak_src = load_peaks()
    total_bytes = stack_bytes(w, n, nnz, layers)
    roofline = None
    if layers == 1:
        kbytes = kernel_algorithmic_bytes(n, nnz, w["f_in"], w["heads"], w["bases"], w["f_out"] // w["heads"], w["aggrs"])
        roofline = dominant_roofline(name, prof, kernels, kbytes, peak, peak_src)
    step_gbs = total_bytes / (ms * 1e-3) / 1e9
    edges = nnz * layers

    cpu = parity = None
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        frac = 1.0 if (name == "arxiv" and layers == 1) else (0.5 if name == "arxiv" else 0.25)
        cjob = cpu_reference_job(w, n, job.ei, layers, frac, args.seed)
        t_cpu = time_cpu(cjob["step"], 2, 1)
        cpu = {"value": cjob["nnz"] * layers / t_cpu, "unit": "edges/s", "cores": cores, "kind": "port",
               "sample": f"{cjob['sample']}; 1 warm-up + 2 timed fwd+bwd steps, {t_cpu:.2f} s/step"}
        if frac == 1.0:
            # the CPU leg's results are the checker: same parameters (the GPU model loaded the oracle's state_dict),
            # same x / grad_out (same generator seed), fp32 run = the timed one, one extra fp64 run = the truth
            cjob["model"].eval()
            cpu32 = cjob["step"]()
            c64 = cpu_reference_job(w, n, job.ei, layers, 1.0, args.seed, torch.float64, train=False)
            parity = parity_vs_cpu(job, cpu32, c64["step"]())

    line = {
        "metric": "EGConv fwd+bwd edges/s", "value": edges / (ms * 1e-3), "unit": "edges/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, w, n, nnz, layers, p_intra, 1),
        "launch_mode": "eager launches" if args.no_graph else "whole step replayed from one CUDA graph (as the N > 1 runs)",
        "eager_ms_per_step": ms_eager,
        "clocks": clocks.summary(),
        "e2e": {"value": edges / (ms_e2e * 1e-3), "unit": "edges/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": 4,
                "input_pipeline": "public API, eager; double-buffered: the H2D copy of step k+1 overlaps the compute of step k"},
        "gpu_launches": launches_per_step * args.steps,
        "step_roofline": {"achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak},
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity_check": parity,
        "kernels": kernels,
    }
    if not args.no_extras and name == "arxiv" and layers == 1:
        del job
        torch.cuda.empty_cache()
        line["other_configs"] = single_gpu_extras(args, dev, p_intra, peak)
    print(json.dumps(line))
    if parity is not None and not parity["ok"]:
        sys.exit("bench.py: GPU results differ from the CPU oracle beyond the bar - see parity_check")


def single_gpu_extras(args, dev, p_intra, peak):
    """The other full-graph configurations BASELINE.json names, timed the same way (graph replay, resident inputs), so
    that the 1-GPU record holds the base of every scaling curve: configs[2] (3-layer arxiv stack), configs[3] (mag),
    plus the default layer on the generator's uniform graph (p_intra = 0, the round-1 headline graph)."""
    out = {}
    for key, name, layers, pi in (("arxiv_3layer", "arxiv", 3, p_intra), ("mag", "mag", 1, p_intra),
                                  ("arxiv_uniform_graph", "arxiv", 1, 0.0)):
        try:
            w = WORKLOADS[name]
            job = SingleGpuJob(name, w, layers, dev, pi, args.seed)
            ms, _ = cuda_timed(job.replay, max(args.steps // 2, 5), 3)
            total = stack_bytes(w, job.n, job.nnz, layers)
            out[key] = {"config": workload_config(name, w, job.n, job.nnz, layers, pi, 1), "ms_per_step": ms,
                        "value": job.nnz * layers / (ms * 1e-3), "unit": "edges/s",
                        "step_roofline_frac": total / (ms * 1e-3) / 1e9 / peak}
            del job
            torch.cuda.empty_cache()
        except Exception as exc:                          # an extra must never cost the headline line
            out[key] = {"error": repr(exc)[:300]}
    return out


def local_roofline(kernels, n_rows, nnz, w, peak, peak_src):
    """`roofline` object of a partitioned run from rank 0's traced kernels: the dominant kernel's algorithmic bytes for
    the LOCAL rows / nnz of one step over its time per step (all its launches of the step), against one GPU's peak."""
    try:
        dim = w["f_out"] // w["heads"]
        kb = kernel_algorithmic_bytes(int(n_rows), int(nnz), w["f_in"], w["heads"], w["bases"], dim, w["aggrs"])
        cand = [k for k in kernels if kb.get(k) and kernels[k]["ms_per_step"] > 0]
        if not cand:
            return None
        dom = max(cand, key=lambda k: kernels[k]["ms_per_step"])
        per_step = kb[dom] * (2 if dom == "k_project_tc" else 1)        # forward and d_x launches move the same bytes
        achieved = per_step / (kernels[dom]["ms_per_step"] * 1e-3) / 1e9
        return {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_step": per_step,
                "ms_per_step": kernels[dom]["ms_per_step"], "launches_per_step": kernels[dom]["launches_per_step"],
                "scope": "rank 0, its local rows and nnz (halo rows not counted), eager traced pass"}
    except Exception:                                                   # never let the extra key break the bench line
        return None


class PartitionedJob:
    """One workload row-partitioned over the ranks of the process group, next to the single-GPU model on the same
    (full) graph - every rank builds the full graph anyway - which is the parity reference and the same-graph base of
    the speed-up."""

    def __init__(self, args, name, w, layers, dev, p_intra):
        import egc_b200
        from egc_b200.dist import PartitionedGraph
        import torch.distributed as dist
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.name, self.w, self.layers, self.dev = name, w, layers, dev
        self.n, ei = synth_graph(name, args.seed, p_intra=p_intra, blocks=8)
        n = self.n
        self.model = make_gpu_model(w, layers, dev, seed=args.seed)       # identical replicated parameters on every rank
        sym = "symnorm" in w["aggrs"]
        if w["kind"] == "edge_index":
            self.g = egc_b200.GraphStructure.from_edge_index(ei.to(dev), n, sym, True)
        else:
            rowptr, col = to_adj_t(ei, n)
            self.g = egc_b200.GraphStructure.from_csr(rowptr.to(dev), col.to(dev), None, n, sym, True)
        self.nnz = self.g.nnz
        self.pg = PartitionedGraph.from_global(self.g, self.rank, self.world, dev, transport=args.transport)
        b, e = self.pg.part.row_begin, self.pg.part.row_end
        gen = torch.Generator().manual_seed(args.seed + 1)
        self.x_full = torch.randn(n, w["f_in"], generator=gen)
        self.go_full = torch.randn(n, out_width(w, layers), generator=gen)
        self.x_loc = self.x_full[b:e].to(dev).requires_grad_(True)
        self.go_loc = self.go_full[b:e].to(dev)
        self.x_host = self.x_loc.detach().cpu().pin_memory()
        self.params = list(self.model.parameters())
        self.b, self.e = b, e

    def run(self, x, graph):
        from egc_b200.dist import PartitionedGraph, partitioned_egconv
        if self.layers == 1 and isinstance(graph, PartitionedGraph):
            return partitioned_egconv(x, graph, self.model)
        return self.model(x, graph)                      # EGConv on a prepared graph, or the EGC stack on either kind

    def step(self):
        out = self.run(self.x_loc, self.pg)
        return (out,) + torch.autograd.grad(out, [self.x_loc] + self.params, self.go_loc)

    def single_gpu_step(self, xs, gos):
        out = self.run(xs, self.g)
        return (out,) + torch.autograd.grad(out, [xs] + self.params, gos)

    def parity_check(self):
        """Rank-local out / d_x rows and the (already summed) parameter gradients of the partitioned step against the
        single-GPU layer on the same graph, dropout off.  Max over ranks."""
        import torch.distributed as dist
        was = self.model.training
        self.model.eval()
        xs = self.x_full.to(self.dev).requires_grad_(True)
        ref = self.single_gpu_step(xs, self.go_full.to(self.dev))
        got = self.step()
        self.model.train(was)
        b, e = self.b, self.e
        errs = [rel_err(got[0], ref[0][b:e]), rel_err(got[1], ref[1][b:e])] + [rel_err(a, r) for a, r in zip(got[2:], ref[2:])]
        t = torch.tensor([errs[0], errs[1], max(errs[2:])], device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tol_out, tol_grad = 1e-6 * self.layers, 1e-5 * self.layers
        o, dx, dp = (float(v) for v in t)
        return {"against": "the single-GPU layer on the same graph, parameters and inputs (max over ranks)",
                "out": o, "d_x": dx, "param_grads": dp, "max_rel_err": max(o, dx, dp), "tol": {"out": tol_out, "grads": tol_grad},
                "ok": bool(o < tol_out and dx < tol_grad and dp < tol_grad)}

    def close(self):
        self.pg.close()


def time_partitioned(args, job, steps, warmup, with_e2e=True):
    """(ms per step max over ranks, e2e ms, launches per step of this rank, single-GPU same-graph ms)."""
    import torch.distributed as dist
    from egc_b200 import _lib
    from egc_b200.dist import GraphedStep
    dev = job.dev
    use_graph = args.transport == "peer" and not args.no_graph
    l0 = _lib.launch_count()
    job.step()
    launches_per_step = _lib.launch_count() - l0
    step = GraphedStep(job.step, warmup=2).replay if use_graph else job.step

    # end-to-end step: this rank's feature rows arrive from pinned host memory every step, the loss is read back.  As on
    # one GPU the copy is double-buffered: the H2D transfer of step k+1 runs on a side stream into a staging buffer while
    # step k computes; the step itself starts with a device-to-device copy into the (graph-captured) input buffer.
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [torch.empty_like(job.x_loc.detach()) for _ in range(2)]
    ev_ready = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    e2e_state = {"k": 0, "primed": False}

    def issue_copy(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[slot])
            stage[slot].copy_(job.x_host, non_blocking=True)
            ev_ready[slot].record(copy_stream)

    def step_e2e():
        k = e2e_state["k"]
        slot = k & 1
        if not e2e_state["primed"]:
            for e in ev_free:
                e.record()
            issue_copy(slot)
            e2e_state["primed"] = True
        issue_copy(slot ^ 1)                                 # prefetch the next step's rows
        torch.cuda.current_stream().wait_event(ev_ready[slot])
        with torch.no_grad():
            job.x_loc.copy_(stage[slot])
        ev_free[slot].record()
        res = step()
        e2e_state["k"] = k + 1
        return float((res[0].detach() * job.go_loc).sum().item())

    def reduce_max(ms):
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ms = reduce_max(cuda_timed(step, steps, warmup, dist.barrier)[0])
    ms_e2e = reduce_max(cuda_timed(step_e2e, max(3, min(steps, 10)), 2, dist.barrier)[0]) if with_e2e else None
    job.pg.check()
    # the single-GPU layer on the SAME graph, same launch mode, timed on every rank's own GPU at the same time
    xs, gos = job.x_full.to(dev).requires_grad_(True), job.go_full.to(dev)
    single = GraphedStep(lambda: job.single_gpu_step(xs, gos), warmup=2).replay if not args.no_graph else (lambda: job.single_gpu_step(xs, gos))
    ms_single = reduce_max(cuda_timed(single, max(steps // 2, 5), 3, dist.barrier)[0])
    return ms, ms_e2e, launches_per_step, ms_single, use_graph


def run_multi_gpu(args, name, w):
    """Row-partitioned layer / stack over N ranks (one per GPU, NCCL bootstrap): strong scaling on the same graph."""
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    p_intra = default_locality(args)
    layers = args.layers
    job = PartitionedJob(args, name, w, layers, dev, p_intra)
    n, nnz = job.n, job.nnz
    parity = job.parity_check()
    with ClockSampler(dev.index or 0) as clocks:
        ms, ms_e2e, launches_per_step, ms_single, use_graph = time_partitioned(args, job, args.steps, args.warmup)
    # per-kernel CUDA-event times of rank 0 (eager launches, separate pass; waits include the time spent on peers)
    prof, kernels = traced_kernels(job.step, args.steps)
    pg = job.pg
    stats = torch.tensor([pg.part.n_halo, pg.part.n_local, pg.part.interior_rows.numel(), launches_per_step * args.steps],
                         device=dev, dtype=torch.float64)
    gathered = [torch.zeros_like(stats) for _ in range(world)]
    dist.all_gather(gathered, stats)
    local_rows, local_nnz = int(pg.part.n_local), int(pg.graph.nnz)
    job.close()
    del job
    torch.cuda.empty_cache()
    others = None
    if not args.no_extras and name == "arxiv" and layers == 1:
        others = multi_gpu_extras(args, dev, p_intra)
    if rank == 0:
        total_bytes = stack_bytes(w, n, nnz, layers)
        peak, peak_src = load_peaks()
        halo_rows = sum(int(t[0]) for t in gathered)
        bd = w["bases"] * (w["f_out"] // w["heads"])
        edges = nnz * layers
        line = {
            "metric": "EGConv fwd+bwd edges/s", "value": edges / (ms * 1e-3), "unit": "edges/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(name, w, n, nnz, layers, p_intra, world),
            "partition": {"scheme": f"contiguous target-row ranges over {world} GPUs (nnz-balanced), halo exchange of basis rows",
                          "halo_rows_total": halo_rows, "interior_rows_total": sum(int(t[2]) for t in gathered),
                          "nvlink_bytes_per_step": 2 * halo_rows * bd * 4 * layers,
                          "transport": ("NVLink peer-memory kernels (posted stores + epoch flags), whole step replayed "
                                        "from one CUDA graph" if use_graph else
                                        ("NVLink peer-memory kernels, eager launches" if args.transport == "peer" else
                                         "NCCL batch_isend_irecv + all_reduce, eager launches"))},
            "parity_check": parity,
            "single_gpu_same_graph": {"ms_per_step": ms_single, "speedup": ms_single / ms,
                                      "note": "the single-GPU layer on the same graph, same launch mode, same box"},
            "clocks": clocks.summary(),
            "e2e": {"value": edges / (ms_e2e * 1e-3), "unit": "edges/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": n * w["f_in"] * 4, "d2h_bytes_per_step": 4 * world,
                    "input_pipeline": "every rank copies its own rows from pinned host memory; double-buffered (the H2D copy "
                                      "of step k+1 overlaps the compute of step k), loss read back on every rank"},
            "gpu_launches": sum(int(t[3]) for t in gathered),
            "step_roofline": {"achieved": total_bytes / (ms * 1e-3) / 1e9, "peak": peak * world, "unit": "GB/s",
                              "frac": total_bytes / (ms * 1e-3) / 1e9 / (peak * world), "peak_source": peak_src + f" x {world}"},
            "roofline": local_roofline(kernels, local_rows, local_nnz, w, peak, peak_src) if layers == 1 else None,
            "cpu_baseline": None, "kernels_rank0": kernels,
        }
        if others is not None:
            line["other_configs"] = others
        print(json.dumps(line))
    dist.destroy_process_group()
    if not parity["ok"]:
        sys.exit(f"bench.py: the partitioned step differs from the single-GPU layer beyond the bar: {parity}")


def multi_gpu_extras(args, dev, p_intra):
    """configs[2] (3-layer arxiv stack) and configs[3] (mag) partitioned over the same ranks: time, same-graph
    single-GPU time and parity, so the scaling record covers the configurations BASELINE.json names."""
    import torch.distributed as dist
    out = {}
    for key, name, layers in (("arxiv_3layer", "arxiv", 3), ("mag", "mag", 1)):
        job = None
        try:
            w = WORKLOADS[name]
            job = PartitionedJob(args, name, w, layers, dev, p_intra)
            parity = job.parity_check()
            ms, _, _, ms_single, _ = time_partitioned(args, job, max(args.steps // 2, 5), 3, with_e2e=False)
            out[key] = {"config": workload_config(name, w, job.n, job.nnz, layers, p_intra, dist.get_world_size()),
                        "ms_per_step": ms, "value": job.nnz * layers / (ms * 1e-3), "unit": "edges/s",
                        "single_gpu_same_graph": {"ms_per_step": ms_single, "speedup": ms_single / ms},
                        "parity_check": parity}
        except Exception as exc:
            out[key] = {"error": repr(exc)[:300]}
        finally:
            if job is not None:
                try:
                    job.close()
                except Exception:
                    pass
            del job
            torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
# mini-batch workloads: synthetic graph lists (shapes from SURVEY.md section 8d) and the runner
# ------------------------------------------------------------------------------------------------
def synth_small_graphs(kind: str, num_graphs: int, seed: int, f_in: int):
    """[(x [n, f_in] fp32, edge_index [2, e] int64 graph-local, n)].  zinc: ~N(23.2, 4.5) nodes in [9, 37], random tree
    + ring closures, both directions; cifar: U{85..150} nodes, 8 nearest neighbours in 2-D as in-edges of every node."""
    gen = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(num_graphs):
        if kind == "zinc":
            n = int(torch.clamp(torch.round(torch.randn((), generator=gen) * 4.5 + 23.2), 9, 37))
            parent = (torch.rand(n - 1, generator=gen) * torch.arange(1, n)).long()
            child = torch.arange(1, n)
            n_ring = max(1, int(round(0.075 * n)))
            a = torch.randint(0, n, (n_ring,), generator=gen)
            b = (a + torch.randint(2, max(n - 1, 3), (n_ring,), generator=gen)) % n
            keep = a != b
            src, dst = torch.cat([parent, a[keep]]), torch.cat([child, b[keep]])
            ei = torch.stack([torch.cat([src, dst]), torch.cat([dst, src])])
        else:
            n = int(torch.randint(85, 151, (), generator=gen))
            pos = torch.rand((n, 2), generator=gen)
            d = torch.cdist(pos, pos)
            d.fill_diagonal_(float("inf"))
            nbr = d.topk(8, largest=False).indices
            ei = torch.stack([nbr.reshape(-1), torch.arange(n).repeat_interleave(8)])
        out.append((torch.randn((n, f_in), generator=gen), ei, n))
    return out


class StaticBatchStep:
    """Fixed-shape mini-batch step: every batch padded on the host (the DataLoader's collate step) to the same node /
    edge counts, so the WHOLE step - collation, CSR + CSC build, the layer stack forward + backward, readout, loss -
    is captured once and replayed from ONE CUDA graph per batch.  `flat_scale` (data-parallel runs): the parameter
    gradients are also packed, scaled, into one flat buffer inside the graph (`self.flat`) for a single all-reduce."""

    def __init__(self, model, packed, n_graphs, f_in, sym, dev, flat_scale=None):
        import egc_b200
        from egc_b200.dist import GraphedStep
        self.n_graphs = n_graphs
        e_cap = max(int(pk[1].size(1)) for pk in packed) + 1
        q_max = e_cap - min(int(pk[1].size(1)) for pk in packed)
        n_cap = max(int(pk[0].size(0)) for pk in packed) + max(64, (q_max + 63) // 64)
        padded = [egc_b200.pad_batch(pk[0], pk[1], pk[2], n_cap, e_cap) for pk in packed]
        shapes = {p_[3] for p_ in padded}
        if len(shapes) != 1:
            raise ValueError("batches with self-loops in their edge lists do not share one prepared-graph size")
        nnz_cap = shapes.pop()
        self.n_cap, self.e_cap = n_cap, e_cap
        self.pinned = [tuple(t.pin_memory() for t in p_[:3]) for p_ in padded]
        self.resident = [tuple(t.to(dev) for t in p_) for p_ in self.pinned]
        self.xs = torch.zeros((n_cap, f_in), device=dev, requires_grad=True)
        self.els = torch.zeros((2, e_cap), dtype=torch.int64, device=dev)
        self.pts = torch.zeros((2, n_graphs + 2), dtype=torch.int32, device=dev)
        params = list(model.parameters())
        self.flat = torch.zeros(sum(p_.numel() for p_ in params), device=dev) if flat_scale is not None else None
        keep = {}

        def static_step():
            edge_index, _ = egc_b200.collate_arrays(self.els, self.pts[1], self.pts[0], num_nodes=n_cap, validate=False)
            g = egc_b200.GraphStructure.from_edge_index(edge_index, n_cap, sym, True, expect={"nnz": nnz_cap})
            keep["g"] = g
            h = self.xs
            for layer in model:
                h = torch.relu(layer(h, g))
            loss = egc_b200.global_mean_pool(h, self.pts[0, :n_graphs + 1]).pow(2).sum(1).mean()
            grads = torch.autograd.grad(loss, [self.xs] + params)
            if self.flat is not None:
                torch.cat([gr.reshape(-1) for gr in grads[1:]], out=self.flat)
                self.flat.mul_(flat_scale)
            return (loss,) + grads

        self.load(0)
        self.graphed = GraphedStep(static_step, warmup=2)
        self.graph = keep["g"]                            # its counters are static buffers of the captured build

    def load(self, k, pinned=False):
        src = (self.pinned if pinned else self.resident)[k % len(self.resident)]
        with torch.no_grad():
            self.xs.copy_(src[0], non_blocking=True)
            self.els.copy_(src[1], non_blocking=True)
            self.pts.copy_(src[2], non_blocking=True)

    def replay(self):
        return self.graphed.replay()

    def verify(self):
        self.graph.verify()


def run_minibatch(args, m):
    """One step = one collated batch of small graphs through `layers` x (EGConv -> ReLU), mean readout, squared-norm
    loss, backward.  The graph structure is NOT cached (every batch is new, as in the reference's mini-batch training):
    the CSR / CSC build is inside the timed step, once per batch and shared by the layers."""
    import egc_b200
    from egc_b200 import _lib
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    dims = [m["f_in"]] + [m["hidden"]] * m["layers"]
    model = torch.nn.ModuleList([egc_b200.EGConv(dims[i], dims[i + 1], aggrs=m["aggrs"], num_heads=m["heads"],
                                                 num_bases=m["bases"]) for i in range(m["layers"])]).to(dev)
    params = list(model.parameters())
    sym = "symnorm" in m["aggrs"]
    n_batches = 8
    host = [synth_small_graphs(args.workload, m["graphs"], args.seed * 100 + b, m["f_in"]) for b in range(n_batches)]
    # pinned, pre-concatenated host arrays of every batch (what a DataLoader worker hands over)
    packed = []
    for graphs in host:
        counts = torch.tensor([[g[2], g[1].size(1)] for g in graphs])
        ptrs = torch.zeros((2, len(graphs) + 1), dtype=torch.int32)
        ptrs[:, 1:] = counts.cumsum(0).t().to(torch.int32)
        packed.append((torch.cat([g[0] for g in graphs]).pin_memory(), torch.cat([g[1] for g in graphs], 1).pin_memory(),
                       ptrs.pin_memory(), len(graphs)))
    resident = [tuple(t.to(dev) if torch.is_tensor(t) else t for t in pk) for pk in packed]
    state = {"k": 0}

    def run(x, edge_local, ptrs, n_graphs, read_loss):
        n = int(x.size(0))
        edge_index, batch = egc_b200.collate_arrays(edge_local, ptrs[1], ptrs[0], num_nodes=n, validate=False)
        g = egc_b200.GraphStructure.from_edge_index(edge_index, n, sym, True)
        h = x.requires_grad_(True)
        for layer in model:
            h = torch.relu(layer(h, g))
        loss = egc_b200.global_mean_pool(h, ptrs[0]).pow(2).sum(1).mean()
        torch.autograd.grad(loss, [x] + params)
        return (float(loss.item()) if read_loss else loss), g.nnz

    def step():
        k = state["k"]; state["k"] = k + 1
        x, el, ptrs, ng = resident[k % n_batches]
        return run(x.detach(), el, ptrs, ng, False)

    def step_e2e():
        k = state["k"]; state["k"] = k + 1
        x, el, ptrs, ng = packed[k % n_batches]
        return run(x.to(dev, non_blocking=True), el.to(dev, non_blocking=True), ptrs.to(dev, non_blocking=True), ng, True)

    nnz_per_step = []
    for b in range(n_batches):                            # also the warm-up of every kernel shape
        nnz_per_step.append(step()[1])
    nnz = sum(nnz_per_step) / n_batches                   # mean aggregated nnz (edges + self-loops) per layer and step
    nodes = sum(int(pk[0].size(0)) for pk in packed) / n_batches

    # ---- fixed-shape path (StaticBatchStep): the eager path above pays ~50 launches and two device-to-host reads of
    # graph preparation per step; padded to one shape the whole step replays from ONE CUDA graph
    static = None
    ms_static = ms_static_e2e = parity_static = None
    n_cap = e_cap = None
    if not args.no_graph:
        try:
            static = StaticBatchStep(model, packed, m["graphs"], m["f_in"], sym, dev)
            n_cap, e_cap = static.n_cap, static.e_cap
        except ValueError:
            static = None
    static_ok = static is not None
    if static_ok:
        def step_static():
            k = state["k"]; state["k"] = k + 1
            static.load(k)
            return static.replay()

        def step_static_e2e():
            k = state["k"]; state["k"] = k + 1
            static.load(k, pinned=True)
            return float(static.replay()[0].item())

        static.load(3)
        res = static.replay()
        # parity of the padded replay against the eager, unpadded step on the same batch (parameter gradients)
        x3, el3, pt3, _ = resident[3]
        x3 = x3.detach().requires_grad_(True)
        ei3, _ = egc_b200.collate_arrays(el3, pt3[1], pt3[0], num_nodes=int(x3.size(0)), validate=False)
        g3 = egc_b200.GraphStructure.from_edge_index(ei3, int(x3.size(0)), sym, True)
        h3 = x3
        for layer in model:
            h3 = torch.relu(layer(h3, g3))
        loss3 = egc_b200.global_mean_pool(h3, pt3[0]).pow(2).sum(1).mean()
        ref3 = torch.autograd.grad(loss3, [x3] + params)
        errs = [rel_err(res[0], loss3), rel_err(res[1][:x3.size(0)], ref3[0])] + [rel_err(a, b) for a, b in zip(res[2:], ref3[1:])]
        static.verify()
        parity_static = {"against": "the eager, unpadded step on the same batch (loss, d_x rows, parameter gradients)",
                         "max_rel_err": max(errs), "tol": 1e-5, "ok": bool(max(errs) < 1e-5)}

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / steps, _lib.launch_count() - l0

    steps = args.steps
    with ClockSampler(dev.index or 0) as clocks:
        ms_eager, launches = timed(step, steps, args.warmup)
        ms_eager_e2e, _ = timed(step_e2e, steps, 2)
        if static_ok:
            ms_static, _ = timed(step_static, steps, args.warmup)
            ms_static_e2e, _ = timed(step_static_e2e, steps, 2)
            static.verify()                               # the replayed builds still match the declared shape
    ms, ms_e2e = (ms_static, ms_static_e2e) if static_ok else (ms_eager, ms_eager_e2e)
    _lib.profile_enable(True)
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    kernels = {k: {"launches_per_step": c / steps, "ms_per_step": t / steps} for k, (c, t) in prof.items()}
    dim = m["hidden"] // m["heads"]
    peak, peak_src = load_peaks()
    n_i, e_i = int(round(nodes)), int(round(nnz))
    bf, bb = algorithmic_bytes(n_i, e_i, m["hidden"], m["heads"], m["bases"], dim, m["aggrs"])
    kbytes = kernel_algorithmic_bytes(n_i, e_i, m["hidden"], m["heads"], m["bases"], dim, m["aggrs"])
    cand = [k for k in kernels if kbytes.get(k)]
    dom = max(cand, key=lambda k: kernels[k]["ms_per_step"]) if cand else None
    roofline = None
    if dom:
        per_launch_ms = prof[dom][1] / prof[dom][0]
        achieved = kbytes[dom] / (per_launch_ms * 1e-3) / 1e9
        roofline = {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": kbytes[dom], "ms_per_launch": per_launch_ms,
                    "note": "launch-latency regime: a launch moves ~1-10 MB"}
    gpu_kernel_ms = sum(v["ms_per_step"] for v in kernels.values())
    cpu = None
    if not args.no_cpu_baseline:
        cpu = minibatch_cpu_baseline(args, m, host[0])
    edges = nnz * m["layers"]
    h2d = sum(pk[0].numel() * 4 + pk[1].numel() * 8 + pk[2].numel() * 4 for pk in packed) / n_batches
    line = {
        "metric": "EGConv fwd+bwd edges/s", "value": edges / (ms * 1e-3), "unit": "edges/s", "n_gpus": 1,
        "steps": steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": m["desc"], "graphs_per_step": m["graphs"], "mean_nodes_per_step": nodes,
                   "mean_nnz_per_layer": nnz, "layers": m["layers"],
                   "edges_counted": "aggregated nnz (edges + self-loops) x layers",
                   "structure": "cold: CSR / CSC / symnorm built every step (once per batch, shared by the layers)",
                   "l2": "working set < L2 (launch-latency regime); batches cycle over 8 different graph lists",
                   "algorithmic_bytes_per_step": (bf + bb) * m["layers"], "us_per_step": ms * 1e3,
                   "gpu_kernel_ms_per_step": gpu_kernel_ms,
                   "launch_mode": (f"fixed-shape batches (host-side padding to {n_cap} nodes / {e_cap} edges), the whole step - "
                                   "collation, CSR + CSC build, layers, readout, backward - replayed from ONE CUDA graph"
                                   if static_ok else "eager launches")},
        "eager": {"ms_per_step": ms_eager, "e2e_ms_per_step": ms_eager_e2e, "launches_per_step": launches / steps},
        "parity_check": parity_static,
        "clocks": clocks.summary(),
        "e2e": {"value": edges / (ms_e2e * 1e-3), "unit": "edges/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "input_pipeline": "pinned host arrays of the batch -> device collation -> stack -> loss read back"},
        "gpu_launches": launches,
        "step_roofline": {"achieved": (bf + bb) * m["layers"] / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                          "frac": (bf + bb) * m["layers"] / (ms * 1e-3) / 1e9 / peak},
        "roofline": roofline, "cpu_baseline": cpu, "kernels": kernels,
    }
    print(json.dumps(line))


def run_minibatch_dp(args, m):
    """Data-parallel mini-batch training over N ranks (BASELINE configs[4]: CIFAR-shaped EGC-M batches, and configs[0]):
    every rank runs the SAME replicated stack on its OWN batch of `graphs` small graphs per step (weak scaling), the
    parameter gradients are all-reduced per layer from inside the backward pass (NCCL, overlapped with the backward of
    the layers below).  Before timing: the all-reduced gradients are compared with ONE process on the concatenation of
    every rank's batch (`parity_check`)."""
    import torch.distributed as dist

    import egc_b200
    from egc_b200 import _lib
    from egc_b200.dist import OverlappedGradientAllReduce
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    dims = [m["f_in"]] + [m["hidden"]] * m["layers"]
    sym = "symnorm" in m["aggrs"]

    def make_model():
        torch.manual_seed(0)                              # identical replicated parameters on every rank
        return torch.nn.ModuleList([egc_b200.EGConv(dims[i], dims[i + 1], aggrs=m["aggrs"], num_heads=m["heads"],
                                                    num_bases=m["bases"]) for i in range(m["layers"])]).to(dev)

    def pack(graphs):
        counts = torch.tensor([[g[2], g[1].size(1)] for g in graphs])
        ptrs = torch.zeros((2, len(graphs) + 1), dtype=torch.int32)
        ptrs[:, 1:] = counts.cumsum(0).t().to(torch.int32)
        return (torch.cat([g[0] for g in graphs]).pin_memory(), torch.cat([g[1] for g in graphs], 1).pin_memory(),
                ptrs.pin_memory(), len(graphs))

    def loss_of(model, x, edge_local, ptrs):
        n = int(x.size(0))
        edge_index, _ = egc_b200.collate_arrays(edge_local, ptrs[1], ptrs[0], num_nodes=n, validate=False)
        g = egc_b200.GraphStructure.from_edge_index(edge_index, n, sym, True)
        h = x
        for layer in model:
            h = torch.relu(layer(h, g))
        return egc_b200.global_mean_pool(h, ptrs[0]).pow(2).sum(1).mean(), g.nnz

    model = make_model()
    sync = OverlappedGradientAllReduce(list(model))
    n_batches = 8
    host = [synth_small_graphs(args.workload, m["graphs"], (args.seed * 100 + b) * 64 + rank, m["f_in"]) for b in range(n_batches)]
    packed = [pack(g) for g in host]
    resident = [tuple(t.to(dev) if torch.is_tensor(t) else t for t in pk) for pk in packed]
    state = {"k": 0}

    def step_on(x, el, ptrs, read_loss):
        for p_ in model.parameters():
            p_.grad = None
        sync.begin(1.0 / world)                           # every rank holds the same number of graphs
        loss, nnz = loss_of(model, x, el, ptrs)
        loss.backward()
        sync.finish()
        return (float(loss.item()) if read_loss else loss), nnz

    def step():
        k = state["k"]; state["k"] = k + 1
        x, el, ptrs, _ = resident[k % n_batches]
        return step_on(x, el, ptrs, False)

    def step_e2e():
        k = state["k"]; state["k"] = k + 1
        x, el, ptrs, _ = packed[k % n_batches]
        return step_on(x.to(dev, non_blocking=True), el.to(dev, non_blocking=True), ptrs.to(dev, non_blocking=True), True)

    # ---- parity: DP gradients of batch 0 == one process on the concatenation of every rank's batch 0
    step_on(*resident[0][:3], False)
    dp_grads = [p_.grad.detach().clone() for p_ in model.parameters()]
    gathered = [None] * world
    dist.all_gather_object(gathered, [(x.clone(), ei.clone(), n) for x, ei, n in host[0]])
    ref_model = make_model()
    xa, ea, pa, _ = pack([g for part in gathered for g in part])
    ref_loss, _ = loss_of(ref_model, xa.to(dev), ea.to(dev), pa.to(dev))
    ref_grads = torch.autograd.grad(ref_loss, list(ref_model.parameters()))
    err = torch.tensor([max(rel_err(a, b) for a, b in zip(dp_grads, ref_grads))], device=dev, dtype=torch.float64)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    tol = 2e-5
    parity = {"against": "one process on the concatenation of every rank's batch (loss = mean over all graphs)",
              "max_rel_err": float(err.item()), "tol": tol, "ok": bool(float(err.item()) < tol)}
    del ref_model, ref_grads

    nnz_local = sum(step()[1] for _ in range(n_batches)) / n_batches      # also the warm-up of every kernel shape
    steps = args.steps

    # fixed-shape path: the whole local step replays from ONE CUDA graph, which also packs the (scaled) parameter
    # gradients into one flat buffer; then ONE NCCL all-reduce of that buffer.  Every rank pads to its own capacity.
    static = None
    if not args.no_graph:
        try:
            static = StaticBatchStep(model, packed, m["graphs"], m["f_in"], sym, dev, flat_scale=1.0 / world)
        except ValueError:
            static = None
    ok_all = torch.tensor([1.0 if static is not None else 0.0], device=dev)
    dist.all_reduce(ok_all, op=dist.ReduceOp.MIN)
    use_static = bool(ok_all.item() > 0)

    def step_static(pinned=False, read_loss=False):
        k = state["k"]; state["k"] = k + 1
        static.load(k, pinned=pinned)
        res = static.replay()
        dist.all_reduce(static.flat, op=dist.ReduceOp.SUM)
        return float(res[0].item()) if read_loss else res[0]

    parity_static = None
    if use_static:
        # same batch as the eager parity above (batch 0): flat buffer == the eager overlapped all-reduce result
        static.load(0)
        static.replay()
        dist.all_reduce(static.flat, op=dist.ReduceOp.SUM)
        e = torch.tensor([rel_err(static.flat, torch.cat([g_.reshape(-1) for g_ in dp_grads]))], device=dev, dtype=torch.float64)
        dist.all_reduce(e, op=dist.ReduceOp.MAX)
        static.verify()
        parity_static = {"against": "the eager data-parallel step on the same batches (all-reduced parameter gradients)",
                         "max_rel_err": float(e.item()), "tol": 1e-5, "ok": bool(float(e.item()) < 1e-5)}
    with ClockSampler(dev.index or 0) as clocks:
        ms_eager, launches = cuda_timed(step, steps, args.warmup, dist.barrier)
        ms_eager_e2e, _ = cuda_timed(step_e2e, steps, 2, dist.barrier)
        if use_static:
            ms, _ = cuda_timed(step_static, steps, args.warmup, dist.barrier)
            ms_e2e, _ = cuda_timed(lambda: step_static(True, True), steps, 2, dist.barrier)
            static.verify()
        else:
            ms, ms_e2e = ms_eager, ms_eager_e2e
    eag = torch.tensor([ms_eager, ms_eager_e2e], device=dev, dtype=torch.float64)
    dist.all_reduce(eag, op=dist.ReduceOp.MAX)
    t = torch.tensor([ms, ms_e2e, nnz_local * m["layers"], launches], device=dev, dtype=torch.float64)
    tmax, tsum = t.clone(), t.clone()
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    if rank == 0:
        ms, ms_e2e = float(tmax[0]), float(tmax[1])
        edges = float(tsum[2])
        n_param = sum(p_.numel() for p_ in model.parameters())
        h2d = sum(pk[0].numel() * 4 + pk[1].numel() * 8 + pk[2].numel() * 4 for pk in packed) / n_batches
        print(json.dumps({
            "metric": "EGConv fwd+bwd edges/s", "value": edges / (ms * 1e-3), "unit": "edges/s", "n_gpus": world,
            "steps": steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": m["desc"] + f", data-parallel over {world} GPUs ({m['graphs']} graphs per GPU and step)",
                       "graphs_per_step": m["graphs"] * world, "layers": m["layers"],
                       "edges_counted": "aggregated nnz (edges + self-loops) x layers, summed over the ranks",
                       "structure": "cold: CSR / CSC / symnorm built every step on every rank",
                       "all_reduce": f"{n_param * 4} B of parameter gradients per step, one NCCL all-reduce per layer launched from "
                                     "inside backward (overlaps the backward of the layers below)",
                       "l2": "working set < L2 (launch-latency regime); batches cycle over 8 different graph lists per rank"},
            "parity_check": parity, "parity_check_graph_replay": parity_static,
            "launch_mode": ("fixed-shape batches: the local step replayed from ONE CUDA graph (it packs the scaled gradients "
                            "into one flat buffer), then ONE NCCL all-reduce" if use_static else
                            "eager launches, one NCCL all-reduce per layer launched from inside backward"),
            "eager_overlapped": {"ms_per_step": float(eag[0]), "e2e_ms_per_step": float(eag[1]),
                                 "note": "eager launches, per-layer all-reduce launched from backward hooks (host-launch-bound)"},
            "clocks": clocks.summary(),
            "e2e": {"value": edges / (ms_e2e * 1e-3), "unit": "edges/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": 4 * world,
                    "input_pipeline": "pinned host arrays of the batch -> device collation -> stack -> loss read back"},
            "gpu_launches": int(float(tsum[3])), "roofline": None, "cpu_baseline": None}))
    dist.destroy_process_group()
    if not parity["ok"] or (parity_static is not None and not parity_static["ok"]):
        sys.exit(f"bench.py: data-parallel gradients differ from the single-process run: {parity} {parity_static}")


def minibatch_cpu_step_factory(m, graphs):
    """The same stack on the host cores through the oracle port (reference path, pure-torch leaf ops)."""
    from oracle import batching as OB
    from oracle import restatement as R
    torch.manual_seed(0)
    dims = [m["f_in"]] + [m["hidden"]] * m["layers"]
    model = torch.nn.ModuleList([R.EGConvOracle(dims[i], dims[i + 1], aggrs=m["aggrs"], num_heads=m["heads"],
                                                num_bases=m["bases"]) for i in range(m["layers"])])
    x, ei, batch, ptr = OB.collate(graphs)
    nnz = int(ei.size(1)) + int(x.size(0))

    def step():
        for p_ in model.parameters():
            p_.grad = None
        h = x.detach().requires_grad_(True)
        for layer in model:                                   # every layer prepares the graph itself, as the reference
            h = torch.relu(layer(h, ei))
        OB.global_pool(h, batch, len(graphs), "mean").pow(2).sum(1).mean().backward()

    return step, nnz * m["layers"]


def minibatch_cpu_baseline(args, m, graphs, steps=3):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, edges = minibatch_cpu_step_factory(m, graphs)
    t = time_cpu(step, steps, 1)
    return {"value": edges / t, "unit": "edges/s", "cores": cores, "kind": "port",
            "sample": f"one batch of {len(graphs)} graphs, 1 warm-up + {steps} timed steps, {t * 1e3:.1f} ms/step"}


def run_minibatch_reference_arm(args, m):
    graphs = synth_small_graphs(args.workload, m["graphs"], args.seed * 100, m["f_in"])
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, edges = minibatch_cpu_step_factory(m, graphs)
    t = time_cpu(step, max(args.steps, 1), args.warmup)
    value = edges / t
    sample = f"one batch of {len(graphs)} graphs per step"
    print(json.dumps({
        "impl": "reference", "metric": "EGConv fwd+bwd edges/s", "value": value, "unit": "edges/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": m["desc"], "sample": sample,
                   "path": "oracle port of the reference's PyG path (pure-torch leaf ops), host CPU"},
        "cpu_baseline": {"value": value, "unit": "edges/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------
# heterogeneous workload: REGConv on an ogbn-mag-shaped heterogeneous graph (SURVEY.md section 8 f-2)
# ------------------------------------------------------------------------------------------------
RMAG_NODES = {"author": 1_134_649, "field_of_study": 59_965, "institution": 8_740, "paper": 736_389}   # ref rmag/models.py:10-15
# directed edge counts of ogbn-mag per stored relation; every non-square relation is used in both directions and
# paper-cites-paper is symmetrised (ref rmag/configs.py:84-98)
RMAG_EDGES = {("author", "affiliated_with", "institution"): 1_043_998, ("author", "writes", "paper"): 7_145_660,
              ("paper", "cites", "paper"): 5_416_271, ("paper", "has_topic", "field_of_study"): 7_505_078}
RMAG = dict(f_in=128, f_out=128, heads=8, bases=4,
            desc="REGConv (mean+max per relation, H8 B4) 128->128 on an ogbn-mag-shaped heterogeneous graph, 1 layer fwd+bwd")


def synth_hetero_csr(scale: float, seed: int):
    """{(src, rel, dst): (rowptr int64, col int64, n_src)} of adj_t (rows = targets, sorted by (target, source),
    duplicates kept), Zipf-like popularity on both endpoints; node / edge counts scaled by `scale`."""
    rng = np.random.default_rng(seed)
    sizes = {t: max(int(n * scale), 4) for t, n in RMAG_NODES.items()}

    def endpoints(n, e, a):
        return np.minimum((n * rng.random(e) ** (1.0 / (1.0 - a))).astype(np.int64), n - 1) if a else rng.integers(0, n, e)

    def to_csr(dst, src, n_dst, n_src):
        order = np.argsort(dst * n_src + src, kind="stable")
        rowptr = np.zeros(n_dst + 1, dtype=np.int64)
        np.cumsum(np.bincount(dst, minlength=n_dst), out=rowptr[1:])
        return torch.from_numpy(rowptr), torch.from_numpy(src[order]), n_src

    out = {}
    for (s, r, d), e0 in RMAG_EDGES.items():
        e = max(int(e0 * scale), 8)
        perm_s, perm_d = rng.permutation(sizes[s]), rng.permutation(sizes[d])
        src, dst = perm_s[endpoints(sizes[s], e, 0.5)], perm_d[endpoints(sizes[d], e, 0.6)]
        if s == d:                                             # to_symmetric(): both directions, duplicates merged
            key = np.unique(np.concatenate([dst * sizes[s] + src, src * sizes[s] + dst]))
            dst, src = key // sizes[s], key % sizes[s]
            out[(s, r, d)] = to_csr(dst, src, sizes[d], sizes[s])
        else:
            out[(s, r, d)] = to_csr(dst, src, sizes[d], sizes[s])
            out[(d, "to", s)] = to_csr(src, dst, sizes[s], sizes[d])
    return sizes, out


def rmag_cpu_step_factory(scale, seed):
    from oracle import hetero as OH
    sizes, csr = synth_hetero_csr(scale, seed)
    torch.manual_seed(0)
    model = OH.REGConvOracle(RMAG["f_in"], RMAG["f_out"], RMAG["heads"], RMAG["bases"])
    x = {t: torch.randn(n, RMAG["f_in"], requires_grad=True) for t, n in sizes.items()}
    go = {t: torch.randn(n, RMAG["f_out"]) for t, n in sizes.items()}
    nnz = sum(int(v[1].numel()) for v in csr.values())

    def step():
        for p_ in model.parameters():
            p_.grad = None
        for v in x.values():
            v.grad = None
        out = model(x, csr)
        sum((out[t] * go[t]).sum() for t in sizes).backward()

    return step, nnz, f"graph scaled to {scale:.4f} of ogbn-mag ({sum(sizes.values())} nodes, {nnz} nnz over 7 relations)"


def run_rmag_reference_arm(args):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, nnz, sample = rmag_cpu_step_factory(1 / 64, args.seed)
    t = time_cpu(step, max(args.steps, 1), args.warmup)
    value = nnz / t
    print(json.dumps({
        "impl": "reference", "metric": "EGConv fwd+bwd edges/s", "value": value, "unit": "edges/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": RMAG["desc"], "sample": sample,
                   "path": "oracle port of the reference's REGConv (pure-torch leaf ops), host CPU"},
        "cpu_baseline": {"value": value, "unit": "edges/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


def run_rmag(args):
    import egc_b200
    from egc_b200 import _lib
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    sizes, csr = synth_hetero_csr(1.0, args.seed)
    torch.manual_seed(0)
    conv = egc_b200.REGConv(RMAG["f_in"], RMAG["f_out"], RMAG["heads"], RMAG["bases"]).to(dev)
    params = list(conv.parameters())
    adj = {k: egc_b200.SparseTensor(rowptr=rp.to(dev), col=col.to(dev), sparse_sizes=(rp.numel() - 1, ns), is_sorted=True)
           for k, (rp, col, ns) in csr.items()}
    rel_nnz = {k: int(v[1].numel()) for k, v in csr.items()}
    nnz = sum(rel_nnz.values())
    del csr
    types = list(sizes)
    # as in the reference only papers carry input features (they arrive from the host in the e2e arm); the other node
    # types hold trainable embeddings that live on the device (ref rmag/models.py:150-175)
    x = {t: torch.randn(n, RMAG["f_in"], device=dev, requires_grad=True) for t, n in sizes.items()}
    go = {t: torch.randn(n, RMAG["f_out"], device=dev) for t, n in sizes.items()}
    x_paper_host = torch.randn(sizes["paper"], RMAG["f_in"]).pin_memory()

    def step():
        out = conv(x, adj)
        torch.autograd.grad([out[t] for t in types], [x[t] for t in types] + params, [go[t] for t in types])
        return out

    def step_e2e():
        with torch.no_grad():
            x["paper"].copy_(x_paper_host, non_blocking=True)
        out = conv(x, adj)
        loss = sum((out[t] * go[t]).sum() for t in types)
        torch.autograd.grad(loss, [x[t] for t in types] + params)
        return float(loss.item())

    step()                                                   # builds + caches CSR / CSC / plans of the 7 relations

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / steps, _lib.launch_count() - l0

    with ClockSampler(dev.index or 0) as clocks:
        ms, launches = timed(step, args.steps, args.warmup)
        ms_e2e, _ = timed(step_e2e, max(3, min(args.steps, 10)), 2)
    _lib.profile_enable(True)
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    kernels = {k: {"launches_per_step": c / args.steps, "ms_per_step": t / args.steps} for k, (c, t) in prof.items()}
    peak, peak_src = load_peaks()
    # unique-bytes model (SURVEY 8d conventions): per node type the projection streams, per relation the fused
    # aggregate + combine forward and its two backward passes (mean: one linear stream; max: one routed slot)
    bd, hb, hd = RMAG["bases"] * (RMAG["f_out"] // RMAG["heads"]), RMAG["heads"] * RMAG["bases"], RMAG["f_out"]
    total = 0
    for t, n in sizes.items():
        r_t = sum(1 for k in adj if k[2] == t)
        hab = hb * (1 + 2 * r_t)
        total += 4 * n * (RMAG["f_in"] + bd + hab) * 3                                  # fwd, d_x and wgrad GEMM streams
        total += 4 * n * (2 * bd + 2 * hb + 3 * hd)                                     # root term fwd + bwd
    for (s_, r_, d_), a in adj.items():
        e = rel_nnz[(s_, r_, d_)]
        nd, ns = sizes[d_], sizes[s_]
        total += 4 * ns * bd + 4 * nd * (2 * hb + hd + 3 * bd) + 4 * (e + nd)            # forward incl. saved + arg
        total += 4 * nd * (hd + 4 * hb + 3 * bd + 2 * bd) + 4 * ns * 2 * bd + 8 * (e + nd)   # backward
    step_gbs = total / (ms * 1e-3) / 1e9
    cand = {k: v for k, v in kernels.items() if k in ("k_aggregate_fwd", "k_scatter_bwd", "k_combine_bwd", "k_project_tc")}
    dom = max(cand, key=lambda k: cand[k]["ms_per_step"]) if cand else None
    cpu = None
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        cstep, cnnz, sample = rmag_cpu_step_factory(1 / 64, args.seed)
        t_cpu = time_cpu(cstep, 2, 1)
        cpu = {"value": cnnz / t_cpu, "unit": "edges/s", "cores": cores, "kind": "port",
               "sample": f"{sample}; 1 warm-up + 2 timed fwd+bwd steps, {t_cpu:.2f} s/step"}
    line = {
        "metric": "EGConv fwd+bwd edges/s", "value": nnz / (ms * 1e-3), "unit": "edges/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": RMAG["desc"], "nodes": sizes, "relations": len(adj), "nnz": nnz,
                   "structure": "cached (7 relation graphs prepared once)", "l2": "no flush: working set >> L2",
                   "algorithmic_bytes_per_step": total},
        "clocks": clocks.summary(),
        "e2e": {"value": nnz / (ms_e2e * 1e-3), "unit": "edges/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": x_paper_host.numel() * 4, "d2h_bytes_per_step": 4},
        "gpu_launches": launches,
        "step_roofline": {"achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak, "peak_source": peak_src},
        "roofline": ({"kernel": dom, "bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                      "traffic": None, "note": "per-kernel byte model not split per relation; see step_roofline",
                      "ms_per_step": cand[dom]["ms_per_step"]} if dom else None),
        "cpu_baseline": cpu, "kernels": kernels,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="arxiv", choices=sorted(WORKLOADS) + sorted(MINIBATCH) + ["rmag"])
    ap.add_argument("--layers", type=int, default=1,
                    help="full-graph workloads: 1 = one EGConv layer (configs[1] / [3]); >= 2 = the reference's EGC stack (configs[2] uses 3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the `other_configs` object (3-layer arxiv stack, mag, uniform graph) of the default run")
    ap.add_argument("--transport", default="peer", choices=["peer", "nccl"],
                    help="multi-GPU halo exchange: our NVLink peer-memory kernels (default) or the NCCL baseline")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--bwd-flags", type=int, default=0, help="EGC_BWD_* tuning bits passed to egc_aggregate_bwd (A/B runs)")
    ap.add_argument("--locality", type=float, default=-1.0,
                    help="p_intra of the synthetic generator (default 0.8 with 8 id blocks, for every GPU count)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (output, d_x, parameter "
                         "gradients) as DIR/<name>.npy; single-GPU full-graph workloads")
    args = ap.parse_args()
    if args.steps < 1:
        sys.exit("--steps must be >= 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS or args.gpus > 1
                              or int(os.environ.get("WORLD_SIZE", 1)) > 1):
        sys.exit("--dump-outputs is implemented for the single-GPU full-graph workloads (" + ", ".join(WORKLOADS) + ")")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    if args.workload == "rmag":
        if rank != 0:
            return
        if args.impl == "reference":
            run_rmag_reference_arm(args)
        else:
            run_rmag(args)
        return
    if args.workload in MINIBATCH:
        if args.impl == "reference":
            if rank == 0:
                run_minibatch_reference_arm(args, MINIBATCH[args.workload])
        elif int(os.environ.get("WORLD_SIZE", 1)) > 1:      # data-parallel: per-rank batches, overlapped gradient all-reduce
            run_minibatch_dp(args, MINIBATCH[args.workload])
        else:
            run_minibatch(args, MINIBATCH[args.workload])
        return
    w = WORKLOADS[args.workload]
    if args.layers < 1:
        sys.exit("--layers must be >= 1")

    if args.impl == "reference":
        if rank != 0:
            return
        run_reference_arm(args, args.workload, w)
        return

    if args.gpus > 1 or int(os.environ.get("WORLD_SIZE", 1)) > 1:
        if "RANK" not in os.environ:
            sys.exit("multi-GPU runs are launched with torch.distributed.run (see the module docstring)")
        run_multi_gpu(args, args.workload, w)
        return
    run_single_gpu(args, args.workload, w)


if __name__ == "__main__":
    main()
