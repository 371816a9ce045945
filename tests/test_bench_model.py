"""Host-side checks of bench.py: the unique-bytes roofline model against the figures SURVEY.md section 8(d) /
BASELINE.md section 2 state, the synthetic generators' shapes, and the JSON contract of the CPU arms (no GPU)."""
import json
import subprocess
import sys

import numpy as np
import torch

import bench


def test_algorithmic_bytes_match_the_survey_figures():
    # cfg2: arxiv-shaped EGC-M, N = 169 343, E = 2 484 941 -> 0.510 + 1.247 = 1.756 GB/layer, 707 B/edge
    bf, bb = bench.algorithmic_bytes(169_343, 2_484_941, 128, 4, 4, 32, ["symnorm", "max", "std"])
    assert abs(bf / 1e9 - 0.510) < 0.002 and abs(bb / 1e9 - 1.247) < 0.002
    assert abs((bf + bb) / 2_484_941 - 707) < 1.5
    # cfg4: mag-shaped EGC-S, N = 736 389, E = 11 529 061 -> 1.372 + 2.458 = 3.829 GB/layer, 332 B/edge
    bf, bb = bench.algorithmic_bytes(736_389, 11_529_061, 128, 8, 4, 16, ["symnorm"])
    assert abs(bf / 1e9 - 1.372) < 0.002 and abs(bb / 1e9 - 2.458) < 0.002
    assert abs((bf + bb) / 11_529_061 - 332) < 1.0


def test_per_kernel_bytes_add_up_to_the_step_model():
    """Every byte of Bf + Bb is attributed to exactly one kernel launch (2 projection launches + wgrad), up to the
    terms the per-kernel model adds on purpose: the saved aggregates, the symnorm weight streams, the routed slab."""
    n, e, aggrs = 169_343, 2_498_405, ["symnorm", "max", "std"]
    bf, bb = bench.algorithmic_bytes(n, e, 128, 4, 4, 32, aggrs)
    k = bench.kernel_algorithmic_bytes(n, e, 128, 4, 4, 32, aggrs)
    step = 2 * k["k_project_tc"] + k["k_wgrad_tc"] + k["k_aggregate_fwd"] + k["k_combine_bwd"] + k["k_route_minmax"] + k["k_scatter_bwd"]
    assert step >= bf + bb                       # the kernel model never undercounts the step model
    assert step < 2.2 * (bf + bb)                # and stays within the saved-state / re-read terms


def test_synthetic_graph_shapes():
    z = bench.synth_small_graphs("zinc", 64, 0, 8)
    n = sum(g[2] for g in z)
    e = sum(g[1].size(1) for g in z)
    assert 20 < n / 64 < 27 and 1.9 < e / n < 2.4
    assert all(int(g[1].max()) < g[2] and g[0].shape == (g[2], 8) for g in z)
    c = bench.synth_small_graphs("cifar", 8, 0, 5)
    assert all(85 <= g[2] <= 150 and g[1].size(1) == 8 * g[2] for g in c)
    sizes, csr = bench.synth_hetero_csr(1 / 512, 0)
    assert set(sizes) == set(bench.RMAG_NODES) and len(csr) == 7
    for (s, r, d), (rowptr, col, n_src) in csr.items():
        assert rowptr.numel() == sizes[d] + 1 and n_src == sizes[s] and int(rowptr[-1]) == col.numel()
        assert int(col.max()) < n_src and bool((rowptr[1:] >= rowptr[:-1]).all())
    rp, col, _ = csr[("paper", "cites", "paper")]                     # symmetrised: (i, j) present iff (j, i) is
    row = torch.repeat_interleave(torch.arange(rp.numel() - 1), rp[1:] - rp[:-1])
    a = set(zip(row.tolist(), col.tolist()))
    assert all((j, i) in a for i, j in list(a)[:500])


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--workload", "zinc", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, cwd=bench.ROOT, timeout=600)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "edges/s" and line["value"] > 0 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_keeps_the_same_seeded_rows(tmp_path):
    n = bench.DUMP_ROWS + 1000
    out = torch.arange(n, dtype=torch.float64)[:, None].repeat(1, 3)          # row i holds i
    grad_w = torch.randn(4, 5)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"out": out, "grad_w": grad_w}, n)
    o = np.load(tmp_path / "a" / "out.npy")
    assert o.dtype == np.float32 and o.shape == (bench.DUMP_ROWS, 3)
    assert (np.diff(o[:, 0]) > 0).all() and o[-1, 0] < n and (o[:, 1] == o[:, 0]).all()
    assert np.array_equal(np.load(tmp_path / "b" / "out.npy"), o)
    assert np.array_equal(np.load(tmp_path / "a" / "grad_w.npy"), grad_w.numpy())


def test_rejected_arguments_exit_before_any_work():
    for extra, msg in ((["--steps", "0"], "--steps must be >= 1"),
                       (["--workload", "zinc", "--dump-outputs", "unused"], "--dump-outputs is implemented for")):
        out = subprocess.run([sys.executable, "bench.py"] + extra, capture_output=True, text=True, cwd=bench.ROOT,
                             timeout=120)
        assert out.returncode != 0 and not out.stdout.strip() and msg in out.stderr


def test_local_roofline_of_partitioned_runs():
    w = bench.WORKLOADS["arxiv"]
    kernels = {"k_scatter_bwd": {"launches_per_step": 1.0, "ms_per_step": 0.25},
               "k_aggregate_fwd": {"launches_per_step": 2.0, "ms_per_step": 0.19},
               "k_peer_wait": {"launches_per_step": 4.0, "ms_per_step": 2.5},            # no byte model: never dominant
               "k_project_tc": {"launches_per_step": 2.0, "ms_per_step": 0.13}}
    r = bench.local_roofline(kernels, 84_000, 1_250_000, w, 6500.0, "test")
    assert r["kernel"] == "k_scatter_bwd" and r["unit"] == "GB/s" and 0 < r["frac"] < 1
    kb = bench.kernel_algorithmic_bytes(84_000, 1_250_000, w["f_in"], w["heads"], w["bases"], 32, w["aggrs"])
    assert abs(r["achieved"] - kb["k_scatter_bwd"] / 0.25e-3 / 1e9) < 1e-6
    assert bench.local_roofline({}, 10, 10, w, 6500.0, "test") is None
    assert bench.local_roofline({"k_scatter_bwd": {"ms_per_step": "bad"}}, 10, 10, w, 6500.0, "test") is None
