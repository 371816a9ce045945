"""Every aggregation kernel the dispatch of egc_aggregate_fwd / _bf16 and egc_aggregate_bwd / _bf16 can select, checked
against the fp64 oracle, with the kernel that served each case asserted by name.

A case runs the aggregation + combination stage alone: random basis rows [n, B*D] and weightings [n, H*A*B] are the
leaves, the oracle is R.aggregate + R.combine (with autograd for d_bases, d_weightings, d_bias and the weightings' column
sums) over the device's own CSR, and the kernels run through functional.aggregate_combine / aggregate_backward.  The bar is
the suite's: max(1e-5, 4 x the fp32 oracle's own error against fp64); argmax source ids are bit-exact.  Basis rows are
dyadic (multiples of 1/4, |x| < 16: exact in fp32 and bf16), so min / max winners are decided by exact values on both
sides.  The graphs have rows and columns on both sides of EGC_CHUNK_EDGES, empty rows and empty columns.

Which kernel served a case is read from torch.profiler and matched against EXPECT, the one table of expected kernel names:
a change of the dispatch fails here and points at the table instead of silently moving coverage.  The switches read once
per process (EGC_FWD_WARP_PER_ROW, EGC_BWD_RING, EGC_BWD_WARP_PER_COLUMN) run in a fresh interpreter per setting.
BRANCHES maps every branch of the dispatch in aggregate_api.cu to the cases that reach it.

Not here: the dropout instantiations (DROP = true) are covered by tests/test_gpu_dropout.py.  Pass 1 with EV = 1 is reached
through D % 4 != 0 only: the target-side streams live in the 16-byte aligned workspace (or in a caller's tstreams_out,
which must be aligned), so no caller pointer can make them unaligned."""
import os
import re
import subprocess
import sys
import zlib
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

import egc_b200
from egc_b200 import _lib
from egc_b200.functional import aggregate_backward, aggregate_combine, make_desc
from oracle import restatement as R
from tests.util import random_graph, rel_err, to_adj_csr

gpu = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWITCHES = ("EGC_FWD_WARP_PER_ROW", "EGC_BWD_RING", "EGC_BWD_WARP_PER_COLUMN")
DET, NO_HUB = _lib.BWD_DETERMINISTIC, _lib.BWD_NO_HUB_PRIVATISATION

# EGC_STATIC_CFGS of aggregate_fast.cuh, in index order: heads, bases, head dim, aggregators
STATIC_CFGS = [(4, 4, 32, ("symnorm", "max", "std")), (8, 4, 16, ("symnorm",)), (4, 4, 32, ("symnorm",)),
               (4, 4, 32, ("symnorm", "max", "mean")), (8, 4, 16, ("mean", "max")), (8, 4, 16, ("sum",))]


def _static_name(i):
    h, b, d, aggrs = STATIC_CFGS[i]
    return f"egc::StaticCfg<{h}, {b}, {d}, {', '.join(str(_lib.AGGR_CODES[a]) for a in aggrs)}>"


def _has_arg(aggrs):
    return any(a in ("max", "min") for a in aggrs)


# ------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    heads: int
    bases: int
    dim: int
    aggrs: tuple
    stage: str                      # "fwd": the forward's kernels are asserted, "bwd": the backward's
    graph: str = "pattern"          # "pattern" or "hubcap" (_graph)
    valued: bool = False            # per-entry linear weights (val_lin)
    bf16: bool = False              # bf16 basis rows (and target-side streams)
    arg: bool = True                # forward: request arg_out and the saved tensors (ARG = true with min / max)
    offset: str = ""                # "bases" / "grad_out": that tensor starts 4 bytes into its allocation
    flags: int = 0


CASES = {}
for _i, (_h, _b, _d, _a) in enumerate(STATIC_CFGS):
    CASES[f"fwd_rows_static{_i}"] = Case(_h, _b, _d, _a, "fwd")
    if _has_arg(_a):                                         # ARG is a template parameter
        CASES[f"fwd_rows_static{_i}_noarg"] = Case(_h, _b, _d, _a, "fwd", arg=False)
    CASES[f"fwd_bf16_static{_i}"] = Case(_h, _b, _d, _a, "fwd", bf16=True)
    if _has_arg(_a):
        CASES[f"fwd_bf16_static{_i}_noarg"] = Case(_h, _b, _d, _a, "fwd", bf16=True, arg=False)
    CASES[f"bwd_p1_static{_i}"] = Case(_h, _b, _d, _a, "bwd")
    CASES[f"bwd_p1_static{_i}_bf16"] = Case(_h, _b, _d, _a, "bwd", bf16=True)
CASES.update({
    # forward, fp32
    "fwd_rows_dyn_g32": Case(4, 4, 32, ("sum", "mean", "min", "var"), "fwd"),
    "fwd_rows_dyn_g16": Case(4, 3, 16, ("max", "mean"), "fwd"),                        # B*D = 48
    # row-block staging above 72 KB (A*B*D + 8 rows of H*A*B weights + the window): the warp-per-row kernel
    "fwd_fast_dyn_g32": Case(4, 4, 32, ("sum", "mean", "symnorm", "min", "max", "var", "std"), "fwd"),
    "fwd_fast_dyn_g16": Case(8, 4, 16, ("sum", "mean", "min", "max", "std"), "fwd"),
    "fwd_general_v4_npass": Case(8, 4, 44, ("symnorm", "max", "mean"), "fwd"),         # B*D = 176: two passes
    "fwd_general_v4_valued": Case(4, 4, 32, ("sum", "max"), "fwd", valued=True),
    "fwd_general_v1_bd30": Case(4, 3, 10, ("sum", "min", "var"), "fwd"),
    "fwd_general_v1_valued": Case(4, 3, 10, ("mean", "max"), "fwd", valued=True),
    "fwd_general_v1_offset_bases": Case(4, 4, 32, ("symnorm", "max", "std"), "fwd", offset="bases"),
    # forward, bf16 basis rows
    "fwd_bf16_dyn_g16": Case(4, 4, 24, ("sum", "max", "std"), "fwd", bf16=True),     # B*D = 96
    "fwd_bf16_dyn_g8": Case(4, 4, 10, ("mean", "min"), "fwd", bf16=True),            # B*D = 40
    # backward pass 1
    "bwd_p1_dyn_ev4": Case(4, 4, 32, ("sum", "mean", "min", "var"), "bwd"),
    "bwd_p1_dyn_ev1": Case(4, 3, 10, ("sum", "min", "var"), "bwd"),
    "bwd_p1_dyn_ev4_linw": Case(4, 4, 32, ("sum", "max"), "bwd", valued=True),
    "bwd_p1_dyn_ev4_bf16": Case(4, 4, 24, ("sum", "max", "std"), "bwd", bf16=True),
    "bwd_p1_dyn_ev1_bf16": Case(4, 4, 10, ("mean", "min"), "bwd", bf16=True),
    "bwd_p1_vec16_off": Case(4, 4, 32, ("symnorm", "max", "std"), "bwd", offset="grad_out"),   # static shape, no vec16
    "bwd_colsum_fused": Case(4, 4, 32, ("sum", "mean"), "bwd"),
    "bwd_colsum_two_stage": Case(8, 8, 16, ("symnorm", "max", "std"), "bwd"),           # H*A*B = 192
    # min / max routing
    "bwd_route_atomic_hubs": Case(4, 4, 16, ("max", "min", "sum"), "bwd"),
    "bwd_route_atomic_no_hub": Case(4, 4, 16, ("max", "min", "sum"), "bwd", flags=NO_HUB),
    "bwd_route_atomic_hubcap": Case(4, 4, 8, ("max", "min"), "bwd", graph="hubcap"),    # > 1024 long columns
    "bwd_route_det_v4": Case(4, 4, 16, ("max", "min", "sum"), "bwd", flags=DET),
    "bwd_route_det_v1": Case(4, 3, 10, ("sum", "min", "var"), "bwd", flags=DET),
    # pass 2
    "bwd_p2_ring": Case(4, 4, 32, ("symnorm", "std"), "bwd"),                           # three streams, G = 32
    "bwd_p2_cols32": Case(4, 4, 32, ("sum",), "bwd"),                                   # one stream
    "bwd_p2_cols16": Case(4, 4, 16, ("symnorm", "std"), "bwd"),                         # B*D = 64
    "bwd_p2_ring_bf16": Case(4, 4, 32, ("symnorm", "std"), "bwd", bf16=True),
    "bwd_p2_cols32_bf16": Case(4, 4, 32, ("sum",), "bwd", bf16=True),
    "bwd_p2_cols16_bf16": Case(4, 4, 16, ("symnorm", "std"), "bwd", bf16=True),
    "bwd_p2_scatter_v1_linw": Case(4, 3, 10, ("mean", "max"), "bwd", valued=True),
    "bwd_p2_scatter_npass": Case(8, 4, 44, ("symnorm", "mean"), "bwd"),                 # two passes: mode-1 merge launch
})

# ------------------------------------------------------------------------------------------------
# EXPECT: case -> {switch setting ("" = none): [expected kernel, ...]}.  An entry is a demangled-name fragment in which
# `#` stands for any number; `name*N` = at least N launches; `!name` = not launched.
# ------------------------------------------------------------------------------------------------
EXPECT = {}
for _i, (_h, _b, _d, _a) in enumerate(STATIC_CFGS):
    _s = _static_name(_i)
    for _arg in ((True, False) if _has_arg(_a) else (False,)):
        _sfx = "" if _arg or not _has_arg(_a) else "_noarg"
        _t = str(_arg).lower()
        EXPECT[f"fwd_rows_static{_i}{_sfx}"] = {
            "": [f"k_aggregate_rows<{_s}, {_t}, float, false>"],
            "EGC_FWD_WARP_PER_ROW=1": [f"k_aggregate_fast<{_s}, {_t}, false>"]}
        EXPECT[f"fwd_bf16_static{_i}{_sfx}"] = {"": [f"k_aggregate_rows<egc::Bf16Cfg<{_s} >, {_t}, __nv_bfloat16, false>"]}
    EXPECT[f"bwd_p1_static{_i}"] = {"": [f"k_combine_bwd<{_s}, 4, false, float>", "k_colsum_partials"]}
    EXPECT[f"bwd_p1_static{_i}_bf16"] = {"": [f"k_combine_bwd<{_s}, 4, false, __nv_bfloat16>"]}
EXPECT.update({
    "fwd_rows_dyn_g32": {"": ["k_aggregate_rows<egc::DynCfg<#, 32>, true, float, false>"],
                         "EGC_FWD_WARP_PER_ROW=1": ["k_aggregate_fast<egc::DynCfg<#, 32>, true, false>"]},
    "fwd_rows_dyn_g16": {"": ["k_aggregate_rows<egc::DynCfg<#, 16>, true, float, false>"],
                         "EGC_FWD_WARP_PER_ROW=1": ["k_aggregate_fast<egc::DynCfg<#, 16>, true, false>"]},
    "fwd_fast_dyn_g32": {"": ["k_aggregate_fast<egc::DynCfg<#, 32>, true, false>", "!k_aggregate_rows"]},
    "fwd_fast_dyn_g16": {"": ["k_aggregate_fast<egc::DynCfg<#, 16>, true, false>", "!k_aggregate_rows"]},
    # general kernel: a second launch (mode 1) merges the chunk partials of the long rows
    "fwd_general_v4_npass": {"": ["k_aggregate<#, 4, false, true, false>*2"]},
    "fwd_general_v4_valued": {"": ["k_aggregate<#, 4, true, true, false>*2"]},
    "fwd_general_v1_bd30": {"": ["k_aggregate<#, 1, false, true, false>*2"]},
    "fwd_general_v1_valued": {"": ["k_aggregate<#, 1, true, true, false>*2"]},
    "fwd_general_v1_offset_bases": {"": ["k_aggregate<#, 1, false, true, false>*2"]},
    "fwd_bf16_dyn_g16": {"": ["k_aggregate_rows<egc::DynCfg<#, 16>, true, __nv_bfloat16, false>"]},
    "fwd_bf16_dyn_g8": {"": ["k_aggregate_rows<egc::DynCfg<#, 8>, true, __nv_bfloat16, false>"]},
    "bwd_p1_dyn_ev4": {"": ["k_combine_bwd<egc::DynCfg<0, 32>, 4, false, float>"]},
    "bwd_p1_dyn_ev1": {"": ["k_combine_bwd<egc::DynCfg<0, 32>, 1, false, float>"]},
    "bwd_p1_dyn_ev4_linw": {"": ["k_combine_bwd<egc::DynCfg<0, 32>, 4, true, float>"]},
    "bwd_p1_dyn_ev4_bf16": {"": ["k_combine_bwd<egc::DynCfg<0, 32>, 4, false, __nv_bfloat16>"]},
    "bwd_p1_dyn_ev1_bf16": {"": ["k_combine_bwd<egc::DynCfg<0, 32>, 1, false, __nv_bfloat16>"]},
    "bwd_p1_vec16_off": {"": ["k_combine_bwd<egc::DynCfg<0, 32>, 4, false, float>", "!k_combine_bwd<egc::StaticCfg"]},
    "bwd_colsum_fused": {"": ["k_colsum_partials", "!k_colsum_stage1"]},
    "bwd_colsum_two_stage": {"": ["k_colsum_stage1<false>*2", "k_colsum_stage2*2", "!k_colsum_partials"]},
    "bwd_route_atomic_hubs": {"": ["k_route_minmax", "!k_route_csc"]},
    "bwd_route_atomic_no_hub": {"": ["k_route_minmax", "!k_route_csc"]},
    "bwd_route_atomic_hubcap": {"": ["k_route_minmax", "!k_scatter"]},                  # min / max only: no pass 2
    "bwd_route_det_v4": {"": ["k_route_csc<4>", "!k_route_minmax"]},
    "bwd_route_det_v1": {"": ["k_route_csc<1>", "!k_route_minmax"]},
    "bwd_p2_ring": {"": ["k_scatter_ring<7, 4, float>"],
                    "EGC_BWD_RING=7": ["k_scatter_ring<7, 7, float>"],
                    "EGC_BWD_RING=0": ["k_scatter_cols<7, 32, true, float>", "!k_scatter_ring"],
                    "EGC_BWD_WARP_PER_COLUMN=1": ["k_scatter_bwd<7, 4, false>", "!k_scatter_ring"]},
    "bwd_p2_cols32": {"": ["k_scatter_cols<2, 32, false, float>"],
                      "EGC_BWD_WARP_PER_COLUMN=1": ["k_scatter_bwd<2, 4, false>", "!k_scatter_cols"]},
    "bwd_p2_cols16": {"": ["k_scatter_cols<7, 16, true, float>"]},
    "bwd_p2_ring_bf16": {"": ["k_scatter_ring<7, 8, __nv_bfloat16>"],
                         "EGC_BWD_RING=4": ["k_scatter_ring<7, 4, __nv_bfloat16>"],
                         "EGC_BWD_WARP_PER_COLUMN=1": ["k_scatter_ring<7, 8, __nv_bfloat16>"]},   # bf16 keeps its column blocks
    "bwd_p2_cols32_bf16": {"": ["k_scatter_cols<2, 32, false, __nv_bfloat16>"]},
    "bwd_p2_cols16_bf16": {"": ["k_scatter_cols<7, 16, true, __nv_bfloat16>"]},
    "bwd_p2_scatter_v1_linw": {"": ["k_combine_bwd<egc::DynCfg<0, 32>, 1, true, float>", "k_scatter_bwd<2, 1, true>"]},
    "bwd_p2_scatter_npass": {"": ["k_scatter_bwd<3, 4, false>*2"]},
})

# every branch of the dispatch in aggregate_api.cu -> the (switch setting, case) pairs that reach it.  A new branch is added
# here with its case; test_every_dispatch_branch_has_a_case checks the mapping against EXPECT.
_ROWS = "EGC_FWD_WARP_PER_ROW=1"
BRANCHES = {
    "fwd: row-block kernel, static cfg 0-5, with / without arg": [("", f"fwd_rows_static{i}{s}") for i in range(6)
                                                                  for s in ("", "_noarg") if f"fwd_rows_static{i}{s}" in CASES],
    "fwd: row-block kernel, dynamic G=32": [("", "fwd_rows_dyn_g32")],
    "fwd: row-block kernel, dynamic G=16": [("", "fwd_rows_dyn_g16")],
    "fwd: warp-per-row kernel, static cfg 0-5": [(_ROWS, f"fwd_rows_static{i}{s}") for i in range(6)
                                                 for s in ("", "_noarg") if f"fwd_rows_static{i}{s}" in CASES],
    "fwd: warp-per-row kernel, dynamic G=32": [("", "fwd_fast_dyn_g32"), (_ROWS, "fwd_rows_dyn_g32")],
    "fwd: warp-per-row kernel, dynamic G=16": [("", "fwd_fast_dyn_g16"), (_ROWS, "fwd_rows_dyn_g16")],
    "fwd: general kernel v4 + mode-1 merge": [("", "fwd_general_v4_npass"), ("", "fwd_general_v4_valued")],
    "fwd: general kernel v1 + mode-1 merge": [("", "fwd_general_v1_bd30"), ("", "fwd_general_v1_valued"),
                                              ("", "fwd_general_v1_offset_bases")],
    "fwd bf16: static cfg 0-5": [("", f"fwd_bf16_static{i}{s}") for i in range(6) for s in ("", "_noarg")
                                 if f"fwd_bf16_static{i}{s}" in CASES],
    "fwd bf16: dynamic g16": [("", "fwd_bf16_dyn_g16")],
    "fwd bf16: dynamic g8": [("", "fwd_bf16_dyn_g8")],
    "EGC_LAUNCH_COMBINE_CFG: StaticCfg x fp32 streams": [("", f"bwd_p1_static{i}") for i in range(6)],
    "EGC_LAUNCH_COMBINE_CFG: StaticCfg x bf16 streams": [("", f"bwd_p1_static{i}_bf16") for i in range(6)],
    "EGC_LAUNCH_COMBINE_CFG: DynCfg EV=4 bf16": [("", "bwd_p1_dyn_ev4_bf16")],
    "EGC_LAUNCH_COMBINE_CFG: DynCfg EV=1 bf16": [("", "bwd_p1_dyn_ev1_bf16")],
    "EGC_LAUNCH_COMBINE_CFG: DynCfg EV=4 fp32": [("", "bwd_p1_dyn_ev4"), ("", "bwd_p1_vec16_off")],
    "EGC_LAUNCH_COMBINE_CFG: DynCfg EV=4 per-entry weights": [("", "bwd_p1_dyn_ev4_linw")],
    "EGC_LAUNCH_COMBINE_CFG: DynCfg EV=1 fp32": [("", "bwd_p1_dyn_ev1")],
    "EGC_LAUNCH_COMBINE_CFG: DynCfg EV=1 per-entry weights": [("", "bwd_p2_scatter_v1_linw")],
    "pass 1: column sums fused": [("", "bwd_colsum_fused")],
    "pass 1: column sums two-stage": [("", "bwd_colsum_two_stage")],
    "route: atomic, hubs privatised": [("", "bwd_route_atomic_hubs")],
    "route: atomic, EGC_BWD_NO_HUB_PRIVATISATION": [("", "bwd_route_atomic_no_hub")],
    "route: atomic, more long columns than kRouteMaxHubs": [("", "bwd_route_atomic_hubcap")],
    "route: deterministic vec4": [("", "bwd_route_det_v4")],
    "route: deterministic vec1": [("", "bwd_route_det_v1")],
    "run_pass2: ring<4>": [("", "bwd_p2_ring")],
    "run_pass2: ring<7>": [("EGC_BWD_RING=7", "bwd_p2_ring")],
    "run_pass2: cols<32>": [("", "bwd_p2_cols32"), ("EGC_BWD_RING=0", "bwd_p2_ring")],
    "run_pass2: cols<16>": [("", "bwd_p2_cols16")],
    "run_pass2: ring<8, bf16>": [("", "bwd_p2_ring_bf16"), ("EGC_BWD_WARP_PER_COLUMN=1", "bwd_p2_ring_bf16")],
    "run_pass2: ring<4, bf16>": [("EGC_BWD_RING=4", "bwd_p2_ring_bf16")],
    "run_pass2: cols<32, bf16>": [("", "bwd_p2_cols32_bf16")],
    "run_pass2: cols<16, bf16>": [("", "bwd_p2_cols16_bf16")],
    "run_pass2: k_scatter vec4 (EGC_BWD_WARP_PER_COLUMN)": [("EGC_BWD_WARP_PER_COLUMN=1", "bwd_p2_ring"),
                                                           ("EGC_BWD_WARP_PER_COLUMN=1", "bwd_p2_cols32")],
    "run_pass2: k_scatter vec1, per-entry weights": [("", "bwd_p2_scatter_v1_linw")],
    "run_pass2: k_scatter n_pass > 1 + mode-1 merge": [("", "bwd_p2_scatter_npass")],
}


def _pattern(entry):
    """(regex, minimum launches, absent) of one EXPECT entry."""
    absent = entry.startswith("!")
    entry = entry.lstrip("!")
    count = 1
    if re.search(r"\*\d+$", entry):
        entry, count = entry.rsplit("*", 1)
        count = int(count)
    return re.compile(re.escape(entry).replace(re.escape("#"), r"\d+")), count, absent


def assert_kernels(case, setting, launched):
    for entry in EXPECT[case][setting]:
        rx, count, absent = _pattern(entry)
        n = sum(1 for k in launched if rx.search(k))
        hint = (f"{case} [{setting or 'default'}]: expected {entry!r} (EXPECT in tests/test_gpu_dispatch.py); "
                f"launched: {sorted(set(launched))}")
        assert (n == 0) if absent else (n >= count), hint


# ------------------------------------------------------------------------------------------------
# graphs, inputs, oracle
# ------------------------------------------------------------------------------------------------
def _edges(kind):
    """pattern: 1500 nodes, row degrees cycling through `degrees` (empty rows, rows of 256 / 257 / 300 / 600 entries), four
    long columns (sources 0-3: 257 to 900 entries) and 8 sources without entries.  hubcap: 1100 sources with 270 entries
    each (more long columns than the per-CTA hub table of the min/max routing holds), 100 empty columns, 50 empty rows."""
    gen = torch.Generator().manual_seed(7 if kind == "pattern" else 8)
    src, dst = [], []
    if kind == "pattern":
        n, degrees, hubs = 1500, [3, 0, 17, 1, 300, 12, 7, 0, 257, 2, 40, 0, 5, 256, 9, 30, 600, 1], [300, 520, 900, 257]
        for i in range(n):
            d = degrees[i % len(degrees)]
            if d:
                src.append(torch.randperm(n - 8, generator=gen)[:d])
                dst.append(torch.full((d,), i, dtype=torch.long))
    else:
        n, hubs = 1200, [270] * 1100
    hi = n if kind == "pattern" else n - 50                 # hubcap: the last 50 rows stay empty
    for j, d in enumerate(hubs):
        dst.append(torch.randperm(hi, generator=gen)[:d])
        src.append(torch.full((d,), j, dtype=torch.long))
    return n, torch.stack([torch.cat(src), torch.cat(dst)])


_GRAPHS = {}


def _graph(kind, symnorm, valued):
    """(device GraphStructure, OracleGraph over the device's own CSR and weights).  No self-loops are added."""
    key = (kind, symnorm, valued)
    if key not in _GRAPHS:
        n, ei = _edges(kind)
        if valued:
            rowptr, col, _ = to_adj_csr(ei, n)
            val = torch.randint(1, 5, (col.numel(),), generator=torch.Generator().manual_seed(9)).float() / 2   # dyadic
            g = egc_b200.GraphStructure.from_csr(rowptr.to(DEV), col.to(DEV), val.to(DEV), n, False, False)
        else:
            g = egc_b200.GraphStructure.from_edge_index(ei.to(DEV), n, symnorm, False)
        og = R.OracleGraph(g.rowptr.cpu().long(), g.col.cpu().long(), g.n_dst, g.n_src,
                           val_sym=g.val_sym.cpu() if g.val_sym is not None else None,
                           val_lin=g.val_lin.cpu() if g.val_lin is not None else None)
        deg = og.rowptr[1:] - og.rowptr[:-1]
        cdeg = torch.bincount(og.col, minlength=n)
        chunk = _lib.EGC_CHUNK_EDGES
        assert (deg == 0).any() and (deg > chunk).any() and (cdeg == 0).any() and (cdeg > chunk).any()
        _GRAPHS[key] = (g, og)
    return _GRAPHS[key]


def _offset(t):
    """`t` copied to a view that starts 4 bytes into an allocation one row larger (not 16-byte aligned)."""
    buf = torch.empty((t.shape[0] + 1) * t.shape[1], dtype=t.dtype, device=DEV)
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4
    return v


def _oracle(og, bases, w, bias, aggrs, heads, go, dtype):
    """R.aggregate + R.combine in `dtype` from the given leaves; with `go`: d_bases, d_weightings, d_bias."""
    grad = go is not None
    b, ww, bb = (t.to(dtype).requires_grad_(grad) for t in (bases, w, bias))
    with torch.set_grad_enabled(grad):
        agg, args = R.aggregate(og, b, aggrs)
        out = R.combine(ww, agg, bb, heads)
    res = {"out": out.detach(), "args": args}
    if grad:
        res["d_bases"], res["d_weightings"], res["d_bias"] = torch.autograd.grad(out, [b, ww, bb], go.to(dtype))
        res["d_lin_colsum"] = res["d_weightings"].sum(0)
    return res


def _src_ids(col, pos):
    nnz = col.numel()
    return torch.where((pos >= 0) & (pos < nnz), col[pos.clamp(0, nnz - 1)], torch.full_like(pos, -1))


def _traced(fn, trace=None):
    """fn()'s result and the demangled names of the CUDA kernels it launched (torch.profiler).  With `trace` (a path) the
    profile is also exported there as a chrome trace, whose kernel events carry the launch's grid and shared memory."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    if trace is not None:
        prof.export_chrome_trace(str(trace))
    return res, [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def _close(what, got, r64, r32):
    bar = max(TOL, 4 * rel_err(r32, r64))
    err = rel_err(got, r64)
    assert err < bar, f"{what}: relative error {err:.3e} >= bar {bar:.3e}"


def run_case(name, setting=""):
    c = CASES[name]
    g, og = _graph(c.graph, "symnorm" in c.aggrs, c.valued)
    n, bd, hd, hab = g.n_dst, c.bases * c.dim, c.heads * c.dim, c.heads * len(c.aggrs) * c.bases
    gen = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    bases = torch.round(torch.randn(n, bd, generator=gen) * 4) / 4                       # dyadic: exact in fp32 and bf16
    bases = bases.clamp(-15.75, 15.75)
    w = torch.randn(n, hab, generator=gen) * 0.5
    bias = torch.randn(hd, generator=gen)
    go = torch.randn(n, hd, generator=gen)
    desc = make_desc(g, c.heads, c.bases, c.dim, list(c.aggrs), False)
    bases_d = bases.to(DEV, torch.bfloat16 if c.bf16 else torch.float32)
    if c.offset == "bases":
        bases_d = _offset(bases_d)
    w_d, bias_d, go_d = w.to(DEV), bias.to(DEV), go.to(DEV)
    if c.offset == "grad_out":
        go_d = _offset(go_d)
    want = c.arg or c.stage == "bwd"
    (out, _, arg, saved, saved_arg), fwd_kernels = _traced(
        lambda: aggregate_combine(desc, g, bases_d, w_d, bias_d, want_arg=want, want_saved=want))
    grad = c.stage == "bwd"
    o64 = _oracle(og, bases, w, bias, c.aggrs, c.heads, go if grad else None, torch.float64)
    o32 = _oracle(og, bases, w, bias, c.aggrs, c.heads, go if grad else None, torch.float32)
    _close(f"{name}: out", out, o64["out"], o32["out"])
    if want:
        for a in ("max", "min"):
            if a in c.aggrs:
                k = c.aggrs.index(a)
                assert torch.equal(g.source_ids(arg[:, k]).cpu(), _src_ids(og.col, o64["args"][a])), f"{name}: {a} winners"
    if not grad:
        assert_kernels(name, setting, fwd_kernels)
        return
    (d_w, d_bases, d_bias, d_lin), bwd_kernels = _traced(
        lambda: aggregate_backward(desc, g, bases_d, w_d, saved, saved_arg, go_d, True, c.flags, want_lin_colsum=True))
    assert_kernels(name, setting, bwd_kernels)
    _close(f"{name}: d_weightings", d_w, o64["d_weightings"], o32["d_weightings"])
    _close(f"{name}: d_bias", d_bias, o64["d_bias"], o32["d_bias"])
    _close(f"{name}: d_lin_colsum", d_lin, o64["d_lin_colsum"], o32["d_lin_colsum"])
    if not c.bf16:
        _close(f"{name}: d_bases", d_bases, o64["d_bases"], o32["d_bases"])
        return
    # bf16 streams: each stored value is rounded once (relative error <= 2^-9), so |error| <= 2^-8 x the column pass over
    # the magnitudes of the stream terms + the fp32 rule (the derivation of tests/test_gpu_bf16.py)
    from tests.test_gpu_bf16 import _layer_from_bases
    ref = _layer_from_bases(og, bases.double(), w.double(), bias.double(), list(c.aggrs), c.heads, go.double())
    bound = 2.0 ** -8 * ref["d_bases_mag"] + TOL * ref["d_bases"].abs().max()
    excess = (d_bases.cpu().double() - ref["d_bases"]).abs() - bound
    assert (excess <= 0).all(), f"{name}: d_bases exceeds the bf16 bound by up to {excess.max().item():.3e}"


def _settings():
    return sorted({s for e in EXPECT.values() for s in e if s})


def run_setting(setting):
    """Every case whose expectation depends on `setting` (run in a process started with that switch)."""
    for name in sorted(k for k, e in EXPECT.items() if setting in e):
        run_case(name, setting)


# ------------------------------------------------------------------------------------------------
# tests
# ------------------------------------------------------------------------------------------------
def test_every_dispatch_branch_has_a_case():
    assert set(EXPECT) == set(CASES), set(EXPECT) ^ set(CASES)
    reached = set()
    for branch, pairs in BRANCHES.items():
        assert pairs, f"dispatch branch without a case: {branch}"
        for setting, case in pairs:
            assert case in EXPECT and setting in EXPECT[case], f"{branch}: no expectation for {case} [{setting}]"
            reached.add((setting, case))
    every = {(s, k) for k, e in EXPECT.items() for s in e}
    assert every == reached, f"expectations outside BRANCHES: {sorted(every - reached)}"
    for k, e in EXPECT.items():
        for entries in e.values():
            for entry in entries:
                _pattern(entry)


@gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_kernel_against_the_oracle(name):
    if any(s in os.environ for s in SWITCHES):
        pytest.skip("a dispatch switch is set in the environment: the default expectations do not apply")
    run_case(name)


@gpu
@pytest.mark.parametrize("setting", _settings())
def test_switch_in_a_fresh_process(setting):
    """The switches are read once per process: a fresh interpreter with only `setting` set runs the affected cases."""
    key, value = setting.split("=")
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env[key] = value
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_dispatch import run_setting; run_setting(%r); "
            "print('ok')" % (ROOT, setting))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-3000:] + r.stderr[-6000:]


# ------------------------------------------------------------------------------------------------
# fused epilogue on layers too wide for pass 1's column sums (H*A*B > 128): d_bias from the two-stage column sum over the
# masked, scaled gradient
# ------------------------------------------------------------------------------------------------
WIDE = dict(aggrs=["symnorm", "max", "std"], num_heads=8, num_bases=8)      # H*A*B = 192


@gpu
def test_wide_layer_fused_relu_equals_relu_after_the_layer():
    n = 3000
    ei = random_graph(n, 30000, seed=81, hub=600).to(DEV)
    torch.manual_seed(12)
    c = egc_b200.EGConv(64, 128, deterministic=True, **WIDE).to(DEV)
    with torch.no_grad():
        c.bias.uniform_(-0.5, 0.5)
    x, go = torch.randn(n, 64, device=DEV), torch.randn(n, 128, device=DEV)
    res = []
    for fused in (False, True):
        xc = x.clone().requires_grad_(True)
        y = c(xc, ei, relu=True) if fused else torch.relu(c(xc, ei))
        res.append([y] + list(torch.autograd.grad(y, [xc] + list(c.parameters()), go)))
    assert float((res[0][0] == 0).float().mean()) > 0.2
    for a, b in zip(*res):
        assert torch.equal(a, b)
    # the folded BatchNorm epilogue: scale multiplies the masked gradient
    scale, shift = torch.rand(128, device=DEV) + 0.5, torch.randn(128, device=DEV) * 0.1
    res = []
    for fused in (False, True):
        xc = x.clone().requires_grad_(True)
        y = c(xc, ei, relu=True, scale=scale, shift=shift) if fused else torch.relu(c(xc, ei) * scale + shift)
        res.append([y] + list(torch.autograd.grad(y, [xc] + list(c.parameters()), go)))
    for a, b in zip(*res):
        assert rel_err(a, b) < TOL


@gpu
@pytest.mark.parametrize("fused_dropout", [False, True])
def test_wide_egc_stack_trains_a_step(fused_dropout):
    """One training step of EGC(heads=8, bases=8, symnorm / max / std): the hidden layers carry the fused ReLU (and, with
    fused_dropout, the dropout) - equal to the composition of plain layers and torch ops."""
    from tests.dropout_model import dropout_constants, keep_mask
    n, p = 3000, 0.5
    ei = random_graph(n, 30000, seed=82, hub=600).to(DEV)
    torch.manual_seed(0)
    m = egc_b200.EGC(128, 3, p, 8, 8, WIDE["aggrs"], in_features=64, out_rounded=40, out_true=37,
                     fused_dropout=fused_dropout, deterministic=True).to(DEV).train()
    x, go = torch.randn(n, 64, device=DEV), torch.randn(n, 37, device=DEV)
    params = list(m.parameters())
    torch.manual_seed(123)
    out = m(x, ei)
    grads = torch.autograd.grad(out, params, go)
    torch.manual_seed(123)
    h = x
    for i, conv in enumerate(m.convs[:-1]):
        h = torch.relu(conv(h, ei))
        if fused_dropout:
            seed = int(m.last_dropout_seeds[i].item()) & 0xFFFFFFFFFFFFFFFF
            keep = torch.from_numpy(keep_mask(seed, 0, n, h.shape[1], p)).to(DEV)
            h = torch.where(keep, h * dropout_constants(p)[1], torch.zeros_like(h))
        else:
            h = F.dropout(h, p=p, training=True)
    ref = m.convs[-1](h, ei)[:, :37].log_softmax(dim=-1)
    grads_ref = torch.autograd.grad(ref, params, go)
    assert torch.equal(out, ref)
    for a, b in zip(grads, grads_ref):
        if fused_dropout:           # (g * k) masked vs g masked, then * k: the same products, summed in another order
            assert rel_err(a, b) <= TOL
        else:
            assert torch.equal(a, b)
