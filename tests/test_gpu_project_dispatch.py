"""Every projection and parameter-gradient kernel the dispatch of egc_project_fwd / _bf16 and egc_project_bwd can select,
checked against fp64, with the kernels that served each case - and the plan they ran with - asserted.

A case is a named (n, f_in, bd, hab, sigmoid, algo, storage, requested outputs, pointer offsets).  It runs the forward and
the backward through the C entry points, twice:

* Exact inputs.  x and the upstream gradients are integers in [-8, 8], the weights and the bias eighths in [-8, 8].  Every
  value is exact in TF32 (so the lo terms of the 3xTF32 split are zero), every product is exact in fp32, and the test
  asserts that sum |a| |b| over the contraction stays below 2^24 units (1/8 for the forward and d_x, 1 for the parameter
  gradients and d_b_comb) for every output element.  Then every partial sum, in any order, is exact: fp32 FFMA, TF32,
  3xTF32, every A feed and every split of the contraction must equal fp64 bit for bit - bases, pre-sigmoid weightings, d_x,
  dW_b, dW_c and d_b_comb.  With sigmoid the weightings get 2^-21 absolute (a few ulp of expf and the division); bf16
  storage must equal the round-to-nearest-even of the fp64 value.  A misplaced tile, a stale ring slot or a garbage pad
  fails with zero tolerance.
* Scaled normal inputs.  Rows and columns of x, of the weights and of the upstream gradients are scaled by 2^e, e in
  [-30, 30].  Each element is held to  |got - ref| <= gamma * (|A| |B|)_ij  (plus |b_comb| for the weightings), K = the
  contraction length (f_in, bd + hab, or n), u = 2^-24:
    FFMA     every product is exact before its fmaf rounding, the split-K slabs and their reduction add a few roundings on
             any path:  gamma = (K + 4) u.
    TF32     a operand is truncated to 10 explicit bits, |a - a_hi| < 2^-10 |a|:  |ab - a_hi b_hi| < 2^-9 |a||b|; the products
             are exact in fp32 and the tensor core's accumulation is allowed one ulp (2u, truncation) per addition:
             gamma = 2^-9 + (K + 4) 2u.
    3xTF32   ab ~ a_hi b_hi + a_hi b_lo + a_lo b_hi (project_tc.cu:6).  The MMA truncates the lo operands to TF32 again
             (|lo - tf32(lo)| < 2^-10 |lo| < 2^-20 |a|) and a_lo b_lo is missing (< 2^-20 |a||b|): three terms of 2^-20;
             3K products summed with one ulp per addition:  gamma = 3 * 2^-20 + 1.002 (3K + 4) 2u.
  With sigmoid the bound is multiplied by 1/4 (the largest slope) plus 2^-21; bf16 storage adds 2^-8 |ref|.  Unlike a
  bar normalised by max |ref|, this catches an error confined to small-magnitude rows.  Because the accumulation term of
  these bounds is loose, a 3xTF32 case is also run with TF32 on the same scaled inputs: the 3xTF32 error (normalised by
  |A||B|) must be at least 32x below the TF32 error, which a dropped lo term would not be.  The measured largest
  |got - ref| / (gamma |A||B|) is printed per case and output (run with -s).  On a B200 it stayed below 0.38 for every
  FFMA and 3xTF32 output (0.05-0.08 for the tcgen05 forward and d_x at f_in >= 100, up to 0.38 where K is tiny, n = 1);
  the TF32 (0.94) and bf16 (0.995) ratios come close to 1 because those bounds are tight: truncation to 10 bits and
  rounding to 8 significant bits are what they bound.

Which kernels served a case is read from torch.profiler and matched against EXPECT, the table of expected demangled names
(`name*N` = at least N launches, `!name` = not launched).  The plan is read from the profile's chrome trace: each kernel
event carries its grid and shared memory, which are compared launch by launch with `mirror`, a Python restatement of
tc_plan / launch_tc (project_tc.cu), wgrad_mn_part (wgrad_mn.cu), wgrad_tc (wgrad_tc.cu) and the FFMA fallbacks
(project.cu).  So a case asserts the n_split, ring depth and grid it claims.  On the B200 (torch 2.11, CUDA 12.8) the
trace's "shared memory" is the dynamic size for the tcgen05 kernels (they have no static shared memory) and the static
arrays for k_gemm_f32; the 1 KB per-block reservation is not included.  The plan is asserted from the default cases' traces;
a profile that misses launches (the library counts its own) is taken again.  torch.profiler on a B200 was seen to drop
more and more of a session's first launches after some forty sessions in one process, so the tests that need no
demangled names - the default reruns of the switch tests and the output subsets - count launches with the library's
own table (egc_profile_enable / egc_profile_collect) or not at all.

BRANCHES maps every branch of egc_project_fwd / _bf16 / _bwd, project_bwd_tc, launch_tc, wgrad_mn and the kernels' edges
(chunk tails, CTAs without a chunk, several TMEM flush segments, empty split-K slabs) to the (switch setting, case) pairs
that reach it; the CPU test checks each pair against the mirror.  Row counts that depend on the SM count are rules (_rows).

The switches are read once per process, so each runs in a fresh interpreter: EGC_TC_NO_TMA, EGC_TC_NO_SWIZZLE,
EGC_TC_TMA_STORE and EGC_TC_MAX_RAW_STAGES change only how k_project_tc moves data (same MMAs in the same order), so their
outputs must be bitwise equal to the default process's.  EGC_WGRAD_TRANSPOSE partitions the nodes differently and is held
to the oracle only.

Every output is a row-prefix of a NaN-filled buffer: each element must be written, and the guard rows after it must stay
bitwise unchanged."""
import json
import os
import subprocess
import sys
import zlib
from dataclasses import dataclass

import pytest
import torch

import egc_b200
from egc_b200 import _lib
from tests.test_gpu_dispatch import _pattern, _traced
from tests.util import random_graph, rel_err

gpu = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWITCHES = ("EGC_TC_NO_TMA", "EGC_TC_NO_SWIZZLE", "EGC_TC_TMA_STORE", "EGC_TC_MAX_RAW_STAGES", "EGC_WGRAD_TRANSPOSE")
AUTO, SIMT, X3, TF32 = _lib.GEMM_AUTO, _lib.GEMM_FP32_SIMT, _lib.GEMM_3XTF32, _lib.GEMM_TF32
OUTS = ("d_x", "d_w_bases", "d_w_comb", "d_b_comb")
GUARD = 3                                   # guard rows after every output
U = 2.0 ** -24


# ------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    n: object                 # rows: an int, or a rule of _rows (depends on the SM count)
    f_in: int
    bd: int
    hab: int
    sigmoid: bool = False
    algo: int = X3
    storage: str = "f32"      # "bf16": egc_project_fwd_bf16
    outs: tuple = OUTS        # requested outputs of the backward
    offset: tuple = ()        # of "x", "d_bases", "d_lin": starts 4 bytes into its allocation


def _rows(n, sms):
    """Row counts that reach an edge for any SM count."""
    if isinstance(n, int):
        return n
    return {
        "tiles3": 128 * 3 * sms + 77,       # >= 3 row tiles per k_project_tc CTA for every n_split: the TMEM double buffer wraps
        "zero_mn": 32 * (sms + 1),          # k_wgrad_mn: 2 chunks per CTA, the last CTAs get none
        "zero_tc": 16 * (sms + 1),          # k_wgrad_tc: the same with 16-node chunks
        "segs": 24 * 32 * sms + 5,          # 25 / 49 chunks per CTA: three TMEM flush segments in both kernels, a chunk tail
        "empty_slabs": 512 * sms + 1,       # FFMA split-K: 2 * SMs slabs of 272 nodes, the last ones get no node
    }[n]


MAG, ARXIV = (128, 64, 32), (128, 128, 48)
CASES = {
    # k_project_tc plans (3xTF32 forced) and k_wgrad_mn
    "mag_n1": Case(1, *MAG),
    "mag_n127": Case(127, *MAG),
    "mag_n128": Case(128, *MAG, sigmoid=True),
    "mag_n129": Case(129, *MAG),
    "mag_tiles3": Case("tiles3", *MAG),
    "arxiv_n129": Case(129, *ARXIV, sigmoid=True),
    "arxiv_tiles3": Case("tiles3", *ARXIV),
    "split3_tiles3": Case("tiles3", 352, 64, 32),                 # f_in > 128: parameter gradients on FFMA
    "split4": Case(1000, 256, 128, 48),                           # f_in > 128: parameter gradients on FFMA
    "ring6": Case(5000, 128, 256, 256),                           # 512 accumulator columns: parameter gradients on FFMA
    "dx_boxes": Case(3000, 100, 52, 32, sigmoid=True),            # d_x: 16-byte boxes, a chunk straddles d_bases | d_lin
    "pad": Case(2001, 20, 36, 48),                                # k_pad and n_pad
    "wide2": Case(5000, 128, 224, 64),                            # k_wgrad_mn in 2 launches
    "wide3": Case(999, 64, 200, 312),                             # k_wgrad_mn in 3 launches
    "tf32_mag": Case(3000, *MAG, algo=TF32),
    "auto_arxiv": Case(3000, *ARXIV, algo=AUTO),
    # bf16 basis rows
    "bf16_mag": Case(3000, *MAG, storage="bf16", sigmoid=True),
    "bf16_ffma64": Case(1000, 20, 36, 48, algo=SIMT, storage="bf16"),
    "bf16_ffma128": Case(1000, 128, 128, 48, algo=SIMT, storage="bf16"),
    # fp32 FFMA
    "ffma_small": Case(129, 20, 36, 48, algo=SIMT, sigmoid=True),
    "ffma_wide": Case(3000, *ARXIV, algo=SIMT),
    "ffma_empty_slabs": Case("empty_slabs", 20, 36, 48, algo=SIMT),
    "auto_unsupported_shape": Case(500, 30, 36, 48, algo=AUTO),   # f_in % 4 != 0: FFMA under AUTO
    # parameter-gradient edges (k_wgrad_mn by default, k_wgrad_tc under EGC_WGRAD_TRANSPOSE)
    **{f"wg_n{k}": Case(k, 20, 36, 48) for k in (15, 16, 17, 31, 32, 33)},
    "wg_zero_mn": Case("zero_mn", 20, 36, 48),
    "wg_zero_tc": Case("zero_tc", 20, 36, 48),
    "wg_segs": Case("segs", 20, 36, 48),
    # alignment: AUTO takes FFMA for the affected products
    "offset_all": Case(1000, *MAG, algo=AUTO, offset=("x", "d_bases", "d_lin")),
    "offset_x": Case(1000, *MAG, algo=AUTO, offset=("x",)),
}

_TC_SWITCHES = ("EGC_TC_NO_TMA=1", "EGC_TC_NO_SWIZZLE=1", "EGC_TC_TMA_STORE=1", "EGC_TC_MAX_RAW_STAGES=4",
                "EGC_TC_MAX_RAW_STAGES=5")
_TRANSPOSE = "EGC_WGRAD_TRANSPOSE=1"
_SWITCH_CASES = {
    "EGC_TC_NO_TMA=1": ("mag_n129", "arxiv_tiles3", "split3_tiles3", "dx_boxes", "pad", "bf16_mag"),
    "EGC_TC_NO_SWIZZLE=1": ("mag_n129", "arxiv_tiles3", "split4", "pad", "bf16_mag"),
    "EGC_TC_TMA_STORE=1": ("mag_tiles3", "arxiv_n129", "ring6", "split3_tiles3", "pad"),
    "EGC_TC_MAX_RAW_STAGES=4": ("mag_tiles3", "arxiv_tiles3", "split3_tiles3"),
    "EGC_TC_MAX_RAW_STAGES=5": ("mag_tiles3", "split4", "dx_boxes"),
    _TRANSPOSE: ("mag_n129", "wide2", "pad", "wg_n15", "wg_n16", "wg_n17", "wg_n31", "wg_n32", "wg_n33", "wg_zero_mn",
                 "wg_zero_tc", "wg_segs"),
}

# ------------------------------------------------------------------------------------------------
# EXPECT: case -> {switch setting ("" = none): [kernel, ...]}.  `#` stands for any number; `name*N` = at least N launches;
# `!name` = not launched.  The forward and the backward of a case are one list.
# ------------------------------------------------------------------------------------------------
TC, TCB, MN, WT, RED = "k_project_tc<false>", "k_project_tc<true>", "k_wgrad_mn", "k_wgrad_tc", "k_wgrad_reduce"
RS, CS = "k_reduce_splits", ["k_colsum_stage1<false>", "k_colsum_stage2"]


def G(bn, a, b, t="float"):
    return f"k_gemm_f32<{bn}, {str(a).lower()}, {str(b).lower()}, {t}>"


_TC_MN = [f"{TC}*2", MN, RED, *CS, "!k_gemm_f32", "!k_wgrad_tc"]              # forward + d_x on tcgen05, dW on k_wgrad_mn
_TC_FFMA_WG = [f"{TC}*2", G(128, False, True), f"{RS}*2", *CS, "!k_wgrad"]     # ... dW on FFMA (f_in > 128 or N > 256)
EXPECT = {
    **{k: {"": _TC_MN} for k in ("mag_n1", "mag_n127", "mag_n128", "mag_n129", "mag_tiles3", "arxiv_n129", "arxiv_tiles3",
                                 "dx_boxes", "pad", "tf32_mag", "auto_arxiv")},
    "split3_tiles3": {"": [f"{TC}*2", G(64, False, True), G(128, False, True), f"{RS}*2", *CS, "!k_wgrad"]},
    "split4": {"": _TC_FFMA_WG},
    "ring6": {"": _TC_FFMA_WG},
    "wide2": {"": [f"{TC}*2", f"{MN}*2", f"{RED}*2", *CS, "!k_gemm_f32"]},
    "wide3": {"": [f"{TC}*2", f"{MN}*3", f"{RED}*3", *CS, "!k_gemm_f32"]},
    "bf16_mag": {"": [TCB, TC, MN, RED, *CS, "!k_gemm_f32"]},
    "bf16_ffma64": {"": [G(64, True, True, "__nv_bfloat16"), G(64, True, False), G(64, True, False), G(64, True, True),
                         G(64, False, True), f"{RS}*2", *CS, "!k_project_tc", "!k_wgrad"]},
    "bf16_ffma128": {"": [G(128, True, True, "__nv_bfloat16"), G(64, True, False), G(128, True, False), G(128, True, True),
                          G(128, False, True), f"{RS}*2", *CS, "!k_project_tc", "!k_wgrad"]},
    "ffma_small": {"": [G(64, True, True), G(64, True, False), G(64, False, True), f"{RS}*2", *CS, "!k_project_tc",
                        "!k_wgrad"]},
    "ffma_wide": {"": [G(128, True, True), G(64, True, False), G(128, True, False), G(128, True, True),
                       G(128, False, True), f"{RS}*2", *CS, "!k_project_tc", "!k_wgrad"]},
    "ffma_empty_slabs": {"": [G(64, True, True), G(64, False, True), f"{RS}*2", *CS, "!k_project_tc", "!k_wgrad"]},
    "auto_unsupported_shape": {"": [G(64, True, True), G(64, False, True), f"{RS}*2", "!k_project_tc", "!k_wgrad"]},
    **{k: {"": _TC_MN} for k in ("wg_n15", "wg_n16", "wg_n17", "wg_n31", "wg_n32", "wg_n33", "wg_zero_mn", "wg_zero_tc",
                                 "wg_segs")},
    "offset_all": {"": [G(64, True, True), G(64, True, False), G(128, True, False), G(128, True, True),
                        G(64, False, True), G(128, False, True), f"{RS}*2", *CS, "!k_project_tc", "!k_wgrad"]},
    "offset_x": {"": [TC, G(64, True, True), G(64, True, False), G(64, False, True), G(128, False, True), f"{RS}*2", *CS,
                      "!k_wgrad"]},
}
for _s, _names in _SWITCH_CASES.items():
    for _k in _names:
        if _s != _TRANSPOSE:                                         # same kernels, other data movement
            EXPECT[_k][_s] = EXPECT[_k][""]
        elif _k == "wide2":                                          # 288 accumulator columns: k_wgrad_tc cannot, FFMA does
            EXPECT[_k][_s] = [f"{TC}*2", G(128, False, True), f"{RS}*2", "!k_wgrad"]
        else:
            EXPECT[_k][_s] = [f"{TC}*2", WT, RED, *CS, "!k_wgrad_mn", "!k_gemm_f32"]

# every branch -> the (switch setting, case) pairs that reach it (checked against `mirror` by the CPU test)
_P = [("", k) for k in CASES]
BRANCHES = {
    "fwd: k_project_tc<false>": [("", "mag_n129"), ("", "auto_arxiv"), ("", "tf32_mag")],
    "fwd: FFMA, algo FP32_SIMT": [("", "ffma_small"), ("", "ffma_wide")],
    "fwd: FFMA under AUTO, shape unsupported": [("", "auto_unsupported_shape")],
    "fwd: FFMA under AUTO, tensors unaligned": [("", "offset_all"), ("", "offset_x")],
    "fwd_bf16: k_project_tc<true>": [("", "bf16_mag")],
    "fwd_bf16: FFMA": [("", "bf16_ffma64"), ("", "bf16_ffma128")],
    "bwd: d_x on k_project_tc": [("", "dx_boxes"), ("", "offset_x")],
    "bwd: d_x FFMA, algo FP32_SIMT": [("", "ffma_wide")],
    "bwd: d_x FFMA under AUTO, shape unsupported": [("", "auto_unsupported_shape")],
    "project_bwd_tc: d_x FFMA, tensors unaligned": [("", "offset_all")],
    "project_bwd_tc: dW on k_wgrad_mn": [("", "mag_n129"), ("", "wg_segs")],
    "project_bwd_tc: dW on k_wgrad_tc": [(_TRANSPOSE, "mag_n129"), (_TRANSPOSE, "wg_segs")],
    "project_bwd_tc: dW on FFMA, shape": [("", "split3_tiles3"), ("", "ring6"), (_TRANSPOSE, "wide2")],
    "project_bwd_tc: dW on FFMA, tensors unaligned": [("", "offset_x")],
    "wgrad_mn: one launch": [("", "mag_n129")],
    "wgrad_mn: 2 launches": [("", "wide2")],
    "wgrad_mn: 3 launches": [("", "wide3")],
    "launch_tc: n_split 1": [("", "mag_tiles3")],
    "launch_tc: n_split 2": [("", "arxiv_tiles3"), ("EGC_TC_MAX_RAW_STAGES=4", "split3_tiles3")],
    "launch_tc: n_split 3": [("", "split3_tiles3")],
    "launch_tc: n_split 4": [("", "split4"), ("", "ring6")],
    "launch_tc: ring depth 4": [("EGC_TC_MAX_RAW_STAGES=4", "mag_tiles3")],
    "launch_tc: ring depth 5": [("EGC_TC_MAX_RAW_STAGES=5", "mag_tiles3")],
    "launch_tc: ring depth 6": [("", "ring6")],
    "launch_tc: ring depth >= 7": [("", "mag_tiles3")],
    "launch_tc: one 64-byte-swizzled box per chunk": [("", "mag_n129")],
    "launch_tc: four 16-byte boxes per chunk": [("", "dx_boxes"), ("EGC_TC_NO_SWIZZLE=1", "mag_n129")],
    "launch_tc: cp.async producers": [("EGC_TC_NO_TMA=1", "mag_n129"), ("EGC_TC_NO_TMA=1", "dx_boxes")],
    "launch_tc: TMA-store epilogue": [("EGC_TC_TMA_STORE=1", "mag_tiles3"), ("EGC_TC_TMA_STORE=1", "ring6")],
    "launch_tc: TMA store requested, columns not in blocks of 32": [("EGC_TC_TMA_STORE=1", "pad")],
    "k_project_tc: n = 1": [("", "mag_n1")],
    "k_project_tc: row tail": [("", "mag_n127"), ("", "mag_n129")],
    "k_project_tc: >= 3 tiles per CTA": [("", "mag_tiles3"), ("", "arxiv_tiles3"), ("", "split3_tiles3")],
    "k_project_tc: padded K and N": [("", "pad")],
    "k_wgrad_mn: chunk tail": [("", "wg_n15"), ("", "wg_n17"), ("", "wg_n31"), ("", "wg_n33")],
    "k_wgrad_mn: CTAs without a chunk": [("", "wg_zero_mn"), ("", "wg_segs")],
    "k_wgrad_mn: >= 2 flush segments": [("", "wg_segs")],
    "k_wgrad_tc: chunk tail": [(_TRANSPOSE, "wg_n15"), (_TRANSPOSE, "wg_n17"), (_TRANSPOSE, "wg_n31")],
    "k_wgrad_tc: CTAs without a chunk": [(_TRANSPOSE, "wg_zero_tc"), (_TRANSPOSE, "wg_segs")],
    "k_wgrad_tc: >= 2 flush segments": [(_TRANSPOSE, "wg_segs")],
    "k_gemm_f32: split-K slab without nodes": [("", "ffma_empty_slabs")],
    "kind::tf32 single pass": [("", "tf32_mag")],
    "every case": _P + [(s, k) for s, ks in _SWITCH_CASES.items() for k in ks],
}


# ------------------------------------------------------------------------------------------------
# mirror of the host-side planning
# ------------------------------------------------------------------------------------------------
def _cdiv(a, b):
    return -(-a // b)


def _r16(v):
    return _cdiv(v, 16) * 16


MAX_SMEM = 227 * 1024
CHUNK_BYTES = 128 * 16 * 4


def tc_plan(k, n, cap=None):
    """tc_plan (project_tc.cu): (n_split, cols_per_group, raw_stages, dynamic smem), or None."""
    k_pad = _r16(k)
    fixed = 4 * CHUNK_BYTES + 4 * 32 * 144 + (3 * 16 + 4 + 4) * 8 + 64
    best = None
    for s in range(1, 5):
        cpg = _r16(_cdiv(n, s))
        if cpg < 16 or cpg > 256:
            continue
        b = 2 * cpg * k_pad * 4
        if b + fixed + 2 * CHUNK_BYTES > MAX_SMEM:
            continue
        r = min(16, (MAX_SMEM - b - fixed) // CHUNK_BYTES)
        if cap is not None:
            r = max(4, min(r, cap))
        if best is None or r > best[2]:
            best = (s, cpg, r, b + fixed + r * CHUNK_BYTES)
        if r >= 8:
            break
    return best if best is not None and best[2] >= 4 else None


def tc_supported(n, f_in, bd, hab, cap=None):
    return (n >= 1 and f_in % 4 == 0 and bd % 4 == 0 and hab % 4 == 0 and tc_plan(f_in, bd + hab, cap) is not None
            and tc_plan(bd + hab, f_in, cap) is not None)


def _env(setting):
    if not setting:
        return {}
    k, v = setting.split("=")
    return {k: v}


def launch_tc(k1, k2, n1, n2, m, sms, env, bf16=False):
    """launch_tc (project_tc.cu): one k_project_tc launch and the branches it takes."""
    cap = int(env["EGC_TC_MAX_RAW_STAGES"]) if "EGC_TC_MAX_RAW_STAGES" in env else None
    s, cpg, r, smem = tc_plan(k1 + k2, n1 + n2, cap)
    tma = "EGC_TC_NO_TMA" not in env
    use_tma = 2 if tma and "EGC_TC_NO_SWIZZLE" not in env and (k2 == 0 or k1 % 16 == 0) else 1 if tma else 0
    want_store = not bf16 and "EGC_TC_TMA_STORE" in env
    store = want_store and n1 % 32 == 0 and cpg % 32 == 0 and (n2 == 0 or n2 % 4 == 0)
    tiles = _cdiv(m, 128)
    per_group = max(1, min(tiles, sms // s))
    labels = {f"launch_tc: n_split {s}", f"launch_tc: ring depth {r if r <= 6 else '>= 7'}",
              ["launch_tc: cp.async producers", "launch_tc: four 16-byte boxes per chunk",
               "launch_tc: one 64-byte-swizzled box per chunk"][use_tma]}
    if store:
        labels.add("launch_tc: TMA-store epilogue")
    elif want_store:
        labels.add("launch_tc: TMA store requested, columns not in blocks of 32")
    if m == 1:
        labels.add("k_project_tc: n = 1")
    if m % 128:
        labels.add("k_project_tc: row tail")
    if tiles >= 3 * per_group:
        labels.add("k_project_tc: >= 3 tiles per CTA")
    if (k1 + k2) % 16 or cpg % 16 or (n1 + n2) % cpg:
        labels.add("k_project_tc: padded K and N")
    launch = dict(kernel="k_project_tc<true>" if bf16 else "k_project_tc<false>", grid=(per_group * s, 1, 1), smem=smem,
                  n_split=s, raw_stages=r, use_tma=use_tma, tma_store=store)
    return [launch], labels


def gemm(m, n, k, splits, a_kcontig, b_ncontig, ct="float"):
    bn = 128 if n > 64 else 64
    smem = 4 * 16 * (128 + 4) + 4 * 16 * (bn + 4)
    return dict(kernel=G(bn, a_kcontig, b_ncontig, ct), grid=(_cdiv(n, bn), _cdiv(m, 128), splits), smem=smem, static=True)


def _slabs(n, sms):
    return max(1, min(2 * sms, _cdiv(n, 256)))


def simt_bwd(n, f_in, bd, hab, d_x, dwb, dwc, dbc, sms):
    """project_bwd_simt (project.cu)."""
    out, labels = [], set()
    if d_x:
        out += [gemm(n, f_in, bd, 1, True, False), gemm(n, f_in, hab, 1, True, True)]
    slabs = _slabs(n, sms)
    kps = _cdiv(_cdiv(n, slabs), 16) * 16
    for want, m, nn in ((dwb, f_in, bd), (dwc, hab, f_in)):
        if want:
            out += [gemm(m, nn, n, slabs, False, True), dict(kernel=RS, grid=(_cdiv(m * nn, 256), 1, 1), smem=None)]
            if (slabs - 1) * kps >= n:
                labels.add("k_gemm_f32: split-K slab without nodes")
    if dbc:
        cslabs = max(1, min(2 * sms, _cdiv(n, 64)))
        out += [dict(kernel=CS[0], grid=(cslabs, 1, 1), smem=None), dict(kernel=CS[1], grid=(_cdiv(hab, 8), 1, 1), smem=None)]
    return out, labels


def _mn_n_pad(bd, hab):
    return _r16(32 * _cdiv(bd, 32) + hab)


def _mn_stage(bd, hab):
    return 4 * 4096 + (_cdiv(bd, 32) + _cdiv(hab, 32)) * 4096


def _mn_raw(bd, hab):
    stage = _mn_stage(bd, hab)
    fixed = 2 * stage + (3 * 6 + 2 + 4) * 8 + 64 + 1024
    return 0 if fixed + 2 * stage > MAX_SMEM else min(6, (MAX_SMEM - fixed) // stage)


def _mn_first(bd, hab):
    return hab if _mn_n_pad(bd, hab) <= 256 else max(0, (256 - 32 * _cdiv(bd, 32)) // 32 * 32)


def mn_supported(n, f_in, bd, hab, env):
    if "EGC_WGRAD_TRANSPOSE" in env or n < 1 or f_in % 4 or bd % 4 or hab % 4 or f_in > 128 or hab < 1:
        return False
    first = _mn_first(bd, hab)
    if first < hab and (first < 32 or _mn_raw(0, min(hab - first, 256)) < 2):
        return False
    return _mn_raw(bd, first) >= 2


def _chunk_labels(kernel, n, chunk, seg_chunks, sms):
    total = _cdiv(n, chunk)
    grid = min(sms, total)
    per_cta = _cdiv(total, grid)
    labels = set()
    if n % chunk:
        labels.add(f"{kernel}: chunk tail")
    if (grid - 1) * per_cta >= total:
        labels.add(f"{kernel}: CTAs without a chunk")
    if per_cta > seg_chunks:
        labels.add(f"{kernel}: >= 2 flush segments")
    return grid, labels


def wgrad_mn(n, f_in, bd, hab, dwb, sms):
    first = _mn_first(bd, hab)
    parts = [(bd, first)] + [(0, min(256, hab - c0)) for c0 in range(first, hab, 256)]
    grid, labels = _chunk_labels("k_wgrad_mn", n, 32, 12, sms)
    out = []
    for n1, n2 in parts:
        smem = (_mn_raw(n1, n2) + 2) * _mn_stage(n1, n2) + (3 * 6 + 2 + 4) * 8 + 64 + 1024
        out += [dict(kernel=MN, grid=(grid, 1, 1), smem=smem),
                dict(kernel=RED, grid=(_cdiv(f_in * (n1 + n2), 32), 1, 1), smem=None)]
    labels.add({1: "wgrad_mn: one launch", 2: "wgrad_mn: 2 launches", 3: "wgrad_mn: 3 launches"}[len(parts)])
    return out, labels


def _wt_raw(n_pad, width):
    op = 2 * (128 * 16 * 4 + n_pad * 16 * 4)
    raw = 16 * width * 4
    fixed = 2 * op + (2 * 12 + 8) * 8 + 64
    return 0 if fixed + 2 * raw > MAX_SMEM else min(12, (MAX_SMEM - fixed) // raw)


def wt_supported(n, f_in, bd, hab):
    if n < 1 or f_in % 4 or bd % 4 or hab % 4 or f_in > 128:
        return False
    return _r16(bd + hab) <= 256 and _wt_raw(_r16(bd + hab), f_in + bd + hab) >= 2


def wgrad_tc(n, f_in, bd, hab, sms):
    n_pad, width = _r16(bd + hab), f_in + bd + hab
    raw = _wt_raw(n_pad, width)
    smem = 2 * 2 * (128 * 16 * 4 + n_pad * 16 * 4) + raw * 16 * width * 4 + (2 * 12 + 8) * 8 + 64
    grid, labels = _chunk_labels("k_wgrad_tc", n, 16, 24, sms)
    return [dict(kernel=WT, grid=(grid, 1, 1), smem=smem),
            dict(kernel=RED, grid=(_cdiv(f_in * (bd + hab), 32), 1, 1), smem=None)], labels


def mirror(c, setting, sms):
    """The launches (kernel, grid, shared memory) of a case's forward + backward, which product ran where, and the
    BRANCHES labels it reaches."""
    env = _env(setting)
    n, f_in, bd, hab = _rows(c.n, sms), c.f_in, c.bd, c.hab
    cap = int(env["EGC_TC_MAX_RAW_STAGES"]) if "EGC_TC_MAX_RAW_STAGES" in env else None
    bf16 = c.storage == "bf16"
    tc = c.algo != SIMT and tc_supported(n, f_in, bd, hab, cap)
    launches, labels, where = [], {"every case"}, {}
    if c.algo == TF32:
        labels.add("kind::tf32 single pass")
    fwd = "fwd_bf16" if bf16 else "fwd"
    # forward
    if tc and "x" not in c.offset:
        lo, lb = launch_tc(f_in, 0, bd, hab, n, sms, env, bf16)
        launches += lo
        labels |= lb | {f"{fwd}: k_project_tc<{str(bf16).lower()}>"}
        where["fwd"] = "tc"
    else:
        launches += [gemm(n, bd, f_in, 1, True, True, "__nv_bfloat16" if bf16 else "float"), gemm(n, hab, f_in, 1, True, False)]
        labels.add("fwd_bf16: FFMA" if bf16 else "fwd: FFMA, algo FP32_SIMT" if c.algo == SIMT else
                   "fwd: FFMA under AUTO, tensors unaligned" if tc else "fwd: FFMA under AUTO, shape unsupported")
        where["fwd"] = "ffma"
    # backward
    want = {o: o in c.outs for o in OUTS}
    if not tc:
        lo, lb = simt_bwd(n, f_in, bd, hab, want["d_x"], want["d_w_bases"], want["d_w_comb"], want["d_b_comb"], sms)
        launches += lo
        labels |= lb
        if want["d_x"]:
            labels.add("bwd: d_x FFMA, algo FP32_SIMT" if c.algo == SIMT else "bwd: d_x FFMA under AUTO, shape unsupported")
        where.update(d_x="ffma", dw="ffma")
        return launches, labels, where
    dx_simt = False
    if want["d_x"]:
        if "d_bases" in c.offset or "d_lin" in c.offset:
            dx_simt = True
            labels.add("project_bwd_tc: d_x FFMA, tensors unaligned")
            where["d_x"] = "ffma"
        else:
            lo, lb = launch_tc(bd, hab, f_in, 0, n, sms, env)
            launches += lo
            labels |= lb | {"bwd: d_x on k_project_tc"}
            where["d_x"] = "tc"
    dwb, dwc = want["d_w_bases"], want["d_w_comb"]
    wg_ok = (dwb or dwc) and not c.offset
    where["dw"] = "ffma"
    if wg_ok and mn_supported(n, f_in, bd, hab, env):
        lo, lb = wgrad_mn(n, f_in, bd, hab, dwb, sms)
        launches += lo
        labels |= lb | {"project_bwd_tc: dW on k_wgrad_mn"}
        dwb = dwc = False
        where["dw"] = "tc"
    elif wg_ok and wt_supported(n, f_in, bd, hab):
        lo, lb = wgrad_tc(n, f_in, bd, hab, sms)
        launches += lo
        labels |= lb | {"project_bwd_tc: dW on k_wgrad_tc"}
        dwb = dwc = False
        where["dw"] = "tc"
    elif wg_ok:
        labels.add("project_bwd_tc: dW on FFMA, shape")
    elif dwb or dwc:
        labels.add("project_bwd_tc: dW on FFMA, tensors unaligned")
    lo, lb = simt_bwd(n, f_in, bd, hab, dx_simt, dwb, dwc, want["d_b_comb"], sms)
    return launches + lo, labels | lb, where


# ------------------------------------------------------------------------------------------------
# inputs, oracle, bounds
# ------------------------------------------------------------------------------------------------
def _inputs(name, c, n, scaled):
    gen = torch.Generator().manual_seed(zlib.crc32(f"{name}:{scaled}".encode()))
    f_in, bd, hab = c.f_in, c.bd, c.hab
    if not scaled:
        def ints(*shape, hi=8):
            return torch.randint(-hi, hi + 1, shape, generator=gen).double()
        return dict(x=ints(n, f_in), wb=ints(f_in, bd, hi=64) / 8, wc=ints(hab, f_in, hi=64) / 8, bc=ints(hab, hi=64) / 8,
                    db=ints(n, bd), dl=ints(n, hab))

    def scaled(rows, cols):                                  # element (i, j) scaled by 2^(r_i + c_j), r, c in [-15, 15]
        e = torch.randint(-15, 16, (rows, 1), generator=gen) + torch.randint(-15, 16, (1, cols), generator=gen)
        return torch.randn(rows, cols, generator=gen, dtype=torch.float64) * torch.exp2(e.double())
    return dict(x=scaled(n, f_in), wb=scaled(f_in, bd), wc=scaled(hab, f_in), bc=scaled(1, hab)[0], db=scaled(n, bd),
                dl=scaled(n, hab))


def _fp32(t):
    return t.float().double()


def _oracle(inp):
    x, wb, wc, bc, db, dl = (_fp32(inp[k]) for k in ("x", "wb", "wc", "bc", "db", "dl"))
    ax, awb, awc, adb, adl = x.abs(), wb.abs(), wc.abs(), db.abs(), dl.abs()
    lin = x @ wc.t() + bc
    return {
        "bases": (x @ wb, ax @ awb, x.shape[1]),
        "lin": (lin, ax @ awc.t() + bc.abs(), x.shape[1] + 1),
        "d_x": (db @ wb.t() + dl @ wc, adb @ awb.t() + adl @ awc, wb.shape[1] + wc.shape[0]),
        "d_w_bases": (x.t() @ db, ax.t() @ adb, x.shape[0]),
        "d_w_comb": (dl.t() @ x, adl.t() @ ax, x.shape[0]),
        "d_b_comb": (dl.sum(0), adl.sum(0), x.shape[0]),
    }


def gamma(kind, n_terms, k):
    if kind == "ffma":
        return (k + 4) * U
    if n_terms == 1:
        return 2.0 ** -9 + (k + 4) * 2 * U
    return 3 * 2.0 ** -20 + 1.002 * (3 * k + 4) * 2 * U


def _offset_view(t):
    buf = torch.empty(t.numel() + 4, dtype=t.dtype, device=DEV)
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4
    return v


def _guarded(rows, *cols, dtype=torch.float32):
    """A NaN-filled buffer with GUARD rows after the first `rows`: (buffer, row-prefix view)."""
    buf = torch.full((rows + GUARD, *cols), float("nan"), dtype=dtype, device=DEV)
    return buf, buf[:rows]


def _guard_intact(what, buf, rows):
    g = buf[rows:]
    bits = g.view(torch.int16 if g.dtype == torch.bfloat16 else torch.int32)
    nan = torch.full_like(g, float("nan")).view(bits.dtype)
    assert torch.equal(bits, nan), f"{what}: a guard row after the output was written"


def _call(c, n, inp, algo, trace=None, record="profiler"):
    """Forward + backward through the C entry points (outputs in guarded NaN buffers); the second backward call's results
    must equal the first's bitwise.  Returns ({output: tensor}, launched kernels): record="profiler" gives the demangled
    names from torch.profiler (and the chrome trace at `trace`), "counters" the library's own launch table
    {LaunchScope name: launches}, None nothing."""
    lib = _lib.load()
    P, st = _lib.ptr, torch.cuda.current_stream().cuda_stream
    f_in, bd, hab = c.f_in, c.bd, c.hab
    dev = {k: v.float().to(DEV) for k, v in inp.items()}
    for k in c.offset:
        dev[{"x": "x", "d_bases": "db", "d_lin": "dl"}[k]] = _offset_view(dev[{"x": "x", "d_bases": "db", "d_lin": "dl"}[k]])
    bf16 = c.storage == "bf16"
    shapes = {"d_x": (n, f_in), "d_w_bases": (f_in, bd), "d_w_comb": (hab, f_in), "d_b_comb": (hab,)}
    nbytes = lib.egc_project_bwd_workspace_bytes(n, f_in, bd, hab)
    ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=DEV)

    def bwd_outs():
        return {o: _guarded(shapes[o][0], *shapes[o][1:]) for o in OUTS if o in c.outs}

    def run(bufs, outs):
        fn = lib.egc_project_fwd_bf16 if bf16 else lib.egc_project_fwd
        _lib.check(fn(P(dev["x"]), P(dev["wb"]), P(dev["wc"]), P(dev["bc"]), n, f_in, bd, hab, int(c.sigmoid),
                      P(bufs["bases"][1]), P(bufs["lin"][1]), algo, st), fn.__name__)
        _lib.check(lib.egc_project_bwd(P(dev["x"]), P(dev["wb"]), P(dev["wc"]), P(dev["db"]), P(dev["dl"]), n, f_in, bd, hab,
                                       *[P(outs[o][1]) if o in outs else None for o in OUTS], algo, P(ws), nbytes, st),
                   "egc_project_bwd")

    def fresh():
        return {"bases": _guarded(n, bd, dtype=torch.bfloat16 if bf16 else torch.float32), "lin": _guarded(n, hab)}, bwd_outs()

    if record == "profiler":
        for _ in range(3):         # the profiler can miss the first launches of a session: such a trace is taken again
            bufs, first = fresh()
            before = _lib.launch_count()
            _, names = _traced(lambda: run(bufs, first), trace)
            if sum("egc::" in k for k in names) == _lib.launch_count() - before:
                break
        assert sum("egc::" in k for k in names) == _lib.launch_count() - before, "the profile misses launches"
    elif record == "counters":
        bufs, first = fresh()
        _lib.profile_enable(True)
        try:
            run(bufs, first)
            names = {k: v[0] for k, v in _lib.profile_collect().items()}
        finally:
            _lib.profile_enable(False)
    else:
        bufs, first = fresh()
        run(bufs, first)
        names = None
    second = bwd_outs()
    _lib.check(lib.egc_project_bwd(P(dev["x"]), P(dev["wb"]), P(dev["wc"]), P(dev["db"]), P(dev["dl"]), n, f_in, bd, hab,
                                   *[P(second[o][1]) if o in second else None for o in OUTS], algo, P(ws), nbytes, st),
               "egc_project_bwd")
    torch.cuda.synchronize()
    res = {}
    for k, (buf, view) in {**bufs, **first}.items():
        _guard_intact(k, buf, view.shape[0])
        res[k] = view.cpu()
    for o in second:
        assert torch.equal(second[o][1].view(torch.int32), first[o][1].view(torch.int32)), f"{o}: two calls differ"
    return res, names


def _check_exact(name, c, res, ref):
    for k, got in res.items():
        want = ref[k][0]
        if k == "bases" and c.storage == "bf16":
            assert torch.equal(got.view(torch.int16), want.to(torch.bfloat16).view(torch.int16)), f"{name}: bf16 bases"
        elif k == "lin" and c.sigmoid:
            err = (got.double() - torch.sigmoid(want)).abs().max().item()
            assert err <= 2.0 ** -21, f"{name}: sigmoid weightings off by {err:.3e}"
        else:
            assert torch.equal(got.double(), want), \
                f"{name}: {k} differs from fp64 ({(got.double() - want).abs().max().item():.3e}, {(got.double() != want).sum()} elements)"


def _exact_bounds_hold(name, ref):
    for k, (_, mag, _) in ref.items():
        unit = 8 if k in ("bases", "lin", "d_x") else 1
        assert mag.max().item() * unit < 2 ** 24, f"{name}: the exact inputs of {k} exceed 2^24 units"


def _ratios(name, c, res, ref, where, algo):
    """max |got - ref| / (gamma |A||B|) per output, and max |got - ref| / |A||B| (the normalised error)."""
    n_terms = 1 if algo == TF32 else 3
    kinds = {"bases": where["fwd"], "lin": where["fwd"], "d_x": where.get("d_x", "ffma"), "d_w_bases": where["dw"],
             "d_w_comb": where["dw"], "d_b_comb": "ffma"}
    out = {}
    for k, got in res.items():
        want, mag, kk = ref[k]
        g = gamma(kinds[k], n_terms, kk)
        bound = g * mag
        if k == "lin" and c.sigmoid:
            want, bound = torch.sigmoid(want), 0.25 * bound + 2.0 ** -21
        elif k == "bases" and c.storage == "bf16":
            bound = bound * (1 + 2.0 ** -8) + 2.0 ** -8 * want.abs()
        err = (got.double() - want).abs()
        ratio = (err / bound.clamp_min(1e-300)).max().item()
        out[k] = (ratio, (err / mag.clamp_min(1e-300)).max().item(), kinds[k])
        assert ratio <= 1.0, f"{name}: {k} exceeds gamma |A||B| by {ratio:.3f}x (gamma {g:.3e}, {kinds[k]})"
    return out


def _kernel_events(trace):
    with open(trace) as f:
        ev = json.load(f)["traceEvents"]
    ks = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    return [(e["name"], tuple(e["args"]["grid"]), e["args"].get("shared memory")) for e in ks]


def assert_kernels(name, setting, launched):
    for entry in EXPECT[name][setting]:
        rx, count, absent = _pattern(entry)
        k = sum(1 for x in launched if rx.search(x))
        hint = (f"{name} [{setting or 'default'}]: expected {entry!r} (EXPECT in tests/test_gpu_project_dispatch.py); "
                f"launched: {sorted(set(launched))}")
        assert (k == 0) if absent else (k >= count), hint


def assert_plan(name, events, launches):
    got = [e for e in events if "egc::" in e[0]]
    assert len(got) == len(launches), f"{name}: launched {[e[0] for e in got]}, the mirror expects {[l['kernel'] for l in launches]}"
    for (kname, grid, smem), want in zip(got, launches):
        assert _pattern(want["kernel"])[0].search(kname), f"{name}: {kname} where the mirror expects {want['kernel']}"
        assert grid == want["grid"], f"{name}: {want['kernel']} grid {grid}, the mirror expects {want['grid']} ({want})"
        if want["smem"] is not None:
            assert smem == want["smem"], f"{name}: {want['kernel']} shared memory {smem}, the mirror expects {want['smem']}"


def _label(kernel):
    """The LaunchScope name under which the library counts a mirror kernel."""
    base = kernel.split("<")[0]
    return "k_wgrad_tc" if base == "k_wgrad_mn" else base


def run_case(name, setting="", tmp=None, c=None, record="profiler"):
    """One case: exact inputs (kernels, plan and fp64 bit-exactness), then scaled normal inputs (gamma bounds).  The
    kernels are checked against EXPECT and, with `tmp`, the plan against the mirror (record="profiler"), or the library's
    launch counts against the mirror's launches (record="counters"), or not at all (None).  Returns the outputs."""
    c = c or CASES[name]
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    n = _rows(c.n, sms)
    launches, _, where = mirror(c, setting, sms)
    exact_in = _inputs(name, c, n, False)
    ref = _oracle(exact_in)
    _exact_bounds_hold(name, ref)
    trace = os.path.join(tmp, f"{name}.json") if tmp is not None else None
    exact, names = _call(c, n, exact_in, c.algo, trace, record)
    if record == "profiler":
        assert_kernels(name, setting, names)
        if trace is not None:
            assert_plan(name, _kernel_events(trace), launches)
    elif record == "counters":
        want = {}
        for l in launches:
            want[_label(l["kernel"])] = want.get(_label(l["kernel"]), 0) + 1
        assert names == want, f"{name}: launched {names}, the mirror expects {want}"
    _check_exact(name, c, exact, ref)
    scaled_in = _inputs(name, c, n, True)
    ref = _oracle(scaled_in)
    scaled, _ = _call(c, n, scaled_in, c.algo, record=None)
    ratios = _ratios(name, c, scaled, ref, where, c.algo)
    if c.algo == X3 and any(r[2] == "tc" for r in ratios.values()):
        tf32, _ = _call(c, n, scaled_in, TF32, record=None)
        single = _ratios(name, c, tf32, ref, where, TF32)
        for k, (_, e3, kind) in ratios.items():
            rounded = (k == "bases" and c.storage == "bf16") or (k == "lin" and c.sigmoid)   # not the product's error
            if kind == "tc" and not rounded and single[k][1] > 0:
                assert e3 * 32 <= single[k][1], f"{name}: {k} 3xTF32 error {e3:.3e} is not 32x below TF32's {single[k][1]:.3e}"
    print(f"gamma ratio {name} [{setting or 'default'}] n={n}: " +
          ", ".join(f"{k} {r:.4f} ({kind})" for k, (r, _, kind) in ratios.items()))
    return {"exact": exact, "scaled": scaled}


def run_setting(setting, out_path, tmp):
    """The cases of `setting` in this process (started with that switch); their outputs go to out_path."""
    res = {name: run_case(name, setting, tmp) for name in _SWITCH_CASES[setting]}
    torch.save(res, out_path)


# ------------------------------------------------------------------------------------------------
# CPU tests
# ------------------------------------------------------------------------------------------------
SMS_CPU = 148


def test_every_dispatch_branch_has_a_case():
    assert set(EXPECT) == set(CASES), set(EXPECT) ^ set(CASES)
    reached, seen = set(), set()
    for branch, pairs in BRANCHES.items():
        assert pairs, f"dispatch branch without a case: {branch}"
        for setting, case in pairs:
            assert case in EXPECT and setting in EXPECT[case], f"{branch}: no expectation for {case} [{setting}]"
            assert branch in mirror(CASES[case], setting, SMS_CPU)[1], f"{branch}: {case} [{setting}] does not reach it"
            reached.add((setting, case))
    every = {(s, k) for k, e in EXPECT.items() for s in e}
    assert every == reached, f"expectations outside BRANCHES: {sorted(every - reached)}"
    for setting, case in every:
        seen |= mirror(CASES[case], setting, SMS_CPU)[1]
        launches = mirror(CASES[case], setting, SMS_CPU)[0]
        names = [l["kernel"] for l in launches]
        for entry in EXPECT[case][setting]:                  # the table and the mirror name the same kernels
            rx, count, absent = _pattern(entry)
            k = sum(1 for x in names if rx.search(x))
            assert (k == 0) if absent else (k >= count), f"{case} [{setting}]: {entry} vs the mirror's {names}"
    assert seen <= set(BRANCHES), f"branches the cases reach but BRANCHES does not list: {sorted(seen - set(BRANCHES))}"


# n_split and ring depth of the forward and of d_x, derived by hand from tc_plan
PLANS = {(128, 64, 32): ((1, 10), (1, 10)), (128, 128, 48): ((2, 10), (2, 11)), (352, 64, 32): ((3, 11), (3, 10)),
         (256, 128, 48): ((4, 10), (4, 11)), (128, 256, 256): ((4, 6), (4, 6)), (100, 52, 32): ((1, 11), (1, 11)),
         (128, 224, 64): ((3, 10), (3, 8)), (64, 200, 312): ((3, 11), (4, 14))}


def test_plan_mirror_claims():
    for (f_in, bd, hab), (fwd, dx) in PLANS.items():
        assert (tc_plan(f_in, bd + hab)[0], tc_plan(f_in, bd + hab)[2]) == fwd, (f_in, bd, hab)
        assert (tc_plan(bd + hab, f_in)[0], tc_plan(bd + hab, f_in)[2]) == dx, (f_in, bd, hab)
    # the ring cap keeps at least 4 stages and can move the column split; the split never leaves a group without columns
    assert tc_plan(352, 96, cap=4)[:3:2] == (2, 4)
    for k in range(4, 1025, 4):
        for nn in range(4, 1025, 12):
            p = tc_plan(k, nn)
            if p is not None:
                assert (p[0] - 1) * p[1] < nn, (k, nn, p)
    # the wide split of k_wgrad_mn: 2 and 3 launches, and the chunk edges of the row rules for any SM count
    assert len(wgrad_mn(5000, 128, 224, 64, True, 148)[0]) == 4 and len(wgrad_mn(999, 64, 200, 312, True, 148)[0]) == 6
    for sms in (132, 148, 160):
        assert {"k_wgrad_mn: CTAs without a chunk"} <= _chunk_labels("k_wgrad_mn", _rows("zero_mn", sms), 32, 12, sms)[1]
        assert {"k_wgrad_tc: CTAs without a chunk"} <= _chunk_labels("k_wgrad_tc", _rows("zero_tc", sms), 16, 24, sms)[1]
        assert {"k_wgrad_mn: >= 2 flush segments", "k_wgrad_mn: chunk tail"} <= \
            _chunk_labels("k_wgrad_mn", _rows("segs", sms), 32, 12, sms)[1]
        assert "k_wgrad_tc: >= 2 flush segments" in _chunk_labels("k_wgrad_tc", _rows("segs", sms), 16, 24, sms)[1]
        assert "k_gemm_f32: split-K slab without nodes" in simt_bwd(_rows("empty_slabs", sms), 20, 36, 48, 0, 1, 1, 0, sms)[1]
        for name in ("mag_tiles3", "arxiv_tiles3", "split3_tiles3"):
            assert "k_project_tc: >= 3 tiles per CTA" in mirror(CASES[name], "", sms)[1], (name, sms)


def test_exact_inputs_stay_below_2_to_the_24_units():
    for name in ("split3_tiles3", "wg_segs", "ffma_empty_slabs", "ring6"):
        c = CASES[name]
        _exact_bounds_hold(name, _oracle(_inputs(name, c, _rows(c.n, SMS_CPU), False)))


# ------------------------------------------------------------------------------------------------
# GPU tests
# ------------------------------------------------------------------------------------------------
def _no_switches():
    if any(s in os.environ for s in SWITCHES):
        pytest.skip("a projection switch is set in the environment: the default expectations do not apply")


@gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_case_against_the_oracle(name, tmp_path):
    _no_switches()
    run_case(name, "", str(tmp_path))


@gpu
@pytest.mark.parametrize("setting", sorted(_SWITCH_CASES))
def test_switch_in_a_fresh_process(setting, tmp_path):
    """The switches are read once per process: a fresh interpreter with only `setting` set runs the affected cases against
    the oracle; the k_project_tc switches must also reproduce this process's outputs bit for bit."""
    _no_switches()
    key, value = setting.split("=")
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env[key] = value
    out = tmp_path / "outputs.pt"
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_project_dispatch import run_setting; "
            "run_setting(%r, %r, %r); print('ok')" % (ROOT, setting, str(out), str(tmp_path)))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT, timeout=1800)
    print(r.stdout[-4000:])
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-3000:] + r.stderr[-6000:]
    if key == "EGC_WGRAD_TRANSPOSE":
        return
    theirs = torch.load(out)
    for name, res in theirs.items():
        mine = run_case(name, record=None)                    # the default process's outputs
        for kind in ("exact", "scaled"):
            for k, t in res[kind].items():
                bits = torch.int16 if t.dtype == torch.bfloat16 else torch.int32
                assert torch.equal(t.view(bits), mine[kind][k].view(bits)), f"{name} [{setting}]: {kind} {k} differs"


@gpu
@pytest.mark.parametrize("algo", [SIMT, X3])
def test_every_subset_of_backward_outputs(algo):
    """All 16 subsets of {d_x, d_w_bases, d_w_comb, d_b_comb}: as many launches of each kernel as the mirror names (the
    library's own launch table), every requested element written, nothing else.  (128, 224, 64) splits k_wgrad_mn over
    two launches, also with d_w_bases NULL."""
    _no_switches()
    for mask in range(16):
        outs = tuple(o for i, o in enumerate(OUTS) if mask >> i & 1)
        c = Case(700, 128, 224, 64, algo=algo, outs=outs)
        run_case(f"subset{mask}_{algo}", c=c, record="counters")


@gpu
def test_unaligned_tensors_under_a_forced_tensor_core_algorithm():
    """A forced tcgen05 algorithm does not fall back: EGC_ERR_UNSUPPORTED when x (forward) or d_bases / d_lin (d_x) are
    not 16-byte aligned."""
    _no_switches()
    lib = _lib.load()
    P, st = _lib.ptr, torch.cuda.current_stream().cuda_stream
    n, (f_in, bd, hab) = 1000, MAG
    x, wb, wc, bc = torch.randn(n, f_in, device=DEV), torch.randn(f_in, bd, device=DEV), torch.randn(hab, f_in, device=DEV), \
        torch.randn(hab, device=DEV)
    bases, lin = torch.empty(n, bd, device=DEV), torch.empty(n, hab, device=DEV)
    for algo in (X3, TF32):
        rc = lib.egc_project_fwd(P(_offset_view(x)), P(wb), P(wc), P(bc), n, f_in, bd, hab, 0, P(bases), P(lin), algo, st)
        assert rc == -3 and b"does not support" in lib.egc_last_error_string()
        rc = lib.egc_project_fwd_bf16(P(_offset_view(x)), P(wb), P(wc), P(bc), n, f_in, bd, hab, 0,
                                      P(bases.to(torch.bfloat16)), P(lin), algo, st)
        assert rc == -3 and b"does not support" in lib.egc_last_error_string()
        nbytes = lib.egc_project_bwd_workspace_bytes(n, f_in, bd, hab)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
        d_x = torch.empty(n, f_in, device=DEV)
        for db, dl in ((_offset_view(bases), lin), (bases, _offset_view(lin))):
            rc = lib.egc_project_bwd(P(x), P(wb), P(wc), P(db), P(dl), n, f_in, bd, hab, P(d_x), None, None, None, algo,
                                     P(ws), nbytes, st)
            assert rc == -3 and b"does not support" in lib.egc_last_error_string()


@gpu
def test_egconv_on_an_offset_x():
    """EGConv asks only for contiguous tensors: x viewed 4 bytes into its storage trains like an aligned copy."""
    _no_switches()
    n, f_in = 3000, 64
    ei = random_graph(n, 24000, seed=5).to(DEV)
    torch.manual_seed(3)
    conv = egc_b200.EGConv(f_in, 128, aggrs=["symnorm", "max"], num_heads=4, num_bases=4).to(DEV)
    x, go = torch.randn(n, f_in, device=DEV), torch.randn(n, 128, device=DEV)
    res = []
    for view in (lambda t: t.clone(), _offset_view):
        xv = view(x).requires_grad_(True)
        out = conv(xv, ei)
        res.append([out] + list(torch.autograd.grad(out, [xv] + list(conv.parameters()), go)))
    for a, b in zip(*res):
        assert rel_err(b, a.double()) < 1e-5


@gpu
def test_projection_on_two_devices_in_one_process():
    """The kernels' shared-memory attribute is set per device: one process projects on cuda:0, then on cuda:1."""
    _no_switches()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    c = CASES["mag_n129"]
    global DEV
    outs = []
    for d in ("cuda:0", "cuda:1"):
        DEV = d
        try:
            with torch.cuda.device(d):
                inp = _inputs("two_devices", c, 5000, False)
                res, _ = _call(c, 5000, inp, X3, record=None)
                _check_exact("two_devices " + d, c, res, _oracle(inp))
                outs.append(res)
        finally:
            DEV = "cuda:0"
