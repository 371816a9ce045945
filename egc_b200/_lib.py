"""Builds (nvcc, sm_100a, in-tree) and loads `libegc_b200.so`, the C-ABI library declared in
`include/egc_b200.h`, through ctypes.  There is no fallback: if the library is missing or a call
fails, the caller gets an exception."""
import ctypes
import os
import subprocess
from ctypes import POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_size_t, c_void_p

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG_DIR)
LIB_PATH = os.path.join(_PKG_DIR, "libegc_b200.so")

ABI_VERSION = 5
EGC_MAX_AGGR = 8
EGC_CHUNK_EDGES = 256
MAX_PUSH_SEGMENTS = 64                     # EGC_MAX_PUSH_SEGMENTS: segments of one egc_peer_push_rows call
META_SLOTS = 8
META_NNZ, META_MAX_DEG, META_N_LONG, META_N_CHUNKS, META_N_LOOPS, META_ERRFLAGS = 0, 1, 2, 3, 4, 7
LOOPS_NONE, LOOPS_ALL_NODES, LOOPS_UP_TO_MAX_ID = 0, 1, 2
GEMM_AUTO, GEMM_FP32_SIMT, GEMM_3XTF32, GEMM_TF32 = 0, 1, 2, 3
BWD_DETERMINISTIC, BWD_SKIP_ROUTING, BWD_NO_HUB_PRIVATISATION = 1, 4, 8
BWD_COLS_HEAD, BWD_COLS_TAIL = 128, 256
BWD_PASS1_ONLY, BWD_ACCUMULATE = 512, 1024

POOL_CODES = {"sum": 0, "add": 0, "mean": 1, "max": 2}
AGGR_CODES = {"sum": 0, "mean": 1, "symnorm": 2, "min": 3, "max": 4, "var": 5, "std": 6}


class LayerDesc(Structure):
    """mirrors `egc_layer_desc`"""
    _fields_ = [("n_dst", c_int32), ("n_src", c_int32), ("heads", c_int32), ("bases", c_int32),
                ("dim", c_int32), ("n_aggr", c_int32), ("aggr", c_int32 * EGC_MAX_AGGR), ("sigmoid", c_int32),
                ("relu", c_int32)]


class Epilogue(Structure):
    """mirrors `egc_epilogue`"""
    _fields_ = [("scale", c_void_p), ("shift", c_void_p), ("add", c_void_p), ("agg_init", c_void_p)]


class Dropout(Structure):
    """mirrors `egc_dropout`"""
    _fields_ = [("seed", c_void_p), ("p", c_float), ("row_offset", c_int64)]


class RowPlan(Structure):
    """mirrors `egc_row_plan`"""
    _fields_ = [("n_long", c_int32), ("n_chunks", c_int32), ("long_rows", c_void_p),
                ("long_chunk_ptr", c_void_p), ("chunk_row", c_void_p), ("chunk_begin", c_void_p)]


# name -> (restype, argtypes); must list every symbol declared in include/egc_b200.h
_P = c_void_p
SIGNATURES = {
    "egc_abi_version": (c_int32, []),
    "egc_last_error_string": (c_char_p, []),
    "egc_build_info": (c_char_p, []),
    "egc_launch_count": (ctypes.c_uint64, []),
    "egc_profile_enable": (c_int32, [c_int32]),
    "egc_profile_collect": (c_int32, [ctypes.c_char_p, c_size_t]),
    "egc_csr_from_edges_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "egc_csr_from_edges": (c_int32, [_P, _P, c_int64, c_int32, c_int32, _P, _P, _P, _P, c_size_t, _P]),
    "egc_csr_fill_diag_workspace_bytes": (c_size_t, [c_int32]),
    "egc_csr_fill_diag": (c_int32, [_P, _P, _P, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P, c_size_t, _P]),
    "egc_symnorm_weights": (c_int32, [_P, _P, _P, c_int32, _P, _P, _P, _P]),
    "egc_csr_transpose_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "egc_csr_transpose": (c_int32, [_P, _P, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P, c_size_t, _P]),
    "egc_permute_f32": (c_int32, [_P, _P, c_int32, _P, _P]),
    "egc_plan_build": (c_int32, [_P, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P, c_size_t, _P]),
    "egc_plan_build_workspace_bytes": (c_size_t, [c_int32]),
    "egc_project_fwd": (c_int32, [_P, _P, _P, _P, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, c_int32, _P]),
    "egc_project_fwd_bf16": (c_int32, [_P, _P, _P, _P, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, c_int32, _P]),
    "egc_project_bwd_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "egc_project_bwd": (c_int32, [_P, _P, _P, _P, _P, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P,
                                  c_int32, _P, c_size_t, _P]),
    "egc_saved_slots": (c_int32, [POINTER(LayerDesc)]),
    "egc_saved_arg_slots": (c_int32, [POINTER(LayerDesc)]),
    "egc_aggregate_fwd_workspace_bytes": (c_size_t, [POINTER(LayerDesc), POINTER(RowPlan)]),
    "egc_aggregate_fwd": (c_int32, [POINTER(LayerDesc), _P, _P, _P, _P, POINTER(RowPlan), _P, _P, _P, POINTER(Epilogue), _P, c_int32,
                                    _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "egc_aggregate_fwd_bf16": (c_int32, [POINTER(LayerDesc), _P, _P, _P, POINTER(RowPlan), _P, _P, _P, POINTER(Epilogue),
                                         _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "egc_aggregate_fwd_dropout": (c_int32, [POINTER(LayerDesc), _P, _P, _P, _P, POINTER(RowPlan), _P, _P, _P, POINTER(Epilogue),
                                            POINTER(Dropout), _P, c_int32, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "egc_aggregate_fwd_bf16_dropout": (c_int32, [POINTER(LayerDesc), _P, _P, _P, POINTER(RowPlan), _P, _P, _P, POINTER(Epilogue),
                                                 POINTER(Dropout), _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "egc_aggregate_bwd_bf16_workspace_bytes": (c_size_t, [POINTER(LayerDesc), POINTER(RowPlan), c_int32]),
    "egc_aggregate_bwd_bf16": (c_int32, [POINTER(LayerDesc), _P, _P, _P, _P, _P, _P, POINTER(RowPlan), _P, _P, _P, _P, _P, _P, _P,
                                         _P, _P, _P, _P, c_int32, _P, c_size_t, _P]),
    "egc_aggregate_bwd_bf16_partitioned": (c_int32, [POINTER(LayerDesc), _P, _P, _P, _P, _P, _P, POINTER(RowPlan), _P, _P, _P, _P,
                                                     _P, _P, _P, _P, _P, _P, _P, _P, c_int32, c_int32, _P, c_size_t, _P]),
    "egc_aggregate_bwd_workspace_bytes": (c_size_t, [POINTER(LayerDesc), POINTER(RowPlan), c_int32]),
    "egc_aggregate_bwd": (c_int32, [POINTER(LayerDesc), _P, _P, _P, _P, _P, _P, _P, _P, POINTER(RowPlan), _P, _P, _P,
                                    _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int32, c_int32, _P, c_size_t, _P]),
    "egc_aggregate_bwd_cols_workspace_bytes": (c_size_t, [POINTER(LayerDesc), POINTER(RowPlan)]),
    "egc_aggregate_bwd_cols": (c_int32, [POINTER(LayerDesc), _P, _P, _P, _P, POINTER(RowPlan), _P, _P, _P, c_int32, _P, c_size_t, _P]),
    "egc_aggregate_bwd_cols_bf16": (c_int32, [POINTER(LayerDesc), _P, _P, _P, POINTER(RowPlan), _P, _P, _P, c_int32, _P,
                                              c_size_t, _P]),
    "egc_gather_rows": (c_int32, [_P, _P, c_int32, c_int32, _P, _P]),
    "egc_peer_alloc": (c_int32, [c_size_t, POINTER(c_void_p), _P]),
    "egc_peer_free": (c_int32, [_P]),
    "egc_peer_open": (c_int32, [_P, POINTER(c_void_p)]),
    "egc_peer_close": (c_int32, [_P]),
    "egc_peer_push_rows": (c_int32, [c_int32, _P, _P, _P, _P, c_int32, _P, c_int32, c_int32, ctypes.c_uint32, _P, _P, _P]),
    "egc_peer_copy": (c_int32, [_P, _P, c_size_t, _P]),
    "egc_peer_epoch_advance": (c_int32, [_P, _P]),
    "egc_peer_signal": (c_int32, [_P, c_int32, c_int32, ctypes.c_uint32, _P, _P]),
    "egc_peer_wait": (c_int32, [_P, c_int32, c_int32, c_int32, _P, ctypes.c_uint32, c_int32, ctypes.c_uint64, _P, _P]),
    "egc_peer_reduce_rows": (c_int32, [_P, _P, _P, _P, c_int32, c_int32, _P, _P]),
    "egc_peer_allreduce": (c_int32, [_P, _P, _P, _P, _P, c_int32, c_int32, c_int32, _P, _P, c_int32, _P, ctypes.c_uint64, _P, _P]),
    "egc_peer_sum_slots": (c_int32, [_P, c_int32, c_int32, _P, _P]),
    "egc_collate_edges": (c_int32, [_P, _P, _P, _P, c_int32, c_int64, c_int64, _P, _P, _P, _P, _P]),
    "egc_segment_ptr": (c_int32, [_P, c_int64, c_int32, _P, _P, _P]),
    "egc_segment_pool_fwd": (c_int32, [_P, _P, c_int32, c_int32, c_int32, _P, _P, _P]),
    "egc_segment_pool_bwd": (c_int32, [_P, _P, _P, c_int32, c_int32, c_int32, _P, _P]),
}

_lib = None


class EGCError(RuntimeError):
    """A libegc_b200 entry point returned a negative status."""


def build(verbose: bool = False, jobs: int = 0) -> str:
    """Compile every CUDA source for sm_100a into egc_b200/libegc_b200.so (nvcc cross-compiles
    without a GPU).  Returns the library path."""
    jobs = jobs or (os.cpu_count() or 4)
    proc = subprocess.run(["make", "-C", _ROOT, f"-j{jobs}"], capture_output=True, text=True)
    if verbose or proc.returncode != 0:
        print(proc.stdout[-4000:])
        print(proc.stderr[-8000:])
    if proc.returncode != 0:
        raise RuntimeError("building libegc_b200.so failed (see nvcc output above)")
    return LIB_PATH


def load() -> ctypes.CDLL:
    """Load the shared library (building is explicit: `egc_b200.build()` / `make`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `make -C {_ROOT} -j` or `python -c 'import egc_b200; "
            "egc_b200.build()'`.  egc_b200 has no Python/CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)     # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.egc_abi_version() != ABI_VERSION:
        raise ImportError(f"libegc_b200 ABI {lib.egc_abi_version()} != {ABI_VERSION} expected by the Python host code")
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().egc_last_error_string().decode("utf-8", "replace")
        raise EGCError(f"{what or 'libegc_b200'} failed with status {status}: {msg}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else c_void_p(t.data_ptr())


def launch_count() -> int:
    """Kernels launched by libegc_b200 in this process so far."""
    return int(load().egc_launch_count())


def profile_enable(on: bool = True) -> None:
    check(load().egc_profile_enable(int(on)), "egc_profile_enable")


def profile_collect() -> dict:
    """{kernel name: (launches, total_ms)} since profile_enable(True); clears the table."""
    buf = ctypes.create_string_buffer(1 << 16)
    n = load().egc_profile_collect(buf, len(buf))
    if n < 0:
        check(n, "egc_profile_collect")
    out = {}
    for line in buf.raw[:n].decode().splitlines():
        name, cnt, ms = line.rsplit(",", 2)
        out[name] = (int(cnt), float(ms))
    return out
