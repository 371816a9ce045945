"""Import the UNMODIFIED reference layers on CPU through the pure-torch shims.

TEST INFRASTRUCTURE ONLY - nothing under `egc_b200/` may import this module.

The reference's `experiments/optimized_layers.py` (EGConv) and
`experiments/layers.py` (EfficientGraphConv) depend on
torch_geometric / torch_scatter / torch_sparse, none of which is installable
offline.  `oracle/shims/` holds original pure-torch stand-ins for the leaf ops;
with them on `sys.path` the reference's own `forward`, `aggregate` and
`message_and_aggregate` run verbatim and autograd yields reference gradients.

The reference sources are not part of this repository.  They are looked for
in `oracle/_ref/` (a checkout of shyam196/egc, ignored by git) or in the
directory `EGC_REFERENCE_ROOT` names.  Without them `available()` is False and
parity rests on `oracle/restatement.py` and on `tests/golden/*.pt` (generated
from this loader by `oracle/make_golden*.py`).
"""
import importlib
import os
import sys
from types import SimpleNamespace

_ORACLE_DIR = os.path.dirname(os.path.abspath(__file__))
REFERENCE_ROOT = os.environ.get("EGC_REFERENCE_ROOT", os.path.join(_ORACLE_DIR, "_ref"))
_SHIMS = os.path.join(_ORACLE_DIR, "shims")
_cache = None


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "experiments", "optimized_layers.py"))


def _ensure_shims() -> None:
    if _SHIMS not in sys.path:
        sys.path.insert(0, _SHIMS)


def shims() -> SimpleNamespace:
    """The shim modules themselves (usable without the reference sources)."""
    _ensure_shims()
    return SimpleNamespace(
        torch_scatter=importlib.import_module("torch_scatter"),
        torch_sparse=importlib.import_module("torch_sparse"),
        torch_geometric=importlib.import_module("torch_geometric"),
        gcn_norm=importlib.import_module("torch_geometric.nn.conv.gcn_conv").gcn_norm,
        add_remaining_self_loops=importlib.import_module("torch_geometric.utils").add_remaining_self_loops,
        to_undirected=importlib.import_module("torch_geometric.utils").to_undirected,
        SparseTensor=importlib.import_module("torch_sparse").SparseTensor,
    )


def load() -> SimpleNamespace:
    """Returns the reference classes: EGConv, EfficientGraphConv, SparseTensor."""
    global _cache
    if _cache is not None:
        return _cache
    if not available():
        raise RuntimeError(f"reference sources not found under {REFERENCE_ROOT}")
    _ensure_shims()
    if REFERENCE_ROOT not in sys.path:
        sys.path.append(REFERENCE_ROOT)          # `experiments` is a namespace package there
    opt = importlib.import_module("experiments.optimized_layers")
    paper = importlib.import_module("experiments.layers")
    _cache = SimpleNamespace(
        EGConv=opt.EGConv,
        EfficientGraphConv=paper.EfficientGraphConv,
        SparseTensor=importlib.import_module("torch_sparse").SparseTensor,
        modules=(opt, paper),
    )
    return _cache
