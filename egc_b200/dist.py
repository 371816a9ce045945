"""Row-partitioned (multi-GPU) execution of the EGConv hot path.  The reference has no counterpart
(it is single-GPU, SURVEY.md 2.2); the contract is "same numbers as the single-GPU layer".

Scheme (one process per GPU, torch.distributed; NCCL over NVLink on the B200 box, gloo in CPU tests):
  * contiguous target-row ranges balanced by nnz; every rank owns x / bases / weightings / out rows of
    its range and the CSR rows of those targets;
  * column ids are remapped to a local "extended" space: [own rows | halo rows], halo = remote
    sources referenced by the local CSR rows, grouped by owner;
  * forward : local projection -> halo exchange of basis rows (point-to-point, only the rows each peer
              needs) overlapped with the aggregation of interior rows -> boundary rows;
  * backward: local passes produce d_bases for own AND halo sources; halo partial sums travel back to
              their owners (reverse exchange) and are added in fixed peer order (deterministic);
              parameter gradients are all-reduced.
              Layers without min / max and with ONE target-side stream (symnorm-only, sum / mean only: EGC-S) instead
              exchange that stream ("T exchange"): pass 1 -> the stream rows of my boundary targets go to the ranks
              whose source columns they touch (a forward-style halo exchange on the TRANSPOSED adjacency) -> pass 2
              over my OWN columns only, complete and in CSC order: no 1-entry halo columns, no partial-sum reduce.
`PartitionPlan` and `HaloExchange` are pure index / communication plumbing (any device, any backend);
`PartitionedGraph` + `partitioned_egconv` bind them to the CUDA kernels.  On the B200 box the data path does not
go through NCCL: `transport="peer"` moves halo rows, halo gradient partial sums and the replicated parameter
gradients with our own kernels over NVLink peer memory (`egc_b200/peer.py`, `csrc/peer.cu`).
"""
from dataclasses import dataclass, replace
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist
from torch import Tensor


def balanced_row_bounds(rowptr: Tensor, world_size: int) -> List[int]:
    """Split rows into `world_size` contiguous ranges with (nearly) equal nnz + rows."""
    n = rowptr.numel() - 1
    work = rowptr[1:].double() + torch.arange(1, n + 1, dtype=torch.float64)     # cumulative nnz + rows
    total = float(work[-1]) if n > 0 else 0.0
    bounds = [0]
    for p in range(1, world_size):
        target = total * p / world_size
        b = int(torch.searchsorted(work, torch.tensor(target, dtype=torch.float64)))
        # every rank owns at least one row whenever there are enough rows (a hub row can outweigh a whole share)
        b = min(max(b, bounds[-1] + 1), n - (world_size - p)) if n >= world_size else min(max(b, bounds[-1]), n)
        bounds.append(b)
    bounds.append(n)
    return bounds


def transpose_csr(rowptr: Tensor, col: Tensor, *values: Optional[Tensor]):
    """Host-side transpose of a square CSR: (rowptr_t, col_t, *values_t), entries of a row of the transpose ascending by
    their original row (stable)."""
    rowptr, col = rowptr.long().cpu(), col.long().cpu()
    n = rowptr.numel() - 1
    row = torch.repeat_interleave(torch.arange(n), rowptr[1:] - rowptr[:-1])
    order = torch.argsort(col, stable=True)
    rowptr_t = torch.zeros(n + 1, dtype=torch.long)
    rowptr_t[1:] = torch.cumsum(torch.bincount(col, minlength=n), 0)
    return (rowptr_t, row[order]) + tuple(v.cpu()[order] if v is not None else None for v in values)


@dataclass
class LocalPartition:
    """What one rank needs (all index tensors int64 on CPU until `.to(device)`).  The column space is [own source rows
    col_begin..col_end | halo rows]; a square graph owns the same range of rows and columns.  The per-type halo tables of
    a `HeteroPartitionPlan` are LocalPartitions without a CSR (rowptr / col / interior / boundary rows are None)."""
    rank: int
    world_size: int
    row_begin: int
    row_end: int
    rowptr: Tensor              # [n_local + 1] local CSR over own target rows
    col: Tensor                 # [nnz_local] column ids in the extended local space
    val_sym: Optional[Tensor]
    val_lin: Optional[Tensor]
    halo_ids: Tensor            # [n_halo] global ids of halo sources, grouped by owner, ascending
    recv_counts: List[int]      # rows received from each peer (sum = n_halo)
    send_rows: List[Tensor]     # per peer: LOCAL row ids whose basis rows that peer needs
    interior_rows: Tensor       # local rows whose sources are all local
    boundary_rows: Tensor       # local rows that touch at least one halo source
    col_begin: Optional[int] = None     # own source-column range (None: the row range)
    col_end: Optional[int] = None

    @property
    def n_local(self) -> int:
        return self.row_end - self.row_begin

    @property
    def n_own_cols(self) -> int:
        return self.n_local if self.col_begin is None else self.col_end - self.col_begin

    def split_by_column(self):
        """The local CSR cut by column locality: (entries whose column is an OWN row, entries whose column is a HALO row),
        each as (rowptr, col, val_sym, val_lin) over the same rows and the same [own | halo] column space.  A sum over a
        row = the sum over the first part (computable while the halo rows are still in flight) + the sum over the second."""
        n = self.n_local
        rows = torch.repeat_interleave(torch.arange(n), self.rowptr[1:] - self.rowptr[:-1])
        is_own = self.col < self.n_own_cols
        parts = []
        for m in (is_own, ~is_own):
            rowptr = torch.zeros(n + 1, dtype=torch.long)
            rowptr[1:] = torch.cumsum(torch.bincount(rows[m], minlength=n), 0)
            parts.append((rowptr, self.col[m], self.val_sym[m] if self.val_sym is not None else None,
                          self.val_lin[m] if self.val_lin is not None else None))
        return parts

    @property
    def n_halo(self) -> int:
        return int(self.halo_ids.numel())


class PartitionPlan:
    """Host-side partition of a prepared global CSR (after self-loops / gcn_norm), so that symnorm
    weights and nnz counts are the GLOBAL ones on every rank.  `col_bounds`: owner ranges of the source columns of a
    rectangular CSR (one relation of a heterogeneous graph: rows = target type, columns = source type); by default the
    columns are owned like the rows."""

    def __init__(self, rowptr: Tensor, col: Tensor, world_size: int, val_sym: Optional[Tensor] = None,
                 val_lin: Optional[Tensor] = None, bounds: Optional[List[int]] = None,
                 col_bounds: Optional[List[int]] = None):
        self.rowptr, self.col = rowptr.long().cpu(), col.long().cpu()
        self.val_sym = val_sym.cpu() if val_sym is not None else None
        self.val_lin = val_lin.cpu() if val_lin is not None else None
        self.world_size = world_size
        self.n = self.rowptr.numel() - 1
        if self.n < world_size:
            raise ValueError(f"cannot partition {self.n} rows over {world_size} ranks: every rank needs at least one row")
        self.bounds = bounds or balanced_row_bounds(self.rowptr, world_size)
        self.col_bounds = list(col_bounds) if col_bounds is not None else self.bounds
        if len(self.bounds) != world_size + 1 or len(self.col_bounds) != world_size + 1:
            raise ValueError(f"row / column bounds need {world_size + 1} entries")
        self._bounds_t = torch.tensor(self.col_bounds, dtype=torch.long)
        self._needs = [self._needed_remote(r) for r in range(world_size)]      # [rank][owner] -> ids

    def owner_of(self, ids: Tensor) -> Tensor:
        """Rank that owns each source column id."""
        return torch.searchsorted(self._bounds_t, ids, right=True) - 1

    def transposed(self) -> "PartitionPlan":
        """The same node ranges over the TRANSPOSED adjacency: rank p's rows are its own SOURCE columns, its halo the
        remote TARGETS that aggregate them - what the backward's T exchange needs (see the module docstring)."""
        if (int(self.col.max()) >= self.n if self.col.numel() else False) or self.col_bounds != self.bounds:
            raise ValueError("the transposed plan needs a square adjacency")
        rowptr_t, col_t, sym_t, lin_t = transpose_csr(self.rowptr, self.col, self.val_sym, self.val_lin)
        return PartitionPlan(rowptr_t, col_t, self.world_size, val_sym=sym_t, val_lin=lin_t, bounds=list(self.bounds))

    def _needed_remote(self, rank: int) -> List[Tensor]:
        b, e = self.bounds[rank], self.bounds[rank + 1]
        cb, ce = self.col_bounds[rank], self.col_bounds[rank + 1]
        cols = self.col[self.rowptr[b]:self.rowptr[e]]
        remote = torch.unique(cols[(cols < cb) | (cols >= ce)])
        owner = self.owner_of(remote)
        return [remote[owner == q] for q in range(self.world_size)]

    def local(self, rank: int) -> LocalPartition:
        b, e = self.bounds[rank], self.bounds[rank + 1]
        lo, hi = int(self.rowptr[b]), int(self.rowptr[e])
        rowptr = self.rowptr[b:e + 1] - lo
        cols = self.col[lo:hi]
        cb, ce = self.col_bounds[rank], self.col_bounds[rank + 1]
        halo_ids = torch.cat(self._needs[rank]) if self.world_size > 1 else cols.new_zeros(0)
        n_local = e - b
        is_local = (cols >= cb) & (cols < ce)
        col_ext = torch.where(is_local, cols - cb, (ce - cb) + torch.searchsorted(halo_ids, cols)
                              if halo_ids.numel() else cols - cb)
        # halo_ids is sorted globally because owners are contiguous ascending ranges
        rows = torch.repeat_interleave(torch.arange(n_local), rowptr[1:] - rowptr[:-1])
        touches = torch.zeros(n_local, dtype=torch.bool)
        touches[rows[~is_local]] = True
        send_rows = [self._needs[q][rank] - cb for q in range(self.world_size)]
        return LocalPartition(
            rank=rank, world_size=self.world_size, row_begin=b, row_end=e, rowptr=rowptr, col=col_ext,
            val_sym=self.val_sym[lo:hi] if self.val_sym is not None else None,
            val_lin=self.val_lin[lo:hi] if self.val_lin is not None else None,
            halo_ids=halo_ids, recv_counts=[int(t.numel()) for t in self._needs[rank]], send_rows=send_rows,
            interior_rows=torch.nonzero(~touches).flatten(), boundary_rows=torch.nonzero(touches).flatten(),
            col_begin=cb, col_end=ce)


@dataclass
class HeteroLocalPartition:
    """One rank's share of a heterogeneous graph: per node type the exchange table (own rows + the union halo of every
    relation that reads that type, a `LocalPartition` without CSR), per relation the local CSR over this rank's target
    rows whose column ids point into the [own | halo] table of its source type (halo fields = those of that table)."""
    tables: Dict[str, LocalPartition]
    relations: Dict[Tuple[str, str, str], LocalPartition]


class HeteroPartitionPlan:
    """Row partition of a heterogeneous graph {(src, rel, dst): (rowptr [n_dst + 1], col)} over node types `sizes`: every
    type gets its own contiguous row ranges, balanced by the rows + nnz of the relations that target it, so every rank
    owns rows of every type.  Each relation is a rectangular `PartitionPlan` (rows owned like its target type, columns
    like its source type); a rank's halo of type s is the union of the remote s ids its target rows reference in every
    relation (s, r, t), grouped by owner and ascending - ONE halo per source type, shared by all relations reading it."""

    def __init__(self, csr_dict, sizes: Dict[str, int], world_size: int, values=None):
        self.types, self.keys, self.world_size = list(sizes), list(csr_dict), world_size
        for t, n in sizes.items():
            if n < world_size:
                raise ValueError(f"cannot partition {n} rows of node type {t!r} over {world_size} ranks: every rank "
                                 "needs at least one row of every type")
        csr = {}
        for k, (rowptr, col) in csr_dict.items():
            if k[0] not in sizes or k[2] not in sizes:
                raise ValueError(f"relation {k} names a node type outside {self.types}")
            if rowptr.numel() != sizes[k[2]] + 1:
                raise ValueError(f"relation {k} has {rowptr.numel() - 1} rows, node type {k[2]!r} has {sizes[k[2]]}")
            csr[k] = (rowptr.long().cpu(), col.long().cpu())
        self.bounds = {}
        for t in self.types:
            rowptr = torch.zeros(sizes[t] + 1, dtype=torch.long)
            for k, (rp, _) in csr.items():
                if k[2] == t:
                    rowptr = rowptr + rp
            self.bounds[t] = balanced_row_bounds(rowptr, world_size)
        values = values or {}
        self.plans = {k: PartitionPlan(rp, col, world_size, val_lin=values.get(k), bounds=self.bounds[k[2]],
                                       col_bounds=self.bounds[k[0]]) for k, (rp, col) in csr.items()}

    def _type_needs(self, s: str, reader: int, owner: int) -> Tensor:
        """Ascending ids of type s owned by `owner` that `reader` reads, over every relation with source s."""
        parts = [p._needs[reader][owner] for k, p in self.plans.items() if k[0] == s]
        return torch.unique(torch.cat(parts)) if parts else torch.zeros(0, dtype=torch.long)

    def local(self, rank: int) -> HeteroLocalPartition:
        w = self.world_size
        tables = {}
        for s in self.types:
            cb, ce = self.bounds[s][rank], self.bounds[s][rank + 1]
            needs = [self._type_needs(s, rank, q) for q in range(w)]
            halo_ids = torch.cat(needs) if w > 1 else torch.zeros(0, dtype=torch.long)
            send_rows = [self._type_needs(s, q, rank) - cb for q in range(w)]
            tables[s] = LocalPartition(rank=rank, world_size=w, row_begin=cb, row_end=ce, rowptr=None, col=None,
                                       val_sym=None, val_lin=None, halo_ids=halo_ids,
                                       recv_counts=[int(t.numel()) for t in needs], send_rows=send_rows,
                                       interior_rows=None, boundary_rows=None, col_begin=cb, col_end=ce)
        relations = {}
        for k, plan in self.plans.items():
            lp, tab = plan.local(rank), tables[k[0]]
            n_own = tab.n_local
            is_halo = lp.col >= n_own                   # relation halo slot -> the same id's slot in the type's halo
            col = lp.col.clone()
            col[is_halo] = n_own + torch.searchsorted(tab.halo_ids, lp.halo_ids[lp.col[is_halo] - n_own])
            relations[k] = replace(lp, col=col, halo_ids=tab.halo_ids, recv_counts=tab.recv_counts,
                                   send_rows=tab.send_rows)
        return HeteroLocalPartition(tables, relations)


class HaloExchange:
    """Point-to-point exchange of feature rows between the ranks of a `PartitionPlan`.

    forward(local_rows [n_local, W]) -> halo rows [n_halo, W] (what the peers own and this rank needs)
    reverse(halo_partial [n_halo, W], into [n_local, W])  adds the peers' partial sums for rows this rank
    owns, in ascending peer order.  `gather` / `scatter_add` can be overridden with device kernels.
    """

    def __init__(self, part: LocalPartition, device, group=None):
        self.part, self.group, self.device = part, group, torch.device(device)
        self.send_rows = [t.to(self.device) for t in part.send_rows]
        self.recv_offsets = [0]
        for c in part.recv_counts:
            self.recv_offsets.append(self.recv_offsets[-1] + c)

    def _peers(self):
        r, w = self.part.rank, self.part.world_size
        return [(r + k) % w for k in range(1, w)]

    def start_forward(self, local_rows: Tensor):
        """Posts the sends/receives; returns (halo buffer, work handles).  Call `finish()` before use."""
        width = local_rows.size(1)
        halo = torch.empty((self.part.n_halo, width), dtype=local_rows.dtype, device=local_rows.device)
        ops, keep = [], []
        for q in self._peers():
            if self.part.recv_counts[q]:
                ops.append(dist.P2POp(dist.irecv, halo[self.recv_offsets[q]:self.recv_offsets[q + 1]], q, self.group))
            if self.send_rows[q].numel():
                buf = self.gather(local_rows, self.send_rows[q])
                keep.append(buf)
                ops.append(dist.P2POp(dist.isend, buf, q, self.group))
        works = dist.batch_isend_irecv(ops) if ops else []
        return halo, (works, keep)

    @staticmethod
    def finish(handle) -> None:
        works, _keep = handle
        for w in works:
            w.wait()

    def forward(self, local_rows: Tensor) -> Tensor:
        halo, handle = self.start_forward(local_rows)
        self.finish(handle)
        return halo

    def reverse(self, halo_partial: Tensor, into: Tensor) -> Tensor:
        width = halo_partial.size(1)
        ops, recv = [], {}
        for q in self._peers():
            if self.send_rows[q].numel():          # rows I own that q used: q sends me its partial sums
                recv[q] = torch.empty((self.send_rows[q].numel(), width), dtype=into.dtype, device=into.device)
                ops.append(dist.P2POp(dist.irecv, recv[q], q, self.group))
            if self.part.recv_counts[q]:
                seg = halo_partial[self.recv_offsets[q]:self.recv_offsets[q + 1]].contiguous()
                ops.append(dist.P2POp(dist.isend, seg, q, self.group))
        for w in (dist.batch_isend_irecv(ops) if ops else []):
            w.wait()
        for q in sorted(recv):                     # fixed order: deterministic sums
            self.scatter_add(into, self.send_rows[q], recv[q])
        return into

    # -- overridable data movers ------------------------------------------------------------
    def gather(self, rows: Tensor, index: Tensor) -> Tensor:
        return rows.index_select(0, index)

    def scatter_add(self, into: Tensor, index: Tensor, src: Tensor) -> None:
        into.index_add_(0, index, src)             # index is unique per peer: no intra-call conflicts


class CudaHaloExchange(HaloExchange):
    """HaloExchange whose packing runs through libegc_b200 (egc_gather_rows)."""

    def __init__(self, part: LocalPartition, device, group=None):
        super().__init__(part, device, group)
        self.send_rows32 = [t.to(torch.int32) for t in self.send_rows]

    def gather(self, rows: Tensor, index: Tensor) -> Tensor:
        from . import _lib
        from .graph import _stream
        q = next(i for i, t in enumerate(self.send_rows) if t is index)
        idx = self.send_rows32[q]
        out = torch.empty((idx.numel(), rows.size(1)), dtype=rows.dtype, device=rows.device)
        words = rows.size(1) * rows.element_size() // 4                # the kernel moves 4-byte words (bf16: B*D % 8 == 0)
        _lib.check(_lib.load().egc_gather_rows(_lib.ptr(rows), _lib.ptr(idx), idx.numel(), words, _lib.ptr(out),
                                               _stream()), "egc_gather_rows")
        return out


# ---------------------------------------------------------------------------------------------------
# CUDA binding
# ---------------------------------------------------------------------------------------------------
class PartitionedGraph:
    """Device-side state of one rank: the rectangular local CSR ([own rows] x [own | halo] columns), the
    interior / boundary row split and the halo exchange.

    transport = "peer" (default): our own kernels over NVLink peer memory (`egc_b200.peer`, csrc/peer.cu) - posted
    stores into the consumer's memory ordered by epoch flags, graph-capturable, no NCCL on the data path;
    transport = "nccl": point-to-point `batch_isend_irecv` + all-reduce (kept as the library baseline).

    storage_dtype=torch.bfloat16 declares that the exchanges of this graph may carry bf16 rows: layers built with
    `EGConv(..., storage_dtype=torch.bfloat16)` then run on it, their halo basis rows and T-exchange stream rows travel as
    bf16 (the halo partial sums stay fp32).  fp32 layers run on either kind of graph."""

    def __init__(self, part: LocalPartition, device, group=None, transport: str = "peer",
                 tpart: Optional[LocalPartition] = None, storage_dtype: torch.dtype = torch.float32):
        from .functional import check_storage_dtype
        from .graph import GraphStructure
        if transport not in ("peer", "nccl"):
            raise ValueError(f"unknown transport {transport!r}")
        self.storage_dtype = check_storage_dtype(storage_dtype)
        if storage_dtype == torch.bfloat16 and part.val_lin is not None:      # same on every rank; nothing collective yet
            raise ValueError("storage_dtype=torch.bfloat16 does not support an adjacency with edge values (without symnorm)")
        self.part = part
        self.tpart = tpart                         # local block of the TRANSPOSED adjacency (T exchange), or None
        self._graph_t = None
        self.exchange_t = CudaHaloExchange(tpart, torch.device(device), group) if tpart is not None else None
        self.device = torch.device(device)
        self.graph = GraphStructure.from_prepared(part.rowptr, part.col, part.n_local + part.n_halo,
                                                  val_sym=part.val_sym, val_lin=part.val_lin, device=self.device)
        self.transport = transport if part.world_size > 1 else "nccl"
        self.exchange = CudaHaloExchange(part, self.device, group)
        self.interior = part.interior_rows.to(self.device, torch.int32)
        self.boundary = part.boundary_rows.to(self.device, torch.int32)
        # Aggregating the interior rows while the halo rows are in flight only pays when there are enough of them:
        # a row subset runs slower than the contiguous whole-graph launch (per-row staging), and with ~15 nnz per
        # row and 20 % remote sources only a few rows are interior.  Below one half: wait, then ONE contiguous launch.
        self.overlap_interior = part.interior_rows.numel() * 2 >= max(part.n_local, 1)
        # backward: halo columns of pass 2 first, their push on a side stream while the own columns run.  Measured on
        # 2 x B200 (profiles/r02c): with a routed (min / max) aggregator the column phases cost more than they hide - the
        # routing has to come first, so d_bases is zeroed and pass 2 turns into a read-modify-write (0.91 vs 0.82 ms per
        # arxiv-shaped EGC-M step) - so "auto" splits only layers without min / max.  EGC_DIST_SPLIT_BWD=0|1 forces it.
        import os
        self.split_backward = os.environ.get("EGC_DIST_SPLIT_BWD", "auto")
        # backward by T exchange (module docstring): "auto" = layers without min / max whose backward has ONE target-side
        # stream - the exchanged rows are then as wide as the partial sums they replace; EGC_DIST_T_EXCHANGE=0|1 forces it
        # (1: every layer without min / max, whatever its stream count)
        self.t_exchange = os.environ.get("EGC_DIST_T_EXCHANGE", "auto")
        # Overlapped exchanges for sum / symnorm-only layers on the peer transport (EGC_DIST_OVERLAP=1, opt-in): the halo
        # rows travel by the copy engine on a side stream while the entries with OWN columns are aggregated; a second
        # launch over the halo entries continues those sums (forward: `agg_init`; backward: EGC_BWD_ACCUMULATE).  Measured
        # on 2 x B200, mag shape (profiles/r02m_bench_2gpu_mag_ov{0,1}.json): 1.105 ms against 1.025 ms without - the second
        # launches pay the per-row work again (forward 0.23 -> 0.36 ms, column pass 0.16 -> 0.28 ms), more than the two
        # hidden pushes (0.22 ms) return - so it stays off by default.
        self.overlap = os.environ.get("EGC_DIST_OVERLAP", "0")
        self._split = {}
        self.group = group
        self._peer_ctx = {}

    @staticmethod
    def from_global(graph, rank: int, world_size: int, device, group=None, transport: str = "peer",
                    t_exchange: Optional[bool] = None, storage_dtype: torch.dtype = torch.float32) -> "PartitionedGraph":
        """Partition a prepared single-device `GraphStructure` (every rank builds the same plan).  `t_exchange`: also
        partition the transposed adjacency (needed by the T-exchange backward; default: yes for square graphs on more
        than one rank unless EGC_DIST_T_EXCHANGE=0).  `storage_dtype`: see the class docstring; bf16 raises ValueError
        for a graph with edge values, on every rank alike and before anything collective."""
        import os
        plan = PartitionPlan(graph.rowptr.cpu(), graph.col.cpu(), world_size,
                             val_sym=graph.val_sym.cpu() if graph.val_sym is not None else None,
                             val_lin=graph.val_lin.cpu() if graph.val_lin is not None else None)
        if t_exchange is None:
            t_exchange = world_size > 1 and graph.n_dst == graph.n_src and os.environ.get("EGC_DIST_T_EXCHANGE", "auto") != "0"
        tpart = plan.transposed().local(rank) if t_exchange else None
        return PartitionedGraph(plan.local(rank), device, group, transport, tpart, storage_dtype)

    @property
    def graph_t(self):
        """Device CSR of this rank's rows of the transposed adjacency: rows = own source columns, column ids = rows of
        the [own | halo] target-stream table."""
        if self._graph_t is None:
            from .graph import GraphStructure
            t = self.tpart
            self._graph_t = GraphStructure.from_prepared(t.rowptr, t.col, t.n_local + t.n_halo, val_sym=t.val_sym,
                                                         val_lin=t.val_lin, device=self.device)
        return self._graph_t

    def split_graphs(self, transposed: bool):
        """(own-column part, halo-column part) of the local block (or of its transposed twin) as device graphs."""
        if transposed not in self._split:
            from .graph import GraphStructure
            part = self.tpart if transposed else self.part
            self._split[transposed] = tuple(
                GraphStructure.from_prepared(rp, col, part.n_local + part.n_halo, val_sym=vs, val_lin=vl, device=self.device)
                for rp, col, vs, vl in part.split_by_column())
        return self._split[transposed]

    def uses_overlap(self, aggrs, storage_dtype: torch.dtype = torch.float32) -> bool:
        """Split launches around a copy-engine exchange: layers whose aggregators are all sum / symnorm (continuable sums
        that do not depend on the row's entry count), peer transport, T-exchange backward.  Never for bf16 layers: the
        second forward launch continues the sums with `agg_init`, which the bf16 forward does not take."""
        return (storage_dtype == torch.float32 and self.transport == "peer" and self.overlap != "0" and
                self.part.n_halo > 0 and all(a in ("sum", "symnorm") for a in aggrs) and self.uses_t_exchange(aggrs))

    def uses_t_exchange(self, aggrs) -> bool:
        if self.tpart is None or self.t_exchange == "0" or any(a in ("max", "min") for a in aggrs):
            return False
        if self.part.val_lin is not None and self.t_exchange != "1":     # per-entry weights: the partial-sum exchange (tested)
            return False
        return self.t_exchange == "1" or n_target_streams(aggrs) == 1

    def peer_context(self, key, bd: int, n_flat: int, t_width: int = 0, storage_dtype: torch.dtype = torch.float32):
        """Exchange state of one layer (collective on first use: every rank must reach it in the same order)."""
        k = (key, int(bd), int(n_flat), int(t_width), storage_dtype)
        ctx = self._peer_ctx.get(k)
        if ctx is None:
            from .peer import PeerLayerContext
            ctx = PeerLayerContext(self.part, bd, n_flat, self.device, self.group,
                                   tpart=self.tpart if t_width else None, t_width=t_width, storage_dtype=storage_dtype)
            self._peer_ctx[k] = ctx
        return ctx

    def check(self):
        """Raise if any exchange of this graph timed out on the device (synchronises)."""
        for ctx in self._peer_ctx.values():
            ctx.check()

    def close(self):
        for ctx in self._peer_ctx.values():
            ctx.close()
        self._peer_ctx = {}


def n_target_streams(aggrs) -> int:
    """Linear target-side streams of the backward: [symnorm] + [sum / mean / var / std] + [var / std] (DESIGN.md 3)."""
    return (int("symnorm" in aggrs) + int(any(a in ("sum", "mean", "var", "std") for a in aggrs)) +
            int(any(a in ("var", "std") for a in aggrs)))


class _PartitionedEGConvFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, bases_weight, comb_weight, comb_bias, bias, pg, heads, num_bases, aggrs, sigmoid, algo, key,
                grad_mode=True, bwd_flags=0, relu=False, storage_dtype=torch.float32, dropout=0.0, dropout_seed=None):
        from . import functional as F
        from . import peer as P
        part, g = pg.part, pg.graph
        x = F._require_cuda_f32("x", x)
        dropout = F.check_dropout(dropout)
        if dropout > 0.0 and not relu:
            raise ValueError("the fused dropout follows the fused ReLU: dropout > 0 needs relu=True")
        bd = bases_weight.size(1)
        desc = F.make_desc(g, heads, num_bases, bd // num_bases, aggrs, sigmoid, relu)
        bf16 = storage_dtype == torch.bfloat16
        if bf16:
            F.check_bf16_layer(desc, g)
        # the bf16 forward has no row subset: bf16 layers wait for the halo rows and run one contiguous launch
        rows_split = pg.overlap_interior and not bf16
        needs_grad = grad_mode and any(ctx.needs_input_grad[:5])       # needs_input_grad ignores torch.no_grad()
        peer = None
        with torch.cuda.device(x.device):
            if pg.transport == "peer":
                n_flat = bases_weight.numel() + comb_weight.numel() + comb_weight.size(0) + heads * (bd // num_bases)
                peer = pg.peer_context(key, bd, n_flat, n_target_streams(aggrs) * bd if pg.uses_t_exchange(aggrs) else 0,
                                       storage_dtype)
                # new epoch; every peer is done with the halo rows of my previous step
                ctx.step_id = peer.begin_step(needs_grad)
                bases_ext = peer.bases_ext
            else:
                bases_ext = torch.empty((part.n_local + part.n_halo, bd), dtype=storage_dtype, device=x.device)
            _, weightings = F.project(x, bases_weight.contiguous(), comb_weight.contiguous(), comb_bias, sigmoid, algo,
                                      bases_out=bases_ext[:part.n_local])
            outs = F.alloc_aggregate_outputs(desc, x.device, want_out=True, want_saved=needs_grad)
            drop = None                                    # this rank's rows of the single-GPU mask: keyed by global row
            if dropout > 0.0:
                seed = F.check_dropout_seed(dropout_seed, x.device) if dropout_seed is not None else F.draw_dropout_seed(x.device)
                drop = (seed, dropout, part.row_begin)
            def interior():
                if rows_split:
                    F.aggregate_combine(desc, g, bases_ext, weightings, bias, row_subset=pg.interior, use_plan=False,
                                        outputs=outs, dropout=drop)

            overlap = peer is not None and pg.uses_overlap(aggrs, storage_dtype)
            if overlap:
                # copy-engine push on the side stream while the entries with own columns are aggregated here; the halo
                # entries then continue those sums (agg_init) and the same launch combines and writes out / saved
                main = torch.cuda.current_stream()
                peer.side_stream.wait_stream(main)
                with torch.cuda.stream(peer.side_stream):
                    peer.push_forward(dma=True)
                g_own, g_halo = pg.split_graphs(False)
                partial = F.aggregate_combine(desc, g_own, bases_ext, None, None, want_out=False, want_agg=True)[1]
                main.wait_stream(peer.side_stream)
                peer.wait(P.SLOT_FWD)
                F.aggregate_combine(desc, g_halo, bases_ext, weightings, bias, outputs=outs,
                                    epilogue=(None, None, None, partial), dropout=drop)
            elif peer is not None:
                peer.push_forward()                        # posted stores into the peers' halo regions, then FWD flag
                interior()
                peer.wait(P.SLOT_FWD)
            else:
                # halo exchange runs on the communication stream while interior rows are aggregated here
                halo, handle = pg.exchange.start_forward(bases_ext[:part.n_local])
                interior()
                pg.exchange.finish(handle)
                bases_ext[part.n_local:].copy_(halo)
            if overlap:
                pass
            elif rows_split:
                F.aggregate_combine(desc, g, bases_ext, weightings, bias, row_subset=pg.boundary, use_plan=True,
                                    outputs=outs, dropout=drop)
            else:                                          # one contiguous launch over every local row
                F.aggregate_combine(desc, g, bases_ext, weightings, bias, outputs=outs, dropout=drop)
            if peer is not None and not needs_grad:
                peer.signal(P.SLOT_CONS)
        out, _, _, saved, saved_arg = outs
        if needs_grad:
            # dropout: out > 0 = ReLU open and kept, so the ReLU's mask scaled by k is the backward (functional.egconv)
            k = (torch.full((desc.heads * desc.dim,), F.dropout_constants(dropout)[1], dtype=torch.float32, device=x.device)
                 if dropout > 0.0 else None)
            ctx.save_for_backward(x, bases_weight, comb_weight, bases_ext, weightings, saved, saved_arg, out if relu else None, k)
        ctx.pg, ctx.desc, ctx.algo, ctx.peer, ctx.bwd_flags, ctx.aggrs = pg, desc, algo, peer, int(bwd_flags), tuple(aggrs)
        ctx.storage_dtype = storage_dtype
        ctx.has_bias, ctx.has_comb_bias = bias is not None, comb_bias is not None
        return out

    @staticmethod
    def backward(ctx, grad_out):
        from . import functional as F
        from . import peer as P
        x, bases_weight, comb_weight, bases_ext, weightings, saved, saved_arg, out_act, epi_scale = ctx.saved_tensors
        pg, part, peer = ctx.pg, ctx.pg.part, ctx.peer
        grad_out = F._require_cuda_f32("grad_out", grad_out)
        need_x, need_wb, need_wc, need_bc, need_b = ctx.needs_input_grad[:5]
        want_b = bool(need_b and ctx.has_bias)
        want_bc = bool(need_bc and ctx.has_comb_bias)
        with torch.cuda.device(x.device):
            use_t = pg.uses_t_exchange(ctx.aggrs)
            if use_t:                                      # descriptor of the column pass over the transposed local block
                desc_t = F.make_desc(pg.graph, ctx.desc.heads, ctx.desc.bases, ctx.desc.dim, ctx.aggrs, False)
                desc_t.n_dst, desc_t.n_src = pg.tpart.n_local + pg.tpart.n_halo, pg.tpart.n_local   # stream rows, own columns
                t_width = n_target_streams(ctx.aggrs) * ctx.desc.bases * ctx.desc.dim
            if peer is None and use_t:
                t_own = torch.empty((part.n_local, t_width), dtype=ctx.storage_dtype, device=x.device)
                d_w, _, d_bias, d_bc = F.aggregate_backward(ctx.desc, pg.graph, bases_ext, weightings, saved, saved_arg,
                                                            grad_out, want_b, ctx.bwd_flags, want_lin_colsum=True,
                                                            out_act=out_act, epi_scale=epi_scale, tstreams_out=t_own)
                t_ext = torch.cat([t_own, pg.exchange_t.forward(t_own)])      # stream rows of the remote targets
                d_bases = F.aggregate_backward_cols(desc_t, pg.graph_t, t_ext, bases_ext[:part.n_local])
            elif peer is None:
                d_w, d_bases_ext, d_bias, d_bc = F.aggregate_backward(ctx.desc, pg.graph, bases_ext, weightings, saved,
                                                                      saved_arg, grad_out, want_b, ctx.bwd_flags,
                                                                      want_lin_colsum=True, out_act=out_act, epi_scale=epi_scale)
                d_bases = d_bases_ext[:part.n_local]
                pg.exchange.reverse(d_bases_ext[part.n_local:], d_bases)     # halo partial sums go home
            if peer is None:
                d_x, d_wb, d_wc, _ = F.project_backward(x, bases_weight.contiguous(), comb_weight.contiguous(), d_bases,
                                                        d_w, need_x, need_wb, need_wc, False, ctx.algo)
                if not want_bc:
                    d_bc = None
                for t in (d_wb, d_wc, d_bc, d_bias):                          # parameters are replicated
                    if t is not None:
                        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=pg.group)
                return (d_x, d_wb, d_wc, d_bc, d_bias) + (None,) * 13
            # ---- peer transport: flat parameter-gradient vector [d_wb | d_wc | d_bc | d_bias] in the exchange context
            n_wb, n_wc, hab = bases_weight.numel(), comb_weight.numel(), comb_weight.size(0)
            hd = ctx.desc.heads * ctx.desc.dim
            flat = peer.flat
            v_wb = flat[:n_wb].view_as(bases_weight)
            v_wc = flat[n_wb:n_wb + n_wc].view_as(comb_weight)
            v_bc = flat[n_wb + n_wc:n_wb + n_wc + hab]
            v_b = flat[n_wb + n_wc + hab:n_wb + n_wc + hab + hd]
            peer.begin_backward(ctx.step_id)
            if not (need_wb and need_wc and want_b):
                flat.zero_()
            main = torch.cuda.current_stream()

            def push_halo(d_ext):                          # halo partial sums go home (posted stores), BWD + CONS flags,
                peer.side_stream.wait_stream(main)         # on a side stream while the own columns of pass 2 run
                with torch.cuda.stream(peer.side_stream):
                    peer.push_backward(d_ext)

            routed = any(a in ("max", "min") for a in ctx.aggrs)
            if use_t:
                # pass 1 writes the streams of my targets into the exchange table; the rows my peers' columns touch go
                # to them (BWD + CONS flags); once theirs are here the column pass over my own columns is complete
                d_w, _, _, _ = F.aggregate_backward(ctx.desc, pg.graph, bases_ext, weightings, saved, saved_arg, grad_out,
                                                    want_b, ctx.bwd_flags, want_lin_colsum=True, out_bias=v_b,
                                                    out_lin_colsum=v_bc, out_act=out_act, epi_scale=epi_scale, tstreams_out=peer.t_ext)
                if pg.uses_overlap(ctx.aggrs, ctx.storage_dtype):
                    peer.side_stream.wait_stream(main)
                    with torch.cuda.stream(peer.side_stream):
                        peer.push_t(dma=True)
                    gt_own, gt_halo = pg.split_graphs(True)
                    d_bases = F.aggregate_backward_cols(desc_t, gt_own, peer.t_ext, bases_ext[:part.n_local])
                    main.wait_stream(peer.side_stream)
                    peer.wait(P.SLOT_BWD)
                    d_bases = F.aggregate_backward_cols(desc_t, gt_halo, peer.t_ext, bases_ext[:part.n_local],
                                                        d_bases=d_bases, accumulate=True)
                else:
                    peer.push_t()
                    peer.wait(P.SLOT_BWD)
                    d_bases = F.aggregate_backward_cols(desc_t, pg.graph_t, peer.t_ext, bases_ext[:part.n_local])
            elif pg.split_backward == "1" or (pg.split_backward == "auto" and not routed):
                d_w, d_bases_ext, _, _ = F.aggregate_backward(ctx.desc, pg.graph, bases_ext, weightings, saved, saved_arg,
                                                              grad_out, want_b, ctx.bwd_flags, want_lin_colsum=True,
                                                              out_bias=v_b, out_lin_colsum=v_bc, col_split=part.n_local,
                                                              between_phases=push_halo, out_act=out_act, epi_scale=epi_scale)
                main.wait_stream(peer.side_stream)
            else:
                d_w, d_bases_ext, _, _ = F.aggregate_backward(ctx.desc, pg.graph, bases_ext, weightings, saved, saved_arg,
                                                              grad_out, want_b, ctx.bwd_flags, want_lin_colsum=True,
                                                              out_bias=v_b, out_lin_colsum=v_bc, out_act=out_act, epi_scale=epi_scale)
                peer.push_backward(d_bases_ext)
            if not use_t:
                peer.wait(P.SLOT_BWD)
                d_bases = d_bases_ext[:part.n_local]
                peer.reduce_into(d_bases)                  # fixed peer order: deterministic
            d_x, _, _, _ = F.project_backward(x, bases_weight.contiguous(), comb_weight.contiguous(), d_bases, d_w,
                                              need_x, need_wb, need_wc, False, ctx.algo, out_wb=v_wb, out_wc=v_wc)
            total = peer.allreduce_flat()
            d_wb = total[:n_wb].view_as(bases_weight).clone() if need_wb else None
            d_wc = total[n_wb:n_wb + n_wc].view_as(comb_weight).clone() if need_wc else None
            d_bc = total[n_wb + n_wc:n_wb + n_wc + hab].clone() if want_bc else None
            d_bias = total[n_wb + n_wc + hab:n_wb + n_wc + hab + hd].clone() if want_b else None
        return (d_x, d_wb, d_wc, d_bc, d_bias) + (None,) * 13


def _bwd_flags_of(conv) -> int:
    from . import _lib
    return (_lib.BWD_DETERMINISTIC if getattr(conv, "deterministic", False) else 0) | int(getattr(conv, "bwd_flags", 0))


def partitioned_egconv(x_local: Tensor, pg: PartitionedGraph, conv, relu: bool = False, dropout: float = 0.0,
                       dropout_seed: Optional[Tensor] = None) -> Tensor:
    """Run `conv` (an `egc_b200.EGConv` with replicated parameters) on this rank's rows of a partitioned graph.
    Output rows / input gradients are local; parameter gradients are summed over the ranks (= single-GPU values).
    With the peer transport every layer keeps its own exchange buffers (keyed by the module), one step in flight.
    A layer with `storage_dtype=torch.bfloat16` needs a graph built with `storage_dtype=torch.bfloat16`; it returns this
    rank's rows of the single-GPU bf16 layer's results.
    `dropout` = p > 0 (with relu=True): the fused dropout of `egc_b200.functional.egconv`, keyed by the GLOBAL row, so each
    rank gets its rows of the single-GPU mask for the same seed.  Without `dropout_seed` every rank draws it from its own
    default CUDA generator: the ranks must be seeded identically (torch.manual_seed with the same value, as every
    multi-rank driver of this project does), or their masks are not one mask."""
    storage_dtype = getattr(conv, "storage_dtype", torch.float32)
    if storage_dtype != torch.float32 and getattr(pg, "storage_dtype", None) != storage_dtype:
        raise NotImplementedError("partitioned_egconv: a layer with storage_dtype=torch.bfloat16 needs a PartitionedGraph "
                                  "built with storage_dtype=torch.bfloat16 (PartitionedGraph.from_global(..., "
                                  "storage_dtype=torch.bfloat16))")
    return _PartitionedEGConvFunction.apply(x_local, conv.bases_weight, conv.comb_weight.weight, conv.comb_weight.bias,
                                            conv.bias, pg, conv.num_heads, conv.num_bases, tuple(conv.aggregators),
                                            bool(conv.sigmoid), int(conv.gemm_algo), id(conv), torch.is_grad_enabled(),
                                            _bwd_flags_of(conv), bool(relu), storage_dtype, float(dropout), dropout_seed)


class PartitionedHeteroGraph:
    """Device-side state of one rank of a row-partitioned heterogeneous graph (`REGConv`): per relation the local CSR
    ([own target rows] x [own | halo] rows of its source type), per node type the halo exchange.  Pass it to
    `REGConv.forward` in place of the adjacency dict; the layer then returns this rank's rows of every type.

    transport = "peer" (default): every layer gets one peer segment holding the [own | halo] basis table of every node
    type; ONE push moves the halo rows of all types, ONE push sends their partial sums home, ONE reduce adds them in fixed
    peer order, ONE kernel all-reduces the parameter gradients (`egc_b200.peer`).  transport = "nccl": one
    `CudaHaloExchange` per node type and `dist.all_reduce` (the library baseline)."""

    def __init__(self, part: HeteroLocalPartition, device, group=None, transport: str = "peer"):
        from .graph import GraphStructure
        if transport not in ("peer", "nccl"):
            raise ValueError(f"unknown transport {transport!r}")
        self.part, self.device, self.group, self.transport = part, torch.device(device), group, transport
        self.types = list(part.tables)
        self.edge_types = list(part.relations)          # the order of the adjacency dict: the accumulation order
        self.graphs = {}
        for k, rel in part.relations.items():
            tab = part.tables[k[0]]
            self.graphs[k] = GraphStructure.from_prepared(rel.rowptr, rel.col, tab.n_local + tab.n_halo,
                                                          val_lin=rel.val_lin, device=self.device)
        self.exchanges = {t: CudaHaloExchange(tab, self.device, group) for t, tab in part.tables.items()}
        self._peer_ctx = {}

    @staticmethod
    def from_global(adj_t_dict, sizes: Dict[str, int], rank: int, world_size: int, device, group=None,
                    transport: str = "peer") -> "PartitionedHeteroGraph":
        """Partition a dict of whole-graph adjacencies {(src, rel, dst): adj_t} (rows = targets) over node types with
        `sizes` rows each (every rank builds the same plan).  Raises ValueError, on every rank alike and before anything
        collective, when a type has fewer rows than there are ranks."""
        from .graph import adjacency_to_csr
        csr, values = {}, {}
        for k, adj in adj_t_dict.items():
            rowptr, col, value, n_src = adjacency_to_csr(adj)
            if k[0] in sizes and n_src != sizes[k[0]]:
                raise ValueError(f"adjacency of {k} has {n_src} columns, node type {k[0]!r} has {sizes[k[0]]} rows")
            csr[k] = (rowptr.cpu(), col.cpu())
            if value is not None:
                values[k] = value.cpu()
        plan = HeteroPartitionPlan(csr, sizes, world_size, values)
        return PartitionedHeteroGraph(plan.local(rank), device, group, transport)

    def row_range(self, node_type: str) -> Tuple[int, int]:
        """(begin, end) of the global rows of `node_type` this rank owns."""
        tab = self.part.tables[node_type]
        return tab.row_begin, tab.row_end

    def peer_context(self, key, bd: int, n_flat: int):
        """Exchange state of one layer (collective on first use: every rank must reach it in the same order)."""
        k = (key, int(bd), int(n_flat))
        ctx = self._peer_ctx.get(k)
        if ctx is None:
            from .peer import PeerLayerContext
            ctx = PeerLayerContext([self.part.tables[t] for t in self.types], bd, n_flat, self.device, self.group)
            self._peer_ctx[k] = ctx
        return ctx

    def exchange(self, key, n_flat: int, bases: Dict[str, Tensor]) -> Dict[str, Tensor]:
        """{type: own basis rows} -> {type: [own | halo] rows}, differentiable (backward: halo partial sums go home)."""
        tables = _HeteroHaloFunction.apply(self, key, int(n_flat), torch.is_grad_enabled(), *[bases[t] for t in self.types])
        return dict(zip(self.types, tables))

    def replicated(self, key, params: Sequence[Tensor]) -> Tuple[Tensor, ...]:
        """The same parameters; their gradients are summed over the ranks (one flat all-reduce per layer)."""
        return _ReplicatedParamsFunction.apply(self, key, *params)

    def end_forward(self, key, bd: int, n_flat: int) -> None:
        """After the last relation launch of a forward that saved nothing for a backward: release the peers' rows (CONS)."""
        from . import peer as P
        ctx = self._peer_ctx.get((key, int(bd), int(n_flat)))
        if ctx is not None and not ctx.outstanding:
            ctx.signal(P.SLOT_CONS)

    def check(self):
        """Raise if any exchange of this graph timed out on the device (synchronises)."""
        for ctx in self._peer_ctx.values():
            ctx.check()

    def close(self):
        for ctx in self._peer_ctx.values():
            ctx.close()
        self._peer_ctx = {}


class _HeteroHaloFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, phg, key, n_flat, grad_mode, *bases):
        from . import peer as P
        types = phg.types
        tabs = [phg.part.tables[t] for t in types]
        bd = bases[0].size(1)
        for t, b, tab in zip(types, bases, tabs):
            if b.dtype != torch.float32 or not b.is_cuda or tuple(b.shape) != (tab.n_local, bd):
                raise ValueError(f"bases of node type {t!r} must be CUDA fp32 [{tab.n_local}, {bd}] (got {b.dtype} "
                                 f"{tuple(b.shape)} on {b.device})")
        needs_grad = grad_mode and any(ctx.needs_input_grad[4:])       # needs_input_grad ignores torch.no_grad()
        peer = None
        with torch.cuda.device(bases[0].device):
            if phg.transport == "peer":
                peer = phg.peer_context(key, bd, n_flat)
                ctx.step_id = peer.begin_step(needs_grad)       # every peer is done with the halo rows of my last step
                out = [peer.table(i) for i in range(len(types))]
                for o, b, tab in zip(out, bases, tabs):
                    o[:tab.n_local].copy_(b)
                peer.push_forward()                             # every type's halo rows to every peer, then FWD flag
                peer.wait(P.SLOT_FWD)
            else:
                out = [torch.cat([b, phg.exchanges[t].forward(b)]) for t, b in zip(types, bases)]
        ctx.phg, ctx.peer, ctx.bd = phg, peer, bd
        return tuple(out)

    @staticmethod
    def backward(ctx, *d_ext):
        from . import peer as P
        phg, peer = ctx.phg, ctx.peer
        tabs = [phg.part.tables[t] for t in phg.types]
        dev = phg.device
        d_ext = [d.contiguous() if d is not None else torch.zeros((tab.n_local + tab.n_halo, ctx.bd), device=dev)
                 for d, tab in zip(d_ext, tabs)]
        with torch.cuda.device(dev):
            if peer is None:
                d_own = []
                for t, d, tab in zip(phg.types, d_ext, tabs):
                    own = d[:tab.n_local].clone()
                    phg.exchanges[t].reverse(d[tab.n_local:], own)       # halo partial sums go home
                    d_own.append(own)
                return (None,) * 4 + tuple(d_own)
            peer.begin_backward(ctx.step_id)
            stacked = torch.cat([d[:tab.n_local] for d, tab in zip(d_ext, tabs)])     # [own t0 | own t1 | ...]
            peer.push_backward(*d_ext)                          # every type's halo partial sums home, BWD + CONS flags
            peer.wait(P.SLOT_BWD)
            peer.reduce_into(stacked)                           # fixed peer order: deterministic
        return (None,) * 4 + tuple(stacked.split([tab.n_local for tab in tabs]))


class _ReplicatedParamsFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, phg, key, *params):
        ctx.phg, ctx.key, ctx.sizes = phg, key, [p.numel() for p in params]
        ctx.set_materialize_grads(False)
        return tuple(p.view_as(p) for p in params)

    @staticmethod
    def backward(ctx, *grads):
        phg, n = ctx.phg, sum(ctx.sizes)
        with torch.cuda.device(phg.device):
            if phg.transport == "peer":                  # the layer's exchange context (made by its forward)
                peer = next(c for k, c in phg._peer_ctx.items() if k[0] == ctx.key and k[2] == n)
                flat = peer.flat
            else:
                flat = torch.empty(n, dtype=torch.float32, device=phg.device)
            off = 0
            for g, m in zip(grads, ctx.sizes):           # fixed layout [param 0 | param 1 | ...], unused ones zero
                if g is not None:
                    flat[off:off + m].copy_(g.reshape(-1))
                else:
                    flat[off:off + m].zero_()
                off += m
            if phg.transport == "peer":
                total = peer.allreduce_flat()
            else:
                dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=phg.group)
                total = flat
            out, off = [], 0
            for g, m in zip(grads, ctx.sizes):
                out.append(total[off:off + m].view_as(g).clone() if g is not None else None)
                off += m
        return (None, None) + tuple(out)


class GraphedStep:
    """Capture `fn(*static_inputs)` - typically one forward + backward of a partitioned layer stack, exchange kernels
    and flags included - into a CUDA graph after `warmup` eager calls; `replay()` re-runs it with the current
    contents of the static input tensors.  `outputs` are the tensors `fn` returned at capture time (static too)."""

    def __init__(self, fn, warmup: int = 3):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        # thread_local: CUDA calls of other threads (the NCCL watchdog polling its events, pinned-memory helpers)
        # must not invalidate the capture; the autograd worker thread still launches into the capturing stream
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
            self.outputs = fn()

    def replay(self):
        self.graph.replay()
        return self.outputs


class GradientAllReduce:
    """Data-parallel mini-batch training (BASELINE configs 1 / 5; SURVEY.md section 8e): every rank runs the same
    model on different collated batches and the parameter gradients are combined with ONE flat all-reduce per
    bucket.  `weight` is this rank's share of the global batch (graphs on this rank / graphs on all ranks), so that
    a loss averaged over the local graphs yields the gradient of the loss averaged over ALL graphs - the parity
    statement of the single-process run on the concatenated batch.  Buckets are persistent flat buffers (no
    allocation per step, CUDA-graph friendly); NCCL on GPUs, gloo in the CPU tests."""

    def __init__(self, params, group=None, bucket_bytes: int = 32 << 20):
        self.params = [p for p in params if p.requires_grad]
        self.group = group
        self.buckets = []                                   # (flat buffer, [(param, offset, numel)])
        cur, cur_bytes = [], 0
        for p in self.params:
            nbytes = p.numel() * p.element_size()
            if cur and (cur_bytes + nbytes > bucket_bytes or cur[0].dtype != p.dtype or cur[0].device != p.device):
                self._close(cur)
                cur, cur_bytes = [], 0
            cur.append(p)
            cur_bytes += nbytes
        if cur:
            self._close(cur)

    def _close(self, ps):
        flat = torch.zeros(sum(p.numel() for p in ps), dtype=ps[0].dtype, device=ps[0].device)
        views, off = [], 0
        for p in ps:
            views.append((p, off, p.numel()))
            off += p.numel()
        self.buckets.append((flat, views))

    @torch.no_grad()
    def __call__(self, weight: float = None):
        """Overwrites every p.grad with sum_r weight_r * grad_r (weight defaults to 1 / world_size)."""
        world = dist.get_world_size(self.group)
        w = (1.0 / world) if weight is None else float(weight)
        handles = []
        for flat, views in self.buckets:
            for p, off, n in views:
                if p.grad is None:
                    flat[off:off + n].zero_()
                else:
                    torch.mul(p.grad.reshape(-1), w, out=flat[off:off + n])
            handles.append(dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True))
        for (flat, views), h in zip(self.buckets, handles):
            h.wait()
            for p, off, n in views:
                if p.grad is None:
                    p.grad = flat[off:off + n].view_as(p).clone()
                else:
                    p.grad.copy_(flat[off:off + n].view_as(p))


class OverlappedGradientAllReduce:
    """`GradientAllReduce` launched from inside the backward pass: one persistent flat bucket per module of
    `modules` (a layer each), all-reduced asynchronously as soon as the LAST gradient of that bucket has been
    accumulated (`register_post_accumulate_grad_hook`), i.e. while autograd is still running the backward of the
    layers below it (SURVEY.md section 8e: "bucketed all-reduce of grads per step overlapped with the previous layer's
    backward").  Protocol per step:  `begin(weight)` -> `loss.backward()` -> `finish()`; afterwards every `p.grad`
    holds  sum_r weight_r * grad_r  (weight = this rank's share of the global batch, default 1 / world_size).
    Works with NCCL (GPU) and gloo (CPU tests)."""

    def __init__(self, modules, group=None):
        self.group = group
        self.buckets = []                                   # [flat, [(param, offset, numel)], pending, handle]
        self._of = {}
        for m in modules:
            ps = [p for p in m.parameters() if p.requires_grad]
            if not ps:
                continue
            flat = torch.zeros(sum(p.numel() for p in ps), dtype=ps[0].dtype, device=ps[0].device)
            views, off = [], 0
            for p in ps:
                views.append((p, off, p.numel()))
                off += p.numel()
            b = {"flat": flat, "views": views, "pending": 0, "handle": None}
            self.buckets.append(b)
            for p in ps:
                self._of[p] = b
                p.register_post_accumulate_grad_hook(self._hook)
        self._weight = None

    def begin(self, weight: float = None):
        world = dist.get_world_size(self.group)
        self._weight = (1.0 / world) if weight is None else float(weight)
        for b in self.buckets:
            b["pending"], b["handle"] = len(b["views"]), None

    def _hook(self, p):
        if self._weight is None:                            # backward outside a begin() / finish() pair: plain local grads
            return
        b = self._of[p]
        b["pending"] -= 1
        if b["pending"] == 0:
            with torch.no_grad():
                for q, off, n in b["views"]:
                    torch.mul(q.grad.reshape(-1), self._weight, out=b["flat"][off:off + n])
            b["handle"] = dist.all_reduce(b["flat"], op=dist.ReduceOp.SUM, group=self.group, async_op=True)

    @torch.no_grad()
    def finish(self):
        for b in self.buckets:
            if b["handle"] is None:                         # a bucket whose parameters received no gradient this step
                for q, off, n in b["views"]:
                    if q.grad is None:
                        b["flat"][off:off + n].zero_()
                    else:
                        torch.mul(q.grad.reshape(-1), self._weight, out=b["flat"][off:off + n])
                b["handle"] = dist.all_reduce(b["flat"], op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        for b in self.buckets:
            b["handle"].wait()
            for q, off, n in b["views"]:
                if q.grad is None:
                    q.grad = b["flat"][off:off + n].view_as(q).clone()
                else:
                    q.grad.copy_(b["flat"][off:off + n].view_as(q))
        self._weight = None
