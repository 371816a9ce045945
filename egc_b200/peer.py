"""NVLink peer-memory plumbing for the row-partitioned layer (one process per GPU of a node).

`PeerSegment` owns this rank's peer-visible device memory (allocated and IPC-exported by
`libegc_b200.so`, csrc/peer.cu), maps the segments of the other ranks and hands out torch views of its
own regions.  `PeerLayerContext` binds a `LocalPartition` to the exchange kernels for ONE layer:

  forward : epoch++ and wait CONS(epoch-1) (one kernel) -> [projection writes own basis rows into the segment]
            -> push the rows each peer needs straight into that peer's halo region (its last CTA raises FWD)
            -> [interior rows aggregate] -> wait FWD -> [boundary rows aggregate]
  backward: [pass 1, routing, pass 2 of the HALO columns] -> on a side stream: push halo partial sums into their owners'
            staging (raises BWD + CONS), overlapped with [pass 2 of the own columns] -> wait BWD -> deterministic
            reduce into own rows -> [projection
            gradients] -> push flat parameter gradients into every rank's slot (raises GRAD) -> wait GRAD
            -> sum the slots in rank order (bit-identical on every rank)
  backward, T exchange (layers without min / max and one target-side stream, `egc_b200.dist`): [pass 1 writes the stream
            rows of my targets into my `t_ext` table] -> push the rows my peers' source columns touch into THEIR tables
            (raises BWD + CONS) -> wait BWD -> [pass 2 over my own columns of the transposed local block: complete sums,
            no staging, no reduce] -> [projection gradients] -> as above

No NCCL call, no host synchronisation and no allocation is on that path, so a whole step can be captured
in a CUDA graph (`egc_b200.dist.GraphedStep`).  The reference has no multi-GPU counterpart.
"""
import ctypes
import os
from typing import Dict, List, Tuple

import torch
import torch.distributed as dist

from . import _lib
from ._lib import check

SLOT_FWD, SLOT_BWD, SLOT_GRAD, SLOT_CONS = 0, 1, 2, 3
N_SLOTS = 4
DEFAULT_TIMEOUT_NS = 20_000_000_000


def _align(v: int, a: int = 256) -> int:
    return (v + a - 1) // a * a


class _RawCuda:
    """Exposes a raw device allocation through __cuda_array_interface__ (no ownership)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class PeerSegment:
    """This rank's peer-visible memory, split into named regions, plus the mapped segments of the peers."""

    def __init__(self, regions: List[Tuple[str, int]], device, group=None):
        lib = _lib.load()
        self.device = torch.device(device)
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if self.world > 8:
            raise ValueError("peer-memory exchange supports up to 8 ranks of one node")
        self.offsets: Dict[str, int] = {}
        off = 0
        for name, nbytes in regions:
            self.offsets[name] = off
            off = _align(off + max(int(nbytes), 4))
        self.nbytes = max(off, 256)
        handle = (ctypes.c_ubyte * 64)()
        base = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(lib.egc_peer_alloc(self.nbytes, ctypes.byref(base), handle), "egc_peer_alloc")
        self.base = int(base.value)
        self._raw = torch.as_tensor(_RawCuda(self.base, self.nbytes), device=self.device)
        infos = [None] * self.world
        dist.all_gather_object(infos, {"handle": bytes(handle), "offsets": self.offsets}, group=group)
        self.peer_base: List[int] = [0] * self.world
        self.peer_offsets: List[Dict[str, int]] = [i["offsets"] for i in infos]
        self._opened: List[int] = []
        for q in range(self.world):
            if q == self.rank:
                self.peer_base[q] = self.base
                continue
            h = (ctypes.c_ubyte * 64).from_buffer_copy(infos[q]["handle"])
            p = ctypes.c_void_p()
            with torch.cuda.device(self.device):
                check(lib.egc_peer_open(h, ctypes.byref(p)), "egc_peer_open")
            self.peer_base[q] = int(p.value)
            self._opened.append(int(p.value))
        dist.barrier(group=group)

    def view(self, name: str, shape, dtype=torch.float32) -> torch.Tensor:
        n = 1
        for s in shape:
            n *= int(s)
        nbytes = n * torch.empty((), dtype=dtype).element_size()
        off = self.offsets[name]
        return self._raw[off:off + nbytes].view(dtype).view(*shape)

    def peer_ptr(self, q: int, name: str, byte_offset: int = 0) -> int:
        return self.peer_base[q] + self.peer_offsets[q][name] + byte_offset

    def close(self):
        lib = _lib.load()
        if getattr(self, "base", 0):
            torch.cuda.synchronize(self.device)
            try:
                dist.barrier(group=self.group)
            except Exception:
                pass
            for p in self._opened:
                lib.egc_peer_close(ctypes.c_void_p(p))
            self._opened = []
            self._raw = None
            lib.egc_peer_free(ctypes.c_void_p(self.base))
            self.base = 0


def _ptr_array(values: List[int]):
    arr = (ctypes.c_void_p * len(values))()
    for i, v in enumerate(values):
        arr[i] = v
    return arr


class PeerLayerContext:
    """Exchange state of one layer (basis width `bd`, `n_flat` replicated parameter-gradient floats) on one rank.
    `part` is one `LocalPartition` (EGConv: one [own | halo] basis table) or a list of them, one table per node type of a
    heterogeneous layer (`egc_b200.dist.PartitionedHeteroGraph`): every table gets its own [own | halo] region and staging
    rows, and each exchange moves the rows of ALL tables in one push - segments per (peer, table), peers in the rotated
    order outside, tables inside - with one flag; the reduce adds the partial sums into the stacked own rows
    [own 0 | own 1 | ...].  The T exchange and the copy-engine pushes take one table.
    storage_dtype=torch.bfloat16: the basis rows (`bases_ext`) and the target-side stream rows (`t_ext`) are stored and
    pushed as bf16 - half the bytes per exchanged row; the halo partial sums (`staging`) and the parameter-gradient slots
    stay fp32."""

    def __init__(self, part, bd: int, n_flat: int, device, group=None, timeout_ns: int = DEFAULT_TIMEOUT_NS,
                 tpart=None, t_width: int = 0, storage_dtype: torch.dtype = torch.float32):
        tables = list(part) if isinstance(part, (list, tuple)) else [part]
        self.tables = tables
        self.part, self.bd, self.device, self.group = tables[0], int(bd), torch.device(device), group
        self.storage_dtype = storage_dtype
        elem = torch.empty((), dtype=storage_dtype).element_size()            # bytes per stored basis / stream value
        self.tpart, self.t_width = (tpart, int(t_width)) if tpart is not None and t_width else (None, 0)
        if len(tables) > 1 and self.tpart is not None:
            raise ValueError("the T exchange takes one table")
        self.rank, self.world = self.part.rank, self.part.world_size
        if (self.world - 1) * len(tables) > _lib.MAX_PUSH_SEGMENTS:           # same on every rank, nothing collective yet
            raise ValueError(f"{len(tables)} tables over {self.world} ranks need {(self.world - 1) * len(tables)} push "
                             f"segments, more than {_lib.MAX_PUSH_SEGMENTS}")
        self.timeout_ns = int(timeout_ns)
        self.n_flat = _align(int(n_flat), 128)                     # rows of 128 floats for the slot pushes
        n_ext = [t.n_local + t.n_halo for t in tables]
        send_counts = [[int(r.numel()) for r in t.send_rows] for t in tables]
        n_send = [sum(c) if self.tpart is None else 0 for c in send_counts]     # T exchange: no partial sums, no staging
        stage_off = [0]                                            # staging rows of table i start at stage_off[i]
        for c in n_send:
            stage_off.append(stage_off[-1] + c)
        own_off = [0]                                              # stacked own rows [own 0 | own 1 | ...]
        for t in tables:
            own_off.append(own_off[-1] + t.n_local)
        n_ext_t = (self.tpart.n_local + self.tpart.n_halo) if self.tpart is not None else 0
        # the push kernels move 4-byte words: row widths of the stored tables in words (bf16 rows: whole 16-byte pieces)
        if elem != 4 and (self.bd % 8 or self.t_width % 8):
            raise ValueError(f"bf16 exchange rows need B*D % 8 == 0 (got {self.bd})")
        self.bd_words, self.t_words = self.bd * elem // 4, self.t_width * elem // 4
        self.seg = PeerSegment([("flags", 4 * N_SLOTS * self.world)] +
                               [(f"bases_ext{i}", elem * n * bd) for i, n in enumerate(n_ext)] +
                               [("staging", 4 * max(stage_off[-1], 1) * bd), ("slots", 4 * self.world * self.n_flat),
                                ("t_ext", elem * n_ext_t * self.t_width)], device, group)
        self.t_ext = self.seg.view("t_ext", (n_ext_t, self.t_width), storage_dtype) if self.tpart is not None else None
        self.flags = self.seg.view("flags", (N_SLOTS * self.world,), torch.int32)
        self.n_ext = n_ext
        self.bases_ext = self.table(0)
        self.staging = self.seg.view("staging", (max(stage_off[-1], 1), bd))
        self.slots = self.seg.view("slots", (self.world, self.n_flat))
        self.epoch = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.err = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.counter = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.flat = torch.zeros(self.n_flat, dtype=torch.float32, device=self.device)
        self.flat_sum = torch.zeros(self.n_flat, dtype=torch.float32, device=self.device)
        # host-side step bookkeeping: a forward that saved state for a backward is "outstanding" until that backward
        # has pushed its halo gradients (which also raises CONS, releasing the peers' halo copies of my rows)
        self.step_id = 0
        self.outstanding = False
        self.side_stream = torch.cuda.Stream(device=self.device)      # carries the backward push next to pass 2

        # what every rank must know about the others: local row counts, halo layout, staging layout (per table)
        recv_off, send_off = [], []
        for t, counts in zip(tables, send_counts):
            r_off, s_off = [0], [0]
            for c in t.recv_counts:
                r_off.append(r_off[-1] + c)
            for c in counts:
                s_off.append(s_off[-1] + c)
            recv_off.append(r_off)
            send_off.append(s_off)
        self.recv_off, self.send_off = recv_off, send_off
        infos = [None] * self.world
        t_recv_off = [0]
        for c in (self.tpart.recv_counts if self.tpart is not None else []):
            t_recv_off.append(t_recv_off[-1] + c)
        dist.all_gather_object(infos, {"n_local": [t.n_local for t in tables], "recv_off": recv_off, "send_off": send_off,
                                       "stage_off": stage_off, "t_recv_off": t_recv_off}, group=group)
        # Destination order of every push: rank + 1, rank + 2, ... (mod world).  The push kernel walks its segments in
        # this order, so at any moment the ranks write to DIFFERENT destinations; with the ascending order every rank
        # started on rank 0 (7 senders into one ingress port), then rank 1, ...  (EGC_PEER_ORDER=ascending: A/B)
        if os.environ.get("EGC_PEER_ORDER", "rotated") == "ascending":
            self.peers = [q for q in range(self.world) if q != self.rank]
        else:
            self.peers = [(self.rank + k) % self.world for k in range(1, self.world)]
        self.segments = [(q, i) for q in self.peers for i in range(len(tables))]      # peers outside, tables inside
        row_bytes = elem * bd

        # forward push: rows send_rows[q] of my table i -> q's halo region of table i, at q's offset for owner = me
        self.fwd_index = (torch.cat([tables[i].send_rows[q] for q, i in self.segments]) if self.segments else
                          torch.zeros(0, dtype=torch.long)).to(self.device, torch.int32)
        self.fwd_seg_ptr = (ctypes.c_int32 * (len(self.segments) + 1))()
        fwd_dst = []
        for s, (q, i) in enumerate(self.segments):
            self.fwd_seg_ptr[s + 1] = self.fwd_seg_ptr[s] + send_counts[i][q]
            fwd_dst.append(self.seg.peer_ptr(q, f"bases_ext{i}",
                                             (infos[q]["n_local"][i] + infos[q]["recv_off"][i][self.rank]) * row_bytes))
        self.fwd_dst = _ptr_array(fwd_dst)
        self.fwd_dst_list, self.fwd_counts = fwd_dst, [send_counts[i][q] for q, i in self.segments]
        self.fwd_src = _ptr_array([self.seg.peer_ptr(self.rank, f"bases_ext{i}") for _, i in self.segments])

        # backward push: my halo rows of table i owned by q (contiguous) -> q's staging, at q's offset for sender = me
        self.bwd_seg_ptr = (ctypes.c_int32 * (len(self.segments) + 1))()
        bwd_dst = []
        for s, (q, i) in enumerate(self.segments):
            self.bwd_seg_ptr[s + 1] = self.bwd_seg_ptr[s] + tables[i].recv_counts[q]
            bwd_dst.append(self.seg.peer_ptr(q, "staging",
                                             (infos[q]["stage_off"][i] + infos[q]["send_off"][i][self.rank]) * 4 * bd))
        self.bwd_dst = _ptr_array(bwd_dst)

        # T exchange: rows tpart.send_rows[q] of my stream table -> q's table, at q's offset for owner = me
        if self.tpart is not None:
            t_counts = [int(t.numel()) for t in self.tpart.send_rows]
            self.t_index = (torch.cat([self.tpart.send_rows[q] for q in self.peers]) if self.peers else
                            torch.zeros(0, dtype=torch.long)).to(self.device, torch.int32)
            self.t_seg_ptr = (ctypes.c_int32 * (len(self.peers) + 1))()
            t_dst = []
            for s, q in enumerate(self.peers):
                self.t_seg_ptr[s + 1] = self.t_seg_ptr[s] + t_counts[q]
                t_dst.append(self.seg.peer_ptr(q, "t_ext", (infos[q]["n_local"][0] + infos[q]["t_recv_off"][self.rank]) * elem * self.t_width))
            self.t_dst = _ptr_array(t_dst)
            self.t_dst_list, self.t_counts = t_dst, [t_counts[q] for q in self.peers]
            self.t_src = _ptr_array([self.t_ext.data_ptr()] * len(self.peers))

        # copy-engine pushes (overlapped exchanges): the rows are packed here first, then one contiguous copy per peer
        pack = max(sum(send_counts[0]) * self.bd_words, sum(self.t_counts) * self.t_words if self.tpart is not None else 0, 4)
        self.send_buf = torch.empty(pack, dtype=torch.float32, device=self.device)      # 4-byte words

        # deterministic reduce plan: stacked own row -> its staging entries in ascending peer order
        red_rows, red_cnt, red_entry = [], [], []
        for i, t in enumerate(tables):
            if not n_send[i]:
                continue
            rows_cat = torch.cat([t.send_rows[q] for q in range(self.world)])           # staging order = peer order
            order = torch.argsort(rows_cat, stable=True)
            uniq, counts = torch.unique_consecutive(rows_cat[order], return_counts=True)
            red_rows.append(uniq + own_off[i])
            red_cnt.append(counts)
            red_entry.append(order + stage_off[i])
        if red_rows:
            counts = torch.cat(red_cnt)
            ptr = torch.zeros(counts.numel() + 1, dtype=torch.long)
            ptr[1:] = torch.cumsum(counts, 0)
            self.red_rows = torch.cat(red_rows).to(self.device, torch.int32)
            self.red_ptr = ptr.to(self.device, torch.int32)
            self.red_entry = torch.cat(red_entry).to(self.device, torch.int32)
        else:
            self.red_rows = self.red_ptr = self.red_entry = None

        # parameter-gradient slots: my flat vector -> slot [me] of every rank (own included), rows of 128 floats
        rows128 = self.n_flat // 128
        self.grad_seg_ptr = (ctypes.c_int32 * (self.world + 1))()
        for q in range(self.world):
            self.grad_seg_ptr[q + 1] = self.grad_seg_ptr[q] + rows128
        self.grad_dst = _ptr_array([self.seg.peer_ptr(q, "slots", self.rank * self.n_flat * 4) for q in range(self.world)])
        self.grad_src = _ptr_array([self.flat.data_ptr()] * self.world)
        self.flag_ptrs = _ptr_array([self.seg.peer_ptr(q, "flags") for q in range(self.world)])

    def table(self, i: int) -> torch.Tensor:
        """[own | halo] rows of table i in this rank's segment (a new view object on every call)."""
        return self.seg.view(f"bases_ext{i}", (self.n_ext[i], self.bd), self.storage_dtype)

    # -- step protocol -----------------------------------------------------------------------------------
    def begin_step(self, needs_grad: bool) -> int:
        """Start a new step of this layer: epoch += 1 after every peer is done with the halo rows of my previous
        step (CONS).  If the previous forward required grad but its backward never ran (validation outside
        `torch.no_grad()`, an exception between forward and backward), nobody raised CONS for it: raise it here -
        the program is SPMD, every rank is in the same situation - instead of stalling all ranks until the timeout."""
        if self.outstanding:
            self.signal(SLOT_CONS)
        self.wait(SLOT_CONS, lag=1, advance=True)
        self.step_id += 1
        self.outstanding = bool(needs_grad)
        return self.step_id

    def begin_backward(self, step_id: int) -> None:
        """The backward of step `step_id` is about to use the exchange buffers: they must still hold that step."""
        if step_id != self.step_id or not self.outstanding:
            raise RuntimeError(
                "egc_b200 partitioned layer: backward of a stale step - the layer ran another forward (or this backward "
                "already ran, e.g. retain_graph=True) since the forward being differentiated, and the exchange buffers "
                "(halo rows, staging) hold one step per layer.  Use a separate module per application, or run the "
                "forward again.")
        self.outstanding = False

    # -- stream-ordered primitives ---------------------------------------------------------------------
    @staticmethod
    def _stream():
        return torch.cuda.current_stream().cuda_stream

    def signal(self, *slots: int):
        mask = sum(1 << s for s in slots)
        check(_lib.load().egc_peer_signal(self.flag_ptrs, self.world, self.rank, mask, self.epoch.data_ptr(), self._stream()),
              "egc_peer_signal")

    def wait(self, slot: int, lag: int = 0, advance: bool = False):
        """(advance: a new step starts - epoch += 1 first.)  Blocks the stream until every peer's `slot` flag has
        reached epoch - lag."""
        check(_lib.load().egc_peer_wait(self.flags.data_ptr(), self.world, self.rank, slot, self.epoch.data_ptr(), lag,
                                        int(advance), self.timeout_ns, self.err.data_ptr(), self._stream()), "egc_peer_wait")

    def _push(self, n_seg, src, dst, seg_ptr, index, width, slots, fused=None):
        # fused=True: the flags are raised by the push kernel's last CTA (one system-scope fence per CTA after a CTA
        # barrier); fused=False: a separate one-warp signal kernel after the push (EGC_PEER_FUSED_SIGNAL picks, A/B)
        if fused is None:
            fused = os.environ.get("EGC_PEER_FUSED_SIGNAL", "0") == "1"
        mask = sum(1 << s for s in slots)
        check(_lib.load().egc_peer_push_rows(n_seg, src, dst, seg_ptr, index, width, self.flag_ptrs, self.world, self.rank,
                                             mask if fused else 0, self.epoch.data_ptr(), self.counter.data_ptr(),
                                             self._stream()), "egc_peer_push_rows")
        if not fused:
            self.signal(*slots)

    def _push_dma(self, table: torch.Tensor, index: torch.Tensor, counts, dst_ptrs, width: int, slots):      # width: words
        """The same transfer by the copy engine: pack the rows (egc_gather_rows, local), one contiguous copy per peer in
        the rotated order, then the flags.  No SM is busy while the bytes travel, so a compute kernel on another stream
        runs at full occupancy meanwhile (the posted-store kernel keeps 8 CTAs per SM resident for the whole transfer)."""
        lib = _lib.load()
        n = int(index.numel())
        if n:
            check(lib.egc_gather_rows(table.data_ptr(), index.data_ptr(), n, width, self.send_buf.data_ptr(), self._stream()),
                  "egc_gather_rows")
        off = 0
        for s_, nrows in enumerate(counts):
            nbytes = nrows * width * 4
            check(lib.egc_peer_copy(dst_ptrs[s_], self.send_buf.data_ptr() + off, nbytes, self._stream()), "egc_peer_copy")
            off += nbytes
        self.signal(*slots)

    def push_forward(self, dma: bool = False):
        """My basis rows -> the halo regions of the peers that need them; the kernel's last CTA raises FWD."""
        if dma:
            return self._push_dma(self.bases_ext, self.fwd_index, self.fwd_counts, self.fwd_dst_list, self.bd_words,
                                  (SLOT_FWD,))
        self._push(len(self.segments), self.fwd_src, self.fwd_dst, self.fwd_seg_ptr, self.fwd_index.data_ptr(),
                   self.bd_words, (SLOT_FWD,))

    def push_backward(self, *d_bases_ext: torch.Tensor):
        """Halo partial sums -> their owners' staging (one contiguous fp32 [own | halo] gradient per table); raises BWD
        and CONS (my halo copy of the peers' basis rows is no longer needed once the local backward passes are done)."""
        src = _ptr_array([d_bases_ext[i].data_ptr() + (self.tables[i].n_local + self.recv_off[i][q]) * self.bd * 4
                          for q, i in self.segments])
        self._push(len(self.segments), src, self.bwd_dst, self.bwd_seg_ptr, None, self.bd, (SLOT_BWD, SLOT_CONS))

    def push_t(self, dma: bool = False):
        """T exchange: the target-side stream rows my peers' source columns touch -> their stream tables; raises BWD and
        CONS (pass 1 is done: neither it nor the column pass reads my halo copy of the peers' basis rows)."""
        if dma:
            return self._push_dma(self.t_ext, self.t_index, self.t_counts, self.t_dst_list, self.t_words, (SLOT_BWD, SLOT_CONS))
        self._push(len(self.peers), self.t_src, self.t_dst, self.t_seg_ptr, self.t_index.data_ptr(), self.t_words,
                   (SLOT_BWD, SLOT_CONS))

    def reduce_into(self, d_bases_local: torch.Tensor):
        """d_bases_local (fp32, the stacked own rows of every table) += the peers' partial sums, in fixed peer order."""
        if self.red_rows is None:
            return
        check(_lib.load().egc_peer_reduce_rows(self.staging.data_ptr(), self.red_rows.data_ptr(), self.red_ptr.data_ptr(),
                                               self.red_entry.data_ptr(), self.red_rows.numel(), self.bd,
                                               d_bases_local.data_ptr(), self._stream()), "egc_peer_reduce_rows")

    def allreduce_flat(self) -> torch.Tensor:
        """Sum `self.flat` over the ranks in ONE kernel (push to every rank's slot, flag, wait, sum in rank order)."""
        check(_lib.load().egc_peer_allreduce(self.flat.data_ptr(), self.grad_dst, self.slots.data_ptr(), self.flag_ptrs,
                                             self.flags.data_ptr(), self.world, self.rank, SLOT_GRAD, self.epoch.data_ptr(),
                                             self.counter.data_ptr(), self.n_flat, self.flat_sum.data_ptr(), self.timeout_ns,
                                             self.err.data_ptr(), self._stream()), "egc_peer_allreduce")
        return self.flat_sum

    def check(self):
        """Host-side check of the device error word (synchronises)."""
        code = int(self.err.item())
        if code:
            names = {1 + SLOT_FWD: "FWD", 1 + SLOT_BWD: "BWD", 1 + SLOT_GRAD: "GRAD", 1 + SLOT_CONS: "CONS"}
            raise RuntimeError(
                f"egc_b200 peer exchange: rank {self.rank} timed out waiting for its peers' {names.get(code, code)} flag "
                f"[epoch {int(self.epoch.item())}, flags {self.flags.view(N_SLOTS, self.world).tolist()}] "
                "(a rank skipped a step or died; the waiting kernel trapped, this CUDA context is unusable)")

    def close(self):
        self.seg.close()
