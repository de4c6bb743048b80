"""Row-sharded embedding tables over NVLink peer memory (SURVEY.md 8(e); C ABI: the psb_peer_* block of
include/psb.h).

One process per GPU.  Every buffer a peer must read -- table shards, the compact gradient lists each rank
produces, the flat bucket of replicated dense gradients, barrier flags -- is allocated by ``PeerGroup.alloc``,
exported as a CUDA IPC handle, exchanged once through ``torch.distributed`` (plumbing) and mapped by every
other rank.  From then on the exchange steps are loads inside hand-written kernels:

  fetch   ``PeerShardedTable.fetch``: out[i] = shard[id % G][id / G]  (psb_peer_gather_rows) into a small
          local *mini table*; the unchanged single-GPU fused kernels then run on it with remapped indices
  push    the table's sink (a ``functional.RowGradSink`` in "stage" mode) runs the usual deterministic sort +
          segmented reduce over GLOBAL row ids into a peer-visible compact list (rows, values, count)
  fold    after a barrier every owner folds the slots it owns of each peer's list, peer by peer in rank order,
          into its dense shard gradient (psb_peer_fold_lists: two launches whatever G is): reproducible, no
          float atomics, no second sort
  dense   replicated parameters: one-shot all-reduce over the peers' flat buckets (psb_peer_allreduce)

Nothing here synchronises with the host, so ``model(batch); backward; sync_grads; optim.step`` is captured
and replayed as ONE CUDA graph per rank (graph_step.GraphedTrainStep).  For the unit tests several ranks can be
simulated inside one process on one GPU (``PeerGroup.simulate``): the kernels only see pointer arrays.
"""
import ctypes

import torch

from . import _lib
from . import functional as F_
from ._lib import c_vp, check, load, stream_ptr


class _Raw(object):
    """Raw device allocation exposed to torch through __cuda_array_interface__."""

    def __init__(self, ptr, nbytes, owner=None):
        self.ptr, self.nbytes, self.owner = ptr, nbytes, owner
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def _as_tensor(ptr, nbytes, device, keep):
    t = torch.as_tensor(_Raw(ptr, nbytes, keep), device=device)
    return t


class PeerBuffer(object):
    """One symmetric allocation: ``local`` (uint8 tensor view of this rank's copy) and the device pointers of
    every rank's copy (``ptrs``), usable from this rank's kernels."""

    def __init__(self, group, seq, ptr, nbytes):
        self.group, self.seq, self.ptr, self.nbytes = group, seq, ptr, nbytes
        self.local = _as_tensor(ptr, nbytes, group.device, self)
        self._ptrs = None

    @property
    def ptrs(self):
        if self._ptrs is None:
            self._ptrs = self.group._resolve(self)
        return self._ptrs

    def ptr_array(self, offset=0):
        """HOST array of G device pointers (ctypes), each advanced by ``offset`` bytes."""
        return (c_vp * len(self.ptrs))(*[p + offset for p in self.ptrs])

    def view(self, dtype, shape, offset=0):
        n = 1
        for s in shape:
            n *= s
        nb = n * torch.empty((), dtype=dtype).element_size()
        return self.local[offset:offset + nb].view(dtype).view(shape)


class _SimHub(object):
    """Shared registry of the simulated ranks of one process (tests)."""

    def __init__(self, world):
        self.world, self.table = world, {}


class PeerGroup(object):
    def __init__(self, group=None, device=None, _sim=None, _rank=None):
        import torch.distributed as dist
        self._sim = _sim
        if _sim is not None:
            self.world, self.rank = _sim.world, _rank
        else:
            self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > _lib.PEER_MAX:
            raise RuntimeError("PeerGroup: at most %d ranks" % _lib.PEER_MAX)
        self.group = group
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._seq = 0
        self._opened = []
        self.flags = self.alloc(4 * _lib.PEER_MAX)
        self.epoch = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.err = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.wait_cycles = torch.zeros(4, dtype=torch.int64, device=self.device)   # per barrier call site (slot)
        self.timeout_cycles = 0

    @classmethod
    def simulate(cls, world, device="cuda"):
        """``world`` ranks inside this process, all on ``device`` (unit tests of the kernels and host logic)."""
        hub = _SimHub(world)
        return [cls(device=device, _sim=hub, _rank=r) for r in range(world)]

    # ---- allocation (collective: every rank calls alloc in the same order with the same size) -------------
    def alloc(self, nbytes):
        # Sizes are rounded up to whole 2 MiB pages.  Measured on B200 / NVLink 5 (profiles/r02n_alloc_probe.jsonl): a
        # 4 GB cudaMalloc whose size is NOT a multiple of 64 KiB is mapped into the peers (CUDA IPC) with small pages
        # and 128-bit row loads from it run at 40 GB/s instead of 630 GB/s -- the "PCIe-class" peer gather of round 1
        # was this, not the kernel and not the link (same kernel, same ids: 6.34 ms vs 0.42 ms per 1M rows).
        nbytes = int(nbytes)
        gran = (2 << 20) if nbytes >= (1 << 20) else 256
        nbytes = (nbytes + gran - 1) // gran * gran
        out = c_vp()
        with torch.cuda.device(self.device):
            check(load().psb_peer_alloc(nbytes, ctypes.byref(out)), "psb_peer_alloc")
        buf = PeerBuffer(self, self._seq, out.value, nbytes)
        self._seq += 1
        if self._sim is not None:
            self._sim.table[(buf.seq, self.rank)] = buf.ptr
        elif self.world > 1:
            buf._ptrs = self._exchange(buf)
        else:
            buf._ptrs = [buf.ptr]
        return buf

    def _resolve(self, buf):
        if self._sim is None:
            return buf._ptrs
        return [self._sim.table[(buf.seq, r)] for r in range(self.world)]

    def _exchange(self, buf):
        import torch.distributed as dist
        handle = ctypes.create_string_buffer(_lib.PEER_HANDLE_BYTES)
        check(load().psb_peer_export(buf.ptr, handle), "psb_peer_export")
        handles = [None] * self.world
        dist.all_gather_object(handles, (self.rank, buf.seq, buf.nbytes, handle.raw), group=self.group)
        ptrs = []
        for r, (rr, seq, nb, raw) in enumerate(handles):
            if rr != r or seq != buf.seq or nb != buf.nbytes:
                raise RuntimeError("PeerGroup.alloc called out of step across ranks")
            if r == self.rank:
                ptrs.append(buf.ptr)
                continue
            out = c_vp()
            check(load().psb_peer_open(raw, ctypes.byref(out)), "psb_peer_open (CUDA IPC / NVLink P2P)")
            self._opened.append(out.value)
            ptrs.append(out.value)
        return ptrs

    # ---- synchronisation ----------------------------------------------------------------------------------
    def barrier(self, slot=0):
        """Stream-ordered barrier of all ranks (graph-capturable); ``slot`` (0..3) names the call site in the
        ``wait_cycles`` statistics.  The simulated ranks of one process share
        a stream and are driven phase by phase in lockstep by the tests, so stream order already is the barrier."""
        if self.world == 1 or self._sim is not None:
            return
        check(load().psb_peer_barrier(self.flags.ptr_array(), self.rank, self.world, self.epoch.data_ptr(),
                                      self.err.data_ptr(), int(self.timeout_cycles), self.wait_cycles.data_ptr(),
                                      int(slot), stream_ptr()),
              "psb_peer_barrier")

    def fold_stamp(self):
        """Device pointer of a uint32 that is constant during one fold and new for the next: the barrier epoch
        (two barriers separate consecutive folds); the simulated ranks, whose barrier is stream order, bump a
        private counter instead."""
        if self._sim is None and self.world > 1:
            return self.epoch.data_ptr()
        if not hasattr(self, "_stamp"):
            self._stamp = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._stamp.add_(1)
        return self._stamp.data_ptr()

    def check_errors(self):
        """Host-synchronising check of the barrier time-out flag."""
        e = int(self.err.item())
        if e:
            raise RuntimeError("peer barrier timed out waiting for rank %d" % (e - 1))

    def allreduce(self, buf, n, out, scale=1.0, offset=0):
        """out[:n] = scale * sum over ranks of the fp32 vectors at ``offset`` of the symmetric ``buf``."""
        check(load().psb_peer_allreduce(buf.ptr_array(offset), self.world, self.rank, int(n), float(scale), out.data_ptr(),
                                        stream_ptr()), "psb_peer_allreduce")
        return out


def try_create(group=None, device=None):
    """PeerGroup of ``group`` if CUDA IPC + P2P work between all its ranks, else None -- the same answer on every
    rank (callers fall back to the NCCL all-to-all transport of sharded.py)."""
    import torch.distributed as dist
    pg, ok = None, 1
    try:
        pg = PeerGroup(group, device)
    except RuntimeError as ex:
        ok = 0
        import sys
        sys.stderr.write("peer memory unavailable on rank %d: %s\n" % (dist.get_rank(group), ex))
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    t = torch.tensor([ok], dtype=torch.int32, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    return pg if int(t.item()) == 1 else None


class PeerShardedTable(object):
    """A [rows, d] fp32 table row-sharded cyclically (owner = id % G, local row = id // G)."""

    def __init__(self, rows, d, peer, pad_idx, full=None, bias=None, stage_cap=0, sparse=False):
        """sparse: the owners update their shard with the row-sparse lazily caught-up Adam (optimizers.FusedAdam): the
        moments and the per-row step stamps live in peer memory next to the shard, because a reader brings a resting
        row up to date on the fly (psb_peer_gather_rows_lazy) and needs them."""
        self.rows, self.d, self.peer, self.pad_idx = int(rows), int(d), peer, int(pad_idx)
        G, r = peer.world, peer.rank
        self.local_rows = (self.rows - r + G - 1) // G
        per = max((self.rows + G - 1) // G, 1)
        self.shard = peer.alloc(per * d * 4)    # the same size on every rank
        self.sparse = bool(sparse)
        self.lazy_optim = None                  # the FusedAdam whose step counter / coefficient history the fetch reads
        if self.sparse:
            self._m_buf, self._v_buf, self._last_buf = peer.alloc(per * d * 4), peer.alloc(per * d * 4), peer.alloc(per * 4)
            self.exp_avg = self._m_buf.view(torch.float32, (self.local_rows, d))
            self.exp_avg_sq = self._v_buf.view(torch.float32, (self.local_rows, d))
            self.last_step = self._last_buf.view(torch.int32, (self.local_rows,))
        w = self.shard.view(torch.float32, (self.local_rows, d))
        if full is not None:
            with torch.no_grad():
                w.copy_(full[r::G].to(w.device))
        self.weight = torch.nn.Parameter(w)
        self.grad = torch.zeros_like(w)                    # dense shard gradient (what Adam reads)
        self.bias = bias                                   # replicated bias vector indexed like the table
        # contributions arrive as mini-table positions (fetch hands the sink their global ids); the reduced rows go
        # into the staging list the owners fold
        self.sink = F_.RowGradSink(self.weight, self.pad_idx, bias, "stage", rows=self.rows)
        self._stage = None
        self._cap = 0
        self._posmap = None
        if stage_cap:
            self._ensure_stage(stage_cap)

    # staging layout (peer-visible): [n_rows int32 | pad to 256][rows int32 cap][vals fp32 cap x d]
    def _ensure_stage(self, cap):
        if self._stage is not None:
            raise RuntimeError("the gradient staging list is sized once (stage_cap / the first step)")
        cap = (cap + 63) // 64 * 64
        self._off_rows = 256
        self._off_vals = 256 + cap * 4
        self._stage = self.peer.alloc(self._off_vals + cap * self.d * 4)   # collective
        self._cap = cap
        self.stage_n = self._stage.view(torch.int32, (1,), 0)
        self.stage_rows = self._stage.view(torch.int32, (cap,), self._off_rows)
        self.stage_vals = self._stage.view(torch.float32, (cap, self.d), self._off_vals)
        self.sink.stage = (self.stage_rows, self.stage_n, self.stage_vals)

    def reserve_stage(self, cap):
        """Size the peer-visible gradient list for ``cap`` contribution slots per step.  Collective (and
        host-synchronising) when it has to grow, free otherwise; growing inside graph capture is an error."""
        if self._stage is None:
            if self.peer.world > 1 and self.peer._sim is None:     # ragged batches: agree on the largest request
                import torch.distributed as dist
                t = torch.tensor([int(cap)], dtype=torch.int64, device=self.peer.device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.peer.group)
                cap = int(t.item())
            self._ensure_stage(cap)

    def fetch(self, index_tensors, stream=None):
        """Gather the rows of ``index_tensors`` (global ids) from their owners into a local mini table.
        Returns (mini [n+1, d], remapped index tensors, pad position): positions of pad ids are remapped to
        the single position n (which holds the pad row), so kernels keep their ``idx != pad_idx`` validity rule.
        stream: run the P2P gather on this side stream (forked from the current one; buffers are allocated on the
        current stream); the CALLER joins it -- ``current_stream().wait_stream(stream)`` -- before the first use."""
        flats = [t.reshape(-1) for t in index_tensors]
        n = sum(f.numel() for f in flats)
        dev = self.weight.device
        pad_t = getattr(self, "_pad_t", None)
        if pad_t is None:
            pad_t = self._pad_t = torch.full((1,), self.pad_idx, dtype=torch.int64, device=dev)
        ids = torch.cat(flats + [pad_t])
        mini = torch.empty((n + 1, self.d), dtype=torch.float32, device=dev)
        remap = torch.empty((n + 1,), dtype=torch.int64, device=dev)
        if stream is not None:
            stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream(dev)):
            opt = self.lazy_optim
            if self.sparse and opt is not None and opt._step_dev is not None:
                lr, b1, b2, eps = opt._hyper()
                check(load().psb_peer_gather_rows_lazy(
                    self.shard.ptr_array(), self._m_buf.ptr_array(), self._v_buf.ptr_array(), self._last_buf.ptr_array(),
                    self.peer.world, self.rows, self.d, ids.data_ptr(), n + 1, mini.data_ptr(), remap.data_ptr(),
                    self.pad_idx, n, None, lr, b1, b2, eps, 1 if opt._last_noam else 0, float(opt._last_warmup),
                    opt._step_dev.data_ptr(), opt._coef_hist.data_ptr() if opt._coef_hist is not None else None,
                    opt.coef_cap, stream_ptr()), "psb_peer_gather_rows_lazy")
            else:
                check(load().psb_peer_gather_rows(self.shard.ptr_array(), self.peer.world, self.rows, self.d,
                                                  ids.data_ptr(), n + 1, mini.data_ptr(), remap.data_ptr(), self.pad_idx, n,
                                                  None, stream_ptr()), "psb_peer_gather_rows")
        # a leaf that requires grad, so the autograd Functions reading it run their backward (which routes the row
        # gradients to the sink; nothing is ever accumulated into mini.grad)
        mini.requires_grad_(self.weight.requires_grad and torch.is_grad_enabled())
        outs, off = [], 0
        origin = {}
        for t, f in zip(index_tensors, flats):
            r = remap[off:off + f.numel()].view(t.shape)
            outs.append(r)
            origin[r.data_ptr()] = f
            off += f.numel()
        self.sink.begin(ids, origin)
        return mini, outs, n

    def fold(self, scale):
        fold_tables([self], scale)

    def _fold_desc(self):
        """psb_fold_table_t of this table; clears the rows the previous fold wrote."""
        from . import ops
        G = self.peer.world
        if self._posmap is None:
            self._posmap = torch.zeros(G * self.local_rows, dtype=torch.int64, device=self.weight.device)
            self._rowwise_zero = self.sparse or self.grad.numel() * 4 > (64 << 20)   # big shard: clear touched rows, not a memset
            if self._rowwise_zero:
                self._touched = torch.zeros(G * self._cap, dtype=torch.int32, device=self.weight.device)
                self._n_touched = torch.zeros(1, dtype=torch.int32, device=self.weight.device)
        if self.sparse:
            self._n_touched.zero_()      # only the rows of THIS fold's list are ever read: nothing to clear
        elif self._rowwise_zero:
            ops.zero_rows(self._touched, self._n_touched, self.d, self.grad, None)
            self._n_touched.zero_()
        else:
            self.grad.zero_()
        t = _lib.FoldTable()
        st = self._stage
        for r in range(G):
            base = st.ptrs[r]
            t.rows[r], t.vals[r], t.n_rows[r] = base + self._off_rows, base + self._off_vals, base
        t.cap, t.d, t.shard_rows = self._cap, self.d, self.local_rows
        t.posmap, t.dense = self._posmap.data_ptr(), self.grad.data_ptr()
        t.touched = self._touched.data_ptr() if self._rowwise_zero else None
        t.n_touched = self._n_touched.data_ptr() if self._rowwise_zero else None
        return t


def fold_tables(tables, scale):
    """Owner side, after the barrier: for up to two tables at once, shard gradient = scale * (rank-ordered sum over
    the peers' compact lists of the rows this rank owns); two launches in total (psb_peer_fold_lists)."""
    peer = tables[0].peer
    arr = (_lib.FoldTable * len(tables))(*[t._fold_desc() for t in tables])
    check(load().psb_peer_fold_lists(arr, len(tables), peer.rank, peer.world, float(scale), peer.fold_stamp(),
                                     stream_ptr()), "psb_peer_fold_lists")
    for t in tables:
        if t.sparse:                     # (rows the fold wrote, the dense shard gradient they index, their count)
            t.weight.grad = None
            t.weight.row_grad = (t._touched, t.grad, t._n_touched)
            t.weight._psb_grad_by_row = True
            t.weight._psb_drop_idx = t.pad_idx // peer.world if t.pad_idx % peer.world == peer.rank else -1
        else:
            t.weight.grad = t.grad


class DenseBucket(object):
    """Flat peer-visible bucket of the replicated parameters' gradients + the one-shot all-reduce."""

    def __init__(self, peer, params):
        self.peer = peer
        self.params = list(params)
        self.n = sum(p.numel() for p in self.params)
        n_pad = (self.n + 3) // 4 * 4
        self.buf = peer.alloc(n_pad * 4)
        self.flat = self.buf.view(torch.float32, (n_pad,))
        self.red = torch.zeros(n_pad, dtype=torch.float32, device=peer.device)
        self.views, off = [], 0
        for p in self.params:
            self.views.append(self.red[off:off + p.numel()].view(p.shape))
            off += p.numel()

    def stage(self):
        """Copy the local gradients into the bucket (before the barrier)."""
        zeros = None
        parts = []
        for p in self.params:
            if p.grad is None:
                if zeros is None:
                    zeros = {}
                z = zeros.get(p.numel())
                if z is None:
                    z = zeros[p.numel()] = torch.zeros(p.numel(), dtype=torch.float32, device=self.peer.device)
                parts.append(z)
            else:
                parts.append(p.grad.reshape(-1))
        torch.cat(parts, out=self.flat[:self.n])

    def reduce(self):
        """After the barrier: mean over ranks into the local reduced bucket; gradients become views of it."""
        self.peer.allreduce(self.buf, self.flat.numel(), self.red, scale=1.0 / self.peer.world)
        for p, v in zip(self.params, self.views):
            p.grad = v
