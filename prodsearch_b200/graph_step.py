"""One training step -- forward, backward, gradient sinks, clipped Adam -- captured in a CUDA graph.

At batch 384 a TEM step moves a few MB and runs ~50 short kernels: launching them one by one from Python
costs more than executing them.  ``GraphedTrainStep`` runs the reference's step sequence
(trainer.py:74-78: ``loss = model(batch); zero_grad; loss.backward(); optim.step()``) once under stream
capture and replays it with new batch contents copied into static input buffers.  Everything the step
needs is device-resident and replay-safe: negatives come from the device generator (``torch.multinomial``,
Philox offsets advance per replay), dropout keys from a device seed, the Adam step counter / clip norm
live in device memory, the gradient sinks keep their touched-row lists in persistent buffers.

Capture rule inherited from torch: no autograd graph of an EARLIER eager pass over the same parameters may still be
alive (a loss tensor kept in a variable): its AccumulateGrad nodes are bound to the stream of that pass -- usually the
legacy default stream -- and the captured backward would try to run them there ("operation would make the legacy
stream depend on a capturing blocking stream").  Drop such tensors before constructing a GraphedTrainStep.
"""
import argparse

import torch

from . import _lib


class PackedBatch(object):
    """A batch as one host byte buffer in the layout of a GraphedTrainStep's static inputs (GraphedTrainStep.pack)."""

    def __init__(self, buf):
        self.buf = buf


class GraphedTrainStep(object):
    def __init__(self, model, optim, sample_batch, pad_values=None, warmup=3, sync_grads=None):
        """sample_batch: a batch whose tensor fields have the LARGEST shapes that will be fed (narrower
        batches are right-padded with ``pad_values[field]``, e.g. the word / item pad ids).
        sync_grads: optional callable run between backward and the optimizer (data-parallel reduce)."""
        self.model, self.optim = model, optim
        self.pad_values = dict(pad_values or {})
        self.static = argparse.Namespace()
        dev = next(model.parameters()).device
        # every tensor field of the batch lives in ONE device allocation (16-byte aligned slices), so that a batch packed
        # the same way on the host (``pack``) arrives with a single host -> device copy
        self._layout, off = {}, 0
        for k, v in vars(sample_batch).items():
            if torch.is_tensor(v):
                nbytes = v.numel() * v.element_size()
                self._layout[k] = (off, nbytes, tuple(v.shape), v.dtype)
                off += (nbytes + 15) // 16 * 16
        self._pack_bytes = max(off, 16)
        self._dev_pack = torch.zeros(self._pack_bytes, dtype=torch.uint8, device=dev)
        for k, v in vars(sample_batch).items():
            if torch.is_tensor(v):
                dst = self._view(self._dev_pack, k)
                dst.copy_(v)
                setattr(self.static, k, dst)
            else:
                setattr(self.static, k, v)
        self.sync_grads = sync_grads
        self._one = None
        snap = self._snapshot()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):        # allocates optimizer state, dense gradient buffers, smem attributes
                self._step_body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._restore(snap)                # the warm-up steps must not count as training
        self.graph = torch.cuda.CUDAGraph()
        n0 = _lib.launch_count()
        with torch.cuda.graph(self.graph):
            self.loss = self._step_body()
        self.launches_per_replay = _lib.launch_count() - n0   # hand-written kernels captured in the graph
        torch.cuda.synchronize()

    def _snapshot(self):
        opt = getattr(self.optim, "optimizer", None)
        snap = dict(params=[p.detach().clone() for p in self.model.parameters()], host_step=getattr(self.optim, "_step", 0),
                    opt_state=None, opt_step=None, acc=None)
        if opt is not None and hasattr(opt, "_step_dev"):
            snap["opt_state"] = {p: {k: v.clone() for k, v in st.items()} for p, st in opt.state.items()}
            snap["opt_step"] = None if opt._step_dev is None else opt._step_dev.clone()
        elif opt is not None:
            import copy
            snap["opt_state"] = copy.deepcopy(opt.state_dict())
        if getattr(self.model, "_ps_acc", None) is not None:
            snap["acc"] = (self.model._ps_acc.clone(), self.model._item_acc.clone())
        return snap

    def _restore(self, snap):
        with torch.no_grad():
            for p, v in zip(self.model.parameters(), snap["params"]):
                p.copy_(v)
            opt = getattr(self.optim, "optimizer", None)
            if opt is not None and hasattr(opt, "_step_dev"):
                if opt._step_dev is not None:
                    if snap["opt_step"] is None:
                        opt._step_dev.zero_()
                    else:
                        opt._step_dev.copy_(snap["opt_step"])
                for p, st in opt.state.items():
                    old = snap["opt_state"].get(p) or {}
                    for k, v in st.items():          # exp_avg, exp_avg_sq, (row-sparse tables) last_step
                        if k in old:
                            v.copy_(old[k])
                        elif k == "last_step":       # created by the warm-up: every row is current at the restored step
                            v.copy_(opt._step_dev.expand_as(v))
                        else:
                            v.zero_()
            elif opt is not None:
                opt.load_state_dict(snap["opt_state"])
            if hasattr(self.optim, "_step"):
                self.optim._step = snap["host_step"]
            if getattr(self.model, "_ps_acc", None) is not None:
                if snap["acc"] is None:
                    self.model._ps_acc.zero_()
                    self.model._item_acc.zero_()
                else:
                    self.model._ps_acc.copy_(snap["acc"][0])
                    self.model._item_acc.copy_(snap["acc"][1])

    def _step_body(self):
        loss = self.model(self.static)
        self.model.zero_grad()
        if self._one is None or self._one.shape != loss.shape:
            self._one = torch.ones_like(loss)
        loss.backward(self._one)           # a persistent root gradient: no fill kernel at the head of every backward pass
        if self.sync_grads is not None:
            self.sync_grads()
        self.optim.step()
        return loss.detach()

    def _view(self, buf, k):
        off, nbytes, shape, dtype = self._layout[k]
        return buf[off:off + nbytes].view(dtype).view(shape)

    def pack(self, batch, pin=True):
        """Host side of the one-copy load: the batch's tensor fields laid out (and right-padded) like the static device
        buffers in one (pinned) byte buffer.  Part of collating a batch, like pinning it; ``load`` / ``__call__`` accept
        the result."""
        buf = torch.zeros(self._pack_bytes, dtype=torch.uint8)
        if pin and torch.cuda.is_available():
            buf = buf.pin_memory()
        for k, v in vars(batch).items():
            if not torch.is_tensor(v):
                continue
            dst = self._view(buf, k)
            v = v.detach().cpu()
            if v.shape == dst.shape:
                dst.copy_(v)
                continue
            if v.dim() != dst.dim() or v.shape[0] != dst.shape[0] or any(a > b for a, b in zip(v.shape, dst.shape)):
                raise ValueError("batch field %s has shape %s, graph was captured for %s" % (k, tuple(v.shape), tuple(dst.shape)))
            if k not in self.pad_values:
                raise ValueError("no pad value for the narrower batch field " + k)
            dst.fill_(self.pad_values[k])
            dst[tuple(slice(0, n) for n in v.shape)].copy_(v)
        return PackedBatch(buf)

    def load(self, batch, non_blocking=True):
        """Copy a (host or device) batch into the static input buffers, right-padding narrower tensors.  A PackedBatch
        (``pack``) takes one copy."""
        if isinstance(batch, PackedBatch):
            if batch.buf.numel() != self._pack_bytes:
                raise ValueError("packed batch of %d bytes, graph was captured for %d" % (batch.buf.numel(), self._pack_bytes))
            self._dev_pack.copy_(batch.buf, non_blocking=non_blocking)
            return
        for k, v in vars(batch).items():
            if not torch.is_tensor(v):
                continue
            dst = getattr(self.static, k)
            if v.shape == dst.shape:
                dst.copy_(v, non_blocking=non_blocking)
                continue
            if v.dim() != dst.dim() or v.shape[0] != dst.shape[0] or any(a > b for a, b in zip(v.shape, dst.shape)):
                raise ValueError("batch field %s has shape %s, graph was captured for %s" % (k, tuple(v.shape), tuple(dst.shape)))
            if k not in self.pad_values:
                raise ValueError("no pad value for the narrower batch field " + k)
            dst.fill_(self.pad_values[k])
            dst[tuple(slice(0, n) for n in v.shape)].copy_(v, non_blocking=non_blocking)

    def __call__(self, batch=None):
        """Run one step; returns the (static, device) loss tensor of that step."""
        if batch is not None:
            self.load(batch)
        self.graph.replay()
        _lib.note_param_write()        # the replayed optimizer wrote the parameters behind autograd's back
        return self.loss
