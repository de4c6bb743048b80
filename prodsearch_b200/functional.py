"""Autograd surface over the C-ABI ops: the piece that lets ``loss.backward()`` in the
reference's trainer (trainer.py:77) drive the sm_100a kernels.

Embedding-table gradients never flow through autograd as dense [rows, d] tensors (the
reference's embedding_dense_backward, SURVEY.md 0.6).  Each op *registers a contribution*
(indices + source rows + per-slot scales) with the table's ``RowGradSink``; when the backward
pass finishes, one deterministic sort + segmented-reduce per table (psb_scatter_reduce_rows)
produces the gradient, either scattered into a persistent dense ``.grad`` (drop-in for the
reference's dense Adam), kept row-sparse as ``param.row_grad = (rows, values, n_rows)``, or written into the
caller-owned staging list a peer-sharded table's owners fold (peer.py).
"""
import torch
from torch.autograd import Function, Variable

from . import ops


def run_forked(sink):
    """Run ``sink.finalize()`` on the sink's own side stream, forked from the stream ``backward()`` runs on; one
    extra engine callback (queued by the first forked sink, so it runs after every finalize callback already queued)
    joins all side streams back before ``backward()`` returns.  Inside a captured CUDA graph the chains become
    parallel branches.  ``sink`` needs ``weight``, ``_pending``, ``_stream``, ``_hold`` and ``finalize()``."""
    dev = sink.weight.device
    cur = torch.cuda.current_stream(dev)
    if sink._stream is None:
        sink._stream = torch.cuda.Stream(device=dev)
    sink._stream.wait_stream(cur)
    sink._hold = list(sink._pending)              # contribution tensors stay alive until the join
    first = not RowGradSink._forked
    RowGradSink._forked.append(sink)
    try:
        with torch.cuda.stream(sink._stream):
            sink.finalize()
    except Exception:
        RowGradSink._forked.remove(sink)
        sink._hold = None
        raise
    if first:
        Variable._execution_engine.queue_callback(RowGradSink._join_forked)


class RowGradSink(object):
    """Gradient collector for one embedding table (and the bias vector indexed like it).

    ``rows``: the id space the sort runs over (and ``drop_idx`` is in), ``weight.shape[0]`` unless the table holds a
    share of the rows (peer-sharded: global ids).  ``mode``: the reduced rows go into a persistent ``weight.grad``
    ("dense"), ``weight.row_grad`` ("rowsparse") or the owner's staging list ``stage = (rows int32 [cap], count int32
    [1], values fp32 [cap, d])``, set before the first step ("stage"; the bias gradient is a dense vector).

    The sort + segmented reduce of different tables are independent, and at batch 384 each is a chain of short,
    narrow launches (one CTA of counting sort, then the reduce): every sink of a CUDA table runs its chain on its own
    side stream, forked from and joined back into the stream ``backward()`` ran on, so the chains of the item and the
    word table overlap (inside a captured CUDA graph they become parallel branches)."""

    _forked = []                      # sinks whose chain is in flight on a side stream (not yet joined)
    _seq = 0                          # global order of expect() / mark_forward_end() calls
    _fwd_mark = {}                    # device -> (event recorded when a model's forward pass ended, its sequence number)

    @staticmethod
    def mark_forward_end(device):
        """A model calls this when its forward pass is complete and every side stream has been joined into the current
        one: an event recorded here covers the producers of ALL index lists announced so far (sampled negatives
        included), so the sinks' sorts can start behind it instead of behind whatever backward has enqueued by the
        time the first contribution arrives."""
        dev = torch.device(device)
        mark = RowGradSink._fwd_mark.get(dev)
        ev = mark[0] if mark is not None else torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        RowGradSink._seq += 1
        RowGradSink._fwd_mark[dev] = (ev, RowGradSink._seq)

    def __init__(self, weight, drop_idx=-1, bias=None, mode="dense", rows=None):
        self.weight = weight
        self.bias = bias
        self.drop_idx = drop_idx
        self.mode = mode              # "dense" | "rowsparse" | "stage"
        self.rows = weight.shape[0] if rows is None else int(rows)
        self.stage = None
        self.ids = None               # begin(): the row id of every position of the fetched mini table
        self._origin = None
        self._pending = []
        self._queued = False
        self._dense = None
        self._dense_bias = None
        self._prev = None             # (unique_rows, n_unique) written into the dense buffers last time
        self._uniq_buf = None         # persistent: a CUDA-graph replay reads last replay's rows from here
        self._nu_buf = None
        self._stream = None
        self._hold = None
        self._expected = []           # index tensors the forward pass announced (expect), in forward order
        self._exp_event = None
        self._sort_stream = None
        self._sort_done = None
        self._presort = None          # dict(exp, ws, uniq, nu, cleared) of the sort launched for this step
        self._sort_bufs = None
        self._last_seq = 0

    def begin(self, ids, origin):
        """A fetch handed out a mini table: contributions now index its positions, and position p is row ``ids[p]``.
        ``origin`` maps each index tensor the fetch returned (by data pointer) to the row ids it was remapped from."""
        self.ids, self._origin = ids, origin
        self._expected = []

    def _origin_of(self, idx):
        g = self._origin.get(idx.data_ptr())
        return g if g is not None and g.numel() == idx.numel() else None

    # -- called from Function.forward ---------------------------------------------------
    def expect(self, idx):
        """Announce an index list that backward will contribute with.  The sort of a step's contributions only needs
        the index lists, and those all exist when the forward pass ends: at the first contribution of the backward
        pass the sink sorts the announced lists on its own stream -- ordered behind the forward pass only, so it runs
        NEXT TO the backward kernels -- and finalize() is left with the segmented reduce.  If what backward delivers
        does not match what forward announced (a branch without gradient, a second forward), finalize() falls back to
        the one-call sort + reduce; the result is the same.  So does a step with more lists than one sort takes, or
        with an index list the fetch (begin) did not hand out."""
        if not (self.weight.is_cuda and self.weight.requires_grad) or self._expected is None:
            return
        if self._origin is not None:
            idx = self._origin_of(idx)
            if idx is None:
                self._expected = None
                return
        t = ops._idx(idx).reshape(-1)
        if t.numel() == 0:
            return
        if len(self._expected) >= ops._lib.MAX_CONTRIBS:
            self._expected = None
            return
        self._expected.append(t)
        RowGradSink._seq += 1
        self._last_seq = RowGradSink._seq

    def _launch_presort(self):
        exp, w = self._expected, self.weight
        if self.mode == "dense" and w.grad is not None and w.grad is self._dense:
            return                                   # gradient accumulation: finalize() takes its own path
        dev = w.device
        n_total = sum(t.numel() for t in exp)
        if self.mode == "stage" and (self.stage is None or n_total > self.stage[0].numel()):
            return                                   # finalize() raises
        if self._sort_stream is None:
            self._sort_stream = torch.cuda.Stream(device=dev)
            self._sort_done = torch.cuda.Event()
        bufs = self._sort_bufs
        wb = ops.scatter_workspace_bytes(n_total, self.rows)
        if bufs is None or bufs[0].numel() < wb or bufs[1].numel() < n_total:
            if self._prev is not None and self._prev != "all" and bufs is not None and self._prev[0] is bufs[1]:
                self._prev = "all"               # the old row list goes away with its buffer: next clear is a memset
            ws = torch.empty(wb, dtype=torch.uint8, device=dev)
            if self.mode == "stage":             # the sort writes the staging list's rows and count (sized once)
                bufs = (ws,) + tuple(self.stage[:2])
            else:
                bufs = (ws, torch.empty(max(n_total, 1), dtype=torch.int32, device=dev),
                        torch.zeros(1, dtype=torch.int32, device=dev))
            self._sort_bufs = bufs
        ws, uniq, nu = bufs
        st = self._sort_stream
        # behind the end of the forward pass when the model marked it after this sink's last announcement, else
        # behind everything enqueued so far (still correct, less overlap)
        mark = RowGradSink._fwd_mark.get(dev)
        if mark is not None and mark[1] >= self._last_seq:
            st.wait_event(mark[0])
        else:
            if self._exp_event is None:
                self._exp_event = torch.cuda.Event()
            self._exp_event.record(torch.cuda.current_stream(dev))
            st.wait_event(self._exp_event)
        cleared = False
        with torch.cuda.stream(st):
            if self.mode == "dense":    # clear last step's rows of the persistent gradient buffers here, off the critical
                # path -- and BEFORE the sort overwrites the row list they are cleared by (a CUDA-graph replay finds
                # the previous replay's rows in the same buffer)
                self._prepare_dense(self.bias is not None and self._dense_bias is not None, clear=True)
                cleared = True
            nu.zero_()
            ops.scatter_sort(exp, self.rows, self.drop_idx, ws, uniq, nu)
            self._sort_done.record(st)
        self._presort = dict(exp=exp, ws=ws, uniq=uniq, nu=nu, cleared=cleared)

    # -- called from Function.backward ------------------------------------------------
    def add(self, idx, src, src_row=None, src_div=1, scale=None, scale2=None, scale2_div=1, to_bias=False):
        if not self.weight.requires_grad and not (to_bias and self.bias is not None and self.bias.requires_grad):
            return
        if self._origin is not None:
            g = self._origin_of(idx)
            idx = g if g is not None else self.ids[idx.reshape(-1)]
        self._pending.append(ops.make_contrib(idx, src, src_row, src_div, scale, scale2, scale2_div,
                                              to_bias and self.bias is not None))
        if not self._queued:
            self._queued = True
            Variable._execution_engine.queue_callback(self._finalize_callback)
            if self._expected and self._presort is None:
                self._launch_presort()

    def _finalize_callback(self):
        if not self.weight.is_cuda:
            return self.finalize()
        run_forked(self)

    @staticmethod
    def _join_forked():
        forked, RowGradSink._forked = RowGradSink._forked, []
        for sink in forked:
            torch.cuda.current_stream(sink.weight.device).wait_stream(sink._stream)
            sink._hold = None

    # -- runs once, after the whole backward graph has executed --------------------------
    def finalize(self):
        self._queued = False
        pending, self._pending = self._pending, []
        ps, self._presort, self._expected = self._presort, None, []
        if ps is not None:            # join the sort stream whatever happens next (a captured graph needs it joined)
            torch.cuda.current_stream(self.weight.device).wait_event(self._sort_done)
        if not pending:
            return
        w = self.weight
        rows, d = self.rows, w.shape[1]
        want_bias = self.bias is not None and any(c.to_bias for c, _ in pending)
        if self.mode == "stage":
            self._prepare_stage(pending, want_bias)
        if ps is not None and self._finalize_presorted(ps, pending, rows, d, want_bias):
            return
        if ps is not None and ps["cleared"]:
            self._prev = None         # the persistent buffers were already cleared next to the sort
        for lo in range(0, len(pending), ops._lib.MAX_CONTRIBS):
            chunk = pending[lo:lo + ops._lib.MAX_CONTRIBS]
            first = lo == 0
            if self.mode == "dense":
                if not first:
                    raise RuntimeError("more than %d contributions to one table in a step" % ops._lib.MAX_CONTRIBS)
                # A second backward() without zero_grad (micro-batch accumulation, two losses sharing a table):
                # param.grad IS the persistent buffer and holds the earlier gradient -- reduce this pass into a
                # scratch buffer and add it, as AccumulateGrad does for the dense parameters.
                acc_w = w.grad is not None and w.grad is self._dense
                acc_b = want_bias and self.bias.grad is not None and self.bias.grad is self._dense_bias
                if acc_w or acc_b:
                    self._accumulate_dense(chunk, rows, d, want_bias)
                    continue
                self._prepare_dense(want_bias, clear=first)
                n_total = sum(int(c.n) for c, _ in chunk)
                if self._uniq_buf is None or self._uniq_buf.numel() < n_total:
                    self._uniq_buf = torch.empty(max(n_total, 1), dtype=torch.int32, device=w.device)
                    self._nu_buf = torch.zeros(1, dtype=torch.int32, device=w.device)
                uniq, _, _, nu = ops.scatter_reduce(chunk, rows, d, self.drop_idx, dense_grad=self._dense,
                                                    dense_bias_grad=self._dense_bias if want_bias else None,
                                                    want_rows=False, device=w.device, out_uniq=self._uniq_buf,
                                                    out_nu=self._nu_buf)
                self._prev = (uniq, nu)
                self._attach(w, self._dense)
                if want_bias:
                    self._attach(self.bias, self._dense_bias)
            elif self.mode == "stage":
                ops.scatter_reduce(chunk, rows, d, self.drop_idx, dense_bias_grad=self._dense_bias if want_bias else None,
                                   want_rows=True, device=w.device, out_uniq=self.stage[0], out_nu=self.stage[1],
                                   out_red=self.stage[2])
            else:
                uniq, red, redb, nu = ops.scatter_reduce(chunk, rows, d, self.drop_idx, want_rows=True,
                                                         want_bias=want_bias, device=w.device)
                w.row_grad = (uniq, red, nu)
                w._psb_drop_idx = self.drop_idx          # the row-sparse optimizer never replays the pad row
                if want_bias:
                    self.bias.row_grad = (uniq, redb, nu)
                    w._psb_row_bias = self.bias          # updated with (and stamped like) the table's rows

    def _finalize_presorted(self, ps, pending, rows, d, want_bias):
        """Reduce over the sort launched at the start of backward.  The contributions are put into the order the
        forward pass announced their index lists in; any mismatch -> False (the caller runs the one-call path)."""
        exp = ps["exp"]
        if len(pending) != len(exp):
            return False
        left = list(pending)
        ordered = []
        for t in exp:
            hit = None
            for j, (c, _) in enumerate(left):
                if c.idx == t.data_ptr() and int(c.n) == t.numel():
                    hit = j
                    break
            if hit is None:
                return False
            ordered.append(left.pop(hit))
        w = self.weight
        if self.mode == "dense":
            if w.grad is not None and w.grad is self._dense:
                return False
            if not ps["cleared"]:
                self._prepare_dense(want_bias, clear=True)
            elif want_bias and self._dense_bias is None:
                self._dense_bias = torch.zeros_like(self.bias)
            ops.scatter_reduce_sorted(ordered, rows, d, self.drop_idx, ps["ws"], ps["uniq"], ps["nu"],
                                      dense_grad=self._dense, dense_bias_grad=self._dense_bias if want_bias else None)
            self._prev = (ps["uniq"], ps["nu"])
            self._attach(w, self._dense)
            if want_bias:
                self._attach(self.bias, self._dense_bias)
        elif self.mode == "stage":
            ops.scatter_reduce_sorted(ordered, rows, d, self.drop_idx, ps["ws"], ps["uniq"], ps["nu"],
                                      dense_bias_grad=self._dense_bias if want_bias else None, want_rows=True,
                                      out_red=self.stage[2])
        else:
            red, redb = ops.scatter_reduce_sorted(ordered, rows, d, self.drop_idx, ps["ws"], ps["uniq"], ps["nu"],
                                                  want_rows=True, want_bias=want_bias)
            w.row_grad = (ps["uniq"], red, ps["nu"])
            w._psb_drop_idx = self.drop_idx
            if want_bias:
                self.bias.row_grad = (ps["uniq"], redb, ps["nu"])
                w._psb_row_bias = self.bias
        return True

    def _accumulate_dense(self, chunk, rows, d, want_bias):
        """Gradient accumulation into the persistent buffers: row-sparse reduce of this pass, then a deterministic
        indexed add (every row occurs once in the reduced list).  The touched-row list of the buffers is now a
        union nobody tracks, so the next clear is a full memset."""
        w = self.weight
        uniq, red, redb, nu = ops.scatter_reduce(chunk, rows, d, self.drop_idx, want_rows=True, want_bias=want_bias,
                                                 device=w.device)
        n = int(nu.item())
        r = uniq[:n].long()
        if w.grad is None:                 # only the bias was accumulating
            self._prepare_dense(False, clear=True)
            self._dense.index_add_(0, r, red[:n])
            w.grad = self._dense
        else:
            w.grad.index_add_(0, r, red[:n])
        if want_bias:
            if self.bias.grad is None:
                if self._dense_bias is None:
                    self._dense_bias = torch.zeros_like(self.bias)
                else:
                    self._dense_bias.zero_()
                self._dense_bias.index_add_(0, r, redb[:n])
                self.bias.grad = self._dense_bias
            else:
                self.bias.grad.index_add_(0, r, redb[:n])
        self._prev = "all"

    def _prepare_dense(self, want_bias, clear):
        w = self.weight
        if self._dense is None:
            self._dense = torch.zeros_like(w)
            self._prev = None
        if want_bias and self._dense_bias is None:
            self._dense_bias = torch.zeros_like(self.bias)
        if clear and self._prev is not None:
            uniq, nu = self._prev if self._prev != "all" else (None, None)
            if uniq is None or w.numel() * 4 <= (64 << 20):       # small table: a memset beats a row list
                self._dense.zero_()
                if self._dense_bias is not None:
                    self._dense_bias.zero_()
            else:
                ops.zero_rows(uniq, nu, w.shape[1], self._dense, self._dense_bias)
            self._prev = None

    def _prepare_stage(self, pending, want_bias):
        if len(pending) > ops._lib.MAX_CONTRIBS:
            raise RuntimeError("more than %d contributions to one table in a step" % ops._lib.MAX_CONTRIBS)
        n_total, cap = sum(int(c.n) for c, _ in pending), self.stage[0].numel() if self.stage is not None else 0
        if n_total > cap:
            raise RuntimeError("gradient staging list too small (%d slots, %d needed): call reserve_stage with the "
                               "largest step first" % (cap, n_total))
        if want_bias:
            if self._dense_bias is None:
                self._dense_bias = torch.empty_like(self.bias)
            self._dense_bias.zero_()
            self.bias.grad = self._dense_bias     # replaced: this mode has no gradient accumulation

    @staticmethod
    def _attach(param, buf):
        if param.grad is None or param.grad is buf:
            param.grad = buf
        else:                          # user-side gradient accumulation: keep torch semantics
            param.grad = param.grad + buf


class LazyFlushMixin(object):
    """nn.Module mixin: tables updated by the row-sparse optimizer are made dense-equivalent before anything reads
    them wholesale -- switching to eval mode (ranking, scoring candidate lists, the review table) and
    ``state_dict()`` (checkpoints)."""

    def flush_lazy_rows(self):
        done = False
        for p in self.parameters():
            lazy = getattr(p, "_psb_lazy", None)
            if lazy is not None:
                lazy.flush()
                done = True
        if done:
            ops._lib.note_param_write()

    def train(self, mode=True):
        if not mode:
            self.flush_lazy_rows()
        return super().train(mode)

    def state_dict(self, *args, **kwargs):
        self.flush_lazy_rows()
        return super().state_dict(*args, **kwargs)


def _expect(sink, idx):
    fn = getattr(sink, "expect", None)
    if fn is not None:
        fn(idx)


_ONES = {}


def _dropout_keep(shape, p, training, device):
    """Dropout mask already scaled by 1/(1-p) (None when inactive): ONE launch -- dropout of a cached tensor of ones
    (a Bernoulli draw followed by a division would be two, at the head of the step's critical path)."""
    if not training or p <= 0.0:
        return None
    key = (tuple(shape), str(device))
    ones = _ONES.get(key)
    if ones is None:
        if len(_ONES) > 16:
            _ONES.clear()
        ones = _ONES[key] = torch.ones(shape, dtype=torch.float32, device=device)
    return torch.nn.functional.dropout(ones, p=p, training=True)


class GatherRowsFn(Function):
    """aten::embedding with the backward routed to the table's RowGradSink."""

    @staticmethod
    def forward(ctx, weight, idx, sink, stream=None):
        ctx.sink, ctx.idx = sink, idx
        if ctx.needs_input_grad[0]:
            _expect(sink, idx)
        return ops.gather_rows(weight, idx, stream=stream)

    @staticmethod
    def backward(ctx, g):
        d = g.shape[-1]
        ctx.sink.add(ctx.idx.reshape(-1), g.contiguous().view(-1, d))
        return None, None, None, None


class MeanPoolFn(Function):
    """Fused gather + masked mean (+dropout, +fs); psb_gather_meanpool_fwd / psb_fs_bwd."""

    @staticmethod
    def forward(ctx, weight, idx, fs_weight, fs_bias, sink, pad_idx, mask, tok_scale, keep_scale, stream=None):
        # validity by pad id with the pad row dropped by the sink anyway: the backward weights valid / count reduce to
        # 1 / count per pool, which the forward kernel hands out for free (no token-weights launch in backward).  A sink
        # that translates mini-table positions (begin) drops a row id, which pad_idx is not.
        ctx.by_count = (mask is None and pad_idx >= 0 and sink is not None and sink.ids is None and
                        sink.drop_idx == pad_idx and ctx.needs_input_grad[0])
        out, mean, inv = ops.gather_meanpool(weight, idx, pad_idx=pad_idx, mask=mask, tok_scale=tok_scale,
                                             keep_scale=keep_scale, fs_weight=fs_weight, fs_bias=fs_bias,
                                             want_inv_count=ctx.by_count, stream=stream)
        ctx.inv_count = inv
        ctx.sink, ctx.idx, ctx.pad_idx, ctx.mask, ctx.keep = sink, idx, pad_idx, mask, keep_scale
        if ctx.needs_input_grad[0]:
            _expect(sink, idx)
        ctx.fs = fs_weight is not None
        if ctx.fs:
            ctx.save_for_backward(out, mean, fs_weight)
        return out

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        gw = gb = None
        if ctx.fs:
            out, mean, fs_weight = ctx.saved_tensors
            gw, gb, gm = ops.fs_bwd(g, out, mean, ctx.keep, fs_weight)
        else:
            gm = g if ctx.keep is None else g * ctx.keep
        idx = ctx.idx
        if ctx.by_count:
            ctx.sink.add(idx.reshape(-1), gm, src_div=idx.shape[1], scale2=ctx.inv_count, scale2_div=idx.shape[1])
        else:
            tw = ops.token_weights(idx, pad_idx=ctx.pad_idx, mask=ctx.mask)
            ctx.sink.add(idx.reshape(-1), gm, src_div=idx.shape[1], scale=tw.view(-1))
        return None, None, gw, gb, None, None, None, None, None, None


class NSLossFn(Function):
    """Fused negative-sampling loss (psb_ns_loss_fwd); returns the per-anchor loss [n]."""

    @staticmethod
    def forward(ctx, anchor_a, anchor_b, weight, bias, pos_idx, neg_idx, sink, pad_idx, mask, neg_weight,
                pos_weight, stream=None):
        loss, cp, cn, ga, gb = ops.ns_loss(anchor_a, weight, pos_idx, neg_idx, anchor_b=anchor_b, bias=bias,
                                           mask=mask, pad_idx=pad_idx, neg_weight=neg_weight,
                                           pos_weight=pos_weight, stream=stream)
        ctx.sink, ctx.pos_idx, ctx.neg_idx = sink, pos_idx, neg_idx
        if ctx.needs_input_grad[2] or (bias is not None and ctx.needs_input_grad[3]):
            _expect(sink, pos_idx)
            if neg_idx.numel() > 0:
                _expect(sink, neg_idx)
        ctx.has_b, ctx.has_bias = anchor_b is not None, bias is not None
        ctx.save_for_backward(anchor_a, anchor_b, cp, cn, ga, gb)
        return loss

    @staticmethod
    def backward(ctx, g):
        anchor_a, anchor_b, cp, cn, ga, gb = ctx.saved_tensors
        g = g.contiguous()
        n, w = ctx.pos_idx.shape
        k = cn.shape[-1]
        ctx.sink.add(ctx.pos_idx.reshape(-1), anchor_a, src_div=w, scale=cp.view(-1), scale2=g, scale2_div=w,
                     to_bias=ctx.has_bias)
        if k > 0:
            if ctx.has_b:
                ctx.sink.add(ctx.neg_idx.reshape(-1), anchor_b, src_div=1, scale=cn.view(-1), scale2=g,
                             scale2_div=w * k, to_bias=ctx.has_bias)
            else:
                ctx.sink.add(ctx.neg_idx.reshape(-1), anchor_a, src_div=w * k, scale=cn.view(-1), scale2=g,
                             scale2_div=w * k, to_bias=ctx.has_bias)
        grad_a = ga * g.unsqueeze(1) if ctx.needs_input_grad[0] else None
        grad_b = None
        if ctx.has_b and ctx.needs_input_grad[1]:
            grad_b = gb * g.repeat_interleave(k).unsqueeze(1)
        return grad_a, grad_b, None, None, None, None, None, None, None, None, None, None


class DensePosLossFn(Function):
    """Positive half of the NS loss against ALREADY GATHERED target rows [n, w, d] -- the reference's call form of
    ParagraphVector.forward / ParagraphVectorCorruption.forward (PV.py:50, PVC.py:69 take ``review_word_emb``, the
    output of ``word_embeddings(idx)``).  Same kernel, identity index over the flattened rows; the gradient goes back
    to the dense tensor through autograd (and from there into whatever produced it), not into a sink."""

    @staticmethod
    def forward(ctx, anchor, dense, mask):
        n, w, d = dense.shape
        flat = dense.contiguous().view(n * w, d)
        idx = torch.arange(n * w, device=dense.device).view(n, w)
        loss, cp, _, ga, _ = ops.ns_loss(anchor.contiguous(), flat, idx, idx.new_empty((n, w, 0)), mask=mask)
        ctx.save_for_backward(anchor, cp, ga)
        return loss

    @staticmethod
    def backward(ctx, g):
        anchor, cp, ga = ctx.saved_tensors
        g = g.contiguous()
        grad_anchor = ga * g.unsqueeze(1) if ctx.needs_input_grad[0] else None
        grad_dense = None
        if ctx.needs_input_grad[1]:
            grad_dense = anchor.unsqueeze(1) * (cp * g.unsqueeze(1)).unsqueeze(-1)
        return grad_anchor, grad_dense, None


def ns_loss_dense_pos(anchor, dense_pos, table, neg_idx, sink, mask=None):
    """NS loss with the positive rows given as a dense tensor [n, w, d] and the negatives as indices into ``table``
    (the reference's PV / PVC forward signature).  Two launches of the fused kernel: positives by identity index over
    the dense rows (k = 0), negatives with the positive term weighted 0 (its index is the dropped pad row); both
    halves are masked means over the same mask, so their sum is the reference's loss [n]."""
    n, w, _ = dense_pos.shape
    pos = DensePosLossFn.apply(anchor, dense_pos, mask)
    pad = torch.full((n, w), table.shape[0] - 1, dtype=torch.int64, device=table.device)
    ensure_current(table, (neg_idx,))
    neg = NSLossFn.apply(anchor, None, table, None, pad, neg_idx, sink, -1, mask, None, 0.0, None)
    return pos + neg


class TemTailFn(Function):
    """The TEM tail in two launches: ranking loss on the encoder's [B, 1 + K, d] output block in place
    (psb_tem_loss_fwd; no repacking copies of the positive / negative rows) and
    ``loss = mean(ps_rows) + mean(item_loss_rows)`` with the trainer's running sums (psb_tem_loss_finish) --
    item_transformer.py:485,:493-520.  The gradient with respect to the block comes out of the forward kernel already
    laid out and scaled by 1 / B, so backward is one multiply by the upstream scalar plus the sink contributions."""

    @staticmethod
    def forward(ctx, enc_out, il_rows, weight, bias, pos_idx, neg_idx, sink, pos_weight, acc_ps, acc_il, src_rows):
        B = pos_idx.numel()
        rows, cp, cn, g_enc = ops.tem_loss(enc_out, weight, pos_idx, neg_idx, bias=bias, pos_weight=pos_weight,
                                           grad_scale=1.0 / B)
        loss = ops.tem_loss_finish(rows, il_rows, acc_ps, acc_il)
        ctx.sink, ctx.pos_idx, ctx.neg_idx, ctx.src_rows = sink, pos_idx, neg_idx, src_rows
        if ctx.needs_input_grad[2] or (bias is not None and ctx.needs_input_grad[3]):
            _expect(sink, pos_idx)
            _expect(sink, neg_idx)
        ctx.has_bias = bias is not None
        ctx.n_il = il_rows.numel()
        ctx.save_for_backward(enc_out, cp, cn, g_enc)
        return loss

    @staticmethod
    def backward(ctx, g):
        enc_out, cp, cn, g_enc = ctx.saved_tensors
        g = g.contiguous()                                      # 0-dim upstream gradient
        B, K = cn.shape
        flat = enc_out.view(B * (1 + K), -1)
        pos_rows, neg_rows = ctx.src_rows
        every = B * K + 1                                       # scale2 index = slot / every = 0: the scalar g
        ctx.sink.add(ctx.pos_idx.reshape(-1), flat, src_row=pos_rows, scale=cp.view(-1), scale2=g.view(1),
                     scale2_div=every, to_bias=ctx.has_bias)
        ctx.sink.add(ctx.neg_idx.reshape(-1), flat, src_row=neg_rows, scale=cn.view(-1), scale2=g.view(1),
                     scale2_div=every, to_bias=ctx.has_bias)
        grad_enc = g_enc * g if ctx.needs_input_grad[0] else None
        grad_il = (g / ctx.n_il).expand(ctx.n_il) if ctx.needs_input_grad[1] else None
        return grad_enc, grad_il, None, None, None, None, None, None, None, None, None


def tem_tail(enc_out, il_rows, weight, pos_idx, neg_idx, sink, bias=None, pos_weight=1.0, acc_ps=None, acc_il=None,
             src_rows=None):
    ensure_current(weight, (pos_idx, neg_idx))
    return TemTailFn.apply(enc_out, il_rows, weight, bias, pos_idx, neg_idx, sink, pos_weight, acc_ps, acc_il, src_rows)


class SeqEncoderFn(Function):
    """Fused last encoder layer + final LayerNorm at one output position (psb_encoder_fwd / _bwd).
    Token inputs: (first [S,d], table, idx [S,T-1]) -- gradients of the table rows go to ``sink`` --
    or a dense [S,T,d] tensor."""

    @staticmethod
    def forward(ctx, first, dense, table, idx, sink, pad_idx, mask, pe, opts, names, *weights):
        params = dict(zip(names, weights))
        out, call = ops.encoder_fwd(params, opts["heads"], first=first, table=table, idx=idx, pad_idx=pad_idx,
                                    dense=dense, mask=mask, pe=pe, copies=opts["copies"], out_pos=opts["out_pos"],
                                    pre_ln=opts["pre_ln"], eps=opts["eps"], p_drop=opts["p_drop"],
                                    seed=opts["seed"], raw_input=opts.get("raw_input", False),
                                    first_ready=opts.get("first_ready"))
        ctx.call, ctx.sink, ctx.idx, ctx.names = call, sink, idx, names
        if call.tem and sink is not None and call.T > 1 and ctx.needs_input_grad[2]:
            _expect(sink, idx)
        ctx.shapes = {n: tuple(w.shape) for n, w in zip(names, weights)}
        ctx.pre_ln = opts["pre_ln"]
        ctx.weights = weights
        return out

    # The weight gradients (split-M partial products + their reduce, ~55 us at batch 384) are needed by nobody
    # before the optimizer, so the library computes them on its side stream next to the rest of the backward pass
    # (data gradients of the encoder, query-encoder backward, the tables' gradient sinks) and records an event; one
    # engine callback at the end of backward() makes the calling stream wait for it.  Only when the weights have no
    # gradient yet and no earlier node of the same pass has gradients of the same weights in flight: AccumulateGrad
    # then merely adopts the new tensors -- an in-place accumulation would touch them on the calling stream too
    # early, so in that case whatever is in flight is joined first and this node runs on the calling stream.
    _events = {}
    _pending = {}          # device -> [event, [(workspace, forward call, grad_out) kept alive], {id(weight) in flight}]

    @staticmethod
    def _join(dev):
        p = SeqEncoderFn._pending.pop(dev, None)
        if p is not None:
            torch.cuda.current_stream(dev).wait_event(p[0])
            p[1].clear()                                        # the side stream is done with the buffers

    @staticmethod
    def backward(ctx, g):
        shapes = ctx.shapes if ctx.pre_ln else {n: s for n, s in ctx.shapes.items() if not n.startswith("ln_attn")}
        dev = g.device
        pend = SeqEncoderFn._pending.get(dev)
        ids = set(id(w) for w in ctx.weights)
        clash = pend is not None and not ids.isdisjoint(pend[2])
        fork = not ctx.pre_ln and not clash and all(w.grad is None for w in ctx.weights)
        if clash or (pend is not None and not fork):
            SeqEncoderFn._join(dev)
            pend = None
        ev = None
        if fork:
            ev = SeqEncoderFn._events.get(dev)
            if ev is None:
                ev = SeqEncoderFn._events[dev] = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(dev))      # creates the underlying cudaEvent_t
        g_first, g_rest, g_dense, grads, ws = ops.encoder_bwd(ctx.call, g, shapes, wgrad_event=ev)
        if ev is not None:
            # the side stream reads the workspace AND the forward's saved activations / inputs (ctx.call) until the
            # event: both stay referenced until the join, or the caching allocator would hand their memory to the
            # next allocation of the calling stream
            alive = (ws, ctx.call, g)
            if pend is None:
                SeqEncoderFn._pending[dev] = [ev, [alive], ids]
                Variable._execution_engine.queue_callback(lambda dev=dev: SeqEncoderFn._join(dev))
            else:                    # same side stream, same event re-recorded behind the earlier work
                pend[1].append(alive)
                pend[2].update(ids)
        if ctx.call.tem and ctx.sink is not None and ctx.call.T > 1:
            ctx.sink.add(ctx.idx.reshape(-1), g_rest.view(-1, g_rest.shape[-1]))
        ctx.call = None
        ctx.weights = None
        return (g_first, g_dense, None, None, None, None, None, None, None, None) + tuple(
            grads.pop(n, None) for n in ctx.names)


def ensure_current(weight, idx_list, stream=None):
    """Row-sparse optimizer (optimizers.FusedAdam): a table whose rows are updated lazily carries ``_psb_lazy``; the
    rows about to be gathered are brought up to the current optimizer step first, on the stream the reader runs on.
    No-op (one attribute lookup) for every other tensor."""
    lazy = getattr(weight, "_psb_lazy", None)
    if lazy is None:
        return
    if stream is None:
        lazy.ensure(idx_list)
    else:
        # fork first: the side stream must be ordered behind the calling stream (the previous optimizer step) -- and,
        # under stream capture, must have JOINED the capture -- before the catch-up is enqueued on it
        stream.wait_stream(torch.cuda.current_stream(weight.device))
        with torch.cuda.stream(stream):
            keep = lazy.ensure(idx_list)
        held = getattr(stream, "_psb_keep", None)       # converted index copies stay alive until the stream is joined
        if held is None:
            held = stream._psb_keep = []
        held.append(tuple(keep or ()))
        del held[:-8]


def gather_rows(weight, idx, sink, stream=None):
    ensure_current(weight, (idx,), stream)
    return GatherRowsFn.apply(weight, idx, sink, stream)


def meanpool(weight, idx, sink, pad_idx=-1, mask=None, tok_scale=None, keep_scale=None, fs_weight=None,
             fs_bias=None, stream=None):
    ensure_current(weight, (idx,), stream)
    return MeanPoolFn.apply(weight, idx, fs_weight, fs_bias, sink, pad_idx, mask, tok_scale, keep_scale, stream)


def ns_loss(anchor_a, weight, pos_idx, neg_idx, sink, anchor_b=None, bias=None, pad_idx=-1, mask=None,
            neg_weight=None, pos_weight=1.0, stream=None):
    """stream: enqueue the forward kernel on a side stream the caller has forked and will join (the autograd node
    -- and therefore its backward -- still belongs to the current stream)."""
    ensure_current(weight, (pos_idx, neg_idx), stream)
    return NSLossFn.apply(anchor_a, anchor_b, weight, bias, pos_idx, neg_idx, sink, pad_idx, mask, neg_weight,
                          pos_weight, stream)


def seq_encoder(params, opts, first=None, table=None, idx=None, sink=None, pad_idx=-1, dense=None, mask=None,
                pe=None):
    """params: ordered dict name -> Parameter (psb_encoder_params_t member names)."""
    if table is not None:
        ensure_current(table, (idx,))
    names = tuple(params.keys())
    return SeqEncoderFn.apply(first, dense, table, idx, sink, pad_idx, mask, pe, opts, names, *params.values())
