"""Optimizer wrapper with the reference's semantics (models/optimizers.py:111-245): Adam with
eps=1e-9 (:186), optional noam schedule (:214-219) and global-norm gradient clipping (:241-242).
Row N2 of SURVEY.md 8(f).  Two forms, both one fused multi-tensor call with the step counter and the global norm in
device memory (CUDA-graph replayable):
  * dense (``psb_adam_step``): the clip + Adam update of every element of every tensor, on the dense ``.grad``
    tensors the gradient sinks attach in ``grad_mode="dense"`` -- literally the reference's sweep;
  * row-sparse (``psb_adam_sparse_step``): embedding tables whose sinks run in ``grad_mode="rowsparse"`` hand over
    ``param.row_grad = (unique_rows, reduced_rows, n)``; only those rows are updated, every other row rests and is
    replayed (``psb_adam_rows_catchup``) right before something reads it -- the gather wrappers of ``functional.py``
    call ``ensure_current`` -- or when ``flush()`` is called (evaluation, checkpoints).  Dense-equivalent results
    within fp32 rounding; the step costs O(rows touched), not O(table).

Known difference from torch.optim.Adam: ONE step counter for all tensors (torch keeps one per parameter; they only
differ for a parameter that receives its first gradient later than the others -- none does in these models).
A step in which a row-sparse table receives no row list (its gradient is None) is a zero-gradient step for every row of
that table -- its moments decay and its rows move, as in a dense step with a zero gradient -- whereas torch.optim.Adam
would leave a parameter without a gradient untouched."""
import torch
from torch.nn.utils import clip_grad_norm_

from . import _lib


class FusedAdam(object):
    """torch.optim.Adam(eps=1e-9) + clip_grad_norm_ in three sm_100a launches (psb_adam_step).  Keeps the
    ``param_groups`` / ``state_dict`` / ``load_state_dict`` surface of torch.optim.Adam that the reference's
    checkpoints use (models/ps_model.py:27-32, trainer.py:234-244)."""

    def __init__(self, params, lr, betas=(0.9, 0.999), eps=1e-9, weight_decay=0.0):
        self.params = list(params)
        self.param_groups = [dict(params=self.params, lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay,
                                  amsgrad=False)]
        self.state = {}
        self._step_dev = None
        self._sqnorm = None
        self._ws = None
        self._norm_given = 0
        self.coef_cap = 1 << 18              # steps whose coefficients the catch-up reads from a table (2 MB)
        self._coef_hist = None
        self._lazy = {}                      # table parameter -> LazyRows

    def _ensure(self, dev):
        if self._step_dev is None:
            self._step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
            self._sqnorm = torch.zeros(1, dtype=torch.float32, device=dev)

    def adopt_state(self, p, exp_avg, exp_avg_sq, last_step=None):
        """Use caller-owned tensors as the optimizer state of ``p`` (row-sharded tables keep their moments and row
        stamps in peer memory, where the readers of a resting row find them)."""
        st = dict(exp_avg=exp_avg, exp_avg_sq=exp_avg_sq)
        if last_step is not None:
            st["last_step"] = last_step
        self.state[p] = st

    def _state_of(self, p):
        st = self.state.get(p)
        if st is None:
            st = self.state[p] = dict(exp_avg=torch.zeros_like(p, memory_format=torch.contiguous_format),
                                      exp_avg_sq=torch.zeros_like(p, memory_format=torch.contiguous_format))
        return st

    def set_global_sqnorm(self, sq):
        """Row-sharded training: the caller supplies the GLOBAL squared gradient norm (device tensor [1]; this
        rank's parameters are only a shard) for the next ``step``.  Stream-ordered copy, CUDA-graph safe."""
        self._ensure(sq.device)
        self._sqnorm.copy_(sq.reshape(1))
        self._norm_given = 1

    def global_norm_slots(self, device):
        """(sqnorm, step) device tensors a caller fills itself (psb_peer_sum_sqnorm) for the next ``step``."""
        self._ensure(device)
        self._norm_given = 2
        return self._sqnorm, self._step_dev

    @property
    def total_norm(self):
        """Global gradient norm of the last step (device tensor; reading it synchronises)."""
        return self._sqnorm.sqrt()

    # ---- row-sparse tables -------------------------------------------------------------------------------
    def _rows_struct(self, p, lists=True):
        """psb_adam_rows_t of table parameter ``p`` (+ the bias vector indexed like it) and the tensors it points to."""
        st = self._state_of(p)
        if "last_step" not in st:
            # every row is current at the optimizer's step: 0 in a fresh run, the checkpoint's step after a resume (a
            # stamp of 0 would read as "never updated" and the row's resting steps would not be replayed)
            st["last_step"] = self._step_stamps(p.shape[0], p.device)
        bias = getattr(p, "_psb_row_bias", None)
        if bias is not None and not bias.requires_grad:
            bias = None
        keep = [st["exp_avg"], st["exp_avg_sq"], st["last_step"]]
        R = _lib.AdamRows()
        R.p, R.m, R.v, R.last_step = p.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), st["last_step"].data_ptr()
        R.d, R.table_rows = p.shape[1], p.shape[0]
        if bias is not None:
            sb = self._state_of(bias)
            R.bias_p, R.bias_m, R.bias_v = bias.data_ptr(), sb["exp_avg"].data_ptr(), sb["exp_avg_sq"].data_ptr()
            keep += [sb["exp_avg"], sb["exp_avg_sq"]]
        if lists:
            rows, vals, nu = p.row_grad
            by_row = bool(getattr(p, "_psb_grad_by_row", False))      # dense buffer indexed by row id (sharded fold)
            R.rows, R.grad, R.n_rows = rows.data_ptr(), vals.data_ptr(), nu.data_ptr()
            R.cap = rows.numel() if by_row else min(rows.numel(), vals.shape[0])
            R.grad_by_row = 1 if by_row else 0
            keep += [rows, vals, nu]
            bg = getattr(bias, "row_grad", None) if bias is not None else None
            if bg is not None:
                if bg[0].data_ptr() != rows.data_ptr():
                    raise RuntimeError("bias row gradient does not share its table's row list")
                R.bias_grad = bg[1].data_ptr()
                keep.append(bg[1])
        return R, keep, bias

    def _step_stamps(self, n, device):
        """int32 [n] holding the current step: a stream-ordered copy of the device counter, no host sync."""
        self._ensure(device)
        return self._step_dev.to(torch.int32).expand(n).clone()

    def _hyper(self):
        g = self.param_groups[0]
        b1, b2 = g["betas"]
        return float(g["lr"]), float(b1), float(b2), float(g["eps"])

    def _catchup(self, p, idx_list, noam=None, warmup=None):
        """Bring the rows of lazily updated table ``p`` up to the current step before they are read
        (``idx_list``: index tensors about to be gathered; None = every row).  Runs on the current stream."""
        if self._step_dev is None:
            return
        R, keep, _ = self._rows_struct(p, lists=False)
        lr, b1, b2, eps = self._hyper()
        noam = self._last_noam if noam is None else noam
        warmup = self._last_warmup if warmup is None else warmup
        n = 0
        ptrs = cnts = None
        if idx_list is not None:
            idx_list = [t if (t.dtype == torch.int64 and t.is_contiguous()) else t.long().contiguous() for t in idx_list
                        if t is not None and t.numel() > 0]
            n = len(idx_list)
            if n == 0:
                return
            if n > _lib.ADAM_MAX_IDX_LISTS:
                raise RuntimeError("more than %d index lists in one catch-up" % _lib.ADAM_MAX_IDX_LISTS)
            ptrs = (_lib.c_vp * n)(*[t.data_ptr() for t in idx_list])
            cnts = (_lib.c_i64 * n)(*[t.numel() for t in idx_list])
            keep += idx_list
        skip = int(getattr(p, "_psb_drop_idx", -1))
        _lib.check(_lib.load().psb_adam_rows_catchup(
            R, ptrs, cnts, n, skip, lr, b1, b2, eps, 1 if noam else 0, float(warmup), self._step_dev.data_ptr(),
            self._coef_hist.data_ptr() if self._coef_hist is not None else None, self.coef_cap, _lib.stream_ptr()),
            "psb_adam_rows_catchup")
        return keep

    def flush(self):
        """Make every lazily updated table dense-equivalent NOW (before evaluation, ranking, checkpoints)."""
        for p in list(self._lazy):
            self._catchup(p, None)
        if self._lazy:
            _lib.note_param_write()

    _last_noam, _last_warmup = False, 4000.0

    def _sparse_step(self, live, sparse, max_grad_norm, noam, warmup_steps):
        g = self.param_groups[0]
        if g["weight_decay"]:
            raise RuntimeError("row-sparse Adam does not support weight_decay (a decayed row never rests): "
                               "use grad_mode='dense'")
        if len(sparse) > _lib.ADAM_MAX_ROW_TABLES:
            raise RuntimeError("more than %d row-sparse tables" % _lib.ADAM_MAX_ROW_TABLES)
        dev = (sparse[0] if sparse else live[0]).device
        self._ensure(dev)
        if self._coef_hist is None:
            self._coef_hist = torch.zeros(self.coef_cap * 2, dtype=torch.float32, device=dev)
        rows_arr = (_lib.AdamRows * max(len(sparse), 1))()
        keep, covered = [], set()
        for i, p in enumerate(sparse):
            if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() and p.dim() == 2):
                raise RuntimeError("row-sparse Adam needs contiguous fp32 CUDA tables")
            R, k, bias = self._rows_struct(p)
            rows_arr[i] = R
            keep.append(k)
            if bias is not None:
                covered.add(id(bias))
            if p not in self._lazy:
                self._lazy[p] = p._psb_lazy = LazyRows(self, p)
        live = [p for p in live if id(p) not in covered]
        if len(live) > _lib.ADAM_MAX_TENSORS:
            raise RuntimeError("FusedAdam: more than %d parameter tensors" % _lib.ADAM_MAX_TENSORS)
        arr = (_lib.AdamTensor * max(len(live), 1))()
        for i, p in enumerate(live):
            st = self._state_of(p)
            grad = p.grad
            if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() and grad.is_contiguous()
                    and grad.dtype == torch.float32 and not grad.is_sparse):
                raise RuntimeError("FusedAdam needs contiguous fp32 CUDA parameters and dense gradients")
            arr[i] = _lib.AdamTensor(p.data_ptr(), grad.data_ptr(), st["exp_avg"].data_ptr(),
                                     st["exp_avg_sq"].data_ptr(), p.numel())
        lib = _lib.load()
        wb = int(lib.psb_adam_sparse_workspace_bytes(arr, len(live), rows_arr, len(sparse)))
        if wb < 0:
            _lib.check(wb, "psb_adam_sparse_workspace_bytes")
        if self._ws is None or self._ws.numel() < wb:
            self._ws = torch.empty(wb, dtype=torch.uint8, device=dev)
        lr, b1, b2, eps = self._hyper()
        self._last_noam, self._last_warmup = bool(noam), float(warmup_steps)
        from . import ops
        ev = None
        if ops.PROFILE is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        _lib.check(lib.psb_adam_sparse_step(arr, len(live), rows_arr, len(sparse), lr, b1, b2, eps,
                                            float(max_grad_norm or 0.0), 1 if noam else 0, float(warmup_steps),
                                            int(self._norm_given), self._step_dev.data_ptr(), self._sqnorm.data_ptr(),
                                            self._coef_hist.data_ptr(), self.coef_cap, self._ws.data_ptr(),
                                            self._ws.numel(), _lib.stream_ptr()), "psb_adam_sparse_step")
        self._norm_given = 0
        for p in sparse:                      # consumed: a step without a new backward must not re-apply them
            p.row_grad = None
            b = getattr(p, "_psb_row_bias", None)
            if b is not None:
                b.row_grad = None
        _lib.note_param_write()
        if ev is not None:
            ev[1].record()
            ops.PROFILE.setdefault("adam_step", []).append(ev)

    def step(self, max_grad_norm=0.0, noam=False, warmup_steps=4000.0):
        g = self.param_groups[0]
        live = [p for p in self.params if p.grad is not None]
        sparse = [p for p in self.params if p.dim() == 2 and getattr(p, "row_grad", None) is not None]
        if any(p in self._lazy for p in live):
            raise RuntimeError("a table that has been updated row-sparsely received a dense gradient: keep its sink in "
                               "grad_mode='rowsparse' (or call flush() and build a new optimizer)")
        if sparse or (self._lazy and live):
            return self._sparse_step(live, sparse, max_grad_norm, noam, warmup_steps)
        if not live:
            return
        if len(live) > _lib.ADAM_MAX_TENSORS:
            raise RuntimeError("FusedAdam: more than %d parameter tensors" % _lib.ADAM_MAX_TENSORS)
        self._ensure(live[0].device)
        arr = (_lib.AdamTensor * len(live))()
        for i, p in enumerate(live):
            st = self._state_of(p)
            grad = p.grad
            if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() and grad.is_contiguous()
                    and grad.dtype == torch.float32 and not grad.is_sparse):
                raise RuntimeError("FusedAdam needs contiguous fp32 CUDA parameters and dense gradients")
            arr[i] = _lib.AdamTensor(p.data_ptr(), grad.data_ptr(), st["exp_avg"].data_ptr(),
                                     st["exp_avg_sq"].data_ptr(), p.numel())
        lib = _lib.load()
        wb = int(lib.psb_adam_workspace_bytes(arr, len(live)))
        if self._ws is None or self._ws.numel() < wb:
            self._ws = torch.empty(wb, dtype=torch.uint8, device=live[0].device)
        b1, b2 = g["betas"]
        from . import ops
        ev = None
        if ops.PROFILE is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        _lib.check(lib.psb_adam_step(arr, len(live), float(g["lr"]), float(b1), float(b2), float(g["eps"]),
                                     float(g["weight_decay"]), float(max_grad_norm or 0.0), 1 if noam else 0,
                                     float(warmup_steps), int(self._norm_given), self._step_dev.data_ptr(),
                                     self._sqnorm.data_ptr(),
                                     self._ws.data_ptr(), self._ws.numel(), _lib.stream_ptr()), "psb_adam_step")
        self._norm_given = 0
        _lib.note_param_write()        # raw-pointer update: tensor._version does not move
        if ev is not None:
            ev[1].record()
            ops.PROFILE.setdefault("adam_step", []).append(ev)

    # ---- torch.optim.Adam-compatible checkpoint format ----------------------------------------
    def state_dict(self):
        self.flush()                       # lazily updated tables: dense-equivalent moments and parameters
        step = int(self._step_dev.item()) if self._step_dev is not None else 0
        state = {}
        for i, p in enumerate(self.params):
            st = self.state.get(p)
            if st is not None:
                state[i] = dict(step=torch.tensor(float(step)), exp_avg=st["exp_avg"], exp_avg_sq=st["exp_avg_sq"])
        g = {k: v for k, v in self.param_groups[0].items() if k != "params"}
        g["params"] = list(range(len(self.params)))
        return dict(state=state, param_groups=[g])

    def load_state_dict(self, sd):
        step = 0
        for i, st in sd["state"].items():
            p = self.params[int(i)]
            mine = self._state_of(p)
            mine["exp_avg"].copy_(st["exp_avg"])
            mine["exp_avg_sq"].copy_(st["exp_avg_sq"])
            step = max(step, int(float(st["step"])))
        for k, v in sd["param_groups"][0].items():
            if k != "params":
                self.param_groups[0][k] = v
        if self.params:
            self._ensure(self.params[0].device)
            self._step_dev.fill_(step)
        for st in self.state.values():     # a torch-format checkpoint is dense: every row is current at ``step``
            if "last_step" in st:
                st["last_step"].fill_(step)

    def zero_grad(self, set_to_none=True):
        for p in self.params:
            p.grad = None


class LazyRows(object):
    """Handle a lazily updated table parameter carries (``param._psb_lazy``): the gather wrappers call ``ensure``
    with the indices they are about to read.  Catch-up launches of one table are chained by an event, so that two
    streams never replay the same table concurrently (a reader on one stream must not meet a row the other stream's
    launch is half-way through); the chain is per step -- the streams of a step are joined before the optimizer."""

    def __init__(self, optim, weight):
        self.optim, self.weight = optim, weight
        self._event = None
        self._key = None
        self._seen = set()          # (data_ptr, numel) of the index tensors already made current in this step

    def ensure(self, idx_list):
        """Index tensors already handled in this step (a model pre-ensures everything it will read in as few launches
        as possible; the gather wrappers then find nothing left to do) are skipped -- by identity of their storage."""
        cur = torch.cuda.current_stream(self.weight.device)
        key = (torch.cuda.is_current_stream_capturing(), _lib.PARAM_EPOCH[0])
        if self._key != key:
            self._seen = set()
        todo = [t for t in idx_list if t is not None and t.numel() > 0 and (t.data_ptr(), t.numel()) not in self._seen]
        if not todo:
            return None
        if self._event is None:
            self._event = torch.cuda.Event()
        elif self._key == key:
            cur.wait_event(self._event)
        keep = self.optim._catchup(self.weight, todo)
        self._event.record(cur)
        self._key = key
        self._seen.update((t.data_ptr(), t.numel()) for t in todo)
        return keep

    def flush(self):
        self.optim._catchup(self.weight, None)


class Optimizer(object):
    def __init__(self, method, learning_rate, max_grad_norm, beta1=0.9, beta2=0.999, decay_method=None,
                 warmup_steps=4000, weight_decay=0.0):
        if method not in ("adam", "sgd"):
            raise RuntimeError("Invalid optim method: " + method)
        self.method = method
        self.learning_rate = learning_rate
        self.original_lr = learning_rate
        self.max_grad_norm = max_grad_norm
        self.betas = [beta1, beta2]
        self.decay_method = decay_method
        self.warmup_steps = warmup_steps
        self.weight_decay = weight_decay
        self._step = 0

    def set_parameters(self, params):
        self.params = [p for _, p in params if p.requires_grad]
        if self.method == "sgd":
            self.optimizer = torch.optim.SGD(self.params, lr=self.learning_rate, weight_decay=self.weight_decay)
        else:
            self.optimizer = FusedAdam(self.params, lr=self.learning_rate, betas=self.betas, eps=1e-9,
                                       weight_decay=self.weight_decay)

    def step(self):
        self._step += 1
        noam = self.decay_method == "noam"
        if noam:      # host mirror of the schedule the kernel evaluates from its device step counter
            self.learning_rate = self.original_lr * min(self._step ** (-0.5),
                                                        self._step * self.warmup_steps ** (-1.5))
        if self.method == "sgd":
            if noam:
                self.optimizer.param_groups[0]["lr"] = self.learning_rate
            if self.max_grad_norm:
                clip_grad_norm_(self.params, self.max_grad_norm)
            self.optimizer.step()
            return
        self.optimizer.param_groups[0]["lr"] = self.original_lr if noam else self.learning_rate
        self.optimizer.step(self.max_grad_norm, noam, self.warmup_steps)

    def flush(self):
        """Row-sparse tables: replay every resting row (before evaluation / saving a checkpoint)."""
        if hasattr(self.optimizer, "flush"):
            self.optimizer.flush()

    def sync_host_step(self):
        """CUDA-graph replays advance only the device step counter: bring the host mirror (``_step``, the noam
        ``learning_rate``) in line before pickling the optimizer into a checkpoint."""
        dev = getattr(self.optimizer, "_step_dev", None)
        if dev is not None:
            self._step = int(dev.item())
            if self.decay_method == "noam" and self._step > 0:
                self.learning_rate = self.original_lr * min(self._step ** (-0.5),
                                                            self._step * self.warmup_steps ** (-1.5))


def build_optim(args, model, checkpoint=None):
    """models/ps_model.py:20-51 (fresh optimizer; checkpoint restore reuses the saved object)."""
    if getattr(args, "train_from", "") and checkpoint is not None:
        optim = checkpoint["optim"]
        saved = optim.optimizer.state_dict()
        optim.set_parameters(list(model.named_parameters()))
        optim.optimizer.load_state_dict(saved)
        return optim
    optim = Optimizer(args.optim, args.lr, args.max_grad_norm, beta1=args.beta1, beta2=args.beta2,
                      decay_method=args.decay_method, warmup_steps=args.warmup_steps,
                      weight_decay=args.l2_lambda)
    optim.set_parameters(list(model.named_parameters()))
    return optim
