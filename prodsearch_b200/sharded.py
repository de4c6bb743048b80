"""Multi-GPU plumbing: one process per GPU over torch.distributed (NCCL on GPUs, gloo in CPU tests).

SURVEY.md 8(e): small dense parameters are replicated and all-reduced; the item table is
row-sharded cyclically (owner = id % G, local row = id // G, which spreads Zipf-popular ids).

Training uses "fetch unique -> compute locally -> push gradients":
  1. every rank collects ALL item ids its step needs (targets, negatives, histories), makes them
     unique, and fetches those rows from their owners with one index all-to-all and one row
     all-to-all (``ShardedTable.fetch``) into a small local *mini table*;
  2. the unchanged single-GPU fused kernels run against the mini table with remapped indices;
  3. the mini table's gradient rows travel back to the owners with one more all-to-all and are
     folded into the shard by the deterministic sort + segmented reduce (``push_grads``): terms
     arrive ordered by (source rank, id), so the result is bit-reproducible.
Duplicated ids (popular items) cross NVLink once per rank per step instead of once per use.

Evaluation: every rank scores the (all-gathered) queries against its shard with
``psb_catalog_topk`` (id_base = rank, id_stride = G), the per-shard top-k lists are all-gathered
and merged by ``psb_topk_merge`` (``sharded_rank_catalog``; the peer-sharded model uses it too).

The exchange logic is backend-agnostic: row gather / gradient fold are injected callables, so the
CPU test-suite drives it with gloo (world_size 2) while the product passes the CUDA ops.
"""
import torch
import torch.distributed as dist


def _world(group):
    return dist.get_world_size(group), dist.get_rank(group)


class DenseGradAllReduce(object):
    """Average the gradients of the replicated parameters in one flat bucket."""

    def __init__(self, module, skip=(), group=None):
        self.group = group
        self.params = [p for n, p in module.named_parameters() if p.requires_grad and n not in skip]

    def reduce(self):
        grads = [p.grad for p in self.params if p.grad is not None]
        if not grads:
            return
        flat = torch.cat([g.reshape(-1) for g in grads])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
        flat.div_(dist.get_world_size(self.group))
        off = 0
        for g in grads:
            n = g.numel()
            g.copy_(flat[off:off + n].view_as(g))
            off += n


def exchange_plan(ids, world):
    """Bucket unique global ids by owner.  Returns (perm, send_counts list, local_ids in send order)."""
    dest = ids % world
    perm = torch.argsort(dest, stable=True)
    counts = torch.bincount(dest, minlength=world)
    return perm, counts, (ids[perm] // world)


def all_to_all_var(send, send_counts, recv_counts, group):
    """all_to_all_single with per-peer row counts (host lists); rows = leading dimension."""
    out = send.new_empty((int(sum(recv_counts)),) + tuple(send.shape[1:]))
    dist.all_to_all_single(out, send.contiguous(), output_split_sizes=list(recv_counts),
                           input_split_sizes=list(send_counts), group=group)
    return out


class ShardedTable(object):
    """A [rows, d] table row-sharded over the ranks of ``group``.

    gather_fn(weight, local_ids) -> rows        (product: ops.gather_rows)
    fold_fn(weight, local_ids, grad_rows)       (product: sort + segmented reduce into weight.grad)
    """

    def __init__(self, rows, d, group, gather_fn, fold_fn, device, pad_idx=None, init="normal", seed=0):
        self.rows, self.d, self.group, self.pad_idx = rows, d, group, pad_idx
        self.world, self.rank = _world(group)
        self.local_rows = (rows - self.rank + self.world - 1) // self.world
        g = torch.Generator(device="cpu").manual_seed(seed + 7919 * self.rank)
        w = torch.randn(self.local_rows, d, generator=g) if init == "normal" else torch.zeros(self.local_rows, d)
        if pad_idx is not None and pad_idx % self.world == self.rank:
            w[pad_idx // self.world] = 0
        self.weight = torch.nn.Parameter(w.to(device))
        self.gather_fn, self.fold_fn = gather_fn, fold_fn
        self._last = None

    @classmethod
    def from_full(cls, full, group, gather_fn, fold_fn, device, pad_idx=None):
        """Shard an existing full table (tests / checkpoint loading)."""
        t = cls(full.shape[0], full.shape[1], group, gather_fn, fold_fn, device, pad_idx, init="zeros")
        with torch.no_grad():
            t.weight.copy_(full[t.rank::t.world].to(device))
        return t

    def fetch(self, index_tensors):
        """Unique the ids of ``index_tensors``, fetch their rows from the owners.
        Returns (mini_table [u, d] leaf tensor, remapped index tensors, remapped pad index or -1)."""
        flat = torch.cat([t.reshape(-1) for t in index_tensors])
        uniq, inverse = torch.unique(flat, sorted=True, return_inverse=True)
        perm, counts, local_ids = exchange_plan(uniq, self.world)
        send_counts = counts.tolist()                                  # host sync #1 (split sizes)
        recv_counts_t = torch.empty_like(counts)
        dist.all_to_all_single(recv_counts_t, counts, group=self.group)
        recv_counts = recv_counts_t.tolist()                           # host sync #2
        want = all_to_all_var(local_ids, send_counts, recv_counts, self.group)
        rows = self.gather_fn(self.weight.detach(), want)
        mini = all_to_all_var(rows, recv_counts, send_counts, self.group)   # rows in `perm` order
        mini.requires_grad_(self.weight.requires_grad)
        inv_perm = torch.empty_like(perm)
        inv_perm[perm] = torch.arange(perm.numel(), device=perm.device)
        remap = inv_perm[inverse]
        outs, off = [], 0
        for t in index_tensors:
            outs.append(remap[off:off + t.numel()].view(t.shape))
            off += t.numel()
        pad = -1
        if self.pad_idx is not None:
            hit = (uniq == self.pad_idx).nonzero()
            if hit.numel():                                            # host sync #3 only via .numel() of nonzero
                pad = int(inv_perm[hit[0, 0]])
        self._last = (want, send_counts, recv_counts)
        return mini, outs, pad

    def push_grads(self, mini_grad):
        """Send the mini table's gradient rows (send order = fetch order) to their owners and fold them
        into the shard.  mini_grad [u, d] (zeros where untouched)."""
        want, send_counts, recv_counts = self._last
        grads = all_to_all_var(mini_grad, send_counts, recv_counts, self.group)
        self.fold_fn(self.weight, want, grads)
        self._last = None


def sharded_rank_catalog(queries, k, shard_topk, merge_fn, group=None):
    """Full-catalog top-k over a row-sharded table (owner = id % G).  queries [m, d]: this rank's, m may differ from
    rank to rank.  Every rank scores the queries of all ranks against its shard,
    ``shard_topk(q_all, k, id_base=rank, id_stride=G) -> (ids, scores)``; the per-shard lists are gathered into
    [G, G * m_max, k] and merged, ``merge_fn(ids, scores) -> (ids, scores)`` [G * m_max, k].  Every collective lands
    in its final layout (all_gather_into_tensor): no host pickles, no list gathers, no cat / stack copies."""
    world, rank = _world(group)
    if world == 1:
        return shard_topk(queries, k, 0, 1)
    m = torch.tensor([queries.shape[0]], device=queries.device)
    ms = torch.empty(world, dtype=m.dtype, device=queries.device)
    dist.all_gather_into_tensor(ms, m, group=group)
    m_max = int(ms.max())
    q_pad = queries
    if queries.shape[0] != m_max:
        q_pad = queries.new_zeros((m_max, queries.shape[1]))
        q_pad[:queries.shape[0]] = queries
    q_all = queries.new_empty((world * m_max, queries.shape[1]))
    dist.all_gather_into_tensor(q_all, q_pad, group=group)
    ids, sc = shard_topk(q_all, k, rank, world)
    ids_all = ids.new_empty((world, world * m_max, k))
    sc_all = sc.new_empty((world, world * m_max, k))
    dist.all_gather_into_tensor(ids_all.view(-1, k), ids, group=group)
    dist.all_gather_into_tensor(sc_all.view(-1, k), sc, group=group)
    mi, ms_ = merge_fn(ids_all, sc_all)
    lo = rank * m_max
    return mi[lo:lo + queries.shape[0]], ms_[lo:lo + queries.shape[0]]
