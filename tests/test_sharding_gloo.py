"""CPU, world_size 2, gloo: the host-side logic of the row-sharded item table (SURVEY.md 8(e)).

The exchange plan, the index / row / gradient all-to-alls and the sharded top-k merge are
backend-agnostic (prodsearch_b200/sharded.py); here the device kernels are replaced by plain torch
CPU stand-ins (test infrastructure only) and the results are compared with the unsharded answer."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cpu_gather(w, ids):
    return w[ids]


def _cpu_fold(w, ids, grads):
    if w.grad is None:
        w.grad = torch.zeros_like(w)
    w.grad.index_add_(0, ids, grads)


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import oracle
        from prodsearch_b200 import sharded
        g = torch.Generator().manual_seed(0)                      # same data on every rank
        P, d, k = 203, 16, 7
        full = torch.randn(P + 1, d, generator=g)
        full[P] = 0
        table = sharded.ShardedTable.from_full(full, None, _cpu_gather, _cpu_fold, "cpu", pad_idx=P)
        assert table.weight.shape[0] == (P + 1 - rank + world - 1) // world
        # per-rank batch: different ids on each rank, duplicates, pad ids, ragged shapes
        gr = torch.Generator().manual_seed(100 + rank)
        tgt = torch.randint(0, P, (9,), generator=gr)
        neg = torch.randint(0, P, (9, 3), generator=gr)
        hist = torch.randint(0, P, (9, 5), generator=gr)
        hist[2, 3:] = P
        hist[4, :] = P
        neg[0, 0] = tgt[0]
        mini, (t2, n2, h2), pad = table.fetch([tgt, neg, hist])
        # bit-exact rows through the two all-to-alls and the remap
        assert torch.equal(mini[t2], full[tgt]) and torch.equal(mini[n2], full[neg]) and torch.equal(mini[h2], full[hist])
        assert pad >= 0 and torch.equal(mini[pad], full[P])
        assert mini.shape[0] == torch.unique(torch.cat([tgt, neg.reshape(-1), hist.reshape(-1)])).numel()
        # gradient push: every rank contributes a dense mini-gradient; owners fold them
        mg = torch.zeros_like(mini)
        up = torch.randn(9, d, generator=gr)
        mg.index_add_(0, t2, up)
        mg.index_add_(0, h2.reshape(-1), up.repeat_interleave(5, 0) * 0.5)
        mg[pad] = 0
        table.push_grads(mg.detach())
        # reference: the same contributions accumulated on the full table, all ranks summed
        ref = torch.zeros(P + 1, d)
        for r in range(world):
            g2 = torch.Generator().manual_seed(100 + r)
            tg = torch.randint(0, P, (9,), generator=g2)
            _ = torch.randint(0, P, (9, 3), generator=g2)
            hs = torch.randint(0, P, (9, 5), generator=g2)
            hs[2, 3:] = P
            hs[4, :] = P
            u2 = torch.randn(9, d, generator=g2)
            ref.index_add_(0, tg, u2)
            ref.index_add_(0, hs.reshape(-1), u2.repeat_interleave(5, 0) * 0.5)
        ref[P] = 0
        assert torch.allclose(table.weight.grad, ref[rank::world], atol=1e-6)
        # sharded catalog ranking == global ranking (lower id first), ragged query counts per rank
        q = torch.randint(-2, 3, (3 + rank, d), generator=gr).float()
        qtab = torch.randint(-2, 3, (P + 1, d), generator=g).float()      # integer data: exact ties
        qtab[10:20] = qtab[3]
        t2b = sharded.ShardedTable.from_full(qtab, None, _cpu_gather, _cpu_fold, "cpu", pad_idx=P)

        def topk(qa, kk, base, stride):
            assert (base, stride) == (rank, world)
            n_local = (P - base + stride - 1) // stride
            w = t2b.weight.detach()
            ids = base + stride * torch.arange(n_local)
            i, s_ = oracle.topk_lower_id_first((qa @ w[:n_local].t()).numpy(), kk, np.tile(ids.numpy(), (qa.shape[0], 1)))
            return torch.from_numpy(i), torch.from_numpy(s_)

        def merge(ids, sc):
            assert ids.shape == (world, world * (3 + world - 1), k)
            i, s_ = oracle.merge_shard_topk(list(ids.numpy()), list(sc.numpy()), k)
            return torch.from_numpy(i), torch.from_numpy(s_)
        ids, sc = sharded.sharded_rank_catalog(q, k, topk, merge)
        ref_i, ref_s = oracle.topk_lower_id_first((q @ qtab[:P].t()).numpy(), k)
        assert np.array_equal(ids.numpy(), ref_i) and np.array_equal(sc.numpy(), ref_s)
        # replicated-parameter gradient averaging
        lin = torch.nn.Linear(4, 3)
        with torch.no_grad():
            for p_ in lin.parameters():
                p_.fill_(1.0)
                p_.grad = torch.full_like(p_, float(rank + 1))
        sharded.DenseGradAllReduce(lin).reduce()
        assert all(torch.allclose(p_.grad, torch.full_like(p_, (1 + world) / 2)) for p_ in lin.parameters())
        out.put((rank, "ok"))
    except Exception as ex:  # noqa: BLE001
        import traceback
        out.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(180)
def test_sharded_table_and_ranking_world2_gloo():
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29500 + os.getpid() % 500
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=150) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    for rank, msg in res:
        assert msg == "ok", "rank %d: %s" % (rank, msg)


# ---------------------------------------------------------------------------------------------------------------
# bench.sharded_regime (extra.sharded_16M of the N>1 bench lines): its control flow contains collectives, so a
# failure on ONE rank must be agreed on before the next collective instead of leaving the others inside it.
# ---------------------------------------------------------------------------------------------------------------
class _FakeShards(object):
    """CPU stand-in for peer.PeerShardedTable (test infrastructure): local shard only, fetch() gathers local rows."""
    fail_ctor_on = None
    fail_fetch_on = None

    def __init__(self, rows, d, pg, pad_idx):
        rank, world = dist.get_rank(), dist.get_world_size()
        if _FakeShards.fail_ctor_on == rank:
            raise MemoryError("simulated allocation failure")
        self.rank, self.world = rank, world
        self.weight = torch.nn.Parameter(torch.zeros((rows - rank + world - 1) // world, d))

    def fetch(self, index_tensors):
        if _FakeShards.fail_fetch_on == self.rank:
            raise RuntimeError("simulated gather failure")
        ids = index_tensors[0]
        return self.weight.detach()[(ids // self.world) % self.weight.shape[0]], [ids], ids.numel()


def _regime_worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import argparse
        import time

        import bench
        import oracle
        from prodsearch_b200 import ops

        def timer(fn, iters, warmup=3):
            for _ in range(warmup):
                fn()
            t0 = time.perf_counter()
            for _ in range(iters):
                fn()
            return max(time.perf_counter() - t0, 1e-9) / iters
        seen = {}

        def prepare(w, n_local):
            return argparse.Namespace(fits=True, n_items=n_local)

        def topk(qa, w, kk, n_items, id_base, id_stride, mode, prepared):
            if seen.get("fail_topk_on") == rank:
                raise RuntimeError("simulated shortlist failure")
            ids = id_base + id_stride * torch.arange(n_items)
            i, s_ = oracle.topk_lower_id_first((qa @ w[:n_items].t()).numpy(), kk, np.tile(ids.numpy(), (qa.shape[0], 1)))
            return torch.from_numpy(i), torch.from_numpy(s_)

        def merge(ids, sc):
            i, s_ = oracle.merge_shard_topk(list(ids.numpy()), list(sc.numpy()), ids.shape[2])
            seen["merged"] = (i, s_)
            return torch.from_numpy(i), torch.from_numpy(s_)
        ops.catalog_prepare_f16, ops.catalog_topk, ops.topk_merge = prepare, topk, merge
        peaks = {"hbm": 6500.0, "bf16": 1600.0, "src": "test"}
        kw = dict(rows=1001, d=8, m_total=6, k=5, n_gather=64, dev="cpu", table_cls=_FakeShards, timer=timer)
        # 1. every rank healthy: both sections measured, the same numbers on every rank (max over ranks)
        r1 = bench.sharded_regime(peaks, None, rank, world, **kw)
        assert "unavailable" not in r1 and r1["peer_gather_rows"]["ms"] > 0, r1
        cat = r1["catalog_topk_16M"]
        assert cat["queries"] == 6 and cat["queries_per_s"] > 0 and cat["mode"] == "tcgen05_f16", cat
        ids, _ = seen["merged"]
        assert ids.shape == (6, 5) and (ids >= 0).all() and (ids < 1001).all()
        both = [None] * world
        dist.all_gather_object(both, (r1["peer_gather_rows"]["ms"], cat["ms"]))
        assert both[0] == both[1]
        # 2. one rank cannot allocate its shard: every rank reports it and nobody waits inside a collective
        _FakeShards.fail_ctor_on = 1
        r2 = bench.sharded_regime(peaks, None, rank, world, **kw)
        assert "unavailable" in r2 and "catalog_topk_16M" not in r2, r2
        assert ("MemoryError" in r2["unavailable"]) == (rank == 1)
        _FakeShards.fail_ctor_on = None
        # 3. the gather fails on one rank: that section is dropped everywhere, the catalog section still runs
        _FakeShards.fail_fetch_on = 0
        r3 = bench.sharded_regime(peaks, None, rank, world, **kw)
        assert "unavailable" in r3["peer_gather_rows"] and r3["catalog_topk_16M"]["queries_per_s"] > 0, r3
        _FakeShards.fail_fetch_on = None
        # 4. the shard-local top-k fails on one rank: found by the local run before the timed loop's collectives
        seen["fail_topk_on"] = 1
        r4 = bench.sharded_regime(peaks, None, rank, world, **kw)
        assert r4["peer_gather_rows"]["ms"] > 0 and "unavailable" in r4["catalog_topk_16M"], r4
        assert ("simulated shortlist" in r4["catalog_topk_16M"]["unavailable"]) == (rank == 1)
        out.put((rank, "ok"))
    except Exception:  # noqa: BLE001
        import traceback
        out.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(180)
def test_bench_sharded_regime_agrees_on_failures_world2_gloo():
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 30100 + os.getpid() % 500
    procs = [ctx.Process(target=_regime_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=150) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    for rank, msg in res:
        assert msg == "ok", "rank %d: %s" % (rank, msg)
