"""One GPU, one rank: the all-to-all (``ShardedItemTransformerRanker``) and the peer-sharded TEM take the training
step, the evaluation and the catalog ranking of the unsharded model.  Both row-sharded models share the model's step
body and differ only in where the rows come from; with one rank the shard is the whole table, so the loss, every
gradient, the candidate scores and the exact full-catalog top-k must equal the local model's.  The all-to-all model
needs a process group, so the check runs in one spawned child that forms a one-rank NCCL group."""
import argparse
import os
import sys
import traceback

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P, V, B = 3001, 2000, 48


def _step(model, batch, negs):
    """One training step on ``batch`` with fixed negatives; the dropout draws start from the same generator state."""
    model.train()
    model.injected_negatives = negs
    torch.manual_seed(11)
    loss = model(batch)
    model.zero_grad()
    loss.backward()
    if hasattr(model, "sync_grads"):
        model.sync_grads()
    torch.cuda.synchronize()
    return float(loss)


def _check(dropout):
    from golden_util import DEFAULTS
    from prodsearch_b200 import _lib, peer, synth
    from prodsearch_b200.item_transformer import (ItemTransformerRanker, PeerShardedItemTransformerRanker,
                                                  ShardedItemTransformerRanker)
    cfg = dict(DEFAULTS)
    cfg.update(embedding_size=128, ff_size=512, heads=8, inter_layers=1, neg_per_pos=5, dropout=dropout)
    cfg = argparse.Namespace(**cfg)
    batch, ni, nw = synth.tem_batch(B, P, V, seed=70)
    b = argparse.Namespace(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(batch).items()})
    negs = (ni.cuda(), nw.cuda())
    g = torch.Generator(device="cuda").manual_seed(5)
    tb = argparse.Namespace(**vars(b))
    tb.candi_prod_idxs = torch.randint(0, P, (B, 17), device="cuda", generator=g)
    q = torch.randn(7, 128, device="cuda", generator=g)

    def build(cls, **kw):
        torch.manual_seed(3)
        return cls(cfg, "cuda", V, P, None, word_dists=synth.word_dists(V), **kw)
    ref = build(ItemTransformerRanker)
    ref_loss = _step(ref, b, negs)
    ref_grads = {k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in ref.named_parameters()}
    ref.eval()
    ref_scores = ref.test(tb)
    ref_ids, ref_sc = ref.rank_catalog(q, k=100, mode=_lib.TOPK_EXACT)
    for name, m in (("all-to-all", build(ShardedItemTransformerRanker)),
                    ("peer", build(PeerShardedItemTransformerRanker, peer=peer.PeerGroup(device="cuda")))):
        where = "%s, dropout %g" % (name, dropout)
        loss = _step(m, b, negs)
        assert abs(loss - ref_loss) <= 1e-5 * abs(ref_loss), (where, loss, ref_loss)
        for k, p in m.named_parameters():
            gr = p.grad if p.grad is not None else torch.zeros_like(p)
            scale = float(ref_grads[k].abs().max()) + 1e-12
            err = float((gr - ref_grads[k]).abs().max())
            assert err <= 1e-4 * scale + 2e-7, (where, k, err, scale)
        m.eval()
        assert torch.allclose(m.test(tb), ref_scores, rtol=1e-4, atol=1e-5), where
        ids, sc = m.rank_catalog(q, k=100, mode=_lib.TOPK_EXACT)
        assert torch.equal(ids, ref_ids) and torch.equal(sc, ref_sc), where


def _child(port, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        for dropout in (0.0, 0.1):          # 0.1: the fused tem_tail ranking loss; 0.0: ns_loss
            _check(dropout)
        out.put("ok")
    except Exception:  # noqa: BLE001
        out.put(traceback.format_exc())
    finally:
        dist.destroy_process_group()


def test_sharded_models_match_local_model_on_one_rank():
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    proc = ctx.Process(target=_child, args=(30700 + os.getpid() % 500, out))
    proc.start()
    try:
        msg = out.get(timeout=600)
    finally:
        proc.join(timeout=60)
        if proc.is_alive():
            proc.kill()
            proc.join()
    assert msg == "ok", msg
