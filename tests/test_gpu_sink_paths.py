"""Which reduce path the gradient sinks take.  Every equality test passes whether a sink reduces over the sort it
launched next to the backward pass (ops.scatter_sort at the first contribution, ops.scatter_reduce_sorted in
finalize) or falls back to the one-call sort + reduce (ops.scatter_reduce): only the first keeps the counting sort off
the critical path.  The three entry points are wrapped with counters (the sink looks them up on the ops module at
call time), one training step runs, and each table that receives a gradient must show one sort and one reduce over
the same number of index lists, and no one-call reduce."""
import argparse
import collections

import numpy as np
import pytest
import torch

from golden_util import DEFAULTS, Golden

pytestmark = pytest.mark.gpu


@pytest.fixture
def calls(monkeypatch):
    """kind -> [(table_rows, number of index lists or contributions)], in call order."""
    from prodsearch_b200 import ops
    log = collections.defaultdict(list)

    def counted(kind, fn):
        def wrapper(lists, table_rows, *a, **k):
            log[kind].append((int(table_rows), len(lists)))
            return fn(lists, table_rows, *a, **k)
        return wrapper
    for kind in ("scatter_sort", "scatter_reduce_sorted", "scatter_reduce"):
        monkeypatch.setattr(ops, kind, counted(kind, getattr(ops, kind)))
    return log


def assert_presorted(calls, lists_per_table):
    """One sort and one reduce over it per table (rows -> number of index lists), no one-call reduce."""
    got = {k: sorted(v) for k, v in calls.items()}
    want = sorted(lists_per_table.items())
    assert got.get("scatter_sort", []) == want, got
    assert got.get("scatter_reduce_sorted", []) == want, got
    assert got.get("scatter_reduce", []) == [], got


def _cuda(ns, pad_query_to=None, pad_word=None):
    out = argparse.Namespace(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(ns).items()})
    if pad_query_to is not None:
        q = torch.full((out.query_word_idxs.shape[0], pad_query_to), pad_word, dtype=torch.int64, device="cuda")
        q[:, :out.query_word_idxs.shape[1]] = out.query_word_idxs
        out.query_word_idxs = q
    return out


def _tem_cfg(dropout):
    c = dict(DEFAULTS)
    c.update(embedding_size=128, ff_size=512, heads=8, inter_layers=1, neg_per_pos=5, dropout=dropout)
    return argparse.Namespace(**c)


P, V, B = 3001, 2000, 48
# item table: target gather, history rows of the encoder, ranking-loss positives and negatives;
# word table: query pooling, item -> word positives and negatives
TEM_LISTS = {P + 1: 4, V: 3}


@pytest.mark.parametrize("dropout", [0.0, 0.1])        # 0.1: the fused tem_tail ranking loss
@pytest.mark.parametrize("grad_mode", ["dense", "rowsparse"])
def test_local_tem_step_reduces_over_the_presort(calls, grad_mode, dropout):
    from prodsearch_b200 import synth
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    torch.manual_seed(3)
    model = ItemTransformerRanker(_tem_cfg(dropout), "cuda", V, P, None, word_dists=synth.word_dists(V),
                                  grad_mode=grad_mode)
    batch, ni, nw = synth.tem_batch(B, P, V, seed=70)
    model.train()
    model.injected_negatives = (ni.cuda(), nw.cuda())
    loss = model(_cuda(batch))
    model.zero_grad()
    loss.backward()
    torch.cuda.synchronize()
    assert_presorted(calls, TEM_LISTS)


def test_second_backward_without_zero_grad_takes_the_one_call_reduce(calls):
    """Gradient accumulation into the persistent dense buffers reduces this pass on its own and adds it."""
    from prodsearch_b200 import synth
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    torch.manual_seed(3)
    model = ItemTransformerRanker(_tem_cfg(0.0), "cuda", V, P, None, word_dists=synth.word_dists(V))
    batch, ni, nw = synth.tem_batch(B, P, V, seed=70)
    model.train()
    model.injected_negatives = (ni.cuda(), nw.cuda())
    model.zero_grad()
    model(_cuda(batch)).backward()
    assert_presorted(calls, TEM_LISTS)
    calls.clear()
    model(_cuda(batch)).backward()
    torch.cuda.synchronize()
    got = {k: sorted(v) for k, v in calls.items()}
    assert got.get("scatter_sort", []) == [] and got.get("scatter_reduce_sorted", []) == [], got
    assert got.get("scatter_reduce", []) == sorted(TEM_LISTS.items()), got


def test_rtm_pv_step_reduces_over_the_presort(calls):
    from prodsearch_b200.ps_model import ProductRanker
    G = Golden("rtm_pv_trainpv", model_name="review_transformer", embedding_size=32, ff_size=48, heads=4)
    R = int(G.z["cfg/review_count"])
    Vr = G.params["word_embeddings.weight"].shape[0]
    G.cfg.do_subsample_mask = True
    torch.manual_seed(3)
    model = ProductRanker(G.cfg, "cuda", Vr, R, 12, 9, G.inputs["review_words"].tolist(), None,
                          word_dists=np.ones(Vr))
    b = G.batch()
    for k in ("pos_prod_rword_idxs_pvc", "neg_prod_rword_idxs_pvc"):
        if not hasattr(b, k):
            setattr(b, k, None)
    draws = [G.draws[k] for k in sorted(G.draws) if k.startswith("multinomial")]
    model.review_encoder.injected_negatives = draws[0].cuda()
    model.train()
    loss = model(_cuda(b), train_pv=True)
    model.zero_grad()
    loss.backward()
    torch.cuda.synchronize()
    tables = [model.word_embeddings, model.review_encoder.review_embeddings, model.seg_embeddings]
    rows = [t.weight.shape[0] for t in tables]
    assert len(set(rows)) == len(rows)
    for t in tables:
        assert t.weight.grad is not None
    # every table's sort runs over the lists its reduce gets, whatever their number
    sorts = dict(calls["scatter_sort"])
    assert sorted(sorts) == sorted(rows), dict(calls)
    assert_presorted(calls, sorts)


@pytest.mark.parametrize("dropout", [0.0, 0.1])        # 0.1: the fused tem_tail ranking loss
def test_peer_tem_step_reduces_over_the_presort(calls, dropout):
    """Two simulated ranks: each rank's item and word sinks sort over GLOBAL row ids into the staging list."""
    from prodsearch_b200 import peer, synth
    from prodsearch_b200.item_transformer import PeerShardedItemTransformerRanker
    groups = peer.PeerGroup.simulate(2, "cuda")
    batches = [synth.tem_batch(B, P, V, seed=70 + r) for r in range(2)]
    wq = max(b.query_word_idxs.shape[1] for b, _, _ in batches)
    models = []
    for g in groups:                   # every rank's shards exist before the first fetch
        torch.manual_seed(3)
        models.append(PeerShardedItemTransformerRanker(_tem_cfg(dropout), "cuda", V, P, None,
                                                       word_dists=synth.word_dists(V), peer=g))
    for m, (b, ni, nw) in zip(models, batches):
        m.train()
        m.injected_negatives = (ni.cuda(), nw.cuda())
        calls.clear()
        loss = m(_cuda(b, wq, V - 1))
        m.zero_grad()
        loss.backward()
        torch.cuda.synchronize()
        assert_presorted(calls, TEM_LISTS)
