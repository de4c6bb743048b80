"""GPU parity, second batch: the configurations round 1 left untested.

  * TEM ``forward_dotproduct`` at BASELINE ``configs[1]`` UNDER DROPOUT 0.1 (the benchmarked configuration): the
    multipliers the device applied -- the query encoder's keep mask and the fused encoder's Philox streams -- are
    handed to the oracle, which then has to reproduce loss and every gradient;
  * RTM (``ProductRanker``) at BASELINE ``configs[2]`` shape (batch 384, 20 + 30 reviews per sequence, 100 words per
    review, pv and pvc, train_pv both ways) and ParagraphVector at N = 19 200 reviews / R = 300k against the oracle;
  * A11: sampled negatives / corruption masks are exactly what the reference's literal calls draw on the same device
    generator (models/item_transformer.py:447,:268, models/PV.py:57, models/PVC.py:51,:83);
  * the reference's call forms of ParagraphVector.forward / ParagraphVectorCorruption.forward (dense target-word
    embeddings, models/PV.py:50, models/PVC.py:69) against the golden files;
  * rank -> optimizer step -> rank (the shortlist caches must follow raw-pointer parameter updates);
  * gradient accumulation over two backward passes through the row-gradient sinks.
"""
import argparse

import numpy as np
import pytest
import torch

import oracle
from golden_util import DEFAULTS

pytestmark = pytest.mark.gpu


def close(a, b, rtol=1e-5, atol=2e-6, what=""):
    a, b = torch.as_tensor(a).detach().cpu().double(), torch.as_tensor(b).detach().cpu().double()
    err = (a - b).abs()
    bound = atol + rtol * b.abs()
    assert bool((err <= bound).all()), "%s: max err %g at bound %g" % (
        what, float(err.max()), float(bound.flatten()[err.argmax()] if err.numel() else 0))


def cuda_batch(ns):
    return argparse.Namespace(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(ns).items()})


def cpu_leaves(model):
    return {k: v.detach().cpu().clone().requires_grad_(v.dtype.is_floating_point) for k, v in model.state_dict().items()}


def check_all_grads(model, params, pad_rows=("product_emb.weight", "word_embeddings.weight",
                                             "review_encoder.review_embeddings.weight", "user_emb.weight")):
    seen = 0
    for k, p in model.named_parameters():
        g = params[k].grad
        if g is None:
            continue
        g = g.clone()
        if k in pad_rows:
            g[-1] = 0                     # nn.Embedding(padding_idx): the pad row gets no gradient
        scale = float(g.abs().max()) + 1e-12
        got = p.grad if p.grad is not None else torch.zeros_like(p)
        close(got, g, rtol=1e-4, atol=max(2e-5 * scale, 2e-7), what="grad " + k)
        seen += 1
    assert seen >= 8


def _cfg(**kw):
    c = dict(DEFAULTS)
    c.update(dict(embedding_size=128, ff_size=512, heads=8, inter_layers=1, neg_per_pos=5))
    c.update(kw)
    return argparse.Namespace(**c)


# ------------------------------------------------------------------ TEM under dropout (the benchmarked configuration)
@pytest.mark.parametrize("qenc,B", [("fs", 384), ("avg", 50)])
def test_tem_forward_dropout_matches_oracle_with_device_multipliers(qenc, B, monkeypatch):
    from prodsearch_b200 import functional as F_
    from prodsearch_b200 import synth
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    from oracle import philox
    p = 0.1
    cfg = _cfg(model_name="item_transformer", dropout=p, query_encoder_name=qenc)
    torch.manual_seed(11)
    P, V, K, L = 18000, 32000, 5, 20
    model = ItemTransformerRanker(cfg, "cuda", V, P, None, word_dists=synth.word_dists(V))
    with torch.no_grad():
        model.word_bias.normal_(0, 0.1)
    batch, neg_items, neg_words = synth.tem_batch(B, P, V, L=L, W=1, K=K, seed=23)
    params = cpu_leaves(model)
    keeps = []
    real_keep = F_._dropout_keep

    def spy(shape, pp, training, device):
        k = real_keep(shape, pp, training, device)
        keeps.append(k)
        return k
    monkeypatch.setattr(F_, "_dropout_keep", spy)
    model.train()
    model.injected_negatives = (neg_items.cuda(), neg_words.cuda())
    loss = model(cuda_batch(batch))
    model.zero_grad()
    loss.backward()
    assert len(keeps) == 1 and keeps[0] is not None             # the query encoder's dropout, drawn once (:450)
    seed = int(model.transformer_encoder._drop_seed.item())
    d, H, ff, T = 128, 8, 512, 1 + L
    m = philox.encoder_dropout_muls(seed, p, B, 1 + K, T, H, d, ff, 0)     # rows = sequence * (1 + K) + copy
    pos, neg = {}, {}
    for k, v in m.items():
        v = torch.from_numpy(v).view((B, 1 + K) + v.shape[1:])
        pos[k] = v[:, 0].contiguous()
        neg[k] = v[:, 1:].reshape((B * K,) + v.shape[2:]).contiguous()
    drop = dict(query_keep=keeps[0].cpu(), enc_pos=pos, enc_neg=neg)
    torch.set_num_threads(8)
    ref, ref_ps, ref_il = oracle.tem_forward(params, cfg, batch.query_word_idxs, batch.target_prod_idxs,
                                             batch.u_item_idxs, batch.pos_iword_idxs, neg_items, neg_words,
                                             training=True, drop=drop)
    ref.backward()
    close(loss, ref, what="loss")
    close(model.ps_loss, ref_ps, what="ps_loss")
    close(model.item_loss, ref_il, what="item_loss")
    check_all_grads(model, params)
    # and the multipliers are a genuine dropout draw: zeros at about rate p, the rest 1/(1-p)
    km = keeps[0]
    assert abs(float((km == 0).float().mean()) - p) < 0.02 and bool(((km == 0) | ((km - 1 / (1 - p)).abs() < 1e-6)).all())


# ------------------------------------------------------------------ RTM at BASELINE configs[2] shape
_RTM_TABLE = {}


def _review_table(R, V, Wr):
    key = (R, V, Wr)
    if key not in _RTM_TABLE:
        from prodsearch_b200 import synth
        _RTM_TABLE[key] = synth.review_words_table(R, V, Wr)
    return _RTM_TABLE[key]


@pytest.mark.parametrize("enc,train_pv,B", [("pv", True, 384), ("pv", False, 384), ("pvc", True, 384),
                                            ("pvc", False, 96)])
def test_rtm_baseline_shape_vs_oracle(enc, train_pv, B):
    from prodsearch_b200 import synth
    from prodsearch_b200.ps_model import ProductRanker
    V, R, P, U, K, Ru, Ri, Wr = 32000, 300000, 18000, 35000, 5, 20, 30, 100
    rate = 0.9                                                   # the reference's default corrupt_rate (main.py:114)
    cfg = _cfg(model_name="review_transformer", review_encoder_name=enc, review_word_limit=Wr, corrupt_rate=rate,
               do_subsample_mask=True, review_pad_idx=R - 1, use_user_emb=(enc == "pv"), use_item_emb=(enc == "pv"))
    rw = _review_table(R, V, Wr)
    torch.manual_seed(3)
    model = ProductRanker(cfg, "cuda", V, R, P, U, rw, None, word_dists=synth.word_dists(V))
    batch, draws = synth.rtm_batch(B, rw, V, P, U, Ru=Ru, Ri=Ri, W=1, K=K, pvc=(enc == "pvc"), train_pv=train_pv, seed=31)
    Rc = Ru + Ri
    masks = []
    if enc == "pvc":
        g = torch.Generator().manual_seed(7)
        masks = [(torch.rand(B * Rc, Wr, generator=g) < rate).float(), (torch.rand(B * K * Rc, Wr, generator=g) < rate).float()]
    params = cpu_leaves(model)
    model.train()
    if draws["multinomial"]:
        model.review_encoder.injected_negatives = draws["multinomial"][0].cuda()
    if masks:
        model.review_encoder.injected_corruption = [m.clone() for m in masks]
    loss = model(cuda_batch(batch), train_pv=train_pv)
    model.zero_grad()
    loss.backward()
    torch.set_num_threads(8)
    ref, _, _ = oracle.rtm_forward(params, cfg, batch, train_pv, draws["multinomial"][0] if draws["multinomial"] else None,
                                   [m.clone() for m in masks], training=True)
    ref.backward()
    close(loss, ref, what="loss")
    check_all_grads(model, params)


def test_pv_train_step_shape_vs_oracle():
    """ParagraphVector alone at the RTM step's size: N = 384 * 50 = 19 200 reviews of a 300k-review table."""
    from prodsearch_b200 import synth
    from prodsearch_b200.pv import ParagraphVector
    V, R, d, N, W, K = 32000, 300000, 128, 19200, 1, 5
    g = torch.Generator().manual_seed(5)
    wemb = torch.nn.Embedding(V, d, padding_idx=V - 1)
    pv = ParagraphVector(wemb, torch.as_tensor(synth.word_dists(V)), R, dropout=0.0).cuda()
    with torch.no_grad():
        wemb.weight.normal_(generator=None)
        pv.review_embeddings.weight.normal_()
    ids = torch.randint(0, R, (N,), generator=g)
    ids[::37] = R - 1
    words = torch.randint(0, V - 1, (N, W), generator=g)
    mask = (torch.rand(N, W, generator=g) < 0.9)
    negs = torch.randint(0, V - 1, (N * W * K,), generator=g)
    pv.injected_negatives = negs.cuda()
    emb, loss = pv(ids.cuda(), words.cuda(), mask.cuda(), K)
    up_e, up_l = torch.randn(N, d, generator=g), torch.randn(N, 1, generator=g)
    ((emb * up_e.cuda()).sum() + (loss * up_l.cuda()).sum()).backward()
    rt = pv.review_embeddings.weight.detach().cpu().clone().requires_grad_(True)
    wt = wemb.weight.detach().cpu().clone().requires_grad_(True)
    r_emb, r_loss = oracle.pv_forward(rt, wt, ids, words, mask, negs, K)
    ((r_emb * up_e).sum() + (r_loss * up_l).sum()).backward()
    assert torch.equal(emb.cpu(), r_emb.detach())                # gathered rows: bit exact
    close(loss, r_loss, what="loss")
    gr, gw = rt.grad.clone(), wt.grad.clone()
    gr[-1] = 0
    gw[-1] = 0
    for got, ref, what in ((pv.review_embeddings.weight.grad, gr, "review table grad"), (wemb.weight.grad, gw, "word table grad")):
        close(got, ref, rtol=1e-4, atol=max(2e-5 * float(ref.abs().max()), 2e-7), what=what)   # sums with cancellation


# ------------------------------------------------------------------ A11: sampled indices on the device generator
def test_sampled_negatives_equal_reference_draws():
    """Same device generator state -> the ids the reference's literal calls draw, in its call order."""
    from prodsearch_b200 import synth
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    cfg = _cfg(model_name="item_transformer")
    P, V, B, W, K = 18000, 32000, 384, 1, 5
    model = ItemTransformerRanker(cfg, "cuda", V, P, None, word_dists=synth.word_dists(V))
    torch.manual_seed(1234)
    neg_items, neg_words = model._draw_negatives(B, W, K)
    torch.manual_seed(1234)
    prod_dists = torch.ones(P, device="cuda")                                     # item_transformer.py:33
    word_dists = torch.tensor(synth.word_dists(V), device="cuda")                # :30-32
    ref_items = torch.multinomial(prod_dists, B * K, replacement=True).view(B, -1)     # :447-448
    ref_words = torch.multinomial(word_dists, B * W * K, replacement=True)             # :268
    assert torch.equal(neg_items, ref_items)
    assert torch.equal(neg_words.reshape(-1), ref_words)
    assert int(neg_items.max()) < P and int(neg_words.max()) < V - 1                # pad word has probability 0
    # the whole forward consumes the generator exactly like the reference's forward does (dropout 0: two draws)
    batch, _, _ = synth.tem_batch(B, P, V, seed=2)
    model.train()
    torch.manual_seed(99)
    model(cuda_batch(batch))
    after_model = torch.cuda.get_rng_state()
    torch.manual_seed(99)
    torch.multinomial(prod_dists, B * K, replacement=True)
    torch.multinomial(word_dists, B * W * K, replacement=True)
    assert torch.equal(after_model, torch.cuda.get_rng_state())


def test_reproducible_draws_are_the_inverse_cdf_of_the_device_uniforms():
    """reproducible_draws: every id is the inverse CDF (float64, summed on the host) of one torch.rand draw of the device
    generator, items first, then words -- a pure function of the generator state, so one seed gives the same ids on
    every run; the ids follow the reference's distributions (uniform items; word_dists, the pad word never); inside a
    captured step they change from replay to replay."""
    from prodsearch_b200 import synth
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    cfg = _cfg(model_name="item_transformer")
    P, V, W, K, n = 18000, 32000, 1, 5, 200_000
    wd = np.asarray(synth.word_dists(V), dtype=np.float64)
    model = ItemTransformerRanker(cfg, "cuda", V, P, None, word_dists=wd)
    model.reproducible_draws = True
    torch.manual_seed(1234)
    neg_items, neg_words = model._draw_negatives(n // K, W, K)
    torch.manual_seed(1234)
    u_items = torch.rand(n, dtype=torch.float64, device="cuda").cpu()
    u_words = torch.rand(n, dtype=torch.float64, device="cuda").cpu()
    for got, u, p in ((neg_items, u_items, np.ones(P)), (neg_words, u_words, np.float32(wd).astype(np.float64))):
        cdf = np.cumsum(p)
        want = np.searchsorted(cdf / cdf[-1], u.numpy(), side="right")
        assert np.array_equal(got.reshape(-1).cpu().numpy(), want)
    items, words = neg_items.reshape(-1).cpu().numpy(), neg_words.reshape(-1).cpu().numpy()
    assert items.min() >= 0 and items.max() < P and words.min() >= 0 and words.max() < V - 1
    # frequencies against the distributions: every id's count within 6 sigma of its expectation
    for ids, p in ((items, np.full(P, 1.0 / P)), (words, wd / wd.sum())):
        cnt = np.bincount(ids, minlength=len(p)).astype(np.float64)
        assert np.all(np.abs(cnt - n * p) <= 6 * np.sqrt(n * p * (1 - p)) + 1)
    g = torch.cuda.CUDAGraph()
    torch.manual_seed(5)
    with torch.cuda.graph(g):
        ni, nw = model._draw_negatives(64, W, K)
    g.replay()
    first = (ni.clone(), nw.clone())
    g.replay()
    assert not torch.equal(first[0], ni) and not torch.equal(first[1], nw)


def test_pv_pvc_draws_equal_reference_draws(monkeypatch):
    from prodsearch_b200 import synth
    from prodsearch_b200.pv import ParagraphVector
    from prodsearch_b200.pvc import ParagraphVectorCorruption
    V, d, N, W, K, Wr, rate = 5000, 64, 700, 3, 5, 40, 0.9
    wd = torch.tensor(synth.word_dists(V), device="cuda")
    g = torch.Generator().manual_seed(8)
    words = torch.randint(0, V - 1, (N, W), generator=g).cuda()
    mask = torch.ones(N, W, dtype=torch.uint8).cuda()
    rwords = torch.randint(0, V - 1, (N, Wr), generator=g).cuda()
    seen = {}
    real_m, real_b = torch.multinomial, torch.bernoulli

    def spy_m(*a, **k):
        out = real_m(*a, **k)
        seen.setdefault("m", []).append(out.clone())
        return out

    def spy_b(*a, **k):
        out = real_b(*a, **k)
        seen.setdefault("b", []).append(out.clone())
        return out
    wemb = torch.nn.Embedding(V, d, padding_idx=V - 1).cuda()
    pv = ParagraphVector(wemb, wd, 1000, dropout=0.0).cuda()
    pvc = ParagraphVectorCorruption(wemb, wd, rate, dropout=0.0).cuda()
    monkeypatch.setattr(torch, "multinomial", spy_m)
    monkeypatch.setattr(torch, "bernoulli", spy_b)
    torch.manual_seed(77)
    pv(torch.randint(0, 999, (N,), generator=g).cuda(), words, mask, K)
    pvc(words, mask, rwords, K)
    monkeypatch.undo()
    torch.manual_seed(77)
    ref_pv = torch.multinomial(wd, N * W * K, replacement=True)                       # PV.py:57
    probs = torch.empty(N, Wr, device="cuda").fill_(rate)                             # PVC.py:49 (.new().resize_().fill_())
    ref_mask = torch.bernoulli(probs)                                                 # PVC.py:51, called from :78
    ref_pvc = torch.multinomial(wd, N * W * K, replacement=True)                      # PVC.py:83
    assert torch.equal(seen["m"][0], ref_pv)
    assert torch.equal(seen["b"][0], ref_mask)
    assert torch.equal(seen["m"][1], ref_pvc)


# ------------------------------------------------------------------ reference call forms of PV / PVC (dense target rows)
def test_pv_reference_signature_golden(golden_dir):
    from prodsearch_b200.pv import ParagraphVector
    z = np.load(golden_dir + "/pv.npz")
    wt = torch.from_numpy(z["word_table"])
    V, d = wt.shape
    wemb = torch.nn.Embedding(V, d, padding_idx=V - 1)
    pv = ParagraphVector(wemb, torch.ones(V), z["review_table"].shape[0], dropout=0.0).cuda()
    with torch.no_grad():
        wemb.weight.copy_(wt)
        pv.review_embeddings.weight.copy_(torch.from_numpy(z["review_table"]))
    pv.injected_negatives = torch.from_numpy(z["neg_word_idxs"]).cuda()
    review_word_emb = wemb(torch.from_numpy(z["pos_word_idxs"]).cuda())              # what ps_model.py:270 passes
    emb, loss = pv(torch.from_numpy(z["review_ids"]).cuda(), review_word_emb, torch.from_numpy(z["word_mask"]).cuda(),
                   int(z["n_negs"]))
    close(emb, z["review_emb"], rtol=0, atol=0)
    close(loss, z["loss"])
    ((emb * torch.from_numpy(z["up_emb"]).cuda()).sum() + (loss * torch.from_numpy(z["up_loss"]).cuda()).sum()).backward()
    close(wemb.weight.grad, z["grad_word_table"], rtol=1e-4)
    close(pv.review_embeddings.weight.grad, z["grad_review_table"], rtol=1e-4)


def test_pvc_reference_signature_golden(golden_dir):
    from prodsearch_b200.pvc import ParagraphVectorCorruption
    z = np.load(golden_dir + "/pvc.npz")
    wt = torch.from_numpy(z["word_table"])
    V, d = wt.shape
    wemb = torch.nn.Embedding(V, d, padding_idx=V - 1)
    pvc = ParagraphVectorCorruption(wemb, torch.ones(V), float(z["corrupt_rate"]), dropout=0.0).cuda()
    with torch.no_grad():
        wemb.weight.copy_(wt)
    pvc.injected_negatives = torch.from_numpy(z["neg_word_idxs"]).cuda()
    pvc.injected_corruption = [torch.from_numpy(z["corrupt_mask"])]
    review_word_emb = wemb(torch.from_numpy(z["pos_word_idxs"]).cuda())              # ps_model.py:273-274
    emb, loss = pvc(review_word_emb, torch.from_numpy(z["word_mask"]).cuda(), torch.from_numpy(z["rword_idxs_pvc"]).cuda(),
                    int(z["n_negs"]))
    close(emb, z["review_emb"])
    close(loss, z["loss"])
    ((emb * torch.from_numpy(z["up_emb"]).cuda()).sum() + (loss * torch.from_numpy(z["up_loss"]).cuda()).sum()).backward()
    close(wemb.weight.grad, z["grad_word_table"], rtol=1e-4)


# ------------------------------------------------------------------ caches follow raw-pointer parameter updates
def test_rank_train_rank_follows_the_updated_table():
    """rank_catalog -> one FusedAdam step (writes the table through raw pointers: tensor._version does not move)
    -> rank_catalog must rank the UPDATED table; the fp16 shortlist copy / error bound / row-norm bound are rebuilt."""
    from prodsearch_b200 import _lib, synth
    from prodsearch_b200.graph_step import GraphedTrainStep
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    from prodsearch_b200.optimizers import Optimizer
    cfg = _cfg(model_name="item_transformer")
    P, V, B = 60000, 8000, 64
    torch.manual_seed(4)
    model = ItemTransformerRanker(cfg, "cuda", V, P, None, word_dists=synth.word_dists(V))
    opt = Optimizer("adam", 0.5, 5.0)                              # a large step: the ranking really changes
    opt.set_parameters(list(model.named_parameters()))
    batch, _, _ = synth.tem_batch(B, P, V, seed=9)
    b = cuda_batch(batch)
    for mode in (_lib.TOPK_TC16, _lib.TOPK_TC):
        model.eval()
        ids0, sc0 = model.rank_catalog(b, k=100, mode=mode)
        model.train()
        loss = model(b)
        model.zero_grad()
        loss.backward()
        opt.step()
        model.eval()
        ids1, sc1 = model.rank_catalog(b, k=100, mode=mode)
        ide, sce = model.rank_catalog(b, k=100, mode=_lib.TOPK_EXACT)
        assert torch.equal(ids1, ide) and torch.equal(sc1, sce)
        assert not torch.equal(sc0, sc1)
    # the same through CUDA-graph replays (the eager loss above still holds its autograd graph, whose AccumulateGrad
    # nodes are bound to the stream of that eager pass: release it before capturing)
    del loss
    model.train()
    step = GraphedTrainStep(model, opt, b)
    model.eval()
    model.rank_catalog(b, k=100)
    model.train()
    step(b)
    step(b)
    model.eval()
    ids1, sc1 = model.rank_catalog(b, k=100)
    ide, sce = model.rank_catalog(b, k=100, mode=_lib.TOPK_EXACT)
    assert torch.equal(ids1, ide) and torch.equal(sc1, sce)


# ------------------------------------------------------------------ gradient accumulation through the sinks
def test_two_backward_passes_accumulate_table_gradients():
    from prodsearch_b200 import synth
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    cfg = _cfg(model_name="item_transformer", sim_func="bias_product")
    P, V, B = 3000, 4000, 48
    torch.manual_seed(6)
    model = ItemTransformerRanker(cfg, "cuda", V, P, None, word_dists=synth.word_dists(V))
    b1, ni1, nw1 = synth.tem_batch(B, P, V, seed=1)
    b2, ni2, nw2 = synth.tem_batch(B, P, V, seed=2)
    model.train()

    def run(batch, ni, nw, zero):
        model.injected_negatives = (ni.cuda(), nw.cuda())
        loss = model(cuda_batch(batch))
        if zero:
            model.zero_grad()
        loss.backward()
        return {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    g1 = run(b1, ni1, nw1, True)
    g2 = run(b2, ni2, nw2, True)
    model.zero_grad()
    run(b1, ni1, nw1, False)
    both = run(b2, ni2, nw2, False)                               # no zero_grad in between: torch semantics = sum
    for k in g1:
        scale = float((g1[k] + g2[k]).abs().max()) + 1e-12
        close(both[k], g1[k] + g2[k], rtol=1e-5, atol=1e-6 * scale, what="accumulated grad " + k)
    # and a following ordinary step starts from zero again
    g1b = run(b1, ni1, nw1, True)
    for k in g1:
        assert torch.equal(g1b[k], g1[k]), k


# ------------------------------------------------------------------ 1M-item catalog: exact mode against fp64
def test_catalog_topk_1m_spot_check_fp64():
    """BASELINE configs[3] exactly (1M items, d = 128, top-100): a few queries of the exact mode (the checker of the
    tensor-core modes at this size) against an fp64 score matrix computed on the device."""
    from prodsearch_b200 import _lib, ops
    n, m, k = 1_000_000, 384, 100
    g = torch.Generator(device="cuda").manual_seed(m + n)
    E = torch.randn(n + 1, 128, generator=g, device="cuda")
    Q = torch.randn(m, 128, generator=g, device="cuda")
    ids, sc = ops.catalog_topk(Q, E, k, n_items=n, mode=_lib.TOPK_EXACT)
    ids16, sc16 = ops.catalog_topk(Q, E, k, n_items=n, mode=_lib.TOPK_TC16, prepared=ops.catalog_prepare_f16(E, n))
    assert torch.equal(ids, ids16) and torch.equal(sc, sc16)
    rows = torch.tensor([0, 1, 127, 128, 200, 255, 256, 383], device="cuda")
    S = Q[rows].double() @ E[:n].double().t()
    tol = 1e-5 * Q[rows].double().norm(dim=1, keepdim=True) * E[:n].double().norm(dim=1).max()
    got = torch.gather(S, 1, ids[rows])
    assert bool(((got - sc[rows].double()).abs() <= tol).all())
    ref_s, ref_i = torch.topk(S, k, dim=1)
    assert bool(((ref_s - sc[rows].double()).abs() <= tol).all())
    # ids are defined at the positions whose score gaps to both neighbours exceed the fp32 noise
    ref_s1 = torch.topk(S, k + 1, dim=1).values
    gaps = ref_s1[:, :-1] - ref_s1[:, 1:]                                      # [rows, k]: gap below position j
    inf = torch.full_like(gaps[:, :1], float("inf"))
    clear = (gaps > 2 * tol) & (torch.cat([inf, gaps[:, :-1]], dim=1) > 2 * tol)
    assert float(clear.float().mean()) > 0.5
    assert torch.equal(ids[rows][clear], ref_i[clear])
    d = sc[:, 1:] - sc[:, :-1]
    assert bool((d <= 0).all()) and bool((ids[:, 1:][d == 0] > ids[:, :-1][d == 0]).all())
