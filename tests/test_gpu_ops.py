"""GPU parity of every C-ABI entry point against the CPU oracle (same seeded inputs).

Bit-exact for gathered rows, indices and top-k ids; losses / means / gradients within
1e-5 relative (BASELINE.json north_star tolerance), stated per test."""
import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

RTOL = 1e-5


@pytest.fixture(scope="module")
def ops():
    from prodsearch_b200 import ops as _ops
    return _ops


def dev(t):
    return t.cuda()


def close(a, b, rtol=RTOL, atol=1e-6):
    a, b = torch.as_tensor(a).detach().cpu().double(), torch.as_tensor(b).detach().cpu().double()
    err = (a - b).abs()
    bound = atol + rtol * b.abs()
    assert bool((err <= bound).all()), "max err %g (bound %g)" % (float(err.max()), float(bound.max()))


# ---------------------------------------------------------------- G1
@pytest.mark.parametrize("d", [128, 64, 132, 512])
@pytest.mark.parametrize("n", [0, 1, 37, 5000])
def test_gather_rows_bit_exact(ops, d, n):
    g = torch.Generator().manual_seed(d * 7 + n)
    table = torch.randn(301, d, generator=g)
    idx = torch.randint(0, 301, (n,), generator=g)
    out = ops.gather_rows(dev(table), dev(idx))
    assert torch.equal(out.cpu(), table[idx])


def test_gather_rows_shapes_and_bounds(ops):
    g = torch.Generator().manual_seed(3)
    table = torch.randn(50, 128, generator=g)
    idx = torch.randint(0, 50, (6, 5, 3), generator=g)
    out = ops.gather_rows(dev(table), dev(idx))
    assert out.shape == (6, 5, 3, 128) and torch.equal(out.cpu(), table[idx])
    bad = idx.clone().view(-1)
    bad[7] = 50
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = ops.gather_rows(dev(table), dev(bad), err_flag=flag)
    assert int(flag.item()) == 1 and float(out[7].abs().sum()) == 0.0


def test_gather_rows_large_table_bit_exact(ops):
    # 2M x 128 fp32 = 1 GiB table (> L2): rows really come from HBM
    g = torch.Generator(device="cuda").manual_seed(5)
    table = torch.randn(2_000_000, 128, generator=g, device="cuda")
    idx = torch.randint(0, 2_000_000, (300_000,), generator=g, device="cuda")
    out = ops.gather_rows(table, idx)
    assert torch.equal(out, table[idx])


# ---------------------------------------------------------------- G4
@pytest.mark.parametrize("d,w", [(128, 12), (128, 100), (64, 5), (256, 33)])
def test_meanpool_vs_oracle(ops, d, w):
    g = torch.Generator().manual_seed(d + w)
    V, n = 97, 41
    table = torch.randn(V, d, generator=g)
    idx = torch.randint(0, V - 1, (n, w), generator=g)
    idx[0, 1:] = V - 1
    idx[1, :] = V - 1                       # fully padded row -> count clamps to 1, mean 0
    idx[2, w // 2:] = V - 1
    ref = oracle.masked_mean(table[idx], idx.ne(V - 1))
    out, _, inv = ops.gather_meanpool(dev(table), dev(idx), pad_idx=V - 1, want_inv_count=True)
    close(out, ref)
    close(inv, 1.0 / idx.ne(V - 1).sum(-1).clamp(min=1).float())
    # explicit uint8 mask (RTM review-word masks) + PVC token scale + dropout multiplier
    mask = (torch.rand(n, w, generator=g) > 0.3)
    scale = torch.where(torch.rand(n, w, generator=g) < 0.5, torch.zeros(()), torch.full((), 2.0))
    keep = torch.where(torch.rand(n, d, generator=g) < 0.1, torch.zeros(()), torch.full((), 1 / 0.9))
    ref2 = oracle.masked_mean(table[idx] * scale.unsqueeze(-1), mask) * keep
    out2, mean2, _ = ops.gather_meanpool(dev(table), dev(idx), mask=dev(mask.to(torch.uint8)), tok_scale=dev(scale),
                                         keep_scale=dev(keep), want_mean=True)
    close(out2, ref2)
    close(mean2, ref2)
    tw = ops.token_weights(dev(idx), pad_idx=V - 1)
    m = idx.ne(V - 1).float()
    close(tw, m / m.sum(-1, keepdim=True).clamp(min=1))


@pytest.mark.parametrize("d", [128, 64])
def test_fs_encoder_fwd_bwd(ops, d):
    g = torch.Generator().manual_seed(d)
    V, n, w = 60, 19, 7
    table = torch.randn(V, d, generator=g)
    idx = torch.randint(0, V - 1, (n, w), generator=g)
    idx[3, 2:] = V - 1
    W = (torch.randn(d, d, generator=g) * (2.0 / (2 * d)) ** 0.5).requires_grad_(True)
    b = (torch.randn(d, generator=g) * 0.1).requires_grad_(True)
    x = table[idx].requires_grad_(True)
    ref = oracle.fs_encoder(x, idx.ne(V - 1), W, b)
    out, mean, _ = ops.gather_meanpool(dev(table), dev(idx), pad_idx=V - 1, fs_weight=dev(W.detach()),
                                       fs_bias=dev(b.detach()))
    close(out, ref)
    up = torch.randn(n, d, generator=g)
    (ref * up).sum().backward()
    gw, gb, gm = ops.fs_bwd(dev(up), out, mean, None, dev(W.detach()))
    close(gw, W.grad, rtol=1e-4, atol=1e-6)
    close(gb, b.grad, rtol=1e-4, atol=1e-6)
    # grad_mean, spread over valid tokens, is the gradient of the gathered rows
    tw = idx.ne(V - 1).float()
    tw = tw / tw.sum(-1, keepdim=True).clamp(min=1)
    close(gm.cpu().unsqueeze(1) * tw.unsqueeze(-1), x.grad, rtol=1e-4, atol=1e-6)


def test_text_encoder_golden(ops, golden_dir):
    z = np.load(golden_dir + "/text_encoder.npz")
    x = torch.from_numpy(z["x"])
    n, w, d = x.shape
    table = x.reshape(n * w, d).contiguous()
    idx = torch.arange(n * w).view(n, w)
    mask = torch.from_numpy(z["mask"]).to(torch.uint8)
    out, _, _ = ops.gather_meanpool(dev(table), dev(idx), mask=dev(mask))
    close(out, z["mean"])
    out, mean, _ = ops.gather_meanpool(dev(table), dev(idx), mask=dev(mask), fs_weight=dev(torch.from_numpy(z["fs_w"])),
                                       fs_bias=dev(torch.from_numpy(z["fs_b"])))
    close(out, z["fs_out"])
    gw, gb, gm = ops.fs_bwd(dev(torch.from_numpy(z["upstream"])), out, mean, None, dev(torch.from_numpy(z["fs_w"])))
    close(gw, z["grad_w"], rtol=1e-4)
    close(gb, z["grad_b"], rtol=1e-4)


# ---------------------------------------------------------------- G3 / A4
@pytest.mark.parametrize("d,w,k", [(128, 1, 5), (128, 3, 4), (64, 2, 3), (256, 1, 16)])
def test_ns_loss_vs_oracle(ops, d, w, k):
    g = torch.Generator().manual_seed(d + 10 * w + k)
    V, n = 83, 29
    table = (torch.randn(V, d, generator=g) * 0.3).requires_grad_(True)
    bias = (torch.randn(V, generator=g) * 0.3).requires_grad_(True)
    anchor = (torch.randn(n, d, generator=g) * 0.5).requires_grad_(True)
    pos = torch.randint(0, V - 1, (n, w), generator=g)
    pos[1, w - 1] = V - 1
    pos[2, :] = V - 1
    neg = torch.randint(0, V - 1, (n * w * k,), generator=g)
    ref = oracle.ns_word_loss(anchor, table, pos, neg, pos.ne(V - 1), k, bias).squeeze(-1)
    loss, cp, cn, ga, _ = ops.ns_loss(dev(anchor.detach()), dev(table.detach()), dev(pos), dev(neg.view(n, w, k)),
                                      bias=dev(bias.detach()), pad_idx=V - 1)
    close(loss, ref)
    up = torch.randn(n, generator=g)
    (ref * up).sum().backward()
    close(ga.cpu() * up.unsqueeze(1), anchor.grad, rtol=1e-4, atol=1e-6)
    # coefficients reproduce the table and bias gradients through an index_add
    coef = torch.cat([cp.cpu().unsqueeze(-1), cn.cpu()], dim=-1) * up.view(n, 1, 1)
    rows = torch.cat([pos.unsqueeze(-1), neg.view(n, w, k)], dim=-1)
    gt = torch.zeros(V, d).index_add_(0, rows.view(-1), (coef.unsqueeze(-1) * anchor.detach().view(n, 1, 1, d)).view(-1, d))
    gbias = torch.zeros(V).index_add_(0, rows.view(-1), coef.view(-1))
    close(gt, table.grad, rtol=1e-4, atol=1e-6)
    close(gbias, bias.grad, rtol=1e-4, atol=1e-6)


def test_score_loss_tail_vs_oracle(ops):
    """TEM tail (item_transformer.py:485,:493-514): per-negative anchors, pos_weight, product bias."""
    g = torch.Generator().manual_seed(77)
    P, n, k, d = 90, 33, 5, 128
    E = (torch.randn(P + 1, d, generator=g) * 0.3).requires_grad_(True)
    pb = (torch.randn(P + 1, generator=g) * 0.2).requires_grad_(True)
    pos_out = (torch.randn(n, d, generator=g) * 0.5).requires_grad_(True)
    neg_out = (torch.randn(n * k, d, generator=g) * 0.5).requires_grad_(True)
    tgt = torch.randint(0, P, (n,), generator=g)
    neg = torch.randint(0, P, (n, k), generator=g)
    ps = (pos_out * E[tgt]).sum(-1) + pb[tgt]
    ns = (neg_out * E[neg.view(-1)]).sum(-1).view(n, k) + pb[neg.view(-1)].view(n, k)
    wts = torch.ones(n, 1 + k)
    wts[:, 0] = k
    tg = torch.cat([torch.ones(n, 1), torch.zeros(n, k)], -1)
    ref = oracle.bce_with_logits(torch.cat([ps.unsqueeze(-1), ns], -1), tg, wts).sum(-1)
    loss, cp, cn, ga, gb = ops.ns_loss(dev(pos_out.detach()), dev(E.detach()), dev(tgt.view(n, 1)), dev(neg.view(n, 1, k)),
                                       anchor_b=dev(neg_out.detach()), bias=dev(pb.detach()), pos_weight=float(k))
    close(loss, ref)
    ref.mean().backward()
    close(ga / n, pos_out.grad, rtol=1e-4, atol=1e-7)
    close(gb / n, neg_out.grad, rtol=1e-4, atol=1e-7)


# ---------------------------------------------------------------- G2
def _dense_ref(table_rows, d, parts, drop):
    """fp64 scatter-add reference + the per-entry sum of |terms| (fp32 accumulation of n terms
    is only accurate to ~eps * sum|terms|, so tolerances scale with it)."""
    gt = torch.zeros(table_rows, d, dtype=torch.float64)
    ga = torch.zeros(table_rows, d, dtype=torch.float64)
    gb = torch.zeros(table_rows, dtype=torch.float64)
    for p in parts:
        idx = p["idx"].view(-1)
        n = idx.numel()
        row = p["src_row"] if p.get("src_row") is not None else torch.arange(n) // p.get("src_div", 1)
        s = p["scale"].double() if p.get("scale") is not None else torch.ones(n, dtype=torch.float64)
        if p.get("scale2") is not None:
            s = s * p["scale2"].double()[torch.arange(n) // p.get("scale2_div", 1)]
        keep = idx != drop
        terms = p["src"].double()[row[keep]] * s[keep].unsqueeze(1)
        gt.index_add_(0, idx[keep], terms)
        ga.index_add_(0, idx[keep], terms.abs())
        if p.get("to_bias"):
            gb.index_add_(0, idx[keep], s[keep])
    return gt, gb, ga


def close_sum(a, ref, abs_sum):
    """|a - ref| <= 1e-6 * sum|terms| + 1e-6: a few fp32 ulps of the accumulated magnitude."""
    a, ref = a.detach().cpu().double(), ref.double()
    assert bool(((a - ref).abs() <= 1e-6 * abs_sum + 1e-6).all()), float((a - ref).abs().max())


@pytest.mark.parametrize("n,rows,d", [(700, 300, 128), (16384, 18001, 128), (16385, 18001, 128),
                                      (250_000, 1_000_003, 128), (9000, 40, 64), (5000, 70000, 260),
                                      (120_000, 5, 128), (2_000_000, 16_000_001, 128)])
def test_scatter_reduce_vs_index_add(ops, n, rows, d):
    g = torch.Generator().manual_seed(n + rows)
    drop = rows - 1
    n2 = n // 3
    # Zipf-ish duplicates + explicit pad rows
    idx1 = (torch.rand(n - n2, generator=g) ** 3 * (rows - 1)).long()
    idx1[::17] = drop
    idx2 = torch.randint(0, rows - 1, (n2,), generator=g)
    src1 = torch.randn(n - n2, d, generator=g)
    anchors = torch.randn((n2 + 5) // 6, d, generator=g)
    scale = torch.randn(n2, generator=g)
    scale2 = torch.randn((n2 + 5) // 6, generator=g)
    parts = [dict(idx=idx1, src=src1),
             dict(idx=idx2, src=anchors, src_div=6, scale=scale, scale2=scale2, scale2_div=6, to_bias=True)]
    gt, gb, ga = _dense_ref(rows, d, parts, drop)
    contribs = [ops.make_contrib(dev(idx1), dev(src1)),
                ops.make_contrib(dev(idx2), dev(anchors), src_div=6, scale=dev(scale), scale2=dev(scale2),
                                 scale2_div=6, to_bias=True)]
    dense = torch.zeros(rows, d, device="cuda")
    dense_b = torch.zeros(rows, device="cuda")
    uniq, red, redb, nu = ops.scatter_reduce(contribs, rows, d, drop_idx=drop, dense_grad=dense,
                                             dense_bias_grad=dense_b, want_bias=True)
    nu = int(nu.item())
    expect_rows = torch.unique(torch.cat([idx1[idx1 != drop], idx2]))
    assert nu == expect_rows.numel()
    assert torch.equal(uniq[:nu].cpu().long(), expect_rows)          # ascending, bit-exact row ids
    close_sum(red[:nu], gt[expect_rows], ga[expect_rows])
    close(redb[:nu], gb[expect_rows], rtol=1e-5, atol=1e-4)
    close_sum(dense, gt, ga)
    close(dense_b, gb, rtol=1e-5, atol=1e-4)
    assert float(dense[drop].abs().sum()) == 0.0                    # padding_idx row stays zero
    # run-to-run bit reproducibility (no float atomics)
    uniq2, red2, redb2, nu2 = ops.scatter_reduce(contribs, rows, d, drop_idx=drop, want_bias=True)
    assert torch.equal(red[:nu], red2[:nu]) and torch.equal(redb[:nu], redb2[:nu])
    # clearing the touched rows restores an all-zero dense gradient in O(batch)
    ops.zero_rows(uniq, nu2, d, dense, dense_b)
    assert float(dense.abs().sum()) == 0.0 and float(dense_b.abs().sum()) == 0.0


@pytest.mark.parametrize("n,rows", [(10_000, 18_001), (7_000, 32_000), (16_384, 50), (3, 33_000)])
def test_count_sort_path_equals_radix_path_bitwise(ops, n, rows):
    """Small tables take the shared-memory counting sort (one bin per row), larger ones the radix sort: both must
    produce THE stable order, so the reduced rows agree bit for bit (declaring more rows than the indices use
    switches the same data to the radix path)."""
    g = torch.Generator().manual_seed(n * 31 + rows)
    idx = (torch.rand(n, generator=g) ** 4 * (rows - 1)).long()          # heavy head: runs of hundreds of slots
    idx[::13] = rows - 1                                                  # dropped
    src = torch.randn(n, 128, generator=g)
    scale = torch.randn(n, generator=g)
    c = [ops.make_contrib(dev(idx), dev(src), scale=dev(scale), to_bias=True)]
    u1, r1, b1, n1 = ops.scatter_reduce(c, rows, 128, drop_idx=rows - 1, want_bias=True)
    u2, r2, b2, n2 = ops.scatter_reduce(c, 1_000_000, 128, drop_idx=rows - 1, want_bias=True)
    k = int(n1.item())
    assert k == int(n2.item()) and torch.equal(u1[:k], u2[:k])
    assert torch.equal(r1[:k], r2[:k]) and torch.equal(b1[:k], b2[:k])


def test_scatter_reduce_all_dropped_and_single(ops):
    idx = torch.full((50,), 9, dtype=torch.int64)
    src = torch.randn(50, 128)
    uniq, red, _, nu = ops.scatter_reduce([ops.make_contrib(dev(idx), dev(src))], 10, 128, drop_idx=9)
    assert int(nu.item()) == 0
    idx[:] = 4
    uniq, red, _, nu = ops.scatter_reduce([ops.make_contrib(dev(idx), dev(src))], 10, 128, drop_idx=9)
    assert int(nu.item()) == 1 and int(uniq[0]) == 4
    assert torch.equal(red[0].cpu(), _bracketed_sum(src, 8))


def _bracketed_sum(src, unit, batch=16, long_units=64):
    """The kernels' fixed bracketing, term by term (so equality is bit-exact): sequential sums inside a unit of
    `unit` sorted slots (seg_reduce_kernel); unit partials combined by the fix-up kernel -- batches of 16 units as a
    binary tree, batches in unit order; a segment of more than 64 units is cut into 8 contiguous chunks (one per
    warp) whose sums are added in chunk order."""
    parts = []
    for u0 in range(0, src.shape[0], unit):
        part = torch.zeros(src.shape[1])
        for r in src[u0:u0 + unit]:
            part = part + r
        parts.append(part)
    if len(parts) == 1:
        return parts[0]

    def fold(ps):
        acc = torch.zeros(src.shape[1])
        for b0 in range(0, len(ps), batch):
            v = list(ps[b0:b0 + batch]) + [torch.zeros(src.shape[1])] * (batch - len(ps[b0:b0 + batch]))
            w = 1
            while w < batch:
                for t in range(0, batch - w, 2 * w):
                    v[t] = v[t] + v[t + w]
                w *= 2
            acc = acc + v[0]
        return acc
    if len(parts) <= long_units:
        return fold(parts)
    per = (len(parts) + 7) // 8
    total = None
    for w in range(8):
        chunk = fold(parts[w * per:(w + 1) * per])
        total = chunk if total is None else total + chunk
    return total


def test_scatter_reduce_long_segment_bracketing(ops):
    """A hot row spanning > 64 units goes through the CTA-cooperative fix-up; all paths are bit-reproducible."""
    g = torch.Generator().manual_seed(3)
    n = 8 * 150 + 5                                       # 151 units of 8 slots: the long path
    idx = torch.full((n,), 7, dtype=torch.int64)
    src = torch.randn(n, 128, generator=g)
    uniq, red, _, nu = ops.scatter_reduce([ops.make_contrib(dev(idx), dev(src))], 20, 128, drop_idx=19)
    assert int(nu.item()) == 1 and int(uniq[0]) == 7
    assert torch.equal(red[0].cpu(), _bracketed_sum(src, 8))
    assert torch.allclose(red[0].cpu(), src.double().sum(0).float(), rtol=1e-5, atol=1e-4)
    uniq2, red2, _, _ = ops.scatter_reduce([ops.make_contrib(dev(idx), dev(src))], 20, 128, drop_idx=19)
    assert torch.equal(red[0], red2[0])


# ---------------------------------------------------------------- G5 (exact mode) + merge
def _check_topk(ids, scores, Q, E, bias, k, n_items):
    S = Q.double() @ E[:n_items].double().t()
    if bias is not None:
        S = S + bias[:n_items].double()
    ids, scores = ids.cpu(), scores.cpu()
    scale = Q.norm(dim=1, keepdim=True).double() * E[:n_items].norm(dim=1).max().double()
    tol = 1e-5 * scale                                              # |score err| <= 1e-5 * |q||e|
    got = torch.gather(S, 1, ids)
    assert bool(((got - scores.double()).abs() <= tol).all())
    # ordering rule on the returned list: descending score, ties -> ascending id
    ds = scores[:, 1:] - scores[:, :-1]
    assert bool((ds <= 0).all())
    tie = ds == 0
    assert bool((ids[:, 1:][tie] > ids[:, :-1][tie]).all())
    # it is a top-k: nothing outside the list beats the k-th entry by more than the tolerance
    kth = scores[:, -1:].double()
    outside = S.clone()
    outside.scatter_(1, ids, float("-inf"))
    assert bool((outside.max(dim=1, keepdim=True).values <= kth + 2 * tol).all())
    for r in range(ids.shape[0]):
        assert len(set(ids[r].tolist())) == k


@pytest.mark.parametrize("m,n,d,k", [(24, 18000, 128, 100), (7, 1000, 64, 10), (130, 70001, 128, 100)])
def test_catalog_topk_exact(ops, m, n, d, k):
    g = torch.Generator().manual_seed(m + n)
    E = torch.randn(n + 1, d, generator=g)
    E[n] = 0
    Q = torch.randn(m, d, generator=g)
    bias = torch.randn(n + 1, generator=g) * 0.1
    ids, sc = ops.catalog_topk(dev(Q), dev(E), k, n_items=n, bias=dev(bias))
    _check_topk(ids, sc, Q, E, bias, k, n)
    ids2, sc2 = ops.catalog_topk(dev(Q), dev(E), k, n_items=n)
    _check_topk(ids2, sc2, Q, E, None, k, n)


def test_catalog_topk_ties_lower_id_first(ops):
    # small-integer data: fp32 dot products are exact, so ties are exact and the id rule decides
    g = torch.Generator().manual_seed(9)
    n, d, m, k = 5000, 128, 9, 100
    E = torch.randint(-2, 3, (n, d), generator=g).float()
    E[1000:1200] = E[17]                                            # 200 duplicates of one row
    Q = torch.randint(-2, 3, (m, d), generator=g).float()
    Q[0] = E[17]                                                    # makes the duplicates the top scores
    ids, sc = ops.catalog_topk(dev(Q), dev(E), k)
    S = (Q.double() @ E.double().t()).float().numpy()
    ref_i, ref_s = oracle.topk_lower_id_first(S, k)
    assert np.array_equal(ids.cpu().numpy(), ref_i)
    assert np.array_equal(sc.cpu().numpy(), ref_s)


def test_catalog_topk_short_catalog(ops):
    g = torch.Generator().manual_seed(10)
    E, Q = torch.randn(30, 128, generator=g), torch.randn(4, 128, generator=g)
    ids, sc = ops.catalog_topk(dev(Q), dev(E), 100)
    assert bool((ids[:, 30:] == -1).all()) and bool((ids[:, :30] >= 0).all())
    ref_i, _ = oracle.topk_lower_id_first((Q @ E.t()).numpy(), 30)
    assert np.array_equal(ids[:, :30].cpu().numpy(), ref_i)


def test_topk_merge_matches_global(ops):
    g = torch.Generator().manual_seed(12)
    G, n, d, m, k = 4, 4000, 128, 16, 100
    E = torch.randint(-2, 3, (n, d), generator=g).float()
    Q = torch.randint(-2, 3, (m, d), generator=g).float()
    parts_i, parts_s = [], []
    for r in range(G):                                              # cyclic row sharding: owner = id % G
        ids, sc = ops.catalog_topk(dev(Q), dev(E[r::G].contiguous()), k, id_base=r, id_stride=G)
        parts_i.append(ids)
        parts_s.append(sc)
    mi, ms = ops.topk_merge(torch.stack(parts_i), torch.stack(parts_s))
    gi, gs = ops.catalog_topk(dev(Q), dev(E), k)
    assert torch.equal(mi, gi) and torch.equal(ms, gs)
    ref_i, _ = oracle.merge_shard_topk([p.cpu().numpy() for p in parts_i], [p.cpu().numpy() for p in parts_s], k)
    assert np.array_equal(mi.cpu().numpy(), ref_i)


# ---------------------------------------------------------------- G5 tensor-core mode (tcgen05 + TMA)
@pytest.mark.parametrize("m,n,k,with_bias", [(24, 100_000, 100, False), (130, 70_001, 100, True),
                                             (384, 1_000_000, 100, False), (5, 40_000, 10, True)])
def test_catalog_topk_tc_equals_exact(ops, m, n, k, with_bias):
    """The TF32 shortlist + exact rescoring returns bit-identical (ids, scores) to the fp32 mode."""
    from prodsearch_b200 import _lib
    g = torch.Generator(device="cuda").manual_seed(m + n)
    E = torch.randn(n + 1, 128, generator=g, device="cuda")
    Q = torch.randn(m, 128, generator=g, device="cuda")
    bias = (torch.randn(n + 1, generator=g, device="cuda") * 0.1) if with_bias else None
    ids_e, sc_e = ops.catalog_topk(Q, E, k, n_items=n, bias=bias, mode=_lib.TOPK_EXACT)
    ids_t, sc_t = ops.catalog_topk(Q, E, k, n_items=n, bias=bias, mode=_lib.TOPK_TC)
    assert torch.equal(ids_e, ids_t)
    assert torch.equal(sc_e, sc_t)
    if n <= 100_000:
        _check_topk(ids_t, sc_t, Q.cpu(), E.cpu(), bias.cpu() if with_bias else None, k, n)


def test_catalog_topk_tc_degenerate_falls_back(ops):
    """Massive ties (every item identical) overflow the shortlist; the exact fallback still returns
    the lower-id-first answer."""
    from prodsearch_b200 import _lib
    n, m, k = 50_000, 3, 100
    E = torch.ones(n, 128, device="cuda")
    Q = torch.ones(m, 128, device="cuda")
    ids, sc = ops.catalog_topk(Q, E, k, mode=_lib.TOPK_TC)
    assert torch.equal(ids.cpu(), torch.arange(k).repeat(m, 1))
    assert bool((sc == 128.0).all())


def test_catalog_topk_tc_scaled_rows(ops):
    """Rows with very different norms (the eps bound uses the max row norm)."""
    from prodsearch_b200 import _lib
    g = torch.Generator(device="cuda").manual_seed(3)
    n, m, k = 200_000, 64, 100
    E = torch.randn(n, 128, generator=g, device="cuda") * torch.logspace(-2, 1, n, device="cuda").unsqueeze(1)
    Q = torch.randn(m, 128, generator=g, device="cuda")
    a = ops.catalog_topk(Q, E, k, mode=_lib.TOPK_EXACT)
    b = ops.catalog_topk(Q, E, k, mode=_lib.TOPK_TC)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ---------------------------------------------------------------- G5 fp16 shortlist (tcgen05 kind::f16, up to 512 queries / pass)
@pytest.mark.parametrize("m,n,k,with_bias", [(24, 100_000, 100, False), (130, 70_001, 100, True),
                                             (384, 1_000_000, 100, False), (5, 40_000, 10, True),
                                             (300, 250_000, 100, True), (513, 120_000, 50, False),
                                             (1100, 90_000, 100, False), (2100, 150_000, 100, True)])
def test_catalog_topk_f16_equals_exact(ops, m, n, k, with_bias):
    """fp16 shortlist (1..4 query tiles per CTA, 1..9 query groups; from 16 query tiles on, 2 tiles per CTA at 128 items
    per MMA) + exact fp32 rescoring == the fp32 mode, bit for bit, incl. ragged last item tile / last query tile and the
    bias path."""
    from prodsearch_b200 import _lib
    g = torch.Generator(device="cuda").manual_seed(m + n)
    E = torch.randn(n + 1, 128, generator=g, device="cuda")
    Q = torch.randn(m, 128, generator=g, device="cuda")
    bias = (torch.randn(n + 1, generator=g, device="cuda") * 0.1) if with_bias else None
    prep = ops.catalog_prepare_f16(E, n)
    assert prep.fits and torch.equal(prep.half, E[:n].half())
    assert abs(float(prep.stats[0]) - float((E[:n] ** 2).sum(1).max())) <= 1e-4 * float(prep.stats[0])
    ids_e, sc_e = ops.catalog_topk(Q, E, k, n_items=n, bias=bias, mode=_lib.TOPK_EXACT)
    ids_t, sc_t = ops.catalog_topk(Q, E, k, n_items=n, bias=bias, mode=_lib.TOPK_TC16, prepared=prep)
    assert torch.equal(ids_e, ids_t)
    assert torch.equal(sc_e, sc_t)


def test_catalog_topk_f16_scaled_rows_ties_and_overflow(ops):
    from prodsearch_b200 import _lib
    g = torch.Generator(device="cuda").manual_seed(3)
    n, m, k = 200_000, 64, 100
    E = torch.randn(n, 128, generator=g, device="cuda") * torch.logspace(-2, 1, n, device="cuda").unsqueeze(1)
    Q = torch.randn(m, 128, generator=g, device="cuda")
    a = ops.catalog_topk(Q, E, k, mode=_lib.TOPK_EXACT)
    b = ops.catalog_topk(Q, E, k, mode=_lib.TOPK_TC16, prepared=ops.catalog_prepare_f16(E))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # massive ties: the shortlist overflows, the exact fallback answers lower-id-first
    E1, Q1 = torch.ones(50_000, 128, device="cuda"), torch.ones(3, 128, device="cuda")
    ids, sc = ops.catalog_topk(Q1, E1, k, mode=_lib.TOPK_TC16, prepared=ops.catalog_prepare_f16(E1))
    assert torch.equal(ids.cpu(), torch.arange(k).repeat(3, 1)) and bool((sc == 128.0).all())
    # a value outside the fp16 range: flagged by the conversion pass, and the call still returns the exact answer
    E2 = E.clone()
    E2[12345, 7] = 1.0e6
    prep = ops.catalog_prepare_f16(E2)
    assert not prep.fits
    a = ops.catalog_topk(Q[:4], E2, k, mode=_lib.TOPK_EXACT)
    b = ops.catalog_topk(Q[:4], E2, k, mode=_lib.TOPK_TC16, prepared=prep)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
