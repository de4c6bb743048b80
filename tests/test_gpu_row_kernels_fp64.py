"""GPU: float64 references for every launch path of the row kernels (csrc/gather.cu, csrc/ns_loss.cu) and for the
catalog's tensor-core top-k modes at every width they accept.

Cases are built from the dispatch conditions of each entry point, and each case id names the template instance it
reaches.  Where the profiler label tells the instances apart, the case asserts that the expected kernel ran, so a
later change of dispatch cannot quietly move a case onto another path.

Every reference restates the contract of include/psb.h in float64 (or runs the oracle's bce_with_logits in float64);
gradients of the loss kernels come from float64 autograd.  Out-of-range row ids read as a zero row with no bias,
which is what every kernel does.

Error bounds.  Each output element e gets a first-order error magnitude M(e): the float64 sum of the absolute
values of every term rounded on its way to e.  For a dot product that is sum |a_c r_c| + |bias|.  Transcendentals
add their own magnitude, and input errors carry through the derivative.  For example, the loss adds
|sigmoid(x) - t| * M(x) + |x| + 1 + bce(x) per score, and a coefficient adds sigmoid'(x) M(x) + sigmoid(x) +
|sigmoid(x) - t|.  The bound is K * 2^-24 * M(e), and K is stated per group.  K is the number of rounding steps
in the kernel's longest chain when that chain is short.  Sums that are long or tree-shaped take K well below their
worst case: the inputs are zero-mean, so the rounding errors of one chain add in quadrature.  The module prints the
worst err / bound of every group when the file has run (pytest -s).  K is set so that this worst is well above 1/30:
a dropped term, a wrong index or a missing scale moves an element by a whole term, far past K ulps of M.

The mean-pool is checked bit for bit instead.  The kernel adds each scaled row, rounded, in token order without FMA
(gather.cu, meanpool_kernel), then divides with IEEE division and applies keep_scale.  A CPU float32 replay of that
order reproduces it exactly.
"""
import math

import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                      # unit roundoff of float32
RATIOS = {}                         # group -> worst err / bound seen in this run


@pytest.fixture(scope="module")
def ops():
    from prodsearch_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    if RATIOS:
        print("\nworst err / bound per group:")
        for g in sorted(RATIOS):
            print("  %-34s %.3g" % (g, RATIOS[g]))


class _Kernels(object):
    """Names of the library kernels launched inside the block (the library's own event profiler, switched off
    again on exit)."""

    def __enter__(self):
        from prodsearch_b200 import _lib
        self._lib = _lib
        _lib.profile_enable(True)
        self.names = set()
        return self

    def __exit__(self, *exc):
        try:
            self.names = set(self._lib.profile_dump())
        finally:
            self._lib.profile_enable(False)
        return False


def _check(group, got, ref, mag, K):
    """|got - ref| <= K * u * mag elementwise (mag == 0: exact)."""
    got = torch.as_tensor(got).detach().cpu().double().reshape(-1)
    ref = torch.as_tensor(ref).detach().cpu().double().reshape(-1)
    mag = torch.as_tensor(mag).detach().cpu().double().reshape(-1)
    assert got.shape == ref.shape == mag.shape
    if got.numel() == 0:
        return
    assert bool(torch.isfinite(got).all()), "%s: non-finite output" % group
    err = (got - ref).abs()
    bound = K * U * mag
    ratio = torch.where(bound > 0, err / torch.where(bound > 0, bound, torch.ones_like(bound)),
                        torch.where(err > 0, torch.full_like(err, float("inf")), torch.zeros_like(err)))
    j = int(ratio.argmax())
    worst = float(ratio[j])
    RATIOS[group] = max(RATIOS.get(group, 0.0), worst)
    assert worst <= 1.0, "%s: err / bound %.3g at flat %d (got %r, ref %r, bound %r)" % (
        group, worst, j, float(got[j]), float(ref[j]), float(bound[j]))


def _d_rows(table, ids):
    """float64 rows table[ids] with out-of-range ids read as zeros; also the in-range mask."""
    V = table.shape[0]
    ok = (ids >= 0) & (ids < V)
    rows = table.double()[torch.where(ok, ids, torch.zeros_like(ids))] * ok.unsqueeze(-1).double()
    return rows, ok


def _scatter_oor(g, ids, V, every):
    """Put ids >= V and < 0 at a spread of positions (never the pad id)."""
    flat = ids.view(-1)
    if flat.numel() == 0:
        return
    sel = torch.randperm(flat.numel(), generator=g)[:max(1, flat.numel() // every)]
    flat[sel[0::2]] = V + 3
    flat[sel[1::2]] = -2


# ------------------------------------------------------------------------------------------------ ns_loss
def _bce_mags(x, Sx, t, wt, m, cnt, gscale):
    """First-order error magnitudes of the loss rows and of the coefficients d loss / d x (see the module doc)."""
    sig = torch.sigmoid(x)
    bce = oracle.bce_with_logits(x, t)
    aw = wt.abs()
    per = aw * ((sig - t).abs() * Sx + 1.0 + x.abs() + bce)
    m_loss = (per.sum(-1) * m).sum(-1) / cnt
    m_coef = abs(gscale) * m.unsqueeze(-1) * aw / cnt.view(-1, *([1] * (x.dim() - 1))) * (
        sig * (1 - sig) * Sx + sig + (sig - t).abs())
    return m_loss, m_coef


def _ns_ref(anchor_a, anchor_b, table, bias, pos, neg, mask, pad_idx, neg_weight, pos_weight):
    """psb_ns_loss_fwd's contract in float64: (loss, coef [n,w,1+k], grad_a, grad_b) and their error magnitudes."""
    n, w = pos.shape
    k = neg.shape[-1]
    d = table.shape[1]
    ids = torch.cat([pos.unsqueeze(-1), neg], -1)                         # [n, w, 1 + k]
    R, ok = _d_rows(table, ids)
    b = bias.double()[torch.where(ok, ids, torch.zeros_like(ids))] * ok.double() if bias is not None \
        else torch.zeros(ids.shape, dtype=torch.float64)
    A = anchor_a.double().requires_grad_(True)
    B = anchor_b.double().requires_grad_(True) if anchor_b is not None else None
    if B is not None:
        anc = torch.cat([A.view(n, 1, 1, d), B.view(n, 1, k, d)], 2)       # w == 1
    else:
        anc = A.view(n, 1, 1, d).expand(n, w, 1 + k, d)
    x = (anc * R).sum(-1) + b
    x.retain_grad()
    Sx = (anc.detach() * R).abs().sum(-1) + b.abs()
    t = torch.zeros_like(x.detach())
    t[..., 0] = 1.0
    wt = torch.ones(n, w, 1 + k, dtype=torch.float64)
    wt[..., 0] = pos_weight
    if neg_weight is not None:
        wt[..., 1:] = neg_weight.double().view(n, 1, k)
    if mask is not None:
        m = mask.ne(0).double()
    elif pad_idx >= 0:
        m = pos.ne(pad_idx).double()
    else:
        m = torch.ones(n, w, dtype=torch.float64)
    cnt = m.sum(-1).clamp(min=1)
    loss = (oracle.bce_with_logits(x, t, wt).sum(-1) * m).sum(-1) / cnt
    loss.sum().backward()
    coef = x.grad
    m_loss, m_coef = _bce_mags(x.detach(), Sx, t, wt, m, cnt, 1.0)
    Ra = R.abs()
    mg_row = (m_coef + coef.abs()).unsqueeze(-1) * Ra                    # [n, w, 1 + k, d]
    if B is not None:
        m_ga = mg_row[:, :, 0].sum(1)
        m_gb = mg_row[:, 0, 1:].reshape(n * k, d)
    else:
        m_ga = mg_row.sum((1, 2))
        m_gb = None
    return dict(loss=loss.detach(), coef=coef, ga=A.grad, gb=B.grad if B is not None else None,
                m_loss=m_loss, m_coef=m_coef, m_ga=m_ga, m_gb=m_gb)


def _ns_inputs(seed, n, w, k, d, V, use_mask, use_bias, use_nw, pos_weight, with_b):
    g = torch.Generator().manual_seed(seed)
    sa = 2.0 / math.sqrt(d)                                  # scores of spread ~2: both sides of the sigmoid
    table = torch.randn(V, d, generator=g)
    anchor_a = torch.randn(n, d, generator=g) * sa
    anchor_b = torch.randn(n * k, d, generator=g) * sa if with_b else None
    bias = torch.randn(V, generator=g) * 0.5 if use_bias else None
    pos = torch.randint(0, V - 1, (n, w), generator=g)
    neg = torch.randint(0, V - 1, (n, w, k), generator=g)
    _scatter_oor(g, pos, V, 9)
    _scatter_oor(g, neg, V, 7)
    pad = V - 1
    pos[1, :] = pad                                          # a fully padded row
    if w > 1:
        pos[2, w // 2] = pad
    if use_mask:                                             # the mask decides; pad ids are then ordinary rows
        mask = (torch.rand(n, w, generator=g) > 0.25).to(torch.uint8)
        mask[1] = 0
        mask[3] = 0                                          # fully masked, with real ids
    else:
        mask = None
    nw = torch.rand(n, k, generator=g) * 1.75 + 0.25 if use_nw else None
    return dict(anchor_a=anchor_a, anchor_b=anchor_b, table=table, bias=bias, pos=pos, neg=neg, mask=mask,
                pad_idx=pad, neg_weight=nw, pos_weight=pos_weight)


def _dev(t):
    return t.cuda() if t is not None else None


# K per group (module doc).  Dot products: 4 fused steps per lane and float4 column, then the 5-level warp tree;
# loss: the bce evaluation and the 1 + k (and w) term sums; coefficients: expf, one division, one subtraction and
# the division by the count; anchor gradients: a sequential FMA chain over the scores of the anchor.
K_NS = dict(loss=4.0, coef=6.0, ga=6.0, gb=4.0)


def _ns_loss_at_rows(inp, table_rows):
    """psb_ns_loss_fwd with table_rows passed in place of the table's row count."""
    from prodsearch_b200 import _lib
    a, b, table, bias, pos, neg, mask, nw = (_dev(inp[x]) for x in ("anchor_a", "anchor_b", "table", "bias", "pos", "neg",
                                                                    "mask", "neg_weight"))
    n, w = pos.shape
    k, d = neg.shape[-1], table.shape[1]
    f = dict(dtype=torch.float32, device="cuda")
    loss, cp, cn, ga = torch.empty(n, **f), torch.empty(n, w, **f), torch.empty(n, w, k, **f), torch.empty(n, d, **f)
    gb = torch.empty(n * k, d, **f) if b is not None else None
    P = _lib.ptr
    _lib.check(_lib.load().psb_ns_loss_fwd(P(a), P(b), P(table), table_rows, d, P(bias), P(pos), P(neg), P(mask),
                                           inp["pad_idx"], P(nw), inp["pos_weight"], n, w, k, P(loss), P(cp), P(cn),
                                           P(ga), P(gb), _lib.stream_ptr()), "psb_ns_loss_fwd")
    return loss, cp, cn, ga, gb


def _run_ns(ops, group, label, case, n, w, k, d, V=1000, table_rows=None):
    """table_rows: passed to the library in place of V.  Ids >= V then become table_rows + 3, so every id is either a
    real row or out of range for the kernel as well: the kernel reads only rows whose id is in [0, table_rows)."""
    use_mask, use_bias, use_nw, pw, with_b = case
    inp = _ns_inputs(n * 131 + w * 17 + k * 5 + d, n, w, k, d, V, use_mask, use_bias, use_nw, pw, with_b)
    if table_rows is not None:
        for t in (inp["pos"], inp["neg"]):
            t[t >= V] = table_rows + 3
    ref = _ns_ref(**inp)
    with _Kernels() as kern:
        if table_rows is not None:
            loss, cp, cn, ga, gb = _ns_loss_at_rows(inp, table_rows)
        else:
            loss, cp, cn, ga, gb = ops.ns_loss(_dev(inp["anchor_a"]), _dev(inp["table"]), _dev(inp["pos"]),
                                               _dev(inp["neg"]), anchor_b=_dev(inp["anchor_b"]), bias=_dev(inp["bias"]),
                                               mask=_dev(inp["mask"]), pad_idx=inp["pad_idx"],
                                               neg_weight=_dev(inp["neg_weight"]), pos_weight=pw)
    assert label in kern.names, (label, kern.names)
    _check(group + "/loss", loss, ref["loss"], ref["m_loss"], K_NS["loss"])
    _check(group + "/coef_pos", cp, ref["coef"][..., 0], ref["m_coef"][..., 0], K_NS["coef"])
    _check(group + "/coef_neg", cn, ref["coef"][..., 1:], ref["m_coef"][..., 1:], K_NS["coef"])
    _check(group + "/grad_a", ga, ref["ga"], ref["m_ga"], K_NS["ga"])
    if with_b:
        _check(group + "/grad_b", gb, ref["gb"], ref["m_gb"], K_NS["gb"])


def _features(i, w=1, k=1):
    """Input options crossed over the cases: (mask or pad_idx, bias, neg_weight, pos_weight)."""
    use_mask = i % 2 == 0
    use_bias = i % 3 != 2
    use_nw = k > 0 and (i % 2 == 1 or w > 1 or i % 5 == 0)
    pw = 1.0 if i % 4 < 2 else 2.5
    return use_mask, use_bias, use_nw, pw


def _fid(f):
    return "%s%s%s%s" % ("mask" if f[0] else "pad", "_bias" if f[1] else "", "_nw" if f[2] else "",
                         "_pw" if f[3] != 1.0 else "")


def _w1_cases():
    out, i = [], 0
    for with_b in (False, True):
        for k in (0, 1, 5, 6, 7):
            for d in (4, 64, 124, 128):
                f = _features(i, 1, k)
                nr = 6 if k <= 5 else 8
                out.append(pytest.param(f + (with_b,), k, d, 67,
                                        id="w1_kernel<%s,NR%d>-k%d-d%d-%s" % ("B" if with_b and k else "noB", nr, k, d,
                                                                               _fid(f))))
                i += 1
    # more anchors than resident warps: every warp takes a second anchor through the prefetching loop
    out.append(pytest.param((False, True, True, 1.0, False), 7, 64, 40000, id="w1_kernel<noB,NR8>-k7-d64-n40000-grid_stride"))
    out.append(pytest.param((True, False, False, 2.5, True), 5, 32, 40000, id="w1_kernel<B,NR6>-k5-d32-n40000-grid_stride"))
    return out


@pytest.mark.parametrize("case,k,d,n", _w1_cases())
def test_ns_loss_w1_kernel(ops, case, k, d, n):
    _run_ns(ops, "ns_w1", "ns_loss_w1_kernel", case, n, 1, k, d)


def _fast_cases():
    out, i = [], 1
    for w in (2, 33):
        for k in (3, 7):
            for d in (60, 128):
                f = _features(i, w, k)
                out.append(pytest.param(f + (False,), w, k, d, 45, id="fast_kernel<noB>-w%d-k%d-d%d-%s" % (w, k, d, _fid(f))))
                i += 1
    out.append(pytest.param((True, True, True, 1.0, False), 2, 3, 32, 38000, id="fast_kernel<noB>-w2-k3-d32-n38000-grid_stride"))
    return out


@pytest.mark.parametrize("case,w,k,d,n", _fast_cases())
def test_ns_loss_fast_kernel(ops, case, w, k, d, n):
    _run_ns(ops, "ns_fast", "ns_loss_fast_kernel", case, n, w, k, d)


def _fast_w1_cases():
    out, i = [], 3
    for with_b in (False, True):
        for k in (1, 5, 7):
            for d in (64, 128):
                f = _features(i, 1, k)
                out.append(pytest.param(f + (with_b,), k, d, id="fast_kernel<%s>-w1-k%d-d%d-rows2^31-%s" % (
                    "B" if with_b else "noB", k, d, _fid(f))))
                i += 1
    return out


@pytest.mark.parametrize("case,k,d", _fast_w1_cases())
def test_ns_loss_fast_kernel_w1_large_table(ops, case, k, d):
    """w == 1 on a table of 2^31 rows or more: ns_loss_w1_kernel carries row ids as int32, so the fast kernel takes
    these calls (the only way to reach ns_loss_fast_kernel<true>).  The small real table stands in for the large one."""
    _run_ns(ops, "ns_fast_w1", "ns_loss_fast_kernel", case, 67, 1, k, d, table_rows=2 ** 31)


def _generic_cases():
    out, i = [], 2
    for d, c in ((128, 1), (256, 2), (260, 4), (512, 4)):
        for k in (8, 16):
            for w in (1, 3):
                f = _features(i, w, k)
                with_b = w == 1 and i % 2 == 0
                out.append(pytest.param(f + (with_b,), w, k, d, 37,
                                        id="ns_loss_kernel<%d>-w%d-k%d-d%d-%s%s" % (c, w, k, d, _fid(f), "-anchor_b" if with_b else "")))
                i += 1
    # d > 128 with k <= 7 also takes the generic kernel, and k = 0 there
    out.append(pytest.param((True, True, False, 2.5, False), 1, 0, 132, 37, id="ns_loss_kernel<2>-w1-k0-d132-mask_bias_pw"))
    out.append(pytest.param((False, True, True, 1.0, False), 2, 5, 508, 37, id="ns_loss_kernel<4>-w2-k5-d508-pad_bias_nw"))
    out.append(pytest.param((False, False, True, 1.0, True), 1, 4, 200, 37, id="ns_loss_kernel<2>-w1-k4-d200-pad_nw-anchor_b"))
    out.append(pytest.param((True, True, True, 1.0, False), 1, 8, 132, 19000, id="ns_loss_kernel<2>-w1-k8-d132-n19000-grid_stride"))
    return out


@pytest.mark.parametrize("case,w,k,d,n", _generic_cases())
def test_ns_loss_generic_kernel(ops, case, w, k, d, n):
    _run_ns(ops, "ns_generic", "ns_loss_kernel", case, n, w, k, d)


# ------------------------------------------------------------------------------------------------ tem_loss
def _tem_ref(enc, table, bias, tgt, neg, pos_weight, grad_scale):
    """The TEM tail of test_gpu_ops.test_score_loss_tail_vs_oracle in float64, with grad_scale on the gradient."""
    n, c, d = enc.shape
    k = c - 1
    E = table.double()
    X = enc.double().requires_grad_(True)
    pos_out, neg_out = X[:, 0], X[:, 1:]
    pb = bias.double() if bias is not None else torch.zeros(table.shape[0], dtype=torch.float64)
    ps = (pos_out * E[tgt]).sum(-1) + pb[tgt]
    ns = (neg_out * E[neg]).sum(-1) + pb[neg]
    x = torch.cat([ps.unsqueeze(-1), ns], -1)
    x.retain_grad()
    wts = torch.ones(n, 1 + k, dtype=torch.float64)
    wts[:, 0] = pos_weight
    tg = torch.cat([torch.ones(n, 1), torch.zeros(n, k)], -1).double()
    rows = oracle.bce_with_logits(x, tg, wts).sum(-1)
    (grad_scale * rows.sum()).backward()
    ids = torch.cat([tgt.unsqueeze(-1), neg], -1)
    R = E[ids]                                                         # [n, 1 + k, d]
    Sx = (X.detach() * R).abs().sum(-1) + pb[ids].abs()
    m_rows, m_coef = _bce_mags(x.detach().unsqueeze(1), Sx.unsqueeze(1), tg.unsqueeze(1), wts.unsqueeze(1),
                               torch.ones(n, 1, dtype=torch.float64), torch.ones(n, dtype=torch.float64), grad_scale)
    m_coef = m_coef.squeeze(1)
    m_g = (m_coef + x.grad.abs()).unsqueeze(-1) * R.abs()
    return rows.detach(), x.grad, X.grad, m_rows, m_coef, m_g


K_TEM = dict(loss=4.0, coef=6.0, grad=4.0)


@pytest.mark.parametrize("with_bias,pos_weight,grad_scale", [(False, 1.0, 1.0), (True, 5.0, 1.0 / 77)],
                         ids=["nobias", "bias_pw5_scale"])
@pytest.mark.parametrize("d", [32, 128])
@pytest.mark.parametrize("k", [1, 5, 6, 7])
def test_tem_loss_vs_fp64_tail(ops, k, d, with_bias, pos_weight, grad_scale):
    """ns_loss_w1_kernel<true, 6> for k <= 5, <true, 8> for k = 6, 7, on the [n, 1 + k, d] block."""
    g = torch.Generator().manual_seed(k * 100 + d + int(with_bias))
    P, n = 3000, 77
    table = torch.randn(P, d, generator=g)
    bias = torch.randn(P, generator=g) * 0.5 if with_bias else None
    enc = torch.randn(n, 1 + k, d, generator=g) * (2.0 / math.sqrt(d))
    tgt = torch.randint(0, P, (n,), generator=g)
    neg = torch.randint(0, P, (n, k), generator=g)
    rows_r, coef_r, genc_r, m_rows, m_coef, m_g = _tem_ref(enc, table, bias, tgt, neg, pos_weight, grad_scale)
    with _Kernels() as kern:
        rows, cp, cn, genc = ops.tem_loss(enc.cuda(), table.cuda(), tgt.cuda(), neg.cuda(), bias=_dev(bias),
                                          pos_weight=pos_weight, grad_scale=grad_scale)
    assert "ns_loss_w1_kernel" in kern.names, kern.names
    _check("tem/loss_rows", rows, rows_r, m_rows, K_TEM["loss"])
    _check("tem/coef_pos", cp, coef_r[:, 0], m_coef[:, 0], K_TEM["coef"])
    _check("tem/coef_neg", cn, coef_r[:, 1:], m_coef[:, 1:], K_TEM["coef"])
    _check("tem/grad_enc_out", genc, genc_r, m_g, K_TEM["grad"])


# one thread sums n / 256 strided terms, then the 5-level warp tree, then 8 warp sums, one division; the running
# sums add one more rounding to a magnitude that already includes the accumulator
K_FINISH = 6.0
K_ACC = 2.0


@pytest.mark.parametrize("n_ps,n_il", [(257, 0), (1000, 300), (4097, 777), (70001, 513)])
def test_tem_loss_finish_vs_fp64_means(ops, n_ps, n_il):
    g = torch.Generator().manual_seed(n_ps + n_il)
    ps = torch.rand(n_ps, generator=g) * 3.0
    il = torch.randn(n_il, generator=g) + 0.5
    acc_ps = torch.full((1,), 2.0, device="cuda")
    acc_il = torch.full((1,), -1.0, device="cuda")
    with _Kernels() as kern:
        out = ops.tem_loss_finish(ps.cuda(), il.cuda() if n_il else None, acc_ps, acc_il)
    assert "tem_loss_finish_kernel" in kern.names
    mps = ps.double().mean()
    mil = il.double().mean() if n_il else torch.zeros((), dtype=torch.float64)
    aps = ps.double().abs().mean()
    ail = il.double().abs().mean() if n_il else torch.zeros((), dtype=torch.float64)
    _check("tem_finish/loss", out, mps + mil, aps + ail, K_FINISH)
    _check("tem_finish/acc_ps", acc_ps, 2.0 + mps, 2.0 + aps, K_ACC)
    _check("tem_finish/acc_il", acc_il, -1.0 + mil, 1.0 + ail, K_ACC)


# ------------------------------------------------------------------------------------------------ score_rows
# per lane 4 C fused steps, then the 5-level warp tree and the bias
K_SCORE = 6.0


@pytest.mark.parametrize("with_bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("c_per", [1, 3, 4, 5, 31, 32, 33, 100, 1001])
@pytest.mark.parametrize("d,C", [(4, 1), (128, 1), (132, 2), (256, 2), (512, 4)],
                         ids=["d4-score_rows_kernel<1>", "d128-score_rows_kernel<1>", "d132-score_rows_kernel<2>",
                              "d256-score_rows_kernel<2>", "d512-score_rows_kernel<4>"])
def test_score_rows_vs_fp64(ops, d, C, c_per, with_bias):
    g = torch.Generator().manual_seed(d * 7 + c_per * 3 + int(with_bias))
    V = 2500
    n = 40 if c_per < 100 else 9
    table = torch.randn(V, d, generator=g)
    bias = torch.randn(V, generator=g) * 0.5 if with_bias else None
    anchor = torch.randn(n, d, generator=g) / math.sqrt(d)
    idx = torch.randint(0, V, (n, c_per), generator=g)
    _scatter_oor(g, idx, V, 6)
    idx[0, -1] = V                                          # the last candidate of a group past the first 32
    R, ok = _d_rows(table, idx)
    b = bias.double()[torch.where(ok, idx, torch.zeros_like(idx))] * ok.double() if with_bias \
        else torch.zeros(idx.shape, dtype=torch.float64)
    prod = anchor.double().unsqueeze(1) * R
    ref = prod.sum(-1) + b
    mag = prod.abs().sum(-1) + b.abs()
    with _Kernels() as kern:
        sc = ops.score_rows(anchor.cuda(), table.cuda(), idx.cuda(), bias=_dev(bias))
    assert "score_rows_kernel" in kern.names
    assert bool((sc.cpu()[~ok] == 0).all())                 # invalid candidate: score 0, no bias
    _check("score_rows", sc, ref, mag, K_SCORE)


# ------------------------------------------------------------------------------------------------ mean-pool / fs
def _pool_inputs(seed, n, w, d, V, use_mask, use_tok, use_keep):
    g = torch.Generator().manual_seed(seed)
    table = torch.randn(V, d, generator=g)
    idx = torch.randint(0, V - 1, (n, w), generator=g)
    _scatter_oor(g, idx, V, 11)
    pad = V - 1
    idx[0, :] = pad                                          # fully padded
    idx[2, w // 2:] = pad
    mask = None
    if use_mask:
        mask = (torch.rand(n, w, generator=g) > 0.3).to(torch.uint8)
        mask[4] = 0
    tok = torch.where(torch.rand(n, w, generator=g) < 0.3, torch.zeros(()), torch.full((), 1 / 0.7)) if use_tok else None
    keep = torch.where(torch.rand(n, d, generator=g) < 0.1, torch.zeros(()), torch.full((), 1 / 0.9)) if use_keep else None
    return table, idx, pad, mask, tok, keep


def _valid(idx, pad, mask):
    return mask.ne(0) if mask is not None else idx.ne(pad)


def _replay_mean(table, idx, pad, mask, tok, keep):
    """meanpool_kernel's float32 arithmetic on the CPU: (row * scale) rounded, added in token order, IEEE division
    by max(#valid, 1), then the keep_scale multiply."""
    n, w = idx.shape
    V, d = table.shape
    valid = _valid(idx, pad, mask)
    acc = torch.zeros(n, d, dtype=torch.float32)
    for j in range(w):
        r = idx[:, j]
        ok = (r >= 0) & (r < V)
        sc = torch.where(valid[:, j] & ok, tok[:, j] if tok is not None else torch.ones(n), torch.zeros(n))
        term = table[torch.where(ok, r, torch.zeros_like(r))] * sc.unsqueeze(1)
        acc = acc + torch.where((sc != 0).unsqueeze(1), term, torch.zeros(()))
    mean = acc / valid.sum(-1).clamp(min=1).float().unsqueeze(1)
    return mean * keep if keep is not None else mean


def _mean64(table, idx, pad, mask, tok, keep):
    """The contract in float64, and the magnitude of the float32 accumulation that approximates it."""
    n, w = idx.shape
    valid = _valid(idx, pad, mask)
    cnt = valid.sum(-1).clamp(min=1).double().unsqueeze(1)
    acc = torch.zeros(n, table.shape[1], dtype=torch.float64)
    mag = torch.zeros_like(acc)
    for j in range(w):
        rows, _ = _d_rows(table, idx[:, j])
        s = valid[:, j].double() * (tok[:, j].double() if tok is not None else 1.0)
        acc += rows * s.unsqueeze(1)
        mag += (rows * s.unsqueeze(1)).abs()
    ks = keep.double().abs() if keep is not None else 1.0
    mean = acc / cnt * (keep.double() if keep is not None else 1.0)
    return mean, mag / cnt * ks + mean.abs()


@pytest.mark.parametrize("w", [1, 31, 32, 33, 100])
@pytest.mark.parametrize("d,C", [(4, 1), (64, 1), (128, 1), (132, 2), (256, 2), (260, 4), (512, 4)],
                         ids=["d4-meanpool_kernel<1,false>", "d64-meanpool_kernel<1,false>",
                              "d128-meanpool_kernel<1,false>", "d132-meanpool_kernel<2,false>",
                              "d256-meanpool_kernel<2,false>", "d260-meanpool_kernel<4,false>",
                              "d512-meanpool_kernel<4,false>"])
def test_meanpool_bit_exact_replay(ops, d, C, w):
    i = d + w
    use_mask, use_tok, use_keep = i % 2 == 0, i % 3 != 0, i % 5 != 1
    n = 300
    table, idx, pad, mask, tok, keep = _pool_inputs(i, n, w, d, 701, use_mask, use_tok, use_keep)
    with _Kernels() as kern:
        out, mean, inv = ops.gather_meanpool(table.cuda(), idx.cuda(), pad_idx=pad, mask=_dev(mask), tok_scale=_dev(tok),
                                             keep_scale=_dev(keep), want_mean=True, want_inv_count=True)
    assert "meanpool_kernel" in kern.names
    ref = _replay_mean(table, idx, pad, mask, tok, keep)
    assert torch.equal(out.cpu(), ref), float((out.cpu() - ref).abs().max())
    assert torch.equal(mean.cpu(), ref)
    valid = _valid(idx, pad, mask)
    cnt = valid.sum(-1).clamp(min=1).float()
    assert torch.equal(inv.cpu(), 1.0 / cnt)
    # the same ids through gather_rows_kernel<8> (zero rows for out-of-range ids) and token_weights_kernel
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    with _Kernels() as kern:
        rows = ops.gather_rows(table.cuda(), idx.cuda(), err_flag=flag)
        tw = ops.token_weights(idx.cuda(), pad_idx=pad, mask=_dev(mask))
    assert "gather_rows_kernel" in kern.names and "token_weights_kernel" in kern.names
    assert torch.equal(rows.cpu(), _d_rows(table, idx)[0].float()) and int(flag) == 1
    assert torch.equal(tw.cpu(), torch.where(valid, (1.0 / cnt).unsqueeze(1), torch.zeros(())))


# fs forward: the pooled row's own rounding (token-order sum) carried through W, the matvec (per-lane FMA chains and
# the warp tree, or the shared-memory FMA chain over d), tanh.  fs_bwd: the 8-warp split over n (grad_weight,
# grad_bias) plus the dz products; grad_mean is one sequential FMA chain of d terms per element, so its K grows as
# sqrt(d) (K_FS_GM * sqrt(d)): a d-term chain of zero-mean terms.
K_FS = dict(out=8.0, gW=8.0, gb=8.0)
K_FS_GM = 1.0


def _fs_cases():
    out = []
    for d, kind in ((64, "meanpool_kernel<1,true,true>"), (128, "meanpool_kernel<1,true,true>"),
                    (132, "meanpool_kernel<2,true>"), (256, "meanpool_kernel<2,true>"), (512, "meanpool_kernel<4,true>")):
        bwd = "fs_bwd_kernel<%d>" % (1 if d <= 128 else 2 if d <= 256 else 4)
        for w in (1, 31, 32, 33, 100):
            n = 4097 if (d + w) % 2 == 0 else 1000
            out.append(pytest.param(d, w, n, id="%s+%s-d%d-w%d-n%d" % (kind, bwd, d, w, n)))
    return out


@pytest.mark.parametrize("d,w,n", _fs_cases())
def test_fs_forward_and_backward_vs_fp64(ops, d, w, n):
    i = d + w
    use_mask, use_tok = i % 2 == 1, i % 3 != 0
    table, idx, pad, mask, tok, keep = _pool_inputs(i * 3 + n, n, w, d, 901, use_mask, use_tok, True)
    g = torch.Generator().manual_seed(i)
    W = torch.randn(d, d, generator=g) * (1.5 / math.sqrt(d))
    b = torch.randn(d, generator=g) * 0.1
    go = torch.randn(n, d, generator=g)
    with _Kernels() as kern:
        out, mean, _ = ops.gather_meanpool(table.cuda(), idx.cuda(), pad_idx=pad, mask=_dev(mask), tok_scale=_dev(tok),
                                           keep_scale=keep.cuda(), fs_weight=W.cuda(), fs_bias=b.cuda())
        gW, gb, gm = ops.fs_bwd(go.cuda(), out, mean, keep.cuda(), W.cuda())
    assert "meanpool_kernel" in kern.names and "fs_bwd_kernel" in kern.names
    assert torch.equal(mean.cpu(), _replay_mean(table, idx, pad, mask, tok, keep))
    # forward: tanh(W mean + b) with the float64 mean of the contract
    m64, m_mag = _mean64(table, idx, pad, mask, tok, keep)
    W64 = W.double()
    o64 = torch.tanh(m64 @ W64.t() + b.double())
    z_mag = m64.abs() @ W64.abs().t() + m_mag @ W64.abs().t() + b.double().abs()
    _check("fs_fwd/out", out, o64, (1 - o64 * o64) * z_mag + o64.abs(), K_FS["out"])
    # backward: the contract on the kernel's own out and mean (its inputs), in float64
    o, mn, go64 = out.cpu().double(), mean.cpu().double(), go.double()
    dz = go64 * (1 - o * o)
    dz_mag = go64.abs()                                           # |dz| + the rounding of 1 - o*o
    _check("fs_bwd/grad_W", gW, dz.t() @ mn, dz_mag.t() @ mn.abs(), K_FS["gW"])
    _check("fs_bwd/grad_b", gb, dz.sum(0), dz_mag.sum(0), K_FS["gb"])
    _check("fs_bwd/grad_mean", gm, keep.double() * (dz @ W64), keep.double().abs() * (dz_mag @ W64.abs()),
           K_FS_GM * math.sqrt(d))


# ------------------------------------------------------------------------------------------------ catalog top-k
def _topk_pair(ops, Q, E, k, n, bias, mode, id_base=0, id_stride=1):
    from prodsearch_b200 import _lib
    prep = ops.catalog_prepare_f16(E, n) if mode == _lib.TOPK_TC16 else None
    return ops.catalog_topk(Q, E, k, n_items=n, bias=bias, mode=mode, id_base=id_base, id_stride=id_stride,
                            prepared=prep)


_TC_LABEL = {1: "tc_score_kernel", 2: "tc16_score_v3_kernel"}


def _tc_cases():
    out = []
    for mode, d in ((1, 32), (1, 64), (1, 96), (2, 64)):
        for k in (1, 128):
            for n in (32767, 32768):
                name = "TC" if mode == 1 else "TC16"
                path = "exact_fallback" if n < 32768 else "tensor"
                out.append(pytest.param(mode, d, k, n, id="%s-d%d-k%d-n%d-%s" % (name, d, k, n, path)))
    return out


@pytest.mark.parametrize("mode,d,k,n", _tc_cases())
def test_catalog_tensor_modes_equal_exact(ops, mode, d, k, n):
    """TOPK_TC (d = 32, 64, 96: 1..3 k-blocks) and TOPK_TC16 (d = 64: one k-block) return the exact mode's ids and
    scores bit for bit; n = 32767 is the last size the tensor path hands to the exact kernels."""
    from test_gpu_ops import _check_topk
    from prodsearch_b200 import _lib
    g = torch.Generator(device="cuda").manual_seed(d * 10 + k + n)
    m = 40
    E = torch.randn(n + 1, d, generator=g, device="cuda")
    E[n] = 0
    Q = torch.randn(m, d, generator=g, device="cuda")
    bias = torch.randn(n + 1, generator=g, device="cuda") * 0.1 if k == 128 else None
    ids_e, sc_e = ops.catalog_topk(Q, E, k, n_items=n, bias=bias, mode=_lib.TOPK_EXACT)
    with _Kernels() as kern:
        ids_t, sc_t = _topk_pair(ops, Q, E, k, n, bias, mode)
    if n >= 32768:
        assert _TC_LABEL[mode] in kern.names and "final_select_kernel" in kern.names, kern.names
    else:
        assert _TC_LABEL[mode] not in kern.names and "exact_scores_kernel" in kern.names, kern.names
    assert torch.equal(ids_e, ids_t) and torch.equal(sc_e, sc_t)
    _check_topk(ids_e, sc_e, Q.cpu(), E.cpu(), bias.cpu() if bias is not None else None, k, n)


@pytest.mark.parametrize("mode,d", [(1, 32), (1, 64), (1, 96), (2, 64)], ids=["TC-d32", "TC-d64", "TC-d96", "TC16-d64"])
def test_catalog_tensor_modes_sharded_ids(ops, mode, d):
    """Cyclic row sharding (owner = id % G): each shard runs the tensor path with id_base = r, id_stride = G.  The ids
    are base + stride * (the exact mode's local ids), and topk_merge of the shards is the unsharded exact list."""
    from test_gpu_ops import _check_topk
    from prodsearch_b200 import _lib
    G, per, m, k = 3, 33000, 24, 100
    n = G * per
    g = torch.Generator(device="cuda").manual_seed(d + mode)
    E = torch.randn(n, d, generator=g, device="cuda")
    Q = torch.randn(m, d, generator=g, device="cuda")
    bias = torch.randn(n, generator=g, device="cuda") * 0.1
    parts_i, parts_s = [], []
    for r in range(G):
        Er, br = E[r::G].contiguous(), bias[r::G].contiguous()
        li, ls = ops.catalog_topk(Q, Er, k, bias=br, mode=_lib.TOPK_EXACT)
        with _Kernels() as kern:
            ti, ts = _topk_pair(ops, Q, Er, k, per, br, mode, id_base=r, id_stride=G)
        assert _TC_LABEL[mode] in kern.names
        assert torch.equal(ti, r + G * li) and torch.equal(ts, ls)
        parts_i.append(ti)
        parts_s.append(ts)
    mi, ms = ops.topk_merge(torch.stack(parts_i), torch.stack(parts_s))
    gi, gs = ops.catalog_topk(Q, E, k, bias=bias, mode=_lib.TOPK_EXACT)
    assert torch.equal(mi, gi) and torch.equal(ms, gs)
    _check_topk(gi, gs, Q.cpu(), E.cpu(), bias.cpu(), k, n)


@pytest.mark.parametrize("mode", [1, 2], ids=["TC", "TC16"])
def test_catalog_tensor_modes_fallback_rows_map_ids(ops, mode):
    """Identical rows overflow the shortlist, so fallback_rows_kernel answers: lower local id first, mapped to
    id_base + id_stride * local id."""
    n, d, m, k, base, stride = 33000, 64, 3, 128, 5, 7
    E = torch.ones(n, d, device="cuda")
    Q = torch.ones(m, d, device="cuda")
    ids, sc = _topk_pair(ops, Q, E, k, n, None, mode, id_base=base, id_stride=stride)
    assert torch.equal(ids.cpu(), (base + stride * torch.arange(k)).repeat(m, 1))
    assert bool((sc == float(d)).all())
