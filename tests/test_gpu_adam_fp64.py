"""GPU: float64 references for the clipped Adam (csrc/optimizer.cu: psb_adam_step, psb_grad_sqnorm(_sparse),
psb_adam_sparse_step's row update, psb_adam_rows_catchup), for the catch-up series the peer lazy fetch applies
(psb_peer_gather_rows_lazy, csrc/peer.cu), and for the FusedAdam flows a run goes through: resume from a checkpoint, a
step in which a row-sparse table gets no row list, a CUDA-graph step built after eager steps.

The reference states the N2 contract of include/psb.h in float64 with the constants rounded as the contract and torch
round them: omb1 = fl(1 - b1), b2 = fl(b2), omb2 = fl(1 - b2), eps = fl(eps), and the per-step step_size_t =
fl(lr_t / (1 - b1^t)) and ibc_t = fl(1 / sqrt(1 - b2^t)), each formed in double and then rounded.  The clip factor is
formed in float64 from the kernel's own squared norm, read back; the squared norm is checked on its own against the
float64 sum of g^2.  A resting row's reference is the dense step applied k times with g = 0, in float64 -- not the
series the kernels sum (a CPU test pins that the two agree to 1e-12 when the series keeps all k terms).

Error bounds.  Every output element gets a first-order error magnitude M, carried through the step: each rounding
of an intermediate x adds K |x| (K per group below, from the operation count), and the magnitudes of the inputs
propagate through the derivative.  The bound is 2^-24 M.  The catch-up's parameter bound is the series' own: K (|p'|
+ sum_k |S_k| + sum_j |t_j| (14 + 1.39 j lambda)), where S_k are the partial sums of the terms t_j in the kernel's
order, 14 counts the roundings of one term and lambda = |log2(1 - omb1)| + |0.5 log2 b2| carries the exp2f of a
growing exponent; plus 2 ulp per __fdividef and the exact float64 tail sum_{j > kmax} |t_j| the series leaves out.
The closed-form moments m (1 - omb1)^k and v b2^k take two roundings.  Multi-step sequences carry their magnitudes
from step to step, so their bounds add up.  Parameters are drawn at 0, about 1e-6 and about 1, so that an update does
not hide under ulp(p).  The module prints the worst err / bound per group (pytest -s).
"""
import math

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

U = 2.0 ** -24
TINY = 2.0 ** -149                  # a result below the float range rounds to a multiple of the smallest subnormal
K_DENSE = 2                         # one step: every rounding is carried in M with weight 1; 2 covers second order
K_SERIES = 2                        # catch-up: the per-term and partial-sum roundings are counted in M
K_FLOW = 4                          # multi-step flows: dense steps and series catch-ups, carried with the dense M
K_SQNORM = 32                       # fp32 partial sums of <= 16 fma per thread, a 32 + 8 tree, then double
RATIOS = {}


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    if RATIOS:
        print("\nworst err / bound per group:")
        for g in sorted(RATIOS):
            print("  %-28s %.3g" % (g, RATIOS[g]))


def _check(group, got, ref, bound):
    """|got - ref| <= bound elementwise (bound == 0: exact)."""
    got = torch.as_tensor(got).detach().cpu().double().reshape(-1)
    ref = torch.as_tensor(ref).detach().cpu().double().reshape(-1)
    bound = torch.as_tensor(bound).detach().cpu().double().reshape(-1)
    assert got.shape == ref.shape == bound.shape
    if got.numel() == 0:
        return
    assert bool(torch.isfinite(got).all()), "%s: non-finite output" % group
    err = (got - ref).abs()
    ratio = torch.where(bound > 0, err / torch.where(bound > 0, bound, torch.ones_like(bound)),
                        torch.where(err > 0, torch.full_like(err, float("inf")), torch.zeros_like(err)))
    j = int(ratio.argmax())
    worst = float(ratio[j])
    RATIOS[group] = max(RATIOS.get(group, 0.0), worst)
    assert worst <= 1.0, "%s: err / bound %.3g at flat %d (got %r, ref %r, bound %r)" % (
        group, worst, j, float(got[j]), float(ref[j]), float(bound[j]))


def _f32(x):
    return float(np.float32(x))


class Hyper(object):
    """The hyper-parameters as the kernels round them (AdamHyper, step_coef, make_coef)."""

    def __init__(self, lr, b1=0.9, b2=0.999, eps=1e-9, max_norm=0.0, wd=0.0, noam=False, warm=4000.0):
        self.lr, self.beta1, self.beta2, self.eps_d = lr, b1, b2, eps
        self.omb1, self.b2, self.omb2, self.eps = _f32(1.0 - b1), _f32(b2), _f32(1.0 - b2), _f32(eps)
        self.base1 = 1.0 - self.omb1                        # m decays by this per zero-gradient step (lerp)
        self.max_norm, self.max_norm_d, self.wd, self.wd_d = _f32(max_norm), max_norm, _f32(wd), wd
        self.noam, self.warm = bool(noam), _f32(warm)

    def coef(self, t):
        lr = self.lr
        if self.noam:
            lr = self.lr * min(1.0 / math.sqrt(t), t * self.warm ** -1.5)
        return _f32(lr / (1.0 - self.beta1 ** t)), _f32(1.0 / math.sqrt(1.0 - self.beta2 ** t))

    def clip(self, sq):
        """(c, clipped) from the kernel's squared norm: c = min(max_norm / (sqrt(sq) + 1e-6), 1)."""
        if self.max_norm <= 0:
            return 1.0, False
        c = self.max_norm / (math.sqrt(sq) + _f32(1e-6))
        return (c, True) if c < 1.0 else (1.0, False)

    def hist(self, cap):
        """The coefficient history the optimizer step writes: float2 (step_size_t, ibc_t) at index t (t >= 1)."""
        h = torch.zeros(cap, 2, dtype=torch.float32)
        for t in range(1, cap):
            h[t, 0], h[t, 1] = self.coef(t)
        return h.reshape(-1).contiguous()

    def lazy_args(self):
        return (self.lr, self.beta1, self.beta2, self.eps_d, 1 if self.noam else 0, float(self.warm))


def _state(p, m, v, M=None):
    z = torch.zeros(p.shape, dtype=torch.float64)
    st = dict(p=p.double().cpu().clone(), m=m.double().cpu().clone(), v=v.double().cpu().clone(),
              Mp=z.clone(), Mm=z.clone(), Mv=z.clone())
    if M is not None:
        st.update(M)
    return st


def step64(st, g, h, t, c=1.0, clipped=False, K=K_DENSE):
    """One dense Adam step in float64 (kernel adam_one); M carried in units of 2^-24."""
    ss, ibc = h.coef(t)
    p, m, v = st["p"], st["m"], st["v"]
    gc = c * g.double()
    Mg = K * 4.0 * gc.abs() if clipped else torch.zeros_like(gc)   # c: sqrtf, + 1e-6f, division; then c g
    if h.wd:
        gn = h.wd * p + gc
        Mg = Mg + K * gn.abs() + h.wd * st["Mp"]
        gc = gn
    dm = gc - m
    m2 = m + h.omb1 * dm
    Mm = K * (m2.abs() + h.omb1 * dm.abs()) + h.omb1 * Mg + (1.0 - h.omb1) * st["Mm"]
    g2 = gc * gc
    v2 = h.b2 * v + h.omb2 * g2
    Mv = K * (v2.abs() + h.b2 * v.abs() + h.omb2 * g2) + h.b2 * st["Mv"] + 2.0 * h.omb2 * gc.abs() * Mg
    s = v2.sqrt()
    Ms = K * s + torch.where(s > 0, Mv / (2.0 * torch.where(s > 0, s, torch.ones_like(s))), torch.zeros_like(s))
    den = s * ibc + h.eps
    Md = K * (den + 2.0 * s * ibc) + ibc * Ms
    q = m2 / den
    Mq = K * q.abs() + Mm / den + q.abs() * Md / den
    p2 = p - ss * q
    Mp = K * (p2.abs() + ss * q.abs()) + ss * Mq + st["Mp"]
    return dict(p=p2, m=m2, v=v2, Mp=Mp, Mm=Mm, Mv=Mv)


def series_terms(m0, v0, h, frm, n):
    """t_j, j = 1..n, of the catch-up series from step frm in float64: [n, *m0.shape]."""
    j = torch.arange(1, n + 1, dtype=torch.float64)
    cf = torch.tensor([h.coef(frm + int(k)) for k in j], dtype=torch.float64)
    a = cf[:, 0] * h.base1 ** j
    b = cf[:, 1] * h.b2 ** (j / 2)
    shp = (n,) + (1,) * m0.dim()
    return a.view(shp) * m0.unsqueeze(0) / (b.view(shp) * v0.sqrt().unsqueeze(0) + h.eps), j.view(shp)


def catchup64(st, h, frm, to, kmax, K=K_SERIES):
    """A row resting over steps frm+1 .. to: the float64 dense replay with g = 0, and the bound of the kernel's
    series (first min(gap, kmax) terms) + closed-form moments."""
    ref = dict(st)
    zero = torch.zeros_like(st["p"])
    for t in range(frm + 1, to + 1):
        ref = step64(ref, zero, h, t)
    gap = to - frm
    terms, j = series_terms(st["m"], st["v"], h, frm, gap)
    n = min(gap, kmax)
    head, tail = terms[:n].abs(), terms[n:].abs().sum(0)
    lam = abs(math.log2(h.base1)) + abs(0.5 * math.log2(h.b2))
    Mp = K * (ref["p"].abs() + terms[:n].cumsum(0).abs().sum(0) + (head * (14.0 + 1.39 * j[:n] * lam)).sum(0))
    Mp = Mp + 4.0 * head.sum(0) + tail / U + st["Mp"]
    out = dict(p=ref["p"], m=ref["m"], v=ref["v"], Mp=Mp,
               Mm=K * 2.0 * ref["m"].abs() + TINY / U + h.base1 ** gap * st["Mm"],
               Mv=K * 2.0 * ref["v"].abs() + TINY / U + h.b2 ** gap * st["Mv"])
    return out


# ------------------------------------------------------------------------------------------------ CPU: the reference
@pytest.mark.parametrize("b1,noam,frm,gap", [(0.9, False, 3, 1), (0.9, False, 40, 199), (0.9, True, 10, 250),
                                             (0.5, False, 7, 120), (0.9, False, 1, 2000)])
def test_series_with_every_term_equals_the_step_by_step_replay(b1, noam, frm, gap):
    """The float64 series plus closed-form moments, summed over all k terms, is the float64 replay of k dense steps
    with g = 0 (what the catch-up kernels approximate by their first kmax terms)."""
    h = Hyper(2e-3, b1=b1, noam=noam, warm=50.0)
    g = torch.Generator().manual_seed(frm + gap)
    m0 = torch.randn(6, 8, generator=g, dtype=torch.float64) * 1e-2
    v0 = torch.rand(6, 8, generator=g, dtype=torch.float64) * 1e-4 + 1e-20
    p0 = torch.zeros(6, 8, dtype=torch.float64)
    ref = catchup64(_state(p0, m0, v0), h, frm, frm + gap, kmax=gap)
    terms, _ = series_terms(m0, v0, h, frm, gap)
    delta = terms.sum(0)
    scale = terms.abs().sum(0)
    assert float(((p0 - delta) - ref["p"]).abs().max() / scale.max()) <= 1e-12
    assert float(((m0 * h.base1 ** gap - ref["m"]).abs() / (ref["m"].abs() + 1e-300)).max()) <= 1e-12
    assert float(((v0 * h.b2 ** gap - ref["v"]).abs() / ref["v"].abs()).max()) <= 1e-12


# ------------------------------------------------------------------------------------------------ GPU helpers
def _lib():
    from prodsearch_b200 import _lib as L
    return L, L.load()


class _Kernels(object):
    """Names of the library kernels launched inside the block (the library's event profiler)."""

    def __enter__(self):
        self.L, _ = _lib()
        self.L.profile_enable(True)
        self.names = set()
        return self

    def __exit__(self, *exc):
        try:
            self.names = set(self.L.profile_dump())
        finally:
            self.L.profile_enable(False)
        return False


def _params(g, n):
    """Parameters at 0, about 1e-6 and about 1 (an update of ~lr is visible next to the first two)."""
    p = torch.randn(n, generator=g)
    sel = torch.randint(0, 3, (n,), generator=g)
    return torch.where(sel == 0, torch.zeros_like(p), torch.where(sel == 1, p * 1e-6, p))


def _moments(g, shape, fresh_every=0):
    n = int(np.prod(shape))
    m = torch.randn(n, generator=g) * 1e-3
    v = torch.rand(n, generator=g) * 1e-5 + 1e-12
    m[::5] = 0.0                                  # m = 0
    v[3::11] = 1e-20                              # sqrt(v) ~ 1e-10, below eps
    return m.view(shape), v.view(shape)


# ------------------------------------------------------------------------------------------------ dense psb_adam_step
_SIZES64 = [1 + (37 * i) % 300 for i in range(64)]
DENSE = {
    "n1": dict(sizes=[1]), "n3": dict(sizes=[3]), "n4": dict(sizes=[4]), "n4095": dict(sizes=[4095]),
    "n4096": dict(sizes=[4096]), "n4097": dict(sizes=[4097]),
    "scalar_misaligned": dict(sizes=[4097, 5], misaligned=True),
    "tensors64": dict(sizes=_SIZES64),
    "partials_gt256": dict(sizes=[1200000, 777]),
    "clip_active": dict(sizes=[4097, 300], max_norm=0.05),
    "clip_inactive": dict(sizes=[4097, 300], max_norm=1e6),
    "max_norm_0": dict(sizes=[4097, 300], max_norm=0.0),
    "weight_decay": dict(sizes=[4097, 300], max_norm=5.0, wd=0.01),
    "noam": dict(sizes=[4097, 300], max_norm=5.0, noam=True),
    "norm_given_1": dict(sizes=[4097, 300], max_norm=0.5, norm_given=1),
    "norm_given_2": dict(sizes=[4097, 300], max_norm=0.5, norm_given=2),
}


@gpu
@pytest.mark.parametrize("case", list(DENSE))
def test_dense_adam_step_fp64(case):
    L, lib = _lib()
    cfg = DENSE[case]
    ng = cfg.get("norm_given", 0)
    h = Hyper(5e-4, max_norm=cfg.get("max_norm", 1.0), wd=cfg.get("wd", 0.0), noam=cfg.get("noam", False), warm=20.0)
    g = torch.Generator().manual_seed(sum(map(ord, case)))
    off = 1 if cfg.get("misaligned") else 0
    host, dev, arr = [], [], (L.AdamTensor * len(cfg["sizes"]))()
    for i, n in enumerate(cfg["sizes"]):
        p = _params(g, n)
        gr = torch.randn(n, generator=g) * 0.1
        gr[::7] = 0.0
        m, v = _moments(g, (n,))
        host.append((p, gr, m, v))
        bufs = []
        for x in (p, gr, m, v):
            b = torch.zeros(n + off, device="cuda")
            b[off:] = x.cuda()
            bufs.append(b[off:])
        dev.append(bufs)
        if off:
            assert bufs[0].data_ptr() % 16 != 0
        arr[i] = L.AdamTensor(bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(), bufs[3].data_ptr(), n)
    t0 = 6
    step_dev = torch.tensor([t0 + (1 if ng == 2 else 0)], dtype=torch.int64, device="cuda")
    sq_true = sum(float((x[1].double() ** 2).sum()) for x in host)
    sq_dev = torch.tensor([_f32(0.75 * sq_true) if ng else 0.0], device="cuda")
    wb = int(lib.psb_adam_workspace_bytes(arr, len(host)))
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
    with _Kernels() as k:
        L.check(lib.psb_adam_step(arr, len(host), h.lr, h.beta1, h.beta2, h.eps_d, h.wd_d, h.max_norm_d,
                                  1 if h.noam else 0, float(h.warm), ng, step_dev.data_ptr(), sq_dev.data_ptr(),
                                  ws.data_ptr(), wb, L.stream_ptr()), "psb_adam_step")
    want = {0: {"sqnorm_partial_kernel", "sqnorm_final_kernel", "adam_kernel"}, 1: {"bump_step_kernel", "adam_kernel"},
            2: {"adam_kernel"}}[ng]
    assert k.names == want, k.names
    assert int(step_dev.item()) == t0 + 1
    sq = float(sq_dev.item())
    if ng == 0:
        _check("sqnorm", sq, sq_true, K_SQNORM * U * sq_true)
    c, clipped = h.clip(sq)
    if case == "clip_active":
        assert clipped
    for (p, gr, m, v), bufs in zip(host, dev):
        ref = step64(_state(p, m, v), gr, h, t0 + 1, c, clipped)
        for name, got in zip(("p", "m", "v"), (bufs[0], bufs[2], bufs[3])):
            _check("dense " + name, got, ref[name], U * ref["M" + name])


@gpu
def test_grad_sqnorm_dense_and_sparse_fp64():
    """psb_grad_sqnorm and psb_grad_sqnorm_sparse against the float64 sum of g^2 (more than 256 partials, compact and
    by-row lists with a bias gradient), bit-identical on a second call."""
    L, lib = _lib()
    g = torch.Generator().manual_seed(11)
    gs = [torch.randn(n, generator=g).cuda() for n in (1200000, 4097, 3)]
    arr = (L.AdamTensor * 3)()
    for i, x in enumerate(gs):
        arr[i] = L.AdamTensor(None, x.data_ptr(), None, None, x.numel())
    wb = int(lib.psb_adam_workspace_bytes(arr, 3))
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
    outs = []
    for _ in range(2):
        out = torch.zeros(1, device="cuda")
        L.check(lib.psb_grad_sqnorm(arr, 3, out.data_ptr(), ws.data_ptr(), wb, L.stream_ptr()), "psb_grad_sqnorm")
        outs.append(out.item())
    ref = sum(float((x.double() ** 2).sum()) for x in gs)
    assert outs[0] == outs[1]
    _check("sqnorm", outs[0], ref, K_SQNORM * U * ref)
    # tables: compact lists (entries past n_rows excluded) and a dense by-row buffer (only listed in-range rows count)
    R, d, cap, n = 300, 132, 45, 37
    rows = torch.randperm(R, generator=g)[:cap].int()
    rows[5], rows[9] = -3, R + 5
    comp = torch.randn(cap, d, generator=g)
    comp_b = torch.randn(cap, generator=g)
    byrow = torch.randn(R, d, generator=g)
    byrow_b = torch.randn(R, generator=g)
    rows_d, nu = rows.cuda(), torch.tensor([n], dtype=torch.int32, device="cuda")
    keep = [rows_d, nu]
    tabs = (L.AdamRows * 2)()
    for i, (gg, bb, by) in enumerate(((comp, comp_b, 0), (byrow, byrow_b, 1))):
        gd, bd = gg.cuda(), bb.cuda()
        keep += [gd, bd]
        T = L.AdamRows()
        T.rows, T.grad, T.n_rows, T.cap, T.d, T.table_rows = rows_d.data_ptr(), gd.data_ptr(), nu.data_ptr(), cap, d, R
        T.bias_grad, T.grad_by_row = bd.data_ptr(), by
        tabs[i] = T
    wb = int(lib.psb_adam_sparse_workspace_bytes(arr, 3, tabs, 2))
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
    outs = []
    for _ in range(2):
        out = torch.zeros(1, device="cuda")
        L.check(lib.psb_grad_sqnorm_sparse(arr, 3, tabs, 2, out.data_ptr(), ws.data_ptr(), wb, L.stream_ptr()),
                "psb_grad_sqnorm_sparse")
        outs.append(out.item())
    ok = rows[:n].long()
    ok = ok[(ok >= 0) & (ok < R)]
    ref += float((comp[:n].double() ** 2).sum() + (comp_b[:n].double() ** 2).sum())
    ref += float((byrow[ok].double() ** 2).sum() + (byrow_b[ok].double() ** 2).sum())
    assert outs[0] == outs[1]
    _check("sqnorm", outs[0], ref, K_SQNORM * U * ref)


# ------------------------------------------------------------------------------------------------ row update
def _hist_dev(h, cap):
    return h.hist(cap).cuda()


@gpu
@pytest.mark.parametrize("d", [4, 128, 132, 512])
@pytest.mark.parametrize("layout", ["compact", "by_row"])
def test_adam_rows_kernel_fp64(d, layout):
    """Three tables in one psb_adam_sparse_step: bias with a gradient, bias without one (bias_grad NULL), no bias.
    Listed rows are fresh, current or stale (caught up first, also past kmax); cap is not a multiple of 8, entries past
    n_rows and out-of-range ids leave memory untouched."""
    L, lib = _lib()
    h = Hyper(1e-3, max_norm=1.0)
    kmax = int(lib.psb_adam_catchup_steps(h.beta1, h.beta2))
    R, cap, n, t = 300, 45, 37, 301
    by = 1 if layout == "by_row" else 0
    g = torch.Generator().manual_seed(d * 7 + by)
    hist = _hist_dev(h, 4096)
    hist[2 * t:2 * t + 2] = 0.0
    step_dev = torch.tensor([t - 1], dtype=torch.int64, device="cuda")
    sq_dev = torch.zeros(1, device="cuda")
    tabs, host, keep = (L.AdamRows * 3)(), [], []
    prevs = [0, t - 1, t - 2, t - 6, t - 41, t - 1 - 250]     # fresh, current, stale by 1, 5, 40, 250 (> kmax) steps
    for i, bias_kind in enumerate(("grad", "nograd", "none")):
        perm = torch.randperm(R, generator=g)
        rows = perm[:cap].int().clone()
        rows[4], rows[11] = -3, R + 5                   # out-of-range ids inside the valid prefix
        p = _params(g, R * d).view(R, d)
        m, v = _moments(g, (R, d))
        last = torch.tensor([prevs[int(x)] for x in torch.randint(0, len(prevs), (R,), generator=g)], dtype=torch.int32)
        m[last == 0], v[last == 0] = 0.0, 0.0
        grad = torch.randn(cap if not by else R, d, generator=g) * 0.2
        bp, bm, bv = _params(g, R), *_moments(g, (R,))
        bm[last == 0], bv[last == 0] = 0.0, 0.0
        bgrad = torch.randn(cap if not by else R, generator=g) * 0.2
        D = dict(p=p.cuda(), m=m.cuda(), v=v.cuda(), last=last.cuda(), rows=rows.cuda(), grad=grad.cuda(),
                 nu=torch.tensor([n], dtype=torch.int32, device="cuda"), bp=bp.cuda(), bm=bm.cuda(), bv=bv.cuda(),
                 bgrad=bgrad.cuda())
        keep.append(D)
        T = L.AdamRows()
        T.p, T.m, T.v, T.last_step = D["p"].data_ptr(), D["m"].data_ptr(), D["v"].data_ptr(), D["last"].data_ptr()
        T.rows, T.grad, T.n_rows = D["rows"].data_ptr(), D["grad"].data_ptr(), D["nu"].data_ptr()
        T.cap, T.d, T.table_rows, T.grad_by_row = cap, d, R, by
        if bias_kind != "none":
            T.bias_p, T.bias_m, T.bias_v = D["bp"].data_ptr(), D["bm"].data_ptr(), D["bv"].data_ptr()
        if bias_kind == "grad":
            T.bias_grad = D["bgrad"].data_ptr()
        tabs[i] = T
        host.append((bias_kind, p, m, v, last, rows, grad, bp, bm, bv, bgrad))
    wb = int(lib.psb_adam_sparse_workspace_bytes(None, 0, tabs, 3))
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
    with _Kernels() as k:
        L.check(lib.psb_adam_sparse_step(None, 0, tabs, 3, h.lr, h.beta1, h.beta2, h.eps_d, h.max_norm_d, 0, 4000.0, 0,
                                         step_dev.data_ptr(), sq_dev.data_ptr(), hist.data_ptr(), 4096, ws.data_ptr(),
                                         wb, L.stream_ptr()), "psb_adam_sparse_step")
    assert k.names == {"sqnorm_rows_partial_kernel", "sqnorm_final_kernel", "adam_rows_kernel"}, k.names
    assert int(step_dev.item()) == t
    assert hist[2 * t:2 * t + 2].cpu().tolist() == list(h.coef(t))
    sq = float(sq_dev.item())
    sq_ref = 0.0
    for bias_kind, p, m, v, last, rows, grad, bp, bm, bv, bgrad in host:
        ids = rows[:n].long()
        valid = ids[(ids >= 0) & (ids < R)]
        if by:
            sq_ref += float((grad[valid].double() ** 2).sum()) + (float((bgrad[valid].double() ** 2).sum())
                                                                  if bias_kind == "grad" else 0.0)
        else:
            sq_ref += float((grad[:n].double() ** 2).sum()) + (float((bgrad[:n].double() ** 2).sum())
                                                               if bias_kind == "grad" else 0.0)
    _check("sqnorm", sq, sq_ref, K_SQNORM * U * sq_ref)
    c, clipped = h.clip(sq)
    assert clipped
    for (bias_kind, p, m, v, last, rows, grad, bp, bm, bv, bgrad), D in zip(host, keep):
        listed = set()
        for i in range(n):
            r = int(rows[i])
            if r < 0 or r >= R:
                continue
            listed.add(r)
            prev = int(last[r])
            gi = r if by else i
            for which, (P, Mo, V, G) in (("row", (p[r], m[r], v[r], grad[gi])),
                                         ("bias", (bp[r:r + 1], bm[r:r + 1], bv[r:r + 1],
                                                   bgrad[gi:gi + 1] if bias_kind == "grad" else torch.zeros(1)))):
                if which == "bias" and bias_kind == "none":
                    continue
                st = _state(P, Mo, V)
                if 0 < prev < t - 1:
                    st = catchup64(st, h, prev, t - 1, kmax)
                ref = step64(st, G, h, t, c, clipped)
                if which == "row":
                    got = (D["p"][r], D["m"][r], D["v"][r])
                else:
                    got = (D["bp"][r:r + 1], D["bm"][r:r + 1], D["bv"][r:r + 1])
                grp = "rows %s%s" % (which, " stale" if 0 < prev < t - 1 else "")
                for name, x in zip(("p", "m", "v"), got):
                    _check(grp + " " + name, x, ref[name], U * ref["M" + name])
            assert int(D["last"][r]) == t
        rest = torch.tensor(sorted(set(range(R)) - listed), dtype=torch.long)
        assert torch.equal(D["p"].cpu()[rest], p[rest]) and torch.equal(D["m"].cpu()[rest], m[rest])
        assert torch.equal(D["v"].cpu()[rest], v[rest]) and torch.equal(D["last"].cpu()[rest], last[rest])
        if bias_kind != "none":
            assert torch.equal(D["bp"].cpu()[rest], bp[rest]) and torch.equal(D["bv"].cpu()[rest], bv[rest])


# ------------------------------------------------------------------------------------------------ catch-up
RESTS = [1, 31, 32, 33, 197, 198, 199, 2000]
CATCHUP = {"b0.9": dict(b1=0.9), "b0.5_past_kmax": dict(b1=0.5), "noam": dict(b1=0.9, noam=True, warm=300.0)}


def _catchup_table(g, R, d, cur):
    """A table whose rows rest for each of RESTS steps, plus fresh (0) and current rows."""
    p = _params(g, R * d).view(R, d)
    m, v = _moments(g, (R, d))
    m[::5] = torch.randn(d, generator=g) * 1e-3                  # no all-zero rows: every rest moves the row
    choices = [cur - r for r in RESTS] + [0, cur]
    last = torch.tensor([choices[i % len(choices)] for i in range(R)], dtype=torch.int32)
    m[last == 0], v[last == 0] = 0.0, 0.0
    bp, bm, bv = _params(g, R), *_moments(g, (R,))
    bm[last == 0], bv[last == 0] = 0.0, 0.0
    return p, m, v, last, bp, bm, bv


def _replay_rows(p, m, v, last, cur, h, kmax, rows):
    """float64 reference + bound of rows brought from last[r] to cur (unchanged if fresh or current)."""
    groups, out = {}, {}
    for r in rows:
        groups.setdefault(int(last[r]), []).append(r)
    for prev, rs in groups.items():
        idx = torch.tensor(rs, dtype=torch.long)
        st = _state(p[idx], m[idx], v[idx])
        if 0 < prev < cur:
            st = catchup64(st, h, prev, cur, kmax)
        for i, r in enumerate(rs):
            out[r] = {k: x[i] for k, x in st.items()}
    return out


@gpu
@pytest.mark.parametrize("case", list(CATCHUP))
def test_rows_catchup_fp64(case):
    """psb_adam_rows_catchup over 8 index lists with duplicates inside and across them, the skip row and out-of-range
    ids among them; then a flush.  coef_hist given, NULL and shorter than the steps: bit-identical."""
    L, lib = _lib()
    cfg = CATCHUP[case]
    h = Hyper(2e-3, b1=cfg["b1"], noam=cfg.get("noam", False), warm=cfg.get("warm", 4000.0))
    kmax = int(lib.psb_adam_catchup_steps(h.beta1, h.beta2))
    if cfg["b1"] == 0.5:
        assert kmax < 40                            # rests of 197 .. 2000 steps have a tail past kmax
    R, d, cur = 120, 132, 2100
    g = torch.Generator().manual_seed(sum(map(ord, case)))
    p, m, v, last, bp, bm, bv = _catchup_table(g, R, d, cur)
    skip = 7
    listed = sorted(set(range(0, R, 2)) - {skip})
    lists = []
    for q in range(8):                             # every listed row in two lists, some twice in one list
        sel = [r for r in listed if (r // 2) % 4 == q % 4]
        lst = sel + sel[:3] + [skip, -1, R + 9]
        lists.append(torch.tensor(lst, dtype=torch.int64))
    step_dev = torch.tensor([cur], dtype=torch.int64, device="cuda")
    results = []
    for variant, (hist, hcap) in (("hist", (_hist_dev(h, 4096), 4096)), ("null", (None, 4096)),
                                  ("short", (_hist_dev(h, 64), 64))):
        D = [x.cuda() for x in (p, m, v, last, bp, bm, bv)]
        T = L.AdamRows()
        T.p, T.m, T.v, T.last_step = D[0].data_ptr(), D[1].data_ptr(), D[2].data_ptr(), D[3].data_ptr()
        T.d, T.table_rows = d, R
        T.bias_p, T.bias_m, T.bias_v = D[4].data_ptr(), D[5].data_ptr(), D[6].data_ptr()
        ld = [x.cuda() for x in lists]
        ptrs = (L.c_vp * 8)(*[x.data_ptr() for x in ld])
        cnts = (L.c_i64 * 8)(*[x.numel() for x in ld])
        with _Kernels() as k:
            L.check(lib.psb_adam_rows_catchup(T, ptrs, cnts, 8, skip, *h.lazy_args(), step_dev.data_ptr(),
                                              hist.data_ptr() if hist is not None else None, hcap, L.stream_ptr()),
                    "psb_adam_rows_catchup")
        assert k.names == {"adam_rows_catchup_kernel"}, k.names
        results.append([x.cpu() for x in D])
    for other in results[1:]:
        for a, b in zip(results[0], other):
            assert torch.equal(a, b)
    got = results[0]
    ref = _replay_rows(p, m, v, last, cur, h, kmax, range(R))
    bias_ref = _replay_rows(bp.view(R, 1), bm.view(R, 1), bv.view(R, 1), last, cur, h, kmax, range(R))
    for r in range(R):
        prev = int(last[r])
        if r in listed:
            for name, x in zip(("p", "m", "v"), got[:3]):
                _check("catchup %s" % name, x[r], ref[r][name], U * ref[r]["M" + name])
            for name, x in zip(("p", "m", "v"), got[4:]):
                _check("catchup bias %s" % name, x[r:r + 1], bias_ref[r][name], U * bias_ref[r]["M" + name])
            assert int(got[3][r]) == cur
        else:                                      # unlisted rows and the skip row: untouched
            for a, b in zip(got, (p, m, v, last, bp, bm, bv)):
                assert torch.equal(a[r], b[r])
            assert prev == int(got[3][r])
    # flush (no lists): every row but the skip row, from the lists' result
    D = [x.cuda() for x in got]
    T = L.AdamRows()
    T.p, T.m, T.v, T.last_step = D[0].data_ptr(), D[1].data_ptr(), D[2].data_ptr(), D[3].data_ptr()
    T.d, T.table_rows = d, R
    T.bias_p, T.bias_m, T.bias_v = D[4].data_ptr(), D[5].data_ptr(), D[6].data_ptr()
    L.check(lib.psb_adam_rows_catchup(T, None, None, 0, skip, *h.lazy_args(), step_dev.data_ptr(), None, 4096,
                                      L.stream_ptr()), "flush")
    flushed = [x.cpu() for x in D]
    for r in range(R):
        if r in listed:
            for a, b in zip(flushed, got):
                assert torch.equal(a[r], b[r])     # already current: nothing replayed twice
        elif r == skip:
            for a, b in zip(flushed, (p, m, v, last, bp, bm, bv)):
                assert torch.equal(a[r], b[r])
        else:
            for name, x in zip(("p", "m", "v"), flushed[:3]):
                _check("catchup %s" % name, x[r], ref[r][name], U * ref[r]["M" + name])
            for name, x in zip(("p", "m", "v"), flushed[4:]):
                _check("catchup bias %s" % name, x[r:r + 1], bias_ref[r][name], U * bias_ref[r]["M" + name])


@gpu
@pytest.mark.parametrize("world", [1, 3])
def test_peer_lazy_fetch_fp64(world):
    """psb_peer_gather_rows_lazy hands out resting rows as the float64 replay of their skipped dense steps, at every
    rest length of the catch-up test; nothing is written back."""
    from prodsearch_b200 import peer
    L, lib = _lib()
    h = Hyper(2e-3)
    kmax = int(lib.psb_adam_catchup_steps(h.beta1, h.beta2))
    rows, d, cur = 301, 128, 2100
    g = torch.Generator().manual_seed(40 + world)
    p, m, v, last, _, _, _ = _catchup_table(g, rows, d, cur)
    groups = peer.PeerGroup.simulate(world, "cuda")
    tabs = [peer.PeerShardedTable(rows, d, grp, pad_idx=rows - 1, full=p.cuda(), sparse=True) for grp in groups]
    for r0, t in enumerate(tabs):
        own = torch.arange(r0, rows, world)[:t.local_rows]
        assert torch.equal(t.weight.detach().cpu()[:own.numel()], p[own])
        t.exp_avg[:own.numel()].copy_(m[own].cuda())
        t.exp_avg_sq[:own.numel()].copy_(v[own].cuda())
        t.last_step[:own.numel()].copy_(last[own].cuda())
    before = [(t.weight.detach().clone(), t.exp_avg.clone(), t.exp_avg_sq.clone(), t.last_step.clone()) for t in tabs]
    ids = torch.cat([torch.arange(rows - 1), torch.arange(0, rows - 1, 3)]).cuda()
    t0 = tabs[0]
    P, M, V, Ls = t0.shard.ptr_array(), t0._m_buf.ptr_array(), t0._v_buf.ptr_array(), t0._last_buf.ptr_array()
    hist = _hist_dev(h, 4096)
    step_dev = torch.tensor([cur], dtype=torch.int64, device="cuda")
    out = torch.empty(ids.numel(), d, device="cuda")
    with _Kernels() as k:
        L.check(lib.psb_peer_gather_rows_lazy(P, M, V, Ls, world, rows, d, ids.data_ptr(), ids.numel(), out.data_ptr(),
                                              None, -1, 0, None, *h.lazy_args(), step_dev.data_ptr(), hist.data_ptr(),
                                              4096, L.stream_ptr()), "psb_peer_gather_rows_lazy")
    assert k.names == {"peer_gather_rows_lazy_kernel"}, k.names
    for t, b in zip(tabs, before):
        for a, c in zip((t.weight.detach(), t.exp_avg, t.exp_avg_sq, t.last_step), b):
            assert torch.equal(a, c)
    ref = _replay_rows(p, m, v, last, cur, h, kmax, range(rows - 1))
    got = out.cpu()
    for i, r in enumerate(ids.cpu().tolist()):
        _check("peer lazy p", got[i], ref[r]["p"], U * ref[r]["Mp"])


# ------------------------------------------------------------------------------------------------ FusedAdam flows
class _Flow(object):
    """A table with a bias (row-sparse) and a dense parameter under FusedAdam, driven by a fixed sequence of steps."""

    R, d, nd = 500, 64, 300

    def __init__(self, init):
        from prodsearch_b200.optimizers import FusedAdam
        self.tab = torch.nn.Parameter(init[0].clone().cuda())
        self.bias = torch.nn.Parameter(init[1].clone().cuda())
        self.dense = torch.nn.Parameter(init[2].clone().cuda())
        self.tab._psb_row_bias = self.bias
        self.opt = FusedAdam([self.tab, self.bias, self.dense], lr=1e-3)
        self.sq = []

    def step(self, s, max_norm):
        rows, vals, bvals, dg = s
        if rows is not None:
            cap = rows.numel() + 5
            rd = torch.full((cap,), -7, dtype=torch.int32)
            rd[:rows.numel()] = rows.int()
            nu = torch.tensor([rows.numel()], dtype=torch.int32).cuda()
            vd = torch.zeros(cap, self.d)
            vd[:rows.numel()] = vals
            bd = torch.zeros(cap)
            bd[:rows.numel()] = bvals
            rd = rd.cuda()
            self.tab.row_grad = (rd, vd.cuda(), nu)
            self.bias.row_grad = (rd, bd.cuda(), nu)
        self.dense.grad = dg.cuda()
        self.opt.step(max_grad_norm=max_norm)
        self.sq.append(float(self.opt._sqnorm.item()))

    def values(self):
        st = self.opt.state
        return [self.tab.detach(), self.bias.detach(), self.dense.detach()] + [
            st[p][k] for p in (self.tab, self.bias, self.dense) for k in ("exp_avg", "exp_avg_sq")]


def _flow_data(seed, steps, no_rows=()):
    g = torch.Generator().manual_seed(seed)
    init = (_params(g, _Flow.R * _Flow.d).view(_Flow.R, _Flow.d), _params(g, _Flow.R), _params(g, _Flow.nd))
    seq = []
    for s in range(1, steps + 1):
        dg = torch.randn(_Flow.nd, generator=g) * 0.05
        if s in no_rows:
            seq.append((None, None, None, dg))
            continue
        rows = torch.randperm(_Flow.R, generator=g)[:40 + s].sort().values
        sc = 2.0 if s % 3 == 0 else 0.02                         # the clip is active at every third step
        seq.append((rows, torch.randn(rows.numel(), _Flow.d, generator=g) * sc,
                    torch.randn(rows.numel(), generator=g) * sc, dg))
    return init, seq


def _flow_ref(init, seq, sq, max_norm):
    """float64 dense replay: every row, every step; rows without a gradient take g = 0."""
    h = Hyper(1e-3, max_norm=max_norm)
    sts = [_state(x, torch.zeros_like(x), torch.zeros_like(x)) for x in init]
    for t, ((rows, vals, bvals, dg), s2) in enumerate(zip(seq, sq), start=1):
        c, clipped = h.clip(s2)
        gt, gb = torch.zeros(_Flow.R, _Flow.d), torch.zeros(_Flow.R)
        if rows is not None:
            gt[rows], gb[rows] = vals, bvals
        sts = [step64(st, gg, h, t, c, clipped, K=K_FLOW) for st, gg in zip(sts, (gt, gb, dg))]
    return sts


def _check_flow(group, flow, ref):
    got = flow.values()
    for i, st in enumerate(ref):
        _check(group + " p", got[i], st["p"], U * st["Mp"])
    for i, st in enumerate(ref):
        _check(group + " m", got[3 + 2 * i], st["m"], U * st["Mm"])
        _check(group + " v", got[4 + 2 * i], st["v"], U * st["Mv"])


@gpu
def test_resume_from_state_dict_equals_uninterrupted_run():
    """S row-sparse steps, state_dict(), a new optimizer that loads it, T more steps, flush: bit-identical to a run that
    flushes at step S and goes on, and within the float64 dense replay's bound.  Rows that rest after the resume must
    still take the decay and the updates of every step."""
    S, T, max_norm = 4, 6, 1.0
    init, seq = _flow_data(21, S + T)
    a = _Flow(init)
    for s in seq[:S]:
        a.step(s, max_norm)
    a.opt.flush()
    for s in seq[S:]:
        a.step(s, max_norm)
    a.opt.flush()
    b = _Flow(init)
    for s in seq[:S]:
        b.step(s, max_norm)
    sd = b.opt.state_dict()
    assert float(sd["state"][0]["step"]) == S
    c = _Flow([x.cpu() for x in (b.tab.detach(), b.bias.detach(), b.dense.detach())])
    c.opt.load_state_dict(sd)
    for s in seq[S:]:
        c.step(s, max_norm)
    c.opt.flush()
    assert int(c.opt._step_dev.item()) == S + T
    for x, y in zip(a.values(), c.values()):
        assert torch.equal(x, y)
    _check_flow("flow resume", c, _flow_ref(init, seq, a.sq, max_norm))


@gpu
def test_step_without_row_list_is_a_zero_gradient_step():
    """A step in which the table gets no row list (only the dense parameter has a gradient) is a zero-gradient step
    for every row of the table: its coefficients enter the history, later catch-ups replay it."""
    steps, max_norm = 7, 1.0
    init, seq = _flow_data(22, steps, no_rows=(3, 4))
    f = _Flow(init)
    for s in seq[:2]:
        f.step(s, max_norm)
    with _Kernels() as k:                          # the step without rows still writes its coefficients
        f.step(seq[2], max_norm)
    assert k.names == {"sqnorm_partial_kernel", "sqnorm_final_kernel", "adam_kernel", "adam_rows_kernel"}, k.names
    for s in seq[3:]:
        f.step(s, max_norm)
    f.opt.flush()
    _check_flow("flow no-rows step", f, _flow_ref(init, seq, f.sq, max_norm))


def _tem_rowsparse():
    import argparse
    from prodsearch_b200 import synth
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    from prodsearch_b200.optimizers import build_optim
    cfg = argparse.Namespace(
        train_review_only=True, embedding_size=128, dropout=0.0, pretrain_emb_dir="", pretrain_up_emb_dir="",
        sep_prod_emb=False, model_name="item_transformer", ff_size=512, heads=8, inter_layers=1,
        query_encoder_name="fs", use_dot_prod=True, use_pos_emb=True, use_item_pos=False, sim_func="bias_product",
        pos_weight=False, neg_per_pos=5, optim="adam", lr=0.0005, max_grad_norm=5.0, beta1=0.9, beta2=0.999,
        decay_method="adam", warmup_steps=8000, l2_lambda=0.0, train_from="")
    torch.manual_seed(7)
    model = ItemTransformerRanker(cfg, "cuda", 5000, 3000, None, word_dists=synth.word_dists(5000),
                                  grad_mode="rowsparse")
    return model, build_optim(cfg, model), cfg


@gpu
@pytest.mark.parametrize("resume", [False, True], ids=["after_eager_steps", "after_resume"])
def test_graphed_step_after_eager_rowsparse_steps(resume):
    """Eager row-sparse TEM steps, then a GraphedTrainStep (optionally on a new optimizer loaded from the eager one's
    state_dict) for more steps: the parameters equal the all-eager run bit for bit."""
    import argparse
    from prodsearch_b200 import synth
    from prodsearch_b200.graph_step import GraphedTrainStep
    from prodsearch_b200.optimizers import Optimizer
    B, P, V, E, G = 96, 3000, 5000, 3, 4
    batches = [synth.tem_batch(B, P, V, seed=70 + i, Wq_max=9) for i in range(E + G)]
    widest = max(b.query_word_idxs.shape[1] for b, _, _ in batches)

    def padded(b):
        q = torch.full((B, widest), V - 1, dtype=torch.int64)
        q[:, :b.query_word_idxs.shape[1]] = b.query_word_idxs
        return argparse.Namespace(**{k: (v.cuda() if torch.is_tensor(v) else v)
                                     for k, v in dict(vars(b), query_word_idxs=q).items()})

    def run(graphed):
        model, optim, cfg = _tem_rowsparse()
        model.train()
        neg_i, neg_w = batches[0][1].cuda(), batches[0][2].cuda()
        model.injected_negatives = (neg_i, neg_w)
        losses, step = [], None
        for s, (b, ni, nw) in enumerate(batches):
            neg_i.copy_(ni)
            neg_w.copy_(nw)
            if s == E and resume:
                sd = optim.optimizer.state_dict()           # flushes
                if graphed:
                    optim = Optimizer("adam", cfg.lr, cfg.max_grad_norm, beta1=cfg.beta1, beta2=cfg.beta2)
                    optim._step = E
                    optim.set_parameters(list(model.named_parameters()))
                    optim.optimizer.load_state_dict(sd)
            if graphed and s == E:
                step = GraphedTrainStep(model, optim, padded(b), pad_values={"query_word_idxs": V - 1,
                                                                             "u_item_idxs": P})
            if step is not None:
                losses.append(float(step(padded(b))))
            else:
                loss = model(padded(b))
                model.zero_grad()
                loss.backward()
                optim.step()
                losses.append(float(loss.detach()))
                del loss
        optim.flush()
        return losses, [p.detach().clone() for p in model.parameters()]

    l_e, p_e = run(False)
    l_g, p_g = run(True)
    assert l_e == l_g, (l_e, l_g)
    for a, b in zip(p_e, p_g):
        assert torch.equal(a, b)
