"""GPU: float64 reference for the fused single-position encoder (psb_encoder_fwd / _bwd) at every tile choice of its
kernels.

The reference is the contract of include/psb.h (one encoder layer, then the final LayerNorm, at out_pos, for S * copies
copy rows) computed by oracle.encoder_layer in float64: every input, parameter, positional row and dropout multiplier
(exactly 0 or the kernels' fp32 1 / (1 - p)) is the fp32 value the kernels read, cast to double, so only the arithmetic
differs.  Gradients come from float64 autograd against a fixed fp32 upstream gradient.

Bar, calibrated per case: for each tensor X (the output, the data gradient, each weight gradient),
e_k = max|kernel - ref64| / max|ref64| must stay within max(8 e_32, 2e-6), where e_32 is the same measure for the fp32
CPU oracle on the same inputs.  A dropped 3xTF32 correction term or a misread tile edge lands at 1e-4 or worse; rounding
does not.  The key bias gradient is exactly 0 (softmax is shift-invariant), so it is bounded in absolute terms by
1e-5 max|grad bq| instead.  pytest -s prints e_k and e_32 of every case's worst tensor.

Cases are built from the host-side tiling choice, replayed below (dims_from_cfg in csrc/encoder_fwd.cu,
tail_bwd_smem_floats in csrc/encoder_bwd.cu, attn_bwd_spt and tail_bwd_fused_for in csrc/encoder_common.cuh): each id
names the route it reaches, the replay asserts it, and the library's profiler labels confirm which tail kernels ran.
"""
import ctypes
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:                     # also run as a script (the PSB_ENC_TC=0 subprocess below)
    sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from oracle.philox import encoder_dropout_muls  # noqa: E402
from test_gpu_encoder import make_params, run_oracle  # noqa: E402

RATIOS = {}                         # case id -> (worst e_k / bar, its tensor, worst e_k / e_32, its tensor)

# ------------------------------------------------------------------------------------------------ tiling replay
NUM_SMS = 148
SMEM_CAP = 227 * 1024


def _red_floats(R, J):
    cg = (J + 127) // 128
    cg = 1 if cg <= 1 else 2 if cg <= 2 else 4 if cg <= 4 else 8
    return (8 // cg) * R * (J + 4)


def _tail_bwd_smem_floats(R, d, F, H, T, spt):
    return (R * max(d, F) + max(_red_floats(R, d), _red_floats(R, F)) + 2 * R * (d + 4) + 2 * R * H * T +
            2 * spt * H * T)


def _attn_bwd_smem_floats(R, d, H, T, spt):
    return 2 * R * (d + 4) + 2 * R * H * T + 2 * spt * H * T + 2 * spt * T * (d + 4)


def tiling(S, T, d, F, H, C, tc=True):
    """The encoder's route for these dimensions: dict(R, spt, attn_spt, fused) or None (PSB_E_UNSUPPORTED).  R is the
    tile rows of the FFMA tail kernels, spt the sequences per tile (R / C unless no R fits at that), attn_spt the
    sequences per CTA of tail_attn_bwd_kernel, fused whether both tails run on tcgen05."""
    def fits(R, spt):
        return _tail_bwd_smem_floats(R, d, F, H, T, spt) * 4 <= SMEM_CAP

    best = None
    for lowered in (False, True):
        for R in (16, 20, 24):
            spt = R // C
            while lowered and spt > 0 and not fits(R, spt):
                spt -= 1
            if spt == 0 or not fits(R, spt):
                continue
            tiles = -(-S // spt)
            cost = -(-tiles // NUM_SMS) * (R + 10)
            if best is None or cost < best[2]:
                best = (R, spt, cost)
        if best is not None:
            break
    if best is None:
        return None
    R, spt = best[0], best[1]
    attn_spt = spt
    while attn_spt > 0 and _attn_bwd_smem_floats(attn_spt * C, d, H, T, attn_spt) * 4 > SMEM_CAP:
        attn_spt -= 1
    fused = tc and d == 128 and F == 512 and attn_spt > 0
    return dict(R=R, spt=spt, attn_spt=attn_spt, fused=fused)


# ------------------------------------------------------------------------------------------------ cases
# (id, S, T, d, ff, heads, copies, options); the id names the route: tail rows R, sequences per tile, sequences per CTA
# of the attention backward, copy rows S * copies around the 128-row tiles of the tcgen05 kernels, heads, T.
CASES = [
    # FFMA tails (d != 128 or ff != 512); every other test of these kernels picks R = 16
    ("ffma-R20", 600, 21, 64, 256, 8, 6, dict(p=0.1)),
    ("ffma-R24", 3000, 5, 64, 64, 8, 1, dict()),
    ("ffma-R24-C24-spt1-T64", 5, 64, 64, 64, 8, 24, dict(tem=False, out_pos=-1, p=0.1)),
    ("ffma-R16-spt6-T64", 40, 64, 64, 1024, 8, 1, dict(tem=False, full_mask_row=True)),
    # tensor-core tails
    ("tc-R24-attnspt4", 500, 21, 128, 512, 8, 6, dict(p=0.1)),
    ("tc-C24-spt1", 7, 21, 128, 512, 8, 24, dict(p=0.1)),
    ("tc-T33-attnspt5", 40, 33, 128, 512, 8, 1, dict(tem=False, out_pos=-1)),
    ("tc-T51-attnspt3-rows256", 256, 51, 128, 512, 8, 1, dict()),
    ("tc-T64-C6", 30, 64, 128, 512, 8, 6, dict(p=0.1)),
    ("tc-T64-C1-spt12", 40, 64, 128, 512, 8, 1, dict(tem=False, out_pos=-1, full_mask_row=True)),
    ("tc-rows128", 128, 21, 128, 512, 8, 1, dict()),
    ("tc-rows129", 129, 13, 128, 512, 8, 1, dict(tem=False, out_pos=-1, full_mask_row=True)),
    ("tc-rows132", 22, 21, 128, 512, 8, 6, dict(p=0.1)),
    ("tc-rows258", 43, 21, 128, 512, 8, 6, dict(tem=False, p=0.1)),
    ("tc-H1-T32", 37, 32, 128, 512, 1, 1, dict(tem=False)),
    ("tc-H2", 37, 21, 128, 512, 2, 6, dict()),
    ("tc-H16", 29, 21, 128, 512, 16, 2, dict(tem=False, out_pos=-1, p=0.1)),
    ("tc-H32-spt5", 29, 21, 128, 512, 32, 1, dict()),
    ("tc-preln-raw-rows130", 65, 10, 128, 512, 8, 2, dict(tem=False, pre_ln=True, raw=True, p=0.1)),
]
# The R = 20 / R = 24 shapes and the lowered-spt shape at the default size, on the FFMA kernels (PSB_ENC_TC=0)
FFMA_DEFAULT_CASES = [
    ("ffma-d128-R20", 600, 21, 128, 512, 8, 6, dict(p=0.1)),
    ("ffma-d128-R24", 3000, 5, 128, 512, 8, 1, dict()),
    ("ffma-d128-R16-spt12-T64", 40, 64, 128, 512, 8, 1, dict(tem=False, out_pos=-1, full_mask_row=True)),
]


def _route_of_id(cid, t):
    """The route a case id names must be the one the replay picks."""
    for part in cid.split("-"):
        if part[0] == "R" and part[1:].isdigit():
            assert t["R"] == int(part[1:]), (cid, t)
        elif part.startswith("attnspt"):
            assert t["attn_spt"] == int(part[7:]), (cid, t)
        elif part.startswith("spt"):
            assert t["spt"] == int(part[3:]), (cid, t)
    assert t["fused"] == cid.startswith("tc-"), (cid, t)


# ------------------------------------------------------------------------------------------------ one case
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


def _rel(a, ref):
    a, ref = a.detach().cpu().double(), ref.detach().cpu().double()
    return float((a - ref).abs().max()) / max(float(ref.abs().max()), 1e-300)


def _inputs(S, T, d, ff, heads, copies, tem, full_mask_row, seed):
    """fp32 inputs as tests/test_gpu_encoder.py run_case draws them: TEM (first, table, idx) or dense (x, mask)."""
    g = torch.Generator().manual_seed(seed)
    P = make_params(d, ff, seed + 1)
    rows = 500
    table = torch.randn(rows + 1, d, generator=g)
    table[rows] = 0
    hist_len = torch.randint(0, T, (S,), generator=g)
    idx = torch.randint(0, rows, (S, T - 1), generator=g)
    idx[torch.arange(T - 1)[None, :] >= hist_len[:, None]] = rows
    first = torch.randn(S, d, generator=g)
    valid = torch.cat([torch.ones(S, 1, dtype=torch.bool), idx.ne(rows)], 1)
    x = torch.cat([first.unsqueeze(1), table[idx]], 1)
    if not tem:
        valid = torch.rand(S, T, generator=g) > 0.4
        valid[:, 0] |= torch.rand(S, generator=g) > 0.3
        if full_mask_row:
            valid[1] = False
        x = torch.randn(S, T, d, generator=g)
    gout = torch.randn(S * copies, d, generator=g)
    return P, table, idx, first, x, valid, gout, rows


def run_case(cid, S, T, d, ff, heads, copies, p=0.0, tem=True, out_pos=0, pre_ln=False, raw=False,
             full_mask_row=False, seed=11):
    from prodsearch_b200 import ops
    t = tiling(S, T, d, ff, heads, copies, tc=os.environ.get("PSB_ENC_TC") != "0")
    assert t is not None, cid
    _route_of_id(cid, t)
    P, table, idx, first, x, valid, gout, rows = _inputs(S, T, d, ff, heads, copies, tem, full_mask_row, seed)
    pe = oracle.sinusoid_table(64, d)[0] if not raw else None
    o = out_pos % T
    seed_val = 0x5EED0000 + seed
    muls = encoder_dropout_muls(seed_val, p, S, copies, T, heads, d, ff, o) if p > 0 else None

    # kernel: two calls, bit-identical
    dev = {k: v.cuda() for k, v in P.items()}
    shapes = {k: tuple(v.shape) for k, v in P.items() if pre_ln or not k.startswith("ln_attn")}
    seed_t = torch.tensor([seed_val], dtype=torch.int64, device="cuda") if p > 0 else None
    kw = dict(copies=copies, out_pos=out_pos, pre_ln=pre_ln, p_drop=p, seed=seed_t, raw_input=raw,
              pe=pe.cuda() if pe is not None else None)
    if tem:
        src = dict(first=first.cuda(), table=table.cuda(), idx=idx.cuda(), pad_idx=rows)
    else:
        src = dict(dense=x.cuda(), mask=valid.cuda())
    runs = []
    for i in range(2):
        with _Kernels() as kn:
            out, call = ops.encoder_fwd(dev, heads, **src, **kw)
            g_first, g_rest, g_dense, grads, _ = ops.encoder_bwd(call, gout.cuda(), shapes)
            torch.cuda.synchronize()
        data = dict(g_first=g_first, g_rest=g_rest) if tem else dict(g_dense=g_dense)
        runs.append(dict(out=out, **data, **{"grad " + k: v for k, v in grads.items()}))
        if i == 0:
            fused = {"tail_fused_tc_kernel", "tail_bwd_fused_tc_kernel", "tail_attn_bwd_kernel"}
            ffma = {"tail_fwd_kernel", "tail_bwd_kernel"}
            want, avoid = (fused, ffma) if t["fused"] else (ffma, fused)
            assert want <= kn.names and not (avoid & kn.names), (cid, sorted(kn.names))
    for k in runs[0]:
        assert torch.equal(runs[0][k], runs[1][k]), "%s: %s differs between two calls" % (cid, k)
    got = runs[0]

    # references: the same fp32 values through the oracle in float64 and in float32
    refs = []
    for dt in (torch.float64, torch.float32):
        Pd = {k: v.to(dt) for k, v in P.items()}
        ref, leaves, xin = run_oracle(Pd, x.to(dt), valid, heads, out_pos, copies, pre_ln, raw,
                                      pe.to(dt) if pe is not None else None, muls)
        (ref * gout.to(dt)).sum().backward()
        gx = xin.grad
        r = dict(out=ref)
        if tem:
            r.update(g_first=gx[:, 0], g_rest=gx[:, 1:] * valid[:, 1:, None].to(dt))
        else:
            r["g_dense"] = gx
        r.update({"grad " + k: leaves[k].grad for k in shapes})
        refs.append(r)
    r64, r32 = refs

    worst_bar, worst_32 = (0.0, ""), (0.0, "")
    for k, ref in r64.items():
        assert bool(torch.isfinite(got[k]).all()), "%s: %s not finite" % (cid, k)
        if k == "grad bk":
            err = float((got[k].cpu().double() - ref).abs().max())
            bound = 1e-5 * float(r64["grad bq"].abs().max())
            assert err <= bound, "%s: grad bk max err %g > %g" % (cid, err, bound)
            continue
        e_k, e_32 = _rel(got[k], ref), _rel(r32[k], ref)
        bar = max(8 * e_32, 2e-6)
        print("  %-26s %-14s e_k %.3g  e_32 %.3g" % (cid, k, e_k, e_32))
        worst_bar, worst_32 = max(worst_bar, (e_k / bar, k)), max(worst_32, (e_k / e_32 if e_32 > 0 else float("inf"), k))
        assert e_k <= bar, "%s: %s e_k %.3g > max(8 e_32, 2e-6) (e_32 %.3g)" % (cid, k, e_k, e_32)
    RATIOS[cid] = worst_bar + worst_32
    print("%-26s worst e_k / bar %.3g (%s), worst e_k / e_32 %.3g (%s)" % ((cid,) + RATIOS[cid]))


# ------------------------------------------------------------------------------------------------ tests
@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    if RATIOS:
        print("\nworst e_k / max(8 e_32, 2e-6) and worst e_k / e_32 per case:")
        for cid in sorted(RATIOS):
            print("  %-26s %.3g (%s)  %.3g (%s)" % ((cid,) + RATIOS[cid]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_encoder_vs_fp64_reference(case):
    cid, S, T, d, ff, heads, copies, opt = case
    run_case(cid, S, T, d, ff, heads, copies, **opt)


@pytest.mark.gpu
def test_encoder_ffma_kernels_at_default_size_vs_fp64_reference():
    """PSB_ENC_TC is read once per process: the FFMA kernels at d = 128, ff = 512 run in a subprocess of their own."""
    env = dict(os.environ, PSB_ENC_TC="0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "test_gpu_encoder_fp64.py")], env=env,
                       capture_output=True, text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count(" worst e_k / bar ") == len(FFMA_DEFAULT_CASES), r.stdout


@pytest.mark.gpu
def test_encoder_rejects_what_its_backward_tail_cannot_hold():
    """copies 21..24 at d = 128, ff = 512, 8 heads: T <= 35 (include/psb.h).  No R >= copies holds the scores."""
    from prodsearch_b200 import ops
    assert tiling(3, 35, 128, 512, 8, 24) is not None and tiling(3, 36, 128, 512, 8, 24) is None
    P = {k: v.cuda() for k, v in make_params(128, 512, 0).items()}
    ops.encoder_fwd(P, 8, dense=torch.randn(3, 35, 128, device="cuda"), copies=24)
    with pytest.raises(RuntimeError, match="status -5"):
        ops.encoder_fwd(P, 8, dense=torch.randn(3, 36, 128, device="cuda"), copies=24)


def test_tiling_replay_matches_the_host_code():
    """CPU: the replay above accepts exactly the shapes the library's host code accepts (psb_encoder_saved_bytes runs
    dims_from_cfg and touches no device); every rejection is PSB_E_UNSUPPORTED."""
    from prodsearch_b200 import _lib
    lib = _lib.load()
    for d, ff in ((128, 512), (64, 1024), (64, 64)):
        for heads in (1, 8, 16, 32):
            for copies in (1, 6, 16, 17, 21, 24):
                for T in (1, 21, 26, 27, 35, 36, 52, 53, 56, 57, 64):
                    cfg = _lib.EncoderCfg(40, T, d, heads, ff, copies, 0, 0, 0, 1e-6, 0.0, None, None, None, 0, None,
                                          -1, ctypes.c_void_p(256), None, None, None, None)
                    st = lib.psb_encoder_saved_bytes(ctypes.byref(cfg))
                    accepted = tiling(40, T, d, ff, heads, copies) is not None
                    assert (st > 0) == accepted and (accepted or st == -5), (d, ff, heads, copies, T, st)


if __name__ == "__main__":
    # test_encoder_ffma_kernels_at_default_size_vs_fp64_reference runs this with PSB_ENC_TC=0
    for c in FFMA_DEFAULT_CASES:
        run_case(c[0], *c[1:7], **c[7])
