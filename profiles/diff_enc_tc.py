"""Stage-by-stage comparison of the encoder forward's tensor-core path (the default, csrc/gemm3_tf32.cu) with the FFMA
kernels (PSB_ENC_TC=0): the same seeded TEM-layout call (batch 384, 21 positions, d 128, ff 512, 8 heads, 1 + 5 copies,
dropout 0.1 on a fixed Philox seed) runs once per path in its own subprocess (the knob is read once per process, and
a tcgen05 hand-off bug hangs), the whole saved-activation buffer is dumped, and every region of it (encoder_common.cuh
saved_layout) is compared with the FFMA path's: the first region that differs by more than fp32 noise names the stage
that is wrong -- qv / kv (projections), ctx, y, n (out-projection + LayerNorm), pre1, h1 (FFN up), z, out (FFN down + LN).
At this shape the backward takes the tensor-core tail, so the tensor-core forward leaves dropout_3 . gelu'(pre1) in the
pre1 slot (all the backward reads of it): that region is compared with the value formed in float64 from the FFMA path's
pre1 and h1 (h1 == 0 where dropout_3 dropped the element; elsewhere the multiplier is 1 / keep).

    timeout 300 python profiles/diff_enc_tc.py        # one JSON line per region"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S, T, D, FF, H, C = 384, 21, 128, 512, 8, 6
KEEP = 0.9                                         # 1 - p_drop
CHILD = r'''
import sys, numpy as np, torch
sys.path.insert(0, %r)
from prodsearch_b200 import ops
S, T, d, ff, heads, copies = %d, %d, %d, %d, %d, %d
g = torch.Generator().manual_seed(0)
shapes = dict(wq=(d, d), bq=(d,), wk=(d, d), bk=(d,), wv=(d, d), bv=(d,), wo=(d, d), bo=(d,), ln_attn_g=(d,), ln_attn_b=(d,),
              ln_ff_g=(d,), ln_ff_b=(d,), w1=(ff, d), b1=(ff,), w2=(d, ff), b2=(d,), ln_out_g=(d,), ln_out_b=(d,))
P = {}
for k, s in shapes.items():
    if len(s) == 2:
        P[k] = (torch.randn(s, generator=g) * (2.0 / (s[0] + s[1])) ** 0.5).cuda()
    elif k.endswith("_g"):
        P[k] = (1.0 + 0.3 * torch.randn(s, generator=g)).cuda()
    else:
        P[k] = (0.1 * torch.randn(s, generator=g)).cuda()
rows = 500
table = torch.randn(rows + 1, d, generator=g); table[rows] = 0
hist_len = torch.randint(0, T, (S,), generator=g)
idx = torch.randint(0, rows, (S, T - 1), generator=g)
idx[torch.arange(T - 1)[None, :] >= hist_len[:, None]] = rows
first = torch.randn(S, d, generator=g)
pos = torch.arange(64)[:, None].float(); div = torch.exp(torch.arange(0, d, 2).float() * -(np.log(10000.0) / d))
pe = torch.zeros(64, d); pe[:, 0::2] = torch.sin(pos * div); pe[:, 1::2] = torch.cos(pos * div)
seed_t = torch.tensor([0x1234ABCD5678], dtype=torch.int64, device="cuda")
out, call = ops.encoder_fwd(P, heads, first=first.cuda(), table=table.cuda(), idx=idx.cuda(), pad_idx=rows, copies=copies,
                            out_pos=0, pre_ln=False, p_drop=0.1, seed=seed_t, raw_input=False, pe=pe.cuda())
torch.cuda.synchronize()
np.savez(sys.argv[1], saved=call.saved.cpu().numpy().view(np.float32), out=out.cpu().numpy())
''' % (ROOT, S, T, D, FF, H, C)


def layout():
    """encoder_common.cuh saved_layout, in floats."""
    a4 = lambda x: (x + 3) & ~3
    sc = S * C
    sizes = [("nact", a4(S)), ("off", a4(S + 1)), ("tok", a4(S * T)), ("xo", S * D), ("xno", S * D), ("qv", S * D),
             ("xn", S * T * D), ("kv", S * T * 2 * D), ("p", a4(S * T * H)), ("ctx", sc * D), ("y", sc * D), ("n", sc * D),
             ("z", sc * D), ("pre1", sc * FF), ("h1", sc * FF), ("wot_hl", 2 * D * D), ("w1t_hl", 2 * D * FF), ("w2t_hl", 2 * FF * D), ("wkv_t", 2 * D * D)]
    out, p = {}, 0
    for name, n in sizes:
        out[name] = (p, n)
        p += n
    return out


def gelu_tanh_grad(x):
    """d/dx of the tanh-form gelu the kernels use (encoder_common.cuh gelu_tanh_grad), float64."""
    c = np.sqrt(2.0 / np.pi)
    t = np.tanh(c * (x + 0.044715 * x ** 3))
    return 0.5 * (1.0 + t) + 0.5 * x * (1.0 - t * t) * c * (1.0 + 3.0 * 0.044715 * x * x)


def run(path_name, path):
    """path_name "ffma": PSB_ENC_TC=0; "tc": the default tensor-core path."""
    env = {k: v for k, v in os.environ.items() if k != "PSB_ENC_TC"}
    if path_name == "ffma":
        env["PSB_ENC_TC"] = "0"
    try:
        r = subprocess.run([sys.executable, "-c", CHILD, path], env=env, capture_output=True, text=True, timeout=120)
    except subprocess.TimeoutExpired:
        print(json.dumps({"path": path_name, "error": "timeout (hang?)"}))
        return None
    if r.returncode != 0:
        print(json.dumps({"path": path_name, "error": r.stderr[-600:]}))
        return None
    return np.load(path)


if __name__ == "__main__":
    tmp = tempfile.mkdtemp()
    base = run("ffma", os.path.join(tmp, "ffma.npz"))
    ok = base is not None
    L = layout()
    got = run("tc", os.path.join(tmp, "tc.npz")) if ok else None
    if got is None:
        ok = False
    else:
        n_act = int(base["saved"].view(np.int32)[L["off"][0] + S])        # active tokens: compact rows beyond hold garbage
        for name, (p, n) in L.items():
            a, b = base["saved"][p:p + n], got["saved"][p:p + n]
            if name.endswith("_hl") or name == "wkv_t":    # operands only the tensor-core backward reads
                continue
            if name in ("nact", "off", "tok"):
                same = bool(np.array_equal(a.view(np.int32), b.view(np.int32)))
                print(json.dumps({"path": "tc", "region": name, "identical": same}))
                ok = ok and same
                continue
            if name in ("xn", "kv", "p"):                                  # compact token rows: only the active ones
                w = {"xn": D, "kv": 2 * D, "p": H}[name]
                a, b = a[:n_act * w], b[:n_act * w]
            if name == "pre1":                                             # dropout_3 . gelu'(pre1), see the docstring
                p1, n1 = L["h1"]
                h1 = base["saved"][p1:p1 + n1]
                a = np.where(h1 == 0, 0.0, gelu_tanh_grad(a.astype(np.float64)) / KEEP)
            err = float(np.abs(a.astype(np.float64) - b).max() / max(np.abs(a).max(), 1e-30))
            good = err < 2e-5 and bool(np.isfinite(b).all())
            ok = ok and good
            print(json.dumps({"path": "tc", "region": name, "max_abs_diff_over_max": err, "ok": good}))
        err = float(np.abs(base["out"].astype(np.float64) - got["out"]).max() / np.abs(base["out"]).max())
        print(json.dumps({"path": "tc", "region": "out", "max_abs_diff_over_max": err, "ok": err < 2e-5}))
        ok = ok and err < 2e-5
    print("VERDICT:", "the tensor-core encoder's saved activations agree with the FFMA kernels stage by stage" if ok else "MISMATCH or failure (see the first bad region)")
    sys.exit(0 if ok else 1)
