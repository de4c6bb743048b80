"""Backward of the encoder on the tensor-core path (the default, csrc/gemm3_tf32.cu tail_bwd_fused_tc_kernel) against
the FFMA kernels (PSB_ENC_TC=0): the same seeded TEM-layout call (batch 384, 21 positions, d 128, ff 512, 8 heads, 1 + 5
copies, dropout 0.1 on a fixed Philox seed) and the same upstream gradient run once per path in their own subprocesses;
every gradient the backward returns (grad_first, grad_rest, all 18 parameter gradients) and the backward workspace's
intermediate regions (g_h2, g_pre, g_o1, gxo, g_qlin, gkv) are compared, largest difference over the tensor's maximum.

    timeout 300 python profiles/diff_enc_bwd_tc.py       # one JSON line per tensor"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S, T, D, FF, H, C = 384, 21, 128, 512, 8, 6
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
gout = torch.randn(S * copies, d, generator=g).cuda()
seed_t = torch.tensor([0x1234ABCD5678], dtype=torch.int64, device="cuda")
out, call = ops.encoder_fwd(P, heads, first=first.cuda(), table=table.cuda(), idx=idx.cuda(), pad_idx=rows, copies=copies,
                            out_pos=0, pre_ln=False, p_drop=0.1, seed=seed_t, raw_input=False)
g_first, g_rest, _, grads, ws = ops.encoder_bwd(call, gout, {k: v.shape for k, v in P.items() if not k.startswith("ln_attn")})
torch.cuda.synchronize()
res = {"g_first": g_first, "g_rest": g_rest}
res.update({"d_" + k: v for k, v in grads.items()})
sc = S * copies
off, wsf = 2 * d * d, ws.view(torch.float32)
for name, n in (("g_h2", sc * d), ("g_pre", sc * ff), ("g_o1", sc * d), ("gxo", S * d), ("g_qlin", S * d)):
    res["ws_" + name] = wsf[off:off + n]
    off += n
np.savez(sys.argv[1], **{k: v.detach().cpu().numpy() for k, v in res.items()})
''' % (ROOT, S, T, D, FF, H, C)


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
        print(json.dumps({"path": path_name, "error": r.stderr[-800:]}))
        return None
    return np.load(path)


if __name__ == "__main__":
    tmp = tempfile.mkdtemp()
    base = run("ffma", os.path.join(tmp, "ffma.npz"))
    got = run("tc", os.path.join(tmp, "tc.npz")) if base is not None else None
    ok = got is not None
    if ok:
        for name in base.files:
            a, b = base[name].astype(np.float64), got[name].astype(np.float64)
            # d_bk is zero in exact arithmetic (a key bias shifts every score of a softmax row alike): measured against d_bv
            scale = np.abs(base["d_bv"]).max() if name == "d_bk" else np.abs(a).max()
            err = float(np.abs(a - b).max() / max(scale, 1e-30))
            good = err < 3e-5 and bool(np.isfinite(b).all())
            ok = ok and good
            print(json.dumps({"path": "tc", "tensor": name, "max_abs_diff_over_max": err, "ok": good}))
    print("VERDICT:", "tensor-core backward agrees with the FFMA kernels" if ok else "MISMATCH or failure")
    sys.exit(0 if ok else 1)
