"""Timeline of the fused tensor-core encoder tail (the default path, PSB_FT_TRACE=1): %globaltimer stamps of CTA 0 at its
phase boundaries, relative to the kernel's first instruction, for a few launches of the TEM-shaped forward call.

    PSB_FT_TRACE=1 timeout 200 python profiles/tail_trace.py"""
import ctypes
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from prodsearch_b200 import _lib, ops  # noqa: E402

S, T, d, ff, heads, copies = 384, 21, 128, 512, 8, 6
g = torch.Generator().manual_seed(0)
shapes = dict(wq=(d, d), bq=(d,), wk=(d, d), bk=(d,), wv=(d, d), bv=(d,), wo=(d, d), bo=(d,), ln_attn_g=(d,), ln_attn_b=(d,),
              ln_ff_g=(d,), ln_ff_b=(d,), w1=(ff, d), b1=(ff,), w2=(d, ff), b2=(d,), ln_out_g=(d,), ln_out_b=(d,))
P = {k: (torch.randn(s, generator=g) * 0.05 + (1.0 if k.endswith("_g") else 0.0)).cuda() for k, s in shapes.items()}
rows = 500
table = torch.randn(rows + 1, d, generator=g)
table[rows] = 0
hist_len = torch.randint(0, T, (S,), generator=g)
idx = torch.randint(0, rows, (S, T - 1), generator=g)
idx[torch.arange(T - 1)[None, :] >= hist_len[:, None]] = rows
first = torch.randn(S, d, generator=g).cuda()
seed_t = torch.tensor([0x1234ABCD5678], dtype=torch.int64, device="cuda")
table, idx = table.cuda(), idx.cuda()
NAMES = {0: "start", 1: "setup done", 2: "ctx tile landed", 3: "mma: A0 ready", 4: "mma: first chunk split (p0)", 5: "mma: p0 issued",
         6: "epi: acc0 full", 7: "mma: A1 ready", 8: "mma: first chunk split (p1)", 9: "mma: p1 issued", 10: "epi: acc1 full",
         11: "mma: A2 ready", 12: "mma: first chunk split (p2)", 13: "mma: p2 issued", 14: "epi: acc2 full",
         15: "cluster sync 1 passed", 16: "final rows stored", 17: "cluster sync 2 passed"}
lib = _lib.load()
BNAMES = {0: "start", 1: "prologue done (tile 0 written)", 2: "epi1: operands ready", 3: "epi1: acc0 full", 4: "epi1: tile 1 written",
          5: "epi1: g_pre stored", 6: "epi2: acc1 full", 7: "epi2: partial tile written", 8: "cluster sync 1 passed",
          9: "final rows done (tile 2 written)", 10: "ln partials reduced", 11: "epi3: acc2 full", 12: "g_ctx stored",
          13: "cluster sync 2 passed"}
gout = torch.randn(S * copies, d, generator=g).cuda()
for it in range(4):
    out, call = ops.encoder_fwd(P, heads, first=first, table=table, idx=idx, pad_idx=rows, copies=copies, out_pos=0,
                                pre_ln=False, p_drop=0.1, seed=seed_t, raw_input=False)
    bw = ops.encoder_bwd(call, gout, {k: v.shape for k, v in P.items() if not k.startswith("ln_attn")})
    torch.cuda.synchronize()
    buf = (ctypes.c_uint64 * 64)()
    if lib.psb_debug_tail_trace(buf) != 0:          # tracing off (e.g. under ncu): the launches are all this run is for
        continue
    t = np.array(list(buf), dtype=np.int64)
    rel = {NAMES[i]: round(float(t[i] - t[0]) / 1000.0, 2) for i in sorted(NAMES) if t[i] != 0}
    print(json.dumps({"launch": it, "us_since_start": rel}))
    if t[48] != 0:
        AN = {0: "start", 1: "loads + dropout multipliers staged", 2: "gxo + gA done", 3: "softmax backward done", 4: "gK | gV stored", 5: "gq stored"}
        print(json.dumps({"launch": it, "attn_backward_us_since_start":
                          {AN[i]: round(float(t[48 + i] - t[48]) / 1000.0, 2) for i in sorted(AN) if t[48 + i] != 0}}))
    if t[32] != 0:
        print(json.dumps({"launch": it, "backward_us_since_start":
                          {BNAMES[i]: round(float(t[32 + i] - t[32]) / 1000.0, 2) for i in sorted(BNAMES) if t[32 + i] != 0}}))
