"""G5 fp16 shortlist: time the main-pass kernel (csrc/catalog_tc.cu tc16_score_v2_kernel) end to end and per kernel, in a
subprocess under a hard timeout (a hand-off bug in a tcgen05 pipeline shows up as a hang, not as a wrong answer).  Run
on ONE GPU:

    timeout 900 python profiles/check_tc16_v2.py            # one JSON line per (N, M): ms, per-kernel us, a hash of the lists
    timeout 900 python profiles/check_tc16_v2.py --quick    # 1M items, M = 384 and 4096 only
    timeout 200 python profiles/check_tc16_v2.py --tmem     # TMEM read bytes / clock / SM (psb_debug_tmem_read_bw)

The hash ("sha") of the ids and scores lets two builds be compared by hand: same seed, same data.  Earlier results:
profiles/r01Z_tc16_v*_stats.jsonl, profiles/r02a_tc16_variants.jsonl."""
import json
import subprocess
import sys
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = r'''
import hashlib, json, os, sys, torch
sys.path.insert(0, %r)
from prodsearch_b200 import _lib, ops
n, d = int(sys.argv[1]), 128
torch.manual_seed(0)
table = torch.empty(n + 1, d, device="cuda").normal_()
prep = ops.catalog_prepare_f16(table, n)
for m in ((384, 4096) if sys.argv[2] == "1" else (24, 128, 384, 1024, 4096)):
    q = torch.randn(m, d, device="cuda")
    f = lambda: ops.catalog_topk(q, table, 100, n_items=n, mode=_lib.TOPK_TC16, prepared=prep)
    ids, sc = f()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5): f()
    b.record(); torch.cuda.synchronize()
    _lib.profile_enable(True)
    for _ in range(3): f()
    split = {k_: round(v[1] / 3 * 1e3, 1) for k_, v in _lib.profile_dump().items()}
    _lib.profile_enable(False)
    h = hashlib.sha256(ids.cpu().numpy().tobytes() + sc.cpu().numpy().tobytes()).hexdigest()[:16]
    print(json.dumps({"n_items": n, "m": m, "ms": round(a.elapsed_time(b) / 5, 4), "kernel_us": split,
                      "tflops": round(2.0 * m * n * d / (a.elapsed_time(b) / 5) / 1e9, 1), "sha": h}), flush=True)
''' % ROOT

TMEM_CHILD = r'''
import ctypes, json, sys
sys.path.insert(0, %r)
import torch
from prodsearch_b200 import _lib
torch.zeros(1, device="cuda")
out = (ctypes.c_double * 2)()
for warps in (4, 8, 12, 16):
    _lib.check(_lib.load().psb_debug_tmem_read_bw(warps, 20000, out), "psb_debug_tmem_read_bw")
    print(json.dumps({"tmem_read": "tcgen05.ld.32x32b.x32 + wait::ld", "warps": warps, "bytes_per_clk_one_cta": round(out[0], 1),
                      "bytes_per_clk_all_sms": round(out[1], 1), "needed_for_f16_peak_at_K128": 128.0}))
''' % ROOT


if __name__ == "__main__":
    if "--tmem" in sys.argv:
        r = subprocess.run([sys.executable, "-c", TMEM_CHILD], capture_output=True, text=True, timeout=120)
        print(r.stdout.strip() or r.stderr[-600:])
        sys.exit(r.returncode)
    quick = "--quick" in sys.argv
    ok = True
    for n in ((1_000_000,) if quick else (1_000_000, 250_000)):
        try:
            r = subprocess.run([sys.executable, "-c", CHILD, str(n), "1" if quick else "0"], capture_output=True, text=True,
                               timeout=25 if quick else 240)
        except subprocess.TimeoutExpired as ex:
            print(json.dumps({"n_items": n, "error": "timeout (hang?)",
                              "partial": (ex.stdout or b"")[-400:].decode("utf8", "replace")}))
            ok = False
            continue
        print(r.stdout.strip() if r.returncode == 0 else json.dumps({"n_items": n, "error": r.stderr[-600:]}))
        ok = ok and r.returncode == 0
    sys.exit(0 if ok else 1)
