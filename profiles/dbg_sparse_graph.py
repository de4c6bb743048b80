"""Debug aid: row-sparse training, eager vs CUDA-graph replays, step by step (which rows / moments diverge first)."""
import argparse, os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_gpu_sparse_adam import _tem, _cuda
from prodsearch_b200 import synth, _lib
from prodsearch_b200.graph_step import GraphedTrainStep
from prodsearch_b200.optimizers import Optimizer
mode = sys.argv[1] if len(sys.argv) > 1 else "default"
a, b = _tem("rowsparse"), _tem("rowsparse")
b.load_state_dict(a.state_dict())
oa, ob = Optimizer("adam", 5e-3, 5.0), Optimizer("adam", 5e-3, 5.0)
oa.set_parameters(list(a.named_parameters())); ob.set_parameters(list(b.named_parameters()))
a.train(); b.train()
P, V, B = 9000, 6000, 96
batches = [synth.tem_batch(B, P, V, seed=40 + s) for s in range(4)]
Wq = max(x[0].query_word_idxs.shape[1] for x in batches)
def padded(x):
    q = torch.full((B, Wq), V - 1, dtype=torch.int64); q[:, :x.query_word_idxs.shape[1]] = x.query_word_idxs
    return argparse.Namespace(**dict(vars(x), query_word_idxs=q))
neg_i = torch.empty(B, 5, dtype=torch.int64, device="cuda"); neg_w = torch.empty(B * 5, dtype=torch.int64, device="cuda")
a.injected_negatives = b.injected_negatives = (neg_i, neg_w)
step_fn = None
for s, (x, ni, nw) in enumerate(batches):
    neg_i.copy_(ni); neg_w.copy_(nw)
    cb = _cuda(padded(x))
    la = a(cb); a.zero_grad(); la.backward(); oa.step(); la = float(la.detach())
    if "eagerb" in mode:
        lb = b(cb); b.zero_grad(); lb.backward(); ob.step(); lb = float(lb.detach())
    else:
        if step_fn is None:
            step_fn = GraphedTrainStep(b, ob, cb)
        lb = float(step_fn(cb))
    torch.cuda.synchronize()
    out = {"mode": mode, "step": s, "loss_a": la, "loss_b": lb}
    sa, sb = oa.optimizer, ob.optimizer
    for name, pa, pb in (("item", a.product_emb.weight, b.product_emb.weight), ("word", a.word_embeddings.weight, b.word_embeddings.weight)):
        sta, stb = sa.state[pa], sb.state[pb]
        dp = (pa.detach() - pb.detach()).abs().max(dim=1).values
        dm = (sta["exp_avg"] - stb["exp_avg"]).abs().max(dim=1).values
        dv = (sta["exp_avg_sq"] - stb["exp_avg_sq"]).abs().max(dim=1).values
        bad = torch.nonzero(dp > 1e-6).flatten()
        out[name] = {"rows_p_differ": int(bad.numel()), "max_dp": float(dp.max()), "max_dm": float(dm.max()), "max_dv": float(dv.max()),
                     "first_rows": bad[:6].tolist(), "last_a": sta["last_step"][bad[:6]].tolist(), "last_b": stb["last_step"][bad[:6]].tolist(),
                     "last_equal": bool(torch.equal(sta["last_step"], stb["last_step"]))}
    print(out, flush=True)
