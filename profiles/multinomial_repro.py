"""Run-to-run reproducibility of the TEM step's negative draws on one GPU.  The same generator state is drawn from T
times -- with a matrix product running on another stream, as the encoder runs next to the draws inside the step -- and
the number of distinct results is counted: the float32 CDF scan inside torch.multinomial (torch.cumsum of the
normalised word distribution), the literal item / word draws of a batch-384 step, and the same draws with
ItemTransformerRanker.reproducible_draws.  One JSON line.

    python profiles/multinomial_repro.py [T]"""
import hashlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from prodsearch_b200 import synth  # noqa: E402
from prodsearch_b200.item_transformer import ItemTransformerRanker  # noqa: E402

T = int(sys.argv[1]) if len(sys.argv) > 1 else 200
P, V, B, K = bench.WORKLOAD["product_size"], bench.WORKLOAD["vocab_size"], bench.WORKLOAD["batch_per_gpu"], 5
model = ItemTransformerRanker(bench.model_args(0.1), "cuda", V, P, None, word_dists=synth.word_dists(V))
busy = torch.randn(4096, 4096, device="cuda")
side = torch.cuda.Stream()


def distinct(fn):
    seen = set()
    for _ in range(T):
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            busy @ busy
        torch.manual_seed(1234)
        seen.add(hashlib.sha1(fn().cpu().numpy().tobytes()).hexdigest())
        torch.cuda.synchronize()
    return len(seen)


def draws(reproducible):
    model.reproducible_draws = reproducible
    items, words = model._draw_negatives(B, 1, K)
    return torch.cat([items.reshape(-1), words.reshape(-1)])


norm = model.word_dists / model.word_dists.sum()
out = {"trials": T, "distinct_results": {
    "cumsum_word_dists_f32": distinct(lambda: torch.cumsum(norm, 0)),
    "literal_multinomial_items_and_words": distinct(lambda: draws(False)),
    "reproducible_draws": distinct(lambda: draws(True))}}
out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                            capture_output=True, text=True).stdout.strip()
print(json.dumps(out))
