#!/usr/bin/env python
"""Benchmark of the ProdSearch embedding-scoring hot path on B200 (contract: see the task brief).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one TEM training step (ItemTransformerRanker.forward_dotproduct + backward + the
reference's clipped Adam) on BASELINE.json configs[1]: Amazon-Sports-shaped synthetic data,
P=18k items, V=32k words, d=128, 1 layer / 8 heads / ff 512, uprev_review_limit 20, batch 384 per GPU,
5 negatives, dropout 0.1 (the reference default).  Rank 0 prints ONE JSON line.

  value  : samples/s with the batches already resident in HBM (CUDA events, max over ranks)
  e2e    : the same step through the module API from pinned HOST batches (H2D inside) + loss.item()
  roofline / extra : the dominant hand-written kernel of the step, and every hot-path kernel in the
           bandwidth regime on a 16M x 128 table (the regime the HBM-roofline target is defined on)
  cpu_baseline : the oracle's CPU restatement of the same step on this box's host cores; cpu_baseline.others: the
           PV step (BASELINE configs[0]), 1M-item catalog ranking and gather / scatter-add on the same cores
  --impl reference : times that CPU path alone (all host threads), same metric / config
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(model="TEM item_transformer", product_size=18000, vocab_size=32000, user_size=35000,
                embedding_size=128, inter_layers=1, heads=8, ff_size=512, uprev_review_limit=20,
                batch_per_gpu=384, neg_per_pos=5, pv_window_size=1, dropout=0.1, lr=0.0005, max_grad_norm=5.0)


def model_args(dropout):
    return argparse.Namespace(
        train_review_only=True, embedding_size=WORKLOAD["embedding_size"], dropout=dropout, pretrain_emb_dir="",
        pretrain_up_emb_dir="", sep_prod_emb=False, model_name="item_transformer", ff_size=WORKLOAD["ff_size"],
        heads=WORKLOAD["heads"], inter_layers=WORKLOAD["inter_layers"], query_encoder_name="fs", use_dot_prod=True,
        use_pos_emb=True, use_item_pos=False, sim_func="product", pos_weight=False,
        neg_per_pos=WORKLOAD["neg_per_pos"], optim="adam", lr=WORKLOAD["lr"],
        max_grad_norm=WORKLOAD["max_grad_norm"], beta1=0.9, beta2=0.999, decay_method="adam", warmup_steps=8000,
        l2_lambda=0.0, train_from="")


def load_traffic():
    """ncu-measured DRAM bytes per launch (profiles/ncu_traffic.json, written by profiles/make_traffic.py from the
    committed ncu exports): {regime: {kernel: {...}}}; empty when the file is absent."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        z = json.load(open(p))
        return dict(hbm=z["hbm_gbs"], bf16=z["bf16_tflops"], bf16_sustained=z["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler(object):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md: "start before, kill after").

    The poller is started BEFORE the warm-up steps: launching nvidia-smi (NVML attach) stalls the polled GPU for a
    fraction of a millisecond, and a bench window is only K x 0.45 ms long -- started at the window's first step
    (as the first version did) that stall landed inside it on rank 0 and every other rank waited for it at the
    step-start barrier (~19 us per step at K = 30).  Samples carry nvidia-smi's own time stamp; the summary uses
    those taken between ``begin()`` and ``end()`` (+- one polling interval: the GPU is under the same load in the
    warm-up steps before and the end-to-end steps after)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    PERIOD_MS = 50

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None

    def start(self):
        if self.index is None:      # other ranks: no sampler (one nvidia-smi poller per box is enough)
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.PERIOD_MS)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def begin(self):
        import datetime
        self.t0 = datetime.datetime.now()

    def end(self):
        import datetime
        self.t1 = datetime.datetime.now()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is not None:
            time.sleep(2.5 * self.PERIOD_MS / 1e3)
            self.proc.terminate()
            self.t.join(timeout=2)
            self.proc = None

    def summary(self):
        import datetime
        rows = [r for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        if self.t0 is not None and self.t1 is not None:
            pad = datetime.timedelta(milliseconds=1.5 * self.PERIOD_MS)
            inside = []
            for r in rows:
                try:
                    ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f")
                except ValueError:
                    continue
                if self.t0 - pad <= ts <= self.t1 + pad:
                    inside.append(r)
            rows = inside or rows
        sm = [float(r[1]) for r in rows]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "poll_ms": self.PERIOD_MS}


def cpu_reference_step_time(steps, warmup, dropout, seed=666):
    import torch
    import oracle
    from prodsearch_b200 import synth
    from prodsearch_b200.transformer import TransformerEncoder
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = model_args(dropout)
    P, V, d, B = WORKLOAD["product_size"], WORKLOAD["vocab_size"], WORKLOAD["embedding_size"], WORKLOAD["batch_per_gpu"]
    g = torch.Generator().manual_seed(seed)
    enc = TransformerEncoder(d, cfg.ff_size, cfg.heads, dropout, cfg.inter_layers)
    enc.initialize_parameters()
    params = {"transformer_encoder." + k: v.detach().clone() for k, v in enc.state_dict().items()}
    params["product_emb.weight"] = torch.randn(P + 1, d, generator=g)
    params["product_emb.weight"][P] = 0
    params["word_embeddings.weight"] = torch.randn(V, d, generator=g)
    params["product_bias"] = torch.zeros(P + 1)
    params["word_bias"] = torch.zeros(V)
    params["query_encoder.f_W.weight"] = torch.randn(d, d, generator=g) * (1.0 / d) ** 0.5
    params["query_encoder.f_W.bias"] = torch.zeros(d)
    leaves = []
    for k, v in params.items():
        if not k.endswith("pos_emb.pe"):
            v.requires_grad_(True)
            leaves.append(v)
    opt = torch.optim.Adam(leaves, lr=cfg.lr, betas=(0.9, 0.999), eps=1e-9)
    wd = torch.as_tensor(synth.word_dists(V))
    pd = torch.ones(P)
    times = []
    for it in range(warmup + steps):
        batch, _, _ = synth.tem_batch(B, P, V, seed=seed + it)
        t0 = time.perf_counter()
        neg_items = torch.multinomial(pd, B * cfg.neg_per_pos, replacement=True).view(B, -1)
        neg_words = torch.multinomial(wd, B * cfg.neg_per_pos, replacement=True)
        loss, _, _ = oracle.tem_forward(params, cfg, batch.query_word_idxs, batch.target_prod_idxs,
                                        batch.u_item_idxs, batch.pos_iword_idxs, neg_items, neg_words, training=True)
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(leaves, cfg.max_grad_norm)
        opt.step()
        float(loss)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return sum(times) / len(times), cores


def cpu_reference_others(seed=666, scale=1):
    """The other CPU timings SURVEY.md 8(d) asks for next to the TEM step, each on a bounded sample (seconds of host
    time in all): (ii) BASELINE configs[0], a ParagraphVector train step (models/PV.py:50-80 through the oracle port,
    dense [R, d] table gradient + Adam as torch does it); (iii) full-catalog ranking over 1M items -- the reference's
    literal path (scores [24, N] then a full argsort, trainer.py:136,:152) and the restated fair baseline (one GEMM +
    torch.topk(100)); (iv) index_select / index_add_ on a large fp32 table.  All host threads.  ``scale`` > 1 divides
    the table sizes (the CPU test of this function)."""
    import torch
    import oracle
    from prodsearch_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(seed)
    d, V, K = WORKLOAD["embedding_size"], WORKLOAD["vocab_size"], WORKLOAD["neg_per_pos"]
    out = {"cores": cores}

    def median_time(fn, iters, warmup=1):
        for _ in range(warmup):
            fn()
        ts = []
        for _ in range(iters):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return statistics.median(ts)

    # (ii) PV train step: R = 300k reviews, N = 384 reviews per batch, one target word each, 5 negatives
    R, N = 300_000 // scale, WORKLOAD["batch_per_gpu"]
    review_table = torch.randn(R, d, generator=g).requires_grad_(True)
    word_table = torch.randn(V, d, generator=g).requires_grad_(True)
    opt = torch.optim.Adam([review_table, word_table], lr=WORKLOAD["lr"], eps=1e-9)
    wd = torch.as_tensor(synth.word_dists(V))
    rid = torch.randint(0, R - 1, (N,), generator=g)
    pos_w = torch.multinomial(wd, N, replacement=True, generator=g).view(N, 1)
    mask = torch.ones(N, 1, dtype=torch.uint8)

    def pv_step():
        neg_w = torch.multinomial(wd, N * K, replacement=True)
        _, loss = oracle.pv_forward(review_table, word_table, rid, pos_w, mask, neg_w, K)
        opt.zero_grad()
        loss.mean().backward()
        opt.step()
    sec = median_time(pv_step, 5)
    out["pv_train_step"] = {"value": N / sec, "unit": "reviews/s", "ms_per_step": sec * 1e3,
                            "sample": "BASELINE configs[0]: 5 ParagraphVector steps (fwd + bwd + Adam), 384 reviews, "
                                      "R = 300k x 128 review table, 5 negatives, oracle port"}
    del review_table, word_table, opt
    # (ii-b) BASELINE configs[2]: an RTM (ProductRanker) train step through the oracle port -- pv at batch 384, pvc at
    #        batch 96 (its [N, 100, 128] gathers need ~20 GB and ~30 s at 384: bounded sample, samples/s is the unit)
    try:
        from prodsearch_b200 import synth as synth_
        from prodsearch_b200.ps_model import ProductRanker
        Vr, Rr, Pr, Ur, Wr = V, 300_000 // scale, 18000 // scale, 35000 // scale, 100
        rw = synth_.review_words_table(Rr, Vr, Wr)
        for enc, Bq in (("pv", WORKLOAD["batch_per_gpu"] // (8 if scale > 1 else 1)), ("pvc", 96 // (8 if scale > 1 else 1))):
            a = model_args(0.0)
            a.model_name, a.review_encoder_name, a.review_word_limit, a.corrupt_rate = "review_transformer", enc, Wr, 0.9
            a.fix_emb, a.do_subsample_mask, a.use_user_emb, a.use_item_emb, a.use_seg_emb = False, True, False, False, True
            a.review_pad_idx = Rr - 1
            torch.manual_seed(1)
            ref_model = ProductRanker(a, "cpu", Vr, Rr, Pr, Ur, rw, None, word_dists=synth_.word_dists(Vr))
            params = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and not k.endswith("pos_emb.pe"))
                      for k, v in ref_model.state_dict().items()}
            leaves = [v for v in params.values() if v.requires_grad]
            opt_r = torch.optim.Adam(leaves, lr=WORKLOAD["lr"], eps=1e-9)
            batch, draws = synth_.rtm_batch(Bq, rw, Vr, Pr, Ur, pvc=(enc == "pvc"), train_pv=True, seed=3)
            gm = torch.Generator().manual_seed(4)
            masks = [(torch.rand(Bq * 50, Wr, generator=gm) < 0.9).float(), (torch.rand(Bq * K * 50, Wr, generator=gm) < 0.9).float()] \
                if enc == "pvc" else None

            def rtm_step():
                loss, _, _ = oracle.rtm_forward(params, a, batch, True, draws["multinomial"][0], [m.clone() for m in masks] if masks else None,
                                                training=True)
                opt_r.zero_grad()
                loss.backward()
                torch.nn.utils.clip_grad_norm_(leaves, WORKLOAD["max_grad_norm"])
                opt_r.step()
            sec = median_time(rtm_step, 2 if enc == "pv" else 1, warmup=1 if enc == "pv" else 0)
            out["rtm_%s_train_step" % enc] = {"value": Bq / sec, "unit": "samples/s", "ms_per_step": sec * 1e3, "batch": Bq,
                                               "sample": "BASELINE configs[2]: RTM train step (fwd + bwd + clipped Adam), %s review encoder "
                                                         "with the review-word objective, 20 + 30 reviews / sequence, 100 words / "
                                                         "review, batch %d, oracle port" % (enc, Bq)}
            del ref_model, params, leaves, opt_r
    except Exception as ex:                                           # noqa: BLE001 -- reported, never fatal
        out["rtm_train_step"] = {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:120])}
    # (iii) full-catalog ranking over N = 1M items
    n_items = 1_000_000 // scale
    chunk = max(n_items // 4, 100)
    table = torch.randn(n_items, d, generator=g)
    q24 = torch.randn(24, d, generator=g)
    sec = median_time(lambda: oracle.reference_rank((q24 @ table.t()).numpy())[:, :100], 1, warmup=0)
    out["catalog_rank_1M_literal"] = {"value": 24 / sec, "unit": "queries/s", "ms": sec * 1e3,
                                      "sample": "one batch of 24 queries: scores [24, 1M] + full argsort (trainer.py:136,:152)"}
    q = torch.randn(384, d, generator=g)

    def gemm_topk():
        best_s, best_i = None, None
        for c0 in range(0, n_items, chunk):                        # [384, 250k] score chunks: 384 MB each
            sc, ix = torch.topk(q @ table[c0:c0 + chunk].t(), 100, dim=1)
            ix = ix + c0
            if best_s is None:
                best_s, best_i = sc, ix
            else:
                sc, sel = torch.topk(torch.cat([best_s, sc], 1), 100, dim=1)
                best_s, best_i = sc, torch.gather(torch.cat([best_i, ix], 1), 1, sel)
        return best_i
    sec = median_time(gemm_topk, 2)
    out["catalog_rank_1M_gemm_topk"] = {"value": 384 / sec, "unit": "queries/s", "ms": sec * 1e3,
                                        "sample": "384 queries x 1M items: chunked GEMM + torch.topk(100) + merge (restated fair CPU baseline)"}
    del table
    # (iv) gather / scatter-add on a table far larger than the CPU caches (bounded: 4M rows = 2 GB, not 16M)
    rows, n = 4_000_000 // scale, 1_000_000 // scale
    big = torch.empty(rows, d).normal_(generator=g)
    idx = synth.gather_indices(n, rows, seed=1, dist="uniform")
    sec = median_time(lambda: big.index_select(0, idx), 3)
    out["gather_rows"] = {"value": n * (d * 4 * 2 + 8) / sec / 1e9, "unit": "GB/s", "ms": sec * 1e3,
                          "sample": "index_select of 1M uniform rows from a 4M x 128 fp32 table (2 GB)"}
    src = torch.randn(n, d, generator=g)
    acc = torch.zeros(rows, d)
    sec = median_time(lambda: acc.index_add_(0, idx, src), 3)
    out["scatter_add_rows"] = {"value": n * (d * 4 * 2 + 8) / sec / 1e9, "unit": "GB/s", "ms": sec * 1e3,
                               "sample": "index_add_ of 1M uniform rows into a 4M x 128 fp32 table (aten::embedding_dense_backward's core)"}
    return out


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = WORKLOAD["batch_per_gpu"]
    sec, cores = cpu_reference_step_time(a.steps, a.warmup, a.dropout)
    value = B / sec
    print(json.dumps({
        "impl": "reference", "metric": "tem_train_samples_per_s", "value": value, "unit": "samples/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(WORKLOAD, workload="BASELINE configs[1]: TEM train step, batch 384, CPU path", dropout=a.dropout),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": "%d full TEM train steps (fwd+bwd+clipped Adam) of batch 384 on the oracle port "
                                   "(same ATen CPU kernels as the reference modules)" % a.steps},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def timed(fn, iters, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters * 1e-3


def dump_outputs(path, loss, model):
    """What a caller of the timed step receives from its last call: the loss it returned and the parameters it left
    (the rank's own shards when the tables are row-sharded), each as ``path/<name>.npy`` in float32.  The inputs are
    seeded and the step is reproducible, so one build writes the same bits on every run with the same arguments, and
    two builds can be compared array by array."""
    import numpy as np
    model.flush_lazy_rows()        # --grad-mode rowsparse: rows the lazily caught-up Adam has not brought current yet
    arrays = {"loss": loss.detach().float().reshape(-1)}
    arrays.update(("param." + k, p.detach().float()) for k, p in model.named_parameters())
    nbytes = sum(v.numel() * 4 for v in arrays.values())
    assert nbytes <= 64 << 20, "outputs of %d bytes: sample them below 64 MB" % nbytes    # TEM workload: ~26 MB
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v.cpu().numpy())


def bandwidth_regime(peaks, rows=16_000_000, d=128):
    """Every hot-path kernel on a table far larger than L2 (8.2 GB): achieved algorithmic GB/s."""
    import torch
    from prodsearch_b200 import _lib, ops, synth
    out = {}
    dev = "cuda"
    table = torch.empty(rows + 1, d, device=dev).normal_()
    table[rows] = 0
    GB = 1e9

    traffic = load_traffic().get("bandwidth", {})
    main_kernel = {"G1": "gather_rows_kernel", "G4": "meanpool_kernel", "G3": "ns_loss_w1_kernel", "G2": "seg_reduce_kernel"}

    def entry(name, sec, nbytes, note):
        out[name] = {"ms": sec * 1e3, "achieved": nbytes / sec / GB, "unit": "GB/s", "peak": peaks["hbm"],
                     "frac": nbytes / sec / GB / peaks["hbm"], "algorithmic_bytes": nbytes, "note": note}
        tr = traffic.get(main_kernel.get(name[:2], ""))
        if tr is not None and not name.endswith("_zipf"):     # ncu DRAM bytes of the entry's main kernel, one launch
            out[name]["traffic"] = tr["dram_bytes_per_launch"]
            out[name]["traffic_kernel"] = main_kernel[name[:2]]

    n = 4_000_000
    idx = synth.gather_indices(n, rows, seed=1, dist="uniform").to(dev)
    sec = timed(lambda: ops.gather_rows(table, idx), 10)
    entry("G1_gather_rows", sec, n * (d * 4 * 2 + 8), "4M uniform rows: read + materialised write + int64 idx")
    idz = synth.gather_indices(n, rows, seed=2, dist="zipf").to(dev)
    sec = timed(lambda: ops.gather_rows(table, idz), 10)
    entry("G1_gather_rows_zipf", sec, n * (d * 4 * 2 + 8), "4M Zipf(1.0) rows")
    nq, w = 400_000, 10
    idx2 = idx[:nq * w].view(nq, w).contiguous()
    sec = timed(lambda: ops.gather_meanpool(table, idx2, pad_idx=rows), 10)
    entry("G4_gather_meanpool", sec, nq * w * (d * 4 + 8) + nq * d * 4, "400k pools of 10 rows (output 1 row each)")
    na, k = 500_000, 5
    anchor = torch.randn(na, d, device=dev)
    pos = idx[:na].view(na, 1).contiguous()
    neg = idx[na:na + na * k].view(na, 1, k).contiguous()
    sec = timed(lambda: ops.ns_loss(anchor, table, pos, neg), 10)
    entry("G3_ns_loss", sec, na * (1 + k) * (d * 4 + 8) + na * d * 4 * 2, "500k anchors x (1+5) rows, fwd + score grad")
    src = torch.randn(n, d, device=dev)
    contrib = [ops.make_contrib(idx, src)]
    holder = {}

    def sr():
        holder["r"] = ops.scatter_reduce(contrib, rows + 1, d, drop_idx=rows)
    sec = timed(sr, 5)
    nu = int(holder["r"][3].item())
    entry("G2_scatter_reduce", sec, n * (d * 4 + 8) + nu * d * 4, "4M uniform slots -> %d rows, sort included in time" % nu)
    # the same reduction with the SORT done beforehand (psb_scatter_sort_rows reads only the indices: in a training
    # step it runs next to the backward pass, RowGradSink.expect): the segmented reduce alone
    try:
        wsb = ops.scatter_workspace_bytes(n, rows + 1)
        ws_ = torch.empty(wsb, dtype=torch.uint8, device=dev)
        uq_ = torch.empty(n, dtype=torch.int32, device=dev)
        nu_ = torch.zeros(1, dtype=torch.int32, device=dev)
        ops.scatter_sort([idx], rows + 1, rows, ws_, uq_, nu_)
        sec = timed(lambda: ops.scatter_reduce_sorted(contrib, rows + 1, d, rows, ws_, uq_, nu_, want_rows=True), 5)
        entry("G2_reduce_presorted", sec, n * (d * 4 + 8) + nu * d * 4, "4M uniform slots, index lists sorted beforehand "
              "(psb_scatter_sort_rows), segmented reduce + fix-up only")
        del ws_, uq_, nu_
    except RuntimeError as ex:
        out["G2_reduce_presorted"] = {"unavailable": str(ex)[:80]}
    contrib_z = [ops.make_contrib(idz, src)]

    def srz():
        holder["z"] = ops.scatter_reduce(contrib_z, rows + 1, d, drop_idx=rows)
    sec = timed(srz, 5)
    nuz = int(holder["z"][3].item())
    entry("G2_scatter_reduce_zipf", sec, n * (d * 4 + 8) + nuz * d * 4, "4M Zipf slots -> %d rows" % nuz)
    # catalog scoring: 1M items, top-100 (the eval table is static: its fp16 shortlist copy / max row norm are
    # prepared once, as rank_catalog caches them)
    n_items = 1_000_000
    cat = {"note": "fp16 shortlist copy and max row norm of the (static) eval table prepared once, as rank_catalog "
                   "caches them; every mode returns the exact-mode ids and scores; tensor peak = measured bf16 cuBLAS "
                   "burst (fp16 shortlist) or half of it (tf32)"}
    norm = ops.table_max_row_sqnorm(table, n_items)
    prep = ops.catalog_prepare_f16(table, n_items)
    for m in (24, 384, 4096):
        q = torch.randn(m, d, device=dev)
        for mode, mname in ((_lib.TOPK_EXACT, "exact_fp32"), (_lib.TOPK_TC, "tcgen05_tf32"), (_lib.TOPK_TC16, "tcgen05_f16")):
            if mode == _lib.TOPK_EXACT and m > 384:
                continue
            try:
                sec = timed(lambda: ops.catalog_topk(q, table, 100, n_items=n_items, mode=mode, max_row_sqnorm=norm,
                                                     prepared=prep if mode == _lib.TOPK_TC16 else None), 3, warmup=1)
            except RuntimeError as ex:
                cat["%s_m%d" % (mname, m)] = {"unavailable": str(ex)[:80]}
                continue
            flops = 2.0 * m * n_items * d
            ent = {"ms": sec * 1e3, "queries_per_s": m / sec, "tflops": flops / sec / 1e12}
            if mode == _lib.TOPK_TC16:
                ent["table_GBps"] = n_items * d * 2 / sec / GB
                ent["frac_of_tensor_peak"] = flops / sec / 1e12 / peaks["bf16"]
                ent["frac_of_hbm_peak"] = n_items * d * 2 / sec / GB / peaks["hbm"]
            else:
                ent["table_GBps"] = n_items * d * 4 / sec / GB
                if mode == _lib.TOPK_TC:
                    ent["frac_of_tensor_peak"] = flops / sec / 1e12 / (peaks["bf16"] / 2)
                ent["frac_of_hbm_peak"] = n_items * d * 4 / sec / GB / peaks["hbm"]
            cat["%s_m%d" % (mname, m)] = ent
    out["G5_catalog_topk_1M"] = cat
    # the same fused top-100 over the whole 16M-row table (BASELINE configs[4] on one GPU: the N=1 end of
    # extra.sharded_16M.catalog_topk_16M of the multi-GPU runs)
    try:
        del prep
        prep16 = ops.catalog_prepare_f16(table, rows)
        mode, mname = (_lib.TOPK_TC16, "tcgen05_f16") if prep16.fits else (_lib.TOPK_TC, "tcgen05_tf32")
        norm16 = ops.table_max_row_sqnorm(table, rows)
        esz = 2 if mode == _lib.TOPK_TC16 else 4
        tpeak = peaks["bf16"] if mode == _lib.TOPK_TC16 else peaks["bf16"] / 2
        for m in (24, 384, 4096):
            q = torch.randn(m, d, device=dev)
            sec = timed(lambda: ops.catalog_topk(q, table, 100, n_items=rows, mode=mode, max_row_sqnorm=norm16,
                                                 prepared=prep16 if mode == _lib.TOPK_TC16 else None), 3, warmup=1)
            flops = 2.0 * m * rows * d
            ent = {"ms": sec * 1e3, "queries": m, "k": 100, "mode": mname, "queries_per_s": m / sec,
                   "tflops": flops / sec / 1e12, "frac_of_tensor_peak": flops / sec / 1e12 / tpeak,
                   "table_GBps": rows * d * esz * ((m + 511) // 512) / sec / GB,
                   "frac_of_hbm_peak": rows * d * esz * ((m + 511) // 512) / sec / GB / peaks["hbm"],
                   "note": "table_GBps counts one shortlist-table pass per 512 queries (M <= 512: the table is streamed "
                           "once, HBM-bound; thousands of queries: tensor-bound)"}
            out["G5_catalog_topk_16M" if m == 4096 else "G5_catalog_topk_16M_m%d" % m] = ent
    except RuntimeError as ex:
        out["G5_catalog_topk_16M"] = {"unavailable": str(ex)[:120]}
    return out


def train_16m_regime(peaks, rows=16_000_000, steps=8):
    """BASELINE configs[4] as a TRAINING step on one GPU: the TEM step of the headline (batch 384, same encoder) with a
    16M-row item table.  grad_mode rowsparse + the row-sparse lazily caught-up Adam: the step touches ~10k rows and its
    cost must not depend on the table size; the dense form (the reference's semantics taken literally: dense table
    gradient + dense Adam sweep, 28 B x 2.05 G parameters per step) is timed next to it on a few steps."""
    import torch
    from prodsearch_b200 import synth
    from prodsearch_b200.graph_step import GraphedTrainStep
    from prodsearch_b200.item_transformer import ItemTransformerRanker
    from prodsearch_b200.optimizers import build_optim
    out = {"table": "%d x 128 fp32 item table (8.2 GB) + Adam moments (16.4 GB), batch 384, dropout 0.1" % rows}
    V, B = WORKLOAD["vocab_size"], WORKLOAD["batch_per_gpu"]
    args = model_args(WORKLOAD["dropout"])
    for mode, a_sampler in (("rowsparse", "randint"), ("rowsparse_aged", "randint"), ("rowsparse_multinomial", "multinomial"),
                            ("dense", "randint")):
        try:
            label, mode = mode, mode.split("_")[0]
            torch.manual_seed(666)
            with torch.device("cuda"):          # the 8.2 GB table is created and initialised on the GPU, not on the host
                model = ItemTransformerRanker(args, "cuda", V, rows, None, word_dists=synth.word_dists(V), grad_mode=mode)
            model.item_negative_sampler = a_sampler
            optim = build_optim(args, model)
            model.train()
            batches = []
            for it in range(steps + 3):
                b, _, _ = synth.tem_batch(B, rows, V, seed=900 + it, permute=False)
                batches.append(argparse.Namespace(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(b).items()}))
            sample = argparse.Namespace(**vars(batches[0]))
            sample.query_word_idxs = torch.full((B, 12), V - 1, dtype=torch.int64)
            step = GraphedTrainStep(model, optim, sample, pad_values={"query_word_idxs": V - 1, "u_item_idxs": rows})
            n = steps if label.startswith("rowsparse") and a_sampler == "randint" else 3
            for it in range(3):
                step(batches[it])
            if label == "rowsparse_aged":
                # steady state of a long run: every row has been updated once, long ago (step 1 of 100 000), so each row a
                # step touches is replayed over the full catch-up window (264 steps) before it is read
                opt = optim.optimizer
                torch.cuda.synchronize()
                for p_, st_ in opt.state.items():
                    if "last_step" in st_:
                        st_["last_step"].fill_(1)
                        st_["exp_avg"].normal_(0, 1e-3)
                        st_["exp_avg_sq"].fill_(1e-6)
                opt._step_dev.fill_(100_000)
                tau = torch.arange(opt.coef_cap, dtype=torch.float64, device="cuda").clamp_(min=1)
                b1, b2 = opt.param_groups[0]["betas"]
                hist = torch.stack([opt.param_groups[0]["lr"] / (1 - b1 ** tau), 1 / torch.sqrt(1 - b2 ** tau)], dim=1)
                opt._coef_hist.copy_(hist.to(torch.float32).reshape(-1))
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for it in range(n):
                step(batches[3 + it])
            s1.record()
            torch.cuda.synchronize()
            ms = s0.elapsed_time(s1) / n
            out[label] = {"ms_per_step": ms, "samples_per_s": B / (ms * 1e-3), "steps": n,
                          "launches_per_step": step.launches_per_replay, "item_negative_sampler": a_sampler}
            if mode == "dense":
                nparam = sum(p.numel() for p in model.parameters())
                out[label]["adam_sweep_GB"] = nparam * 28 / 1e9
                out[label]["note"] = "dominated by the dense Adam / clip-norm sweep and the dense gradient buffer"
            if a_sampler == "multinomial":
                out[label]["note"] = ("the reference's literal torch.multinomial(ones(P)) draw: ATen renormalises the 16M-entry "
                                      "distribution with one thread block on every call (~10 ms)")
            del step, model, optim
        except Exception as ex:                                       # noqa: BLE001 -- reported, never fatal
            out[label] = {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:160])}
        torch.cuda.empty_cache()
    if "ms_per_step" in out.get("rowsparse", {}) and "ms_per_step" in out.get("dense", {}):
        out["dense_over_rowsparse"] = out["dense"]["ms_per_step"] / out["rowsparse"]["ms_per_step"]
    return out


def rtm_regime(peaks, steps=5):
    """BASELINE configs[2]: an RTM (ProductRanker) train step at batch 384, 20 + 30 reviews per sequence, 100 words per
    review, R = 300k reviews, pv and pvc review encoders with the review-word objective (train_pv) -- forward,
    backward, gradient sinks, clipped Adam, launched eagerly.  The gather-heavy kernels of the step are reported
    against the HBM roofline (library profiler: CUDA events around every launch); the encoder over 2304 sequences
    of 51 tokens is the rest of the step."""
    import torch
    from prodsearch_b200 import _lib, synth
    from prodsearch_b200.optimizers import build_optim
    from prodsearch_b200.ps_model import ProductRanker
    V, R, P, U, K, B, Wr, d = 32000, 300_000, 18000, 35000, 5, WORKLOAD["batch_per_gpu"], 100, 128
    rw = synth.review_words_table(R, V, Wr)
    out = {"shape": "batch %d, 20 + 30 reviews / sequence, %d words / review, R = %d, V = %d, d = %d, K = %d" % (B, Wr, R, V, d, K)}
    for enc in ("pv", "pvc"):
        try:
            a = model_args(0.0)
            a.model_name, a.review_encoder_name, a.review_word_limit, a.corrupt_rate = "review_transformer", enc, Wr, 0.9
            a.fix_emb, a.do_subsample_mask, a.use_user_emb, a.use_item_emb, a.use_seg_emb = False, True, False, False, True
            torch.manual_seed(666)
            model = ProductRanker(a, "cuda", V, R, P, U, rw, None, word_dists=synth.word_dists(V))
            optim = build_optim(a, model)
            model.train()
            batch, _ = synth.rtm_batch(B, rw, V, P, U, pvc=(enc == "pvc"), train_pv=True, seed=5)
            cb = argparse.Namespace(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(batch).items()})

            def one():
                loss = model(cb, train_pv=True)
                model.zero_grad()
                loss.backward()
                optim.step()
                return loss
            for _ in range(2):
                one()
            sec_eager = timed(one, steps, warmup=1)
            # the same step captured once and replayed (graph_step.GraphedTrainStep, as the TEM headline): the eager step
            # is bound by the host launching ~150 kernels
            sec = sec_eager
            launch = "eager"
            try:
                from prodsearch_b200.graph_step import GraphedTrainStep
                gstep = GraphedTrainStep(model, optim, cb)
                sec = timed(lambda: gstep(cb), steps, warmup=2)
                launch = "CUDA graph replay"
                del gstep
            except Exception as ex:                                   # noqa: BLE001 -- the eager number stands
                launch = "eager (graph capture failed: %s)" % str(ex)[:80]
            _lib.profile_enable(True)
            for _ in range(2):
                one()
            kp = _lib.profile_dump()
            _lib.profile_enable(False)
            ent = {"ms_per_step": sec * 1e3, "samples_per_s": B / sec, "launch": launch, "eager_ms_per_step": sec_eager * 1e3}
            Rc = 50
            if enc == "pvc":     # PVC: clean + corrupted mean of the positives, mean of the negatives: (2 + K) * B * Rc pools of Wr rows
                pools = (2 + K) * B * Rc
                nbytes = pools * (Wr * (d * 4 + 8) + d * 4)
                k_ = kp.get("meanpool_kernel")
                if k_:
                    ms = k_[1] / 2
                    ent["meanpool_kernel"] = {"ms_per_step": ms, "launches_per_step": k_[0] / 2, "algorithmic_bytes": nbytes,
                                              "achieved": nbytes / (ms * 1e-3) / 1e9, "unit": "GB/s", "peak": peaks["hbm"],
                                              "frac": nbytes / (ms * 1e-3) / 1e9 / peaks["hbm"],
                                              "note": "fused gather + masked mean over %d pools of %d word rows (the [N, Wr, d] "
                                                      "tensors of PVC.py:76-79 / ps_model.py:293-297 never exist); the 32k x "
                                                      "128 word table is L2-resident, so this is requested bytes/s" % (pools, Wr)}
            else:                # PV: review rows gathered for positives (B * Rc) and negatives (B * K * Rc)
                rows_ = B * Rc * (1 + K)
                nbytes = rows_ * (d * 4 * 2 + 8)
                k_ = kp.get("gather_rows_kernel")
                if k_:
                    ms = k_[1] / 2
                    ent["gather_rows_kernel"] = {"ms_per_step": ms, "launches_per_step": k_[0] / 2, "algorithmic_bytes": nbytes,
                                                 "achieved": nbytes / (ms * 1e-3) / 1e9, "unit": "GB/s", "peak": peaks["hbm"],
                                                 "frac": nbytes / (ms * 1e-3) / 1e9 / peaks["hbm"],
                                                 "note": "review-table row gathers (PV.py:46-48, ps_model.py:281,:290) plus the "
                                                         "segment-row gathers of the step; 154 MB review table"}
            top = sorted(kp.items(), key=lambda kv: -kv[1][1])[:6]
            ent["top_kernels_ms_per_step"] = {k: round(v[1] / 2, 4) for k, v in top}
            out[enc] = ent
            del model, optim
        except Exception as ex:                                       # noqa: BLE001
            out[enc] = {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:160])}
        torch.cuda.empty_cache()
    return out


def guarded(fn, seconds, on_timeout):
    """Run fn() with a watchdog: if it has not returned after ``seconds``, on_timeout() runs on the watchdog thread
    and the process exits with status 0.  extra.sharded_16M contains collectives and peer-memory kernels that had no
    GPU run when they were written; whatever happens inside, the headline JSON line of the bench must still appear."""
    import threading
    done = threading.Event()

    def watch():
        if not done.wait(seconds):
            try:
                on_timeout()
                sys.stdout.flush()
            finally:
                os._exit(0)
    threading.Thread(target=watch, daemon=True).start()
    try:
        return fn()
    finally:
        done.set()


def sharded_regime(peaks, pg, rank, world, rows=16_000_000, d=128, m_total=4096, k=100, n_gather=1_000_000, dev="cuda",
                   table_cls=None, timer=None):
    """BASELINE configs[4]: a 16M x 128 fp32 table row-sharded over the ranks of one box (owner = id % G), in peer
    memory.  (1) training-side row gathers of global ids from their owners over NVLink (psb_peer_gather_rows),
    (2) sharded full-catalog top-100: all-gather the queries, local fused top-k per shard, all-gather the per-shard
    lists, merge (psb_topk_merge).  Every rank runs this; seconds are the MAX over ranks.  A failure on one rank is
    agreed on by all ranks BEFORE the next collective, so nobody is left waiting inside NCCL.
    ``dev`` / ``table_cls`` / ``timer`` exist for the world-2 gloo test of this control flow (tests/test_sharding_gloo.py)."""
    import torch
    import torch.distributed as dist
    from prodsearch_b200 import _lib, ops, synth
    if table_cls is None:
        from prodsearch_b200.peer import PeerShardedTable as table_cls
    timer = timer or timed

    def sync():
        dist.barrier()
        if str(dev).startswith("cuda"):
            torch.cuda.synchronize()
    out = {"table": "%d x %d fp32 row-sharded over %d ranks (%.2f GB per rank), peer memory" %
                    (rows, d, world, (rows // world) * d * 4 / 1e9)}
    GB = 1e9

    def agree(err):
        """True when every rank got here without an error (one small all-reduce)."""
        t = torch.tensor([0 if err is None else 1], device=dev, dtype=torch.int32)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return int(t.item()) == 0

    def max_over_ranks(sec):
        t = torch.tensor([sec], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    table = None
    err = None
    try:
        table = table_cls(rows + 1, d, pg, pad_idx=rows)                  # collective: alloc + IPC handle exchange
        with torch.no_grad():
            table.weight.normal_()
            if rows % world == rank:
                table.weight[rows // world] = 0                           # the pad row lives on rank rows % G
        table.weight.requires_grad_(False)
    except Exception as ex:                                               # noqa: BLE001 -- reported in the JSON line
        err = "%s: %s" % (type(ex).__name__, str(ex)[:120])
    if not agree(err):
        out["unavailable"] = err or "another rank failed to allocate its shard"
        return out
    sync()
    # ---- (1) row gathers from the owners: 1M uniform global ids per rank, (G-1)/G of them cross NVLink
    n = int(n_gather)
    sec = None
    try:
        idx = synth.gather_indices(n, rows, seed=11 + rank, dist="uniform").to(dev)
        sec_fetch = None
        with torch.no_grad():
            if hasattr(table, "shard"):          # the kernel alone: psb_peer_gather_rows on preallocated buffers
                buf = torch.empty(n, d, device=dev)
                lib = _lib.load()

                def kernel_only():
                    _lib.check(lib.psb_peer_gather_rows(table.shard.ptr_array(), world, rows + 1, d, idx.data_ptr(), n,
                                                        buf.data_ptr(), None, -1, 0, None, _lib.stream_ptr()),
                               "psb_peer_gather_rows")
                sec = timer(kernel_only, 5, warmup=2)
                sec_fetch = timer(lambda: table.fetch([idx]), 5, warmup=2)
            else:
                sec = timer(lambda: table.fetch([idx]), 5, warmup=2)
    except Exception as ex:                                               # noqa: BLE001
        err = "%s: %s" % (type(ex).__name__, str(ex)[:120])
    if agree(err):
        sec = max_over_ranks(sec)
        nbytes = n * (d * 4 * 2 + 8)
        wire = n * (world - 1) / world * d * 4
        out["peer_gather_rows"] = {
            "ms": sec * 1e3, "rows_per_rank": n, "algorithmic_bytes_per_rank": nbytes,
            "achieved_per_rank": nbytes / sec / GB, "achieved": world * nbytes / sec / GB, "unit": "GB/s",
            "nvlink_GBps_per_rank": wire / sec / GB, "frac_of_nvlink_peak": wire / sec / GB / 900.0,
            "fetch_ms": None if sec_fetch is None else max_over_ranks(sec_fetch) * 1e3,
            "note": "1M uniform global ids per rank read from their owners by psb_peer_gather_rows (128-bit loads from "
                    "peer memory inside the kernel; read + materialised write + int64 id); (G-1)/G of the rows travel "
                    "over NVLink, so the link (900 GB/s per direction per GPU), not HBM, is the ceiling.  fetch_ms = "
                    "PeerShardedTable.fetch around it: id concat, remap list and a fresh 512 MB mini table per call "
                    "(what round 1 reported as the gather: the allocation, not the link, was the 6-13 ms)"}
    else:
        out["peer_gather_rows"] = {"unavailable": err or "failed on another rank"}
        err = None
    sync()
    # ---- (2) sharded full-catalog top-k: m_total queries in all, m_total / G contributed by every rank
    n_local = max(0, (rows - rank + world - 1) // world)
    m_local = max(1, m_total // world)
    sec = None
    mode_name = "tcgen05_f16"
    try:
        w = table.weight.detach()
        prep = ops.catalog_prepare_f16(w, n_local)
        mode = _lib.TOPK_TC16
        if not prep.fits:
            mode, prep, mode_name = _lib.TOPK_TC, None, "tcgen05_tf32"
        q = torch.randn(m_local, d, device=dev)
        # the shard-local kernel once on its own (same shapes as below, no collective): a rank whose kernel fails
        # says so at the agree() below instead of leaving the others inside the all-gather of the timed loop
        ops.catalog_topk(q.repeat(world, 1), w, k, n_items=n_local, id_base=rank, id_stride=world, mode=mode, prepared=prep)
        if str(dev).startswith("cuda"):
            torch.cuda.synchronize()

        q_all = torch.empty(world * m_local, d, device=dev)
        ids_all = torch.empty(world, world * m_local, k, dtype=torch.int64, device=dev)
        sc_all = torch.empty(world, world * m_local, k, dtype=torch.float32, device=dev)

        def ranked():
            # three collectives straight into their final layouts (no list gathers, no cat / stack copies)
            dist.all_gather_into_tensor(q_all, q)
            ids, sc = ops.catalog_topk(q_all, w, k, n_items=n_local, id_base=rank, id_stride=world, mode=mode, prepared=prep)
            dist.all_gather_into_tensor(ids_all.view(-1, k), ids)
            dist.all_gather_into_tensor(sc_all.view(-1, k), sc)
            return ops.topk_merge(ids_all, sc_all)
    except Exception as ex:                                               # noqa: BLE001
        err = "%s: %s" % (type(ex).__name__, str(ex)[:120])
    if agree(err):
        # the timed function contains collectives: every rank runs the same number of calls
        sec = max_over_ranks(timer(ranked, 3, warmup=1))
        m_all = m_local * world
        out["catalog_topk_16M"] = {
            "ms": sec * 1e3, "queries": m_all, "k": k, "mode": mode_name, "queries_per_s": m_all / sec,
            "tflops": 2.0 * m_all * rows * d / sec / 1e12,
            "frac_of_tensor_peak": 2.0 * m_all * rows * d / sec / 1e12 /
                                   ((peaks["bf16"] if mode_name == "tcgen05_f16" else peaks["bf16"] / 2) * world),
            "table_GBps": rows * d * (2 if mode_name == "tcgen05_f16" else 4) * ((m_all + 511) // 512) / sec / GB,
            "note": "all-gather of the queries (NCCL), per-shard fused top-k on the shard's rows (ids = rank + G * "
                    "local row), all-gather of the [M, k] lists (NCCL), psb_topk_merge; exact-mode ids and scores.  "
                    "table_GBps counts one shortlist-table pass per 512 queries (fp16 copy), over all ranks; tensor "
                    "peak = measured bf16 cuBLAS burst (half of it in tf32 mode) x ranks"}
    else:
        out["catalog_topk_16M"] = {"unavailable": err or "failed on another rank"}
        err = None
    # ---- (3) the TEM training step on the 16M-row item table, row-sharded over the ranks (peer-memory fetch / fold,
    #      one CUDA graph per rank) -- BASELINE configs[4] as a training step
    if pg is None or not str(dev).startswith("cuda"):
        return out
    del table
    torch.cuda.empty_cache()
    sync()
    step = None
    try:
        from prodsearch_b200.graph_step import GraphedTrainStep
        from prodsearch_b200.item_transformer import PeerShardedItemTransformerRanker
        from prodsearch_b200.optimizers import build_optim
        V, B = WORKLOAD["vocab_size"], WORKLOAD["batch_per_gpu"]
        args = model_args(WORKLOAD["dropout"])
        torch.manual_seed(666)
        with torch.device("cuda"):
            model = PeerShardedItemTransformerRanker(args, "cuda", V, rows, None, word_dists=synth.word_dists(V), peer=pg,
                                                     grad_mode="rowsparse")
        model.item_negative_sampler = "randint"      # the literal multinomial(ones(16M)) draw alone is ~10 ms (see the class)
        optim = build_optim(args, model)
        model.train()
        torch.manual_seed(666 + 7919 * rank)
        batches = []
        for it in range(8):
            b, _, _ = synth.tem_batch(B, rows, V, seed=700 + 100 * rank + it, permute=False)
            batches.append(argparse.Namespace(**{k_: (v.cuda() if torch.is_tensor(v) else v) for k_, v in vars(b).items()}))
        sample = argparse.Namespace(**vars(batches[0]))
        sample.query_word_idxs = torch.full((B, 12), V - 1, dtype=torch.int64)
        step = GraphedTrainStep(model, optim, sample, pad_values={"query_word_idxs": V - 1, "u_item_idxs": rows},
                                sync_grads=lambda: model.sync_grads(optim))
    except Exception as ex:                                               # noqa: BLE001
        err = "%s: %s" % (type(ex).__name__, str(ex)[:160])
    if agree(err):
        for it in range(3):
            step(batches[it])
        sync()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for it in range(5):
            step(batches[3 + it])
        s1.record()
        torch.cuda.synchronize()
        sec = max_over_ranks(s0.elapsed_time(s1) / 5 * 1e-3)
        out["train_step_16M"] = {
            "ms_per_step": sec * 1e3, "samples_per_s": B * world / sec, "batch_per_gpu": B,
            "launches_per_step": step.launches_per_replay, "item_negative_sampler": "randint",
            "note": "TEM step of the headline (batch 384 / GPU, dropout 0.1) with the 16M x 128 item table row-sharded "
                    "over the ranks: peer-memory fetch of the rows the batch needs (resting rows brought up to date on "
                    "the fly by the reader), compact gradient lists folded by their owners, one-shot all-reduce of the "
                    "replicated gradients, global clip norm, row-sparse Adam on the owned rows the step touched -- one "
                    "CUDA graph per rank; step cost independent of the table size (the dense owner-side sweep would move "
                    "%.1f GB per rank and step)" % ((rows // world) * d * 28 / 1e9)}
        try:
            pg.check_errors()
            # per-kernel split of the same step, launched eagerly with the library's profiler (all ranks take part: the
            # step contains cross-GPU barriers)
            def eager():
                loss = model(batches[0])
                model.zero_grad()
                loss.backward()
                model.sync_grads(optim)
                optim.step()
            for _ in range(2):
                eager()
            sync()
            _lib.profile_enable(True)
            for _ in range(3):
                eager()
            sync()
            kp = _lib.profile_dump()
            _lib.profile_enable(False)
            out["train_step_16M"]["kernels_us_per_step"] = {k_: round(v_[1] / 3 * 1e3, 1) for k_, v_ in
                                                            sorted(kp.items(), key=lambda kv: -kv[1][1])[:14]}
        except Exception as ex:                                           # noqa: BLE001
            out["train_step_16M"]["peer_error"] = str(ex)[:120]
    else:
        out["train_step_16M"] = {"unavailable": err or "failed on another rank"}
    return out


def summarize_regimes(line):
    """Compact per-kernel fractions inside ``roofline`` (the key the driver keeps): the bandwidth-regime kernels G1-G5
    on the 16M-row table, the 16M-row training step and the RTM step, next to the dominant kernel of the headline
    step."""
    rf = line.get("roofline")
    ex = line.get("extra") or {}
    if rf is None:
        return
    bw = ex.get("bandwidth_regime") or {}
    tab = {}
    for k in ("G1_gather_rows", "G4_gather_meanpool", "G3_ns_loss", "G2_scatter_reduce", "G2_reduce_presorted",
              "G2_scatter_reduce_zipf"):
        if isinstance(bw.get(k), dict) and "frac" in bw[k]:
            tab[k] = {"frac_of_hbm_peak": round(bw[k]["frac"], 3), "GBps": round(bw[k]["achieved"], 0)}
    c1 = bw.get("G5_catalog_topk_1M") or {}
    for k in ("tcgen05_f16_m384", "tcgen05_f16_m4096", "tcgen05_tf32_m24"):
        if isinstance(c1.get(k), dict) and "ms" in c1[k]:
            tab["G5_1M_" + k] = {"ms": round(c1[k]["ms"], 3), "frac_of_tensor_peak": round(c1[k].get("frac_of_tensor_peak", 0.0), 3),
                                 "frac_of_hbm_peak": round(c1[k].get("frac_of_hbm_peak", 0.0), 3)}
    for key, name in (("G5_catalog_topk_16M_m24", "G5_16M_m24"), ("G5_catalog_topk_16M_m384", "G5_16M_m384"),
                      ("G5_catalog_topk_16M", "G5_16M_m4096")):
        c16 = bw.get(key) or {}
        if "ms" in c16:
            tab[name] = {"ms": round(c16["ms"], 3), "tflops": round(c16["tflops"], 0),
                         "frac_of_tensor_peak": round(c16["frac_of_tensor_peak"], 3),
                         "frac_of_hbm_peak": round(c16.get("frac_of_hbm_peak", 0.0), 3)}
    t16 = ex.get("train_16M") or {}
    for m in ("rowsparse", "rowsparse_aged", "rowsparse_multinomial", "dense"):
        if isinstance(t16.get(m), dict) and "ms_per_step" in t16[m]:
            tab["train_16M_" + m] = {"ms_per_step": round(t16[m]["ms_per_step"], 3)}
    rtm = ex.get("rtm_configs2") or {}
    for enc in ("pv", "pvc"):
        if isinstance(rtm.get(enc), dict) and "ms_per_step" in rtm[enc]:
            e = {"ms_per_step": round(rtm[enc]["ms_per_step"], 3)}
            if "gather_rows_kernel" in rtm[enc]:
                e["gather_rows_kernel_frac_of_hbm_peak"] = round(rtm[enc]["gather_rows_kernel"]["frac"], 3)
            if "meanpool_kernel" in rtm[enc]:      # 16 MB word table: served from L2, so requested bytes exceed the HBM peak
                e["meanpool_kernel_requested_GBps"] = round(rtm[enc]["meanpool_kernel"]["achieved"], 0)
                e["meanpool_kernel_requested_over_hbm_peak_L2_resident"] = round(rtm[enc]["meanpool_kernel"]["frac"], 3)
            tab["rtm_" + enc] = e
    sh = ex.get("sharded_16M") or {}
    pgr = sh.get("peer_gather_rows") or {}
    if "nvlink_GBps_per_rank" in pgr:
        tab["peer_gather_rows_16M"] = {"ms": round(pgr["ms"], 3), "nvlink_GBps_per_gpu": round(pgr["nvlink_GBps_per_rank"], 0),
                                       "frac_of_nvlink_peak": round(pgr.get("frac_of_nvlink_peak", 0.0), 3)}
    c16s = sh.get("catalog_topk_16M") or {}
    if "ms" in c16s:
        tab["sharded_catalog_16M_m4096"] = {"ms": round(c16s["ms"], 3), "frac_of_tensor_peak_all_gpus": round(c16s["frac_of_tensor_peak"], 3)}
    t16s = sh.get("train_step_16M") or {}
    if "ms_per_step" in t16s:
        tab["sharded_train_step_16M"] = {"ms_per_step": round(t16s["ms_per_step"], 3)}
    # the encoder's kernels in the headline step (eager per-launch times of the profiled pass, cold L2; the ncu capture of
    # the same kernels is profiles/r02X_tails_full_raw.csv: tensor pipe active 19 % / 15 % of the cluster kernels' cycles)
    kn = line.get("kernels") or {}
    for k, name in (("tail_fused_tc_kernel", "N1_tail_fwd_tcgen05"), ("tail_bwd_fused_tc_kernel", "N1_tail_bwd_tcgen05"),
                    ("tail_fwd_kernel", "N1_tail_fwd_ffma"), ("tail_bwd_kernel", "N1_tail_bwd_ffma"), ("wgrad_kernel", "N1_wgrad_ffma")):
        if isinstance(kn.get(k), dict) and "frac" in kn[k]:
            tab[name] = {"us_per_launch": round(kn[k]["avg_launch_us"], 1), "launches_per_step": kn[k]["launches_per_step"],
                         "frac_of_tf32_peak": round(kn[k]["frac"], 4)}
    rf["regimes"] = tab
    rf["regimes_note"] = ("bandwidth regime = 16M x 128 fp32 table (8.2 GB >> L2); fractions of the measured peaks "
                          "(MEASURED_PEAKS.json); full entries under extra")


def run_b200_arm(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl b200 needs a GPU (there is no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        # one launching thread per rank on its own cores: the replayed step is ~1 ms, so a descheduled host thread
        # on one rank stalls every rank at the next cross-GPU barrier
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            os.sched_setaffinity(0, set(cores[local * per:(local + 1) * per]) or set(cores))
        except (AttributeError, OSError):
            pass
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from prodsearch_b200 import _lib, ops, synth
    from prodsearch_b200.item_transformer import ItemTransformerRanker, ShardedItemTransformerRanker
    from prodsearch_b200.optimizers import build_optim
    peaks = load_peaks()
    args = model_args(a.dropout)
    P, V, B = WORKLOAD["product_size"], WORKLOAD["vocab_size"], WORKLOAD["batch_per_gpu"]
    torch.manual_seed(666)
    transport = "local"
    if world > 1:
        # item + word tables row-sharded over the ranks.  Preferred transport: NVLink peer memory (P2P loads inside
        # the kernels, whole step = one CUDA graph per rank); if CUDA IPC is unavailable, NCCL all-to-all (eager).
        from prodsearch_b200 import peer
        pg = None if a.transport == "nccl" else peer.try_create()
        if pg is not None:
            from prodsearch_b200.item_transformer import PeerShardedItemTransformerRanker
            model = PeerShardedItemTransformerRanker(args, "cuda", V, P, None, word_dists=synth.word_dists(V), peer=pg)
            transport = "nvlink-peer"
        else:
            model = ShardedItemTransformerRanker(args, "cuda", V, P, None, word_dists=synth.word_dists(V))
            transport = "nccl-all-to-all"
    else:
        model = ItemTransformerRanker(args, "cuda", V, P, None, word_dists=synth.word_dists(V), grad_mode=a.grad_mode)
    # the step's negatives by inverse CDF on the device generator: the literal torch.multinomial calls are not
    # reproducible on CUDA, and with them a run's results would not be a function of its arguments (--dump-outputs)
    model.reproducible_draws = True
    optim = build_optim(args, model)
    model.train()
    torch.manual_seed(666 + 7919 * rank)      # per-rank negatives / dropout masks from here on
    n_total = a.warmup + a.steps
    host, devb = [], []
    for it in range(n_total):
        b, _, _ = synth.tem_batch(B, P, V, seed=666 + 1000 * rank + it)
        hb = argparse.Namespace(**{k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in vars(b).items()})
        host.append(hb)
        devb.append(argparse.Namespace(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(b).items()}))
    h2d = sum(v.numel() * v.element_size() for v in vars(host[0]).values() if torch.is_tensor(v))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def eager_step(batch):
        loss = model(batch)
        model.zero_grad()
        loss.backward()
        if transport == "nvlink-peer":
            model.sync_grads(optim)
        elif world > 1:
            model.sync_grads()
        optim.step()
        return loss

    graphed = None
    if transport in ("local", "nvlink-peer") and not a.eager:
        # the whole step (fwd + bwd + gradient sinks + clipped Adam) replays as ONE CUDA graph; batches are
        # copied into its static input buffers (query matrix right-padded to the widest batch)
        from prodsearch_b200.graph_step import GraphedTrainStep
        wq = max(b.query_word_idxs.shape[1] for b in host)
        sample = argparse.Namespace(**vars(host[0]))
        sample.query_word_idxs = torch.full((B, wq), V - 1, dtype=torch.int64)
        wq = max(wq, 12)      # synthetic queries have at most 12 words: the same static shape on every rank
        sample.query_word_idxs = torch.full((B, wq), V - 1, dtype=torch.int64)
        graphed = GraphedTrainStep(model, optim, sample, pad_values={"query_word_idxs": V - 1, "u_item_idxs": P},
                                   sync_grads=(lambda: model.sync_grads(optim)) if transport == "nvlink-peer" else None)

    def step(batch):
        return graphed(batch) if graphed is not None else eager_step(batch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local if rank == 0 else None).start()     # before the warm-up: see the class docstring
    for it in range(a.warmup):
        step(devb[it])
    # ---- timed region 1: device-resident batches, CUDA events per step, L2 flushed between steps
    barrier()
    if transport == "nvlink-peer":
        pg.wait_cycles.zero_()
    l0 = _lib.launch_count()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps)]
    clocks.begin()
    t_host = time.perf_counter()
    for it in range(a.steps):
        flush.zero_()
        starts[it].record()
        loss = step(devb[a.warmup + it])
        ends[it].record()
    host_enqueue_ms = (time.perf_counter() - t_host) / a.steps * 1e3     # host time to enqueue one step
    barrier()
    clocks.end()
    barrier_wait = None
    if transport == "nvlink-peer":
        # SM cycles every rank spent inside the three cross-GPU barriers of a step (waiting for the slowest peer)
        wc = pg.wait_cycles.to(torch.float64) / a.steps / 1965.0      # us per step at the nominal SM clock
        allw = [torch.empty_like(wc) for _ in range(world)]
        dist.all_gather(allw, wc)
        st_ = torch.stack(allw)
        mine = torch.tensor([sum(s_.elapsed_time(e_) for s_, e_ in zip(starts, ends)) / a.steps, host_enqueue_ms],
                            device="cuda", dtype=torch.float64)
        allm = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allm, mine)
        barrier_wait = {"us_per_step_by_rank": [[round(float(x), 1) for x in r_[:3]] for r_ in st_],
                        "slots": ["A: step start", "B: gradient lists complete", "C: shard norms published"],
                        "device_ms_per_step_by_rank": [round(float(x[0]), 4) for x in allm],
                        "host_enqueue_ms_per_step_by_rank": [round(float(x[1]), 4) for x in allm]}
        pg.check_errors()
    launches = _lib.launch_count() - l0
    if graphed is not None:       # replays do not pass through the library's host counter
        launches = graphed.launches_per_replay * a.steps
    dev_sec = sum(s.elapsed_time(e) for s, e in zip(starts, ends)) * 1e-3
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, loss, model)
    # ---- timed region 2: end to end from pinned host batches (H2D + step + loss.item()).  The host batches are collated
    #      into the graph's input layout beforehand (GraphedTrainStep.pack: one pinned buffer per batch, like pinning --
    #      not timed), so a step's inputs cross PCIe in one copy
    packed = [graphed.pack(host[a.warmup + it]) for it in range(a.steps)] if graphed is not None else None
    if packed is not None:
        h2d = packed[0].buf.numel()
    barrier()
    e2e_sec = 0.0
    for it in range(a.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hb = host[a.warmup + it]
        if graphed is not None:
            float(step(packed[it]).item())  # pinned, packed host batch -> static device buffers (ONE H2D copy) -> replay -> loss
        else:
            db = argparse.Namespace(**{k: (v.cuda(non_blocking=True) if torch.is_tensor(v) else v) for k, v in vars(hb).items()})
            float(step(db).item())
        e2e_sec += time.perf_counter() - t0
    barrier()
    clocks.stop()
    if world > 1:
        t = torch.tensor([dev_sec, e2e_sec], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_sec, e2e_sec = float(t[0]), float(t[1])
    # ---- per-KERNEL timing inside the same step: a separate eager pass with the library's own profiler
    #      (CUDA events on the launching stream around every hand-written kernel, L2 flushed between steps);
    #      all ranks take part because the sharded step contains cross-GPU barriers
    n_prof = min(a.steps, 10)
    for it in range(2):
        eager_step(devb[it])      # warm-up batches: there are at least 3 of them, and --steps may be 1
    barrier()
    _lib.profile_enable(True)
    for it in range(n_prof):
        flush.zero_()
        eager_step(devb[a.warmup + it])
    barrier()
    kprof = _lib.profile_dump()
    _lib.profile_enable(False)
    do_sharded = world > 1 and transport == "nvlink-peer" and not a.no_extra
    if rank != 0:
        if do_sharded:      # every rank takes part; a rank that hangs leaves after the same time-out as rank 0
            def take_part():
                try:
                    sharded_regime(peaks, pg, rank, world)
                except Exception:                                     # noqa: BLE001
                    # a rank that leaves now (non-zero exit: torchrun tears the job down; exit 0: NCCL reports the lost
                    # peer to the others) could take rank 0 down before it has printed the headline line -- stay until
                    # the watchdog ends this process, which is when rank 0's own watchdog prints the line
                    while True:
                        time.sleep(1.0)
            guarded(take_part, a.extra_timeout + 5, lambda: None)
        if world > 1:
            try:
                dist.destroy_process_group()
            except Exception:                                         # noqa: BLE001 -- after a failed collective
                pass
        return
    d = WORKLOAD["embedding_size"]
    K, L, W, F = WORKLOAD["neg_per_pos"], WORKLOAD["uprev_review_limit"], 1, WORKLOAD["ff_size"]
    hb = devb[a.warmup]
    Wq = int(hb.query_word_idxs.shape[1])
    ntok = int(B + (hb.u_item_idxs != P).sum().item())
    C = 1 + K
    n_item_slots = B * (L + 2 + K)            # history + target (loss) + negatives + target (item->word anchor)
    n_word_slots = B * (Wq + W + W * K)
    n_param = sum(p.numel() for p in model.parameters() if p.grad is not None)
    row = d * 4 + 8
    tail_flop = 2.0 * B * C * (d * d + 2 * d * F)
    # ALGORITHMIC work per STEP of every hand-written kernel (DESIGN.md section 4): ("hbm", bytes) | ("tensor", flop)
    alg = {
        "meanpool_kernel": ("hbm", B * Wq * row + B * d * 4 * 2 + d * d * 4),
        "fs_bwd_kernel": ("hbm", B * d * 4 * 4 + d * d * 4 * 2),
        "token_weights_kernel": ("hbm", B * Wq * 12),
        "gather_rows_kernel": ("hbm", B * (d * 4 * 2 + 8)),
        "ns_loss_fast_kernel": ("hbm", B * (1 + K) * row + B * d * 4 * 2 + B * K * d * 4 * 2      # score + loss tail
                                + B * W * (1 + K) * row + B * d * 4 * 2),                         # item -> words
        "ns_loss_w1_kernel": ("hbm", B * (1 + K) * row + B * d * 4 * 2 + B * K * d * 4 * 2
                              + B * W * (1 + K) * row + B * d * 4 * 2),
        "small_sort_segments_kernel": ("hbm", (n_item_slots + n_word_slots) * 8),
        "seg_reduce_kernel": ("hbm", (n_item_slots + n_word_slots) * row),
        "seg_fixup_kernel": ("hbm", 0),
        "sqnorm_partial_kernel": ("hbm", n_param * 4),
        "adam_kernel": ("hbm", n_param * 28),
        "embed_kernel": ("hbm", ntok * d * 4 * 3),
        "embed_bwd_kernel": ("hbm", ntok * d * 4 * 3),
        "peer_gather_rows_kernel": ("hbm", (n_item_slots - B + n_word_slots) * (d * 4 * 2 + 8)),
        "peer_fold_rows_kernel": ("hbm", (n_item_slots + n_word_slots) * (d * 4 * 3 + 4)),
        "peer_allreduce_kernel": ("hbm", 0),
        "rows_gemm_kernel": ("tensor", 2.0 * (ntok * d * 2 * d + B * d * d) * 2),    # K|V and q projections + their dgrads
        "gemm3_tf32_kernel": ("tensor", 2.0 * (ntok * d * 2 * d + B * d * d)),       # PSB_ENC_TC=1: forward K|V and q projections
        "gemm3_out_proj_ln_kernel": ("tensor", 2.0 * B * C * d * d),                 # PSB_ENC_TC=2: the forward tail as three GEMMs
        "gemm3_ffn_up_kernel": ("tensor", 2.0 * B * C * d * F),
        "gemm3_ffn_down_ln_kernel": ("tensor", 2.0 * B * C * d * F),
        "attn_fwd_kernel": ("tensor", 2.0 * 2 * ntok * d),
        "tail_fwd_kernel": ("tensor", tail_flop),                                    # PSB_ENC_TC=0: fp32 FFMA tails
        "tail_bwd_kernel": ("tensor", tail_flop),                                    # dgrad half; dW is wgrad_kernel
        "tail_fused_tc_kernel": ("tensor", tail_flop),                               # default: the tails on tcgen05 (3xTF32)
        "tail_bwd_fused_tc_kernel": ("tensor", tail_flop),
        "tail_ctx_kernel": ("hbm", B * C * d * 4 * 3 + ntok * (d * 4 + 32)),         # ctx + its hi / lo parts out, V rows + P in
        "tail_attn_bwd_kernel": ("hbm", B * C * d * 4 * 2 + ntok * 2 * d * 4 * 2 + B * d * 4 * 3),
        "count_sort_segments_kernel": ("hbm", (n_item_slots + n_word_slots) * 8),
        "transpose_kernel": ("hbm", (3 * d * d + 2 * d * F) * 4 * 5),
        "wgrad_kernel": ("tensor", tail_flop + 2.0 * (ntok * d * 2 * d + B * d * d)),
    }
    sm_mhz = (clocks.summary().get("sm_mhz") or 1965.0)
    ffma_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    tf32_peak = peaks["bf16"] / 2.0
    kernels = {}
    for name, (cnt, tot_ms, mn, mx) in kprof.items():
        per_step_ms = tot_ms / n_prof
        ent = {"launches_per_step": cnt / n_prof, "ms_per_step": round(per_step_ms, 5),
               "avg_launch_us": round(tot_ms / cnt * 1e3, 3)}
        if name in alg and alg[name][1] > 0:
            bound, amount = alg[name]
            if bound == "hbm":
                ach = amount / (per_step_ms * 1e-3) / 1e9
                ent.update(bound="hbm", algorithmic_bytes_per_step=int(amount), achieved=round(ach, 2), unit="GB/s",
                           peak=peaks["hbm"], frac=round(ach / peaks["hbm"], 5))
            else:
                ach = amount / (per_step_ms * 1e-3) / 1e12
                ent.update(bound="tensor", algorithmic_flop_per_step=amount, achieved=round(ach, 3), unit="TFLOP/s",
                           peak=tf32_peak, frac=round(ach / tf32_peak, 5), frac_of_fp32_ffma_peak=round(ach / ffma_peak, 4))
        kernels[name] = ent
    roofline = None
    if kernels:
        # the cross-GPU barrier kernels are excluded: in this eager, per-kernel-timed pass they absorb the host-launch
        # skew between the ranks (hundreds of us), not device work; what the barriers cost inside the replayed graph is
        # config.peer_barrier_wait (clock64 cycles every rank spent waiting, 8-20 us per barrier)
        # ... and so are the one-CTA index sorts: the step launches them on side streams when its forward pass ends, next
        # to the whole backward pass (functional.RowGradSink.mark_forward_end), so their launch time is not step time
        # (sum of kernel times per step ~0.53 ms, step 0.31 ms); they stay in `kernels`
        side = ("peer_barrier_kernel", "peer_norm_exchange_kernel", "count_sort_segments_kernel", "small_sort_segments_kernel")
        cands = {k_: v_ for k_, v_ in kernels.items() if k_ not in side} or kernels
        name, ent = max(cands.items(), key=lambda kv: kv[1]["ms_per_step"])
        roofline = {"kernel": name, "bound": ent.get("bound", "hbm"), "achieved": ent.get("achieved"),
                    "peak": ent.get("peak"), "unit": ent.get("unit"), "frac": ent.get("frac"), "traffic": None,
                    "peak_source": peaks["src"] + (" bf16 cuBLAS burst / 2 (TF32 rate)" if ent.get("bound") == "tensor" else " copy bandwidth"),
                    "launch_us": ent["avg_launch_us"], "launches_per_step": ent["launches_per_step"],
                    "regime": "dominant hand-written kernel of the batch-384 step (%.0f%% of the %.3f ms of kernel time "
                              "per step), timed per launch with CUDA events in an eager pass with a cold L2.  The step moves "
                              "~25 MB and ~3 GFLOP: every kernel is latency-bound at this size; extra.bandwidth_regime has "
                              "the same gather / loss / scatter kernels on a 16M-row table where the roofline binds."
                              % (100.0 * ent["ms_per_step"] / sum(k["ms_per_step"] for k in cands.values()),
                                 sum(k["ms_per_step"] for k in cands.values()))}
        tr = load_traffic().get("step", {}).get(name)
        if tr is not None:
            roofline["traffic"] = tr["dram_bytes_per_launch"]
            roofline["traffic_source"] = "ncu dram__bytes_read.sum + dram__bytes_write.sum, one launch, " + tr["source"]
        if ent.get("bound") == "tensor" and "_tc_" in name:
            roofline["note"] = ("three chained products (B*(1+K) rows x 128 -> 512 -> 128) on tcgen05 as 3xTF32 (three MMAs per "
                                "k-step to hold the 1e-5 parity bar: the hardware rate for ALGORITHMIC flops is a third of "
                                "the TF32 peak) in one cluster kernel on 72 of the 148 SMs; the launch is a latency chain "
                                "(TMA -> MMA -> epilogue, three times) at this size, see profiles/ for its phase trace")
        elif ent.get("bound") == "tensor":
            roofline["note"] = ("GEMM-shaped but computed in fp32 FFMA on CUDA cores; %.1f%% of the fp32 FFMA peak "
                                "(%.1f TFLOP/s at the sampled clock)"
                                % (100.0 * ent.get("frac_of_fp32_ffma_peak", 0.0), ffma_peak))
    cpu = None
    if world == 1 and not a.no_cpu:
        sec, cores = cpu_reference_step_time(a.cpu_steps, 2, a.dropout)
        cpu = {"value": B / sec, "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": "%d TEM train steps of batch 384 (fwd+bwd+clipped Adam) on the oracle port, %.0f ms/step"
                         % (a.cpu_steps, sec * 1e3)}
        try:        # the other CPU timings of SURVEY.md 8(d): PV step, catalog ranking, gather / scatter-add (~20 s)
            cpu["others"] = cpu_reference_others()
        except Exception as ex:                                       # noqa: BLE001 -- reported, never fatal
            cpu["others"] = {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:120])}
    value = B * a.steps * world / dev_sec
    line = {
        "metric": "tem_train_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": dev_sec / a.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(WORKLOAD, workload="BASELINE configs[1]: TEM item_transformer train step, batch 384/GPU",
                       dropout=a.dropout, l2="flushed between timed steps (256 MiB write), flush not timed",
                       parallelism="dp%d, item/word tables %s" % (world, "row-sharded (%s)" % transport if world > 1 else "local"),
                       launch="CUDA graph replay of the whole step" if graphed is not None else "eager",
                       encoder_products=("3xTF32 on tcgen05, fp32 accumulation in TMEM (PSB_ENC_TC=%s): within 1e-6 of the fp32 "
                                         "FFMA kernels, which PSB_ENC_TC=0 selects" % os.environ.get("PSB_ENC_TC", "4 (default)")),
                       peer_barrier_wait=barrier_wait),
        "clocks": clocks.summary(),
        "e2e": {"value": B * a.steps * world / e2e_sec, "unit": "samples/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "ms_per_step": e2e_sec / a.steps * 1e3},
        "gpu_launches": launches, "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu,
        "extra": None,
    }
    if world == 1 and not a.no_extra:
        # everything above is final; the 16M-row section (seconds of GPU time when healthy) runs last, under the same
        # watchdog as the multi-GPU one: its 16M-row catalog entry had no GPU run when it was written
        def give_up_bw():
            line["extra"] = {"bandwidth_regime": {"unavailable": "no result after %d s (watchdog)" % a.extra_timeout}}
            print(json.dumps(line))
        try:
            line["extra"] = {"bandwidth_regime": guarded(lambda: bandwidth_regime(peaks), a.extra_timeout, give_up_bw),
                             "table": "16M x 128 fp32 (8.2 GB), inputs >> L2, no flush needed"}
        except Exception as ex:                                       # noqa: BLE001 -- the headline line must appear
            line["extra"] = {"bandwidth_regime": {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:160])}}
        summarize_regimes(line)
        for key, fn in (("train_16M", train_16m_regime), ("rtm_configs2", rtm_regime)):
            def give_up_x(key=key):
                line["extra"][key] = {"unavailable": "no result after %d s (watchdog)" % a.extra_timeout}
                print(json.dumps(line))
            try:
                line["extra"][key] = guarded(lambda fn=fn: fn(peaks), a.extra_timeout, give_up_x)
            except Exception as ex:                                   # noqa: BLE001
                line["extra"][key] = {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:160])}
        summarize_regimes(line)
    if do_sharded:
        # everything above is final; the 16M-row section runs last, under a watchdog that prints the line without it
        def give_up():
            line["extra"] = {"sharded_16M": {"unavailable": "no result after %d s (watchdog)" % a.extra_timeout}}
            print(json.dumps(line))
        try:
            line["extra"] = {"sharded_16M": guarded(lambda: sharded_regime(peaks, pg, rank, world), a.extra_timeout,
                                                    give_up)}
            summarize_regimes(line)
        except Exception as ex:                                       # noqa: BLE001 -- the headline line must appear
            line["extra"] = {"sharded_16M": {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:160])}}
            # the other ranks may be inside a collective this rank has left: no orderly shutdown is possible (it could
            # block on them); they leave through their own watchdogs
            print(json.dumps(line))
            sys.stdout.flush()
            os._exit(0)
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        try:
            dist.destroy_process_group()
        except Exception:                                             # noqa: BLE001 -- after a failed collective
            pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dropout", type=float, default=WORKLOAD["dropout"])
    ap.add_argument("--cpu-steps", type=int, default=8)
    ap.add_argument("--no-extra", action="store_true", help="skip the 16M-row bandwidth-regime section")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-variants", action="store_true", dest="no_variants", help="accepted and ignored (round-1 flag)")
    ap.add_argument("--extra-timeout", type=int, default=120, dest="extra_timeout",
                    help="seconds the 16M-row section (extra) may take before the line is printed without it")
    ap.add_argument("--transport", default="auto", choices=["auto", "nccl"],
                    help="N>1: auto = NVLink peer memory when CUDA IPC works, else NCCL all-to-all; nccl forces the latter")
    ap.add_argument("--grad-mode", default="dense", choices=["dense", "rowsparse"], dest="grad_mode",
                    help="N=1: dense = the reference's dense table gradients + dense Adam sweep; rowsparse = compact row "
                         "gradients + row-sparse lazily caught-up Adam (dense-equivalent results, O(rows touched))")
    ap.add_argument("--eager", action="store_true", help="launch the step kernel by kernel instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", dest="dump_outputs",
                    help="b200 arm: after the timed steps, write the loss of the last one and the parameters it left as "
                         "DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes what the b200 arm's timed step computed; --impl %s has none" % a.impl)
    a.warmup = max(a.warmup, 3)
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_b200_arm(a)


if __name__ == "__main__":
    main()
