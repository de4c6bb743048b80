"""TEM: ``ItemTransformerRanker`` (reference models/item_transformer.py) on the sm_100a hot path.

Drop-in for the reference class behind ``model(batch)`` / ``model.test(batch)``
(trainer.py:74,:201): same constructor, same state_dict keys, same ``ps_loss`` /
``item_loss`` / ``clear_loss()`` bookkeeping, same RNG draw order (item negatives, then word
negatives: item_transformer.py:447,:268).  Implemented paths: ``forward_dotproduct`` (:440),
``test_dotproduct`` (:111), ``item_to_words`` (:260) -- the defaults of the reference
(``--use_dot_prod True``).  The ``*_trans`` / ``*_attn`` / ``*_seq`` variants are out of scope
(SURVEY.md 2.1 C1).  New, additive: ``rank_catalog`` (full-catalog top-k without the
[M, N] matrix) and ``encode_queries``.
"""
import torch
import torch.nn as nn

from . import _lib
from . import functional as F_
from . import ops
from .text_encoder import AVGEncoder, FSEncoder
from .transformer import TransformerEncoder


class ItemTransformerRanker(F_.LazyFlushMixin, nn.Module):
    overlap_query_pooling = True     # query pooling on a side stream under the encoder's plan / transpose kernels
    overlap_item_to_words = True     # item -> word loss kernels on a side stream next to the encoder
    fused_loss_tail = True           # training under dropout: ranking loss on the encoder's output block in place
    # Item negatives (item_transformer.py:447: torch.multinomial(ones(P), B * K, replacement=True)).  "multinomial" is
    # that literal call -- bit-identical ids on the same device generator (tests/test_gpu_parity_r2.py).  Its cost is
    # O(P) per draw: ATen renormalises the distribution with ONE thread block and rebuilds the CDF every call --
    # 15 us at P = 18k, ~10 ms at P = 16M, measured (profiles/r02k_bench.json: the whole 16M-row step was 10.9 ms
    # with it).  "randint": torch.randint(0, P) -- the same uniform distribution, O(1), a different random stream;
    # for catalogs where the literal call is the bottleneck.
    item_negative_sampler = "multinomial"
    # Opt-in for runs that must repeat bit for bit.  The literal torch.multinomial calls (item and word negatives) are
    # not reproducible on CUDA: every call rebuilds the distribution's CDF with a float32 scan whose rounding varies from
    # run to run (torch lists CUDA cumsum as nondeterministic), and a draw next to a bucket boundary then takes the
    # neighbouring id (profiles/multinomial_repro.py).  With reproducible_draws the same distributions are sampled by
    # inverse CDF instead: each constant distribution's CDF is summed once in float64 on the host, and a draw is one
    # torch.rand on the device generator plus a search -- a different random stream from the reference's.
    reproducible_draws = False

    def __init__(self, args, device, vocab_size, product_size, vocab_words, word_dists=None,
                 grad_mode="dense"):
        super().__init__()
        if args.model_name != "item_transformer" or not args.use_dot_prod:
            raise NotImplementedError("only the default TEM path (item_transformer + use_dot_prod) is built")
        if getattr(args, "pretrain_emb_dir", "") or getattr(args, "pretrain_up_emb_dir", ""):
            import os
            if os.path.exists(args.pretrain_emb_dir) or os.path.exists(args.pretrain_up_emb_dir):
                raise NotImplementedError("pretrained embedding files: build the table with data_files.pretrained_word_table "
                                          "and copy it into word_embeddings.weight (requires_grad False to freeze it)")
        self.args = args
        self.device = device
        self.train_review_only = args.train_review_only
        self.embedding_size = args.embedding_size
        self.vocab_words = vocab_words
        self.word_dists = None
        if word_dists is not None:
            self.word_dists = torch.as_tensor(word_dists, dtype=torch.float32, device=device)
        self.prod_dists = torch.ones(product_size, device=device)
        self.prod_pad_idx = product_size
        self.word_pad_idx = vocab_size - 1
        self.seg_pad_idx = 3
        self.emb_dropout = args.dropout
        d = self.embedding_size
        self.product_emb = nn.Embedding(product_size + 1, d, padding_idx=self.prod_pad_idx)
        if args.sep_prod_emb:
            self.hist_product_emb = nn.Embedding(product_size + 1, d, padding_idx=self.prod_pad_idx)
        self.product_bias = nn.Parameter(torch.zeros(product_size + 1), requires_grad=True)
        self.word_bias = nn.Parameter(torch.zeros(vocab_size), requires_grad=True)
        self.word_embeddings = nn.Embedding(vocab_size, d, padding_idx=self.word_pad_idx)
        self.transformer_encoder = TransformerEncoder(d, args.ff_size, args.heads, args.dropout, args.inter_layers)
        if args.query_encoder_name == "fs":
            self.query_encoder = FSEncoder(d, self.emb_dropout)
        else:
            self.query_encoder = AVGEncoder(d, self.emb_dropout)
        self.seg_embeddings = nn.Embedding(4, d, padding_idx=self.seg_pad_idx)
        self.initialize_parameters()
        self.to(device)
        self.grad_mode = grad_mode
        self._make_sinks()
        self.injected_negatives = None      # (neg_item_idxs [B,K], neg_word_idxs [B*W*K]) for parity runs
        self._ps_acc = None
        self._item_acc = None

    # ---- bookkeeping the trainer reads (trainer.py:88-98) ---------------------------------
    def _make_sinks(self):
        # nn.Embedding(padding_idx) zeroes the pad row's gradient -> drop_idx
        self.item_sink = F_.RowGradSink(self.product_emb.weight, self.prod_pad_idx, self.product_bias,
                                        self.grad_mode)
        self.hist_sink = (F_.RowGradSink(self.hist_product_emb.weight, self.prod_pad_idx, None, self.grad_mode)
                          if self.args.sep_prod_emb else self.item_sink)
        self.word_sink = F_.RowGradSink(self.word_embeddings.weight, self.word_pad_idx, self.word_bias,
                                        self.grad_mode)

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        if hasattr(self, "item_sink"):
            self._make_sinks()              # parameters may have been re-created (.to / .cuda)
        return out

    @property
    def ps_loss(self):
        return 0 if self._ps_acc is None else float(self._ps_acc)

    @property
    def item_loss(self):
        return 0 if self._item_acc is None else float(self._item_acc)

    def clear_loss(self):
        if self._ps_acc is not None:
            self._ps_acc.zero_()
            self._item_acc.zero_()

    def load_cp(self, pt, strict=True):
        self.load_state_dict(pt["model"], strict=strict)

    def initialize_parameters(self, logger=None):
        """item_transformer.py:576-586: N(0,1) word and segment tables (pad row included),
        default nn.Embedding init for product tables (pad row zero)."""
        nn.init.normal_(self.word_embeddings.weight)
        nn.init.normal_(self.seg_embeddings.weight)
        self.query_encoder.initialize_parameters(logger)
        self.transformer_encoder.initialize_parameters(logger)

    # ---- shared front half -----------------------------------------------------------
    def encode_queries(self, query_word_idxs, u_item_idxs, copies=1, hist=None):
        """Query encoder + [query, purchased items] sequence through the transformer, read at ``out_pos``
        (item_transformer.py:449-484 / :118-140) -> [B*copies, d], copy-minor.  The history rows are
        gathered inside the fused encoder kernels.  ``hist`` = (weight, sink, remapped idx, pad idx) when
        the item table is sharded and the rows live in a fetched mini table."""
        # the query pooling runs on a side stream; the encoder call enqueues its token plan and weight transposes
        # (which do not read the pooled queries) and waits for the event only before the kernel that does
        side = ready = None
        if self.overlap_query_pooling and self.word_embeddings.weight.is_cuda:
            if getattr(self, "_q_stream", None) is None:
                self._q_stream = torch.cuda.Stream(device=self.word_embeddings.weight.device)
                self._q_ready = torch.cuda.Event()
            side, ready = self._q_stream, self._q_ready
        q_emb = self.query_encoder.encode_indices(self.word_embeddings.weight, query_word_idxs, self.word_sink,
                                                  pad_idx=self.word_pad_idx, stream=side)
        if ready is not None:
            ready.record(side)
        if hist is None:
            hist_w = self.hist_product_emb.weight if self.args.sep_prod_emb else self.product_emb.weight
            hist = (hist_w, self.hist_sink, u_item_idxs, self.prod_pad_idx)
        out_pos = -1 if self.args.use_item_pos else 0
        return self.transformer_encoder.encode_position(
            first=q_emb.contiguous(), table=hist[0], idx=hist[2], sink=hist[1], pad_idx=hist[3],
            use_pos=self.args.use_pos_emb, out_pos=out_pos, copies=copies, first_ready=ready)

    def _resolve_item_rows(self, target_prod_idxs, neg_item_idxs, u_item_idxs):
        """(item weight, item sink, target idx, negative idx, hist triple or None) of this step.
        Single GPU: the full local table.  The sharded subclass fetches a mini table instead."""
        return self.product_emb.weight, self.item_sink, target_prod_idxs, neg_item_idxs, None

    # ---- training -----------------------------------------------------------------------
    def forward(self, batch_data, train_pv=False):
        return self.forward_dotproduct(batch_data)

    def _draw_negatives(self, B, W, K):
        if self.injected_negatives is not None:
            neg_items, neg_words = self.injected_negatives
            return neg_items.view(B, K), neg_words.view(B, W, K)
        # items first, then words: the reference's call order (item_transformer.py:447, :268)
        if self.item_negative_sampler == "randint":
            neg_items = torch.randint(0, self.prod_pad_idx, (B, K), device=self.prod_dists.device)
        else:
            neg_items = self._multinomial("prod_dists", B * K).view(B, K)
        neg_words = self._multinomial("word_dists", B * W * K).view(B, W, K)
        return neg_items, neg_words

    def _multinomial(self, name, n):
        """n draws with replacement from the constant distribution ``self.<name>`` (see reproducible_draws)."""
        dist = getattr(self, name)
        if not self.reproducible_draws:
            return torch.multinomial(dist, n, replacement=True)
        cache = self.__dict__.setdefault("_cdfs", {})
        if name not in cache or cache[name][0] is not dist:
            cdf = torch.cumsum(dist.detach().to("cpu", torch.float64), 0)
            cache[name] = (dist, (cdf / cdf[-1]).to(dist.device))
        cdf = cache[name][1]
        # u in [0, 1) and cdf[-1] == 1: the id is the number of CDF entries <= u, so zero-probability ids (the pad
        # word) are never drawn
        return torch.searchsorted(cdf, torch.rand(n, dtype=torch.float64, device=cdf.device), right=True)

    def forward_dotproduct(self, batch_data, train_pv=False):
        query_word_idxs = batch_data.query_word_idxs
        target_prod_idxs = batch_data.target_prod_idxs
        u_item_idxs = batch_data.u_item_idxs
        pos_iword_idxs = batch_data.pos_iword_idxs
        B, _ = u_item_idxs.shape
        K = self.args.neg_per_pos
        W = pos_iword_idxs.shape[1]
        # Neither the negatives nor the item -> word objective are needed by the encoder: the two torch.multinomial
        # chains (renorm + scan + sample, ~70 us of serialised kernels for two constant distributions) and the item ->
        # word kernels run on a side stream -- a parallel branch of the captured graph -- and are joined right before
        # the ranking loss, the first reader of the sampled items.  The draw ORDER on the device generator is the
        # reference's (items, then words: item_transformer.py:447, :268); only where the kernels are enqueued moves.
        dev_t = self.product_emb.weight
        cur = torch.cuda.current_stream(dev_t.device) if dev_t.is_cuda else None
        side = None
        if cur is not None and self.overlap_item_to_words:
            if getattr(self, "_iw_stream", None) is None:
                self._iw_stream = torch.cuda.Stream(device=dev_t.device)
            side = self._iw_stream
            side.wait_stream(cur)
        sharded = type(self)._resolve_item_rows is not ItemTransformerRanker._resolve_item_rows
        if not sharded:
            # row-sparse optimizer: the rows this step reads are brought up to date in as few launches as possible
            # (no-ops for ordinary tables) -- history + target rows and query + target words now, the sampled
            # negatives on the side branch as soon as they exist; the gather wrappers then find nothing left to do
            F_.ensure_current(self.hist_product_emb.weight if self.args.sep_prod_emb else self.product_emb.weight,
                              (u_item_idxs,))
            F_.ensure_current(self.product_emb.weight, (target_prod_idxs,))
            F_.ensure_current(self.word_embeddings.weight, (query_word_idxs, pos_iword_idxs))
        if side is not None and not sharded and self.injected_negatives is None:
            with torch.cuda.stream(side):
                neg_item_idxs, neg_word_idxs = self._draw_negatives(B, W, K)
                F_.ensure_current(self.product_emb.weight, (neg_item_idxs,))
                F_.ensure_current(self.word_embeddings.weight, (neg_word_idxs,))
            # (allocated on the side stream and alive until backward has run; the side stream's next allocation
            # happens after its next wait on the current stream, so the allocator cannot recycle them early)
        else:
            neg_item_idxs, neg_word_idxs = self._draw_negatives(B, W, K)
            if side is not None:
                side.wait_stream(cur)
        item_w, item_sink, tgt_idx, neg_idx, hist = self._resolve_item_rows(target_prod_idxs, neg_item_idxs,
                                                                            u_item_idxs)
        if side is not None and sharded:
            side.wait_stream(cur)                # the fetched mini table is produced on the current stream
        item_loss_rows = self.item_to_words(tgt_idx, pos_iword_idxs, K, neg_word_idxs, item_w, item_sink, stream=side,
                                            reduce=False)
        stochastic = self.training and self.args.dropout > 0
        bias = self.product_bias if self.args.sim_func == "bias_product" else None
        pos_weight = float(K) if self.args.pos_weight else 1.0
        if stochastic:
            # dropout makes the positive and the K negative encodes differ (transformer.py:56, neural.py:226):
            # 1 + K dropout draws of the SAME sequence, K/V projections shared between them
            out = self.encode_queries(query_word_idxs, u_item_idxs, copies=1 + K, hist=hist).view(B, 1 + K, -1)
            if self.fused_loss_tail and K <= 7 and self.embedding_size <= 128 and out.is_cuda:
                # ranking loss on the encoder's output block in place + loss combination and running sums: two launches
                if side is not None:
                    cur.wait_stream(side)        # sampled item negatives and the item -> word losses are ready
                if self._ps_acc is None:
                    self._ps_acc = torch.zeros((), device=out.device)
                    self._item_acc = torch.zeros((), device=out.device)
                loss = F_.tem_tail(out, item_loss_rows, item_w, tgt_idx, neg_idx, item_sink, bias=bias,
                                   pos_weight=pos_weight, acc_ps=self._ps_acc, acc_il=self._item_acc,
                                   src_rows=self._tail_src_rows(B, K, out.device))
                F_.RowGradSink.mark_forward_end(out.device)     # every index list of the step exists: sorts may start
                return loss
            pos_out = out[:, 0].contiguous()
            neg_out = out[:, 1:].reshape(B * K, -1)
        else:
            # deterministic encoder: the K copies the reference re-encodes (:473-476) are identical
            pos_out = self.encode_queries(query_word_idxs, u_item_idxs, hist=hist)
            neg_out = pos_out.unsqueeze(1).expand(-1, K, -1).reshape(B * K, -1)
        if side is not None:
            cur.wait_stream(side)                # the sampled item negatives (and the item -> word losses) are ready
        ps = F_.ns_loss(pos_out.contiguous(), item_w, tgt_idx.view(B, 1), neg_idx.view(B, 1, K), item_sink,
                        anchor_b=neg_out.contiguous(), bias=bias, pos_weight=pos_weight)
        ps_loss = ps.mean()
        item_loss = item_loss_rows.mean()
        with torch.no_grad():   # lazily synchronised running sums (the reference calls .item() here); in place,
            if self._ps_acc is None:   # so a CUDA-graph replay keeps accumulating into the same buffers
                self._ps_acc = torch.zeros((), device=ps_loss.device)
                self._item_acc = torch.zeros((), device=ps_loss.device)
            self._ps_acc.add_(ps_loss.detach())
            self._item_acc.add_(item_loss.detach())
        if ps_loss.is_cuda:
            F_.RowGradSink.mark_forward_end(ps_loss.device)
        return ps_loss + item_loss

    def _tail_src_rows(self, B, K, device):
        """Rows of the encoder's [B * (1 + K), d] output block that score the target item (b, 0) and the negatives
        (b, 1 + c): the source-row lists of the item table's gradient contributions (cached: static across replays)."""
        key = (B, K, str(device))
        cache = getattr(self, "_tail_rows_cache", None)
        if cache is None or cache[0] != key:
            base = torch.arange(B, device=device, dtype=torch.int64) * (1 + K)
            neg = (base.view(B, 1) + 1 + torch.arange(K, device=device, dtype=torch.int64).view(1, K)).reshape(-1)
            cache = self._tail_rows_cache = (key, (base.contiguous(), neg.contiguous()))
        return cache[1]

    def item_to_words(self, target_prod_idxs, target_word_idxs, n_negs, neg_sample_idxs=None, item_w=None,
                      item_sink=None, stream=None, reduce=True):
        """item_transformer.py:260-283.  stream / reduce=False: forward kernels on a side stream the caller forked
        and joins before reading the per-item losses that are then returned un-averaged."""
        B, W = target_word_idxs.shape
        if neg_sample_idxs is None:
            neg_sample_idxs = self._multinomial("word_dists", B * W * n_negs)
        if item_w is None:
            item_w, item_sink = self.product_emb.weight, self.item_sink
        anchor = F_.gather_rows(item_w, target_prod_idxs, item_sink, stream=stream)
        loss = F_.ns_loss(anchor, self.word_embeddings.weight, target_word_idxs,
                          neg_sample_idxs.view(B, W, n_negs), self.word_sink, bias=self.word_bias,
                          pad_idx=self.word_pad_idx, stream=stream)
        return loss.mean() if reduce else loss

    # ---- evaluation ---------------------------------------------------------------------
    def test(self, batch_data):
        return self.test_dotproduct(batch_data)

    def test_dotproduct(self, batch_data):
        """Scores of an explicit candidate list [B, candi_k] (item_transformer.py:111-146).  The
        encoder output does not depend on the candidate (SURVEY.md 0.4), so it is computed once
        per query instead of candi_k times."""
        self.flush_lazy_rows()
        with torch.no_grad():
            q = self.encode_queries(batch_data.query_word_idxs, batch_data.u_item_idxs).contiguous()
            bias = self.product_bias if self.args.sim_func == "bias_product" else None
            return ops.score_rows(q, self.product_emb.weight, batch_data.candi_prod_idxs, bias)

    def _max_row_sqnorm(self):
        """|e|^2 bound of the tensor-core shortlist, cached while the item table is unchanged."""
        w = self.product_emb.weight
        key = (w.data_ptr(), w._version, _lib.PARAM_EPOCH[0])
        if getattr(self, "_norm_cache", (None, None))[0] != key:
            self._norm_cache = (key, ops.table_max_row_sqnorm(w, self.prod_pad_idx))
        return self._norm_cache[1]

    def _prepared_catalog(self):
        """fp16 shortlist copy of the item table, rebuilt when the table changes (evaluation: once)."""
        w = self.product_emb.weight
        key = (w.data_ptr(), w._version, _lib.PARAM_EPOCH[0])      # FusedAdam / graph replays bump the epoch
        if getattr(self, "_prep_cache", (None, None))[0] != key:
            self._prep_cache = (key, ops.catalog_prepare_f16(w.detach(), self.prod_pad_idx))
        return self._prep_cache[1]

    def rank_catalog(self, batch_or_queries, k=100, mode=_lib.TOPK_TC16):
        """Top-k over the whole catalog (items 0..P-1) with fused selection; replaces
        get_prod_scores + host argsort (trainer.py:189-226,:152).  Returns (ids [M,k], scores [M,k]).
        mode TOPK_TC16 (default): tcgen05 fp16 shortlist on a cached half-precision copy of the table + exact fp32
        rescoring; TOPK_TC: tf32 shortlist straight from the fp32 table.  Both return exactly what TOPK_EXACT
        returns; shapes they do not cover (and tables that overflow fp16) run the next mode down."""
        self.flush_lazy_rows()             # row-sparse optimizer: every resting row is replayed before a full scan
        with torch.no_grad():
            if torch.is_tensor(batch_or_queries):
                q = batch_or_queries
            else:
                q = self.encode_queries(batch_or_queries.query_word_idxs, batch_or_queries.u_item_idxs)
            bias = self.product_bias if self.args.sim_func == "bias_product" else None
            prepared = None
            if mode == _lib.TOPK_TC16:
                prepared = self._prepared_catalog()
                if not prepared.fits:
                    mode, prepared = _lib.TOPK_TC, None
            norm = self._max_row_sqnorm() if mode == _lib.TOPK_TC else None
            return ops.catalog_topk(q.contiguous(), self.product_emb.weight, k, n_items=self.prod_pad_idx,
                                    bias=bias, mode=mode, max_row_sqnorm=norm, prepared=prepared)


# the north star names the class ProdSearchModel; the reference's real name is kept as primary
ProdSearchModel = ItemTransformerRanker


class ShardedItemTransformerRanker(ItemTransformerRanker):
    """TEM with the item table row-sharded over the ranks of a process group (SURVEY.md 8(e)).

    ``product_emb`` holds only this rank's rows (owner = id % G, local row = id // G).  Each step
    fetches the unique rows it needs into a mini table (index + row all-to-all), runs the same fused
    kernels on it, and ``sync_grads()`` pushes the mini table's gradient rows back to the owners and
    all-reduces the replicated dense parameters.  Call order per step (all ranks, SPMD):
    ``loss = model(batch); model.zero_grad(); loss.backward(); model.sync_grads(); optim.step()``."""

    def __init__(self, args, device, vocab_size, product_size, vocab_words, word_dists=None, group=None,
                 grad_mode="dense"):
        if args.sep_prod_emb or args.sim_func == "bias_product":
            raise NotImplementedError("sharded TEM: sep_prod_emb / bias_product are not sharded yet")
        import torch.distributed as dist
        from . import sharded
        self._group = group
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        super().__init__(args, device, vocab_size, product_size, vocab_words, word_dists, grad_mode)
        full = self.product_emb.weight.detach()
        fold_sink = {}

        def fold(weight, ids, grads):
            sink = fold_sink.get("s")
            if sink is None or sink.weight is not weight:
                pad_local = self.prod_pad_idx // world if self.prod_pad_idx % world == rank else -1
                sink = fold_sink["s"] = F_.RowGradSink(weight, pad_local, None, grad_mode)
            sink._pending.append(ops.make_contrib(ids, grads))
            sink.finalize()

        self.item_table = sharded.ShardedTable.from_full(full, group, ops.gather_rows, fold, device,
                                                         pad_idx=self.prod_pad_idx)
        # the module's parameter becomes the local shard (same state_dict key, 1/G of the rows)
        self.product_emb = nn.Embedding(self.item_table.local_rows, self.embedding_size)
        self.product_emb.weight = self.item_table.weight
        self._make_sinks()
        self._mini = None
        self._dense = sharded.DenseGradAllReduce(self, skip=("product_emb.weight",), group=group)

    def _resolve_item_rows(self, target_prod_idxs, neg_item_idxs, u_item_idxs):
        mini, (tgt, neg, hist), pad = self.item_table.fetch([target_prod_idxs, neg_item_idxs, u_item_idxs])
        sink = F_.RowGradSink(mini, pad, None, "dense")
        self._mini = mini
        return mini, sink, tgt, neg, (mini, sink, hist, pad)

    def sync_grads(self):
        if self._mini is not None:
            g = self._mini.grad if self._mini.grad is not None else torch.zeros_like(self._mini)
            # data-parallel mean over ranks, like the replicated parameters
            self.item_table.push_grads(g / self.item_table.world)
            self._mini = None
        self._dense.reduce()

    def test_dotproduct(self, batch_data):
        with torch.no_grad():
            mini, (cand, hist), pad = self.item_table.fetch([batch_data.candi_prod_idxs, batch_data.u_item_idxs])
            q = self.encode_queries(batch_data.query_word_idxs, batch_data.u_item_idxs, hist=(mini, None, hist, pad))
            return ops.score_rows(q.contiguous(), mini, cand, None)

    def rank_catalog(self, batch_or_queries, k=100, mode=_lib.TOPK_TC):
        from . import sharded
        with torch.no_grad():
            if torch.is_tensor(batch_or_queries):
                q = batch_or_queries
            else:
                raise NotImplementedError("sharded rank_catalog takes encoded query vectors")

            def topk(qa, w, kk, n_local, base, stride, bias):
                return ops.catalog_topk(qa, w, kk, n_items=n_local, bias=bias, id_base=base, id_stride=stride, mode=mode)
            return sharded.sharded_rank_catalog(q.contiguous(), self.item_table, self.prod_pad_idx, k, topk,
                                                ops.topk_merge)


class PeerShardedItemTransformerRanker(ItemTransformerRanker):
    """TEM with the item AND word tables row-sharded over NVLink peer memory (prodsearch_b200/peer.py).

    ``product_emb`` / ``word_embeddings`` hold this rank's rows (owner = id % G, local row = id // G; same
    state_dict keys, 1/G of the rows); encoder, fs projection and biases are replicated.  Per step every rank
    fetches the rows its batch needs with P2P loads into two mini tables, runs the unchanged fused kernels,
    reduces its gradient contributions by GLOBAL row id into a peer-visible compact list, and -- in
    ``sync_grads`` -- folds the slots it owns of every peer's list into its shard gradient, all-reduces the
    replicated gradients over peer memory and forms the global clip norm.  No host synchronisation anywhere:
    ``GraphedTrainStep(model, optim, batch, sync_grads=lambda: model.sync_grads(optim))`` replays the whole
    multi-GPU step as one CUDA graph per rank.  Gradients are the data-parallel MEAN over ranks, i.e. the
    model behaves like the unsharded one trained on the concatenated batch."""

    def __init__(self, args, device, vocab_size, product_size, vocab_words, word_dists=None, peer=None,
                 grad_mode="dense"):
        if args.sep_prod_emb or args.sim_func == "bias_product":
            raise NotImplementedError("peer-sharded TEM: sep_prod_emb / bias_product are not sharded yet")
        from . import peer as peer_mod
        super().__init__(args, device, vocab_size, product_size, vocab_words, word_dists, grad_mode)
        self.peer = peer if peer is not None else peer_mod.PeerGroup(device=device)
        d = self.embedding_size
        full_items = self.product_emb.weight.detach()
        full_words = self.word_embeddings.weight.detach()
        # grad_mode "rowsparse": the owners update the item shard with the row-sparse Adam (O(rows touched) per step
        # whatever the catalog size); readers bring resting rows up to date on the fly.  The word table stays dense.
        self.item_table = peer_mod.PeerShardedTable(product_size + 1, d, self.peer, self.prod_pad_idx, full=full_items,
                                                    sparse=(grad_mode == "rowsparse"))
        self.word_table = peer_mod.PeerShardedTable(vocab_size, d, self.peer, self.word_pad_idx, full=full_words,
                                                    bias=self.word_bias)
        self.product_emb = nn.Embedding(self.item_table.local_rows, d)
        self.product_emb.weight = self.item_table.weight
        self.word_embeddings = nn.Embedding(self.word_table.local_rows, d)
        self.word_embeddings.weight = self.word_table.weight
        del full_items, full_words
        self._make_sinks()
        skip = {"product_emb.weight", "word_embeddings.weight"}
        if args.sim_func != "bias_product":
            # product_bias [P + 1] is not part of this model's loss (item_transformer.py:495-499 only adds it for
            # bias_product): keeping it in the all-reduced bucket would move 4 (P + 1) bytes per rank over NVLink and
            # 28 (P + 1) bytes through Adam every step -- 64 MB / 457 MB at 16M items -- for a gradient that is always zero
            skip.add("product_bias")
        dense = [p for n, p in self.named_parameters() if p.requires_grad and n not in skip]
        self._bucket = peer_mod.DenseBucket(self.peer, dense)
        self._sq = self.peer.alloc(16)                      # this rank's shard-gradient |g|^2 (peer-visible)
        self._sq_local = self._sq.view(torch.float32, (4,))
        self._sq_total = torch.zeros(4, dtype=torch.float32, device=self.peer.device)
        self._sq_dense = torch.zeros(1, dtype=torch.float32, device=self.peer.device)
        self._norm_ws = None

    def _make_sinks(self):
        if hasattr(self, "item_table"):
            self.item_sink = self.hist_sink = self.item_table.sink
            self.word_sink = self.word_table.sink
        else:
            super()._make_sinks()

    def _apply(self, fn, *a, **k):
        if hasattr(self, "item_table"):
            raise RuntimeError("a peer-sharded model cannot be moved / cast after construction")
        return super()._apply(fn, *a, **k)

    # ---- training ----------------------------------------------------------------------------------------
    def forward_dotproduct(self, batch_data, train_pv=False):
        query_word_idxs = batch_data.query_word_idxs
        target_prod_idxs = batch_data.target_prod_idxs
        u_item_idxs = batch_data.u_item_idxs
        pos_iword_idxs = batch_data.pos_iword_idxs
        B, _ = u_item_idxs.shape
        K = self.args.neg_per_pos
        W = pos_iword_idxs.shape[1]
        neg_item_idxs, neg_word_idxs = self._negatives_for_step(B, W, K)
        L = u_item_idxs.shape[1]
        self.item_table.reserve_stage(2 * B * (L + 2 + K))                       # collective on first use only
        self.word_table.reserve_stage(2 * B * (query_word_idxs.shape[1] + W * (1 + K)))
        self.peer.barrier(0)       # every owner has finished last step's optimizer update / staging reads
        # the item rows travel on a side stream while the word rows are fetched and the queries pooled
        if getattr(self, "_fetch_stream", None) is None:
            self._fetch_stream = torch.cuda.Stream(device=self.peer.device)
        items, (tgt, neg, hist), item_pad = self.item_table.fetch([target_prod_idxs, neg_item_idxs, u_item_idxs],
                                                                  stream=self._fetch_stream)
        words, (qw, pw, nw), word_pad = self.word_table.fetch([query_word_idxs, pos_iword_idxs, neg_word_idxs])
        isink, wsink = self.item_table.sink, self.word_table.sink
        cur = torch.cuda.current_stream(self.peer.device)
        # query pooling on a side stream: the encoder call below enqueues its plan / weight transposes first and
        # waits for the pooled queries only before the kernel that reads them (psb_encoder_cfg_t.first_ready)
        if getattr(self, "_q_stream", None) is None:
            self._q_stream = torch.cuda.Stream(device=self.peer.device)
            self._q_ready = torch.cuda.Event()
            self._iw_stream = torch.cuda.Stream(device=self.peer.device)
        q_emb = self.query_encoder.encode_indices(words, qw, wsink, pad_idx=word_pad, stream=self._q_stream)
        self._q_ready.record(self._q_stream)
        wb = self.word_bias
        bias_mini = None
        if wb is not None:     # bias values at the mini positions (the bias vector itself is replicated)
            bias_mini = _BiasAtFn.apply(wb, self.word_table.sink._ids)
        cur.wait_stream(self._fetch_stream)      # join: the item rows are needed by both branches below
        # the item -> word objective shares nothing with the encoder: a parallel branch, joined before the sum
        self._iw_stream.wait_stream(cur)
        anchor = F_.gather_rows(items, tgt, isink, stream=self._iw_stream)
        il = F_.ns_loss(anchor, words, pw, nw.view(B, W, K), wsink, bias=bias_mini, pad_idx=word_pad,
                        stream=self._iw_stream)
        out_pos = -1 if self.args.use_item_pos else 0
        stochastic = self.training and self.args.dropout > 0
        copies = 1 + K if stochastic else 1
        out = self.transformer_encoder.encode_position(first=q_emb.contiguous(), table=items, idx=hist, sink=isink,
                                                       pad_idx=item_pad, use_pos=self.args.use_pos_emb,
                                                       out_pos=out_pos, copies=copies, first_ready=self._q_ready)
        pos_weight = float(K) if self.args.pos_weight else 1.0
        if stochastic and self.fused_loss_tail and K <= 7 and self.embedding_size <= 128:
            # ranking loss on the encoder's output block in place + loss combination: two launches (see the base class)
            cur.wait_stream(self._iw_stream)
            if self._ps_acc is None:
                self._ps_acc = torch.zeros((), device=out.device)
                self._item_acc = torch.zeros((), device=out.device)
            self._join_negative_prefetch(cur)
            loss = F_.tem_tail(out.view(B, 1 + K, -1), il, items, tgt, neg, isink, pos_weight=pos_weight,
                               acc_ps=self._ps_acc, acc_il=self._item_acc,
                               src_rows=self._tail_src_rows(B, K, out.device))
            F_.RowGradSink.mark_forward_end(out.device)
            return loss
        self._join_negative_prefetch(cur)
        if stochastic:
            out = out.view(B, 1 + K, -1)
            pos_out = out[:, 0].contiguous()
            neg_out = out[:, 1:].reshape(B * K, -1)
        else:
            pos_out = out
            neg_out = pos_out.unsqueeze(1).expand(-1, K, -1).reshape(B * K, -1)
        ps = F_.ns_loss(pos_out.contiguous(), items, tgt.view(B, 1), neg.view(B, 1, K), isink,
                        anchor_b=neg_out.contiguous(), pos_weight=pos_weight)
        ps_loss = ps.mean()
        cur.wait_stream(self._iw_stream)
        item_loss = il.mean()
        with torch.no_grad():
            if self._ps_acc is None:
                self._ps_acc = torch.zeros((), device=ps_loss.device)
                self._item_acc = torch.zeros((), device=ps_loss.device)
            self._ps_acc.add_(ps_loss.detach())
            self._item_acc.add_(item_loss.detach())
        F_.RowGradSink.mark_forward_end(ps_loss.device)
        return ps_loss + item_loss

    # The sharded step needs the sampled negatives before anything else (their rows are part of the peer fetch), so the
    # two torch.multinomial chains (~70 us of serialised kernels) would sit at the head of its critical path.  The
    # distributions are constant: the draws for step t + 1 are made on a side stream DURING step t (fetch + encoder take
    # longer) into a second pair of buffers and copied into the live pair at the start of step t + 1.  Same generator,
    # same draw order (items, words, items, words, ...); each draw is merely issued one step early.
    prefetch_negatives = True

    def _negatives_for_step(self, B, W, K):
        if self.injected_negatives is not None or not self.prefetch_negatives or not self.training:
            self._neg_fork = None
            ni, nw = self._draw_negatives(B, W, K)
            return ni, nw
        dev = self.peer.device
        key = (B, W, K)
        if getattr(self, "_neg_key", None) != key:
            self._neg_key = key
            self._neg_cur = (torch.empty((B, K), dtype=torch.int64, device=dev),
                             torch.empty((B, W, K), dtype=torch.int64, device=dev))
            self._neg_next = (torch.empty_like(self._neg_cur[0]), torch.empty_like(self._neg_cur[1]))
            self._neg_ready = False
            self._neg_stream = torch.cuda.Stream(device=dev)
        cur = torch.cuda.current_stream(dev)
        if self._neg_ready:
            self._neg_cur[0].copy_(self._neg_next[0])
            self._neg_cur[1].copy_(self._neg_next[1])
        else:
            ni, nw = self._draw_negatives(B, W, K)
            self._neg_cur[0].copy_(ni)
            self._neg_cur[1].copy_(nw)
        st = self._neg_stream
        st.wait_stream(cur)                       # the copies above have read the "next" pair
        with torch.cuda.stream(st):
            ni, nw = self._draw_negatives(B, W, K)
            self._neg_next[0].copy_(ni)
            self._neg_next[1].copy_(nw)
        self._neg_ready = True
        self._neg_fork = st
        return self._neg_cur

    def _join_negative_prefetch(self, cur):
        st = getattr(self, "_neg_fork", None)
        if st is not None:
            cur.wait_stream(st)
            self._neg_fork = None

    def sync_grads(self, optim=None):
        """Between ``loss.backward()`` and ``optim.step()`` (all ranks): fold the peers' gradient lists into the
        owned shards, all-reduce the replicated gradients, hand the GLOBAL clip norm to the optimizer.  Three
        phases separated by peer barriers (the single-process simulation of the tests calls them in lockstep)."""
        if self.item_table.sparse and optim is not None and self.item_table.lazy_optim is None:
            opt = getattr(optim, "optimizer", optim)
            if hasattr(opt, "adopt_state"):
                it = self.item_table
                opt.adopt_state(it.weight, it.exp_avg, it.exp_avg_sq, it.last_step)
                it.lazy_optim = opt
        self.sync_stage()
        self.peer.barrier(1)       # every rank's compact lists and dense bucket are complete
        fused = (optim is not None and hasattr(getattr(optim, "optimizer", optim), "global_norm_slots")
                 and self.peer.world > 1 and self.peer._sim is None and self.fused_norm_exchange)
        self.sync_fold(norm_exchange=optim if fused else None)
        if fused or optim is None or not hasattr(getattr(optim, "optimizer", optim), "set_global_sqnorm"):
            return
        self.peer.barrier(2)       # every rank's shard norm is published
        self.sync_norm(optim)

    fused_norm_exchange = True     # shard norm, barrier and global norm in one tail launch (psb_peer_norm_exchange)

    def sync_stage(self):
        self._bucket.stage()

    def sync_fold(self, norm_exchange=None):
        """norm_exchange: the optimizer, when the shard norm, the barrier behind it and the global norm are to run as
        one chain (real multi-process groups); None: only the shard norm is formed here (the simulated ranks of the
        tests meet at explicit phases: sync_grads then runs barrier + sync_norm)."""
        G = self.peer.world
        from .peer import fold_tables
        # the owner-side fold of the two tables and the all-reduce of the replicated gradients are independent:
        # the all-reduce runs on a side stream (a parallel branch of the captured graph)
        cur = torch.cuda.current_stream(self.peer.device)
        if getattr(self, "_reduce_stream", None) is None:
            self._reduce_stream = torch.cuda.Stream(device=self.peer.device)
        self._reduce_stream.wait_stream(cur)
        with torch.cuda.stream(self._reduce_stream):
            self._bucket.reduce()
        fold_tables([self.item_table, self.word_table], 1.0 / G)
        cur.wait_stream(self._reduce_stream)
        # partial |g|^2 of this rank: its two shard gradients; rank 0 adds the (replicated, identical) dense bucket
        lib = _lib.load()
        if self.item_table.sparse:
            # item shard: only the rows this fold wrote count (everything else in the buffer is stale, not zero)
            it = self.item_table
            n = 2 if self.peer.rank == 0 else 1
            arr = (_lib.AdamTensor * 2)(
                _lib.AdamTensor(None, self.word_table.grad.data_ptr(), None, None, self.word_table.grad.numel()),
                _lib.AdamTensor(None, self._bucket.red.data_ptr(), None, None, self._bucket.n))
            R = _lib.AdamRows()
            R.rows, R.grad, R.n_rows = it._touched.data_ptr(), it.grad.data_ptr(), it._n_touched.data_ptr()
            R.cap, R.d, R.table_rows, R.grad_by_row = it._touched.numel(), it.d, it.local_rows, 1
            rows_arr = (_lib.AdamRows * 1)(R)
            wb = int(lib.psb_adam_sparse_workspace_bytes(arr, n, rows_arr, 1))
            if self._norm_ws is None or self._norm_ws.numel() < wb:
                self._norm_ws = torch.empty(wb, dtype=torch.uint8, device=self.peer.device)
            if norm_exchange is not None:
                return self._norm_exchange(norm_exchange, arr, n, rows_arr, 1, wb)
            _lib.check(lib.psb_grad_sqnorm_sparse(arr, n, rows_arr, 1, self._sq_local.data_ptr(), self._norm_ws.data_ptr(),
                                                  wb, _lib.stream_ptr()), "psb_grad_sqnorm_sparse")
            return
        n = 3 if self.peer.rank == 0 else 2
        arr = (_lib.AdamTensor * 3)(
            _lib.AdamTensor(None, self.item_table.grad.data_ptr(), None, None, self.item_table.grad.numel()),
            _lib.AdamTensor(None, self.word_table.grad.data_ptr(), None, None, self.word_table.grad.numel()),
            _lib.AdamTensor(None, self._bucket.red.data_ptr(), None, None, self._bucket.n))
        wb = int(lib.psb_adam_workspace_bytes(arr, n))
        if self._norm_ws is None or self._norm_ws.numel() < wb:
            self._norm_ws = torch.empty(wb, dtype=torch.uint8, device=self.peer.device)
        if norm_exchange is not None:
            return self._norm_exchange(norm_exchange, arr, n, None, 0, wb)
        _lib.check(lib.psb_grad_sqnorm(arr, n, self._sq_local.data_ptr(), self._norm_ws.data_ptr(), wb,
                                       _lib.stream_ptr()), "psb_grad_sqnorm")

    def _norm_exchange(self, optim, arr, n, rows_arr, n_tables, wb):
        """Partial sums, then ONE kernel: finish + publish the shard norm, barrier C, global norm, step counter."""
        pg = self.peer
        sq, step = getattr(optim, "optimizer", optim).global_norm_slots(pg.device)
        _lib.check(_lib.load().psb_peer_norm_exchange(
            arr, n, rows_arr, n_tables, self._sq.ptr_array(), pg.flags.ptr_array(), pg.rank, pg.world, pg.epoch.data_ptr(),
            pg.err.data_ptr(), int(pg.timeout_cycles), pg.wait_cycles.data_ptr(), 2, sq.data_ptr(), step.data_ptr(),
            self._norm_ws.data_ptr(), wb, _lib.stream_ptr()), "psb_peer_norm_exchange")

    def sync_norm(self, optim):
        sq, step = getattr(optim, "optimizer", optim).global_norm_slots(self.peer.device)
        _lib.check(_lib.load().psb_peer_sum_sqnorm(self._sq.ptr_array(), self.peer.world, sq.data_ptr(), step.data_ptr(),
                                                   _lib.stream_ptr()), "psb_peer_sum_sqnorm")

    # ---- evaluation -----------------------------------------------------------------------------------------
    def encode_queries(self, query_word_idxs, u_item_idxs, copies=1, hist=None):
        with torch.no_grad():
            items, (h,), item_pad = self.item_table.fetch([u_item_idxs])
            words, (qw,), word_pad = self.word_table.fetch([query_word_idxs])
            q_emb = self.query_encoder.encode_indices(words, qw, None, pad_idx=word_pad)
            out_pos = -1 if self.args.use_item_pos else 0
            return self.transformer_encoder.encode_position(first=q_emb.contiguous(), table=items, idx=h, sink=None,
                                                            pad_idx=item_pad, use_pos=self.args.use_pos_emb,
                                                            out_pos=out_pos, copies=copies)

    def test_dotproduct(self, batch_data):
        with torch.no_grad():
            q = self.encode_queries(batch_data.query_word_idxs, batch_data.u_item_idxs).contiguous()
            items, (cand,), _ = self.item_table.fetch([batch_data.candi_prod_idxs])
            return ops.score_rows(q, items, cand, None)

    def _shard_topk(self, q, k, n_local, id_base, id_stride, mode):
        """Top-k of this rank's shard; TOPK_TC16 uses a cached fp16 copy of the shard (rebuilt when it changes)."""
        w = self.item_table.weight.detach()
        prepared = None
        if mode == _lib.TOPK_TC16:
            key = (w.data_ptr(), self.item_table.weight._version, n_local, _lib.PARAM_EPOCH[0])
            if getattr(self, "_shard_prep", (None, None))[0] != key:
                self._shard_prep = (key, ops.catalog_prepare_f16(w, n_local))
            prepared = self._shard_prep[1]
            if not prepared.fits:
                mode, prepared = _lib.TOPK_TC, None
        return ops.catalog_topk(q, w, k, n_items=n_local, id_base=id_base, id_stride=id_stride, mode=mode,
                                prepared=prepared)

    def rank_catalog(self, batch_or_queries, k=100, mode=_lib.TOPK_TC16):
        """Sharded full-catalog top-k: every rank scores the all-gathered queries against its shard
        (id = rank + G * local row), the per-shard lists are all-gathered and merged (psb_topk_merge).
        Every mode returns the exact mode's lists (the shortlists are rescored in fp32)."""
        import torch.distributed as dist
        with torch.no_grad():
            q = batch_or_queries if torch.is_tensor(batch_or_queries) else self.encode_queries(
                batch_or_queries.query_word_idxs, batch_or_queries.u_item_idxs)
            q = q.contiguous()
            G, r = self.peer.world, self.peer.rank
            n_local = max(0, (self.prod_pad_idx - r + G - 1) // G)
            if G == 1:
                return self._shard_topk(q, k, n_local, 0, 1, mode)
            # every collective lands in its final layout (all_gather_into_tensor): no list gathers, no cat / stack
            m = torch.tensor([q.shape[0]], device=q.device)
            ms = torch.empty(G, dtype=m.dtype, device=q.device)
            dist.all_gather_into_tensor(ms, m, group=self.peer.group)
            m_max = int(ms.max())
            q_pad = q
            if q.shape[0] != m_max:
                q_pad = q.new_zeros((m_max, q.shape[1]))
                q_pad[:q.shape[0]] = q
            q_all = torch.empty((G * m_max, q.shape[1]), dtype=q.dtype, device=q.device)
            dist.all_gather_into_tensor(q_all, q_pad, group=self.peer.group)
            ids, sc = self._shard_topk(q_all, k, n_local, r, G, mode)
            ids_all = torch.empty((G, G * m_max, k), dtype=ids.dtype, device=q.device)
            sc_all = torch.empty((G, G * m_max, k), dtype=sc.dtype, device=q.device)
            dist.all_gather_into_tensor(ids_all.view(-1, k), ids, group=self.peer.group)
            dist.all_gather_into_tensor(sc_all.view(-1, k), sc, group=self.peer.group)
            mi, ms_ = ops.topk_merge(ids_all, sc_all)
            lo = r * m_max
            return mi[lo:lo + q.shape[0]], ms_[lo:lo + q.shape[0]]


class _BiasAtFn(torch.autograd.Function):
    """bias[ids] for the mini-table positions; the gradient reaches the bias through the table's sink
    (``to_bias`` contributions), so nothing flows back here."""

    @staticmethod
    def forward(ctx, bias, ids):
        return bias.detach()[ids]

    @staticmethod
    def backward(ctx, g):
        return None, None
