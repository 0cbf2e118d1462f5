"""Cached-corpus dev/test scoring (BASELINE config 3; SURVEY 8f-1/f-2).

The reference's ``util.compute_scores`` re-encodes the user's 50 history news for every (impression,
candidate) pair (util.py:19-50, README.md:125).  Here the news corpus is encoded ONCE with the CNE kernels
and kept resident in HBM as a [news_num, 900] table; an impression is then just 50 history ids + n candidate
ids: the history graph / category mask / cluster indices are built on the device from the cached category ids
(``nnr_sue_graph_build``, bit-exact with MIND_corpus.py:178-213), followed by SUE and the dot product.

Parity note (SURVEY finding 2): a news vector depends on the composition of the ``news_encoder`` call it is
encoded in (sort-rank pairing of the selective gate).  The cache is therefore defined per corpus chunk: news
[c*chunk, (c+1)*chunk) are encoded as ONE call of shape [1, chunk]; the oracle test encodes the same chunks.

Data parallel (SURVEY 8e): with a ``process_group``, ``encode_corpus`` and ``evaluate`` are collectives.  Each rank
runs the single-GPU computation on a contiguous share of the same corpus chunks / impression batches
(``contiguous_blocks``) and one NCCL all-gather assembles the whole result on every rank, so the cache, the ranks and
the metrics are bit-identical to one GPU.  The all-gathers run on the current stream, outside any captured graph.
``recommend(collective=True)`` shares the pool tiles the same way: each rank folds its tiles into a k-entry best list, and
the all-gathered rank lists are merged into one on every rank (``nnr_topk_merge_lists``).
"""
import numbers

import torch

from . import engine, metrics, ops


def contiguous_blocks(nblocks, world):
    """Split blocks [0, nblocks) into ``world`` contiguous runs: rank r owns [r*k, min((r+1)*k, nblocks)) with
    k = ceil(nblocks / world), so the ranks' k-block send buffers all-gather in global order.  Ranks past the last block
    own an empty run.  Returns (k, [(first, end) per rank])."""
    k = -(-nblocks // world)
    return k, [(min(r * k, nblocks), min((r + 1) * k, nblocks)) for r in range(world)]


def _checksum(t):
    """position-weighted int64 sum of an integer tensor: cheap, and changes when ids are edited or permuted"""
    t = t.reshape(-1).long()
    w = torch.arange(t.numel(), device=t.device) % 65521 + 1
    return (t * w).sum()


class CorpusScorer:
    """``process_group=None`` scores on this process's device alone.  With an NCCL group, ``encode_corpus`` and
    ``evaluate`` are collectives: every rank of the group calls them with the same arguments (and the same weights, as
    ``TrainStep`` keeps them) and gets the whole result.  ``score`` is always rank-local; ``recommend`` is rank-local unless
    called with ``collective=True``.
    ``graph_flags`` = ``ops.graph_flags(...)`` of the options the model was trained with (no_self_connection,
    no_adjacent_normalization, gcn_normalization_type); 0 is the reference's default symmetric graph."""

    # recommend(): candidates per pool tile by default = this many rows of the cluster tail, B * T * (C + 1).  Each row holds
    # four D-wide fp32-sized buffers (intra-cluster features, their GEMM operand planes, the relu stash, the cluster
    # features): about 7.5 GB at D = 900, plus ~11 KB per (user, candidate) pair on the candidate side.
    TAIL_ROWS = 1 << 19

    def __init__(self, model, news_title_text, news_title_mask, news_content_text, news_content_mask, news_category,
                 news_subCategory, chunk=4096, process_group=None, graph_flags=0):
        self.model = model
        self.graph_flags = graph_flags                          # ops.graph_flags(...) of the model's training configuration
        self.dev = next(model.parameters()).device
        to = lambda t: torch.as_tensor(t).to(self.dev)
        self.tt, self.tm, self.ct, self.cm = to(news_title_text), to(news_title_mask).clone(), to(news_content_text), to(news_content_mask).clone()
        self.cat, self.sub = to(news_category).to(torch.int32), to(news_subCategory).to(torch.int32)
        self.chunk = chunk
        self.cache = None
        self._graphs = {}
        self._num_groups = None                                 # recommend(max_per_category=): 1 + largest category id
        self.group = process_group
        if process_group is not None:
            import torch.distributed as dist
            self._check_group()
            self.rank, self.world = dist.get_rank(process_group), dist.get_world_size(process_group)
            self._corpus_sum = None

    def _check_group(self):
        """the collectives run over NCCL on the model's device, which must be the current device"""
        import torch.distributed as dist
        if dist.get_backend(self.group) != 'nccl':
            raise ValueError('CorpusScorer: process_group must be an NCCL group, got %s' % dist.get_backend(self.group))
        if self.dev.type != 'cuda' or self.dev.index != torch.cuda.current_device():
            raise RuntimeError('CorpusScorer: the model is on %s but the current CUDA device is cuda:%d; call '
                               'torch.cuda.set_device() with the rank\'s device first' % (self.dev, torch.cuda.current_device()))

    def _graphed(self, key, fn, example_inputs):
        """capture ``fn(*static_inputs)`` once per shape key and replay it: an encode of one corpus chunk is ~100 kernels of a
        few microseconds to a millisecond, i.e. host-launch bound when issued one by one (eval mode: no dropout, no seeds)"""
        g = self._graphs.get(key)
        if g is None:
            static = [x.clone() for x in example_inputs]
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):                           # warm-up outside capture: lazy attributes, workspaces, weight planes
                    fn(*[x.clone() for x in static])
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = fn(*static)
            g = (static, graph, out)
            self._graphs[key] = g
        static, graph, out = g
        for s_, x in zip(static, example_inputs):
            s_.copy_(x, non_blocking=True)
        graph.replay()
        return out

    # fields of the descriptor every rank contributes before the first collective of a call
    _FIELDS = ('call', 'news_num', 'chunk', 'D', 'I', 'n_max', 'H', 'batch', 'corpus ids checksum', 'history_ids checksum',
               'history_len checksum', 'candidate_ids checksum', 'candidate_count checksum', 'labels checksum', 'B', 'P', 'k',
               'T', 'm', 'exclude_history', 'pool_ids checksum', 'exact', 'argument error')

    def _agree(self, call, **fields):
        """all-gather a small int64 descriptor of this call's inputs and raise on every rank if any field differs between
        ranks, so that no rank enters an all-gather with a shape or data the others do not share"""
        import torch.distributed as dist
        mine = torch.zeros(len(self._FIELDS), dtype=torch.int64, device=self.dev)
        mine[0] = call
        for name, v in fields.items():
            mine[self._FIELDS.index(name)] = v
        table = torch.empty(self.world * len(self._FIELDS), dtype=torch.int64, device=self.dev)
        dist.all_gather_into_tensor(table, mine, group=self.group)
        table = table.view(self.world, -1).cpu()
        bad = [i for i in range(len(self._FIELDS)) if not bool((table[:, i] == table[0, i]).all())]
        if bad:
            what = '; '.join('%s: %s' % (self._FIELDS[i], table[:, i].tolist()) for i in bad)
            raise RuntimeError('CorpusScorer.%s: the ranks of the process group were called with different arguments (%s). '
                               'Every rank must pass the same inputs.' % (('encode_corpus', 'evaluate', 'recommend')[call - 1], what))

    def _corpus_fields(self):
        return dict(news_num=self.tt.shape[0], chunk=self.chunk, D=self.model.news_encoder.news_embedding_dim)

    @torch.no_grad()
    def encode_corpus(self, cuda_graph=True):
        """news table -> [news_num, news_embedding_dim] fp32 cache; returns it.  Full chunks replay one captured graph.
        With a process group: a collective; each rank encodes its contiguous share of the chunks and every rank returns
        the whole cache."""
        self.model.eval()
        enc = self.model.news_encoder
        n = self.tt.shape[0]

        def encode(tt, tm, ct, cm, cat, sub):
            return enc(tt.unsqueeze(0), tm.unsqueeze(0), None, ct.unsqueeze(0), cm.unsqueeze(0), None, cat.unsqueeze(0), sub.unsqueeze(0), None)[0]

        def encode_chunk(a):
            b = min(n, a + self.chunk)
            args = (self.tt[a:b], self.tm[a:b], self.ct[a:b], self.cm[a:b], self.cat[a:b], self.sub[a:b])
            if cuda_graph and b - a == self.chunk and n >= 3 * self.chunk:
                return self._graphed(('encode', self.chunk), encode, args)
            return encode(*args)

        if self.group is None:
            out = torch.empty(n, enc.news_embedding_dim, device=self.dev)
            for a in range(0, n, self.chunk):
                out[a:min(n, a + self.chunk)] = encode_chunk(a)
            self.cache = out
            return out

        self._corpus_sum = int(sum(int(_checksum(t)) for t in (self.tt, self.ct, self.cat, self.sub)))
        self._agree(1, **self._corpus_fields(), **{'corpus ids checksum': self._corpus_sum})
        self.cache = self._sharded(n, self.chunk, enc.news_embedding_dim, encode_chunk)
        return self.cache

    def _sharded(self, nitems, block, width, compute):
        """rows [0, nitems) in blocks [a, a + block): this rank computes its contiguous share of the blocks (``compute(a)``)
        into a zero-padded [k * block, width] buffer, and one all-gather returns all [nitems, width] rows on every rank"""
        import torch.distributed as dist
        k, parts = contiguous_blocks(-(-nitems // block), self.world)
        first, end = parts[self.rank]
        send = torch.zeros(k * block, width, device=self.dev)
        for a in range(first * block, end * block, block):
            lo = a - first * block
            send[lo:lo + min(nitems, a + block) - a] = compute(a)
        gathered = torch.empty(self.world * k * block, width, device=self.dev)
        dist.all_gather_into_tensor(gathered, send, group=self.group)
        return gathered[:nitems]

    @torch.no_grad()
    def score(self, history_ids, history_len, candidate_ids, cuda_graph=True, exact=True):
        """history_ids [B,H] (0-padded at the end), history_len [B], candidate_ids [B,n] -> scores [B,n].  Rank-local:
        never a collective, also with a process group.  Full shapes with B >= 64 replay one captured CUDA graph per shape.

        ``exact=False`` scores every entry through the factored cluster tail (nnr_cluster_tail_scores_packed, each user's
        n candidates as one list): the cluster affine is applied once per history row instead of to C + 1 cluster
        features per (user, candidate) pair, and the candidate projections run once per candidate.  The scores are those
        of the SUE formula, within a relative error of 1e-4 of ``exact=True`` (fp32 sums in another order), but not
        bit-identical to it.  The call is deterministic.  The candidate ids must lie in [0, news_num) (ValueError before
        any launch otherwise).  SUE_wo_HCA, whose user vector does not depend on the candidate, returns the
        ``exact=True`` result bit for bit."""
        if not exact:
            cid, cnt = self._packed_inputs('score', candidate_ids, None)
            return self._score_packed(history_ids, history_len, cid, cnt, cuda_graph)
        assert self.cache is not None, 'call encode_corpus() first'
        hid = torch.as_tensor(history_ids).to(self.dev).long()
        cid = torch.as_tensor(candidate_ids).to(self.dev).long()
        hl = torch.as_tensor(history_len).to(self.dev).to(torch.int32)
        if cuda_graph and hid.shape[0] >= 64:
            key = ('score', tuple(hid.shape), tuple(cid.shape), self.cache.data_ptr())
            return self._graphed(key, self._score_impl, (hid, hl, cid)).clone()
        return self._score_impl(hid, hl, cid)

    def _packed_inputs(self, who, candidate_ids, candidate_count):
        """the checks of score() / evaluate() with exact=False, once per call and before any launch: candidate_ids [I, n]
        integers, candidate_count [I] in [0, n] (None: all n), the valid candidate ids in [0, news_num).  Returns
        (candidate ids [I, n] int64, counts [I] int32) as given, on the device they came on."""
        if self.cache is None:
            raise RuntimeError('CorpusScorer.%s: call encode_corpus() first' % who)
        cid = torch.as_tensor(candidate_ids)
        if cid.dim() != 2 or cid.dtype.is_floating_point or cid.dtype == torch.bool:
            raise ValueError('CorpusScorer.%s: candidate_ids must be a 2-D integer tensor, got %s of shape %s'
                             % (who, cid.dtype, tuple(cid.shape)))
        I, n = cid.shape
        cnt = torch.full((I,), n, dtype=torch.int64) if candidate_count is None else torch.as_tensor(candidate_count)
        if tuple(cnt.shape) != (I,) or cnt.dtype.is_floating_point or cnt.dtype == torch.bool:
            raise ValueError('CorpusScorer.%s: candidate_count must be an integer tensor of shape [%d], got %s of shape %s'
                             % (who, I, cnt.dtype, tuple(cnt.shape)))
        if I and (int(cnt.min()) < 0 or int(cnt.max()) > n):
            raise ValueError('CorpusScorer.%s: candidate_count must be in [0, %d], got [%d, %d]'
                             % (who, n, int(cnt.min()), int(cnt.max())))
        valid = torch.arange(n, device=cnt.device)[None, :] < cnt[:, None]
        if bool(valid.any()):
            cid_v = cid.to(cnt.device)
            lo = int(torch.where(valid, cid_v, torch.zeros_like(cid_v)).min())
            hi = int(torch.where(valid, cid_v, torch.zeros_like(cid_v)).max())
            news_num = self.cache.shape[0]
            if lo < 0 or hi >= news_num:
                raise ValueError('CorpusScorer.%s: the valid candidate ids must be in [0, %d), got [%d, %d]'
                                 % (who, news_num, lo, hi))
        return cid.long(), cnt.to(torch.int32)

    def _score_packed(self, history_ids, history_len, cid, cnt, cuda_graph):
        """scores [B, n] of the first cnt[b] candidates of each row of cid [B, n] through the factored cluster tail (0 past
        the counts); B >= 64 replays one captured graph per shape"""
        hid = torch.as_tensor(history_ids).to(self.dev).long()
        hl = torch.as_tensor(history_len).to(self.dev).to(torch.int32)
        cid, cnt = cid.to(self.dev), cnt.to(self.dev)
        if cid.numel() == 0:
            return torch.zeros(cid.shape, device=self.dev)
        if cuda_graph and hid.shape[0] >= 64:
            key = ('score_factored', tuple(hid.shape), tuple(cid.shape), self.cache.data_ptr())
            return self._graphed(key, self._score_packed_impl, (hid, hl, cid, cnt)).clone()
        return self._score_packed_impl(hid, hl, cid, cnt)

    def _score_packed_impl(self, hid, hl, cid, cnt):
        """the candidates are packed back to back on the device (prefix sum of the counts; no host synchronisation): list b
        is rows [row_off[b], row_off[b + 1]) of a [B * n, D] buffer whose rows past row_off[B] hold news 0 and are not
        scored.  Padding entries of cid are never read."""
        B, n = cid.shape
        row_off = torch.zeros(B + 1, dtype=torch.int32, device=self.dev)
        torch.cumsum(cnt, 0, dtype=torch.int32, out=row_off[1:])
        j = torch.arange(n, device=self.dev)
        # packed row of every valid entry; padding goes to a dump slot past the end
        dest = torch.where(j[None, :] < cnt[:, None], row_off[:B, None].long() + j[None, :], B * n)
        ids = torch.zeros(B * n + 1, dtype=torch.int64, device=self.dev).scatter_(0, dest.view(-1), cid.reshape(-1))[:B * n]
        ue = self.model.user_encoder
        side = ue.user_side(self.cache[hid], *self._history_graph(hid, hl), factored=True)
        return ue.packed_scores_factored(side, self.cache[ids], row_off, torch.zeros(B, n, device=self.dev))

    def _category_num(self):
        ue = self.model.user_encoder
        return ue.proxy_node_embedding.shape[0] if hasattr(ue, 'proxy_node_embedding') else ue.category_num - 1   # SUE_wo_GCN

    def _history_graph(self, hid, hl):
        """graph, cluster mask and cluster indices of the histories hid [B, H], built on the device from the cached
        category ids"""
        B, H = hid.shape
        C = self._category_num()
        cats = self.cat[hid].contiguous()
        graph = torch.empty(B, H + C, H + C, device=self.dev)
        cmask = torch.empty(B, C + 1, dtype=torch.bool, device=self.dev)
        cidx = torch.empty(B, H, dtype=torch.int64, device=self.dev)
        ops.sue_graph_build(cats, hl, C, graph, cmask, cidx, flags=self.graph_flags)
        return graph, cmask, cidx

    def _score_impl(self, hid, hl, cid):
        graph, cmask, cidx = self._history_graph(hid, hl)
        hist = self.cache[hid]                                  # [B, H, D]
        cand = self.cache[cid]                                  # [B, n, D]
        user = self.model.user_encoder.encode_user(hist, graph, cmask, cidx, cand)
        return engine.RowDot.apply(user, cand)

    def default_pool_tile(self, B):
        """recommend()'s candidates per tile for B users: B * T * (C + 1) <= TAIL_ROWS, 1 <= T <= ops.TOPK_MAX_TILE"""
        return max(1, min(ops.TOPK_MAX_TILE, self.TAIL_ROWS // (max(B, 1) * (self._category_num() + 1))))

    def _category_groups(self):
        """number of groups of the capped merge (1 + the largest corpus category id), after checking once that every
        category id is in [0, ops.TOPK_MAX_GROUPS)"""
        if self._num_groups is None:
            lo, hi = (int(self.cat.min()), int(self.cat.max())) if self.cat.numel() else (0, 0)
            if lo < 0 or hi >= ops.TOPK_MAX_GROUPS:
                raise ValueError('CorpusScorer.recommend: max_per_category needs corpus category ids in [0, %d), got [%d, %d]'
                                 % (ops.TOPK_MAX_GROUPS, lo, hi))
            self._num_groups = hi + 1
        return self._num_groups

    @torch.no_grad()
    def recommend(self, history_ids, history_len, pool_ids, k, exclude_history=True, pool_tile=None, cuda_graph=True,
                  max_per_category=None, collective=False, exact=True):
        """The k best news of a candidate pool for each user: history_ids [B, H] (0-padded at the end) and history_len [B]
        as in ``score``, pool_ids [P] corpus row ids shared by the B users.  Returns (ids [B, k] int64, scores [B, k] fp32),
        best first.

        Order: score descending; equal scores in ascending pool position (a stable descending sort of the user's whole
        [P] score row, the convention of ``metrics.rank_impressions``); a NaN score ranks below every number.  With
        ``exclude_history`` a pool entry whose id is among the user's first history_len[b] history ids is never returned.
        When fewer than k entries are eligible, the tail is filled with id -1 and score -inf (a real candidate scoring
        -inf still ranks before the fill).  Duplicate pool ids are separate entries.

        The scores are those of ``score(history_ids, history_len, tile.expand(B, T))`` for each tile of the pool, bit for
        bit: the user side (graph, GCN, intra-cluster keys) is computed once, then the pool is scored in tiles of
        ``pool_tile`` candidates, each folded into a running top-k list by nnr_topk_merge.  Memory does not grow with P.
        The default tile holds B * T * (C + 1) <= TAIL_ROWS = 2^19 rows of the cluster tail (about 7.5 GB at D = 900,
        C = 18; T = 107 for B = 256) and at most 4096 candidates.  Full tiles replay one captured CUDA graph per
        (B, H, T); a last partial tile runs eagerly.
        Limits: 1 <= k <= ops.TOPK_MAX_K (1024), 1 <= pool_tile <= ops.TOPK_MAX_TILE (4096), H <= ops.TOPK_MAX_EXCLUDE
        with ``exclude_history``.

        ``max_per_category = m`` caps how many of a user's k news may share a ``news_category`` (the corpus category ids
        the history is clustered by): the user's eligible pool entries are taken in the order above, each unless m
        entries of its category were already taken, until k are taken; the rest is filled as above.  Excluded history
        entries count toward no cap, duplicate pool ids count once per entry.  None, or any m >= k, returns exactly the
        uncapped result.  m < k runs nnr_topk_merge_capped, which keeps the same k entries of state per user, so memory
        still does not grow with P.  Corpus category ids must be in [0, ops.TOPK_MAX_GROUPS) (1024).

        ``collective=False`` is rank-local: never a collective, also with a process group.  ``collective=True`` needs a
        scorer with a process group and is a collective: every rank calls it with the same arguments, after
        ``encode_corpus()``.  Rank r scores the pool tiles [a, a + T) of its contiguous share (``contiguous_blocks`` of the
        ceil(P / T) tiles) into its own k-entry list, one all-gather brings every rank's list to every rank, and
        nnr_topk_merge_lists[_capped] folds them in rank order.  Every rank returns the whole result, bit-identical to a
        plain call with the same arguments (the same ``pool_tile``) on one GPU.  The ranks first all-gather a descriptor
        of their arguments: if it differs between ranks, or the arguments fail a check on some ranks only, every rank
        raises RuntimeError naming the fields; a check that fails on every rank raises its ValueError there.  Either way
        no rank is left in a collective, and the group can be used for the next call.

        ``exact=False`` scores the tiles through the factored cluster tail (nnr_cluster_tail_scores): the intra-cluster
        weights of a non-empty cluster sum to 1, so the cluster affine is applied once per history row (Wg = g W^T, with
        the user side) instead of to C + 1 cluster features per (user, candidate) pair, and the candidate projections run
        once per pool row instead of once per (user, row).  The scores are those of the SUE formula, within a relative
        error of 1e-4 of ``score()`` (fp32 sums in another order), but not bit-identical to it or to ``exact=True``, so
        ids whose scores lie that close to the k-th score may differ between the two.  Everything else is as above: the
        checks, the order, the exclusions and the fill, ``max_per_category``, ``collective`` (bit-identical to the plain
        ``exact=False`` call with the same ``pool_tile``), graph replay of full tiles, memory that does not grow with P.
        The call is deterministic: the same arguments give the same bits.  The default tile is min(P, 4096) candidates
        (the factored tail holds no per-pair buffers).  SUE_wo_HCA, whose user vector does not depend on the candidate,
        returns the ``exact=True`` result."""
        if collective:
            return self._recommend_collective(history_ids, history_len, pool_ids, k, exclude_history, pool_tile, cuda_graph,
                                              max_per_category, exact)
        hid, hl, pool, k, T, m, groups = self._recommend_inputs(history_ids, history_len, pool_ids, k, exclude_history,
                                                                pool_tile, max_per_category, exact)
        B, P = hid.shape[0], pool.numel()
        if P == 0 or B == 0:
            best_score, best_pos, _ = self._fill(B, k)
            return best_pos, best_score                         # ids -1, scores -inf
        best_score, best_pos, _ = self._recommend_tiles(hid, hl, pool, k, T, 0, -(-P // T), exclude_history, m, groups,
                                                        cuda_graph, exact)
        return self._pool_ids(pool, best_pos), best_score

    def _recommend_inputs(self, history_ids, history_len, pool_ids, k, exclude_history, pool_tile, max_per_category,
                          exact=True):
        """recommend()'s argument checks, before any kernel launch.  Returns (hid [B, H] int64, hl [B] int32, pool [P] int64
        on the device, k, T, m (None when uncapped), the number of category groups (None when uncapped))."""
        if self.cache is None:
            raise RuntimeError('CorpusScorer.recommend: call encode_corpus() first')
        k = int(k)
        if not 1 <= k <= ops.TOPK_MAX_K:
            raise ValueError('CorpusScorer.recommend: k must be in [1, %d], got %d' % (ops.TOPK_MAX_K, k))
        m = max_per_category
        if m is not None and (isinstance(m, bool) or not isinstance(m, numbers.Integral) or m < 1):
            raise ValueError('CorpusScorer.recommend: max_per_category must be None or an int >= 1, got %r' % (m,))
        capped = m is not None and m < k
        groups = self._category_groups() if capped else None
        pool = torch.as_tensor(pool_ids)
        if pool.dim() != 1 or pool.dtype.is_floating_point or pool.dtype == torch.bool:
            raise ValueError('CorpusScorer.recommend: pool_ids must be a 1-D integer tensor, got %s of shape %s'
                             % (pool.dtype, tuple(pool.shape)))
        news_num = self.cache.shape[0]
        if pool.numel() and (int(pool.min()) < 0 or int(pool.max()) >= news_num):
            raise ValueError('CorpusScorer.recommend: pool_ids must be in [0, %d), got [%d, %d]'
                             % (news_num, int(pool.min()), int(pool.max())))
        hid = torch.as_tensor(history_ids).to(self.dev).long().contiguous()
        hl = torch.as_tensor(history_len).to(self.dev).to(torch.int32)
        B, H = hid.shape
        if pool_tile is not None:
            T = int(pool_tile)
        else:
            T = self.default_pool_tile(B) if exact else max(1, min(pool.numel(), ops.TOPK_MAX_TILE))
        if not 1 <= T <= ops.TOPK_MAX_TILE:
            raise ValueError('CorpusScorer.recommend: pool_tile must be in [1, %d], got %d' % (ops.TOPK_MAX_TILE, T))
        if exclude_history and H > ops.TOPK_MAX_EXCLUDE:
            raise ValueError('CorpusScorer.recommend: exclude_history takes at most %d history ids, got %d' % (ops.TOPK_MAX_EXCLUDE, H))
        return hid, hl, pool.to(self.dev).long(), k, T, (int(m) if capped else None), groups

    def _fill(self, B, k, capped=False):
        """an empty best list: (score -inf, position -1, group -1 or None)"""
        return (torch.full((B, k), float('-inf'), device=self.dev), torch.full((B, k), -1, dtype=torch.int64, device=self.dev),
                torch.full((B, k), -1, dtype=torch.int32, device=self.dev) if capped else None)

    @staticmethod
    def _pool_ids(pool, best_pos):
        return torch.where(best_pos >= 0, pool[best_pos.clamp(min=0)], torch.full_like(best_pos, -1))

    def _recommend_tiles(self, hid, hl, pool, k, T, first, end, exclude_history, m, groups, cuda_graph, exact=True):
        """the best list of pool tiles [first, end) (tile t: pool positions [t * T, min((t + 1) * T, P))): returns
        (best_score [B, k], best_pos [B, k] pool positions, best_group [B, k] or None when m is None).  No tiles: the fill.
        ``exact=False``: the tiles are scored through the factored cluster tail."""
        B, H = hid.shape
        P = pool.numel()
        if first >= end:
            return self._fill(B, k, m is not None)
        ue = self.model.user_encoder
        graph = self._history_graph(hid, hl)
        side = ue.user_side(self.cache[hid], *graph) if exact else ue.user_side(self.cache[hid], *graph, factored=True)

        def tile_scores(*args):
            *user, ids = args
            if not exact:
                return ue.tile_scores_factored(tuple(user), self.cache[ids])
            return ue.tile_scores(tuple(user), self.cache[ids].unsqueeze(0).expand(B, -1, -1))

        best_score = torch.empty(B, k, device=self.dev)
        best_pos = torch.empty(B, k, dtype=torch.int64, device=self.dev)
        best_group = torch.empty(B, k, dtype=torch.int32, device=self.dev) if m is not None else None
        key = ('recommend' if exact else 'recommend_factored', B, H, T, self.cache.data_ptr())
        for a in range(first * T, min(end * T, P), T):
            ids = pool[a:a + T]
            if cuda_graph and ids.numel() == T:
                scores = self._graphed(key, tile_scores, (*side, ids))
                # from now on hand the graph its own static copy of the user side: copy_ onto itself is a no-op, so only
                # the tile's ids are copied per replay
                side = self._graphs[key][0][:-1]
            else:
                scores = tile_scores(*side, ids)
            init = a == first * T
            if m is not None:
                ops.topk_merge_capped(scores, a, ids, hid if exclude_history else None, hl if exclude_history else None,
                                      self.cat.contiguous(), groups, m, init, best_score, best_pos, best_group)
            else:
                ops.topk_merge(scores, a, ids, hid if exclude_history else None, hl if exclude_history else None, init,
                               best_score, best_pos)
        return best_score, best_pos, best_group

    def _merge_rank_lists(self, scores, pos, grp, m, groups):
        """fold W best lists scores / pos (/ grp) [W, B, k] of disjoint pool positions into one, in rank order
        (nnr_topk_merge_lists[_capped], one launch per list).  Returns (best_score [B, k], best_pos [B, k])."""
        W, B, k = scores.shape
        best_score = torch.empty(B, k, device=self.dev)
        best_pos = torch.empty(B, k, dtype=torch.int64, device=self.dev)
        best_group = torch.empty(B, k, dtype=torch.int32, device=self.dev) if m is not None else None
        for r in range(W):
            if m is not None:
                ops.topk_merge_lists_capped(scores[r], pos[r], grp[r], groups, m, r == 0, best_score, best_pos, best_group)
            else:
                ops.topk_merge_lists(scores[r], pos[r], r == 0, best_score, best_pos)
        return best_score, best_pos

    def _recommend_collective(self, history_ids, history_len, pool_ids, k, exclude_history, pool_tile, cuda_graph,
                              max_per_category, exact):
        """recommend(collective=True): agree on the arguments, score this rank's share of the tiles, all-gather the rank
        lists and merge them"""
        if self.group is None:
            raise ValueError('CorpusScorer.recommend: collective=True needs a scorer built with a process_group')
        err = None
        try:
            hid, hl, pool, k, T, m, groups = self._recommend_inputs(history_ids, history_len, pool_ids, k, exclude_history,
                                                                    pool_tile, max_per_category, exact)
        except (ValueError, RuntimeError) as e:        # raised after the agreement, so that no rank waits in a collective
            err = e
        fields = {'argument error': int(err is not None), 'exact': int(bool(exact))}
        if err is None:
            fields.update({'B': hid.shape[0], 'H': hid.shape[1], 'P': pool.numel(), 'k': k, 'T': T,
                           'm': 0 if max_per_category is None else int(max_per_category),
                           'exclude_history': int(bool(exclude_history)), 'pool_ids checksum': _checksum(pool),
                           'history_ids checksum': _checksum(hid), 'history_len checksum': _checksum(hl)})
        try:
            self._agree(3, **self._corpus_fields(), **{'corpus ids checksum': self._corpus_sum or 0}, **fields)
        except RuntimeError as e:
            if err is not None:
                raise RuntimeError('%s On this rank: %s' % (e, err)) from err
            raise
        if err is not None:
            raise err
        B, P = hid.shape[0], pool.numel()
        if P == 0 or B == 0:
            best_score, best_pos, _ = self._fill(B, k)
            return best_pos, best_score                         # ids -1, scores -inf
        _, parts = contiguous_blocks(-(-P // T), self.world)
        first, end = parts[self.rank]
        mine = self._recommend_tiles(hid, hl, pool, k, T, first, end, exclude_history, m, groups, cuda_graph, exact)
        best_score, best_pos = self._gather_and_merge(mine, m, groups)
        return self._pool_ids(pool, best_pos), best_score

    def _gather_and_merge(self, mine, m, groups):
        """all-gather every rank's best list ``mine`` = (score, pos, group or None) [B, k] and fold them into one"""
        import torch.distributed as dist
        B, k = mine[0].shape
        gathered = []
        for t in mine:
            if t is not None:
                out = torch.empty(self.world * B, k, dtype=t.dtype, device=self.dev)
                dist.all_gather_into_tensor(out, t, group=self.group)
                gathered.append(out.view(self.world, B, k))
        return self._merge_rank_lists(gathered[0], gathered[1], gathered[2] if m is not None else None, m, groups)

    @torch.no_grad()
    def _impression_scores(self, history_ids, history_len, candidate_ids, batch, candidate_count=None, labels=None,
                           exact=True):
        """scores [I, n_max] of impressions batched as [a, a + batch) from 0.  With a process group: a collective; each rank
        scores its contiguous share of the batches and every rank returns the whole matrix.  ``exact=False``: only the
        first candidate_count[i] entries of each row are scored, through the factored cluster tail (0 past them)."""
        cid = torch.as_tensor(candidate_ids)
        err = None
        if not exact:
            try:
                cid, cnt = self._packed_inputs('evaluate', cid, candidate_count)
            except (ValueError, RuntimeError) as e:
                if self.group is None:
                    raise
                err = e                                  # raised after the agreement, so that no rank waits in a collective

        def scores(a):
            if exact:
                return self.score(history_ids[a:a + batch], history_len[a:a + batch], cid[a:a + batch])
            return self._score_packed(history_ids[a:a + batch], history_len[a:a + batch], cid[a:a + batch],
                                      cnt[a:a + batch], True)

        if self.group is None:
            return torch.cat([scores(a) for a in range(0, cid.shape[0], batch)])

        fields = {'exact': int(bool(exact)), 'argument error': int(err is not None)}
        if err is None:
            assert self.cache is not None, 'call encode_corpus() first'
            ids = dict(history_ids=history_ids, history_len=history_len, candidate_ids=cid, candidate_count=candidate_count,
                       labels=labels)
            fields.update({k + ' checksum': int(_checksum(torch.as_tensor(v).to(self.dev))) for k, v in ids.items()
                           if v is not None})
            fields.update(I=cid.shape[0], n_max=cid.shape[1], H=torch.as_tensor(history_ids).shape[1], batch=batch)
        try:
            self._agree(2, **self._corpus_fields(), **{'corpus ids checksum': self._corpus_sum or 0}, **fields)
        except RuntimeError as e:
            if err is not None:
                raise RuntimeError('%s On this rank: %s' % (e, err)) from err
            raise
        if err is not None:
            raise err
        return self._sharded(cid.shape[0], batch, cid.shape[1], scores)

    @torch.no_grad()
    def evaluate(self, history_ids, history_len, candidate_ids, candidate_count, labels, batch=256, exact=True):
        """Dev-set metrics with the cached corpus and on-device ranking (SURVEY 8f-2; replaces util.compute_scores +
        evaluate.scoring): impressions are padded to [I, n_max] candidate ids with ``candidate_count`` valid entries
        and 0/1 ``labels``.  Returns (auc, mrr, ndcg5, ndcg10, ranks [I, n_max]).  With a process group: a collective;
        the impression batches are shared out between the ranks, the scores all-gathered, and every rank ranks the whole
        matrix and returns the same metrics as one GPU.

        ``exact=False`` scores each batch of ``batch`` impressions through the factored cluster tail
        (nnr_cluster_tail_scores_packed): only the first candidate_count[i] candidates of each impression are scored,
        packed back to back on the device, so the work follows the sum of the counts instead of I * n_max, and the cluster
        affine is applied once per history row instead of once per (impression, candidate) cluster feature.  Padding
        entries are never read: their ids may be anything, -1 for instance.  The scores are those of the SUE formula,
        within a relative error of 1e-4 of ``exact=True`` (fp32 sums in another order), but not bit-identical to it, so
        ranks of candidates whose scores lie that close may differ between the two, and with them the metrics.  The ranks
        and metrics are computed from these scores as above, and the call is deterministic.  candidate_count must have
        shape [I] with values in [0, n_max], and the valid candidate ids must lie in [0, news_num): ValueError, checked
        once per call before any launch (with a process group, after the ranks' argument agreement, which includes
        ``exact``; the sharded result equals the plain ``exact=False`` call bit for bit).  Full batches replay one
        captured CUDA graph per (batch, H, n_max).  SUE_wo_HCA, whose user vector does not depend on the candidate,
        returns the ``exact=True`` scores of the valid entries bit for bit."""
        scores = self._impression_scores(history_ids, history_len, candidate_ids, batch, candidate_count, labels, exact)
        cnt = torch.as_tensor(candidate_count).to(self.dev)
        lab = torch.as_tensor(labels).to(self.dev)
        ranks, _ = metrics.rank_impressions(scores, cnt)
        return metrics.scoring(scores, lab, cnt) + (ranks,)
