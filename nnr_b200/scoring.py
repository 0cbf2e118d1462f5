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
"""
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
    ``TrainStep`` keeps them) and gets the whole result.  ``score`` is always rank-local."""

    def __init__(self, model, news_title_text, news_title_mask, news_content_text, news_content_mask, news_category,
                 news_subCategory, chunk=4096, process_group=None):
        self.model = model
        self.dev = next(model.parameters()).device
        to = lambda t: torch.as_tensor(t).to(self.dev)
        self.tt, self.tm, self.ct, self.cm = to(news_title_text), to(news_title_mask).clone(), to(news_content_text), to(news_content_mask).clone()
        self.cat, self.sub = to(news_category).to(torch.int32), to(news_subCategory).to(torch.int32)
        self.chunk = chunk
        self.cache = None
        self._graphs = {}
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
               'history_len checksum', 'candidate_ids checksum', 'candidate_count checksum', 'labels checksum')

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
                               'Every rank must pass the same inputs.' % (('encode_corpus', 'evaluate')[call - 1], what))

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
    def score(self, history_ids, history_len, candidate_ids, cuda_graph=True):
        """history_ids [B,H] (0-padded at the end), history_len [B], candidate_ids [B,n] -> scores [B,n].  Rank-local:
        never a collective, also with a process group."""
        assert self.cache is not None, 'call encode_corpus() first'
        hid = torch.as_tensor(history_ids).to(self.dev).long()
        cid = torch.as_tensor(candidate_ids).to(self.dev).long()
        hl = torch.as_tensor(history_len).to(self.dev).to(torch.int32)
        if cuda_graph and hid.shape[0] >= 64:
            key = ('score', tuple(hid.shape), tuple(cid.shape), self.cache.data_ptr())
            return self._graphed(key, self._score_impl, (hid, hl, cid)).clone()
        return self._score_impl(hid, hl, cid)

    def _score_impl(self, hid, hl, cid):
        ue = self.model.user_encoder
        B, H = hid.shape
        C = ue.proxy_node_embedding.shape[0]
        cats = self.cat[hid].contiguous()
        graph = torch.empty(B, H + C, H + C, device=self.dev)
        cmask = torch.empty(B, C + 1, dtype=torch.bool, device=self.dev)
        cidx = torch.empty(B, H, dtype=torch.int64, device=self.dev)
        ops.sue_graph_build(cats, hl, C, graph, cmask, cidx)
        hist = self.cache[hid]                                  # [B, H, D]
        cand = self.cache[cid]                                  # [B, n, D]
        user = ue.encode_user(hist, graph, cmask, cidx, cand)
        return engine.RowDot.apply(user, cand)

    @torch.no_grad()
    def _impression_scores(self, history_ids, history_len, candidate_ids, batch, candidate_count=None, labels=None):
        """scores [I, n_max] of impressions batched as [a, a + batch) from 0.  With a process group: a collective; each rank
        scores its contiguous share of the batches and every rank returns the whole matrix."""
        cid = torch.as_tensor(candidate_ids)
        if self.group is None:
            out = []
            for a in range(0, cid.shape[0], batch):
                out.append(self.score(history_ids[a:a + batch], history_len[a:a + batch], cid[a:a + batch]))
            return torch.cat(out)

        assert self.cache is not None, 'call encode_corpus() first'
        I, n_max = cid.shape
        ids = dict(history_ids=history_ids, history_len=history_len, candidate_ids=cid, candidate_count=candidate_count, labels=labels)
        sums = {k + ' checksum': int(_checksum(torch.as_tensor(v).to(self.dev))) for k, v in ids.items() if v is not None}
        self._agree(2, **self._corpus_fields(), **{'corpus ids checksum': self._corpus_sum}, I=I, n_max=n_max,
                    H=torch.as_tensor(history_ids).shape[1], batch=batch, **sums)
        return self._sharded(I, batch, n_max,
                             lambda a: self.score(history_ids[a:a + batch], history_len[a:a + batch], cid[a:a + batch]))

    @torch.no_grad()
    def evaluate(self, history_ids, history_len, candidate_ids, candidate_count, labels, batch=256):
        """Dev-set metrics with the cached corpus and on-device ranking (SURVEY 8f-2; replaces util.compute_scores +
        evaluate.scoring): impressions are padded to [I, n_max] candidate ids with ``candidate_count`` valid entries
        and 0/1 ``labels``.  Returns (auc, mrr, ndcg5, ndcg10, ranks [I, n_max]).  With a process group: a collective;
        the impression batches are shared out between the ranks, the scores all-gathered, and every rank ranks the whole
        matrix and returns the same metrics as one GPU."""
        scores = self._impression_scores(history_ids, history_len, candidate_ids, batch, candidate_count, labels)
        cnt = torch.as_tensor(candidate_count).to(self.dev)
        lab = torch.as_tensor(labels).to(self.dev)
        ranks, _ = metrics.rank_impressions(scores, cnt)
        return metrics.scoring(scores, lab, cnt) + (ranks,)
