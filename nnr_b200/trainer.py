"""The training-step contract of reference trainer.py:64-66,105-120 (single GPU) and :285-300 (DDP).

    logits = model(*21 tensors); loss = mean(-log_softmax(logits)[:, 0]); zero_grad; backward;
    clip_grad_norm_(params, 4); Adam(lr=1e-4).step()

B200-native layout: all parameters live in ONE flat fp32 buffer (``param.data`` are views), gradients
in a second flat buffer (``param.grad`` are views), Adam moments in two more.  Data parallelism is
one process per GPU and exactly one ``ncclAllReduce`` over the flat gradient buffer per step
(the reference's DDP issues bucketed all-reduces, trainer.py:219,297); the 1/world averaging is
folded into the fused clip+Adam kernel (``nnr_flat_clip_adam``).
"""
import torch
import torch.distributed as dist

from . import engine, ops


def negative_log_softmax(logits):
    """trainer.py:64-66"""
    return (-torch.log_softmax(logits, dim=1).select(dim=1, index=0)).mean()


class PackedBatch:
    """The 21 model inputs of one batch in ONE contiguous byte buffer (device, or pinned host memory) plus the layout needed
    to view it as tensors again: a step then needs a single copy into the static input buffer of the captured graph instead
    of one copy per field (the reference issues 21 ``.cuda(non_blocking=True)`` calls per step, trainer.py:83-103)."""

    def __init__(self, flat, layout):
        self.flat, self.layout = flat, layout
        self.staged = None                   # (device staging buffer, event) after TrainStep.prefetch

    @staticmethod
    def layout_of(batch):
        layout, o = [], 0
        for t in batch:
            if torch.is_tensor(t):
                nbytes = t.numel() * t.element_size()
                layout.append((o, tuple(t.shape), t.dtype, nbytes))
                o += (nbytes + 255) // 256 * 256
            else:
                layout.append(None)
        return layout, max(o, 256)

    @classmethod
    def pack(cls, batch, device=None, pin=False):
        layout, total = cls.layout_of(batch)
        if pin:
            flat = torch.empty(total, dtype=torch.uint8).pin_memory()
        else:
            flat = torch.empty(total, dtype=torch.uint8, device=device if device is not None else 'cpu')
        pb = cls(flat, layout)
        for v, t in zip(pb.views(), batch):
            if v is not None:
                v.copy_(t)
        return pb

    def views(self, flat=None):
        flat = self.flat if flat is None else flat
        out = []
        for e in self.layout:
            if e is None:
                out.append(None)
                continue
            o, shape, dtype, nbytes = e
            out.append(flat[o:o + nbytes].view(dtype).view(shape))
        return out

    def key(self):
        return tuple(None if e is None else (e[1], e[2]) for e in self.layout)


class TrainStep:
    def __init__(self, model, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, gradient_clip_norm=4.0, process_group=None,
                 world_size=None, cuda_graph=False):
        """cuda_graph=True: every distinct batch layout is captured once (zero-grad, forward, loss, backward, gradient
        all-reduce, clip+Adam, weight-plane refresh: a few hundred kernels) and replayed with one launch per step; dropout
        seeds and Adam's step counter then live on the device (engine.SeedSource, nnr_flat_clip_adam_dev)."""
        self.model = model
        self.cuda_graph = bool(cuda_graph)
        self._graphs = {}
        self._copy_stream = None
        self._stage = {}
        self.lr, self.betas, self.eps, self.max_norm = lr, betas, eps, gradient_clip_norm
        self.pg = process_group
        if world_size is None:
            world_size = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.world_size = world_size
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]     # unique parameters, first name
        # flat-buffer order = the order in which the backward pass finishes the gradients, so that each group is one
        # contiguous slice that can be reduced as soon as it is final (engine.grads_ready): the user encoder's own
        # parameters ('sue'), the news encoder without the word table ('cne'), the word-embedding table ('table', the last
        # kernels of the backward pass and 60 % of the bytes)
        def stage_of(name):
            if name.endswith('word_embedding.weight'):
                return 2
            return 0 if (name.startswith('user_encoder.') and not name.startswith('user_encoder.news_encoder.')) else 1
        named.sort(key=lambda np_: stage_of(np_[0]))                                 # stable: keeps the module order inside a group
        params = [p for _, p in named]
        dev = params[0].device          # flat buffers / all-reduce are device agnostic; the optimizer kernel is CUDA only
        sizes = [(p.numel() + 3) // 4 * 4 for p in params]            # keep every slice 16-byte aligned
        total = sum(sizes)
        self.flat = torch.zeros(total, device=dev)
        self.gflat = torch.zeros(total, device=dev)
        self.exp_avg = torch.zeros(total, device=dev)
        self.exp_avg_sq = torch.zeros(total, device=dev)
        o = 0
        bounds = [0, 0, 0, 0]
        for (name, p), s in zip(named, sizes):
            n = p.numel()
            self.flat[o:o + n].copy_(p.data.reshape(-1))
            p.data = self.flat[o:o + n].view(p.shape)
            p.grad = self.gflat[o:o + n].view(p.shape)
            p._nnr_flat_grad = True          # engine._param_grads adds straight into these views
            o += s
            bounds[stage_of(name) + 1] = o
        for i in range(1, 4):
            bounds[i] = max(bounds[i], bounds[i - 1])
        self.stage_bounds = {'sue': (bounds[0], bounds[1]), 'cne': (bounds[1], bounds[2]), 'table': (bounds[2], bounds[3])}
        self.overlap = True          # reduce each group as soon as it is final, on a side stream (world_size > 1)
        self._comm_stream = None
        self._reduced = set()
        self.params = params
        # operand planes of every GEMM weight matrix, refreshed by one launch after each optimizer step (instead of one
        # small split launch per weight per step); embedding tables are gathered, not multiplied
        self._gemm_weights = [p for n, p in model.named_parameters()
                              if p.requires_grad and p.dim() == 2 and p.is_cuda and 'embedding' not in n and '_lstm.' not in n]
        self._gemm_weights = list({id(p): p for p in self._gemm_weights}.values())
        self._split = ops.SplitMany(self._gemm_weights) if dev.type == 'cuda' else None
        self._refresh_weight_planes()
        self.step_count = 0
        self.grad_norm = torch.zeros(1, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=dev) if dev.type == 'cuda' else None   # graph mode
        self.seeds = engine.SeedSource(dev) if (self.cuda_graph and dev.type == 'cuda') else None
        self.launches_per_graph = {}

    def _refresh_weight_planes(self):
        engine.weights_changed()
        if self._split is not None and self._split.n:
            self._split.refresh()
            for w, pl in zip(self._gemm_weights, self._split.planes):
                engine.install_weight_planes(w, pl)

    def zero_grad(self):
        self.gflat.zero_()
        for p in self.params:                                          # keep .grad bound to the flat views
            if p.grad is None or p.grad.data_ptr() < self.gflat.data_ptr() or \
                    p.grad.data_ptr() >= self.gflat.data_ptr() + self.gflat.numel() * 4:
                raise RuntimeError('parameter .grad was rebound; use TrainStep.zero_grad() only')

    def step(self, *batch):
        """one full training step; returns the (device) loss tensor without synchronising.  ``batch`` is the 21 positional
        tensors of Model.forward, or a single PackedBatch.  In graph mode the returned tensor is the graph's static loss
        buffer: read (or copy) it before the next step."""
        if len(batch) == 1 and isinstance(batch[0], PackedBatch):
            if self.cuda_graph:
                return self._graph_step(batch[0])
            batch = batch[0].views(batch[0].flat.to(self.flat.device, non_blocking=True))
        elif self.cuda_graph:
            return self._graph_step(batch)
        return self._eager_step(*batch)

    def _eager_step(self, *batch):
        if not self.model.training:
            self.model.train()
        self._check_grad_bindings()
        logits = self.model(*batch)
        loss = negative_log_softmax(logits)
        self.gflat.zero_()
        self._reduced = set()
        engine.grads_ready = self._on_grads_ready
        try:
            loss.backward()
        finally:
            engine.grads_ready = None
        self.optimizer_step()
        return loss

    def _check_grad_bindings(self):
        """the engine adds gradients straight into the flat-buffer views; a ``model.zero_grad()`` / ``optimizer.zero_grad()``
        with set_to_none=True unbinds them and the optimizer kernel would then see only zeros"""
        lo, hi = self.gflat.data_ptr(), self.gflat.data_ptr() + self.gflat.numel() * 4
        for p in self.params:
            g = p.grad
            if g is None or not (lo <= g.data_ptr() < hi):
                raise RuntimeError('nnr_b200.TrainStep: a parameter .grad is no longer a view of the flat gradient buffer '
                                   '(zero_grad(set_to_none=True)?); use TrainStep.zero_grad()')

    # ---- graph mode -------------------------------------------------------------------------------------------------
    def _graph_for(self, layout_key, example_views, layout):
        g = self._graphs.get(layout_key)
        if g is not None:
            return g
        dev = self.flat.device
        total = PackedBatch.layout_of(example_views)[1]
        static_flat = torch.empty(total, dtype=torch.uint8, device=dev)
        spb = PackedBatch(static_flat, layout)
        static = spb.views()
        for s, t in zip(static, example_views):
            if s is not None:
                s.copy_(t)
        # warm-up outside capture (lazy kernel attributes, workspaces, allocator), then restore the training state so that
        # graph mode and eager mode walk the same trajectory
        saved = [x.clone() for x in (self.flat, self.exp_avg, self.exp_avg_sq, self.step_dev, self.seeds.base)]
        saved_count = self.step_count
        engine.seed_source = self.seeds
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    self.seeds.advance()
                    self._eager_step(*[s.clone() if torch.is_tensor(s) and s.dtype == torch.bool else s for s in static])
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            for dst, src in zip((self.flat, self.exp_avg, self.exp_avg_sq, self.step_dev, self.seeds.base), saved):
                dst.copy_(src)
            self.step_count = saved_count
            self._refresh_weight_planes()
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            n0 = ops.launch_count()
            # lane 0 (the critical path: content branch, user encoder, optimizer) is captured on a stream above the side lanes'
            # priority; the kernel nodes inherit it, so the block scheduler serves lane 0 first whenever two lanes have CTAs
            # waiting (7.44 -> 7.28 ms per step)
            with torch.cuda.graph(graph, stream=torch.cuda.Stream(priority=-1)):
                self.seeds.advance()
                loss = self._eager_step(*static)
            self.launches_per_graph[layout_key] = ops.launch_count() - n0
            self.step_count = saved_count
        finally:
            engine.seed_source = None
        g = (static_flat, static, graph, loss)
        self._graphs[layout_key] = g
        return g

    def _graph_step(self, batch):
        if isinstance(batch, PackedBatch):
            pb = batch
            static_flat, static, graph, loss = self._graph_for(pb.key(), pb.views() if pb.flat.is_cuda else
                                                               pb.views(pb.flat.to(self.flat.device)), pb.layout)
            if pb.staged is not None:                        # prefetched on the copy stream: wait, then one D2D copy
                buf, ev, ring, i = pb.staged
                torch.cuda.current_stream().wait_event(ev)
                static_flat.copy_(buf, non_blocking=True)
                done = torch.cuda.Event()
                done.record()                                # the next prefetch into this staging buffer waits for this read
                ring['events'][i] = done
                pb.staged = None
            else:
                static_flat.copy_(pb.flat, non_blocking=True)
        else:
            layout, _ = PackedBatch.layout_of(batch)
            key = tuple(None if e is None else (e[1], e[2]) for e in layout)
            static_flat, static, graph, loss = self._graph_for(key, batch, layout)
            for s, t in zip(static, batch):
                if s is not None:
                    s.copy_(t, non_blocking=True)
        graph.replay()
        self.step_count += 1
        return loss

    def prefetch(self, pb):
        """enqueue the host-to-device copy of a pinned PackedBatch on a side stream (two rotating staging buffers), so that it
        overlaps the step that is running; ``step(pb)`` then waits for it and moves it into the graph's input buffer"""
        dev = self.flat.device
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        n = pb.flat.numel()
        ring = self._stage.setdefault(n, {'bufs': [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(2)],
                                          'events': [None, None], 'i': 0})
        i = ring['i']
        ring['i'] = 1 - i
        buf = ring['bufs'][i]
        if ring['events'][i] is not None:                    # the step that consumed this buffer last must have read it
            self._copy_stream.wait_event(ring['events'][i])
        with torch.cuda.stream(self._copy_stream):
            buf.copy_(pb.flat, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
        pb.staged = (buf, ev, ring, i)
        return pb

    def step_ids(self, corpus, history_ids, history_len, candidate_ids):
        """index-only training step (SURVEY 8f-1): the batch is gathered from a ``corpus.DeviceCorpus`` on the device"""
        return self.step(*corpus.batch_from_ids(history_ids, history_len, candidate_ids))

    def reduce_gradients(self):
        """the collective of the step: SUM over ranks of the flat gradient buffer (the 1/world average of DDP, trainer.py:219,
        is applied inside the fused clip+Adam kernel as grad_scale).  Groups that were already reduced during the backward
        pass (``_on_grads_ready``) are skipped; what is left goes out as one all-reduce; the compute stream then waits for
        the side stream."""
        if self.world_size <= 1:
            return
        pending = [k for k in ('sue', 'cne', 'table') if k not in self._reduced]
        if len(pending) == 3:
            dist.all_reduce(self.gflat, op=dist.ReduceOp.SUM, group=self.pg)
        else:
            for k in pending:
                a, b = self.stage_bounds[k]
                if b > a:
                    dist.all_reduce(self.gflat[a:b], op=dist.ReduceOp.SUM, group=self.pg)
            if self._comm_stream is not None:
                torch.cuda.current_stream().wait_stream(self._comm_stream)
        self._reduced = set()

    def _on_grads_ready(self, stage):
        """engine.grads_ready callback: the gradients of `stage` are final in the flat buffer once the CURRENT stream gets here
        (the engine announces the word table from the lane that runs the embedding scatters) -> start their all-reduce on
        the communication stream while the backward pass goes on: the table's reduction runs under the weight-gradient GEMMs
        of the content branch"""
        if self.world_size <= 1 or not self.overlap or self.flat.device.type != 'cuda':
            return
        a, b = self.stage_bounds[stage]
        if b <= a or stage in self._reduced:
            return
        if self._comm_stream is None:
            self._comm_stream = torch.cuda.Stream(device=self.flat.device)
        self._comm_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._comm_stream):
            dist.all_reduce(self.gflat[a:b], op=dist.ReduceOp.SUM, group=self.pg)
        self._reduced.add(stage)

    def optimizer_step(self):
        self.reduce_gradients()
        if self.flat.device.type != 'cuda':
            raise RuntimeError('nnr_b200.TrainStep.optimizer_step needs CUDA (nnr_flat_clip_adam has no CPU path)')
        self.step_count += 1
        if self.cuda_graph:      # the step counter lives on the device so that a captured step advances it on every replay
            ops.flat_clip_adam_dev(self.flat, self.gflat, self.exp_avg, self.exp_avg_sq, self.lr, self.betas[0], self.betas[1],
                                   self.eps, self.max_norm, 1.0 / self.world_size, self.step_dev, self.grad_norm)
        else:
            ops.flat_clip_adam(self.flat, self.gflat, self.exp_avg, self.exp_avg_sq, self.lr, self.betas[0], self.betas[1],
                               self.eps, self.max_norm, 1.0 / self.world_size, self.step_count, self.grad_norm)
        self._refresh_weight_planes()   # the kernel updates the parameters through raw pointers: re-split them (one launch)


class LossLog:
    """Per-step loss read-back without stalling the launch queue.

    The reference adds ``float(loss) * batch`` to the epoch loss every step (trainer.py:115,295), which blocks the host
    until the step has finished before the next one is enqueued.  Here every step's loss is copied into a pinned host
    slot with a non-blocking D2H copy + an event; ``push`` returns the values whose copies have completed (normally the
    previous step's), ``drain`` waits for the rest.  Every step is still read exactly once and the epoch sum is the
    same -- the host just consumes step i while the device runs step i+1."""

    def __init__(self, slots=8):
        self.buf = torch.empty(slots, dtype=torch.float32).pin_memory()
        self.pending = []          # (slot, event, weight) in issue order
        self.slots = slots
        self.next = 0
        self.total = 0.0           # sum of weight * loss over the consumed steps (the reference's epoch_loss)
        self.count = 0

    def _consume(self, block):
        out = []
        while self.pending and (block or self.pending[0][1].query()):
            slot, ev, wt = self.pending.pop(0)
            ev.synchronize()
            v = float(self.buf[slot])
            self.total += v * wt
            self.count += 1
            out.append(v)
        return out

    def push(self, loss, weight=1.0, lag=1):
        """enqueue the read of this step's (device) loss; returns the losses that are complete, waiting only if more than
        ``lag`` reads are outstanding"""
        out = []
        if len(self.pending) >= self.slots:                  # ring full (lag >= slots): that value is returned too
            out += self._consume_one()
        slot = self.next
        self.next = (self.next + 1) % self.slots
        self.buf[slot:slot + 1].copy_(loss.detach().reshape(1), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.pending.append((slot, ev, weight))
        while len(self.pending) > lag:
            out += self._consume_one()
        return out + self._consume(False)

    def _consume_one(self):
        slot, ev, wt = self.pending.pop(0)
        ev.synchronize()
        v = float(self.buf[slot])
        self.total += v * wt
        self.count += 1
        return [v]

    def drain(self):
        return self._consume(True)


def balanced_shards(cost, world_size):
    """Token-balanced sharding of one global batch over the ranks of a synchronous data-parallel step.

    ``cost[i]`` is the work of impression i (its number of valid tokens).  Every rank gets exactly ``len(cost) // world_size``
    impressions; they are dealt longest first, each to the rank with the smallest total so far that still has room (greedy
    LPT).  A synchronous step runs at the pace of its slowest rank, and with variable-length news the token count of a random
    shard of 64 impressions varies by +-6 % (the slowest of 8 random shards is ~12 % above the mean), which is what limits the
    weak scaling of the reference's DistributedSampler shards (trainer.py:256-258); the set of impressions in the global batch
    -- hence the averaged gradient's meaning -- is unchanged.  Deterministic: every rank computes the same assignment.
    Returns a list of ``world_size`` index lists (ascending inside a shard)."""
    import numpy as np
    cost = np.asarray(cost, dtype=np.int64)
    n = len(cost)
    if n % world_size:
        raise ValueError('batch size %d not divisible by world size %d' % (n, world_size))
    per = n // world_size
    order = np.argsort(-cost, kind='stable')
    totals = [0] * world_size
    shards = [[] for _ in range(world_size)]
    for i in order:
        r = min((r for r in range(world_size) if len(shards[r]) < per), key=lambda r: (totals[r], r))
        shards[r].append(int(i))
        totals[r] += int(cost[i])
    return [sorted(s) for s in shards]


def shard_batch(batch, rank, world_size):
    """Reference DDP sharding (trainer.py:218,256-258): rank r takes impressions [r*B/W, (r+1)*B/W) of a global
    batch whose size is divisible by the world size (config.py:116).  Works on dicts or sequences of tensors;
    non-tensor entries (the unused entity fields may be None) are passed through."""
    def cut(v):
        if not torch.is_tensor(v):
            return v
        B = v.shape[0]
        if B % world_size:
            raise ValueError('batch size %d not divisible by world size %d' % (B, world_size))
        per = B // world_size
        return v[rank * per:(rank + 1) * per]
    if isinstance(batch, dict):
        return {k: cut(v) for k, v in batch.items()}
    return [cut(v) for v in batch]
