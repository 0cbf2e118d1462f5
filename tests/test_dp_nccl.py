"""GPU tests of the data-parallel path on the REAL model over NCCL (skipped with fewer than 2 GPUs):

SURVEY 8c "DP parity" / reference trainer.py:212-219,285-300: with the global batch sharded over N ranks, the all-reduced flat
gradient times 1/N equals the mean of the single-process oracle gradients of the N shards (each shard is its own sort-rank
pairing domain, exactly as under the reference's DDP), with the bucketed / overlapped reduction, without it, and inside a
captured CUDA graph; the parameters after two optimizer steps are identical on all ranks and match the oracle's clip+Adam.
"""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, q):
    try:
        os.environ['MASTER_ADDR'] = '127.0.0.1'
        os.environ['MASTER_PORT'] = str(port)
        torch.cuda.set_device(rank)
        dev = torch.device('cuda', rank)
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
        import nnr_b200
        from nnr_b200 import engine
        from nnr_b200.synthetic import SyntheticMIND, batch_args
        from nnr_b200.trainer import TrainStep, negative_log_softmax, shard_batch
        from oracle import nnr_oracle as O
        engine.sort_fn = O.stable_sort
        cfg = O.make_config(vocabulary_size=500, max_history_num=6, max_title_length=12, max_abstract_length=24, subCategory_num=30,
                            gcn_layer_num=2, dropout_rate=0.0)
        syn = SyntheticMIND(news_num=200, vocabulary_size=500, subCategory_num=30, max_title_length=12, max_abstract_length=24,
                            max_history_num=6, lengths='uniform', seed=3)
        full = syn.batch(2 * world, seed=1)                              # global batch, 2 impressions per rank
        p = O.formula_params(cfg)
        cfg.pretrained_word_embedding = p['news_encoder.word_embedding.weight']

        def build():
            m = nnr_b200.Model(cfg)
            m.initialize()
            m.load_state_dict(O.alias_state_dict(p))
            return m.to(dev).train()

        # oracle: per-shard gradients on the CPU (every rank computes all of them; tiny)
        shard_grads, shard_losses = [], []
        for r in range(world):
            _, loss_r, g_r = O.forward_backward(p, cfg, shard_batch(full, r, world), sort_fn=O.stable_sort)
            shard_grads.append(g_r)
            shard_losses.append(float(loss_r))
        mean_grads = {k: sum(g[k] for g in shard_grads) / world for k in shard_grads[0]}
        gmax = max(float(v.abs().max()) for v in mean_grads.values())
        mine = shard_batch(full, rank, world)

        def check_grads(ts, m, tag):
            named = dict(m.named_parameters())
            for k, ref in mean_grads.items():
                got = named[k].grad.detach().cpu() / world           # the 1/world of DDP is folded into the optimizer kernel
                tol = 1e-4 * max(float(ref.abs().max()), 1e-2 * gmax)
                assert float((got - ref).abs().max()) <= tol, (tag, k, float((got - ref).abs().max()), tol)

        # (1) overlapped bucket reduction (groups reduced on the side stream as the backward pass finishes them)
        for overlap in (True, False):
            m = build()
            ts = TrainStep(m, lr=1e-3, world_size=world)
            ts.overlap = overlap
            logits = m(*batch_args({k: (v.clone() if torch.is_tensor(v) else v) for k, v in mine.items()}, dev))
            loss = negative_log_softmax(logits)
            ts.gflat.zero_()
            ts._reduced = set()
            engine.grads_ready = ts._on_grads_ready
            loss.backward()
            engine.grads_ready = None
            if overlap:
                # the three stages of the flat buffer, each announced when its gradients are final: the user encoder, the news
                # encoder's weights, and the word table (announced from the lane that runs the embedding scatters)
                assert ts._reduced == {'sue', 'cne', 'table'}, ts._reduced
            ts.reduce_gradients()
            torch.cuda.synchronize()
            assert abs(loss.item() - shard_losses[rank]) < 1e-5
            check_grads(ts, m, 'overlap=%s' % overlap)

        # (2) two full steps, host-launched and as a captured graph: same parameters on every rank, equal to the oracle's
        #     clip_grad_norm_ + Adam on the mean gradient
        ref = {k: v.clone() for k, v in p.items()}
        state = {}
        for step in (1, 2):
            gs = [O.forward_backward(ref, cfg, shard_batch(full, r, world), sort_fn=O.stable_sort)[2] for r in range(world)]
            O.clip_and_adam(ref, {k: sum(g[k] for g in gs) / world for k in gs[0]}, state, step, lr=1e-3, max_norm=4.0)
        for graph in (False, True):
            m = build()
            ts = TrainStep(m, lr=1e-3, gradient_clip_norm=4.0, world_size=world, cuda_graph=graph)
            for step in (1, 2):
                ts.step(*batch_args({k: (v.clone() if torch.is_tensor(v) else v) for k, v in mine.items()}, dev))
            torch.cuda.synchronize()
            flat = ts.flat.clone()
            gathered = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(gathered, flat)
            for g in gathered:
                assert torch.equal(g, gathered[0]), 'parameters diverged across ranks (graph=%s)' % graph
            named = dict(m.named_parameters())
            for k in ref:
                d = (named[k].detach().cpu() - ref[k]).abs().max().item()
                assert d <= 2.5e-3, (graph, k, d)            # nothing moves more than 2 steps of lr plus slack
            big = [k for k in ref if ref[k].numel() > 1000]
            close = sum(int((named[k].detach().cpu() - ref[k]).abs().median().item() < 2e-5) for k in big)
            assert close >= len(big) - 2, (graph, close, len(big))
        del ts, m
        import gc
        gc.collect()
        torch.cuda.synchronize()
        q.put((rank, 'ok'))
    except Exception as ex:                                   # surface the failure in the parent
        import traceback
        q.put((rank, 'FAILED: %s\n%s' % (ex, traceback.format_exc())))
    finally:
        # no destroy_process_group(): tearing down a communicator whose collectives were captured in CUDA graphs takes minutes;
        # the worker process ends here anyway
        import sys
        sys.stdout.flush()
        q.close()
        q.join_thread()                                        # the result must reach the parent before the hard exit
        os._exit(0)


def test_nccl_gradients_equal_mean_of_oracle_shard_gradients():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    world = 2
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=600) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for rank, msg in sorted(results):
        assert msg == 'ok', 'rank %d: %s' % (rank, msg)
