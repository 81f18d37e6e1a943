"""GPU, world size 2 (needs two visible GPUs; skipped otherwise): the data-parallel training path end to end.

ADVICE r1 (high): the per-bucket events the backward records for the gradient all-reduce were never created, so the
side-stream all-reduce ran with no dependency on the backward kernels. Here two ranks run forward + BPTT on their
shard of a batch in the "events" mode of bench.py (external event-record nodes of the replayed backward graph ->
in-place NCCL all-reduce of the gradient buckets on a side stream) and every reduced gradient must equal the gradient
of the whole batch computed by one process. Repeated several times so that the CUDA-graph replay path (third call on)
and any race between the all-reduce and a still-running backward show up.
"""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

CFG = dict(vocab_size=500, image_feature_size=128, embedding_size=600, hidden_size=64, attention_projection_size=48,
           z_space=24, sentiment_vae=1, simple_vae=False, max_caption_length=20, prior_std=1.0, senti_prior_multip=0.5)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _batch(B):
    g = torch.Generator().manual_seed(3)
    feats = torch.rand(B, 9, 128, generator=g)
    toks = torch.randint(2, 500, (B, 20), generator=g)
    lens = torch.randint(4, 21, (B,), generator=g)
    for b in range(B):
        toks[b, lens[b]:] = 0
    sent = torch.randint(-1, 2, (B, 1), generator=g).float()
    eps = torch.randn(21, B, 24, generator=g)
    return feats, toks, sent, eps


def _grads(m, feats, toks, sent, eps, scale):
    m._eps_override = eps.cuda()
    for p in m.parameters():
        p.grad = None
    out = m(feats.cuda(), None, None, toks.cuda(), sent.cuda())
    ((out["loss"].sum() + out["kld"].sum() / 750.0) * scale).backward()


def _worker(rank, world, port, ret):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import sscvae
    from sscvae import _lib
    from helpers import module_from_cfg
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.manual_seed(0)
    m = module_from_cfg(CFG, device=f"cuda:{rank}")
    m.train()
    B = 12
    feats, toks, sent, eps = _batch(B)
    # reference: the whole batch on this rank, objective = mean over the GLOBAL batch
    _grads(m, feats, toks, sent, eps, 1.0 / B)
    torch.cuda.synchronize()
    want = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    # data parallel: every rank its shard; the reducer AVERAGES over ranks, so each rank scales by 1 / (B / world)
    named = [(k, p) for k, p in m.named_parameters() if p.requires_grad]
    reducer = sscvae.BucketedGradReducer(named)
    m._group_events = [torch.cuda.Event() for _ in range(_lib.GRAD_GROUPS)]
    sl = sscvae.shard_batch(B, rank, world)
    worst = 0.0
    for it in range(6):
        _grads(m, feats[sl], toks[sl], sent[sl], eps[:, sl].contiguous(), 1.0 / (B / world))
        reducer.reduce(m._group_events, buckets=m.grad_buckets())
        torch.cuda.synchronize()
        assert all(e.cuda_event for e in m._group_events)
        for k, p in m.named_parameters():
            if p.grad is None:
                continue
            err = ((p.grad - want[k]).abs().max() / (want[k].abs().max() + 1e-12)).item()
            worst = max(worst, err)
    # different ranks must draw different Philox noise (ADVICE r1 medium): same torch seed on both ranks
    m._eps_override = None
    torch.manual_seed(0)
    m._call_counter = 0
    m(feats[:4].cuda(), None, None, toks[:4].cuda(), sent[:4].cuda())
    e = m.train_region(4, 9, "eps", torch.float32, (21 * 4 * 24,)).clone()
    gathered = [torch.empty_like(e) for _ in range(world)]
    dist.all_gather(gathered, e)
    distinct = not torch.equal(gathered[0], gathered[1])
    ret[rank] = (worst, distinct)
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two visible GPUs")
def test_two_rank_gradients_equal_the_single_process_gradient():
    world = 2
    port = _free_port()
    ret = mp.get_context("spawn").Manager().dict()
    mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
    for rank in range(world):
        worst, distinct = ret[rank]
        # shards are summed in a different order than the single-process batch and the bf16 operand roundings of the
        # batched weight-gradient GEMMs differ (K = T*B/2 vs T*B): bf16-level agreement
        assert worst < 2e-2, (rank, worst)
        assert distinct
