"""GPU: checkpoint and resume with FusedClipSGD in torch.optim.SGD's state format (SURVEY 8(f)-1).

  * a run saved as {"model", "optimizer"} (checkpointing.py:101-103) and resumed into a fresh module and optimizer
    (train.py:142-151) equals the run that was never stopped, bit for bit, with the decoder-LSTM freeze interval
    (train.py:156-161) straddling the save, in both zero_grad semantics, and with or without the reference's LambdaLR;
  * a checkpoint of torch.optim.SGD + LambdaLR resumes into FusedClipSGD, and one of FusedClipSGD into torch.optim.SGD;
  * the same resume through the captioner's real forward and backward is bit-exact.
"""
import io

import pytest
import torch

import sscvae
from conftest import load_golden
from helpers import module_from_cfg

pytestmark = pytest.mark.gpu

CFG = dict(vocab_size=300, image_feature_size=64, embedding_size=600, hidden_size=32, attention_projection_size=24,
           z_space=16, sentiment_vae=1, simple_vae=False, max_caption_length=20, prior_std=1.0, senti_prior_multip=0.5)
LR, MOM, WD, CLIP, NIT = 0.05, 0.9, 1e-3, 0.5, 40            # small clip threshold: the clip is active
DEC = "_updown_cell._language_lstm_cell_decoder"
FROZEN = {2, 3, 4}                                            # decoder LSTM frozen on these; the save follows step 2
SAVE, STEPS = 3, 7


def _gradients():
    torch.manual_seed(0)
    m = module_from_cfg(CFG, device="cpu")
    g = torch.Generator().manual_seed(1)
    return [{k: torch.randn(p.shape, generator=g) * (3.0 if it % 2 else 0.01)
             for k, p in m.named_parameters() if p.requires_grad} for it in range(STEPS)]


def _set_grads(m, grads, it):
    for k, p in m.named_parameters():
        if k in grads[it] and not (it in FROZEN and k.startswith(DEC)):   # frozen: backward leaves no gradient
            p.grad = grads[it][k].to(p.device)


def _checkpoint(m, opt):
    f = io.BytesIO()
    torch.save({"model": m.state_dict(), "optimizer": opt.state_dict()}, f)
    return f.getvalue()


def _load(blob):
    """A fresh copy per load: Optimizer.load_state_dict keeps loaded tensors that are already on the parameter's
    device, so two optimizers loaded from one dict would share their momentum buffers."""
    return torch.load(io.BytesIO(blob))


def _fused(m, legacy=False):
    return sscvae.FusedClipSGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD, max_norm=CLIP, num_iterations=NIT,
                               legacy_zero_grad=legacy)


def _lambda_lr(opt, last_epoch=-1):
    return torch.optim.lr_scheduler.LambdaLR(opt, lr_lambda=lambda it: 1 - it / NIT, last_epoch=last_epoch)  # train.py:132-134


def _snapshot(m, opt):
    return ({k: p.detach().clone() for k, p in m.named_parameters()},
            {k: opt.state[p]["momentum_buffer"].clone() for k, p in m.named_parameters() if p in opt.state},
            opt.param_groups[0]["lr"])


def _run_fused(m, opt, grads, its, sched=None):
    trace = []
    for it in its:
        opt.zero_grad()
        _set_grads(m, grads, it)
        opt.step()
        if sched is not None:
            sched.step()
        trace.append(_snapshot(m, opt))
    return trace


def _run_torch(m, opt, sched, grads, its):
    trace = []
    for it in its:
        opt.zero_grad()
        _set_grads(m, grads, it)
        torch.nn.utils.clip_grad_norm_(m.parameters(), CLIP)     # train.py:173-176
        opt.step()
        sched.step()
        trace.append(_snapshot(m, opt))
    return trace


def _assert_equal(a, b):
    for (pa, ba, lra), (pb, bb, lrb) in zip(a, b, strict=True):
        assert lra == lrb
        assert pa.keys() == pb.keys() and ba.keys() == bb.keys()
        assert all(torch.equal(pa[k], pb[k]) for k in pa), [k for k in pa if not torch.equal(pa[k], pb[k])]
        assert all(torch.equal(ba[k], bb[k]) for k in ba), [k for k in ba if not torch.equal(ba[k], bb[k])]


def _assert_close(a, b):
    for step, ((pa, ba, lra), (pb, bb, lrb)) in enumerate(zip(a, b, strict=True)):
        assert lra == lrb, step
        assert pa.keys() == pb.keys() and ba.keys() == bb.keys()
        for k in pa:
            assert torch.allclose(pa[k], pb[k], rtol=2e-5, atol=2e-6), (step, k)
        for k in ba:
            assert torch.allclose(ba[k], bb[k], rtol=2e-5, atol=2e-6), (step, k)


@pytest.mark.parametrize("scheduler", [False, True])
@pytest.mark.parametrize("legacy", [False, True])
def test_resume_equals_the_uninterrupted_run(legacy, scheduler):
    grads = _gradients()
    torch.manual_seed(0)
    m = module_from_cfg(CFG)
    whole = _run_fused(m, _fused(m, legacy), grads, range(STEPS))
    assert whole[-1][2] == LR * (1 - STEPS / NIT)

    torch.manual_seed(0)
    m = module_from_cfg(CFG)
    opt = _fused(m, legacy)
    head = _run_fused(m, opt, grads, range(SAVE), _lambda_lr(opt) if scheduler else None)
    ckpt = _load(_checkpoint(m, opt))
    del m, opt
    torch.manual_seed(1)                                      # a different initialisation, overwritten by the load
    m = module_from_cfg(CFG, ckpt["model"])
    opt = _fused(m, legacy)
    opt.load_state_dict(ckpt["optimizer"])
    assert opt.iteration == SAVE
    # a LambdaLR attached to the resumed optimizer continues at the saved iteration
    sched = _lambda_lr(opt, last_epoch=opt.iteration - 1) if scheduler else None
    tail = _run_fused(m, opt, grads, range(SAVE, STEPS), sched)
    _assert_equal(head + tail, whole)


def test_torch_sgd_checkpoint_resumes_into_fused_clip_sgd():
    grads = _gradients()
    torch.manual_seed(0)
    m = module_from_cfg(CFG)
    opt = torch.optim.SGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD)
    _run_torch(m, opt, _lambda_lr(opt), grads, range(SAVE))
    blob = _checkpoint(m, opt)

    ckpt = _load(blob)
    m = module_from_cfg(CFG, ckpt["model"])
    ours = _fused(m)
    ours.load_state_dict(ckpt["optimizer"])
    assert ours.iteration == 0 and ours.lr == LR               # no iteration in the dict: the schedule restarts
    got = _run_fused(m, ours, grads, range(SAVE, STEPS))

    ckpt = _load(blob)
    m = module_from_cfg(CFG, ckpt["model"])
    opt = torch.optim.SGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD)
    opt.load_state_dict(ckpt["optimizer"])
    want = _run_torch(m, opt, _lambda_lr(opt), grads, range(SAVE, STEPS))     # a fresh LambdaLR: restarts at 0 too
    _assert_close(got, want)


def test_fused_clip_sgd_checkpoint_resumes_into_torch_sgd():
    grads = _gradients()
    torch.manual_seed(0)
    m = module_from_cfg(CFG)
    ours = _fused(m)
    _run_fused(m, ours, grads, range(SAVE))
    blob = _checkpoint(m, ours)

    ckpt = _load(blob)
    m = module_from_cfg(CFG, ckpt["model"])
    opt = torch.optim.SGD(m.parameters(), lr=1.0)
    opt.load_state_dict(ckpt["optimizer"])
    assert (opt.param_groups[0]["momentum"], opt.param_groups[0]["weight_decay"]) == (MOM, WD)
    want = _run_torch(m, opt, _lambda_lr(opt, last_epoch=opt.param_groups[0]["iteration"] - 1), grads,
                      range(SAVE, STEPS))

    ckpt = _load(blob)
    m = module_from_cfg(CFG, ckpt["model"])
    ours = _fused(m)
    ours.load_state_dict(ckpt["optimizer"])
    got = _run_fused(m, ours, grads, range(SAVE, STEPS))
    _assert_close(got, want)


def test_resume_through_the_captioner_is_bit_exact():
    """Real forward + BPTT + FusedClipSGD: 4 steps in one go against 2 steps, save, a new module and optimizer, load,
    2 more. The decoder LSTM is frozen on steps 1 and 2, across the save."""
    g = load_golden("train_tied_sv1")
    cfg = g["cfg"]
    args = (g["image_features"].cuda(), None, None, g["caption_tokens"].cuda(), g["sentiment"].cuda())

    def make(params):
        m = module_from_cfg(cfg, params)
        m.train()
        m._eps_override = g["eps"].cuda()
        return m, sscvae.FusedClipSGD(m.parameters(), lr=0.5, momentum=0.9, weight_decay=1e-3, max_norm=12.5,
                                      num_iterations=100)

    def run(m, opt, its):
        out = []
        for it in its:
            m._updown_cell._language_lstm_cell_decoder.requires_grad_(it not in (1, 2))     # train.py:156-161
            opt.zero_grad()
            o = m(*args)
            (o["loss"].mean() + o["kld"].mean() / 750.0).backward()
            opt.step()
            out.append((o["loss"].clone(), o["kld"].clone()))
        return out

    m, opt = make(g["params"])
    whole = run(m, opt, range(4))
    whole_state = m.state_dict()
    whole_bufs = opt.state_dict()["state"]

    m, opt = make(g["params"])
    head = run(m, opt, range(2))
    ckpt = _load(_checkpoint(m, opt))
    del m, opt
    torch.manual_seed(1)
    m, opt = make(ckpt["model"])
    opt.load_state_dict(ckpt["optimizer"])
    tail = run(m, opt, range(2, 4))

    for it, ((la, ka), (lb, kb)) in enumerate(zip(whole, head + tail, strict=True)):
        assert torch.equal(la, lb) and torch.equal(ka, kb), it
    state = m.state_dict()
    assert all(torch.equal(state[k], v) for k, v in whole_state.items()), \
        [k for k, v in whole_state.items() if not torch.equal(state[k], v)]
    bufs = opt.state_dict()["state"]
    assert bufs.keys() == whole_bufs.keys()
    assert all(torch.equal(bufs[i]["momentum_buffer"], whole_bufs[i]["momentum_buffer"]) for i in bufs)
