"""CPU: FusedClipSGD's checkpoint surface (SURVEY 8(f)-1, checkpoint format {"model", "optimizer"}).

Its state_dict is torch.optim.SGD's (one group, state keyed by parameter index, momentum buffers under
"momentum_buffer"), so a reference checkpoint written by SGD + LambdaLR (checkpointing.py:101-103) resumes into it
(train.py:142-151). The optimizer is only constructed and loaded here; its step() needs the GPU
(tests/test_gpu_resume.py)."""
import copy

import pytest
import torch

import sscvae
from helpers import module_from_cfg

CFG = dict(vocab_size=300, image_feature_size=64, embedding_size=600, hidden_size=32, attention_projection_size=24,
           z_space=16, sentiment_vae=1, simple_vae=False, max_caption_length=20, prior_std=1.0, senti_prior_multip=0.5)
LR, MOM, WD, CLIP, NIT = 0.05, 0.9, 1e-3, 0.5, 40


def _module():
    torch.manual_seed(0)
    return module_from_cfg(CFG, device="cpu")


def _reference_checkpoint(m, steps=3):
    """The reference loop's optimizer (train.py:126-134,173-176) after a few CPU steps: its state_dict."""
    opt = torch.optim.SGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lr_lambda=lambda it: 1 - it / NIT)
    g = torch.Generator().manual_seed(1)
    for _ in range(steps):
        for p in m.parameters():
            if p.requires_grad:
                p.grad = torch.randn(p.shape, generator=g)
        torch.nn.utils.clip_grad_norm_(m.parameters(), CLIP)
        opt.step()
        sched.step()
    return opt, opt.state_dict()


def test_state_dict_has_torch_sgd_layout():
    m = _module()
    ours = sscvae.FusedClipSGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD, max_norm=CLIP, num_iterations=NIT)
    ref = torch.optim.SGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD)
    assert isinstance(ours, torch.optim.Optimizer)
    a, b = ours.state_dict(), ref.state_dict()
    assert a.keys() == b.keys()
    assert [g["params"] for g in a["param_groups"]] == [g["params"] for g in b["param_groups"]]
    assert len(a["param_groups"][0]["params"]) == 22           # model.parameters(): the tied embedding counted once
    assert set(b["param_groups"][0]) <= set(a["param_groups"][0])
    group = a["param_groups"][0]
    assert (group["lr"], group["initial_lr"], group["momentum"], group["weight_decay"]) == (LR, LR, MOM, WD)
    assert (group["dampening"], group["nesterov"], group["maximize"]) == (0, False, False)
    assert (group["max_norm"], group["num_iterations"], group["iteration"]) == (CLIP, NIT, 0)
    assert (ours.lr, ours.iteration) == (LR, 0)
    # the reference's scheduler accepts it (isinstance check) and finds the base of the decay where it looks for it
    sched = torch.optim.lr_scheduler.LambdaLR(ours, lr_lambda=lambda it: 1 - it / NIT)
    assert sched.base_lrs == [LR] and ours.lr == LR


def test_torch_sgd_checkpoint_loads_and_restarts_the_schedule():
    m = _module()
    ref, sd = _reference_checkpoint(m)
    assert sd["param_groups"][0]["lr"] < LR                    # the saved schedule had moved on
    ours = sscvae.FusedClipSGD(m.parameters(), lr=0.5, momentum=0.5, weight_decay=0.0, max_norm=CLIP,
                               num_iterations=NIT)
    ours.load_state_dict(copy.deepcopy(sd))
    trainable = [p for p in m.parameters() if p.requires_grad]
    assert len(ours.state) == len(trainable) == 21
    for p in trainable:
        assert torch.equal(ours.state[p]["momentum_buffer"], ref.state[p]["momentum_buffer"])
    group = ours.param_groups[0]
    assert ours.iteration == 0 and ours.lr == group["initial_lr"] == LR
    assert (group["momentum"], group["weight_decay"]) == (MOM, WD)       # from the checkpoint
    assert (group["max_norm"], group["num_iterations"]) == (CLIP, NIT)   # not in it: from the constructor
    # without LambdaLR's initial_lr, the saved lr is the base of the restarted schedule
    del sd["param_groups"][0]["initial_lr"]
    ours = sscvae.FusedClipSGD(m.parameters(), lr=0.5, num_iterations=NIT)
    ours.load_state_dict(sd)
    assert ours.iteration == 0 and ours.lr == ours.param_groups[0]["initial_lr"] == sd["param_groups"][0]["lr"]


def test_fused_checkpoint_keeps_its_schedule_and_hyperparameters():
    m = _module()
    src = sscvae.FusedClipSGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD, max_norm=CLIP, num_iterations=NIT)
    src.param_groups[0].update(iteration=5, lr=LR * (1 - 5 / NIT))
    dst = sscvae.FusedClipSGD(m.parameters(), lr=1.0, momentum=0.0, weight_decay=0.0, max_norm=99.0, num_iterations=7)
    dst.load_state_dict(src.state_dict())
    assert {k: v for k, v in dst.param_groups[0].items() if k != "params"} == \
        {k: v for k, v in src.param_groups[0].items() if k != "params"}
    assert dst.iteration == 5 and dst.lr == LR * (1 - 5 / NIT)
    # torch's SGD takes the same dict: it ignores the extra keys, and they survive its load
    ref = torch.optim.SGD(m.parameters(), lr=1.0)
    ref.load_state_dict(src.state_dict())
    assert ref.param_groups[0]["iteration"] == 5 and ref.param_groups[0]["lr"] == dst.lr


@pytest.mark.parametrize("change", [dict(dampening=0.1), dict(nesterov=True), dict(maximize=True), "size"])
def test_load_refuses_what_the_kernel_does_not_implement(change):
    m = _module()
    _, sd = _reference_checkpoint(m, steps=1)
    if change == "size":
        sd["param_groups"][0]["params"] = sd["param_groups"][0]["params"][:-1]
    else:
        sd["param_groups"][0].update(change)
    ours = sscvae.FusedClipSGD(m.parameters(), lr=LR, num_iterations=NIT)
    with pytest.raises(ValueError):
        ours.load_state_dict(sd)
    assert len(ours.state) == 0 and ours.lr == LR                  # left as it was


def test_one_parameter_group_only():
    m = _module()
    ps = [p for p in m.parameters() if p.requires_grad]
    with pytest.raises(ValueError):
        sscvae.FusedClipSGD([{"params": ps[:3]}, {"params": ps[3:]}])
