"""Fused training-step tail (SURVEY §8(f)-1): clip_grad_norm_ + SGD(momentum, weight decay) + the
linear-decay learning-rate schedule of var_updown/scripts/train.py:126-134,173-176, as three kernel
launches over all parameter tensors instead of ~100 eager launches."""
import ctypes as C
from typing import Iterable

import torch

from . import _lib
from .captioner import PACKED_OWNERS


class FusedClipSGD(torch.optim.Optimizer):
    """`step()` == clip_grad_norm_(params, max_norm); SGD.step(); LambdaLR.step() of the reference loop.

    Parameters that currently have no gradient are left untouched, as torch's SGD does for
    `p.grad is None` (frozen embedding; decoder LSTM under the freeze schedule, train.py:156-161).

    `legacy_zero_grad=True` reproduces the reference's PINNED torch 1.1.0 (requirements.txt:12) instead:
    there `optimizer.zero_grad()` leaves zero tensors, not None, so a parameter that has had a gradient once
    and is then frozen keeps being updated with a zero gradient (weight decay + momentum coasting). With it,
    `zero_grad()` zeroes nothing on the device: such parameters are handed to the kernel with a NULL gradient.

    Checkpoints: `state_dict()` / `load_state_dict()` use torch.optim.SGD's format (one parameter group, state keyed
    by parameter index, `state[p]["momentum_buffer"]`). The kernel applies the same momentum rule with dampening 0, so
    buffers move between the two unchanged: `torch.optim.SGD(...).load_state_dict(opt.state_dict())` works, and so does
    the reverse. Besides SGD's keys the group carries `initial_lr` (base of the linear decay, the key LambdaLR uses),
    `max_norm`, `num_iterations` and `iteration`. A dict without `iteration` (a torch.optim.SGD checkpoint) restarts the
    schedule at iteration 0 from its `initial_lr` (or its `lr`), as the reference's own resume does (train.py:142-151);
    keys it lacks are taken from the constructor.

    Packed operands: when the parameters being updated all belong to one UpDownCaptioner whose packed bf16 / fp32
    operands are current, `step()` writes the updated operands in the same pass (one launch instead of the update
    followed by a re-pack of every updated weight at the next forward); results are bit-identical. `fuse_pack=False`
    always takes the plain update, after which the next forward re-packs."""

    def __init__(self, params: Iterable[torch.nn.Parameter], lr=0.015, momentum=0.9, weight_decay=0.001,
                 max_norm=12.5, num_iterations=70000, legacy_zero_grad=False, fuse_pack=True):
        defaults = dict(lr=lr, momentum=momentum, dampening=0, weight_decay=weight_decay, nesterov=False,
                        maximize=False, foreach=None, differentiable=False, fused=None,
                        max_norm=max_norm, num_iterations=num_iterations, iteration=0)
        super().__init__(params, defaults)
        if len(self.param_groups) != 1:
            raise ValueError("FusedClipSGD takes one parameter group")
        self.param_groups[0].setdefault("initial_lr", self.param_groups[0]["lr"])
        self.legacy_zero_grad = legacy_zero_grad
        self.fuse_pack = fuse_pack
        self._partial = None

    def __setstate__(self, state):
        super().__setstate__(state)
        for group in self.param_groups:
            if "iteration" not in group:
                group["lr"] = group.setdefault("initial_lr", group["lr"])
            for k, v in self.defaults.items():
                group.setdefault(k, v)

    def load_state_dict(self, state_dict):
        """torch.optim.Optimizer.load_state_dict, refusing options the kernel does not implement."""
        for g in state_dict["param_groups"]:
            if g.get("dampening", 0) != 0 or g.get("nesterov", False) or g.get("maximize", False):
                raise ValueError("FusedClipSGD implements SGD with dampening=0, nesterov=False, maximize=False; the "
                                 f"loaded group has dampening={g.get('dampening')}, nesterov={g.get('nesterov')}, "
                                 f"maximize={g.get('maximize')}")
        super().load_state_dict(state_dict)

    @property
    def lr(self) -> float:
        """Learning rate of the next step: initial_lr · (1 − iteration / num_iterations) (train.py:132-134), unless a
        scheduler has set it since."""
        return self.param_groups[0]["lr"]

    @property
    def iteration(self) -> int:
        return self.param_groups[0]["iteration"]

    def zero_grad(self):
        for p in self.param_groups[0]["params"]:
            p.grad = None

    @torch.no_grad()
    def step(self, grad_scale: float = 1.0):
        """`grad_scale` multiplies every gradient before clipping and the update. Data-parallel training passes
        1 / world_size together with `BucketedGradReducer.reduce(..., average=False)`: the all-reduce leaves the SUM in
        the buckets and no extra pass divides them."""
        L = _lib.lib()
        group, state = self.param_groups[0], self.state

        def buffer(p):                     # `state` is a defaultdict: look up without creating entries
            s = state.get(p)
            return None if s is None else s.get("momentum_buffer")

        legacy = self.legacy_zero_grad
        ps = [p for p in group["params"] if p.grad is not None or (legacy and buffer(p) is not None)]
        if not ps:
            return
        dev = ps[0].device
        if not ps[0].is_cuda:
            raise RuntimeError("FusedClipSGD runs only on CUDA parameters; there is no CPU fallback")
        # all tensors in three launches: squared-norm partials over a fixed chunking, their ordered sum, the update
        if len(ps) > 32:
            raise RuntimeError("FusedClipSGD handles at most 32 parameter tensors (the captioner has 22, 21 trainable)")
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        grads = [None if p.grad is None else p.grad.contiguous() for p in ps]
        bufs, firsts, new = [], [], []
        for p in ps:
            b = buffer(p)
            first = b is None
            if first:                      # the kernel writes the buffer without reading it
                b = torch.empty_like(p, dtype=torch.float32, memory_format=torch.contiguous_format)
                new.append((p, b))
            elif b.dtype != torch.float32 or b.device != p.device or not b.is_contiguous():
                # a loaded buffer the kernel cannot write through a raw pointer: replace it once
                b = state[p]["momentum_buffer"] = b.to(device=p.device, dtype=torch.float32,
                                                       memory_format=torch.contiguous_format)
            if b.shape != p.shape:
                raise ValueError(f"momentum buffer of shape {tuple(b.shape)} for a parameter of shape {tuple(p.shape)}")
            bufs.append(b)
            firsts.append(int(first))
        n = len(ps)
        chunks = sum((p.numel() + 16383) // 16384 for p in ps)
        if self._partial is None or self._partial.numel() < chunks + 1 or self._partial.device != dev:
            self._partial = torch.empty(chunks + 1, dtype=torch.float32, device=dev)
        hyper = (group["max_norm"], group["lr"], group["momentum"], group["weight_decay"], grad_scale)
        owner = PACKED_OWNERS.get(ps[0]) if self.fuse_pack else None
        owner = owner() if owner is not None else None
        if owner is None or not owner._sgd_step_packed(ps, grads, bufs, firsts, hyper, self._partial):
            vp = C.c_void_p
            _lib.check(L.sscvae_sgd_step_multi(
                n, (vp * n)(*[p.data_ptr() for p in ps]), (vp * n)(*[None if g is None else g.data_ptr() for g in grads]),
                (vp * n)(*[b.data_ptr() for b in bufs]), (C.c_uint64 * n)(*[p.numel() for p in ps]),
                (C.c_int32 * n)(*firsts), *[float(h) for h in hyper], _lib.ptr(self._partial), self._partial.numel(),
                stream))
            for p in ps:
                # the kernel wrote through raw pointers: tell autograd (and the captioner's packed-weight cache, which
                # is keyed on the version counters) that the parameters changed
                torch.autograd.graph.increment_version(p)
        for p, b in new:
            state[p]["momentum_buffer"] = b
        group["iteration"] += 1
        group["lr"] = group["initial_lr"] * (1 - group["iteration"] / group["num_iterations"])    # train.py:132-134
