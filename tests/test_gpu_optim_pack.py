"""GPU: FusedClipSGD's fused update of the weights and of the captioner's packed operands (sscvae_sgd_step_packed).

Two copies of a model take the same steps from the same gradients: one with the fused path, one with
`fuse_pack=False` (sscvae_sgd_step_multi, then a re-pack at the next use). After every step
  * parameters and momentum buffers are bit-equal between the two;
  * the fused model's packed buffer is byte-equal to a full pack (sscvae_pack_weights, dirty = NULL) of its updated
    weights, and to the other model's re-packed buffer.
Covered: first and later steps, clipping active and inactive, grad_scale != 1, legacy_zero_grad with NULL gradients over
the decoder-LSTM freeze interval, a weight edited in place between steps (the step falls back, the forward re-packs), an
optimizer over a subset of the parameters, and dims whose blocks have ragged and unaligned edges.
"""
import ctypes as C

import pytest
import torch

import sscvae
from sscvae import _lib
from helpers import module_from_cfg

pytestmark = pytest.mark.gpu

# H % 8 != 0, Z % 4 != 0, odd W_ih row lengths: scalar fp32 accesses and element stores at the edges of the bf16 images
CFG_SV1 = dict(vocab_size=300, image_feature_size=72, embedding_size=600, hidden_size=36, attention_projection_size=24,
               z_space=10, sentiment_vae=1, simple_vae=False, max_caption_length=20, prior_std=1.0,
               senti_prior_multip=0.5)
CFG_SV2 = dict(CFG_SV1, embedding_size=40, hidden_size=64, z_space=16, sentiment_vae=2)      # untied, [W_z | W_c] blocks
DEC = "_updown_cell._language_lstm_cell_decoder"


def _full_pack(m):
    L = _lib.lib()
    ws = m._weight_tensors()
    buf = torch.empty(L.sscvae_packed_bytes(m._handle), dtype=torch.uint8, device="cuda")
    _lib.check(L.sscvae_pack_weights(m._handle, _lib.ptr_array(ws), _lib.ptr(buf), buf.numel(), None,
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return buf


def _run(cfg, legacy=False, subset=None, edit_at=None, steps=5):
    torch.manual_seed(0)
    a = module_from_cfg(cfg)
    b = module_from_cfg(cfg, {k: v.detach().cpu() for k, v in a.state_dict().items()})
    named_a = [(k, p) for k, p in a.named_parameters() if p.requires_grad and (subset is None or subset(k))]
    named_b = [(k, p) for k, p in b.named_parameters() if p.requires_grad and (subset is None or subset(k))]
    kw = dict(lr=0.05, momentum=0.9, weight_decay=1e-3, max_norm=0.5, num_iterations=40, legacy_zero_grad=legacy)
    opt_a = sscvae.FusedClipSGD([p for _, p in named_a], fuse_pack=True, **kw)
    opt_b = sscvae.FusedClipSGD([p for _, p in named_b], fuse_pack=False, **kw)
    g = torch.Generator().manual_seed(1)
    fused_steps = 0
    for it in range(steps):
        a._packed_weights()                                 # the forward's pack (a no-op when it is current)
        b._packed_weights()
        if it == edit_at:                                   # an in-place edit between steps: the packed copy is stale
            with torch.no_grad():
                for m in (a, b):
                    m._updown_cell._attention_lstm_cell.weight_hh.mul_(0.5)
        frozen = legacy and it in (2, 3)                    # train.py:156-161: decoder LSTM frozen
        opt_a.zero_grad()
        opt_b.zero_grad()
        for (k, pa), (_, pb) in zip(named_a, named_b):
            if frozen and k.startswith(DEC):
                continue
            gr = torch.randn(pa.shape, generator=g) * (3.0 if it % 2 else 0.01)     # clip active / inactive
            pa.grad, pb.grad = gr.cuda(), gr.cuda()
        scale = 0.5 if it == 3 else 1.0
        opt_a.step(grad_scale=scale)
        opt_b.step(grad_scale=scale)
        current = a._packed_key == a._weights_key(a._weight_tensors())
        assert current == (it != edit_at), it               # fused unless the packed copy was stale
        fused_steps += current
        for (k, pa), (_, pb) in zip(named_a, named_b):
            assert torch.equal(pa, pb), (it, k)
            ma, mb = opt_a.state[pa].get("momentum_buffer"), opt_b.state[pb].get("momentum_buffer")
            assert (ma is None) == (mb is None) and (ma is None or torch.equal(ma, mb)), (it, k)
        pk = a._packed_weights()
        assert torch.equal(pk, _full_pack(a)), it
        assert torch.equal(pk, b._packed_weights()), it
    return fused_steps


@pytest.mark.parametrize("cfg", [CFG_SV1, CFG_SV2], ids=["sv1_tied", "sv2_untied"])
@pytest.mark.parametrize("legacy", [False, True])
def test_fused_step_equals_update_then_pack(cfg, legacy):
    assert _run(cfg, legacy=legacy) == 5


def test_weight_edited_in_place_falls_back_and_repacks():
    assert _run(CFG_SV1, edit_at=2) == 4


@pytest.mark.parametrize("cfg", [CFG_SV1, CFG_SV2], ids=["sv1_tied", "sv2_untied"])
def test_optimizer_over_a_subset_of_the_parameters(cfg):
    # without the attention LSTM's W_hh and b_hh: its folds and bias sums read them without updating them
    assert _run(cfg, legacy=True, subset=lambda k: not k.endswith(("weight_hh", "bias_hh"))) == 5
