"""GPU parity of the training path (forward loss / KL / per-step tensors and BPTT gradients) against
the CPU oracle and the reference's golden vectors, through the drop-in module -> C ABI -> sm_100a kernels.

Tolerances (stated per north_star): the CUDA path feeds bf16 operands to the tensor cores with fp32
accumulation and keeps cell states / softmax / KL / CE in fp32.
  * against the oracle run with the SAME operand rounding (Rounding("bf16")):  tight — differences come
    only from accumulation order, tanh.approx in the attention scores and bf16 re-rounding flips;
  * against the reference's fp32 golden outputs: bf16-level.
"""
import pytest
import torch

from conftest import load_golden
from helpers import module_from_cfg, oracle_params, rel_err
from oracle import updown_oracle as uo

pytestmark = pytest.mark.gpu

TRAIN = ["train_tied_sv1", "train_tied300_sv0", "train_untied_sv1", "train_tied_simple"]

# per-step logits: |diff| / max|logit|
TOL_LOGITS_VS_BF16_ORACLE = 6e-3
TOL_LOGITS_VS_FP32_REF = 3e-2
TOL_LOSS_VS_BF16_ORACLE = 3e-3       # relative, per caption
TOL_LOSS_VS_FP32_REF = 2e-2
TOL_GRAD_VS_FP32_REF = 6e-2          # max-abs error relative to the largest entry of that gradient


def _run_cuda(name, train=True):
    g = load_golden(name)
    cfg = g["cfg"]
    m = module_from_cfg(cfg, g["params"])
    m.train()
    m._eps_override = g["eps"].cuda()
    out = m(g["image_features"].cuda(), None, None, g["caption_tokens"].cuda(), g["sentiment"].cuda())
    return g, cfg, m, out


@pytest.mark.parametrize("name", TRAIN)
def test_forward_matches_oracle_and_reference(name, monkeypatch):
    # the product path never writes the (T*B, V) logits (the head GEMM's epilogue keeps softmax statistics only);
    # this debug switch, read when the module is created, makes the forward store them as well
    monkeypatch.setenv("SSCVAE_DEBUG_LOGITS", "1")
    g, cfg, m, out = _run_cuda(name)
    ocfg = uo.OracleConfig(**cfg)
    B, N, _ = g["image_features"].shape
    T, V, Z = cfg["max_caption_length"] + 1, cfg["vocab_size"], cfg["z_space"]
    ob = uo.train_forward(oracle_params(g["params"], ocfg), ocfg, g["image_features"], g["caption_tokens"],
                          g["sentiment"], g["eps"], q=uo.Rounding("bf16"), record=True)
    torch.cuda.synchronize()
    logits = m.train_region(B, N, "logits", torch.float32, (T, B, V)).cpu().permute(1, 0, 2)
    tmask = m.train_region(B, N, "tmask", torch.float32, (T, B)).cpu().t()
    alpha = m.train_region(B, N, "alpha", torch.float32, (T, B, N)).cpu()
    mean = m.train_region(B, N, "mean", torch.float32, (T, B, Z)).cpu()
    logvar = m.train_region(B, N, "logvar", torch.float32, (T, B, Z)).cpu()
    # token bookkeeping (a16) is integer work: exact
    assert torch.equal(tmask, (ob["tokens"][:, 1:] != 0).float())
    # per-step intermediates vs the same-rounding oracle
    o_alpha = torch.stack([s["alpha"] for s in ob["steps"]])
    o_mean = torch.stack([s["mean"] for s in ob["steps"]])
    o_logvar = torch.stack([s["log_var"] for s in ob["steps"]])
    assert (alpha - o_alpha).abs().max() < 5e-3
    assert rel_err(mean, o_mean) < 1e-2 and rel_err(logvar, o_logvar) < 1e-2
    assert rel_err(logits, ob["logits"]) < TOL_LOGITS_VS_BF16_ORACLE
    assert rel_err(logits, g["logits"]) < TOL_LOGITS_VS_FP32_REF
    loss, kld = out["loss"].cpu(), out["kld"].cpu()
    scale = g["loss"].abs().clamp(min=1.0)
    assert ((loss - ob["loss"].detach()).abs() / scale).max() < TOL_LOSS_VS_BF16_ORACLE
    assert ((loss - g["loss"]).abs() / scale).max() < TOL_LOSS_VS_FP32_REF
    kscale = g["kld"].abs().clamp(min=1.0)
    assert ((kld - ob["kld"].detach()).abs() / kscale).max() < TOL_LOSS_VS_BF16_ORACLE
    assert ((kld - g["kld"]).abs() / kscale).max() < TOL_LOSS_VS_FP32_REF


@pytest.mark.parametrize("name", TRAIN)
def test_backward_matches_reference_gradients(name):
    g, cfg, m, out = _run_cuda(name)
    (out["loss"].mean() + out["kld"].mean() / 750.0).backward()        # train.py:168-172
    torch.cuda.synchronize()
    named = dict(m.named_parameters())
    assert set(g["grads"]) == {k for k, p in named.items() if p.grad is not None}
    worst = {}
    for k, ref in g["grads"].items():
        worst[k] = rel_err(named[k].grad, ref)
    bad = {k: v for k, v in worst.items() if not v < TOL_GRAD_VS_FP32_REF}
    assert not bad, bad


def test_frozen_decoder_lstm_gets_no_gradient():
    """train.py:156-161 toggles requires_grad of the decoder LSTM; its grads must then stay None and the
    other gradients must be unchanged."""
    g, cfg, m, out = _run_cuda("train_tied_sv1")
    for p in m._updown_cell._language_lstm_cell_decoder.parameters():
        p.requires_grad = False
    m._eps_override = g["eps"].cuda()
    out = m(g["image_features"].cuda(), None, None, g["caption_tokens"].cuda(), g["sentiment"].cuda())
    (out["loss"].mean() + out["kld"].mean() / 750.0).backward()
    assert all(p.grad is None for p in m._updown_cell._language_lstm_cell_decoder.parameters())
    k = "_updown_cell.fc_mean.weight"
    assert rel_err(dict(m.named_parameters())[k].grad, g["grads"][k]) < TOL_GRAD_VS_FP32_REF


def test_philox_path_is_seeded_and_stochastic():
    g, cfg, m, _ = _run_cuda("train_tied_sv1")
    m._eps_override = None
    args = (g["image_features"].cuda(), None, None, g["caption_tokens"].cuda(), g["sentiment"].cuda())
    torch.manual_seed(5); m._call_counter = 0
    a = m(*args)["loss"].clone()
    b = m(*args)["loss"].clone()
    torch.manual_seed(5); m._call_counter = 0
    c = m(*args)["loss"].clone()
    assert torch.equal(a, c) and not torch.equal(a, b)
    eps = m.train_region(6, g["image_features"].shape[1], "eps", torch.float32, (21 * 6 * cfg["z_space"],)).cpu()
    assert abs(eps.mean()) < 0.1 and abs(eps.std() - 1) < 0.1


def test_reference_rng_mode_replays_cpu_generator():
    """rng_mode='reference' draws one (B,Z) CPU normal per step like updown_cell.py:206, so seeding the CPU
    generator reproduces the golden run without passing eps."""
    g = load_golden("train_tied_sv1")
    m = module_from_cfg(g["cfg"], g["params"])
    m.train()
    m.rng_mode = "reference"
    torch.manual_seed(1234)
    out = m(g["image_features"].cuda(), None, None, g["caption_tokens"].cuda(), g["sentiment"].cuda())
    assert ((out["loss"].cpu() - g["loss"]).abs() / g["loss"].abs().clamp(min=1)).max() < TOL_LOSS_VS_FP32_REF


def test_optimizer_step_repacks_the_bf16_operand_copies():
    """FusedClipSGD writes the fp32 parameters through raw pointers; the next forward must run on re-packed bf16
    weights: it has to equal a fresh module built from the updated state_dict, not the previous step's loss."""
    import sscvae
    g = load_golden("train_tied_sv1")
    cfg = g["cfg"]
    m = module_from_cfg(cfg, g["params"])
    m.train()
    m._eps_override = g["eps"].cuda()
    args = (g["image_features"].cuda(), None, None, g["caption_tokens"].cuda(), g["sentiment"].cuda())
    opt = sscvae.FusedClipSGD([p for p in m.parameters() if p.requires_grad], lr=0.5, momentum=0.9, weight_decay=1e-3,
                              max_norm=12.5, num_iterations=100)
    out1 = m(*args)
    (out1["loss"].mean() + out1["kld"].mean() / 750.0).backward()
    before = {k: v.detach().clone() for k, v in m.state_dict().items()}
    grads = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
    opt.step()
    # the update itself: clip_grad_norm_(12.5) + SGD(momentum, wd), first step (train.py:173-176)
    norm = torch.sqrt(sum((v.double() ** 2).sum() for v in grads.values()))
    coef = min(1.0, 12.5 / (norm.item() + 1e-6))
    for k, p in m.named_parameters():
        if k in grads:
            want = before[k] - 0.5 * (grads[k] * coef + 1e-3 * before[k])
            assert torch.allclose(p.detach(), want, rtol=1e-5, atol=1e-6), k
    out2 = m(*args)
    fresh = module_from_cfg(cfg, {k: v.detach().cpu() for k, v in m.state_dict().items()})
    fresh.train()
    fresh._eps_override = g["eps"].cuda()
    out3 = fresh(*args)
    assert torch.equal(out2["loss"], out3["loss"]) and torch.equal(out2["kld"], out3["kld"])
    assert not torch.allclose(out2["loss"], out1["loss"])


def test_full_size_properties():
    """BASELINE config 2 shape (B=256, 36x2048, V=10k, L=20, dims Y): size-independent properties."""
    torch.manual_seed(0)
    cfg = dict(vocab_size=10000, image_feature_size=2048, embedding_size=600, hidden_size=900,
               attention_projection_size=768, z_space=150, sentiment_vae=1, simple_vae=False, max_caption_length=20,
               prior_std=1.0, senti_prior_multip=0.5)
    m = module_from_cfg(cfg)
    m.train()
    B = 256
    g = torch.Generator().manual_seed(0)
    feats = torch.rand(B, 36, 2048, generator=g)
    toks = torch.randint(2, 10000, (B, 20), generator=g)
    lens = torch.randint(5, 21, (B,), generator=g)
    for b in range(B):
        toks[b, lens[b]:] = 0
    sent = torch.randint(-1, 2, (B, 1), generator=g).float()
    eps = torch.randn(21, B, 150, generator=g)
    m._eps_override = eps.cuda()
    out = m(feats.cuda(), None, None, toks.cuda(), sent.cuda())
    loss = out["loss"]
    assert torch.isfinite(loss).all() and torch.isfinite(out["kld"]).all() and (out["kld"] >= 0).all()
    # rows are independent captions: the first 3 rows must match the oracle run on just those rows
    ocfg = uo.OracleConfig(**cfg)
    params = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    o = uo.train_forward(oracle_params(params, ocfg), ocfg, feats[:3], toks[:3], sent[:3], eps[:, :3].contiguous(),
                         q=uo.Rounding("bf16"))
    assert ((loss[:3].cpu() - o["loss"]).abs() / o["loss"].abs().clamp(min=1)).max() < 1e-2
    assert ((out["kld"][:3].cpu() - o["kld"]).abs() / o["kld"].abs().clamp(min=1)).max() < 1e-2
    (out["loss"].mean() + out["kld"].mean() / 750.0).backward()
    grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    assert all(torch.isfinite(v).all() for v in grads.values())
    # linearity / DP invariance: gradient of the full batch == sum of the two half-batch gradients
    acc = {k: torch.zeros_like(v) for k, v in grads.items()}
    for sl in (slice(0, 128), slice(128, 256)):
        for p in m.parameters():
            p.grad = None
        m._eps_override = eps[:, sl].contiguous().cuda()
        o = m(feats[sl].cuda(), None, None, toks[sl].cuda(), sent[sl].cuda())
        ((o["loss"].sum() + o["kld"].sum() / 750.0) / B).backward()
        for k, p in m.named_parameters():
            if p.grad is not None:
                acc[k] += p.grad
    for k in grads:
        assert rel_err(acc[k], grads[k]) < 2e-2, k
    # captions are independent rows: permuting the batch permutes the losses
    perm = torch.randperm(B, generator=g)
    m._eps_override = eps[:, perm].contiguous().cuda()
    o2 = m(feats[perm].cuda(), None, None, toks[perm].cuda(), sent[perm].cuda())
    assert torch.allclose(o2["loss"], loss[perm.cuda()], rtol=2e-3, atol=2e-2)
