"""GPU: UpDownCaptioner._decode_step in training mode (`stepwise_training = True`), the reference's differentiable training
step (updown_captioner.py:371-455, driven by its training loop, updown_captioner.py:263-323), against the reference's golden
training runs, the bf16 oracle under autograd, and the fused training forward / backward it shares its kernels with."""
import pytest
import torch

from conftest import load_golden
from helpers import module_from_cfg, oracle_params, rel_err
from oracle import updown_oracle as uo

pytestmark = pytest.mark.gpu

TRAIN = ["train_tied_sv1", "train_tied300_sv0", "train_untied_sv1", "train_tied_simple", "train_tied_sv2_glove",
         "train_untied_sv2_swn"]
TOL_LOGITS_VS_FP32_REF = 3e-2        # the bars tests/test_gpu_train.py holds the fused path to
TOL_LOSS_VS_FP32_REF = 2e-2
TOL_GRAD_VS_FP32_REF = 6e-2
TOL_LOGITS_VS_BF16_ORACLE = 6e-3     # the decode-step bars (tests/test_gpu_decode_step.py)
TOL_ALPHA = 5e-3
TOL_STATE = 1e-2
TOL_GRAD_VS_BF16_ORACLE = 2e-2
TOL_LOSS_VS_FUSED = 3e-3             # relative per caption
TOL_GRAD_VS_FUSED = 4e-3             # of the largest entry: the bar between the two backward paths
KEYS = ("h1", "c1", "h_encoder", "c_encoder", "h_decoder", "c_decoder")


def stepwise_train(m, feats, caps, sent, eps, obj=None):
    """The reference's training branch (updown_captioner.py:263-323) on top of model._decode_step: boundary tokens, one step
    per timestep with the prior mean reassigned from the step, the per-step KL masked by the token mask, _get_loss.
    eps: (T, B, Z), one slice per step. Returns {"loss", "kld", "logits" (B, T, V)}."""
    ocfg = uo.OracleConfig(**m._test_cfg)
    tokens = uo.add_boundary_tokens(caps, 0, 1)
    T = tokens.shape[1] - 1
    tmask = (tokens[:, 1:] != 0).float()
    B, Z = feats.shape[0], m.z_space
    prior_var = torch.full((B, Z), float(m.prior_std), device=feats.device).pow(2)
    prior_mean, states, logits_t, kl_t = None, None, [], []
    for t in range(T):
        m._eps_override = None if eps is None else eps[t]
        logits, states, mean, log_var, prior_mean, prior_log_var, alpha = m._decode_step(
            feats, obj, tokens[:, t], states, sentiment=sent, prior_mean=prior_mean, prior_var=prior_var)
        kl_t.append(uo.kl_step(ocfg, mean, log_var, prior_mean, prior_var))
        logits_t.append(logits)
    logits = torch.stack(logits_t, dim=1)
    klds = torch.stack(kl_t, dim=1) * tmask
    logp = torch.log_softmax(logits, dim=-1)
    nll = -logp.gather(2, tokens[:, 1:].unsqueeze(-1)).squeeze(-1) * tmask
    lengths = tmask.sum(-1)
    return {"loss": lengths * (nll.sum(1) / (lengths + 1e-13)), "kld": klds.sum(1), "logits": logits}


def objective(out):
    return out["loss"].mean() + out["kld"].mean() / 750.0          # train.py:168-171


def _module(cfg, params=None, **kw):
    m = module_from_cfg(cfg, params, use_cbs=False, **kw)
    m._test_cfg = cfg
    m.train()
    m.stepwise_training = True
    return m


def _golden(name):
    g = load_golden(name)
    obj = g["obj_means"].cuda() if "obj_means" in g else None
    return g, (g["image_features"].cuda(), g["caption_tokens"].cuda(), g["sentiment"].cuda(), g["eps"].cuda(), obj)


def _grads(m):
    return {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}


@pytest.mark.parametrize("name", TRAIN)
def test_stepwise_loop_matches_reference_fixture(name):
    g, (feats, caps, sent, eps, obj) = _golden(name)
    m = _module(g["cfg"], g["params"])
    out = stepwise_train(m, feats, caps, sent, eps, obj)
    objective(out).backward()
    scale, kscale = g["loss"].abs().clamp(min=1.0), g["kld"].abs().clamp(min=1.0)
    assert ((out["loss"].detach().cpu() - g["loss"]).abs() / scale).max() < TOL_LOSS_VS_FP32_REF
    assert ((out["kld"].detach().cpu() - g["kld"]).abs() / kscale).max() < TOL_LOSS_VS_FP32_REF
    assert rel_err(out["logits"], g["logits"]) < TOL_LOGITS_VS_FP32_REF
    grads = _grads(m)
    assert set(grads) == set(g["grads"])
    bad = {k: rel_err(grads[k], ref) for k, ref in g["grads"].items() if not rel_err(grads[k], ref) < TOL_GRAD_VS_FP32_REF}
    assert not bad, bad


def _cfg(sv=1, E=600, le="glove", simple=False, V=300, H=40, Z=16):
    return dict(vocab_size=V, image_feature_size=64, embedding_size=E, hidden_size=H, attention_projection_size=24, z_space=Z,
                sentiment_vae=sv, simple_vae=simple, max_caption_length=20, prior_std=0.8, senti_prior_multip=0.5,
                latent_embedding=le)


CASES = [(0, "glove", 600, False), (1, "glove", 600, False), (1, "glove", 48, False), (2, "glove", 600, False),
         (2, "senti_word_net", 48, False), (2, "glove", 48, True), (1, "glove", 600, True)]


@pytest.mark.parametrize("sv,le,E,simple", CASES)
def test_step_and_its_gradients_match_bf16_oracle(sv, le, E, simple):
    """All seven outputs against the oracle's training decoder_step in Rounding("bf16") from random states; then random
    upstream gradients on every differentiable output against oracle autograd."""
    cfg = _cfg(sv, E, le, simple)
    torch.manual_seed(sv * 10 + E + simple)
    m = _module(cfg)
    B, N, Z, H, V = 5, 6, cfg["z_space"], cfg["hidden_size"], cfg["vocab_size"]
    gen = torch.Generator().manual_seed(3)
    feats = torch.rand(B, N, 64, generator=gen)
    feats[1, 4:] = 0                                                          # ragged boxes
    sent = torch.tensor([[1.0], [-1.0], [0.0], [1.0], [0.0]])
    obj = torch.randn(B, N, Z, generator=gen) if sv == 2 and not simple else None
    prev = torch.randint(0, V, (B,), generator=gen)
    prev[2] = 0                                                               # the padding token
    eps = torch.randn(B, Z, generator=gen)
    states = {k: torch.randn(B, H, generator=gen) * 0.5 for k in KEYS}
    prior_mean, prior_var = torch.randn(B, Z, generator=gen), torch.rand(B, Z, generator=gen) + 0.3
    ocfg = uo.OracleConfig(**cfg)
    p = oracle_params({k: v.detach().cpu() for k, v in m.state_dict().items()}, ocfg, grad=True)
    q = uo.Rounding("bf16")
    o_st = {k: v.clone().requires_grad_(True) for k, v in states.items()}
    o_feats, o_mask, o_avg, o_proj = uo.image_precompute(p, ocfg, feats, q)
    # (simple_vae with sentiment_vae == 2 zeroes the attention-weighted prior mean; the oracle still forms it)
    o_obj = obj if obj is not None or sv != 2 else torch.zeros(B, N, Z)
    o_logits, o_new, aux = uo.decoder_step(p, ocfg, o_feats, o_mask, o_avg, o_proj, prev, o_st, sent, prior_mean, prior_var,
                                           eps, True, q, o_obj)
    d_st = {k: v.cuda().requires_grad_(True) for k, v in states.items()}
    m._eps_override = eps.cuda()
    logits, st, mean, log_var, pm, plv, alpha = m._decode_step(
        feats.cuda(), None if obj is None else obj.cuda(), prev.cuda(), d_st, sentiment=sent.cuda(),
        prior_mean=prior_mean.cuda(), prior_var=prior_var.cuda())
    assert rel_err(logits, o_logits) < TOL_LOGITS_VS_BF16_ORACLE
    for k in KEYS:
        assert rel_err(st[k], o_new[k]) < TOL_STATE, k
    assert rel_err(mean, aux["mean"]) < TOL_STATE and rel_err(log_var, aux["log_var"]) < TOL_STATE
    assert (alpha.detach().cpu() - aux["alpha"].detach()).abs().max() < TOL_ALPHA
    assert (pm.detach().cpu() - aux["prior_mean"].detach()).abs().max() < TOL_ALPHA * max(1.0, 0 if obj is None else obj.abs().max())
    assert torch.allclose(plv.cpu(), prior_var.log())
    if simple:
        assert not pm.any()
    # backward: random upstream gradients on every differentiable output
    outs = [("logits", logits, o_logits), ("mean", mean, aux["mean"]), ("log_var", log_var, aux["log_var"]),
            ("alpha", alpha, aux["alpha"])] + [(k, st[k], o_new[k]) for k in KEYS]
    if sv == 2 and not simple:
        outs.append(("prior_mean", pm, aux["prior_mean"]))
    assert all(t.requires_grad for _, t, _ in outs)
    up = {k: torch.randn(t.shape, generator=gen) for k, t, _ in outs}
    sum(((t * up[k].cuda()).sum() for k, t, _ in outs)).backward()
    sum(((t * up[k]).sum() for k, _, t in outs)).backward()
    for k in KEYS:
        assert rel_err(d_st[k].grad, o_st[k].grad) < TOL_GRAD_VS_BF16_ORACLE, k
    named = dict(m.named_parameters())
    if not m._tied:
        p["_embedding_layer.weight"].grad[0] = 0                               # nn.Embedding(padding_idx=0)
    bad = {}
    for k, prm in named.items():
        if not prm.requires_grad:
            assert prm.grad is None, k
            continue
        e = rel_err(prm.grad, p[k].grad)
        if not e < TOL_GRAD_VS_BF16_ORACLE:
            bad[k] = e
    assert not bad, bad


def _bench_batch(cfg, B, N, seed=0):
    g = torch.Generator().manual_seed(seed)
    feats = torch.rand(B, N, cfg["image_feature_size"], generator=g)
    feats[0, N // 2:] = 0
    toks = torch.randint(2, cfg["vocab_size"], (B, cfg["max_caption_length"]), generator=g)
    lens = torch.randint(3, cfg["max_caption_length"] + 1, (B,), generator=g)
    for b in range(B):
        toks[b, lens[b]:] = 0
    sent = torch.randint(-1, 2, (B, 1), generator=g).float()
    eps = torch.randn(cfg["max_caption_length"] + 1, B, cfg["z_space"], generator=g)
    return feats.cuda(), toks.cuda(), sent.cuda(), eps.cuda()


BENCH_CFG = dict(vocab_size=10000, image_feature_size=2048, embedding_size=600, hidden_size=900, attention_projection_size=768,
                 z_space=150, sentiment_vae=1, simple_vae=False, max_caption_length=20, prior_std=1.0, senti_prior_multip=0.5)


def _against_fused(m, feats, caps, sent, eps, obj=None):
    m._eps_override = eps
    fused = m(feats, obj, None, caps, sent)
    objective(fused).backward()
    g_fused = _grads(m)
    m.zero_grad(set_to_none=True)
    step = stepwise_train(m, feats, caps, sent, eps, obj)
    objective(step).backward()
    g_step = _grads(m)
    for k in ("loss", "kld"):
        a, b = step[k].detach(), fused[k].detach()
        assert ((a - b).abs() / b.abs().clamp(min=1.0)).max() < TOL_LOSS_VS_FUSED, k
    assert set(g_step) == set(g_fused)
    bad = {k: rel_err(g_step[k], g_fused[k]) for k in g_fused if not rel_err(g_step[k], g_fused[k]) < TOL_GRAD_VS_FUSED}
    assert not bad, bad


@pytest.mark.parametrize("name", ["train_tied_sv1", "train_untied_sv2_swn"])
def test_stepwise_loop_matches_fused_forward_at_golden_size(name):
    g, (feats, caps, sent, eps, obj) = _golden(name)
    _against_fused(_module(g["cfg"], g["params"]), feats, caps, sent, eps, obj)


def test_stepwise_loop_matches_fused_forward_at_bench_dims():
    torch.manual_seed(0)
    m = _module(BENCH_CFG)
    _against_fused(m, *_bench_batch(BENCH_CFG, 256, 36))


def test_frozen_parameters_get_no_gradient():
    g, (feats, caps, sent, eps, obj) = _golden("train_tied_sv1")
    m = _module(g["cfg"], g["params"])
    objective(stepwise_train(m, feats, caps, sent, eps)).backward()
    full = _grads(m)
    m.zero_grad(set_to_none=True)
    dec = list(m._updown_cell._language_lstm_cell_decoder.parameters())
    for p in dec:
        p.requires_grad_(False)
    objective(stepwise_train(m, feats, caps, sent, eps)).backward()
    assert all(p.grad is None for p in dec)
    assert m._embedding_layer.weight.grad is None                              # the tied (frozen GloVe) embedding
    part = _grads(m)
    assert set(part) == set(full) - {n for n, p in m.named_parameters() if any(p is q for q in dec)}
    for k in part:
        assert rel_err(part[k], full[k]) < 1e-6, k
    # untied: the learned embedding gets a scatter-add of its rows; the padding row stays zero (padding_idx)
    g, (feats, caps, sent, eps, obj) = _golden("train_untied_sv1")
    m = _module(g["cfg"], g["params"])
    objective(stepwise_train(m, feats, caps, sent, eps)).backward()
    emb = m._embedding_layer.weight.grad
    assert emb is not None and not emb[0].any() and emb.abs().sum() > 0


def _run_alone(m, batch):
    m.zero_grad(set_to_none=True)
    out = stepwise_train(m, *batch)
    objective(out).backward()
    return out["loss"].detach().clone(), _grads(m)


def test_interleaved_graphs_over_different_features_are_independent():
    g, (feats, caps, sent, eps, _) = _golden("train_tied_sv1")
    m = _module(g["cfg"], g["params"])
    A = (feats, caps, sent, eps)
    B = (torch.rand_like(feats), caps.flip(0).contiguous(), sent.flip(0).contiguous(), torch.randn_like(eps))
    la, ga = _run_alone(m, A)
    lb, gb = _run_alone(m, B)
    m.zero_grad(set_to_none=True)
    oa = stepwise_train(m, *A)
    ob = stepwise_train(m, *B)
    objective(ob).backward()
    gb2 = _grads(m)
    m.zero_grad(set_to_none=True)
    # neither a fused forward nor a sample() call between a step's forward and its backward changes anything
    m._eps_override = eps
    m(feats, None, None, caps, sent)
    m.eval()
    m._eps_override = None
    m.sample(feats, sentiment=sent, n_samples=2)
    m.train()
    objective(oa).backward()
    ga2 = _grads(m)
    assert torch.equal(oa["loss"], la) and torch.equal(ob["loss"], lb)
    for k in ga:
        assert torch.equal(ga[k], ga2[k]) and torch.equal(gb[k], gb2[k]), k


def test_inplace_parameter_edit_before_backward_raises():
    g, (feats, caps, sent, eps, _) = _golden("train_tied_sv1")
    m = _module(g["cfg"], g["params"])
    out = stepwise_train(m, feats, caps, sent, eps)
    with torch.no_grad():
        m._updown_cell.fc_mean.weight.mul_(1.0)
    with pytest.raises(RuntimeError, match="inplace"):
        objective(out).backward()


def test_step_and_backward_do_not_synchronise_the_host():
    g, (feats, caps, sent, eps, _) = _golden("train_tied_sv1")
    m = _module(g["cfg"], g["params"])
    B, Z = feats.shape[0], m.z_space
    prev = caps[:, 0].contiguous()
    pv = torch.ones(B, Z, device="cuda")

    def two_steps():
        m._eps_override = None                                                   # Philox normals
        lg, st, mean, lv, pm, plv, a = m._decode_step(feats, None, prev, None, sentiment=sent, prior_var=pv)
        lg2, st, mean2, lv2, pm, plv, a2 = m._decode_step(feats, None, prev, st, sentiment=sent, prior_var=pv)
        return lg.sum() + lg2.sum() + mean2.sum() + a2.sum() + st["h_decoder"].sum()

    two_steps().backward()                                                       # warm-up: workspaces, packed weights
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        two_steps().backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    with torch.no_grad():
        lg, st, mean, lv, pm, plv, a = m._decode_step(feats, None, prev, None, sentiment=sent, prior_var=pv)
    assert not any(t.requires_grad for t in (lg, mean, lv, a, *st.values()))


def test_rows_must_equal_images_and_eval_mode_is_unchanged():
    g, (feats, caps, sent, eps, _) = _golden("train_tied_sv1")
    m = _module(g["cfg"], g["params"])
    with pytest.raises(ValueError, match="one per image"):
        m._decode_step(feats, None, torch.ones(2 * feats.shape[0], dtype=torch.long).cuda(), None, sentiment=sent)
    m.stepwise_training = False
    with pytest.raises(NotImplementedError, match="stepwise_training"):
        m._decode_step(feats, None, caps[:, 0], None, sentiment=sent)
    m.eval()
    m.stepwise_training = True
    logp = m._decode_step(feats, None, caps[:, 0], None, sentiment=sent)[0]
    assert not logp.requires_grad and torch.allclose(logp.exp().sum(1), torch.ones(feats.shape[0], device="cuda"), atol=1e-4)
