"""GPU: UpDownCaptioner._decode_step, the reference's per-step decode (updown_captioner.py:371-455), against the reference's
golden step, the bf16 oracle, the fused decode it shares its kernels with, and the searches it drives."""
from functools import partial

import pytest
import torch

import sscvae
from conftest import load_golden
from helpers import module_from_cfg, rel_err
from oracle import fsm_oracle as fo
from oracle import search_oracle as so
from oracle import updown_oracle as uo

pytestmark = pytest.mark.gpu

TOL_LOGITS_VS_FP32_REF = 3e-2        # the decode / training tolerances against fp32 golden data and the bf16 oracle
TOL_LOGITS_VS_BF16_ORACLE = 6e-3
TOL_ALPHA = 5e-3
TOL_STATE = 1e-2                     # max-abs difference of a state relative to its largest entry (bf16 oracle)
KEYS = ("h1", "c1", "h_encoder", "c_encoder", "h_decoder", "c_decoder")


def _cfg(sv=1, E=600, le="glove", V=300, H=40, Z=16, L=20):
    return dict(vocab_size=V, image_feature_size=64, embedding_size=E, hidden_size=H, attention_projection_size=24, z_space=Z,
                sentiment_vae=sv, simple_vae=False, max_caption_length=L, prior_std=0.8, senti_prior_multip=0.5,
                latent_embedding=le)


def test_step_matches_reference_fixture():
    """decode_step_tied.npz: the unmodified reference's _decode_step on random input states, with its eps."""
    g = load_golden("decode_step_tied")
    cfg = g["cfg"]
    m = module_from_cfg(cfg, g["params"])
    m.eval()
    B, Z = g["image_features"].shape[0], cfg["z_space"]
    m._eps_override = g["eps"].cuda()
    sent = g["sentiment"].cuda()
    logp, st, pm, plv, alpha = m._decode_step(g["image_features"].cuda(), None, g["prev"].cuda(),
                                              {k: v.cuda() for k, v in g["state_in"].items()}, sentiment=sent,
                                              prior_mean=sent.repeat(1, Z) * 0.5, prior_var=torch.ones(B, Z).cuda())
    assert rel_err(logp, g["logp"]) < TOL_LOGITS_VS_FP32_REF
    for k in KEYS:
        assert rel_err(st[k], g["state_out"][k]) < TOL_LOGITS_VS_FP32_REF, k
    assert torch.equal(st["h_encoder"].cpu(), g["state_in"]["h_encoder"])            # eval: the encoder pair passes through
    R = g["prev"].numel()
    assert torch.allclose(pm.cpu(), torch.full((R, Z), 0.5)) and torch.equal(plv.cpu(), torch.zeros(R, Z))
    assert torch.allclose(alpha.sum(1).cpu(), torch.ones(R), atol=1e-5)


CASES = [(0, "glove", 600), (1, "glove", 600), (1, "glove", 48), (2, "glove", 600), (2, "senti_word_net", 48)]


@pytest.mark.parametrize("rows_per_image", [1, 5, 40])
@pytest.mark.parametrize("sv,le,E", CASES)
def test_step_matches_bf16_oracle(sv, le, E, rows_per_image):
    """Every element of the 5-tuple against the oracle's decoder_step in Rounding("bf16"), with zero states and the
    default prior, and with random states and a caller-given per-image prior."""
    cfg = _cfg(sv, E, le)
    torch.manual_seed(sv * 10 + E)
    m = module_from_cfg(cfg, use_cbs=False)
    m.eval()
    B, N, Z, H = 3, 6, cfg["z_space"], cfg["hidden_size"]
    R = B * rows_per_image
    gen = torch.Generator().manual_seed(7)
    feats = torch.rand(B, N, 64, generator=gen)
    feats[1, 4:] = 0                                                      # ragged boxes
    sent = torch.tensor([[1.0], [-1.0], [0.0]])
    obj = torch.randn(B, N, Z, generator=gen) if sv == 2 else None
    ocfg = uo.OracleConfig(**cfg)
    p = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    q = uo.Rounding("bf16")
    o_feats, o_mask, o_avg, o_proj = uo.image_precompute(p, ocfg, feats, q)
    rep = lambda x: None if x is None else x.repeat_interleave(rows_per_image, dim=0)
    for given in (False, True):
        prev = torch.randint(0, cfg["vocab_size"], (R,), generator=gen)
        eps = torch.randn(R, Z, generator=gen)
        if given:
            states = {k: torch.randn(R, H, generator=gen) * 0.5 for k in KEYS}
            prior_mean, prior_var = torch.randn(B, Z, generator=gen), torch.rand(B, Z, generator=gen) + 0.3
        else:
            states, (prior_mean, prior_var) = None, (None, None)
        m._eps_override = eps.cuda()
        cuda = lambda x: None if x is None else x.cuda()
        out = m._decode_step(feats.cuda(), cuda(obj), prev.cuda(), None if states is None else {k: v.cuda() for k, v in states.items()},
                             sentiment=sent.cuda(), prior_mean=cuda(prior_mean), prior_var=cuda(prior_var))
        logp, st, pm, plv, alpha = [x if isinstance(x, dict) else x.cpu() for x in out]
        o_pm, o_pv = uo.prior(ocfg, sent, B)
        if given:
            o_pm, o_pv = prior_mean, prior_var
        logits, o_st, aux = uo.decoder_step(p, ocfg, rep(o_feats), rep(o_mask), rep(o_avg), rep(o_proj), prev,
                                            states if states is not None else uo.zero_states(R, H), rep(sent), rep(o_pm),
                                            rep(o_pv), eps, False, q, rep(obj))
        o_logp = torch.log_softmax(logits, dim=1)
        assert logp.shape == (R, cfg["vocab_size"]) and alpha.shape == (R, N) and pm.shape == (R, Z)
        assert rel_err(logp, o_logp) < TOL_LOGITS_VS_BF16_ORACLE, given
        for k in KEYS:
            assert rel_err(st[k], o_st[k]) < TOL_STATE, (k, given)
        assert (alpha - aux["alpha"]).abs().max().item() < TOL_ALPHA
        assert rel_err(pm, aux["prior_mean"]) < (1e-2 if sv == 2 else 1e-6)
        assert torch.allclose(plv, aux["log_var"], rtol=1e-6, atol=1e-6)


def test_step_search_equals_fused_decode():
    """sscvae.ConstrainedBeamSearch driven by partial(model._decode_step, ...) as the reference does
    (updown_captioner.py:325-343), S 8 (three constraints), K 5, external eps: the same search as the fused sscvae_decode.

    The step's logits come from the same head GEMM on the same bf16 operands as the fused decode's (at 120 rows the fused
    decode stores them from the 64-column tile kernel, the step from the 128-column one that carries the softmax
    statistics; both run the same K loop), so they are expected to be bit-identical, and checked as far as log_probs
    can show it. The log-sum-exp is merged from the GEMM's per-tile partials (exp2 based), so log_probs match
    `logits - torch.logsumexp(logits)` to a few ulp of the log-sum-exp, not bit for bit."""
    cfg = _cfg(1, 600, V=1000, H=64, L=8)
    torch.manual_seed(11)
    B, N, S, K, P, Z, L = 3, 6, 8, 5, 2, cfg["z_space"], cfg["max_caption_length"]
    SK, R = S * K, B * S * K
    m = module_from_cfg(cfg, beam_size=K, use_cbs=True)
    m.eval()
    gen = torch.Generator().manual_seed(5)
    feats = torch.rand(B, N, 64, generator=gen).cuda()
    sent = torch.tensor([[1.0], [-1.0], [0.0]]).cuda()
    fsm = torch.from_numpy(fo.single_word_fsm([[5, 6], [9], [12]], cfg["vocab_size"]))[None].repeat(B, 1, 1, 1)
    eps = torch.randn(L, R, Z, generator=gen)
    m._eps_override = eps.cuda()
    m(feats, None, None, fsm=fsm.cuda(), num_constraints=torch.tensor([3] * B).cuda(), sentiment=sent)
    fused = m.last_search["predictions"].cpu()
    ws_logits = m.decode_region(B, N, S, K, "logits", torch.float32, (R, cfg["vocab_size"])).clone()

    prior_mean = sent.repeat(1, Z) * cfg["senti_prior_multip"]              # what the reference's forward passes
    prior_var = torch.full((B, Z), cfg["prior_std"]).pow(2).cuda()             # (prior_std * prior_std) in fp32, as forward
    decode_step = partial(m._decode_step, feats, None, sentiment=sent, prior_mean=prior_mean, prior_var=prior_var)
    recorded = []

    def step(last, states):
        t = len(recorded)
        m._eps_override = (eps[0, ::SK] if t == 0 else eps[t]).cuda()     # the fused decode's rows of step t
        out = decode_step(last, states)
        recorded.append(out[0].cpu())
        return out
    cbs = sscvae.ConstrainedBeamSearch(1, max_steps=L, beam_size=K, per_node_beam_size=P)
    preds, scores = cbs.search(torch.ones(B, dtype=torch.long, device="cuda"), None, step, fsm.cuda())
    m._eps_override = None
    # the oracle search replayed on the recorded log-probabilities: the repo's standard of exactness
    ctr = {"t": 0}

    def replay(last, state):
        t = ctr["t"]; ctr["t"] += 1
        return recorded[t], {}
    op, os_ = so.cbs_search(torch.ones(B, dtype=torch.long), replay, fsm, K, P, 1, L)
    assert torch.equal(preds.cpu(), op) and torch.equal(scores.cpu(), os_)
    # same search as the fused decode, and at its last step the same rows: compare with its workspace logits
    assert len(recorded) == L, "a beam search that exits early leaves nothing to compare at the last step"
    assert torch.equal(preds.cpu(), fused)
    ref = (ws_logits - torch.logsumexp(ws_logits, dim=1, keepdim=True)).cpu()
    lse = torch.logsumexp(ws_logits, dim=1).abs().max().item()
    assert (recorded[-1] - ref).abs().max().item() <= 8 * torch.finfo(torch.float32).eps * max(1.0, lse)
    # the logits themselves agree: every row of the step's log_probs is exactly fl(logits - c) of the fused decode's logits
    # for one fp32 c (its log-sum-exp, recovered from the row's largest entry, where |logit - c| is smallest, +-2 ulp).
    # log_probs cannot resolve every last bit of a logit, but a different summation order, which moves many logits of a
    # row by an ulp, fails this check
    x, y = ws_logits.cpu(), recorded[-1]
    top = x.argmax(dim=1, keepdim=True)
    c0 = (x.gather(1, top).double() - y.gather(1, top).double()).float()
    exact = torch.zeros(x.shape[0], dtype=torch.bool)
    c = c0.clone()
    for _ in range(2):
        c = torch.nextafter(c, torch.full_like(c, -float("inf")))
    for _ in range(5):
        exact |= ((x - c) == y).all(dim=1)
        c = torch.nextafter(c, torch.full_like(c, float("inf")))
    assert bool(exact.all()), f"{int((~exact).sum())} of {x.shape[0]} rows: logits differ from the fused decode's"


def test_greedy_step_search_equals_forward():
    cfg = _cfg(1, 48, L=20)
    torch.manual_seed(2)
    B, N, Z, L = 4, 5, cfg["z_space"], cfg["max_caption_length"]
    m = module_from_cfg(cfg, beam_size=1, use_cbs=False)
    m.eval()
    gen = torch.Generator().manual_seed(9)
    feats = torch.rand(B, N, 64, generator=gen).cuda()
    sent = torch.tensor([[1.0], [-1.0], [0.0], [0.5]]).cuda()
    eps = torch.randn(L, B, Z, generator=gen)
    m._eps_override = eps.cuda()
    pred = m(feats, sentiment=sent)["predictions"].cpu()
    calls = []

    def step(last, states):
        m._eps_override = eps[len(calls)].cuda()
        calls.append(1)
        return m._decode_step(feats, None, last, states, sentiment=sent)
    preds, _ = sscvae.BeamSearch(1, max_steps=L, beam_size=1).search(torch.ones(B, dtype=torch.long, device="cuda"), None, step)
    m._eps_override = None
    got = preds[:, 0].cpu()
    n = min(got.shape[1], pred.shape[1])
    assert torch.equal(got[:, :n], pred[:, :n])
    assert bool((got[:, n:] == 1).all()) and bool((pred[:, n:] == 1).all())


def test_image_state_cache():
    """The same feature tensor reuses the per-image state (3 launches fewer); a new tensor or an in-place edit recomputes it."""
    cfg = _cfg(1, 600)
    torch.manual_seed(4)
    B, N, Z, H = 3, 6, cfg["z_space"], cfg["hidden_size"]
    R = B * 5
    m = module_from_cfg(cfg, use_cbs=False)
    m.eval()
    gen = torch.Generator().manual_seed(1)
    feats = torch.rand(B, N, 64, generator=gen).cuda()
    sent = torch.tensor([[1.0], [-1.0], [0.0]]).cuda()
    prev = torch.randint(0, cfg["vocab_size"], (R,), generator=gen).cuda()
    states = {k: (torch.randn(R, H, generator=gen) * 0.5).cuda() for k in KEYS}
    pm, pv = sent.repeat(1, Z) * 0.5, torch.ones(B, Z).cuda()
    m._eps_override = torch.randn(R, Z, generator=gen).cuda()
    run = lambda f: m._decode_step(f, None, prev, states, sentiment=sent, prior_mean=pm, prior_var=pv)[0]

    def launches(f):
        torch.cuda.synchronize()
        n0 = sscvae._lib.launch_count()
        out = run(f)
        torch.cuda.synchronize()
        return sscvae._lib.launch_count() - n0, out.cpu()
    run(feats)                                                     # packs the weights, sizes the workspace
    n_same, a = launches(feats)
    # one step on cached image state: import, embedding, 2 x (gate GEMM + LSTM), query GEMM, attention, latent,
    # output projection + head GEMM (tied), log-softmax
    assert n_same == 12, n_same
    other = feats.clone()
    n_new, b = launches(other)
    assert n_new == n_same + 3 and torch.equal(a, b)               # image_prep, W_v projection, mean-feature gate block
    assert launches(other)[0] == n_same
    other.mul_(0.5)                                                # in place: the version counter moves
    n_edit, c = launches(other)
    assert n_edit == n_same + 3
    assert torch.equal(c, launches(other.clone())[1]) and not torch.equal(c, a)
    # inputs the module converts (fp16, non-contiguous) go through a temporary copy whose storage the allocator may hand to
    # the next call's copy: the decision follows the caller's tensor, so different features of the same shape recompute
    f1 = torch.rand(B, N, 64, generator=gen).half().cuda()
    f2 = torch.rand(B, N, 64, generator=gen).half().cuda()
    launches(f1)
    assert launches(f1)[0] == n_same
    n_f2, d = launches(f2)
    assert n_f2 == n_same + 3 and torch.equal(d, launches(f2.float())[1])
    wide = torch.rand(B, N, 128, generator=gen).cuda()
    s1, s2 = wide[..., :64], wide[..., 64:]
    launches(s1)
    assert launches(s1)[0] == n_same
    n_s2, e = launches(s2)
    assert n_s2 == n_same + 3 and torch.equal(e, launches(s2.contiguous())[1])


def test_step_calls_leave_forward_and_sample_unchanged():
    cfg = _cfg(1, 48)
    torch.manual_seed(6)
    B, N, Z, L, J = 3, 5, cfg["z_space"], cfg["max_caption_length"], 4
    m = module_from_cfg(cfg, beam_size=1, use_cbs=False)
    m.eval()
    m.return_attention = True
    gen = torch.Generator().manual_seed(3)
    feats = torch.rand(B, N, 64, generator=gen).cuda()
    sent = torch.tensor([[1.0], [-1.0], [0.0]]).cuda()
    eps_f, eps_s = torch.randn(L, B, Z, generator=gen).cuda(), torch.randn(L, B * J, Z, generator=gen).cuda()

    def both():
        m._eps_override = eps_f
        f = m(feats, sentiment=sent)
        m._eps_override = eps_s
        s = m.sample(feats, sentiment=sent, n_samples=J)
        m._eps_override = None
        return {k: v.cpu() for k, v in f.items()}, {k: v.cpu() for k, v in s.items()}
    f0, s0 = both()
    st = None
    last = torch.ones(B * 2, dtype=torch.long, device="cuda")
    for _ in range(3):
        logp, st, *_ = m._decode_step(feats, None, last, st, sentiment=sent)
        last = logp.argmax(1)
    f1, s1 = both()
    for a, b in ((f0, f1), (s0, s1)):
        assert a.keys() == b.keys()
        for k in a:
            assert torch.equal(a[k], b[k]), k


def test_training_mode_and_bad_rows_are_refused():
    cfg = _cfg(1, 48)
    m = module_from_cfg(cfg, use_cbs=False)
    feats, sent = torch.rand(2, 3, 64).cuda(), torch.zeros(2, 1).cuda()
    m.train()
    with pytest.raises(NotImplementedError, match="training"):
        m._decode_step(feats, None, torch.ones(2, dtype=torch.long).cuda(), None, sentiment=sent)
    m.eval()
    with pytest.raises(ValueError, match="multiple"):
        m._decode_step(feats, None, torch.ones(3, dtype=torch.long).cuda(), None, sentiment=sent)
