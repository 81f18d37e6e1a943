"""GPU: the attention weights behind every word (`return_attention`): from eval forward(), sample() and the training
forward. Checked against the bf16 oracle replayed along the device's tokens, against a host back-trace over the decode
workspace's step histories, and for the switch leaving every other output and the launch plan unchanged."""
import pytest
import torch

import sscvae
from conftest import load_golden
from helpers import module_from_cfg, oracle_params
from oracle import fsm_oracle as fo
from oracle import updown_oracle as uo

pytestmark = pytest.mark.gpu

# the small dims of tests/test_gpu_sample_search.py
CFG = dict(vocab_size=400, image_feature_size=64, embedding_size=600, hidden_size=40, attention_projection_size=24,
           z_space=12, simple_vae=False, max_caption_length=20, prior_std=0.7, senti_prior_multip=0.5)
BENCH = dict(vocab_size=10000, image_feature_size=2048, embedding_size=600, hidden_size=900, attention_projection_size=768,
             z_space=150, sentiment_vae=1, simple_vae=False, max_caption_length=20, prior_std=1.0, senti_prior_multip=0.5)
B, J, N, Z, L = 3, 5, 6, 12, 20
TOL_ALPHA = 5e-3                     # the alpha tolerance of the training tests against the bf16 oracle


def _inputs(sv, seed=2, rows=B * J):
    gen = torch.Generator().manual_seed(seed)
    feats = torch.rand(B, N, 64, generator=gen)
    feats[0, 3:] = 0                                                # ragged boxes
    feats[2, 5:] = 0
    sent = torch.tensor([[1.0], [-1.0], [0.0]]) if sv == 1 else None
    obj = torch.randn(B, N, Z, generator=gen) * 0.5 if sv == 2 else None
    eps = torch.randn(L, rows, Z, generator=gen)
    return feats, sent, obj, eps


def _model(sv, K=1, use_cbs=False, min_sat=2, end_boost=0.0):
    torch.manual_seed(3)
    m = module_from_cfg(dict(CFG, sentiment_vae=sv), beam_size=K, use_cbs=use_cbs, min_sat=min_sat)
    m.eval()
    if end_boost:                   # searches end after a few steps, at a step that depends on the latent draws
        with torch.no_grad():
            e1 = m._embedding_layer.weight[1]
            m._output_projection[0].bias += end_boost * e1 / e1.norm()
    return m


def _cuda(t):
    return None if t is None else t.cuda()


def _first_boundary(tokens):
    """(rows, n) tokens -> index of each row's first boundary token (n when there is none)."""
    n = tokens.shape[1]
    hit = tokens == 1
    return torch.where(hit.any(1), hit.float().argmax(1), torch.full((tokens.shape[0],), n))


# ---- 1. the switch is inert ------------------------------------------------------------------------------------------
def _twice(m, call):
    """call() with the switch off, then on (each after a warm-up call of its own): outputs, launches of each."""
    res = []
    for on in (False, True):
        m.return_attention = on
        call()
        c0 = sscvae._lib.launch_count()
        out = call()
        torch.cuda.synchronize()
        res.append((out, sscvae._lib.launch_count() - c0))
    m.return_attention = False
    return res


def _same(a, b):
    if isinstance(a, dict):                     # the keys of the switched-off call: everything but "attention"
        return all(_same(a[k], b[k]) for k in a)
    if torch.is_tensor(a):
        return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a.cpu(), b.cpu())
    return a == b


def _check_inert(m, call):
    """call() -> (output dict, last_search dict)"""
    (off, n_off), (on, n_on) = _twice(m, call)
    assert _same(off[0], on[0]) and _same(off[1], on[1])
    assert "attention" not in off[0] and "attention" in on[0]
    assert n_on == n_off + 1, (n_off, n_on)            # one launch more: the trace kernel
    return on[0]


def test_switch_is_inert_for_greedy_decode_and_sample():
    m = _model(1)
    feats, sent, _, eps = _inputs(1)

    def fwd():
        m._eps_override = eps[:, :B].contiguous().cuda()
        out = m(feats.cuda(), sentiment=sent.cuda())
        return out, dict(m.last_search)
    _check_inert(m, fwd)

    def smp():
        m._eps_override = eps.cuda()
        return m.sample(feats.cuda(), sentiment=sent.cuda(), n_samples=J), {}
    on = _check_inert(m, smp)
    assert on["attention"].shape == (B, J, on["predictions"].shape[2], N)


@pytest.mark.parametrize("per_sample", [0, 1])
def test_switch_is_inert_for_cbs_decode_and_sample(per_sample):
    S, K = 4, 3
    m = _model(1, K=K, use_cbs=True)
    feats, sent, _, eps = _inputs(1, rows=B * J * S * K)
    fsm = torch.from_numpy(fo.single_word_fsm([[5, 6], [9]], 400))[None].repeat(B, 1, 1, 1)

    def fwd():
        m._eps_override = eps[:, :B * S * K].contiguous().cuda()
        out = m(feats.cuda(), sentiment=sent.cuda(), fsm=fsm.cuda(), num_constraints=torch.tensor([2] * B).cuda())
        return out, dict(m.last_search)
    _check_inert(m, fwd)

    T = B * J if per_sample else B
    f = fsm.repeat_interleave(J, dim=0) if per_sample else fsm

    def smp():
        m._eps_override = eps.cuda()
        out = m.sample(feats.cuda(), sentiment=sent.cuda(), n_samples=J, fsm=f.cuda(), num_constraints=torch.tensor([2] * T).cuda())
        return out, dict(m.last_search)
    _check_inert(m, smp)


# ---- 2. values match the oracle ----------------------------------------------------------------------------------------
def _oracle_alphas(m, feats, sent, obj, eps, tokens, per_image):
    """The bf16 oracle cell replayed along the device's tokens: (rows, steps, N) alpha, rows = B * per_image, row r reading
    image r // per_image and eps row r."""
    cfg = uo.OracleConfig(**dict(CFG, sentiment_vae=m.sentiment_vae))
    p = oracle_params({k: v.detach().cpu() for k, v in m.state_dict().items()}, cfg)
    q = uo.Rounding("bf16")
    rows, steps = tokens.shape
    fe, mask, avg, proj = uo.image_precompute(p, cfg, feats, q)
    rep = lambda x: None if x is None else x.repeat_interleave(per_image, dim=0)
    prior_mean, prior_var = uo.prior(cfg, sent, B)
    states = uo.zero_states(rows, cfg.hidden_size)
    last = torch.ones(rows, dtype=torch.long)
    out = []
    for t in range(steps):
        _, states, aux = uo.decoder_step(p, cfg, rep(fe), rep(mask), rep(avg), rep(proj), last, states, rep(sent),
                                         rep(prior_mean), rep(prior_var), eps[t], False, q, rep(obj))
        out.append(aux["alpha"])
        last = tokens[:, t]
    return torch.stack(out, dim=1), rep(mask)


def _check_against_oracle(att, tokens, oracle, mask):
    """att (rows, n, N) from the device, tokens (rows, n), oracle (rows, n, N)."""
    first = _first_boundary(tokens)
    worst = 0.0
    for r in range(tokens.shape[0]):
        e = int(first[r]) + 1 if int(first[r]) < tokens.shape[1] else tokens.shape[1]
        a = att[r, :e]
        worst = max(worst, (a - oracle[r, :e]).abs().max().item())
        assert bool((a[:, ~mask[r]] == 0).all()), r                  # masked boxes: exactly 0
        assert (a.sum(1) - 1).abs().max().item() < 1e-5, r            # a distribution over the unmasked boxes
        assert bool((att[r, e:] == 0).all()), r                       # after the first boundary token: exactly 0
    assert worst < TOL_ALPHA, worst


@pytest.mark.parametrize("sv", [1, 2])
def test_sample_attention_matches_the_oracle(sv):
    m = _model(sv)
    feats, sent, obj, eps = _inputs(sv)
    m._eps_override = eps.cuda()
    m.return_attention = True
    out = m.sample(feats.cuda(), sentiment=_cuda(sent), n_samples=J, obj_atts=_cuda(obj))
    pred, att = out["predictions"].cpu(), out["attention"]
    n = pred.shape[2]
    assert att.shape == (B, J, n, N) and att.dtype == torch.float32 and not att.requires_grad
    oracle, mask = _oracle_alphas(m, feats, sent, obj, eps[:n], pred.view(B * J, n), J)
    _check_against_oracle(att.cpu().view(B * J, n, N), pred.view(B * J, n), oracle, mask)


@pytest.mark.parametrize("sv", [1, 2])
def test_greedy_decode_attention_matches_the_oracle(sv):
    m = _model(sv)
    feats, sent, obj, eps = _inputs(sv, rows=B)
    m._eps_override = eps.cuda()
    m.return_attention = True
    out = m(feats.cuda(), sentiment=_cuda(sent), obj_atts=_cuda(obj))
    pred, att = out["predictions"].cpu(), out["attention"].cpu()
    n = pred.shape[1]
    assert att.shape == (B, n, N)
    assert m.last_search["attention"].shape == (B, 1, 1, n, N)
    assert torch.equal(m.last_search["attention"][:, 0, 0].cpu(), att)
    oracle, mask = _oracle_alphas(m, feats, sent, obj, eps[:n], pred, 1)
    _check_against_oracle(att, pred, oracle, mask)


# ---- 3. the gather is exact along the CBS path ---------------------------------------------------------------------------
def _host_trace(tok, bp, alpha, g, SK, w, n, steps):
    """The back-trace of search group g, beam w from step n - 1 over the workspace histories: (tokens (n,), attention
    (steps, N)) with the zeros after the first boundary token and from step n on."""
    base = g * SK
    toks, rows = [0] * n, [0] * n
    cur = w
    for t in range(n - 1, 0, -1):
        toks[t] = int(tok[t, base + cur])
        cur = int(bp[t, base + cur])
        rows[t] = base + cur
    toks[0] = int(tok[0, base + cur])
    rows[0] = g
    out = torch.zeros(steps, alpha.shape[2])
    for t in range(n):
        out[t] = alpha[t, rows[t]]
        if toks[t] == 1:
            break
    return torch.tensor(toks), out


def _chosen_state(scores0, nc, min_sat, valid):
    """The selection rules of decoding.py:82-135 over the beam-0 scores (S,) of one search."""
    S = scores0.shape[0]
    if valid is not None:
        ok = [bool(valid[s]) for s in range(S)]
    else:
        need = min(nc, min_sat)
        ok = [s < (1 << nc) and bin(s).count("1") >= need for s in range(S)]
    best, bv = 0, None
    for s in range(S):
        if ok[s] and (bv is None or float(scores0[s]) > bv):
            best, bv = s, float(scores0[s])
    return best


def _words(S):
    return {4: [[5, 6], [9]], 8: [[5, 6], [9], [11]]}[S]


def _c2s(S):
    """object c0 with attributes (constraint i moves to the states with bit i): (constraints, constraint2states, the
    valid-state mask the object / attribute rule gives with min_sat 1)."""
    names = ["c0", "c1", "c2"][:{4: 2, 8: 3}[S]]
    c2s = {c: [s for s in range(S) if s >> i & 1] for i, c in enumerate(names)}
    cons = [("c0", names[1:])]
    valid = torch.zeros(S, dtype=torch.uint8)
    valid[sscvae.valid_states_with_attributes(len(names), cons, c2s, 1)] = 1
    return cons, c2s, valid


@pytest.mark.parametrize("S,K", [(4, 3), (8, 5)])
@pytest.mark.parametrize("cbs_simple", [True, False])
def test_cbs_decode_attention_is_the_gather_along_the_back_trace(S, K, cbs_simple):
    m = _model(1, K=K, use_cbs=True, min_sat=1)
    m.cbs_simple = cbs_simple
    SK, R = S * K, B * S * K
    feats, sent, _, eps = _inputs(1, rows=R)
    fsm = torch.from_numpy(fo.single_word_fsm(_words(S), 400))[None].repeat(B, 1, 1, 1)
    nc = torch.tensor([len(_words(S))] * B)
    kw = {}
    valid = None
    if not cbs_simple:
        cons, c2s, valid = _c2s(S)
        kw = dict(constraints=[cons] * B, constraint2states=[c2s] * B)
    m._eps_override = eps.cuda()
    m.return_attention = True
    out = m(feats.cuda(), sentiment=sent.cuda(), fsm=fsm.cuda(), num_constraints=nc.cuda(), **kw)
    pred, att = out["predictions"].cpu(), out["attention"].cpu()
    ls = m.last_search
    n = ls["n_steps"]
    every, allp, sc = ls["attention"].cpu(), ls["predictions"].cpu(), ls["log_probs"].cpu()
    assert every.shape == (B, S, K, n, N) and att.shape == (B, n, N)
    tok = m.decode_region(B, N, S, K, "tok_hist", torch.int32, (L, R)).cpu()
    bp = m.decode_region(B, N, S, K, "bp_hist", torch.int32, (L, R)).cpu()
    alpha = m.decode_region(B, N, S, K, "alpha_hist", torch.float32, (L, R, N)).cpu()
    for g in range(B):
        for w in range(SK):
            toks, expect = _host_trace(tok, bp, alpha, g, SK, w, n, L)
            assert torch.equal(toks, allp[g, w // K, w % K]), (g, w)
            assert torch.equal(every[g, w // K, w % K], expect[:n]), (g, w)
        st = _chosen_state(sc[g, :, 0], int(nc[g]), 1, valid)
        assert torch.equal(att[g], every[g, st, 0]), g
        assert torch.equal(pred[g], allp[g, st, 0]), g


@pytest.mark.parametrize("per_sample", [0, 1])
@pytest.mark.parametrize("cbs_simple", [True, False])
def test_sample_search_attention_is_the_gather_along_the_back_trace(per_sample, cbs_simple):
    S, K = 4, 3
    SK, R = S * K, B * J * S * K
    m = _model(1, K=K, use_cbs=True, min_sat=1, end_boost=0.4)
    m.cbs_simple = cbs_simple
    feats, sent, _, eps = _inputs(1, rows=R)
    T = B * J if per_sample else B
    words = [[[5, 6], [9]], [[7], [11, 12]], [[20], [21]]]
    fsm = torch.stack([torch.from_numpy(fo.single_word_fsm(words[t % 3], 400)) for t in range(T)])
    nc = torch.tensor([2] * T)
    kw = {}
    valid = None
    if not cbs_simple:
        cons, c2s, valid = _c2s(S)
        kw = dict(constraints=[cons] * T, constraint2states=[c2s] * T)
    m._eps_override = eps.cuda()
    m.return_attention = True
    out = m.sample(feats.cuda(), sentiment=sent.cuda(), n_samples=J, fsm=fsm.cuda(), num_constraints=nc.cuda(), **kw)
    pred, att, ns = out["predictions"].cpu(), out["attention"].cpu(), out["n_steps"].cpu()
    ls = m.last_search
    every, allp, sc = ls["attention"].cpu(), ls["predictions"].cpu(), ls["log_probs"].cpu()
    n = int(ns.max())
    assert int(ns.min()) < n                                        # searches stop at different steps
    assert every.shape == (B, J, S, K, n, N) and att.shape == (B, J, n, N)
    tok = m.sample_search_region(B, N, J, S, K, per_sample, "tok_hist", torch.int32, (L, R)).cpu()
    bp = m.sample_search_region(B, N, J, S, K, per_sample, "bp_hist", torch.int32, (L, R)).cpu()
    alpha = m.sample_search_region(B, N, J, S, K, per_sample, "alpha_hist", torch.float32, (L, R, N)).cpu()
    for g in range(B * J):
        b, j = divmod(g, J)
        ng = int(ns[b, j])
        for w in range(SK):
            toks, expect = _host_trace(tok, bp, alpha, g, SK, w, ng, L)
            assert torch.equal(toks, allp[b, j, w // K, w % K, :ng]), (g, w)
            assert torch.equal(every[b, j, w // K, w % K], expect[:n]), (g, w)
            assert bool((every[b, j, w // K, w % K, ng:] == 0).all())     # its own zero tail
        st = _chosen_state(sc[b, j, :, 0], 2, 1, valid)
        assert torch.equal(att[b, j], every[b, j, st, 0]), g
        assert torch.equal(pred[b, j], allp[b, j, st, 0]), g


# ---- 4. images are independent ---------------------------------------------------------------------------------------------
def test_decode_attention_of_a_batch_is_independent_per_image():
    """Mirrors test_decode_batch_of_images_is_independent_per_image: attention of image b in a batch equals the attention
    of image b decoded alone with the same eps rows."""
    g = load_golden("decode_e2e_cbs_k5")
    cfg = g["cfg"]
    S, K, Z = g["fsm"].shape[1], 5, cfg["z_space"]
    m = module_from_cfg(cfg, g["params"], beam_size=K, use_cbs=True)
    m.eval()
    m.return_attention = True
    gen = torch.Generator().manual_seed(0)
    nb = 3
    feats = torch.rand(nb, 7, cfg["image_feature_size"], generator=gen)
    feats[1, 4:] = 0
    fsm = g["fsm"].repeat(nb, 1, 1, 1)
    sent = torch.tensor([[1.0], [-1.0], [0.0]])
    eps = torch.randn(20, nb * S * K, Z, generator=gen)
    nc = g["num_constraints"].repeat(nb)
    m._eps_override = eps.cuda()
    full = m(feats.cuda(), None, None, fsm=fsm.cuda(), num_constraints=nc.cuda(), sentiment=sent.cuda())["attention"].cpu()
    for b in range(nb):
        m._eps_override = eps[:, b * S * K:(b + 1) * S * K].contiguous().cuda()
        one = m(feats[b:b + 1].cuda(), None, None, fsm=fsm[b:b + 1].cuda(), num_constraints=nc[b:b + 1].cuda(),
                sentiment=sent[b:b + 1].cuda())["attention"].cpu()
        n = min(one.shape[1], full.shape[1])
        assert torch.equal(one[0, :n], full[b, :n]), b
        assert bool((one[0, n:] == 0).all()) and bool((full[b, n:] == 0).all())   # both captions have ended by then


# ---- 5. training --------------------------------------------------------------------------------------------------------
def _train_case(cfg, Bt, Nt, obj=False):
    torch.manual_seed(0)
    m = module_from_cfg(cfg)
    m.train()
    gen = torch.Generator().manual_seed(1)
    F, Zt, T = cfg["image_feature_size"], cfg["z_space"], cfg["max_caption_length"] + 1
    feats = torch.rand(Bt, Nt, F, generator=gen)
    feats[0, Nt // 2:] = 0
    toks = torch.randint(2, cfg["vocab_size"], (Bt, cfg["max_caption_length"]), generator=gen)
    for b in range(Bt):
        toks[b, 3 + b % 15:] = 0
    sent = torch.randint(-1, 2, (Bt, 1), generator=gen).float()
    om = torch.randn(Bt, Nt, Zt, generator=gen) * 0.5 if obj else None
    eps = torch.randn(T, Bt, Zt, generator=gen)
    m._eps_override = eps.cuda()

    def step(on):
        m.return_attention = on
        m.zero_grad(set_to_none=True)
        out = m(feats.cuda(), _cuda(om), None, toks.cuda(), sent.cuda())
        (out["loss"].mean() + out["kld"].mean() / 750.0).backward()
        grads = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
        return out, grads
    return m, step, T


@pytest.mark.parametrize("cfg,Bt,Nt,obj", [
    (BENCH, 4, 36, False),                                          # persistent forward kernel
    (BENCH, 256, 36, False),
    (dict(CFG, sentiment_vae=2), 6, 7, True),                      # per-launch forward path
], ids=["sv1_b4", "sv1_b256", "sv2_b6"])
def test_training_attention_is_the_stored_alpha(cfg, Bt, Nt, obj):
    m, step, T = _train_case(cfg, Bt, Nt, obj)
    if not obj:
        assert sscvae._lib.lib().sscvae_train_backward_is_persistent(m._handle, Bt, Nt) == 1
    off, g_off = step(False)
    assert "attention" not in off
    on, g_on = step(True)
    att = on["attention"]
    assert att.shape == (Bt, T, Nt) and att.dtype == torch.float32 and not att.requires_grad and att.is_contiguous()
    alpha = m.train_region(Bt, Nt, "alpha", torch.float32, (T, Bt, Nt))
    assert torch.equal(att, alpha.transpose(0, 1))
    assert att.data_ptr() != alpha.data_ptr()
    assert torch.equal(off["loss"], on["loss"]) and torch.equal(off["kld"], on["kld"])
    assert g_off.keys() == g_on.keys()
    for k in g_off:
        assert torch.equal(g_off[k], g_on[k]), k
    # a distribution over each image's boxes at every step
    assert (att.sum(-1) - 1).abs().max().item() < 1e-4
