"""GPU: sample() with use_cbs=True (sscvae_decode_samples_search): one constrained beam search per (image, latent sample)
in one call, against the reference's inference loop of one call per sample (var_updown/scripts/inference.py:138-167),
which runs each search as its own batch-1 call (inference.py:95, cbs.py:167)."""
import pytest
import torch

import sscvae
from helpers import module_from_cfg
from oracle import fsm_oracle as fo
from oracle import updown_oracle as uo

pytestmark = pytest.mark.gpu

# The small dims of test_decode_large_batch_path_replay. The batched call runs the cell's GEMMs with M = B*J*S*K = 144 rows
# (B*J = 12 at step 0), a batch-1 call with M = S*K = 12 (1 at step 0). Both take the same gemm_bf16_tn dispatch for every
# GEMM of the cell (N = the gate rows, A = 24, E = 600, V = 400): M <= 256 with N < 1024 stays off the CTA-pair kernel,
# M < 1024 off the 2-CTA tile kernel, and ceil(M/128) * ceil(N/128) <= 2 * 5 < 96 tiles on the same 64-wide (N > 32) or
# 32-wide (N = A) tile kernel, so every row is accumulated in the same order and results are comparable token for token.
CFG = dict(vocab_size=400, image_feature_size=64, embedding_size=600, hidden_size=40, attention_projection_size=24,
           z_space=12, simple_vae=False, max_caption_length=20, prior_std=0.7, senti_prior_multip=0.5)
B, J, S, K, N, Z, L = 3, 4, 4, 3, 6, 12, 20
SK = S * K


def _setup(sv, min_sat=2, end_boost=0.0):
    torch.manual_seed(3)
    m = module_from_cfg(dict(CFG, sentiment_vae=sv), beam_size=K, use_cbs=True, min_sat=min_sat)
    m.eval()
    if end_boost:
        # push the output projection towards the boundary token's embedding: searches end after a few steps, at a step that
        # depends on the latent draws
        with torch.no_grad():
            e1 = m._embedding_layer.weight[1]
            m._output_projection[0].bias += end_boost * e1 / e1.norm()
    gen = torch.Generator().manual_seed(2)
    feats = torch.rand(B, N, 64, generator=gen)
    feats[0, 3:] = 0
    feats[2, 5:] = 0
    sent = torch.tensor([[1.0], [-1.0], [0.0]]) if sv == 1 else None
    obj = torch.randn(B, N, Z, generator=gen) * 0.5 if sv == 2 else None
    eps = torch.randn(L, B * J * SK, Z, generator=gen)
    return m, feats, sent, obj, eps


def _cuda(t):
    return None if t is None else t.cuda()


def _table(fsm, rows):
    return sscvae.FsmBits(fsm.bits[rows]) if isinstance(fsm, sscvae.FsmBits) else fsm[rows].cuda()


def _sample(m, feats, sent, obj, eps, fsm, nc, **kw):
    m._eps_override = eps.cuda()
    out = m.sample(feats.cuda(), sentiment=_cuda(sent), n_samples=J, obj_atts=_cuda(obj), fsm=_table(fsm, slice(None)),
                   num_constraints=nc.cuda(), **kw)
    ls = m.last_search
    return (out["predictions"].cpu(), out["n_steps"].cpu(), ls["predictions"].cpu(), ls["log_probs"].cpu(),
            ls["n_steps"].cpu())


def _loop(m, feats, sent, obj, eps, fsm, nc, per_sample, constraints=None, c2s=None):
    """The reference's loop: B*J batch-1 forward() calls, call (b, j) fed the eps rows of search group b*J + j."""
    res = []
    for b in range(B):
        for j in range(J):
            g = b * J + j
            t = g if per_sample else b
            m._eps_override = eps[:, g * SK:(g + 1) * SK].contiguous().cuda()
            kw = {} if constraints is None else dict(constraints=[constraints[t]], constraint2states=[c2s[t]])
            best = m(feats[b:b + 1].cuda(), obj_atts=None if obj is None else obj[b:b + 1].cuda(),
                     sentiment=None if sent is None else sent[b:b + 1].cuda(), fsm=_table(fsm, slice(t, t + 1)),
                     num_constraints=nc[t:t + 1].cuda(), **kw)["predictions"].cpu()
            ls = m.last_search
            res.append((best[0], ls["predictions"][0].cpu(), ls["log_probs"][0].cpu(), ls["n_steps"]))
    return res


def _assert_same(batched, loop):
    pred, ns, allp, sc, ns2 = batched
    assert pred.shape[:2] == (B, J) and allp.shape[:4] == (B, J, S, K) and ns.shape == (B, J)
    assert torch.equal(ns, ns2) and pred.shape[2] == int(ns.max()) and allp.shape[4] == int(ns.max())
    for g, (best, beams, scores, n) in enumerate(loop):
        b, j = divmod(g, J)
        assert int(ns[b, j]) == n, (b, j, int(ns[b, j]), n)
        assert torch.equal(pred[b, j, :n], best), (b, j)
        assert bool((pred[b, j, n:] == 1).all())                   # after its own exit: the boundary token
        assert torch.equal(allp[b, j, ..., :n], beams), (b, j)
        assert bool((allp[b, j, ..., n:] == 1).all())
        fin = scores > -1e19
        assert torch.equal(fin, sc[b, j] > -1e19), (b, j)
        assert (sc[b, j][fin] - scores[fin]).abs().max().item() <= 1e-5, (b, j)


@pytest.mark.parametrize("sv", [1, 2])
def test_sample_search_equals_the_loop_of_batch1_calls(sv):
    m, feats, sent, obj, eps = _setup(sv)
    fsm = torch.from_numpy(fo.single_word_fsm([[5, 6], [9]], 400))[None].repeat(B, 1, 1, 1)
    nc = torch.tensor([2] * B)
    batched = _sample(m, feats, sent, obj, eps, fsm, nc)
    _assert_same(batched, _loop(m, feats, sent, obj, eps, fsm, nc, False))
    assert not torch.equal(batched[0][:, 0], batched[0][:, 1])     # the samples of an image differ


def test_sample_search_per_sample_machines_as_fsm_bits():
    """fsm_per_sample = 1 with the device bit table: every sample has its own constraints (row b*J + j)."""
    m, feats, sent, obj, eps = _setup(1)
    words = [[[5, 6], [9]], [[7], [11, 12]], [[20], [21]], [[9], [5]]]
    table = torch.stack([torch.from_numpy(fo.single_word_fsm(words[g % 4], 400)) for g in range(B * J)])
    bits = torch.zeros(B * J, S, 400, dtype=torch.int32)
    for i in range(S):                                             # bit i of bits[g, s, w] = table[g, s, i, w]
        bits |= table[:, :, i, :].to(torch.int32) << i
    fsm = sscvae.FsmBits(bits.cuda().contiguous())
    nc = torch.tensor([2, 2, 1, 2] * B)
    batched = _sample(m, feats, sent, obj, eps, fsm, nc)
    _assert_same(batched, _loop(m, feats, sent, obj, eps, fsm, nc, True))
    allp, sc = batched[2], batched[3]
    for g in range(B * J):                                         # a finite beam of state 3 used a word of each of ITS constraints
        b, j = divmod(g, J)
        for k in range(K):
            if sc[b, j, 3, k] > -1e19:
                toks = set(allp[b, j, 3, k].tolist())
                assert all(any(w in toks for w in c) for c in words[g % 4]), (g, k)


def test_sample_search_attribute_rule_selects_per_sample():
    """cbs_simple=False: the per-image valid-state mask (valid_states_with_attributes) is applied to every sample."""
    m, feats, sent, obj, eps = _setup(1, min_sat=1)
    m.cbs_simple = False
    fsm = torch.from_numpy(fo.single_word_fsm([[5, 6], [9]], 400))[None].repeat(B, 1, 1, 1)
    nc = torch.tensor([2] * B)
    # object c0 with attribute c1: only state 3 (both seen) counts, where the simple rule with min_sat 1 takes 1, 2 or 3
    constraints = [[("c0", ["c1"])]] * B
    c2s = [{"c0": [1, 3], "c1": [2, 3]}] * B
    batched = _sample(m, feats, sent, obj, eps, fsm, nc, constraints=constraints, constraint2states=c2s)
    _assert_same(batched, _loop(m, feats, sent, obj, eps, fsm, nc, False, constraints, c2s))
    pred, allp = batched[0], batched[2]
    for b in range(B):
        for j in range(J):
            assert torch.equal(pred[b, j], allp[b, j, 3, 0])


def test_sample_search_exits_per_search():
    """Each search stops when its own beams have all emitted the boundary token, like its batch-1 call; a batch-wide exit
    would give every sample of the batch the largest step count."""
    m, feats, sent, obj, eps = _setup(1, end_boost=0.4)
    fsm = torch.from_numpy(fo.single_word_fsm([[5, 6], [9]], 400))[None].repeat(B, 1, 1, 1)
    nc = torch.tensor([2] * B)
    batched = _sample(m, feats, sent, obj, eps, fsm, nc)
    ns = batched[1]
    assert int(ns.min()) < L
    assert any(len(set(ns[b].tolist())) > 1 for b in range(B)), ns   # samples of one image stop at different steps
    _assert_same(batched, _loop(m, feats, sent, obj, eps, fsm, nc, False))


def test_sample_search_full_dims_path_replay():
    """Bench dims: 4 images x 20 samples x S 8 x K 5 = 3 200 rows (large-tile GEMMs, grouped attention with 800 rows per
    image). The bf16 oracle cell is replayed along the path each search took, up to that search's own n_steps: every
    finite score = parent score + oracle log-prob of its token, every transition allowed by the FSM."""
    from bench import synthetic_fsm
    cfg = dict(vocab_size=10000, image_feature_size=2048, embedding_size=600, hidden_size=900, attention_projection_size=768,
               z_space=150, sentiment_vae=1, simple_vae=False, max_caption_length=20, prior_std=1.0, senti_prior_multip=0.5)
    Bf, Jf, Kf, Nf, Zf = 4, 20, 5, 36, 150
    torch.manual_seed(0)
    m = module_from_cfg(cfg, beam_size=Kf, use_cbs=True)
    m.eval()
    gen = torch.Generator().manual_seed(5)
    feats = torch.rand(Bf, Nf, 2048, generator=gen)
    feats[1, 20:] = 0
    sent = torch.tensor([[1.0], [-1.0], [0.0], [1.0]])
    fsm = synthetic_fsm(Bf, 10000, [[11, 12], [57], [300, 301, 302]])
    Sf = fsm.shape[1]
    SKf, R = Sf * Kf, Bf * Jf * Sf * Kf
    eps = torch.randn(20, R, Zf, generator=gen)
    m._eps_override = eps.cuda()
    out = m.sample(feats.cuda(), sentiment=sent.cuda(), n_samples=Jf, fsm=fsm.cuda(),
                   num_constraints=torch.full((Bf,), 3).cuda())
    ns = out["n_steps"].cpu()
    assert out["predictions"].shape[:2] == (Bf, Jf) and ns.shape == (Bf, Jf)
    tok = m.sample_search_region(Bf, Nf, Jf, Sf, Kf, 0, "tok_hist", torch.int32, (20, R)).cpu().long()
    bp = m.sample_search_region(Bf, Nf, Jf, Sf, Kf, 0, "bp_hist", torch.int32, (20, R)).cpu().long()
    sc = m.sample_search_region(Bf, Nf, Jf, Sf, Kf, 0, "score_hist", torch.float32, (20, R)).cpu()
    ocfg = uo.OracleConfig(**cfg)
    params = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    s_of = torch.arange(SKf) // Kf
    worst = 0.0
    for b, j in [(0, 0), (1, 7), (2, 13), (3, 19)]:                # one search per image, the CPU replay is slow at V 10 000
        g = b * Jf + j
        rows = slice(g * SKf, (g + 1) * SKf)
        stepper = uo.DecodeStepper(params, ocfg, feats[b:b + 1], sent[b:b + 1], q=uo.Rounding("bf16"))
        t_tok, t_bp, t_sc, e = tok[:, rows], bp[:, rows], sc[:, rows], eps[:, rows]
        logp0, state = stepper(torch.ones(1, dtype=torch.long), None, e[0, :1])
        fin = t_sc[0] > -1e19
        assert fin.any()
        rng = (logp0.max() - logp0.min()).item()
        worst = max(worst, (t_sc[0][fin] - logp0[0, t_tok[0]][fin]).abs().max().item() / rng)
        assert bool(fsm[b, 0, s_of, t_tok[0]][fin].bool().all())
        state = {k: v.repeat_interleave(SKf, dim=0) for k, v in state.items()}
        for t in range(1, int(ns[b, j])):
            logp, new_state = stepper(t_tok[t - 1], state, e[t])
            parent = t_bp[t]
            ended = t_tok[t - 1][parent] == 1
            expect = t_sc[t - 1][parent] + torch.where(ended, torch.zeros(SKf), logp[parent, t_tok[t]])
            fin = t_sc[t] > -1e19
            rng = (logp.max() - logp.min()).item()
            worst = max(worst, (t_sc[t][fin] - expect[fin]).abs().max().item() / rng)
            assert bool((t_tok[t][ended & fin] == 1).all())
            assert bool(fsm[b, (parent // Kf), s_of, t_tok[t]][fin].bool().all())
            state = {k: v[parent] for k, v in new_state.items()}
    assert worst < 6e-3, worst
