"""CPU: re-runs the live comparison oracle <-> unmodified reference (visinf/style-seqcvae, imported in place
through oracle/ref_harness.py from the checkout SSCVAE_REFERENCE_ROOT names). The reference is not part of this
repository, so these tests skip without that checkout; the same comparison runs self-contained in
tests/test_oracle_golden.py and tests/test_sentiment_vae2.py against the reference outputs stored in tests/golden/."""
import pytest
import torch

from oracle import ref_harness as rh
from oracle import updown_oracle as uo

pytestmark = pytest.mark.skipif(not rh.reference_available(),
                                reason="no checkout of the reference project (set SSCVAE_REFERENCE_ROOT)")


@pytest.mark.parametrize("E,sv,simple", [(600, 1, False), (300, 0, False), (48, 1, False)])
def test_live_train_parity(E, sv, simple):
    V, F, H, A, Z, B, L = 90, 48, 24, 16, 12, 4, 20
    vocab = rh.make_vocabulary(V)
    m = rh.build_reference_model(vocab, image_feature_size=F, embedding_size=E, hidden_size=H,
                                 attention_projection_size=A, z_space=Z, sentiment_vae=sv, simple_vae=simple, seed=21)
    cfg = uo.OracleConfig(vocab_size=V, image_feature_size=F, embedding_size=E, hidden_size=H,
                          attention_projection_size=A, z_space=Z, sentiment_vae=sv, simple_vae=simple)
    g = torch.Generator().manual_seed(3)
    feats = torch.rand(B, 6, F, generator=g)
    feats[1, 3:] = 0
    toks = torch.randint(2, V, (B, L), generator=g)
    toks[0, 9:] = 0
    toks[2, 1:] = 0
    s = torch.tensor([[1.], [0.], [-1.], [0.]])
    m.train()
    torch.manual_seed(99)
    out = m(feats.clone(), None, None, toks, s)
    torch.manual_seed(99)
    eps = torch.stack([torch.randn(B, Z) for _ in range(L + 1)])
    p = {k: v.detach().clone() for k, v in m.state_dict().items()}
    o = uo.train_forward(p, cfg, feats, toks, s, eps)
    torch.testing.assert_close(o["loss"], out["loss"], rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(o["kld"], out["kld"], rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("E,le,Z", [(48, "senti_word_net", 12), (600, "glove", 150)])
def test_live_train_parity_sentiment_vae_2(E, le, Z):
    """SENTIMENT_VAE = 2 (attribute-grounded prior): the reference forward (constructed as oracle/ref_harness.py
    describes) against the oracle, from attribute lists."""
    from oracle.gen_golden import make_mean_choice, make_obj_atts
    V, F, H, A, B, L, N = 90, 48, 24, 16, 4, 20, 6
    vocab = rh.make_vocabulary(V)
    m = rh.build_reference_model(vocab, image_feature_size=F, embedding_size=E, hidden_size=H, attention_projection_size=A,
                                 z_space=Z, sentiment_vae=2, latent_embedding=le, seed=5, latent_embedding_multip=3.0,
                                 mean_choice=make_mean_choice(Z, le, 8))
    cfg = uo.OracleConfig(vocab_size=V, image_feature_size=F, embedding_size=E, hidden_size=H, attention_projection_size=A,
                          z_space=Z, sentiment_vae=2, latent_embedding=le)
    g = torch.Generator().manual_seed(3)
    feats = torch.rand(B, N, F, generator=g)
    feats[1, 3:] = 0
    toks = torch.randint(2, V, (B, L), generator=g)
    toks[0, 9:] = 0
    obj_atts = make_obj_atts(B, N, 4)
    m.train()
    torch.manual_seed(99)
    out = m(feats.clone(), obj_atts, None, toks, torch.zeros(B, 1))
    torch.manual_seed(99)
    eps = torch.stack([torch.randn(B, Z) for _ in range(L + 1)])
    p = {k: v.detach().clone() for k, v in m.state_dict().items()}
    o = uo.train_forward(p, cfg, feats, toks, None, eps, obj_means=m.translate_obj_atts2obj_means(obj_atts))
    torch.testing.assert_close(o["loss"], out["loss"], rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(o["kld"], out["kld"], rtol=1e-5, atol=1e-4)
