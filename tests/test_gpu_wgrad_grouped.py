"""GPU: the weight-gradient phase's grouped CTA-pair GEMM, its job-table transpose, and the W_hh gradients that are
copies of a W_ih column block."""
import ctypes as C

import pytest
import torch

from helpers import module_from_cfg
from sscvae import _lib

pytestmark = pytest.mark.gpu

SENTINEL = -5.0


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ints(xs):
    return (C.c_int * len(xs))(*xs)


def _ptrs(ts):
    return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def test_grouped_gemm_mixed_shapes_match_torch():
    """One launch mixing the phase's shapes: M 3600 / 768 / 150 / 100, N 2048 / 900 / 600 / 150, K 5376 / 256 / 9216.
    Two problems write column blocks of one matrix with an odd row pitch and one an odd ldc (scalar epilogue), three own
    outputs with ldc % 4 == 0 and N % 4 == 0 (TMA stores), and one has ldc % 4 == 0 but N % 4 != 0 (vectorised staged
    epilogue); M = 150 and M = 100 leave the second CTA of a pair partly / wholly outside M. Rows and columns outside
    each problem keep their sentinel."""
    g = torch.Generator(device="cuda").manual_seed(11)
    # (M, N, K, output: ("shared", column) or ("own", ldc))
    specs = [(3600, 2048, 5376, ("shared", 0)), (3600, 900, 256, ("shared", 2048)), (768, 2048, 9216, ("own", 2052)),
             (150, 900, 5376, ("own", 904)), (100, 150, 256, ("own", 151)), (768, 600, 5376, ("own", 604)),
             (150, 150, 5376, ("own", 152))]
    shared_ld = 3999
    shared = torch.full((3600 + 2, shared_ld), SENTINEL, device="cuda")
    A, B, Cs, views, ldc = [], [], [], [], []
    for M, N, K, (kind, x) in specs:
        A.append(torch.randn(M, K, device="cuda", generator=g).bfloat16())
        B.append(torch.randn(N, K, device="cuda", generator=g).bfloat16())
        if kind == "shared":
            Cs.append(shared[:, x:])
            views.append(shared[:, x:x + N])
            ldc.append(shared_ld)
        else:
            own = torch.full((M + 2, x), SENTINEL, device="cuda")
            Cs.append(own)
            views.append(own[:, :N])
            ldc.append(x)
    n = len(specs)
    _lib.check(_lib.lib().sscvae_test_gemm_grouped(
        n, _ptrs(A), _ints([s[2] for s in specs]), _ptrs(B), _ints([s[2] for s in specs]), _ints([s[0] for s in specs]),
        _ints([s[1] for s in specs]), _ints([s[2] for s in specs]), _ptrs(Cs), _ints(ldc), _stream()))
    torch.cuda.synchronize()
    for i, (M, N, K, (kind, x)) in enumerate(specs):
        ref = A[i].float() @ B[i].float().t()
        err = (views[i][:M] - ref).abs().max().item()
        assert err <= 2e-3 * (K ** 0.5), (i, err, M, N, K)
        assert (views[i][M:] == SENTINEL).all(), i                  # rows beyond M
        if kind == "own":
            assert (Cs[i][:, N:] == SENTINEL).all(), i              # columns beyond N
    assert (shared[:, 2048 + 900:] == SENTINEL).all()               # columns behind the last block of the shared matrix


def test_transpose_job_table_matches_torch_bit_for_bit():
    """out[c, r] = in[r, c] for c < cols, zero padding for rows <= r < ld_out, nothing written for c >= cols; a ragged
    column count (cols % 8 != 0), partial 64 x 64 tiles on both sides and a K = batch operand in one launch."""
    g = torch.Generator(device="cuda").manual_seed(5)
    # (rows, cols, ld_in, ld_out)
    jobs = [(5376, 3600, 3648, 5376), (5376, 900, 1920, 5376), (256, 2048, 2048, 320), (100, 150, 152, 128),
            (9216, 2048, 2048, 9216)]
    ins, outs = [], []
    for rows, cols, ld_in, ld_out in jobs:
        x = torch.randn(rows, ld_in, device="cuda", generator=g).bfloat16()
        ins.append(x)
        outs.append(torch.full((cols + 3, ld_out), SENTINEL, device="cuda", dtype=torch.bfloat16))
    _lib.check(_lib.lib().sscvae_test_transpose_bf16(
        len(jobs), _ptrs(ins), _ints([j[0] for j in jobs]), _ints([j[1] for j in jobs]), _ints([j[2] for j in jobs]),
        _ptrs(outs), _ints([j[3] for j in jobs]), _stream()))
    torch.cuda.synchronize()
    for (rows, cols, ld_in, ld_out), x, o in zip(jobs, ins, outs):
        assert torch.equal(o[:cols, :rows].view(torch.int16), x[:, :cols].t().contiguous().view(torch.int16)), (rows, cols)
        assert (o[:cols, rows:].float() == 0).all(), (rows, cols)
        assert (o[cols:].float() == SENTINEL).all(), (rows, cols)


CFG = dict(vocab_size=500, image_feature_size=128, embedding_size=600, hidden_size=64, attention_projection_size=48,
           z_space=24, sentiment_vae=1, simple_vae=False, max_caption_length=20, prior_std=1.0, senti_prior_multip=0.5)
DEC = "_updown_cell._language_lstm_cell_decoder."
ATT = "_updown_cell._attention_lstm_cell."


def _grads(frozen=()):
    torch.manual_seed(0)
    m = module_from_cfg(CFG)
    g = torch.Generator().manual_seed(1)
    B, N = 8, 9
    feats = torch.rand(B, N, CFG["image_feature_size"], generator=g)
    toks = torch.randint(2, CFG["vocab_size"], (B, 20), generator=g)
    for b in range(B):
        toks[b, 3 + 2 * b:] = 0
    sent = torch.randint(-1, 2, (B, 1), generator=g).float()
    eps = torch.randn(21, B, CFG["z_space"], generator=g)
    params = dict(m.named_parameters())
    for k in frozen:
        params[k].requires_grad_(False)
    m.train()
    m._eps_override = eps.cuda()
    out = m(feats.cuda(), None, None, toks.cuda(), sent.cuda())
    (out["loss"].mean() + out["kld"].mean() / 750.0).backward()
    torch.cuda.synchronize()
    return {k: p.grad.clone() for k, p in params.items() if p.grad is not None}


def test_hh_gradients_are_the_ih_column_blocks():
    """W_hh multiplies the same operand as one W_ih column block, so its gradient is computed once, into W_ih's block,
    and copied out of it (row pitch and column offset of the 2-D copy); with W_ih frozen it is computed straight into
    W_hh and agrees (to fp32 summation order, should the rest of the backward run differently)."""
    F, E, H = CFG["image_feature_size"], CFG["embedding_size"], CFG["hidden_size"]
    g = _grads()
    assert torch.equal(g[DEC + "weight_hh"], g[DEC + "weight_ih"][:, F + H:F + 2 * H])
    assert torch.equal(g[ATT + "weight_hh"], g[ATT + "weight_ih"][:, E + F:E + F + H])
    assert g[DEC + "weight_hh"].abs().max() > 0 and g[ATT + "weight_hh"].abs().max() > 0
    gf = _grads(frozen=(DEC + "weight_ih", ATT + "weight_ih"))
    assert DEC + "weight_ih" not in gf and ATT + "weight_ih" not in gf
    for k in (DEC + "weight_hh", ATT + "weight_hh"):
        assert (gf[k] - g[k]).abs().max() <= 1e-5 * g[k].abs().max(), k
