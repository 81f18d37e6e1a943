"""GPU: the tcgen05 / TMA GEMM against torch on the same bf16 operands."""
import ctypes as C

import pytest
import torch

from sscvae import _lib

pytestmark = pytest.mark.gpu

SHAPES = [
    (128, 64, 64), (256, 3600, 1808), (256, 768, 904), (256, 300, 904), (5376, 3600, 600), (9216, 768, 2048),
    (37, 50, 72), (1, 8, 8), (300, 129, 1000), (3600, 1808, 5376), (256, 3856, 3600), (130, 10000, 600),
    # skinny (M <= 256, N >= 1024) -> swapped-operand CTA-pair kernel, cluster split-K; large long-K -> CTA-pair tiles
    (256, 3600, 4928), (200, 4160, 3648), (8, 1920, 3648), (3600, 2048, 5376), (1100, 520, 2100),
]


@pytest.mark.parametrize("M,N,K", SHAPES)
def test_gemm_matches_torch(M, N, K):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    lda, ldb = (K + 7) // 8 * 8 + 8, (K + 7) // 8 * 8
    A = torch.zeros(M, lda, device="cuda", dtype=torch.bfloat16)
    B = torch.zeros(N, ldb, device="cuda", dtype=torch.bfloat16)
    A[:, :K] = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    B[:, :K] = torch.randn(N, K, device="cuda", generator=g).bfloat16()
    A[:, K:] = 7.0            # garbage beyond K must not be read
    bias = torch.randn(N, device="cuda", generator=g)
    ldc = N + 3
    Cm = torch.full((M, ldc), -5.0, device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(_lib.lib().sscvae_test_gemm(_lib.ptr(A), lda, _lib.ptr(B), ldb, M, N, K, _lib.ptr(Cm), ldc, _lib.ptr(bias), 0, 0, s))
    torch.cuda.synchronize()
    ref = A[:, :K].float() @ B[:, :K].float().t() + bias
    err = (Cm[:, :N] - ref).abs().max().item()
    assert err <= 2e-3 * (K ** 0.5), (err, M, N, K)
    assert (Cm[:, N:] == -5.0).all()          # nothing written outside the tile's valid columns
    # accumulate + tanh epilogue
    _lib.check(_lib.lib().sscvae_test_gemm(_lib.ptr(A), lda, _lib.ptr(B), ldb, M, N, K, _lib.ptr(Cm), ldc, None, 0, 1, s))
    torch.cuda.synchronize()
    ref2 = ref + A[:, :K].float() @ B[:, :K].float().t()
    assert (Cm[:, :N] - ref2).abs().max().item() <= 4e-3 * (K ** 0.5)
    _lib.check(_lib.lib().sscvae_test_gemm(_lib.ptr(A), lda, _lib.ptr(B), ldb, M, N, K, _lib.ptr(Cm), ldc, None, 1, 0, s))
    torch.cuda.synchronize()
    ref3 = torch.tanh(A[:, :K].float() @ B[:, :K].float().t())
    assert (Cm[:, :N] - ref3).abs().max().item() <= 2e-2


@pytest.mark.parametrize("M,N,K", [(256, 3600, 1808), (5376, 1000, 640), (256, 4160, 3648), (3600, 2048, 5376),
                                   (130, 516, 200), (256, 768, 960)])
def test_tma_store_epilogue_matches_staged_epilogue(M, N, K):
    """ldc % 4 == 0 and N % 4 == 0 select the TMA-store epilogue, an odd ldc the staged one: same bits."""
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    B = torch.randn(N, K, device="cuda", generator=g).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    outs = []
    for ldc in (N + 3, N + 4):
        Cm = torch.full((M, ldc), -5.0, device="cuda")
        _lib.check(_lib.lib().sscvae_test_gemm(_lib.ptr(A), K, _lib.ptr(B), K, M, N, K, _lib.ptr(Cm), ldc, _lib.ptr(bias), 0, 0, s))
        torch.cuda.synchronize()
        assert (Cm[:, N:] == -5.0).all()
        outs.append(Cm[:, :N].clone())
    assert torch.equal(outs[0], outs[1])
    ref = A.float() @ B.float().t() + bias
    assert (outs[1] - ref).abs().max().item() <= 2e-3 * (K ** 0.5)


@pytest.mark.parametrize("splits", [1, 2, 3, 4])
@pytest.mark.parametrize("M,N,K", [(256, 3600, 1920), (77, 1300, 4928), (256, 300, 960), (8, 4160, 3648), (129, 256, 512),
                                   (256, 7200, 3968)])
def test_swapped_pair_kernel_forced_split(M, N, K, splits):
    """The CTA-pair form of the swapped-operand kernel (tcgen05.mma.cta_group::2, cluster (2,1,S), DSMEM reduce-scatter),
    forced with a split count; ragged weight rows (second CTA of the last pair fully out of range), batch rows
    below one half tile, TMA-store and staged epilogues give the same bits."""
    g = torch.Generator(device="cuda").manual_seed(M * 3 + N + K + splits)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    B = torch.randn(N, K, device="cuda", generator=g).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ref = A.float() @ B.float().t() + bias
    outs = []
    for ldc in (N + 1, N + 4):
        Cm = torch.full((M, ldc), -5.0, device="cuda")
        _lib.check(_lib.lib().sscvae_test_gemm_splitk(_lib.ptr(A), K, _lib.ptr(B), K, M, N, K, _lib.ptr(Cm), ldc, splits,
                                                      _lib.ptr(bias), s))
        torch.cuda.synchronize()
        assert (Cm[:, :N] - ref).abs().max().item() <= 2e-3 * (K ** 0.5)
        assert (Cm[:, N:] == -5.0).all()
        outs.append(Cm[:, :N].clone())
    if N % 4 == 0:
        assert torch.equal(outs[0], outs[1])
