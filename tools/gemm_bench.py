"""Micro-benchmark of the tcgen05 GEMM at the shapes of the training step against cuBLAS (torch.matmul): the
library's own dispatch, plus the skinny-M CTA-pair kernel forced to a K split of N for every config pkN (N = 1..4).
Usage on the GPU box: python tools/gemm_bench.py [pk1 pk2 pk3 pk4]

Timing: ITERS launches back to back between two CUDA events with no Python in between (ours: the repeat loop of
sscvae_test_gemm; cuBLAS: a captured CUDA graph), operands L2-resident."""
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sscvae  # noqa: E402,F401
from sscvae import _lib  # noqa: E402

SHAPES = [  # (M, N, K, what)
    (256, 3600, 1920, "att gates"), (256, 3600, 4928, "enc gates"), (256, 768, 960, "q"), (256, 300, 960, "fc"),
    (256, 4160, 3648, "bwd dXEZ"), (256, 4928, 3648, "bwd dXEH"), (256, 1920, 3648, "bwd dXA"), (256, 900, 768, "bwd dh1_q"),
    (3600, 2048, 5376, "wgrad"), (5376, 10000, 640, "vocab"), (5376, 3600, 640, "emb gates"),
]
if os.environ.get("GEMM_BENCH_SKINNY"):
    SHAPES = [s for s in SHAPES if s[0] == 256]
ITERS = 40


def time_ours(fn):
    """(GPU time per launch inside a captured CUDA graph, per-launch time when launched from the host in a C loop)."""
    os.environ["SSCVAE_TEST_GEMM_REPEAT"] = "3"
    fn()
    os.environ["SSCVAE_TEST_GEMM_REPEAT"] = str(ITERS)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    host = e0.elapsed_time(e1) / ITERS * 1e3
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay()
    torch.cuda.synchronize()
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / ITERS * 1e3, host


def time_graph(fn):
    """ITERS calls of a torch op captured in one CUDA graph (no CPU launch overhead)."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(ITERS):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / ITERS * 1e3


def main():
    configs = [None] + sys.argv[1:]
    L = _lib.lib()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for (M, N, K, what) in SHAPES:
        A = torch.randn(M, K, device="cuda").bfloat16()
        B = torch.randn(N, K, device="cuda").bfloat16()
        Cm = torch.zeros(M, N, device="cuda")
        ref = time_graph(lambda: torch.matmul(A, B.t()))
        line = f"{what:10s} {M}x{N}x{K}: cublas {ref:6.1f} us |"
        for cfg in configs:
            def fn():
                st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                _lib.check(L.sscvae_test_gemm(_lib.ptr(A), K, _lib.ptr(B), K, M, N, K, _lib.ptr(Cm), N, None, 0, 0, st))
            if cfg is not None:
                if M > 256 or N < 256:
                    continue
                S = int(cfg[2:])                 # pkN: CTA-pair kernel, K split N

                def fn():
                    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                    _lib.check(L.sscvae_test_gemm_splitk(_lib.ptr(A), K, _lib.ptr(B), K, M, N, K, _lib.ptr(Cm), N, S, None, st))
            try:
                gpu, host = time_ours(fn)
                line += f" [{cfg or 'auto'}] {gpu:5.1f}/{host:5.1f}"
            except Exception:
                line += f" [{cfg}] ERR"
        print(line, flush=True)


if __name__ == "__main__":
    main()
