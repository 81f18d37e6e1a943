"""Weight-gradient phase of the training step at the benchmark's shapes (batch 256, T = 21, dims E600 / H900 / A768 /
Z150, 36 boxes, sentiment_vae 1), one gradient group at a time, in two forms:
  per-block: one transpose launch per operand and one GEMM launch per weight block through the library's dispatch
             (gemm_bf16_tn), W_hh computed a second time as its own block. The transposes run on the job-table kernel
             with one job per launch, so the transpose columns compare batched against separate launches of the same
             kernel, not against the per-operand transpose kernel that the job table replaced;
  grouped:   one transpose launch and one grouped CTA-pair GEMM launch per group, W_hh taken from W_ih's block.
Each group's launches are captured into a CUDA graph (no host time in the window) and timed with CUDA events over
windows of >= 1 s, alternating the two forms. Reports useful TFLOP/s (the deduplicated FLOPs of the group over its
time in either form) and the transposes' GB/s (bytes read + written). The working set of every group is larger than L2
except group 4's transposes; nothing flushes the cache between graph replays.
Usage on the GPU box: python tools/wgrad_bench.py [rounds]"""
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sscvae  # noqa: E402,F401
from sscvae import _lib  # noqa: E402

TB, B, BN = 21 * 256, 256, 256 * 36
G, Gp, H, Hp, F, E, Ep, Z, Z2p, A = 3600, 3648, 900, 960, 2048, 600, 640, 150, 320, 768
KX, ZC = F + 2 * Hp, 192
ldD, ldE, ldA = F + 2 * H + 1 + Z, F + 2 * H + 1, E + F + 2 * H

# group: (transposes [(rows, cols, ld_in, ld_out)],
#         GEMM blocks [(name, M, N, K, ldc, W_ih column or None)], duplicated W_hh blocks [(M, N, K)])
GROUPS = {
    "1 decoder": ([(TB, KX, KX, TB), (TB, ZC, ZC, TB), (TB, G, Gp, TB)],
                  [("xhat", G, F, TB, ldD, 0), ("h1", G, H, TB, ldD, F), ("h_dec", G, H, TB, ldD, F + H),
                   ("z", G, Z, TB, ldD, F + 2 * H + 1)], [(G, H, TB)]),
    "2 encoder+fc": ([(TB, G, Gp, TB), (TB, Hp, Hp, TB), (TB, Z2p, Z2p, TB), (TB, Hp, Hp, TB)],
                     [("xhat", G, F, TB, ldE, 0), ("h1", G, H, TB, ldE, F), ("h_dec", G, H, TB, ldE, F + H),
                      ("W_hh", G, H, TB, H, None), ("fc_mean", Z, H, TB, H, None), ("fc_log_var", Z, H, TB, H, None)], []),
    "3 attention": ([(TB, G, Gp, TB), (TB, 2 * Hp, 2 * Hp, TB), (TB, Ep, Ep, TB), (B, G, Gp, B), (B, F, F, B)],
                    [("emb", G, E, TB, ldA, 0), ("avg", G, F, B, ldA, E), ("h1", G, H, TB, ldA, E + F),
                     ("h_dec", G, H, TB, ldA, E + F + H)], [(G, H, TB)]),
    "4 W_q+image": ([(TB, A, A, TB), (BN, F, F, BN)],
                    [("W_q", A, H, TB, H, None), ("image", A, F, BN, F, None)], []),
}


def ints(xs):
    return (C.c_int * len(xs))(*xs)


def ptrs(ts):
    return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def build(name):
    trans, blocks, dups = GROUPS[name]
    tin = [torch.randn(r, ld, device="cuda").bfloat16() for r, c, ld, lo in trans]
    tout = [torch.empty(c, lo, device="cuda", dtype=torch.bfloat16) for r, c, ld, lo in trans]
    ops = []
    wide = {}
    for bname, M, N, K, ldc, col in blocks:
        a = torch.randn(M, K, device="cuda").bfloat16()
        b = torch.randn(N, K, device="cuda").bfloat16()
        if col is not None:
            if ldc not in wide:
                wide[ldc] = torch.empty(M, ldc, device="cuda")
            c = wide[ldc][:, col:]
        else:
            c = torch.empty(M, ldc, device="cuda")
        ops.append((a, b, c, M, N, K, ldc))
    dup_ops = [(torch.randn(M, K, device="cuda").bfloat16(), torch.randn(N, K, device="cuda").bfloat16(),
                torch.empty(M, N, device="cuda"), M, N, K, N) for M, N, K in dups]
    L = _lib.lib()

    def transposes(s, grouped):
        rows, cols, ldi, ldo = [list(x) for x in zip(*trans)]
        if grouped:
            _lib.check(L.sscvae_test_transpose_bf16(len(trans), ptrs(tin), ints(rows), ints(cols), ints(ldi), ptrs(tout),
                                                    ints(ldo), s))
        else:
            for i in range(len(trans)):
                _lib.check(L.sscvae_test_transpose_bf16(1, ptrs(tin[i:i + 1]), ints(rows[i:i + 1]), ints(cols[i:i + 1]),
                                                        ints(ldi[i:i + 1]), ptrs(tout[i:i + 1]), ints(ldo[i:i + 1]), s))

    def gemms(s, grouped):
        if grouped:
            a, b, c, M, N, K, ldc = zip(*ops)
            _lib.check(L.sscvae_test_gemm_grouped(len(ops), ptrs(a), ints(K), ptrs(b), ints(K), ints(M), ints(N), ints(K),
                                                  ptrs(c), ints(ldc), s))
        else:
            for a, b, c, M, N, K, ldc in ops + dup_ops:
                _lib.check(L.sscvae_test_gemm(_lib.ptr(a), K, _lib.ptr(b), K, M, N, K, _lib.ptr(c), ldc, None, 0, 0, s))

    flops = sum(2.0 * M * N * K for _, M, N, K, _, _ in blocks)
    tbytes = sum(4.0 * r * c for r, c, _, _ in trans)
    return transposes, gemms, flops, tbytes


def graph_of(fn, reps):
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        fn(C.c_void_p(s.cuda_stream))                      # first launches configure the kernels outside the capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            for _ in range(reps):
                fn(C.c_void_p(s.cuda_stream))
    torch.cuda.synchronize()
    return g


def time_graph(g, reps, min_s=1.0):
    """ms per repetition over a window of >= min_s seconds"""
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n, ms = 1, 0.0
    while True:
        e0.record()
        for _ in range(n):
            g.replay()
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= min_s * 1e3:
            return ms / (n * reps)
        n = max(n * 2, int(n * 1.2 * min_s * 1e3 / max(ms, 1e-3)))


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(f"# device: {torch.cuda.get_device_name(0)}; nvidia-smi: {smi[0] if smi else 'n/a'}")
    out = {}
    tot = {"per-block": [0.0, 0.0], "grouped": [0.0, 0.0]}
    for name in GROUPS:
        transposes, gemms, flops, tbytes = build(name)
        graphs = {}
        for form, grouped in (("per-block", False), ("grouped", True)):
            graphs[form] = (graph_of(lambda s, gr=grouped: transposes(s, gr), 20), graph_of(lambda s, gr=grouped: gemms(s, gr), 5))
        res = {f: {"transpose_ms": [], "gemm_ms": []} for f in graphs}
        for _ in range(rounds):
            for form, (gt, gg) in graphs.items():
                res[form]["transpose_ms"].append(time_graph(gt, 20))
                res[form]["gemm_ms"].append(time_graph(gg, 5))
        out[name] = {}
        for form, r in res.items():
            t = sorted(r["transpose_ms"])[len(r["transpose_ms"]) // 2]
            m = sorted(r["gemm_ms"])[len(r["gemm_ms"]) // 2]
            tot[form][0] += t
            tot[form][1] += m
            out[name][form] = {"transpose_ms": round(t, 4), "transpose_GBs": round(tbytes / t / 1e6, 1),
                               "gemm_ms": round(m, 4), "gemm_TFLOPs": round(flops / m / 1e9, 1),
                               "spread_gemm_ms": [round(min(r["gemm_ms"]), 4), round(max(r["gemm_ms"]), 4)]}
            print(f"group {name:14s} {form:9s}: transposes {t * 1e3:7.1f} us {tbytes / t / 1e6:7.1f} GB/s | "
                  f"GEMMs {m * 1e3:7.1f} us {flops / m / 1e9:7.1f} TFLOP/s (min {min(r['gemm_ms']) * 1e3:.1f} "
                  f"max {max(r['gemm_ms']) * 1e3:.1f})")
        del graphs
        torch.cuda.empty_cache()
    for form, (t, m) in tot.items():
        print(f"all groups {form:9s}: transposes {t:.3f} ms + GEMMs {m:.3f} ms = {t + m:.3f} ms")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
