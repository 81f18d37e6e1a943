"""Bring-up diagnostics (prints, never asserts): GEMM error over shapes and per-tensor diffs of the
training path against the oracle. Usage on the GPU box: python tools/gpu_probe.py"""
import ctypes as C
import os
import sys
import traceback

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import sscvae  # noqa: E402
from sscvae import _lib  # noqa: E402
from conftest import load_golden  # noqa: E402
from helpers import module_from_cfg, oracle_params, rel_err  # noqa: E402
from oracle import updown_oracle as uo  # noqa: E402


def gemm_probe():
    L = _lib.lib()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for (M, N, K) in [(128, 64, 64), (128, 64, 128), (128, 128, 64), (256, 256, 512), (200, 100, 72), (256, 3600, 1808),
                      (5376, 10000, 600)]:
        g = torch.Generator(device="cuda").manual_seed(1)
        A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
        B = torch.randn(N, K, device="cuda", generator=g).bfloat16()
        Cm = torch.zeros(M, N, device="cuda")
        try:
            _lib.check(L.sscvae_test_gemm(_lib.ptr(A), K, _lib.ptr(B), K, M, N, K, _lib.ptr(Cm), N, None, 0, 0, s))
            torch.cuda.synchronize()
            ref = A.float() @ B.float().t()
            print(f"gemm {M}x{N}x{K}: max err {(Cm - ref).abs().max().item():.3e} (ref max {ref.abs().max().item():.1f})", flush=True)
        except Exception as e:
            print(f"gemm {M}x{N}x{K}: FAILED {e}", flush=True)
            raise


def train_probe(name):
    g = load_golden(name)
    cfg = g["cfg"]
    ocfg = uo.OracleConfig(**cfg)
    m = module_from_cfg(cfg, g["params"])
    m.train()
    m._eps_override = g["eps"].cuda()
    out = m(g["image_features"].cuda(), None, None, g["caption_tokens"].cuda(), g["sentiment"].cuda())
    torch.cuda.synchronize()
    B, N, _ = g["image_features"].shape
    T, V, Z, H, A = cfg["max_caption_length"] + 1, cfg["vocab_size"], cfg["z_space"], cfg["hidden_size"], cfg["attention_projection_size"]
    p = oracle_params(g["params"], ocfg, grad=True)
    ob = uo.train_forward(p, ocfg, g["image_features"], g["caption_tokens"], g["sentiment"], g["eps"],
                          q=uo.Rounding("bf16"), record=True)
    reg = lambda n, shp: m.train_region(B, N, n, torch.float32, shp).cpu()
    print(f"[{name}] loss cuda {out['loss'].detach().cpu().numpy().round(3)}")
    print(f"[{name}] loss ref  {g['loss'].numpy().round(3)}")
    print(f"[{name}] kld  cuda {out['kld'].detach().cpu().numpy().round(3)}")
    print(f"[{name}] kld  ref  {g['kld'].numpy().round(3)}")
    print(f"[{name}] alpha  max abs diff {(reg('alpha', (T, B, N)) - torch.stack([s['alpha'] for s in ob['steps']])).abs().max().item():.3e}")
    print(f"[{name}] mean   rel {rel_err(reg('mean', (T, B, Z)), torch.stack([s['mean'] for s in ob['steps']])):.3e}")
    print(f"[{name}] logvar rel {rel_err(reg('logvar', (T, B, Z)), torch.stack([s['log_var'] for s in ob['steps']])):.3e}")
    lg = reg("logits", (T, B, V)).permute(1, 0, 2)
    print(f"[{name}] logits rel vs bf16-oracle {rel_err(lg, ob['logits']):.3e}  vs fp32 ref {rel_err(lg, g['logits']):.3e}")
    for t in (0, 1, 5, 20):
        print(f"   step {t}: logits rel {rel_err(lg[:, t], ob['logits'][:, t]):.3e}")
    (out["loss"].mean() + out["kld"].mean() / 750.0).backward()
    torch.cuda.synchronize()
    uo.train_objective(ob).backward()
    for k, prm in m.named_parameters():
        if prm.grad is None:
            continue
        ref = g["grads"].get(k)
        print(f"[{name}] grad {k:70s} rel vs ref {rel_err(prm.grad, ref):.3e}  vs bf16-oracle {rel_err(prm.grad, p[k].grad):.3e}")


if __name__ == "__main__":
    print("device", torch.cuda.get_device_name(0))
    try:
        gemm_probe()
    except Exception:
        traceback.print_exc()
    for n in sys.argv[1:] or ["train_tied_sv1", "train_untied_sv1"]:
        try:
            train_probe(n)
        except Exception:
            traceback.print_exc()
