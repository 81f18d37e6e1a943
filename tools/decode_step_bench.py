"""Time per decode step of UpDownCaptioner._decode_step (one sscvae_decode_step call, the reference's step function) against
the fused decode's time per step at the same rows.

Workloads at the bench dims (E 600 tied, H 900, A 768, Z 150, F 2048, V 10 000, 36 boxes, sentiment_vae 1, max length 20):
  (a) sampling: 64 images x 100 rows. Fused: sample(n_samples=100), one sscvae_decode_samples call of 20 steps.
  (b) constrained: 16 images, 3 single-word constraints (S = 8), beam 5: 640 rows. Fused: forward(), one sscvae_decode
      call of 20 steps (the early exit is resolved after the last step, so every call runs all 20).
The step runs on the same feature tensor with given states (the image state is reused, as inside a search). Both forms are
warmed up, then timed alternately in windows of >= --min-seconds with a device synchronise around each; fused time per
step = call time / 20. A separate profiled run of the step gives the log-softmax kernel's time; its bytes (R*V*4 read +
R*V*4 written + the tile partials) over that time is reported against the HBM3e figure of 7.7 TB/s. The working set of
(a) (256 MB of log-probs) exceeds the 126 MB L2; that of (b) (26 MB) does not. Prints one JSON object with the GPU name
and power limit.

    python tools/decode_step_bench.py [--rounds 3] [--min-seconds 1] [--out result.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from sscvae import _lib  # noqa: E402
from bench import DIMS, N_BOXES, synthetic_fsm  # noqa: E402
from sample_search_bench import build, gpu_info, window  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
KEYS = ("h1", "c1", "h_encoder", "c_encoder", "h_decoder", "c_decoder")


def run(name, m, n_img, rows, fused, feats, sent, rounds, min_s, g):
    dev = feats.device
    H, Z, V, L = DIMS["hidden_size"], DIMS["z_space"], DIMS["vocab_size"], DIMS["max_caption_length"]
    prev = torch.randint(2, V, (rows,), generator=g).to(dev)
    states = {k: (torch.randn(rows, H, generator=g) * 0.3).to(dev) for k in KEYS}
    pm = sent.repeat(1, Z) * DIMS["senti_prior_multip"]
    pv = torch.ones(n_img, Z, device=dev)

    def step():
        return m._decode_step(feats, None, prev, states, sentiment=sent, prior_mean=pm, prior_var=pv)
    for _ in range(4):
        step()
        fused()
    torch.cuda.synchronize()
    step_ms, fused_ms = [], []
    for _ in range(rounds):
        step_ms.append(window(step, min_s)[0])
        fused_ms.append(window(fused, min_s)[0] / L)
    _lib.profile(True)
    for _ in range(20):
        step()
    prof = _lib.profile_report()
    _lib.profile(False)
    ls = prof["log_softmax"]
    ls_ms = ls["ms"] / ls["count"]
    ls_bytes = ls["bytes"] / ls["count"]
    return {
        "workload": name, "images": n_img, "rows": rows,
        "step_ms": min(step_ms), "step_ms_all_rounds": step_ms,
        "fused_ms_per_step": min(fused_ms), "fused_ms_per_step_all_rounds": fused_ms,
        "step_over_fused": min(step_ms) / min(fused_ms),
        "log_softmax": {"us": ls_ms * 1e3, "bytes": ls_bytes, "bytes_per_s": ls_bytes / (ls_ms / 1e3),
                        "fraction_of_7.7_TB_s": ls_bytes / (ls_ms / 1e3) / HBM_BYTES_PER_S},
        "profile_one_step": {k: {"count": v["count"] // 20, "us": round(v["ms"] / 20 * 1e3, 2)} for k, v in prof.items()},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="alternating timed windows per form")
    ap.add_argument("--min-seconds", type=float, default=1.0, help="length of one timed window")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decode_step_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu, power = gpu_info()
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(7)
    V = DIMS["vocab_size"]
    res = {"gpu": gpu, "power_limit": power, "dims": DIMS, "boxes": N_BOXES, "workloads": []}
    with torch.no_grad():
        m = build(1, dev, None)
        m._use_cbs = False                                  # (a) the unconstrained beam-1 sampling path
        n_img, J = 64, 100
        feats = torch.rand(n_img, N_BOXES, DIMS["image_feature_size"], generator=g).to(dev)
        sent = torch.randint(-1, 2, (n_img, 1), generator=g).float().to(dev)
        res["workloads"].append(run("sampling_64x100", m, n_img, n_img * J,
                                    lambda: m.sample(feats, sentiment=sent, n_samples=J), feats, sent, a.rounds,
                                    a.min_seconds, g))
        sd = m.state_dict()
        del m
        torch.cuda.empty_cache()
        m = build(5, dev, sd)                               # (b) CBS S 8, K 5
        n_img = 16
        feats, sent = feats[:n_img].contiguous(), sent[:n_img].contiguous()
        fsm = synthetic_fsm(n_img, V, [[11, 12], [57], [300, 301, 302]]).to(dev)
        nc = torch.full((n_img,), 3, dtype=torch.long, device=dev)
        res["workloads"].append(run("cbs_16_s8_k5", m, n_img, n_img * 8 * 5,
                                    lambda: m(feats, None, None, fsm=fsm, num_constraints=nc, sentiment=sent), feats, sent,
                                    a.rounds, a.min_seconds, g))
    text = json.dumps(res)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
