"""Diverse sampling under constrained beam search: the reference's inference loop of one forward() per latent sample
(var_updown/scripts/inference.py:138-167, USE_CBS) against one UpDownCaptioner.sample() call (sscvae_decode_samples_search).

Workloads at the bench dims (E 600 tied, H 900, A 768, Z 150, F 2048, V 10 000, 36 boxes, sentiment_vae 1, max length 20):
  (a) shipped: S = 1 with an all-allowed FSM, beam 1, 64 images x 20 samples
  (b) constrained: 3 single-word constraints (S = 8), beam 5, 16 images x 20 samples
For each, the two forms run on the same feature tensor (the loop reuses the per-image state), each warmed up 4 times (the
graph is captured on the second call), then timed alternately in windows of >= ~1 s with a device synchronise around each.
Prints one JSON object: GPU name and power limit, captions/s and ms per call of both forms, the fraction of best captions
the two forms share (GEMM dispatch differs between M = S*K and M = B*J*S*K rows, so near-ties may resolve differently),
and the library's per-class kernel times of one batched call.

    python tools/sample_search_bench.py [--rounds 3] [--min-seconds 1] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import sscvae  # noqa: E402
from sscvae import _lib  # noqa: E402
from bench import DIMS, N_BOXES, synthetic_fsm  # noqa: E402


class _Vocab:
    def __init__(self, n):
        self.n = n

    def get_vocab_size(self, namespace="tokens"):
        return self.n

    def get_token_index(self, token, namespace="tokens"):
        return {"@@UNKNOWN@@": 0, "@@BOUNDARY@@": 1}.get(token, 0)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:          # the timing does not depend on it; report what went wrong
        return torch.cuda.get_device_name(0), f"unknown ({type(e).__name__})"


def build(beam, dev, sd):
    m = sscvae.UpDownCaptioner(_Vocab(DIMS["vocab_size"]), DIMS["image_feature_size"], DIMS["embedding_size"],
                               DIMS["hidden_size"], DIMS["attention_projection_size"], max_caption_length=20,
                               beam_size=beam, use_cbs=True, min_constraints_to_satisfy=2, z_space=DIMS["z_space"],
                               prior_std=1.0, simple_vae=False, latent_embedding="glove", sentiment_vae=1,
                               senti_prior_multip=0.5, cbs_simple=True, device=dev).to(dev)
    if sd is not None:
        m.load_state_dict(sd)
    m.eval()
    return m


def window(fn, min_s):
    """Calls fn until >= min_s seconds have passed; returns (ms per call, calls)."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n = 0
    while True:
        fn()
        n += 1
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        if el >= min_s:
            return el * 1e3 / n, n


def run(name, m, mb, n_img, J, fsm, nc, feats, sent, rounds, min_s):
    """m runs the loop, mb (same weights) the batched call: each keeps its own decode workspace and graphs."""
    def loop():
        return [m(feats, None, None, fsm=fsm, num_constraints=nc, sentiment=sent)["predictions"] for _ in range(J)]

    def batched():
        return mb.sample(feats, sentiment=sent, n_samples=J, fsm=fsm, num_constraints=nc)["predictions"]

    for _ in range(4):
        loop()
        batched()
    torch.cuda.synchronize()
    # best captions the two forms share: both read the same explicit normals (loop call j gets the rows of the searches
    # b*J + j), since their Philox draws are laid out differently
    Z, S, K = DIMS["z_space"], fsm.shape[1], m.beam_size
    g = torch.Generator().manual_seed(11)
    eps = torch.randn(20, n_img * J * S * K, Z, generator=g)
    mb._eps_override = eps.to(feats.device)
    b_best = batched()
    mb._eps_override = None
    same = total = 0
    for j in range(J):
        idx = torch.cat([torch.arange((b * J + j) * S * K, (b * J + j + 1) * S * K) for b in range(n_img)])
        m._eps_override = eps[:, idx].contiguous().to(feats.device)
        # the batch of n_img images stops together here; compare up to each sample's own exit
        one = m(feats, None, None, fsm=fsm, num_constraints=nc, sentiment=sent)["predictions"]
        n = min(one.shape[1], b_best.shape[2])
        same += int((one[:, :n] == b_best[:, j, :n]).all(dim=1).sum())
        total += n_img
    m._eps_override = None
    loop_ms, batched_ms, loop_calls, batched_calls = [], [], 0, 0
    for _ in range(rounds):
        ms, n = window(loop, min_s)
        loop_ms.append(ms)
        loop_calls += n
        ms, n = window(batched, min_s)
        batched_ms.append(ms)
        batched_calls += n
    _lib.profile(True)
    batched()
    prof = _lib.profile_report()
    _lib.profile(False)
    lm, bm = min(loop_ms), min(batched_ms)
    return {
        "workload": name, "images": n_img, "samples_per_image": J, "fsm_states": S, "beam": K,
        "loop": {"ms_per_sample_loop": lm, "captions_per_s": n_img * J / (lm / 1e3), "ms_all_rounds": loop_ms,
                 "forward_calls_per_loop": J},
        "batched": {"ms_per_call": bm, "captions_per_s": n_img * J / (bm / 1e3), "ms_all_rounds": batched_ms},
        "speedup": lm / bm,
        "best_caption_identical_fraction": same / total,
        "profile_batched_call": {k: {"count": v["count"], "ms": round(v["ms"], 3)} for k, v in prof.items()},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="alternating timed windows per form")
    ap.add_argument("--min-seconds", type=float, default=1.0, help="length of one timed window")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sample_search_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu, power = gpu_info()
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(7)
    V = DIMS["vocab_size"]
    res = {"gpu": gpu, "power_limit": power, "dims": DIMS, "boxes": N_BOXES, "workloads": []}
    m1 = build(1, dev, None)
    sd = m1.state_dict()
    m1b = build(1, dev, sd)
    # (a) the shipped shape: every decode is CBS, S = 1 (all words allowed), beam 1
    n_img, J = 64, 20
    feats = torch.rand(n_img, N_BOXES, DIMS["image_feature_size"], generator=g).to(dev)
    sent = torch.randint(-1, 2, (n_img, 1), generator=g).float().to(dev)
    fsm = torch.ones(n_img, 1, 1, V, dtype=torch.uint8, device=dev)
    nc = torch.zeros(n_img, dtype=torch.long, device=dev)
    res["workloads"].append(run("shipped_s1_k1", m1, m1b, n_img, J, fsm, nc, feats, sent, a.rounds, a.min_seconds))
    del m1, m1b
    torch.cuda.empty_cache()
    # (b) constrained: 3 single-word constraints -> 8 states, beam 5
    n_img = 16
    m5, m5b = build(5, dev, sd), build(5, dev, sd)
    feats, sent = feats[:n_img].contiguous(), sent[:n_img].contiguous()
    fsm = synthetic_fsm(n_img, V, [[11, 12], [57], [300, 301, 302]]).to(dev)
    nc = torch.full((n_img,), 3, dtype=torch.long, device=dev)
    res["workloads"].append(run("cbs_s8_k5", m5, m5b, n_img, J, fsm, nc, feats, sent, a.rounds, a.min_seconds))
    text = json.dumps(res)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
