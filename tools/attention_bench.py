"""Cost of `return_attention` (the per-word attention weights, sscvae_decode_attention) on the two sampling workloads.

Workloads at the bench dims (E 600 tied, H 900, A 768, Z 150, F 2048, V 10 000, 36 boxes, sentiment_vae 1, max length 20):
  (a) diverse sampling, beam 1: 64 images x 100 samples per sample() call (bench.py's batched sampling leg)
  (b) constrained: 3 single-word constraints (S = 8), beam 5, 16 images x 20 samples per sample() call
Each leg runs the same model and inputs with the switch off and on: both are warmed up 4 times (the decode graph is
captured on the second call), then timed alternately in windows of >= ~1 s with a device synchronise around each call;
the best window of each counts. Also reported: the kernel launches of one call with each setting (the switch adds the
trace kernel) and the library's per-class kernel times of one call with the switch on ("search_attention" is the trace).
Prints one JSON object that starts with the GPU name and power limit read in the same run.

    python tools/attention_bench.py [--rounds 3] [--min-seconds 1] [--out result.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from sscvae import _lib  # noqa: E402
from bench import DIMS, N_BOXES, synthetic_fsm  # noqa: E402
from sample_search_bench import build, gpu_info, window  # noqa: E402


def run(name, m, call, images, samples, rounds, min_s):
    def with_switch(on):
        def f():
            m.return_attention = on
            return call()
        return f
    off, on = with_switch(False), with_switch(True)
    for _ in range(4):
        off()
        on()
    torch.cuda.synchronize()
    launches = {}
    for key, f in (("off", off), ("on", on)):
        c0 = _lib.launch_count()
        f()
        torch.cuda.synchronize()
        launches[key] = _lib.launch_count() - c0
    ms = {"off": [], "on": []}
    for _ in range(rounds):
        ms["off"].append(window(off, min_s)[0])
        ms["on"].append(window(on, min_s)[0])
    _lib.profile(True)
    on()
    prof = _lib.profile_report()
    _lib.profile(False)
    m.return_attention = False
    best = {k: min(v) for k, v in ms.items()}
    return {
        "workload": name, "images": images, "samples_per_image": samples, "fsm_states": call.states, "beam": m.beam_size,
        "ms_per_call": best, "ms_all_rounds": ms,
        "captions_per_s": {k: images * samples / (v / 1e3) for k, v in best.items()},
        "on_over_off": best["on"] / best["off"],
        "launches_per_call": launches,
        "trace_kernel_ms": round(prof.get("search_attention", {}).get("ms", float("nan")), 4),
        "profile_call_on": {k: {"count": v["count"], "ms": round(v["ms"], 3)} for k, v in prof.items()},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="alternating timed windows per setting")
    ap.add_argument("--min-seconds", type=float, default=1.0, help="length of one timed window")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu, power = gpu_info()
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(7)
    V = DIMS["vocab_size"]
    res = {"gpu": gpu, "power_limit": power, "dims": DIMS, "boxes": N_BOXES, "workloads": []}
    # (a) beam-1 diverse sampling, bench.py's batched sampling leg
    m1 = build(1, dev, None)
    sd = m1.state_dict()
    m1._use_cbs = False
    n_img, J = 64, 100
    feats = torch.rand(n_img, N_BOXES, DIMS["image_feature_size"], generator=g).to(dev)
    sent = torch.randint(-1, 2, (n_img, 1), generator=g).float().to(dev)

    def sample_greedy():
        return m1.sample(feats, sentiment=sent, n_samples=J)["predictions"]
    sample_greedy.states = 1
    res["workloads"].append(run("sample_b1", m1, sample_greedy, n_img, J, a.rounds, a.min_seconds))
    del m1
    torch.cuda.empty_cache()
    # (b) constrained beam search per sample
    n_img, J = 16, 20
    m5 = build(5, dev, sd)
    feats, sent = feats[:n_img].contiguous(), sent[:n_img].contiguous()
    fsm = synthetic_fsm(n_img, V, [[11, 12], [57], [300, 301, 302]]).to(dev)
    nc = torch.full((n_img,), 3, dtype=torch.long, device=dev)

    def sample_cbs():
        return m5.sample(feats, sentiment=sent, n_samples=J, fsm=fsm, num_constraints=nc)["predictions"]
    sample_cbs.states = fsm.shape[1]
    res["workloads"].append(run("sample_cbs_s8_k5", m5, sample_cbs, n_img, J, a.rounds, a.min_seconds))
    text = json.dumps(res)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
