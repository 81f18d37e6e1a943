"""Time one training iteration through the stepwise training step (UpDownCaptioner._decode_step with
`stepwise_training = True`, one differentiable step per timestep) against the fused training forward + backward.

Workload: the bench dims (E 600 tied, H 900, A 768, Z 150, F 2048, V 10 000, 36 boxes, sentiment_vae 1, max length 20),
256 captions of random lengths 5..20, fixed eps. One iteration is
  stepwise: 21 calls of _decode_step, the reference's loss (per-step KL masked by the token mask, _get_loss,
            loss.mean() + kld.mean() / 750) in torch, backward through autograd;
  fused:    forward() and backward() of the same objective.
Both are warmed up, then timed alternately in windows of >= --min-seconds, each iteration ending in a device synchronise.
Reported per form: ms per iteration (best and all windows), kernel launches per iteration from the library's counter (the
torch kernels of the stepwise loss are not counted), and the peak device memory of one iteration. Prints one JSON object with
the GPU name and power limit.

    python tools/train_step_bench.py [--rounds 3] [--min-seconds 1] [--out result.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

import sscvae  # noqa: E402
from sscvae import _lib  # noqa: E402
from bench import DIMS, KLD_WEIGHT, N_BOXES  # noqa: E402
from sample_search_bench import _Vocab, gpu_info, window  # noqa: E402

BATCH = 256


def stepwise_objective(m, feats, caps, sent, eps):
    """The reference's training branch (updown_captioner.py:263-323) over model._decode_step."""
    B, L = caps.shape
    Z = m.z_space
    tokens = torch.cat([torch.ones(B, 1, dtype=caps.dtype, device=caps.device), caps,
                        torch.zeros(B, 1, dtype=caps.dtype, device=caps.device)], dim=1)
    lengths = (caps != 0).sum(1)
    tokens[torch.arange(B, device=caps.device), lengths + 1] = 1                 # add_sentence_boundary_token_ids
    tmask = (tokens[:, 1:] != 0).float()
    prior_var = torch.full((B, Z), float(m.prior_std) ** 2, device=feats.device)
    prior_mean, states, logits_t, kl_t = None, None, [], []
    for t in range(L + 1):
        m._eps_override = eps[t]
        logits, states, mean, log_var, prior_mean, prior_log_var, _ = m._decode_step(
            feats, None, tokens[:, t], states, sentiment=sent, prior_mean=prior_mean, prior_var=prior_var)
        kl = 1 + log_var - prior_log_var - ((mean - prior_mean).pow(2) + log_var.exp()) / (prior_var + 0.00001)
        kl_t.append(-0.5 * kl.sum(1))
        logits_t.append(logits)
    logp = torch.log_softmax(torch.stack(logits_t, dim=1), dim=-1)
    nll = -logp.gather(2, tokens[:, 1:].unsqueeze(-1)).squeeze(-1) * tmask
    n = tmask.sum(-1)
    loss = n * (nll.sum(1) / (n + 1e-13))
    kld = (torch.stack(kl_t, dim=1) * tmask).sum(1)
    return loss.mean() + kld.mean() / KLD_WEIGHT


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_step_bench.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda")
    torch.manual_seed(0)
    m = sscvae.UpDownCaptioner(_Vocab(DIMS["vocab_size"]), DIMS["image_feature_size"], DIMS["embedding_size"],
                               DIMS["hidden_size"], DIMS["attention_projection_size"], max_caption_length=20,
                               z_space=DIMS["z_space"], prior_std=1.0, simple_vae=False, latent_embedding="glove",
                               sentiment_vae=1, senti_prior_multip=0.5, device=dev).to(dev)
    m.train()
    m.stepwise_training = True
    g = torch.Generator().manual_seed(1)
    L = DIMS["max_caption_length"]
    feats = torch.rand(BATCH, N_BOXES, DIMS["image_feature_size"], generator=g).to(dev)
    caps = torch.randint(2, DIMS["vocab_size"], (BATCH, L), generator=g)
    lens = torch.randint(5, L + 1, (BATCH,), generator=g)
    for b in range(BATCH):
        caps[b, lens[b]:] = 0
    caps = caps.to(dev)
    sent = torch.randint(-1, 2, (BATCH, 1), generator=g).float().to(dev)
    eps = torch.randn(L + 1, BATCH, DIMS["z_space"], generator=g).to(dev)

    def stepwise():
        m.zero_grad(set_to_none=True)
        stepwise_objective(m, feats, caps, sent, eps).backward()

    def fused():
        m.zero_grad(set_to_none=True)
        m._eps_override = eps
        out = m(feats, None, None, caps, sent)
        (out["loss"].mean() + out["kld"].mean() / KLD_WEIGHT).backward()

    forms = {"stepwise": stepwise, "fused": fused}
    for _ in range(3):
        for fn in forms.values():
            fn()
    torch.cuda.synchronize()
    res = {}
    for name, fn in forms.items():
        l0 = _lib.launch_count()
        fn()
        torch.cuda.synchronize()
        launches = _lib.launch_count() - l0
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        res[name] = {"launches_per_iter": int(launches), "peak_mib": round(torch.cuda.max_memory_allocated() / 2**20, 1),
                     "peak_above_resident_mib": round((torch.cuda.max_memory_allocated() - base) / 2**20, 1), "ms": []}
    for _ in range(args.rounds):
        for name, fn in forms.items():
            res[name]["ms"].append(round(window(fn, args.min_seconds)[0], 3))
    for r in res.values():
        r["ms_best"] = min(r["ms"])
    name, power = gpu_info()
    out = {"gpu": name, "power_limit": power, "batch": BATCH, "num_boxes": N_BOXES, "dims": DIMS, **res,
           "stepwise_over_fused": round(res["stepwise"]["ms_best"] / res["fused"]["ms_best"], 2)}
    print(json.dumps(out), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
