#!/usr/bin/env python
"""Benchmark of the Style-SeqCVAE var_updown hot path (BASELINE.json): training captions/s.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU

Workload at N GPUs (BASELINE configs[1] / [2], SURVEY §8d): per GPU one batch of 256 captions,
36x2048 fp32 region features, vocabulary 10 000, max length 20 (21 teacher-forced steps), shipped dims
(E=600 tied/frozen, H=900, A=768, Z=150, SENTIMENT_VAE=1), synthetic data, random-init weights.
One step = forward + loss + BPTT + (gradient all-reduce) + grad-clip + SGD(momentum, wd) update, i.e.
the body of the reference loop var_updown/scripts/train.py:163-176. A caption = one (image, caption) row.

`value`: K steps on inputs already resident in HBM (2 distinct batches are cycled: 151 MB of inputs
> 126 MB L2, and the ~1.6 GB per-step working set never stays L2-resident), CUDA events, max over ranks.
`e2e`: the same steps through UpDownCaptioner.forward with the batch in PINNED HOST memory: every
step does its own host->device copy (prefetched on a copy stream, inside the timed region) and a
device->host read of the step's loss.
After the timed region two extra instrumented steps give the per-kernel-class times for `roofline`.

`--dump-outputs DIR` writes what the last timed step of the device-resident arm computed (rank 0) as
DIR/<name>.npy, see dump_outputs(). Inputs, weights and noise are seeded, so two builds run with the same
arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

DIMS = dict(vocab_size=10000, image_feature_size=2048, embedding_size=600, hidden_size=900,
            attention_projection_size=768, z_space=150, sentiment_vae=1, simple_vae=False, max_caption_length=20,
            prior_std=1.0, senti_prior_multip=0.5)
N_BOXES = 36
KLD_WEIGHT = 750.0
# SURVEY §8d: model FLOPs of one training caption (fwd+bwd, x3 convention), dims Y
GFLOP_PER_CAPTION = 8.10
WORKLOAD = "style-seqcvae var_updown training step, batch 256/GPU, 36x2048 features, V=10k, L=20, dims E600/H900/A768/Z150"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


def synthetic_batch(B, seed, pin):
    g = torch.Generator().manual_seed(seed)
    feats = torch.rand(B, N_BOXES, DIMS["image_feature_size"], generator=g)
    lens = torch.randint(5, 21, (B,), generator=g)
    toks = torch.randint(2, DIMS["vocab_size"], (B, 20), generator=g)
    toks[torch.arange(20)[None, :] >= lens[:, None]] = 0
    sent = torch.randint(-1, 2, (B, 1), generator=g).float()
    if pin:
        feats, toks, sent = feats.pin_memory(), toks.pin_memory(), sent.pin_memory()
    return feats, toks, sent


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_run(steps, warmup, B=8):
    """The reference algorithm on the host CPU: the oracle port (oracle/updown_oracle.py, pinned against the
    unmodified reference by tests/golden) — forward + loss + backward (autograd BPTT) on BASELINE config 0
    (B=8), all host threads, dims and shapes of the GPU workload."""
    from oracle import updown_oracle as uo
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = uo.OracleConfig(**DIMS)
    p = uo.init_params(cfg, seed=0)
    for k, v in p.items():
        if not (cfg.tied and k in ("_embedding_layer.weight", "_output_layer.weight")):
            v.requires_grad_(True)
    feats, toks, sent = synthetic_batch(B, 0, False)
    feats = feats[:, :N_BOXES]
    g = torch.Generator().manual_seed(1234)
    eps = torch.randn(21, B, DIMS["z_space"], generator=g)

    def step():
        for v in p.values():
            v.grad = None
        out = uo.train_forward(p, cfg, feats, toks, sent, eps)
        uo.train_objective(out, KLD_WEIGHT).backward()
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return dict(value=B * steps / dt, unit="captions/s", cores=torch.get_num_threads(), kind="port",
                sample=f"{steps} steps of fwd+loss+bwd on a batch of {B} captions (BASELINE config 0), fp32, torch CPU",
                seconds=dt)


def gpu_eager_reference_run(dev, B, steps=3, warmup=2):
    """SURVEY 8(d) last sentence / BASELINE.md 3.5: "the reference PyTorch path on the B200" - the pinned oracle port of
    the reference module (plain torch ops, autograd BPTT) run by torch eager ON THE GPU, same workload as the timed
    arm: batch B, fwd + loss + backward + clip_grad_norm_(12.5) + torch.optim.SGD(momentum, wd). Three arithmetic
    modes: fp32 (the reference's own), tf32 matmuls, bf16 autocast. Baseline leg only: never on the product path."""
    from oracle import updown_oracle as uo
    out = {}
    cfg = uo.OracleConfig(**DIMS)
    feats, toks, sent = (t.to(dev) for t in synthetic_batch(B, 0, False))
    for mode in ("fp32", "tf32", "bf16_autocast"):
        torch.backends.cuda.matmul.allow_tf32 = mode == "tf32"
        p = {k: v.to(dev) for k, v in uo.init_params(cfg, seed=0).items()}
        train = [v.requires_grad_(True) for k, v in p.items()
                 if not (cfg.tied and k in ("_embedding_layer.weight", "_output_layer.weight"))]
        opt = torch.optim.SGD(train, lr=0.015, momentum=0.9, weight_decay=0.001)
        g = torch.Generator(device=dev).manual_seed(1234)

        def step():
            opt.zero_grad()
            eps = torch.randn(21, B, DIMS["z_space"], generator=g, device=dev)
            with torch.device(dev), torch.autocast("cuda", dtype=torch.bfloat16, enabled=mode == "bf16_autocast"):
                o = uo.train_forward(p, cfg, feats, toks, sent, eps)
            uo.train_objective(o, KLD_WEIGHT).backward()
            torch.nn.utils.clip_grad_norm_(train, 12.5)
            opt.step()
        try:
            for _ in range(warmup):
                step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {"value": B / (ms / 1e3), "unit": "captions/s", "ms_per_step": ms}
        except Exception as ex:                                     # e.g. an op autocast cannot handle
            out[mode] = {"error": f"{type(ex).__name__}: {ex}"[:200]}
        del p, train, opt
    torch.backends.cuda.matmul.allow_tf32 = False
    out["what"] = (f"oracle port of var_updown UpDownCaptioner (oracle/updown_oracle.py, pinned to the reference by tests/golden) "
                   f"in torch {torch.__version__} eager on this GPU, batch {B}, fwd+loss+bwd+clip+SGD, {steps} timed steps")
    return out


def synthetic_fsm(n_images, vocab, constraint_ids):
    """(B, 2^k, 2^k, V) uint8 adjacency tensor of k single-word constraints (the shape the reference's
    FiniteStateMachineBuilder hands to ConstrainedBeamSearch, updown-baseline/updown/utils/constraints.py:329-361):
    fsm[b, s, s2, w] = 1 iff emitting word w moves state s -> s2. State = bitmask of satisfied constraints."""
    k = len(constraint_ids)
    S = 1 << k
    fsm = torch.zeros(S, S, vocab, dtype=torch.uint8)
    for s in range(S):
        fsm[s, s, :] = 1
        for i, ids in enumerate(constraint_ids):
            if not (s >> i) & 1:
                for w in ids:
                    fsm[s, s, w] = 0
                    fsm[s, s | (1 << i), w] = 1
    return fsm[None].repeat(n_images, 1, 1, 1).contiguous()


DUMP_SAMPLE = 1 << 16          # elements kept per parameter / gradient tensor
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, out, named):
    """What a caller of one training step receives, from the last timed step: the per-caption losses `loss` and `kld`
    (B,), and for every trainable parameter its gradient (`grad.<name>`) and its value after the clip + SGD update
    (`param.<name>`). Tensors larger than DUMP_SAMPLE elements are reduced to a fixed sample: the flat indices of the
    first DUMP_SAMPLE entries of a permutation seeded with 0, in ascending order, so every run picks the same ones."""
    import numpy as np
    arrays = {"loss": out["loss"], "kld": out["kld"]}
    for k, p in named:
        if p.grad is not None:
            arrays["grad." + k] = p.grad
        arrays["param." + k] = p.detach()
    torch.cuda.synchronize()
    host = {}
    for name, t in arrays.items():
        t = t.detach().float().reshape(-1)
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            t = t[idx.to(t.device)]
        host[name] = t.cpu().numpy().astype(np.float32)
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_MAX_BYTES, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def decode_legs(sscvae, vocab, train_model, dev, world, max_over_ranks, barrier):
    """BASELINE configs[3] and [4]: decode throughput through UpDownCaptioner.forward (eval), images sharded over
    ranks with no collective. (a) diverse sampling: 100 latent samples per image, greedy decode - the reference loop
    `for k in range(N_Z_SAMPLES): model(image_features, ...)` (var_updown/scripts/inference.py:138-167);
    (b) constrained beam search, beam 5, 3 single-word constraints (8 FSM states, 40 rows per image)."""
    out = {}
    sd = train_model.state_dict()

    def build(beam, cbs):
        m = sscvae.UpDownCaptioner(vocab, DIMS["image_feature_size"], DIMS["embedding_size"], DIMS["hidden_size"],
                                   DIMS["attention_projection_size"], max_caption_length=20, beam_size=beam, use_cbs=cbs,
                                   min_constraints_to_satisfy=2, z_space=DIMS["z_space"], prior_std=1.0, simple_vae=False,
                                   latent_embedding="glove", sentiment_vae=1, senti_prior_multip=0.5, cbs_simple=True,
                                   device=dev).to(dev)
        m.load_state_dict(sd)
        m.eval()
        return m

    def timed(fn, calls, warm):
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    g = torch.Generator().manual_seed(7)
    # (a) diverse sampling, greedy
    n_img, n_samples = 256, 100
    feats = torch.rand(n_img, N_BOXES, DIMS["image_feature_size"], generator=g).to(dev)
    sent = torch.randint(-1, 2, (n_img, 1), generator=g).float().to(dev)
    m1 = build(1, False)
    ms = timed(lambda: m1(feats, None, None, sentiment=sent)["predictions"], n_samples, 3)
    out["sampling_greedy"] = {"value": n_img * n_samples * world / (ms / 1e3), "unit": "captions/s",
                              "images_per_gpu": n_img, "samples_per_image": n_samples, "ms_per_call": ms / n_samples,
                              "config": "BASELINE configs[3]: 100 latent samples per image, greedy decode, max length 20"}
    # the same workload through the batched entry point (UpDownCaptioner.sample -> sscvae_decode_samples): the
    # 100 sequences of an image are rows of one batch sharing its region features; 64 images x 100 samples per call
    n_img_b, calls = 64, 3
    fb, sb = feats[:n_img_b].contiguous(), sent[:n_img_b].contiguous()
    # 4 warm-up calls: the first computes the per-image state, the second is the first sighting of the "reuse" key, the
    # third captures the call into a graph (tens of ms, measured inside the timed region with 2 warm-up calls)
    ms = timed(lambda: m1.sample(fb, sentiment=sb, n_samples=n_samples)["predictions"], calls, 4)
    out["sampling_greedy_batched"] = {"value": n_img_b * n_samples * calls * world / (ms / 1e3), "unit": "captions/s",
                                      "images_per_gpu": n_img_b, "samples_per_image": n_samples, "ms_per_call": ms / calls,
                                      "config": "BASELINE configs[3] in one call per 64 images: rows = images x 100 samples"}
    del m1
    # (b) CBS beam 5, 3 constraints -> 8 states
    n_img, calls = 64, 5
    feats = feats[:n_img].contiguous()
    sent = sent[:n_img].contiguous()
    fsm = synthetic_fsm(n_img, DIMS["vocab_size"], [[11, 12], [57], [300, 301, 302]]).to(dev)
    nc = torch.full((n_img,), 3, dtype=torch.long, device=dev)
    m5 = build(5, True)
    ms = timed(lambda: m5(feats, None, None, fsm=fsm, num_constraints=nc, sentiment=sent)["predictions"], calls, 4)
    out["cbs_beam5"] = {"value": n_img * calls * world / (ms / 1e3), "unit": "captions/s", "images_per_gpu": n_img,
                        "fsm_states": 8, "beam": 5, "rows_per_image": 40, "ms_per_call": ms / calls,
                        "config": "BASELINE configs[4]: constrained beam search, beam 5, 3 word constraints, max length 20"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="captions per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed training step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    # a stalled run ends itself with every thread's stack on stderr instead of waiting for the caller's timeout
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("SSCVAE_BENCH_WATCHDOG_S", "420")), exit=True)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # >= 4: the library replays a call as a CUDA graph from its third sighting on (eager, capture, replay); with the
    # two resident batches below every call signature has been captured before the timed region starts
    warmup = max(args.warmup, 4) if args.impl == "ours" else max(args.warmup, 1)

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of --impl ours")
        if rank != 0:
            return
        r = cpu_reference_run(args.steps, warmup)
        line = dict(metric="train_captions_per_sec", value=r["value"], unit="captions/s", n_gpus=args.gpus,
                    steps=args.steps, warmup=warmup, ms_per_step=1e3 * r["seconds"] / args.steps,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                    impl="reference", config={"workload": WORKLOAD, "sample_batch": 8},
                    cpu_baseline={k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                    e2e={"value": r["value"], "unit": "captions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                    gpu_launches=0)
        print(json.dumps(line), flush=True)
        return

    import sscvae
    from sscvae import _lib

    class _Vocab:                      # the four methods the captioner needs (SURVEY §8b)
        def get_vocab_size(self, namespace="tokens"):
            return DIMS["vocab_size"]

        def get_token_index(self, token, namespace="tokens"):
            return {"@@UNKNOWN@@": 0, "@@BOUNDARY@@": 1}[token]

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch

    def progress(msg):                 # stderr breadcrumbs: where a multi-rank run is when something stalls
        if rank == 0:
            print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)
    progress(f"process group up: world {world}")
    torch.manual_seed(0)
    model = sscvae.UpDownCaptioner(
        _Vocab(), DIMS["image_feature_size"], DIMS["embedding_size"], DIMS["hidden_size"],
        DIMS["attention_projection_size"], max_caption_length=20, beam_size=5, use_cbs=True,
        min_constraints_to_satisfy=2, z_space=DIMS["z_space"], prior_std=1.0, simple_vae=False,
        latent_embedding="glove", sentiment_vae=1, senti_prior_multip=0.5, cbs_simple=True, device=dev).to(dev)
    model.train()
    named = [(k, p) for k, p in model.named_parameters() if p.requires_grad]
    opt = sscvae.FusedClipSGD([p for _, p in named], lr=0.015, momentum=0.9, weight_decay=0.001, max_norm=12.5,
                              num_iterations=70000)
    reducer = sscvae.BucketedGradReducer(named) if world > 1 else None
    # data-parallel mode: "events" (default): the backward records one event per gradient bucket as soon as it is final
    # (external event-record nodes of the replayed graph) and the in-place all-reduce of that bucket starts on a side
    # stream; "plain": all buckets are reduced after the backward has finished
    dp_mode = os.environ.get("SSCVAE_BENCH_DP", "events")
    if world > 1 and dp_mode == "events":
        model._group_events = [torch.cuda.Event() for _ in range(_lib.GRAD_GROUPS)]
        for e in model._group_events:      # torch creates the cudaEvent_t at the first record: a handle of 0 would be skipped
            e.record()
        assert all(e.cuda_event for e in model._group_events)

    n_batches = 2
    host = [synthetic_batch(B, 100 * rank + i, True) for i in range(n_batches)]
    resident = [tuple(t.to(dev) for t in b) for b in host]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host[0])

    last = {}                          # outputs of the latest step (for --dump-outputs)

    def train_step(feats, toks, sent):
        opt.zero_grad()
        out = model(feats, None, None, toks, sent)
        last["out"] = out
        loss = out["loss"].mean() + out["kld"].mean() / KLD_WEIGHT        # train.py:168-171
        loss.backward()
        if reducer is not None:
            if comm["on"]:
                comm["bwd_end"].append(torch.cuda.Event(enable_timing=True))
                comm["bwd_end"][-1].record()
            # the all-reduce leaves the SUM in the buckets; the optimizer kernel takes the mean (grad_scale) on the fly
            reducer.reduce(model._group_events, buckets=model.grad_buckets(), average=False)
            if comm["on"] and reducer.last_comm_done is not None:
                comm["comm_end"].append(reducer.last_comm_done)
        opt.step(grad_scale=1.0 / world)                                  # clip 12.5 + SGD + lr schedule
        return loss.detach()

    comm = {"on": False, "bwd_end": [], "comm_end": []}      # timed region of the device-resident arm: exposed all-reduce time

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---------------------------------------------------------------- device-resident arm
    for i in range(warmup):
        train_step(*resident[i % n_batches])
    barrier()
    progress("warm-up done")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    comm["on"] = world > 1
    e0.record()
    for i in range(args.steps):
        train_step(*resident[i % n_batches])
    e1.record()
    barrier()
    comm["on"] = False
    ms_dev = max_over_ranks(e0.elapsed_time(e1))
    # all-reduce time that is NOT hidden behind backward: end of the last collective minus end of the backward graph
    comm_exposed_ms = None
    if comm["comm_end"]:
        ex = [max(0.0, a.elapsed_time(b)) for a, b in zip(comm["bwd_end"], comm["comm_end"])]
        comm_exposed_ms = max_over_ranks(sum(ex) / len(ex))
    launches = _lib.launch_count() - launches0
    progress(f"device-resident arm done: {ms_dev / args.steps:.3f} ms/step")
    if args.dump_outputs and rank == 0:
        nbytes = dump_outputs(args.dump_outputs, last["out"], named)
        progress(f"outputs of the last timed step written to {args.dump_outputs} ({nbytes / 1e6:.1f} MB)")

    # ---------------------------------------------------------------- end-to-end arm (host buffers)
    copy_stream = torch.cuda.Stream()
    dbuf = [tuple(torch.empty_like(t, device=dev) for t in host[0]) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    loss_host = torch.zeros(args.steps + warmup, dtype=torch.float32).pin_memory()

    def prefetch(slot, batch):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            for d, h in zip(dbuf[slot], batch):
                d.copy_(h, non_blocking=True)
            ready[slot].record(copy_stream)

    def e2e_loop(n, base):
        for s in (0, 1):
            consumed[s].record()
        prefetch(0, host[0])
        for i in range(n):
            slot = i & 1
            if i + 1 < n:
                prefetch(slot ^ 1, host[(i + 1) % n_batches])
            torch.cuda.current_stream().wait_event(ready[slot])
            loss = train_step(*dbuf[slot])
            consumed[slot].record()
            loss_host[base + i].copy_(loss, non_blocking=True)          # device->host read of the step's loss
    e2e_loop(warmup, 0)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    e2e_loop(args.steps, warmup)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    progress(f"end-to-end arm done: {ms_e2e / args.steps:.3f} ms/step")
    assert torch.isfinite(loss_host).all(), "non-finite loss in the end-to-end arm"

    # ---------------------------------------------------------------- instrumented steps -> roofline
    peaks = load_peaks()
    _lib.profile(True)
    for i in range(args.profile_steps):
        train_step(*resident[i % n_batches])
    rep = _lib.profile_report()
    _lib.profile(False)
    kernels, total_ms = {}, sum(v["ms"] for v in rep.values())
    for k, v in sorted(rep.items(), key=lambda kv: -kv[1]["ms"]):
        ms = v["ms"] / args.profile_steps
        e = {"launches_per_step": v["count"] / args.profile_steps, "ms_per_step": round(ms, 4),
             "share": round(v["ms"] / total_ms, 4)}
        if v["flops"] > 0:
            e["tflops"] = round(v["flops"] / v["ms"] / 1e9, 2)
        if v["bytes"] > 0:
            e["gbs"] = round(v["bytes"] / v["ms"] / 1e6, 1)
        kernels[k] = e
    # Dominant kernel = the instrumented class with the largest share of the step. Since round 2 these are the two
    # persistent recurrent kernels: "recurrent_bwd" (the BPTT loop) and "recurrent_fwd" (the forward recurrence), each one
    # cooperative launch for all 21 timesteps. The per-launch instrumentation serialises the
    # stream, so a class's SHARE of the instrumented step is applied to the timed step: duration = share x ms_per_step.
    step_ms = ms_dev / args.steps
    Hh, Ff, Zz, Ee, Aa, Tt = (DIMS["hidden_size"], DIMS["image_feature_size"], DIMS["z_space"], DIMS["embedding_size"],
                              DIMS["attention_projection_size"], 21)
    # ALGORITHMIC flops per training step (reference math, unpadded dims, 2 flops per MAC):
    #   recurrent_fwd : per row and timestep the in-loop part of the three LSTMs (attention: emb + h1 + h_dec + W_hh h1
    #                   columns; encoder: xhat + h1 + h_dec + W_hh h_enc; decoder: xhat + h1 + h_dec + z + W_hh h_dec), the
    #                   query projection, fc_mean / fc_log_var and the region attention (scores + weighted sum)
    #   gemm.recurrent: the three BPTT data gradients dX = dG W of the same LSTM blocks (per-launch backward only)
    #   recurrent_bwd : the persistent BPTT kernel: those three GEMMs + d z (inside the decoder block above), the latent heads
    #                   and the query projection transposed, and the region attention backward (d alpha + d q)
    alg = {
        "recurrent_fwd": 2.0 * B * Tt * (4 * Hh * ((Ee + 3 * Hh) + (Ff + 3 * Hh) + (Ff + 3 * Hh + Zz)) + Hh * Aa + 2 * Hh * Zz
                                         + N_BOXES * (Aa + Ff)),
        "gemm.recurrent": 2.0 * B * Tt * 4 * Hh * (2 * Hh + (Ff + 3 * Hh) + (Ff + 2 * Hh + Zz)),
        "recurrent_bwd": 2.0 * B * Tt * (4 * Hh * (2 * Hh + (Ff + 3 * Hh) + (Ff + 2 * Hh + Zz)) + Hh * Aa + 2 * Hh * Zz
                                         + N_BOXES * (Aa + Ff)),
    }
    names = {"recurrent_fwd": "recurrent_fwd_kernel (persistent cooperative kernel, all T steps of the UpDown cell)",
             "gemm.recurrent": "gemm_tcgen05_swapped_pair_kernel (BPTT data-gradient GEMMs, M = batch)",
             "recurrent_bwd": "recurrent_bwd_kernel (persistent cooperative kernel, all T reverse steps of the BPTT loop)"}
    traffic_file = os.path.join(ROOT, "profiles", "ncu_traffic_r02.json")        # dram read+write per launch, from ncu --set full
    traffic = json.load(open(traffic_file)) if os.path.exists(traffic_file) else {}
    gemm_all = [v for k, v in rep.items() if k.startswith("gemm")]
    roofline, roofline_other = None, {}
    # "gemm.recurrent" only counts as the BPTT class when the per-launch backward ran (3 launches per timestep)
    ranked = sorted((k for k in rep if k in alg and (k != "gemm.recurrent" or rep[k]["count"] / args.profile_steps > Tt)),
                    key=lambda k: -rep[k]["ms"])
    for k in ranked:
        v = rep[k]
        share = v["ms"] / total_ms
        n_launch = v["count"] / args.profile_steps
        r = {"kernel": names[k], "class": k, "bound": "tensor", "achieved": alg[k] / (share * step_ms) / 1e9,
             "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": alg[k] / (share * step_ms) / 1e9 / peaks["tf_sustained"],
             "traffic": traffic.get(k), "flops_per_launch": alg[k] / n_launch, "executed_flops_per_launch": v["flops"] / v["count"],
             "peak_source": peaks["src"] + " bf16_tflops_sustained", "share_of_step": share, "launches_per_step": n_launch,
             "avg_launch_us": 1e3 * share * step_ms / n_launch}
        if roofline is None:
            roofline = r
        else:
            roofline_other[k] = r
    if roofline is not None:
        roofline["all_gemm_share_of_step"] = sum(v["ms"] for v in gemm_all) / total_ms
        roofline["other_classes"] = roofline_other
    for k in ("attention_bwd", "attention_fwd", "ce_fwd", "ce_bwd"):            # HBM-bound classes: achieved GB/s of their algorithmic bytes
        if k in rep and rep[k]["bytes"] > 0:
            share = rep[k]["ms"] / total_ms
            gbs = rep[k]["bytes"] / args.profile_steps / (share * step_ms) / 1e6
            roofline_other[k] = {"class": k, "bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s",
                                 "frac": gbs / peaks["hbm"], "share_of_step": share}

    progress("instrumented steps done")
    decode = None
    if not args.no_decode:
        decode = decode_legs(sscvae, _Vocab(), model, dev, world, max_over_ranks, barrier)
        progress("decode legs done")

    captions = B * world * args.steps
    value = captions / (ms_dev / 1e3)
    e2e_value = captions / (ms_e2e / 1e3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = dict(
        metric="train_captions_per_sec", value=value, unit="captions/s", n_gpus=world, steps=args.steps, warmup=warmup,
        ms_per_step=ms_dev / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
        data="synthetic",
        config={"workload": WORKLOAD, "global_batch": B * world, "parallelism": f"dp{world}",
                "l2": f"{n_batches} distinct input batches cycled ({n_batches * h2d_bytes / 1e6:.0f} MB > 126 MB L2); no explicit flush",
                "step": "fwd + loss + BPTT + grad all-reduce + clip 12.5 + SGD(momentum 0.9, wd 1e-3)"},
        clocks=clocks,
        e2e={"value": e2e_value, "unit": "captions/s", "ms_per_step": ms_e2e / args.steps,
             "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
        gpu_launches=int(launches),
        comm_exposed_ms=comm_exposed_ms,
        roofline=roofline,
        roofline_step={"bound": "tensor", "achieved": value * GFLOP_PER_CAPTION / 1e3, "peak": peaks["tf_sustained"] * world,
                       "unit": "TFLOP/s", "frac": value * GFLOP_PER_CAPTION / 1e3 / (peaks["tf_sustained"] * world),
                       "note": "model FLOPs (8.10 GFLOP/caption, SURVEY §8d) / step time"},
        kernels=kernels,
        decode=decode,
    )
    if not args.no_gpu_eager and world == 1:
        del model, opt
        torch.cuda.empty_cache()
        line["gpu_eager_baseline"] = gpu_eager_reference_run(dev, B)
        progress("gpu eager reference leg done")
    if not args.no_cpu_baseline and world == 1:
        r = cpu_reference_run(20, 1)           # ~12 s of host work
        line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    else:
        line["cpu_baseline"] = None
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
