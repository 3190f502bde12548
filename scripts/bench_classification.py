#!/usr/bin/env python
"""Training throughput of the classification pretext models on one GPU: `Trainer.step` at batch 256.

For token classification (V = 10000, 30 labels per image) and multilabel classification (V = 81, 12 labels per image)
it reports, on the same GPU:
  * ours: `Trainer.step` images/s and ms/step, plus a phase split from CUDA events (forward; output-layer backward;
    pool + backbone backward; optimiser; and, timed apart, the backbone forward and the head forward: pool + logits
    GEMM + K-hot loss) -- the step is expected to be dominated by the backbone;
  * eager: torchvision ResNet-50 + global average pooling + nn.Linear under bf16 autocast, channels_last,
    cudnn.benchmark, torch.optim.SGD with global-norm clipping, once with the reference's per-image Python loss loop
    (virtex/models/classification.py:80-95, which reads labels back to the host image by image) and once with a
    vectorised K-hot loss, so that the host-bound loop does not overstate the speedup;
  * a torch.profiler run of one step of ours (separate from the timed loop): the time of the three new kernels
    against the least time their bytes take at 7.7 TB/s (the HGX B200 data-sheet HBM bandwidth).

    python scripts/bench_classification.py [--steps 10] [--warmup 3] [--loop-steps 2]

Prints the card name and power limit and ONE JSON line.  Writes nothing to the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TASKS = {  # config, labels per image
    "token_classification": ("task_ablations/token_classification_R_50.yaml", 30),
    "multilabel_classification": ("task_ablations/multilabel_classification_R_50.yaml", 12),
}
HBM_BYTES_S = 7.7e12


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001 -- the measurement still stands, the card is then named by torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def make_batch(B, V, L, kind, seed=0):
    g = torch.Generator().manual_seed(seed)
    image = torch.randn(B, 3, 224, 224, generator=g)
    if kind == "token_classification":  # [SOS] caption [EOS], right-padded
        labels = torch.randint(4, V, (B, L), generator=g)
        n = torch.randint(8, L + 1, (B,), generator=g)
        labels[torch.arange(L)[None, :] >= n[:, None]] = 0
        labels[:, 0] = 1
        labels[torch.arange(B), n - 1] = 2
    else:  # category ids with duplicates, 0-padded
        labels = torch.randint(1, V, (B, L), generator=g)
        labels[:, L // 2:] = 0
    return image.cuda(), labels.cuda()


def events(n):
    return [torch.cuda.Event(enable_timing=True) for _ in range(n)]


def ours(kind, B, steps, warmup):
    from virtex_b200.config import Config
    from virtex_b200.factories import PretrainingModelFactory
    from virtex_b200.trainer import Trainer

    cfg_name, L = TASKS[kind]
    cfg = Config(cfg_name)
    torch.manual_seed(0)
    model = PretrainingModelFactory.from_config(cfg).cuda().train()
    with torch.no_grad():  # zero-init residual branches would make the backbone a near-identity
        for n, p in model.named_parameters():
            if "bn3.weight" in n:
                p.fill_(0.25)
    tr = Trainer(model, cfg)
    eng = tr.engine
    image, labels = make_batch(B, cfg.DATA.VOCAB_SIZE, L, kind)
    batch = {"image": image, "labels": labels}
    for _ in range(warmup):
        tr.step(batch)
    torch.cuda.synchronize()
    e0, e1 = events(2)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        loss = tr.step(batch)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    wall = (time.perf_counter() - t0) * 1e3 / steps
    # phase split of the same step (events between the phases, averaged)
    ph = {"forward": 0.0, "output_layer_backward": 0.0, "pool_and_backbone_backward": 0.0, "optimizer": 0.0,
          "backbone_forward": 0.0}
    for _ in range(steps):
        ev = events(5)
        ev[0].record()
        eng.forward(image, None, None, None, training=True, with_grad=True, labels=labels)
        ev[1].record()
        eng.backward(zero_grads=True, bucket_cb=lambda tag: ev[2].record() if tag == "head" else None)
        ev[3].record()
        tr.optimizer_step()
        ev[4].record()
        torch.cuda.synchronize()
        ph["forward"] += ev[0].elapsed_time(ev[1]) / steps
        ph["output_layer_backward"] += ev[1].elapsed_time(ev[2]) / steps
        ph["pool_and_backbone_backward"] += ev[2].elapsed_time(ev[3]) / steps
        ph["optimizer"] += ev[3].elapsed_time(ev[4]) / steps
    ph["head_forward"] = 0.0
    for _ in range(steps):  # the two halves of the forward, timed apart
        a, b, c = events(3)
        a.record()
        feat, h, w = eng.backbone_forward(image, True)
        b.record()
        eng._classify(feat, B, h * w, labels, True)  # pool + logits GEMM + K-hot loss
        c.record()
        torch.cuda.synchronize()
        ph["backbone_forward"] += a.elapsed_time(b) / steps
        ph["head_forward"] += b.elapsed_time(c) / steps
    ph = {k: round(v, 3) for k, v in ph.items()}
    # one profiled step, plus one eval forward for the top-10 kernel
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tr.step(batch)
        model.eval()
        with torch.no_grad():
            model(batch)
        model.train()
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA and e.device_time_total > 0:
            kern[e.key] = (e.device_time_total / 1e3, e.count)
    V, C, S = cfg.DATA.VOCAB_SIZE, 2048, 49
    ldl = (V + 7) // 8 * 8
    pool_bytes = B * S * C * 2 + B * C * 2
    need = {  # bytes each kernel has to move at least (its own inputs and outputs)
        "avgpool_fwd_kernel": pool_bytes,
        "avgpool_bwd_kernel": B * S * C * 2 + B * C * 4,
        "khot_xent_kernel": B * ldl * 4 + B * L * 8 + B * ldl * 2,
        "topk_rows_kernel": B * ldl * 4 + B * 10 * 8,
    }
    new = {}
    for short, nbytes in need.items():
        hits = [(t, c) for k, (t, c) in kern.items() if short in k]
        if hits:
            t, c = hits[0]
            us = t * 1e3 / c
            new[short] = {"us": round(us, 2), "bytes": nbytes, "byte_bound_us": round(nbytes / HBM_BYTES_S * 1e6, 2),
                          "share_of_hbm_bound": round(nbytes / HBM_BYTES_S * 1e6 / us, 3)}
    busy = sum(t for t, _ in kern.values())
    return {"images_s": round(B / ms * 1e3, 1), "ms_per_step": round(ms, 3), "host_wall_ms_per_step": round(wall, 3),
            "loss": round(float(loss[0]), 4), "phases_ms": ph,
            "backbone_share_of_step": round((ph["backbone_forward"] + ph["pool_and_backbone_backward"]) / ms, 3),
            "profiled_step_plus_eval_gpu_busy_ms": round(busy, 3), "new_kernels": new}


def eager(kind, B, steps, warmup, loss_kind):
    import torchvision
    from torch import nn

    cfg_name, L = TASKS[kind]
    from virtex_b200.config import Config
    cfg = Config(cfg_name)
    V = cfg.DATA.VOCAB_SIZE
    ignore = [0, 1, 2, 3] if kind == "token_classification" else [0]
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(0)
    cnn = torchvision.models.resnet50(weights=None, zero_init_residual=True)
    cnn.fc = nn.Identity()
    head = nn.Linear(2048, V)
    model = nn.ModuleDict({"cnn": cnn, "head": head}).cuda().to(memory_format=torch.channels_last).train()
    opt = torch.optim.SGD([{"params": cnn.parameters(), "lr": 0.2}, {"params": head.parameters(), "lr": 0.001}],
                          momentum=0.9, weight_decay=1e-4)
    image, labels = make_batch(B, V, L, kind)
    image = image.contiguous(memory_format=torch.channels_last)
    ign = torch.tensor(ignore, device="cuda")

    def loss_loop(logits):  # the reference's per-image loop
        logprobs = torch.log_softmax(logits, dim=1)
        loss = torch.tensor(0.0, device=logits.device)
        for b in range(logits.shape[0]):
            unique = labels[b].unique()
            keep = [l for l in unique if l not in ignore]
            loss = loss - logprobs[b, keep].mean()
        return loss / logits.shape[0]

    def loss_vec(logits):  # K-hot matrix: duplicates collapse in scatter, ignored ids are cleared
        logprobs = torch.log_softmax(logits, dim=1)
        khot = torch.zeros_like(logprobs).scatter_(1, labels, 1.0)
        khot[:, ign] = 0
        return (-(logprobs * khot).sum(1) / khot.sum(1)).mean()

    loss_fn = loss_loop if loss_kind == "loop" else loss_vec

    def step():
        opt.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            logits = head(cnn(image))  # torchvision's forward pools globally before fc
        loss = loss_fn(logits.float())
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 10.0)
        opt.step()
        return loss

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = events(2)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"variant": f"eager torch {torch.__version__} + torchvision {torchvision.__version__}, bf16 autocast, "
                       f"channels_last, cudnn.benchmark, {loss_kind} loss",
            "images_s": round(B / ms * 1e3, 1), "ms_per_step": round(ms, 3), "steps": steps,
            "loss": round(float(loss), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tasks", default=",".join(TASKS))
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--loop-steps", type=int, default=2, help="timed steps of the host-bound per-image loss loop")
    ap.add_argument("--no-eager", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_classification.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    info = card()
    print(f"card: {info}", flush=True)
    result = {"card": info, "batch": args.batch, "tasks": {}}
    for kind in args.tasks.split(","):
        r = {"ours": ours(kind, args.batch, args.steps, args.warmup)}
        print(kind, "ours", json.dumps(r["ours"]), flush=True)
        torch.cuda.empty_cache()
        if not args.no_eager:
            r["eager_vectorised"] = eager(kind, args.batch, args.steps, args.warmup, "vectorised")
            print(kind, "eager", json.dumps(r["eager_vectorised"]), flush=True)
            r["eager_loop"] = eager(kind, args.batch, args.loop_steps, 1, "loop")
            print(kind, "eager", json.dumps(r["eager_loop"]), flush=True)
            r["speedup_vs_vectorised"] = round(r["ours"]["images_s"] / r["eager_vectorised"]["images_s"], 2)
            r["speedup_vs_loop"] = round(r["ours"]["images_s"] / r["eager_loop"]["images_s"], 2)
            torch.cuda.empty_cache()
        result["tasks"][kind] = r
    print(json.dumps(result))


if __name__ == "__main__":
    main()
