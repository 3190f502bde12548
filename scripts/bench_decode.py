#!/usr/bin/env python
"""Throughput of beam-search captioning on one GPU: `model.eval(); model({"image": ...})["predictions"]`.

For each config (batch 256, beam 5, per-node 2, 30 steps; random weights, so EOS is rare and most batches run all 30
steps) it reports images/s of this project's KV-cached decode and of an eager-PyTorch decode on the same GPU: the
`scripts/gpu_incumbent.py` model under bf16 autocast driving `oracle.decode_oracle.beam_search`, which -- like the
reference's `decoding_step` -- re-runs the textual head over the whole prefix at every step.  A separate
torch.profiler run of one decode gives the GPU-busy time (sum of kernel times) against the host wall time, and the
kernel launches per step: when the GPU is busy for much less than the wall time, the loop is host-bound.

    python scripts/bench_decode.py [--configs base,l4,r101_h2048] [--reps 3] [--no-eager]

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
sys.path.insert(0, os.path.join(ROOT, "scripts"))

CONFIGS = {
    "base": ("_base_bicaptioning_R_50_L1_H1024.yaml", []),
    "l4": ("depth_ablations/bicaptioning_R_50_L4_H1024.yaml", []),
    "r101_h2048": ("backbone_ablations/bicaptioning_R_101_L1_H1024.yaml",
                   ["MODEL.TEXTUAL.NAME", "transdec_postnorm::L1_H2048_A32_F8192"]),
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001 -- the measurement still stands, the card is then named by torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def timed(fn, reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    outs = [fn() for _ in range(reps)]
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, (time.perf_counter() - t0) * 1e3 / reps, outs[-1]


def ours(cfg_name, overrides, image, reps):
    from virtex_b200 import ops
    from virtex_b200.config import Config
    from virtex_b200.factories import PretrainingModelFactory

    torch.manual_seed(0)
    cfg = Config(cfg_name, overrides)
    model = PretrainingModelFactory.from_config(cfg).cuda().eval()
    run = lambda: model({"image": image})["predictions"]
    run()  # warm-up: every workspace buffer and module load
    ms, wall_ms, pred = timed(run, reps)
    L = pred.shape[1]
    n0 = ops.launch_count
    run()
    launches = ops.launch_count - n0
    # profiled run of its own: GPU busy vs host wall
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        run()
        torch.cuda.synchronize()
        prof_wall = (time.perf_counter() - t0) * 1e3
    kernels = {e.key: e.device_time_total / 1e3 for e in prof.key_averages()
               if e.device_type == torch.autograd.DeviceType.CUDA and e.device_time_total > 0}
    busy = sum(kernels.values())
    top = {k: round(v, 3) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])[:8]}
    B = image.shape[0]
    return {"images_s": round(B / (ms / 1e3), 1), "ms_per_decode": round(ms, 2), "host_wall_ms": round(wall_ms, 2),
            "steps": L, "ms_per_step": round(ms / L, 3), "launches_per_decode": launches,
            "launches_per_step": round(launches / L, 1),
            "profiled": {"wall_ms": round(prof_wall, 2), "gpu_busy_ms": round(busy, 2),
                         "gpu_busy_share": round(busy / prof_wall, 3), "top_kernels_ms": top}}


def eager(cfg_name, overrides, image, reps):
    from gpu_incumbent import Bicaptioning
    from oracle import decode_oracle as D
    from virtex_b200.config import Config

    cfg = Config(cfg_name, overrides)
    arch = cfg.MODEL.VISUAL.NAME.split("::")[-1]
    L, H, A, F = [int(x[1:]) for x in cfg.MODEL.TEXTUAL.NAME.split("::")[-1].split("_")]
    torch.manual_seed(0)
    model = Bicaptioning(arch, cfg.DATA.VOCAB_SIZE, H, L, A, F, dropout=0.0).cuda().eval()
    dec = cfg.MODEL.DECODER
    B = image.shape[0]

    @torch.no_grad()
    def run():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            x = image
            for name, layer in model.cnn.named_children():
                x = layer(x)
                if name == "layer4":
                    break

            def step(partial):
                if partial.dim() == 1:
                    partial = partial.unsqueeze(1)
                rows, T = partial.shape
                feats = x.repeat_interleave(rows // B, 0)  # the reference repeats the features per beam
                lengths = torch.full((rows,), T, dtype=torch.int64, device=partial.device)
                return model.textual(feats, partial, lengths)[:, -1].float()

            start = torch.full((B,), cfg.DATA.SOS_INDEX, dtype=torch.int64, device="cuda")
            return D.beam_search(start, step, cfg.DATA.EOS_INDEX, dec.MAX_DECODING_STEPS, dec.BEAM_SIZE, 2)[0]

    run()
    ms, wall_ms, pred = timed(run, reps)
    return {"images_s": round(B / (ms / 1e3), 1), "ms_per_decode": round(ms, 2), "steps": pred.shape[1],
            "variant": f"eager torch {torch.__version__}, bf16 autocast, full-prefix recompute per step"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="base,l4,r101_h2048")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-eager", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_decode.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    info = card()
    print(f"card: {info}", flush=True)
    g = torch.Generator(device="cuda").manual_seed(1)
    image = torch.randn(args.batch, 3, 224, 224, device="cuda", generator=g)
    result = {"card": info, "batch": args.batch, "beam": 5, "max_steps": 30, "configs": {}}
    for name in args.configs.split(","):
        cfg_name, over = CONFIGS[name]
        r = {"ours": ours(cfg_name, over, image, args.reps)}
        print(name, "ours", json.dumps(r["ours"]), flush=True)
        if not args.no_eager:
            r["eager"] = eager(cfg_name, over, image, args.reps)
            r["speedup"] = round(r["ours"]["images_s"] / r["eager"]["images_s"], 2)
            print(name, "eager", json.dumps(r["eager"]), flush=True)
        result["configs"][name] = r
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
