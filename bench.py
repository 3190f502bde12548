#!/usr/bin/env python
"""Benchmark of the bicaptioning pretraining step (BASELINE.json metric: image-caption pairs/sec, R50-L1-H1024).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference algorithm on the host cores (oracle port)

A "step" is one full optimisation step (forward + backward + gradient all-reduce + clip + SGD/Lookahead) on a synthetic
batch of 256 pairs per GPU (weak scaling), random-init weights of the named architecture, dropout 0.1 as configured.
Rank 0 prints ONE JSON line.  `value` = device-resident inputs, CUDA-event timed, max over ranks; `e2e` = the same
step through `Trainer.step` fed from pinned HOST buffers (H2D copy of every batch and D2H read of every loss inside
the timed region).  `roofline` is for the dominant kernel (the tcgen05 GEMM, which runs every conv and linear layer).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "image-caption pairs/sec bicaptioning R50-L1-H1024"
GFLOP_PER_PAIR = 35.17  # fwd+bwd conv+matmul work per pair, vis-proj de-duplicated (SURVEY.md section 8d-2)


def synth_host_batch(B, T=30, vocab=10000, seed=0, pin=True):
    g = torch.Generator().manual_seed(seed)
    image = torch.randn(B, 3, 224, 224, generator=g)
    tokens = torch.randint(4, vocab, (B, T), generator=g)
    tokens[:, 0], tokens[:, -1] = 1, 2
    batch = {"image": image, "caption_tokens": tokens, "noitpac_tokens": tokens.flip(1).contiguous(),
             "caption_lengths": torch.full((B,), T, dtype=torch.int64)}
    if pin:
        batch = {k: v.pin_memory() for k, v in batch.items()}
    return batch


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.perf_counter()] + [x.strip() for x in line.split(",")])

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        inside = [r[1:] for r in self.rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or r[0])]
        rows = inside if inside else [r[1:] for r in self.rows]  # sampler started under load (warm-up) as a fallback
        sm = sorted(float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(rows), "samples_in_timed_region": len(inside)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p.get("bf16_tflops_sustained", 1412.4), p.get("hbm_gbs", 6590.9), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------- CPU / reference
def usable_cores():
    """Host cores this process may really use: min(affinity mask, cgroup CPU quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(quota) // int(period)))
    except (OSError, ValueError):
        pass
    return n


def run_cpu_reference(steps, warmup, batch, threads=None):
    """The reference algorithm (oracle port, fp32, CPU autograd) timed on the host cores: full optimisation steps."""
    from oracle import virtex_oracle as O
    threads = threads or usable_cores()
    torch.set_num_threads(threads)
    spec = O.Spec()
    tr = O.OracleTrainer(O.synth_state(spec, 0, randomize_bn=False), spec)
    hb = synth_host_batch(batch, pin=False)
    hb["image_id"] = torch.arange(batch)
    for _ in range(warmup):
        tr.step(hb)
    t0 = time.perf_counter()
    for _ in range(steps):
        tr.step(hb)
    dt = time.perf_counter() - t0
    return steps * batch / dt, dt / steps, threads


def main_reference(args, rank, world):
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    warm = 1
    B = args.cpu_batch
    v, sec, threads = run_cpu_reference(steps, warm, B)
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": round(sec * 1e3, 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "bicaptioning R50_L1_H1024 full optimisation step, batch 256 per GPU",
                       "sample": f"reference algorithm on the host cores, each step = {B} pairs of that workload",
                       "global_batch": B},
            "cpu_baseline": {"value": round(v, 3), "unit": "pairs/s", "cores": threads, "kind": "port",
                             "sample": f"{steps} full steps at batch {B} after {warm} warm-up (oracle port of the reference, fp32)"},
            "e2e": {"value": round(v, 3), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------- incumbent (eager GPU)
def run_incumbent(args, cfg):
    """The reference's own GPU path on the same box: eager PyTorch (cuDNN / cuBLASLt / SDPA) under bf16 autocast,
    channels_last -- scripts/gpu_incumbent.py in a subprocess (its own CUDA context and memory), N = 1 only."""
    m = __import__("re").match(r"L(\d+)_H(\d+)_A(\d+)_F(\d+)", cfg.MODEL.TEXTUAL.NAME.split("::")[1])
    cmd = [sys.executable, os.path.join(ROOT, "scripts", "gpu_incumbent.py"), "--variant", "channels_last",
           "--arch", cfg.MODEL.VISUAL.NAME.split("::")[-1], "--layers", m.group(1), "--hidden", m.group(2),
           "--batch", str(args.batch_per_gpu), "--steps", "10", "--warmup", "4"]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
        for line in reversed(out.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)["incumbent"]
        return {"unavailable": (out.stderr.strip().splitlines() or ["no output"])[-1][:200]}
    except Exception as e:  # noqa: BLE001 -- a reported baseline must never take the bench line down
        return {"unavailable": repr(e)[:200]}


def dp_gradient_check(trainer, dev_batch, world):
    """Data-parallel parity on real NCCL (scripts/pretrain_virtex.py:121-123, DDP semantics): the gradients the
    optimiser consumes -- bucketed SUM all-reduce on the side stream, 1/world folded in afterwards -- must equal the
    mean over ranks of the per-rank gradients.  Checked on every bucket; the reference value comes from an
    all_gather of the un-reduced gradients."""
    import torch.distributed as dist
    eng = trainer.engine
    eng.seed.add_(1)
    eng.forward(dev_batch["image"], dev_batch["caption_tokens"], dev_batch["noitpac_tokens"],
                dev_batch["caption_lengths"], training=True, with_grad=True)
    eng.backward(zero_grads=True, bucket_cb=None)
    torch.cuda.synchronize()
    local = eng.arena.grads.clone()
    worst = 0.0
    for tag in trainer._ranges:
        trainer._on_bucket(tag)
    for w in trainer._pending:
        w.wait()
    trainer._pending.clear()
    torch.cuda.synchronize()
    for tag, r in trainer._ranges.items():
        if r is None:
            continue
        n = min(r[1] - r[0], 1 << 22)  # first 4 Mi elements of every bucket: all_gather of the whole arena is not needed
        mine = local[r[0]:r[0] + n].contiguous()
        gathered = torch.empty(world * n, dtype=mine.dtype, device=mine.device)
        dist.all_gather_into_tensor(gathered, mine)
        mean = gathered.view(world, n).double().mean(0)
        got = eng.arena.grads[r[0]:r[0] + n].double() / world
        err = ((got - mean).abs().max() / (mean.abs().max() + 1e-30)).item()
        worst = max(worst, err)
    t = torch.tensor([worst], device=local.device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return {"max_rel_err": float(t.item()), "ok": bool(t.item() < 1e-6), "buckets": [k for k, v in trainer._ranges.items() if v]}


DUMP_SAMPLE = 1 << 22  # elements of the parameter and gradient vectors written by --dump-outputs (16 MiB each)


def dump_outputs(out_dir, trainer, loss):
    """What the last timed step produced, as float32 .npy files: its per-direction losses, the pre-clip gradient norm,
    a sample of the updated parameters and of the gradients the step applied, and the BatchNorm running statistics.
    The sample positions are drawn with a fixed seed over all parameters concatenated in name order, so they do not
    depend on the arena layout and two builds can be compared element for element."""
    import numpy as np
    arena, eng = trainer.arena, trainer.engine
    names = sorted(arena.names)
    sizes = torch.tensor([arena.numels[n] for n in names])
    ends = sizes.cumsum(0)
    total = int(ends[-1])
    pos = torch.randint(total, (min(DUMP_SAMPLE, total),), generator=torch.Generator().manual_seed(0)).sort().values
    which = torch.searchsorted(ends, pos, right=True)
    local = pos - (ends - sizes)[which]
    bounds = torch.searchsorted(which, torch.arange(len(names) + 1)).tolist()
    params, grads = [], []
    for i, n in enumerate(names):
        sel = local[bounds[i]:bounds[i + 1]].to(arena.device)
        params.append(arena.p(n).flatten()[sel])
        grads.append(arena.g(n).flatten()[sel])
    bn = [eng.buffers[n].float().flatten() for n in sorted(eng.buffers) if not n.endswith("num_batches_tracked")]
    out = {"loss": loss, "grad_norm": trainer.grad_norm.reshape(1), "params_sample": torch.cat(params),
           "grads_sample": torch.cat(grads), "bn_running_stats": torch.cat(bn)}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------- ours
def main_ours(args, rank, world, local):
    import torch.distributed as dist
    from virtex_b200 import ops
    from virtex_b200.config import Config
    from virtex_b200.factories import PretrainingModelFactory
    from virtex_b200.trainer import Trainer

    dev = torch.device("cuda", local)
    B = args.batch_per_gpu
    cfg = Config(args.config, ["OPTIM.BATCH_SIZE", B * world] + args.config_override)
    torch.manual_seed(cfg.RANDOM_SEED)
    model = PretrainingModelFactory.from_config(cfg).to(dev)
    model.train()
    trainer = Trainer(model, cfg)
    T = cfg.DATA.MAX_CAPTION_LENGTH
    host = [synth_host_batch(B, T, cfg.DATA.VOCAB_SIZE, seed=rank * 100 + i) for i in range(2)]
    dev_batch = {k: v.to(dev) for k, v in host[0].items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()
        return ms

    # ---- warm-up (allocates every workspace buffer), then the device-resident timed region
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()  # started before the warm-up so that it is already sampling when the timed region begins
    for _ in range(max(args.warmup, 3)):
        trainer.step(dev_batch)
    barrier()
    launches0 = ops.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.mark_begin()
    e0.record()
    for _ in range(args.steps):
        loss = trainer.step(dev_batch)
    e1.record()
    barrier()
    clocks.mark_end()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = ops.launch_count - launches0
    clk = clocks.stop() if rank == 0 else None
    loss_val = float(loss.sum().item())
    value = args.steps * B * world / (ms / 1e3)
    if args.dump_outputs and rank == 0:  # before the end-to-end and profiled steps below train the model further
        dump_outputs(args.dump_outputs, trainer, loss)

    # ---- end to end: pinned host batches -> H2D (prefetched on a copy stream) -> step -> D2H loss read, every step
    copy_stream = torch.cuda.Stream(device=dev)
    slots = [{k: torch.empty_like(v, device=dev) for k, v in host[0].items()} for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    loss_host = torch.zeros(2, 2).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())

    def upload(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])
            for k, v in host[i % 2].items():
                slots[i % 2][k].copy_(v, non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_run(n):
        for e in consumed:
            e.record()
        upload(0)
        seen = []
        for i in range(n):
            if i + 1 < n:
                upload(i + 1)
            torch.cuda.current_stream().wait_event(ready[i % 2])
            l = trainer.step(slots[i % 2])
            consumed[i % 2].record()
            loss_host[i % 2].copy_(l, non_blocking=True)
            done = torch.cuda.Event()
            done.record()
            if seen:  # read the previous step's loss on the host (one step of slack keeps the launch queue full)
                ev, slot = seen.pop()
                ev.synchronize()
                _ = float(loss_host[slot].sum())
            seen.append((done, i % 2))
        ev, slot = seen.pop()
        ev.synchronize()
        return float(loss_host[slot].sum())

    e2e_run(2)
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    e2e_run(args.steps)
    t1.record()
    barrier()
    ms_e2e = max_over_ranks(t0.elapsed_time(t1))
    e2e_value = args.steps * B * world / (ms_e2e / 1e3)

    # ---- roofline of the dominant kernel: CUDA events around every tcgen05 GEMM launch of 2 further steps
    roof = None
    if rank == 0:
        ops.start_gemm_profile()
    e0.record()
    for _ in range(2):  # every rank runs the steps (they contain collectives); only rank 0 records events
        trainer.step(dev_batch)
    e1.record()
    if rank == 0:
        prof = ops.stop_gemm_profile()
        prof_ms = e0.elapsed_time(e1) / 2
        if args.dump_gemm_profile:
            os.makedirs(os.path.dirname(os.path.abspath(args.dump_gemm_profile)), exist_ok=True)
            with open(args.dump_gemm_profile, "w") as f:
                json.dump([dict(ms=p[0], flops=p[1], M=p[2], N=p[3], K=p[4], conv_mode=p[5], a_mn=p[6], b_mn=p[7],
                                extra_bytes=p[8])
                           for p in prof[len(prof) // 2:]], f)
        peak_tf, peak_bw, peak_src = measured_peaks()
        half = prof[len(prof) // 2:]  # the launches of the second profiled step
        g_ms = sum(p[0] for p in prof) / 2
        g_fl = sum(p[1] for p in prof) / 2

        def min_bytes(ms, fl, M, N, K, mode, a_mn, b_mn, extra):
            # operands read once + output written once (im2col-free for the implicit convs: the activation is counted
            # once, not once per tap) + what the epilogue reads besides (residual tile, ReLU bit mask)
            if mode in (1, 3, 5):
                return 2 * (M * K // (9 if mode != 5 else 16) + N * K) + 2 * M * N + extra
            if mode in (2, 6):
                return 2 * (K * M + K * N // (9 if mode != 6 else 16)) + 4 * M * N + extra
            if mode == 4:
                return 2 * (K * N + K * 64) + 4 * M * N + extra
            return 2 * (M * K + N * K) + (4 if (a_mn and b_mn) else 2) * M * N + extra

        g_by = sum(min_bytes(*p) for p in half)
        t_min = sum(max(p[1] / (peak_tf * 1e12), min_bytes(*p) / (peak_bw * 1e9)) for p in half) * 1e3  # ms
        # DRAM bytes cannot be counted without ncu: `traffic` is the per-launch average of the committed ncu capture of
        # this same command (profiles/, newest round first); traffic_source says which capture and at which commit
        traffic = traffic_src = None
        tnames = sorted((n for n in os.listdir(os.path.join(ROOT, "profiles")) if n.endswith("_gemm_dram_traffic.json")),
                        reverse=True)  # newest capture first (r02s_ > r02_ > r01_)
        for tname in tnames:
            tpath = os.path.join(ROOT, "profiles", tname)
            if os.path.exists(tpath):
                with open(tpath) as f:
                    tj = json.load(f)
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), f"profiles/{tname} @ {tj.get('commit', 'round-1 kernel')}"
                break
        roof = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 GEMM: all convs + linears)",
                "achieved": round(g_fl / (g_ms * 1e-3) / 1e12, 1), "peak": peak_tf, "unit": "TFLOP/s",
                "frac": round(g_fl / (g_ms * 1e-3) / 1e12 / peak_tf, 4), "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src,
                "launches_per_step": len(prof) // 2, "gemm_ms_per_step": round(g_ms, 3),
                "gemm_share_of_step": round(g_ms / prof_ms, 3),
                "algorithmic_gflop_per_launch": round(g_fl / 1e9 / (len(prof) // 2), 2),
                "algorithmic_bytes_per_launch": int(g_by / (len(prof) // 2)),
                "hbm_view": {"achieved_gbs": round(g_by / (g_ms * 1e-3) / 1e9, 1), "peak_gbs": peak_bw,
                             "frac": round(g_by / (g_ms * 1e-3) / 1e9 / peak_bw, 4)},
                "per_launch_roofline_frac": round(t_min / g_ms, 4),
                "note": "launches of mixed shapes: 'frac' is sum(2MNK)/sum(time) against the bf16 peak; about half of the "
                        "launches (layer1-2 convs, all wgrads) are HBM-bound, so per_launch_roofline_frac = "
                        "sum(max(flops/peak_tf, min_bytes/peak_bw))/sum(time) is the tighter figure; the kernel's time "
                        "includes the BN statistics / BN-backward reductions fused into its epilogues (their y / residual / "
                        "mask reads are counted in min_bytes)"}
    barrier()
    dp = dp_gradient_check(trainer, dev_batch, world) if world > 1 else None
    name = f"{cfg.MODEL.VISUAL.NAME.split('::')[-1]} + {cfg.MODEL.TEXTUAL.NAME}"

    if rank == 0:
        incumbent = None
        if world == 1 and not args.skip_incumbent:
            del trainer, model
            torch.cuda.empty_cache()
            incumbent = run_incumbent(args, cfg)
        cpu_v, cpu_sec, cpu_threads = run_cpu_reference(2, 1, args.cpu_batch) if not args.skip_cpu else (None, None, 0)
        line = {"metric": METRIC, "value": round(value, 1), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"bicaptioning {name} full optimisation step, batch {B} per GPU",
                           "config_file": args.config, "global_batch": B * world, "seq_len": T,
                           "parallelism": f"dp{world}", "dropout": cfg.MODEL.TEXTUAL.DROPOUT,
                           "l2_policy": "per-step working set (>= 150 MB of inputs, GBs of activations) exceeds the 126 MB L2"},
                "loss": round(loss_val, 4), "clocks": clk,
                "e2e": {"value": round(e2e_value, 1), "unit": "pairs/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": 8, "ms_per_step": round(ms_e2e / args.steps, 3),
                        "api": "virtex_b200.trainer.Trainer.step on pinned host batches"},
                "gpu_launches": launches, "roofline": roof,
                "model_tflops": round(value * (roof["algorithmic_gflop_per_launch"] * roof["launches_per_step"] / B) / 1e3, 1),
                "incumbent": incumbent,
                "vs_incumbent": (round(value / incumbent["pairs_s"], 3) if incumbent and "pairs_s" in incumbent else None),
                "dp_check": dp,
                "cpu_baseline": None if cpu_v is None else {
                    "value": round(cpu_v, 3), "unit": "pairs/s", "cores": cpu_threads, "kind": "port",
                    "sample": f"2 full steps at batch {args.cpu_batch} after 1 warm-up (oracle port of the reference, fp32)"}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-per-gpu", type=int, default=256)
    ap.add_argument("--cpu-batch", type=int, default=32)
    ap.add_argument("--config", default="_base_bicaptioning_R_50_L1_H1024.yaml")
    ap.add_argument("--config-override", nargs="*", default=[])
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-incumbent", action="store_true")
    ap.add_argument("--dump-gemm-profile", default="")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        main_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU baseline)")
    from virtex_b200.distributed import init_from_env
    rank, world, local = init_from_env()
    main_ours(args, rank, world, local)


if __name__ == "__main__":
    main()
