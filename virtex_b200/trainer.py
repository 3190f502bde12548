"""`Trainer.step(batch)`: the reference loop body (scripts/pretrain_virtex.py:145-163) on the B200 engine.

    zero_grad -> forward (bf16 compute) -> backward -> [data-parallel gradient all-reduce, overlapped with backward]
    -> global-norm clip -> SGD(momentum, per-parameter lr / weight decay) -> Lookahead every k steps -> LR schedule

The optimiser tail runs as fused kernels over the flat arenas (virtex_b200/csrc/optim.cu) with the arithmetic of
torch.optim.SGD + virtex/optim/lookahead.py + virtex/optim/lr_scheduler.py; bf16 needs no GradScaler.
Gradient all-reduce: NCCL over NVLink on a side stream, one bucket per completed gradient range in backward order
(backward-direction decoder; forward-direction decoder + shared embedding / projection; layer4; layer3; layer2; the
rest), SUM on the wire and the 1/world_size folded into the clip coefficient,
so averaged gradients equal the mean of per-rank gradients like DistributedDataParallel's.
"""
import struct
from typing import Dict, Optional

import torch
import torch.distributed as dist

from . import ops
from .config import Config
from .factories import param_group_hparams
from .ops import _stream, call
from .optim import lr_multiplier_fn

_CHUNK = 65536
# completion order of gradient ranges in backward: the backward-direction decoder finishes first (its gradients are the
# last contiguous range of the arena), then everything shared / forward-direction of the head, then the backbone layers
BUCKET_ORDER = ("head_b", "head", "layer4", "layer3", "layer2", "rest")


def bucket_ranges(names, offsets, numels) -> Dict[str, Optional[tuple]]:
    """Contiguous [begin, end) element ranges of the flat gradient arena per all-reduce bucket (pure host logic)."""

    def rng(pred):
        sel = [n for n in names if pred(n)]
        if not sel:
            return None
        return offsets[sel[0]], offsets[sel[-1]] + numels[sel[-1]]

    out = {"head_b": rng(lambda n: n.startswith("backward_textual.")),
           "head": rng(lambda n: not n.startswith("visual.") and not n.startswith("backward_textual."))}
    for l in ("layer4", "layer3", "layer2"):
        out[l] = rng(lambda n, l=l: n.startswith(f"visual.cnn.{l}."))
    out["rest"] = rng(lambda n: n.startswith("visual.cnn.") and (".layer1." in n or ".layer" not in n))
    return out


def optimizer_segments(names, offsets, numels, hparams, chunk=_CHUNK):
    """[(begin, end, lr, wd)] chunks of <= `chunk` elements; hparams(name) -> (lr, wd) or None for frozen tensors."""
    segs = []
    for name in names:
        hp = hparams(name)
        if hp is None:
            continue
        b, e = offsets[name], offsets[name] + numels[name]
        for c in range(b, e, chunk):
            segs.append((c, min(e, c + chunk), hp[0], hp[1]))
    return segs


class Trainer:
    def __init__(self, model, config: Config, process_group=None):
        if config.OPTIM.OPTIMIZER_NAME != "sgd":
            raise NotImplementedError("the fused optimiser tail implements the reference's SGD recipe")
        self.model = model
        self.config = config
        self.engine = eng = model.engine
        self.arena = arena = eng.arena
        dev = eng.device
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.group = process_group
        O = config.OPTIM
        self.max_norm = float(O.CLIP_GRAD_NORM)
        self.momentum = float(O.SGD_MOMENTUM)
        self.use_lookahead = bool(O.LOOKAHEAD.USE)
        self.la_alpha = float(O.LOOKAHEAD.ALPHA)
        self.la_k = int(O.LOOKAHEAD.STEPS)
        self.lr_fn = lr_multiplier_fn(O.LR_DECAY_NAME, O.NUM_ITERATIONS, O.WARMUP_STEPS, O.LR_STEPS, O.LR_GAMMA)
        # ---- per-parameter (lr, wd) by NAME, split into <= 64 Ki-element chunks for load balance
        segs = optimizer_segments(
            arena.names, arena.offsets, arena.numels,
            lambda n: param_group_hparams(config, n) if arena._param_objs[n].requires_grad else None)
        blob = b"".join(struct.pack("<qqff", *s) for s in segs)
        self.nseg = len(segs)
        self.segs = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)
        self.mom = torch.zeros_like(arena.params)
        self.slow = arena.params.clone() if self.use_lookahead else None
        self.sumsq = torch.zeros(1, dtype=torch.float32, device=dev)
        self.ctl = torch.zeros(2, dtype=torch.float32, device=dev)
        self.hyper = torch.zeros(4, dtype=torch.float32, device=dev)
        self._hyper_ring = [torch.zeros(4, dtype=torch.float32).pin_memory() for _ in range(16)]
        self.iteration = 0
        self._k_counter = 0
        self.momentum_ready = False  # torch.optim.SGD: the first step with a gradient initialises the buffer to it
        # dropout seed of step i = base + i (restored from the iteration on resume); ranks get decorrelated streams
        rank = dist.get_rank(process_group) if dist.is_initialized() else 0
        self._seed_base = (int(config.RANDOM_SEED) << 24) + rank * 1000003
        eng.seed.fill_(self._seed_base)
        self.comm_stream = torch.cuda.Stream(device=dev) if self.world > 1 else None
        # (The GEMM's dynamic tile schedule -- ops.set_dynamic_gemm_schedule -- was built for the case that NCCL's CTAs
        # hold SMs while a bucket is in flight; measured on 2 x B200 it is 0.15 ms/step SLOWER than the static schedule
        # (23.81 vs 23.66 ms, profiles/r02n_*), so the trainer leaves the static schedule on.)
        self._pending = []
        self._ranges = self._bucket_ranges()
        if self.world > 1:  # DDP constructor semantics: rank 0's parameters and buffers everywhere
            dist.broadcast(arena.params, src=0, group=self.group)
            for b in eng.buffers.values():
                dist.broadcast(b, src=0, group=self.group)
            if self.slow is not None:
                self.slow.copy_(arena.params)
        eng.prepare_weights()

    # ------------------------------------------------------------------------------------------------- DP buckets
    def _bucket_ranges(self) -> Dict[str, tuple]:
        a = self.arena
        return bucket_ranges(a.names, a.offsets, a.numels)

    def _on_bucket(self, tag):
        r = self._ranges.get(tag)
        if r is None:
            return
        self.comm_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.comm_stream):
            w = dist.all_reduce(self.arena.grads[r[0]:r[1]], op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        self._pending.append(w)

    # ------------------------------------------------------------------------------------------------------- step
    def step(self, batch) -> torch.Tensor:
        """One optimisation step on a device-resident batch dict; returns the per-direction losses (device, [2]).  A
        classification model takes {"image", "labels"} and returns [loss, 0]."""
        eng = self.engine
        if self.model.engine is not eng:
            raise RuntimeError("the model rebuilt its engine (model.to() / .cuda() after Trainer construction): "
                               "create a new Trainer, this one would update a stale parameter arena")
        eng.seed.add_(1)
        m = self.model
        if eng.classification:
            loss = eng.forward(batch["image"], None, None, None, training=True, with_grad=True, labels=batch["labels"])
        else:
            loss = eng.forward(batch["image"], batch["caption_tokens"],
                               batch["noitpac_tokens"] if m.caption_backward else batch["caption_tokens"],
                               batch["caption_lengths"], training=True, with_grad=True)
        eng.backward(zero_grads=True, bucket_cb=self._on_bucket if self.world > 1 else None)
        for w in self._pending:
            w.wait()
        self._pending.clear()
        self.optimizer_step()
        return loss

    def optimizer_step(self):
        eng, arena = self.engine, self.arena
        s = _stream()
        self.sumsq.zero_()
        call("vtx_sumsq", arena.grads.data_ptr(), arena.total, self.sumsq.data_ptr(), s)
        call("vtx_clip_coef", self.sumsq.data_ptr(), self.world, self.max_norm, self.ctl.data_ptr(), s)
        self._k_counter += 1
        do_la = self.use_lookahead and self._k_counter >= self.la_k
        if do_la:
            self._k_counter = 0
        h = self._hyper_ring[self.iteration % len(self._hyper_ring)]
        h[0] = self.lr_fn(self.iteration)  # the optimiser step of iteration i uses lambda(i - 1 + 1 - 1) = lambda(i)
        h[1] = 0.0 if self.momentum_ready else 1.0
        h[2] = 1.0 if do_la else 0.0
        self.hyper.copy_(h, non_blocking=True)
        call("vtx_sgd_step", arena.params.data_ptr(), arena.grads.data_ptr(), self.mom.data_ptr(),
             0 if self.slow is None else self.slow.data_ptr(), arena.mirror.data_ptr(), self.segs.data_ptr(), self.nseg,
             self.ctl.data_ptr(), self.hyper.data_ptr(), self.momentum, self.la_alpha, s)
        eng.prepare_weights(mirror=False)  # the step kernel refreshed the bf16 mirror; re-pack the k>1 conv weights
        self.momentum_ready = True
        self.iteration += 1

    def sync_dropout_seed(self):
        """Dropout stream position as a function of the iteration (called after a checkpoint load)."""
        self.engine.seed.fill_(self._seed_base + self.iteration)

    def broadcast_buffers(self):
        """BN running statistics of rank 0 everywhere -- what DistributedDataParallel(broadcast_buffers=True) does at
        every forward; here on demand (before an evaluation or a checkpoint written by a non-master rank), since
        training itself never reads them."""
        if self.world > 1:
            for b in self.engine.buffers.values():
                dist.broadcast(b, src=0, group=self.group)

    # ------------------------------------------------------------------------------------------- checkpoint views
    def reset_lookahead(self):
        """Slow weights restart from the current parameters (what the reference's Lookahead does after a load)."""
        self._k_counter = 0
        if self.slow is not None:
            self.slow.copy_(self.arena.params)

    @property
    def optimizer(self):
        """`torch.optim.SGD`-layout state view for checkpoint interchange (virtex_b200/checkpointing.py)."""
        from .checkpointing import FusedOptimizerState
        return FusedOptimizerState(self)

    @property
    def scheduler(self):
        from .checkpointing import FusedSchedulerState
        return FusedSchedulerState(self)

    @property
    def grad_norm(self) -> torch.Tensor:
        return self.ctl[1]
