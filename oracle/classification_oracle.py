"""CPU oracle of the classification pretext models -- TEST INFRASTRUCTURE, NOT PRODUCT.

A restatement, over basic torch CPU ops, of what the reference's `TokenClassificationModel` /
`MultiLabelClassificationModel` compute (virtex/models/classification.py:12-164 with the `LinearTextualHead` of
virtex/modules/textual_heads.py:46-95), written from these rules:

  * features = the ResNet backbone of `virtex_oracle.backbone_forward`, pooled = their mean over h * w,
    logits = pooled . W^T + b;
  * the label set of image b = the distinct ids of labels[b] inside [0, V) minus `ignore`;
  * loss = sum_b -mean(log_softmax(logits)[b, set_b]) / B -- an empty set gives NaN (the mean of nothing) and,
    under autograd, no gradient into its row;
  * predictions = the 10 best ids of each row: NaN above every number, then larger value, then lower index.

Gradients come from CPU autograd.  `oracle/make_classification_golden.py` pins this module against the live reference;
`tests/test_classification_cpu.py` re-checks it against the committed goldens.
"""
from collections import OrderedDict
from typing import Dict, Iterable, List, Optional

import numpy as np
import torch

from oracle import virtex_oracle as O

TOKEN_IGNORE = (0, 1, 2, 3)       # [UNK], [SOS], [EOS], [MASK] (virtex/factories.py:446-455)
MULTILABEL_IGNORE = (0,)          # COCO background
FEATURES = 2048


def _backbone_spec() -> O.Spec:
    return O.Spec(hidden=128, layers=1, heads=2, ffn=256, vocab=16, caption_backward=False)


def synth_state(vocab: int, seed: int = 0, bn3_gain: float = 0.25) -> "OrderedDict[str, torch.Tensor]":
    """Backbone weights of `virtex_oracle.synth_state(seed)` (the backbone part does not depend on the head) plus
    `textual.output.{weight,bias}` drawn like torch's default nn.Linear init, U(-1/sqrt(2048), 1/sqrt(2048))."""
    full = O.synth_state(_backbone_spec(), seed, bn3_gain=bn3_gain)
    state = OrderedDict((k, v) for k, v in full.items() if k.startswith("visual."))
    g = torch.Generator().manual_seed(50000 + seed)
    bound = 1.0 / FEATURES ** 0.5
    state["textual.output.weight"] = (torch.rand(vocab, FEATURES, generator=g) * 2 - 1) * bound
    state["textual.output.bias"] = (torch.rand(vocab, generator=g) * 2 - 1) * bound
    return state


def synth_label_batch(kind: str, batch_size: int, seed: int = 0, vocab: int = 10000, image_size: int = 224,
                      empty_rows: Iterable[int] = ()) -> Dict[str, torch.Tensor]:
    """kind "token": the labels are ragged captions ([SOS] ... [EOS], 0-padded) with an [UNK], a [MASK] and repeated
    tokens inside; kind "multilabel": 12 category ids in [1, vocab) per image with duplicates, 0-padded.  Rows in
    `empty_rows` hold only ignored ids.  `caption_tokens` repeats the labels (what `log_predictions` prints)."""
    g = torch.Generator().manual_seed(7000 + seed)
    image = torch.randn(batch_size, 3, image_size, image_size, generator=g)
    if kind == "token":
        L = 30
        labels = torch.zeros(batch_size, L, dtype=torch.int64)
        for b in range(batch_size):
            n = L if b == 0 else int(torch.randint(8, L + 1, (1,), generator=g))
            row = torch.randint(4, vocab, (n,), generator=g)
            row[0], row[-1] = 1, 2
            row[3], row[5] = 0, 3           # [UNK], [MASK]
            row[6] = row[7] = row[4]        # a token three times
            labels[b, :n] = row
    elif kind == "multilabel":
        L = 12
        labels = torch.zeros(batch_size, L, dtype=torch.int64)
        for b in range(batch_size):
            n = int(torch.randint(3, L + 1, (1,), generator=g))
            row = torch.randint(1, vocab, (n,), generator=g)
            row[1] = row[0]                 # one category with two instances
            labels[b, :n] = row
    else:
        raise ValueError(kind)
    for b in empty_rows:
        labels[b] = 0
        if kind == "token":
            labels[b, :4] = torch.tensor([1, 0, 3, 2])
    return {"image": image, "labels": labels, "caption_tokens": labels.clone()}


def label_sets(labels: torch.Tensor, vocab: int, ignore: Iterable[int]) -> List[List[int]]:
    """Sorted label set of every row: distinct ids inside [0, vocab) that are not ignored."""
    ign = set(int(i) for i in ignore)
    return [sorted({int(v) for v in row.tolist() if 0 <= v < vocab and v not in ign}) for row in labels]


def khot_loss(logits: torch.Tensor, labels: torch.Tensor, ignore: Iterable[int]) -> torch.Tensor:
    """sum_b -mean(log_softmax(logits)[b, set_b]) / B (NaN when a set is empty, with a zero gradient row)."""
    logp = torch.log_softmax(logits, dim=1)
    B, V = logits.shape
    total = logits.new_zeros(())
    for b, s in enumerate(label_sets(labels, V, ignore)):
        total = total - logp[b, torch.tensor(s, dtype=torch.int64)].mean()
    return total / B


def topk(x: torch.Tensor, k: int = 10) -> torch.Tensor:
    """Indices of the k best entries of each row, best first: NaN above every number, then larger, then lower index."""
    a = x.detach().double().numpy()
    nan = np.isnan(a)
    val = np.where(nan, 0.0, a)
    idx = np.broadcast_to(np.arange(a.shape[1]), a.shape)
    out = [np.lexsort((idx[r], -val[r], ~nan[r]))[:k] for r in range(a.shape[0])]
    return torch.from_numpy(np.stack(out).astype(np.int64)) if out else torch.zeros(0, k, dtype=torch.int64)


def forward(P, batch, ignore, training=True, new_buffers=None, emulate_bf16=False):
    """`emulate_bf16` rounds where the CUDA path materialises bf16 tensors (backbone activations, the pooled features,
    the GEMM weights), as `virtex_oracle.backbone_forward` does for the backbone."""
    rb = O._rb if emulate_bf16 else (lambda t: t)
    vf = O.backbone_forward(P, batch["image"], _backbone_spec(), training, new_buffers, emulate_bf16=emulate_bf16)
    pooled = rb(vf.mean(dim=(2, 3)))
    logits = pooled @ rb(P["textual.output.weight"]).t() + P["textual.output.bias"]
    loss = khot_loss(logits, batch["labels"], ignore)
    out = {"loss": loss, "loss_components": {"classification": loss.detach().clone()}, "logits": logits,
           "pooled": pooled}
    if not training:
        out["predictions"] = topk(logits, 10)
    return out


def loss_and_grads(state, batch, ignore, dtype=torch.float32, training=True, emulate_bf16=False):
    """One forward (+ backward when training).  Returns (output dict, grads by name, new BN buffers)."""
    P = {k: (v.clone().to(dtype).requires_grad_(training) if not O.is_buffer(k)
             else (v.clone().to(dtype) if v.is_floating_point() else v.clone())) for k, v in state.items()}
    b = dict(batch)
    b["image"] = batch["image"].to(dtype)
    new_buffers: Dict[str, torch.Tensor] = {}
    with torch.set_grad_enabled(training):
        out = forward(P, b, ignore, training=training, new_buffers=new_buffers, emulate_bf16=emulate_bf16)
    grads = {}
    if training:
        out["loss"].backward()
        grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in P.items() if not O.is_buffer(k)}
    out = {k: (v.detach() if torch.is_tensor(v) else v) for k, v in out.items()}
    return out, grads, new_buffers


class OracleTrainer:
    """Reference step sequence (scripts/pretrain_virtex.py:145-163) on the classification model, fp32 CPU: clip to
    the global norm, SGD with momentum and per-name (lr, weight decay), LR schedule, Lookahead."""

    def __init__(self, state, ignore, cfg: Optional[O.OptimCfg] = None):
        self.cfg = cfg or O.OptimCfg()
        self.ignore = tuple(ignore)
        self.state = OrderedDict((k, v.clone()) for k, v in state.items())
        self.momentum_buf: Dict[str, torch.Tensor] = {}
        self.slow = {k: v.clone() for k, v in self.state.items() if not O.is_buffer(k)}
        self.iteration = 0
        self.k_counter = 0

    def step(self, batch) -> Dict[str, torch.Tensor]:
        cfg = self.cfg
        out, grads, new_buffers = loss_and_grads(self.state, batch, self.ignore)
        self.state.update(new_buffers)
        total = torch.sqrt(sum((g.double() ** 2).sum() for g in grads.values())).float()
        clip = min(1.0, cfg.clip_grad_norm / (float(total) + 1e-6))
        mult = O.lr_multiplier(self.iteration, cfg)
        for name, g in grads.items():
            lr, wd = O.param_hparams(name, cfg)
            p = self.state[name]
            g = g * clip + wd * p
            if name not in self.momentum_buf:
                self.momentum_buf[name] = g.clone()
            else:
                self.momentum_buf[name].mul_(cfg.momentum).add_(g)
            p.add_(self.momentum_buf[name], alpha=-lr * mult)
        if cfg.lookahead:
            self.k_counter += 1
            if self.k_counter >= cfg.lookahead_steps:
                self.k_counter = 0
                for name, slow in self.slow.items():
                    slow.add_(self.state[name] - slow, alpha=cfg.lookahead_alpha)
                    self.state[name].copy_(slow)
        self.iteration += 1
        out["grad_norm"] = total
        return out
