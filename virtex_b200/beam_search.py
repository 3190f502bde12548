"""Beam search for autoregressive captioning: drop-in for virtex/utils/beam_search.py (`AutoRegressiveBeamSearch`).

Same constructor, attributes and `search(start_predictions, step, only_return_best=True)` contract as the reference,
with any step callable that returns CUDA logits.  The selection of every step (log_softmax, the repetition penalty,
forcing of ended beams, the per-row and per-image top-k) is one `vtx_beam_step` launch and the history follows the
selected parents through `vtx_beam_reorder` (csrc/decode.cu); the only host synchronisation per step is the read of the
"every beam ended" flag that stops the loop early, as the reference's `.all()` check does.

Ties, which torch leaves unspecified, are broken towards the lower token id within a row and the lower
(beam, rank) candidate within an image; NaN ranks above every number (include/virtex_b200.h, vtx_beam_step).
`CaptioningModel` hands an `AutoRegressiveBeamSearch` decoder to `Engine.decode`, which runs the same selection over
a KV-cached decoder step instead of calling a step function.
"""
import warnings
from typing import Callable, Tuple

import torch

from .ops import call, _p, _stream

_EMPTY_WARNING = ("Empty captions predicted. You may want to increase beam size or ensure your step function is "
                  "working properly.")
_INF_WARNING = ("Infinite log probs encountered. Some final captions may not make sense. This can happen when the "
                "beam size is larger than the number of valid (non-zero probability) transitions that the step "
                "function produces.")


class BeamState:
    """Device state of one beam search: ping-pong history [rows, max_steps] int64 (and, for a KV-cached decoder, the
    cache index [rows, max_steps] int32 of vtx_decode_attn), running scores, last tokens and the ended flag."""

    def __init__(self, device, batch_size, beam_size, per_node, eos, max_steps, with_table=False, ws=None):
        self.B, self.beam, self.per_node, self.eos, self.max_steps = batch_size, beam_size, per_node, eos, max_steps
        rows = batch_size * beam_size
        self.rows = rows
        self.ldh = max_steps + 1
        get = (lambda name, shape, dtype: ws.get("beam." + name, shape, dtype)) if ws is not None else \
            (lambda name, shape, dtype: torch.empty(shape, dtype=dtype, device=device))
        self.hist = [get("hist0", (rows, self.ldh), torch.int64), get("hist1", (rows, self.ldh), torch.int64)]
        self.scores = [get("sc0", (rows,), torch.float32), get("sc1", (rows,), torch.float32)]
        self.tokens = [get("tok0", (rows,), torch.int64), get("tok1", (rows,), torch.int64)]
        self.parents = get("par", (rows,), torch.int64)
        self.ended = get("ended", (1,), torch.int32)
        self.table = [get("tab0", (rows, self.ldh), torch.int32), get("tab1", (rows, self.ldh), torch.int32)] \
            if with_table else None
        self.cur = 0
        self.length = 0

    # the newest selection (valid after first()/step())
    @property
    def last_tokens(self):
        return self.tokens[self.cur]

    @property
    def history(self):
        """[rows, L] int64 view of the current histories."""
        return self.hist[self.cur][:, :self.length]

    @property
    def cache_table(self):
        return self.table[self.cur] if self.table is not None else None

    def _select(self, logits, images, beam_in, per_node, last, scores_in):
        V = logits.shape[1]
        nxt = 1 - self.cur
        call("vtx_beam_step", logits.data_ptr(), logits.stride(0), V, images, beam_in, per_node, self.beam, self.eos,
             _p(last), _p(scores_in), self.tokens[nxt].data_ptr(), self.parents.data_ptr(),
             self.scores[nxt].data_ptr(), self.ended.data_ptr(), _stream())
        n_tab = self.length if (self.table is not None and self.length >= 1) else 0
        call("vtx_beam_reorder", self.parents.data_ptr(), self.tokens[nxt].data_ptr(),
             self.hist[self.cur].data_ptr() if self.length else 0, self.hist[nxt].data_ptr(), self.ldh, self.length,
             self.table[self.cur].data_ptr() if n_tab > 1 else 0,
             self.table[nxt].data_ptr() if n_tab else 0, self.ldh, max(n_tab, 1), self.rows, _stream())
        self.cur = nxt
        self.length += 1

    def first(self, logits):
        """Step 1: logits [B, V] of the start tokens -> top `beam` tokens per image."""
        self._select(logits, self.B, 1, self.beam, None, None)

    def step(self, logits):
        """Steps 2...: logits [B * beam, V] of every beam's newest position."""
        self._select(logits, self.B, self.beam, self.per_node, self.tokens[self.cur], self.scores[self.cur])

    def all_ended(self) -> bool:
        return bool(self.ended.item())  # the one host synchronisation of a step

    def result(self, only_return_best: bool):
        preds = self.history.reshape(self.B, self.beam, self.length).clone()
        scores = self.scores[self.cur].view(self.B, self.beam).clone()
        if not bool(torch.isfinite(scores).all()):
            warnings.warn(_INF_WARNING, RuntimeWarning)
        if only_return_best:
            return preds[:, 0, :], scores[:, 0]
        return preds, scores

    def empty_result(self):
        """beam_size == 1 and every first token is EOS: the reference returns right after the first step."""
        warnings.warn(_EMPTY_WARNING, RuntimeWarning)
        return (self.tokens[self.cur].view(self.B, 1, 1).clone(), self.scores[self.cur].view(self.B, 1).clone())


def _as_logits(logits: torch.Tensor, rows: int) -> torch.Tensor:
    if not isinstance(logits, torch.Tensor) or logits.device.type != "cuda":
        raise RuntimeError("the beam-search step function must return CUDA logits (virtex_b200 has no CPU path)")
    if logits.dim() != 2 or logits.shape[0] != rows:
        raise ValueError(f"step returned logits of shape {tuple(logits.shape)}, expected ({rows}, vocab_size)")
    if logits.dtype != torch.float32 or logits.stride(1) != 1 or logits.stride(0) % 4:
        logits = logits.float().contiguous()
    return logits


class AutoRegressiveBeamSearch:
    """Beam search over the most likely captions (virtex/utils/beam_search.py).

    Args: eos_index: the [EOS] token; max_steps: most decoding steps; beam_size: beams kept per image;
    per_node_beam_size: candidates taken from each beam per step (default 2; 0 / None means beam_size)."""

    def __init__(self, eos_index: int, max_steps: int = 50, beam_size: int = 5, per_node_beam_size: int = 2) -> None:
        self._eos_index = eos_index
        self.max_steps = max_steps
        self.beam_size = beam_size
        self.per_node_beam_size = per_node_beam_size or beam_size

    def search(self, start_predictions: torch.Tensor, step: Callable[..., torch.Tensor],
               only_return_best: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
        """start_predictions (B,) -> (predictions (B, L) or (B, beam, L) int64, logprobs (B,) or (B, beam)).
        `step(partial_captions)` gets (B,) start tokens first, then (B * beam, t) predictions so far (no start token),
        and returns (rows, vocab) logits of the next token."""
        B = start_predictions.shape[0]
        st = BeamState(start_predictions.device, B, self.beam_size, self.per_node_beam_size, self._eos_index,
                       self.max_steps)
        st.first(_as_logits(step(start_predictions), B))
        if self.beam_size == 1 and st.all_ended():
            return st.empty_result()
        for _ in range(self.max_steps - 1):
            if st.all_ended():
                break
            st.step(_as_logits(step(st.history.contiguous()), st.rows))
        return st.result(only_return_best)
