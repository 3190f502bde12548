"""CPU oracle of beam-search captioning -- TEST INFRASTRUCTURE, NOT PRODUCT.

A plain restatement, on top of `virtex_oracle.head_forward` / `backbone_forward`, of what the reference runs for
`model.eval(); model({"image": ...})["predictions"]` (virtex/models/captioning.py:144-213 with
virtex/utils/beam_search.py).  The rules, in the order the search applies them:

  1. visual features in the backbone's eval BN mode; every image starts from [SOS].
  2. step 1 runs the head on [SOS] (B rows) and keeps the top `beam` tokens of log_softmax, no penalty.
     beam == 1 and every first token EOS: return the (B, 1, 1) first tokens at once (with a RuntimeWarning).
  3. steps 2... run the head on each beam's predictions so far WITHOUT [SOS] (positions 0..t-1, caption length t) and
     use the last position's logits.
  4. per row: log_softmax, then the row's last token gets exactly -10000; a row whose last token is EOS gets 0 at EOS
     and -inf elsewhere; top per_node plus the beam's running score; per image: top beam of the beam * per_node
     candidates, each continuing its parent's history.
  5. stop before a step when every beam's last token is EOS; L = steps taken.
  6. order: NaN above every number, then larger, then lower token id (row) / lower (beam, rank) candidate (image).

`beam_search` also reports, per step, the selection margins: for every image ("image") the smallest gap between
consecutive candidates up to the first dropped one (the order of the kept ones is the beam order, and beam 0 is the
returned caption), and for every row ("row", inf for an ended one) the gap between its last kept and first dropped
token.  Where every margin exceeds the numerical error of
an implementation, its selections are determined by the math alone.
"""
from __future__ import annotations

import warnings
from typing import Callable, Dict, List

import torch

from oracle import virtex_oracle as O

EMPTY_WARNING = "Empty captions predicted"
INF_WARNING = "Infinite log probs encountered"


def rank(x: torch.Tensor) -> torch.Tensor:
    """Indices that order the last dim by rule 6 (NaN first, then descending value, then ascending index)."""
    nan = torch.isnan(x)
    v = torch.where(nan, torch.full_like(x, float("inf")), x)
    o1 = torch.sort(v, dim=-1, descending=True, stable=True).indices
    o2 = torch.sort(nan.gather(-1, o1).to(torch.int8), dim=-1, descending=True, stable=True).indices
    return o1.gather(-1, o2)


def log_softmax_f32(x: torch.Tensor) -> torch.Tensor:
    """(x - max) - log(sum exp(x - max)): the formula the CUDA beam step evaluates, in the input's dtype."""
    m = x.max(dim=-1, keepdim=True).values
    return (x - m) - torch.log(torch.exp(x - m).sum(dim=-1, keepdim=True))


def _gap(sorted_vals: torch.Tensor, k: int, first: int) -> torch.Tensor:
    """Smallest gap between consecutive entries j-1, j (first <= j <= k) of rows sorted by rule 6; a pair of -infs
    counts as inf (their order is the index rule, exactly), as does a missing entry k."""
    n = min(k, sorted_vals.shape[-1] - 1)
    if n < first:
        return torch.full(sorted_vals.shape[:-1], float("inf"), dtype=sorted_vals.dtype)
    a, b = sorted_vals[..., first - 1:n], sorted_vals[..., first:n + 1]
    g = a - b
    g = torch.where((a == float("-inf")) & (b == float("-inf")), torch.full_like(g, float("inf")), g)
    return g.min(dim=-1).values


def penalise(lp: torch.Tensor, last: torch.Tensor, eos: int) -> torch.Tensor:
    """Rule 4 before the top-k: the row's last token gets -10000, a row ended by EOS gets 0 at EOS, -inf elsewhere."""
    lp = lp.clone()
    lp[torch.arange(lp.shape[0], device=lp.device), last] = -10000.0
    ended = last == eos
    lp[ended] = float("-inf")
    lp[ended, eos] = 0.0
    return lp


def select(lp: torch.Tensor, last, scores, eos: int, beam: int, per_node: int):
    """One selection (rule 4) on log-probabilities lp [B * beam_in, V]; last None = step 1 (no penalty / forcing,
    running score 0, beam_in = 1, per_node = beam).  Returns tokens, parent rows, scores [B, beam] and the margins."""
    rows, V = lp.shape
    if last is not None:
        lp = penalise(lp, last, eos)
        live = last != eos
    else:
        live = torch.ones(rows, dtype=torch.bool, device=lp.device)
        scores = torch.zeros(rows, dtype=lp.dtype, device=lp.device)
    o = rank(lp)
    top_idx = o[:, :per_node]
    top_v = lp.gather(1, top_idx)
    row_gap = _gap(lp.gather(1, o[:, :per_node + 1]), per_node, per_node)
    row_gap = torch.where(live, row_gap, torch.full_like(row_gap, float("inf")))  # an ended row's choice is fixed
    B = rows // beam if last is not None else rows
    beam_in = rows // B
    cand = (top_v + scores.reshape(-1, 1)).reshape(B, beam_in * per_node)
    co = rank(cand)
    sel = co[:, :beam]
    img_gap = _gap(cand.gather(1, co), beam, 1)
    tokens = top_idx.reshape(B, -1).gather(1, sel)
    parents = torch.arange(B, device=lp.device)[:, None] * beam_in + sel // per_node
    return tokens, parents, cand.gather(1, sel), {"row": row_gap, "image": img_gap}


def beam_search(start: torch.Tensor, step: Callable[[torch.Tensor], torch.Tensor], eos: int, max_steps: int = 50,
                beam: int = 5, per_node: int = 2, only_return_best: bool = True, log_softmax=None):
    """The reference's AutoRegressiveBeamSearch.search under rules 2-6 -> (predictions, scores, margins), margins a
    list with one {"row", "image"} dict per step."""
    log_softmax = log_softmax or (lambda x: torch.log_softmax(x, dim=-1))
    per_node = per_node or beam
    B = start.shape[0]
    tokens, _, scores, m = select(log_softmax(step(start)), None, None, eos, beam, beam)
    margins: List[Dict[str, torch.Tensor]] = [m]
    if beam == 1 and bool((tokens == eos).all()):
        warnings.warn(EMPTY_WARNING, RuntimeWarning)
        return tokens.unsqueeze(-1), scores, margins
    preds = tokens.unsqueeze(-1)  # [B, beam, 1]
    for _ in range(max_steps - 1):
        last = preds[:, :, -1].reshape(-1)
        if bool((last == eos).all()):
            break
        L = preds.shape[-1]
        lp = log_softmax(step(preds.reshape(B * beam, L)))
        tokens, parents, scores, m = select(lp, last, scores.reshape(-1), eos, beam, per_node)
        margins.append(m)
        preds = torch.cat([preds.reshape(B * beam, L)[parents.reshape(-1)].reshape(B, beam, L),
                           tokens.unsqueeze(-1)], dim=-1)
    if not bool(torch.isfinite(scores).all()):
        warnings.warn(INF_WARNING, RuntimeWarning)
    if only_return_best:
        return preds[:, 0, :], scores[:, 0], margins
    return preds, scores, margins


def decode(P, image: torch.Tensor, spec: O.Spec, sos: int = 1, eos: int = 2, beam: int = 5, per_node: int = 2,
           max_steps: int = 30, only_return_best: bool = True):
    """`model.eval(); model({"image": image})["predictions"]` of the forward direction -> (predictions, scores,
    margins); the dtype of P and image sets the arithmetic."""
    vf = O.backbone_forward(P, image, spec, training=False)
    B = image.shape[0]

    def step(partial):
        if partial.dim() == 1:
            partial = partial.unsqueeze(1)
        rows, T = partial.shape
        v = vf.repeat_interleave(rows // B, dim=0)
        return O.head_forward(P, v, partial, torch.full((rows,), T, dtype=torch.int64), spec)[:, -1]

    start = torch.full((B,), sos, dtype=torch.int64)
    return beam_search(start, step, eos, max_steps, beam, per_node, only_return_best)


def min_margin(margins) -> float:
    vals = [t.min().item() for m in margins for t in (m["row"], m["image"]) if t.numel()]
    return min(vals) if vals else float("inf")
