"""`CaptioningModel` family and the classification pretext models: drop-ins for virtex/models/captioning.py:12-283,
virtex/models/masked_lm.py:11-86 and virtex/models/classification.py:12-164 on the B200 engine.

Same constructor arguments, attribute names, weight sharing between the two directions
(captioning.py:57-63) and the same `forward(batch) -> {"loss", "loss_components", ["predictions"]}` contract.
`output["loss"]` carries a grad_fn: `loss.backward()` runs the engine's hand-written backward and delivers gradients
for every parameter (so torch optimisers, GradScaler-free AMP loops and DistributedDataParallel hooks keep working).
The throughput path (`virtex_b200.trainer.Trainer`) drives the same engine without autograd in between.
"""
import copy
import functools
from typing import Any, Dict, List

import torch
from torch import nn

from .beam_search import AutoRegressiveBeamSearch
from .engine import Engine
from .modules import LinearTextualHead, TextualHead, VisualBackbone


class _StepFunction(torch.autograd.Function):
    """Whole-model forward/backward as one autograd node; the kernels are scheduled by `Engine`."""

    @staticmethod
    def forward(ctx, model, image, tokens, noitpac, lengths, labels, *params):
        eng = model.engine
        eng.seed.add_(1)  # fresh dropout masks every training forward (nn.Dropout draws from an advancing RNG stream)
        loss = eng.forward(image, tokens, noitpac, lengths, training=model.training, with_grad=True, labels=labels)
        ctx.model = model
        ctx.generation = eng.generation
        ctx.n_params = len(params)
        out = loss.clone()
        return out[0], out[1]

    @staticmethod
    def backward(ctx, g_fwd, g_bwd):
        model = ctx.model
        eng = model.engine
        if eng.generation != ctx.generation:
            raise RuntimeError(
                "the engine ran another forward since this loss was computed (a validation forward, or a second "
                "micro-batch): its single activation tape was overwritten; call backward() before the next forward")
        # d(loss_f + loss_b): both components enter the total with weight 1 (captioning.py:133).  A common factor (a loss
        # scaler) is applied to every gradient; DIFFERENT weights per direction are not representable after the fused
        # cross-entropy has written dlogits, so they are rejected instead of being silently ignored.
        if g_bwd is not g_fwd and getattr(model, "caption_backward", False) and not torch.equal(g_fwd, g_bwd):
            raise NotImplementedError("the two captioning directions must enter the loss with the same weight")
        eng.backward(zero_grads=True)
        arena = eng.arena
        scaled = arena.grads * g_fwd  # ONE fused scale over the flat arena; parameter gradients are views of the result
        by_id = model._engine_param_names
        grads = []
        for p in model._engine_params:
            name = by_id.get(id(p))
            if name is None or not p.requires_grad:
                grads.append(None)
            else:
                grads.append(arena.view(scaled, name))
        return (None, None, None, None, None, None, *grads)


class _EngineModel(nn.Module):
    """Engine plumbing shared by every model family: the lazily (re)built `Engine` that adopts the parameters, and the
    hooks that invalidate it (`_apply`: moved / cast parameters) or its bf16 weight copies (`load_state_dict`)."""

    def _new_engine(self) -> Engine:
        raise NotImplementedError

    @property
    def engine(self) -> Engine:
        eng = self._engine
        if eng is None or not eng.arena.intact():
            eng = self._new_engine()
            object.__setattr__(self, "_engine", eng)
            names = {}
            for n in eng.arena.names:
                names[id(eng.arena._param_objs[n])] = n
            object.__setattr__(self, "_engine_param_names", names)
            object.__setattr__(self, "_engine_params", [eng.arena._param_objs[n] for n in eng.arena.names])
        return eng

    def _apply(self, fn, *a, **k):
        # moving / casting the module invalidates the arena views; rebuild lazily afterwards
        object.__setattr__(self, "_engine", None)
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        if self._engine is not None:
            self._engine.mark_weights_dirty()
        return out


class CaptioningModel(_EngineModel):
    def __init__(self, visual: VisualBackbone, textual: TextualHead, caption_backward: bool = False,
                 sos_index: int = 1, eos_index: int = 2, decoder: Any = None):
        super().__init__()
        self.visual = visual
        self.textual = textual
        self.padding_idx = self.textual.padding_idx
        self.caption_backward = caption_backward
        if self.caption_backward:
            self.backward_textual = copy.deepcopy(self.textual)
            # share visual projection and input/output embeddings between directions (captioning.py:60-63)
            self.backward_textual.visual_projection = self.textual.visual_projection
            self.backward_textual.embedding = self.textual.embedding
            self.backward_textual.output = self.textual.output
        self.sos_index = sos_index
        self.eos_index = eos_index
        self.decoder = decoder
        self._engine = None

    # ---------------------------------------------------------------------------------------------------- engine
    def _new_engine(self) -> Engine:
        return Engine(self.visual, self.textual, self.backward_textual if self.caption_backward else None)

    # ---------------------------------------------------------------------------------------------------- forward
    def forward(self, batch: Dict[str, torch.Tensor]) -> Dict[str, Any]:
        if "caption_tokens" not in batch:
            if self.decoder is None:
                raise ValueError("Decoder for predicting captions is missing!")
            return {"predictions": self._decode(batch["image"])}
        image = batch["image"]
        if image.device.type != "cuda":
            raise RuntimeError("virtex_b200 has no CPU path: the batch must live on the model's CUDA device")
        image = image.contiguous().float()
        tokens = batch["caption_tokens"].contiguous()
        lengths = batch["caption_lengths"].contiguous()
        noitpac = batch["noitpac_tokens"].contiguous() if self.caption_backward else tokens
        eng = self.engine
        eng.mark_weights_dirty()  # parameters may have been updated by any optimiser since the last call
        if self.training and torch.is_grad_enabled():
            loss_f, loss_b = _StepFunction.apply(self, image, tokens, noitpac, lengths, None, *self._engine_params)
        else:
            loss = eng.forward(image, tokens, noitpac, lengths, training=self.training, with_grad=False).clone()
            loss_f, loss_b = loss[0], loss[1]
        output: Dict[str, Any] = {"loss": loss_f, "loss_components": {"captioning_forward": loss_f.detach().clone()}}
        if self.caption_backward:
            output["loss"] = loss_f + loss_b
            output["loss_components"]["captioning_backward"] = loss_b.detach().clone()
        if not self.training:
            output["predictions"] = eng.predictions().clone()
        return output

    @torch.no_grad()
    def _decode(self, image):
        """Captions of `image` by the stored decoder (captioning.py:144-163): the KV-cached `Engine.decode` for an
        `AutoRegressiveBeamSearch`, otherwise the decoder's own `search` over `decoding_step`."""
        if image.device.type != "cuda":
            raise RuntimeError("virtex_b200 has no CPU path: the batch must live on the model's CUDA device")
        if self.training:
            raise RuntimeError("caption decoding runs in eval mode only (call model.eval()): the reference would decode "
                               "with dropout active, which cannot be reproduced")
        eng = self.engine
        eng.mark_weights_dirty()
        dec = self.decoder
        if isinstance(dec, AutoRegressiveBeamSearch):
            predictions, _ = eng.decode(image, self.sos_index, dec._eos_index, dec.beam_size, dec.per_node_beam_size,
                                        dec.max_steps, only_return_best=True)
            return predictions
        visual_features = eng.visual_features(image)
        start = torch.full((image.shape[0],), self.sos_index, dtype=torch.int64, device=image.device)
        predictions, _ = dec.search(start, functools.partial(self.decoding_step, visual_features))
        return predictions

    @torch.no_grad()
    def decoding_step(self, visual_features, partial_captions):
        """Logits (rows, V) of the next token after each partial caption (captioning.py:165-213).  Rows beyond the batch
        are beams: image r // beam (the reference repeats the features per beam; the head sees the same inputs)."""
        B, C, h, w = visual_features.shape
        if partial_captions.dim() == 1:
            partial_captions = partial_captions.unsqueeze(1)
        rows, T = partial_captions.shape
        beam = rows // B
        if beam > 1:
            visual_features = visual_features.unsqueeze(1).expand(B, beam, C, h, w).reshape(rows, C, h, w)
        lengths = torch.full((rows,), T, dtype=torch.int64, device=partial_captions.device)
        eng = self.engine
        if not eng._weights_fresh:
            eng.prepare_weights()
        logits = eng.head_logits(visual_features, partial_captions, lengths, training=self.training)
        return logits[:, -1, :].clone()


class ForwardCaptioningModel(CaptioningModel):
    def __init__(self, visual, textual, sos_index: int = 1, eos_index: int = 2, decoder: Any = None):
        super().__init__(visual, textual, sos_index=sos_index, eos_index=eos_index, caption_backward=False,
                         decoder=decoder)


class BidirectionalCaptioningModel(CaptioningModel):
    def __init__(self, visual, textual, sos_index: int = 1, eos_index: int = 2, decoder: Any = None):
        super().__init__(visual, textual, sos_index=sos_index, eos_index=eos_index, caption_backward=True,
                         decoder=decoder)


VirTexModel = BidirectionalCaptioningModel


class MaskedLMModel(CaptioningModel):
    """Drop-in for virtex/models/masked_lm.py:11-86 on the same engine: one textual head whose self-attention masks
    padded keys only (`mask_future_positions=False`, textual_heads.py:255-262), cross entropy between the logits of
    EVERY position and `batch["masked_labels"]` (ignore_index = padding), and in eval mode the argmax predictions with
    the positions that carry no label set to the padding index (masked_lm.py:78-84)."""

    def __init__(self, visual: VisualBackbone, textual: TextualHead):
        super().__init__(visual, textual, caption_backward=False)
        if getattr(textual, "mask_future_positions", False):
            raise ValueError("masked language modelling needs a textual head built with mask_future_positions=False")

    def forward(self, batch: Dict[str, torch.Tensor]) -> Dict[str, Any]:
        image = batch["image"]
        if image.device.type != "cuda":
            raise RuntimeError("virtex_b200 has no CPU path: the batch must live on the model's CUDA device")
        image = image.contiguous().float()
        tokens = batch["caption_tokens"].contiguous()
        lengths = batch["caption_lengths"].contiguous()
        labels = batch["masked_labels"].contiguous()
        eng = self.engine
        eng.mark_weights_dirty()
        if self.training and torch.is_grad_enabled():
            loss, _ = _StepFunction.apply(self, image, tokens, tokens, lengths, labels, *self._engine_params)
        else:
            loss = eng.forward(image, tokens, tokens, lengths, training=self.training, with_grad=False,
                               labels=labels).clone()[0]
        output: Dict[str, Any] = {"loss": loss, "loss_components": {"masked_lm": loss.detach().clone()}}
        if not self.training:
            predictions = eng.predictions().clone()
            predictions[labels == self.padding_idx] = self.padding_idx
            output["predictions"] = predictions
        return output


class ClassificationModel(_EngineModel):
    """Drop-in for virtex/models/classification.py:12-102: a `LinearTextualHead` over the visual features and the
    K-hot loss -- per image, the negative mean log-probability of its unique labels minus `ignore_indices`, averaged
    over the batch.  An image without any such label makes the loss NaN (the mean of nothing) and receives a zero
    gradient, as under the reference's autograd.  In eval mode `predictions` holds the top-10 label ids, best first."""

    def __init__(self, visual: VisualBackbone, textual: TextualHead, ignore_indices: List[int]):
        super().__init__()
        if not isinstance(textual, LinearTextualHead):
            raise ValueError("classification models take a LinearTextualHead (textual head name 'none')")
        self.visual = visual
        self.textual = textual
        self.ignore_indices = ignore_indices
        self._engine = None

    def _new_engine(self) -> Engine:
        return Engine(self.visual, self.textual, ignore_indices=self.ignore_indices)

    def forward(self, batch: Dict[str, torch.Tensor]) -> Dict[str, Any]:
        labels = batch["labels"]
        image = batch["image"]
        if not self.training and self.textual.vocab_size < 10:
            raise ValueError(f"top-10 predictions need at least 10 classes, the head has {self.textual.vocab_size}")
        if image.device.type != "cuda" or labels.device != image.device:
            raise RuntimeError("virtex_b200 has no CPU path: the batch must live on the model's CUDA device")
        image = image.contiguous().float()
        labels = labels.long().contiguous()
        eng = self.engine
        eng.mark_weights_dirty()  # parameters may have been updated by any optimiser since the last call
        if self.training and torch.is_grad_enabled():
            loss, _ = _StepFunction.apply(self, image, None, None, None, labels, *self._engine_params)
        else:
            loss = eng.forward(image, None, None, None, training=self.training, with_grad=False,
                               labels=labels).clone()[0]
        output: Dict[str, Any] = {"loss": loss, "loss_components": {"classification": loss.detach().clone()}}
        if not self.training:
            output["predictions"] = eng.predictions().clone()
        return output

    def _eval_predictions(self, batch):
        self.eval()
        with torch.no_grad():
            predictions = self.forward(batch)["predictions"]
        self.train()
        return predictions


class TokenClassificationModel(ClassificationModel):
    """Labels are the caption tokens, minus [UNK], [SOS], [EOS] and [MASK] (virtex/models/classification.py:105-134)."""

    def log_predictions(self, batch: Dict[str, torch.Tensor], tokenizer) -> str:
        """Caption and top-10 tokens of every image, for logging; `tokenizer` needs `decode(ids)` and
        `id_to_token(id)`.  Runs an eval-mode forward and leaves the model in training mode, like the reference."""
        predictions = self._eval_predictions(batch)
        lines = []
        for tokens, preds in zip(batch["caption_tokens"], predictions):
            words = " ".join(tokenizer.id_to_token(p) for p in preds.tolist())
            lines += [f"Caption tokens : {tokenizer.decode(tokens.tolist())}", f"Predictions (f): {words}", ""]
        return "\n".join(lines)


class MultiLabelClassificationModel(ClassificationModel):
    """Labels are the COCO category ids of an image's instances, minus the background id 0
    (virtex/models/classification.py:137-164)."""

    def log_predictions(self, batch: Dict[str, torch.Tensor], tokenizer: Any = None) -> str:
        """Sorted ground-truth ids of every image beside as many of its best predicted ids, sorted, for logging.
        `tokenizer` is accepted for a uniform interface and not used."""
        predictions = self._eval_predictions(batch)
        lines = []
        for tokens, preds in zip(batch["caption_tokens"], predictions):
            gt = sorted(t for t in tokens.tolist() if t != 0)
            lines += [f"COCO Instance IDs (GT)   : {gt}", f"COCO Instance IDs (Pred) : {sorted(preds.tolist()[:len(gt)])}",
                      ""]
        return "\n".join(lines)
