"""Factories: drop-in for the model/optimiser side of virtex/factories.py (:40-78 base class, :306-341 visual
backbone, :344-407 textual head, :410-466 pretraining model, :503-545 optimiser, :548-584 LR scheduler).

Same `PRODUCTS` names, `create` / `from_config` semantics and name mini-DSLs (`torchvision::resnet50`,
`transdec_postnorm::L1_H1024_A16_F4096`).  Dataset / tokenizer / image-transform factories are outside the hot path
(SURVEY.md section 2.1 #3) and are not provided; the products of the factories below run on the B200 engine.
"""
import re
from functools import partial
from typing import Any, Callable, Dict, Iterable

from torch import nn, optim

from . import models as vmodels
from . import modules
from . import optim as voptim
from .beam_search import AutoRegressiveBeamSearch
from .config import Config


class Factory:
    PRODUCTS: Dict[str, Callable] = {}

    def __init__(self):
        raise ValueError(f"Cannot instantiate {self.__class__.__name__} object, use `create` classmethod to create a "
                         "product from this factory.")

    @classmethod
    def create(cls, name: str, *args, **kwargs) -> Any:
        if name not in cls.PRODUCTS:
            raise KeyError(f"{cls.__name__} cannot create {name}.")
        return cls.PRODUCTS[name](*args, **kwargs)

    @classmethod
    def from_config(cls, config: Config) -> Any:
        raise NotImplementedError


class VisualBackboneFactory(Factory):
    PRODUCTS: Dict[str, Callable] = {"torchvision": modules.TorchvisionVisualBackbone}

    @classmethod
    def from_config(cls, config: Config) -> modules.VisualBackbone:
        _C = config
        kwargs = {"visual_feature_size": _C.MODEL.VISUAL.FEATURE_SIZE}
        if "torchvision" in _C.MODEL.VISUAL.NAME:
            cnn_name = _C.MODEL.VISUAL.NAME.split("::")[-1]
            kwargs["pretrained"] = _C.MODEL.VISUAL.PRETRAINED
            kwargs["frozen"] = _C.MODEL.VISUAL.FROZEN
            return cls.create("torchvision", cnn_name, **kwargs)
        return cls.create(_C.MODEL.VISUAL.NAME, **kwargs)


class TextualHeadFactory(Factory):
    # the transformer decoder heads, named by the `transdec_*::L.._H.._A.._F..` mini-DSL
    PRODUCTS: Dict[str, Callable] = {
        "transdec_prenorm": partial(modules.TransformerDecoderTextualHead, norm_first=True),
        "transdec_postnorm": partial(modules.TransformerDecoderTextualHead, norm_first=False),
    }
    # MODEL.TEXTUAL.NAME "none": no language-modelling head, only the pooled linear classifier of the token /
    # multilabel classification pretext tasks (virtex/factories.py:344-407).  Kept apart from the decoder architectures
    # in PRODUCTS, which stays the set of transformer heads.
    LINEAR_HEAD = "none"

    @classmethod
    def create(cls, name: str, *args, **kwargs) -> Any:
        if name == cls.LINEAR_HEAD:
            return modules.LinearTextualHead(*args, **kwargs)
        return super().create(name, *args, **kwargs)

    @classmethod
    def from_config(cls, config: Config) -> nn.Module:
        _C = config
        name = _C.MODEL.TEXTUAL.NAME
        kwargs = {"visual_feature_size": _C.MODEL.VISUAL.FEATURE_SIZE, "vocab_size": _C.DATA.VOCAB_SIZE}
        if "trans" in name:
            name, architecture = name.split("::")
            m = re.match(r"L(\d+)_H(\d+)_A(\d+)_F(\d+)", architecture)
            mask_future = _C.MODEL.NAME in {"virtex", "captioning", "bicaptioning"}
            kwargs.update(hidden_size=int(m.group(2)), num_layers=int(m.group(1)), attention_heads=int(m.group(3)),
                          feedforward_size=int(m.group(4)), dropout=_C.MODEL.TEXTUAL.DROPOUT,
                          mask_future_positions=mask_future, max_caption_length=_C.DATA.MAX_CAPTION_LENGTH,
                          padding_idx=_C.DATA.UNK_INDEX)
        return cls.create(name, **kwargs)


class _DecoderSpec:
    """Inert stand-in for the reference's nucleus-sampling decoder: the reference samples with torch.multinomial, which
    cannot be reproduced token for token, so the model only stores it and its `search()` raises."""

    def __init__(self, name, **kwargs):
        self.name = name
        self.__dict__.update(kwargs)

    def search(self, *a, **k):
        raise NotImplementedError("nucleus sampling is not implemented; use beam_search")


class CaptionDecoderFactory(Factory):
    PRODUCTS: Dict[str, Callable] = {"beam_search": AutoRegressiveBeamSearch,
                                     "nucleus_sampling": partial(_DecoderSpec, "nucleus_sampling")}

    @classmethod
    def from_config(cls, config: Config):
        _C = config
        kwargs = {"eos_index": _C.DATA.EOS_INDEX, "max_steps": _C.MODEL.DECODER.MAX_DECODING_STEPS}
        if _C.MODEL.DECODER.NAME == "beam_search":
            kwargs["beam_size"] = _C.MODEL.DECODER.BEAM_SIZE
        elif _C.MODEL.DECODER.NAME == "nucleus_sampling":
            kwargs["nucleus_size"] = _C.MODEL.DECODER.NUCLEUS_SIZE
        return cls.create(_C.MODEL.DECODER.NAME, **kwargs)


class PretrainingModelFactory(Factory):
    PRODUCTS: Dict[str, Callable] = {
        "virtex": vmodels.VirTexModel,
        "bicaptioning": vmodels.BidirectionalCaptioningModel,
        "captioning": vmodels.ForwardCaptioningModel,
        "masked_lm": vmodels.MaskedLMModel,
        "token_classification": vmodels.TokenClassificationModel,
        "multilabel_classification": vmodels.MultiLabelClassificationModel,
    }

    @classmethod
    def from_config(cls, config: Config) -> nn.Module:
        _C = config
        visual = VisualBackboneFactory.from_config(_C)
        textual = TextualHeadFactory.from_config(_C)
        kwargs = {}
        if _C.MODEL.NAME in {"virtex", "captioning", "bicaptioning"}:
            kwargs = {"sos_index": _C.DATA.SOS_INDEX, "eos_index": _C.DATA.EOS_INDEX,
                      "decoder": CaptionDecoderFactory.from_config(_C)}
        elif _C.MODEL.NAME == "token_classification":
            kwargs = {"ignore_indices": [_C.DATA.UNK_INDEX, _C.DATA.SOS_INDEX, _C.DATA.EOS_INDEX, _C.DATA.MASK_INDEX]}
        elif _C.MODEL.NAME == "multilabel_classification":
            kwargs = {"ignore_indices": [0]}  # COCO background category
        return cls.create(_C.MODEL.NAME, visual, textual, **kwargs)


def param_group_hparams(config: Config, name: str):
    """(lr, weight_decay) of a parameter from its NAME: virtex/factories.py:529-533."""
    _C = config
    wd = 0.0 if re.match(_C.OPTIM.NO_DECAY, name) else _C.OPTIM.WEIGHT_DECAY
    lr = _C.OPTIM.CNN_LR if "cnn" in name else _C.OPTIM.LR
    return lr, wd


class OptimizerFactory(Factory):
    PRODUCTS: Dict[str, Callable] = {"sgd": optim.SGD, "adamw": optim.AdamW}

    @classmethod
    def from_config(cls, config: Config, named_parameters: Iterable[Any]) -> optim.Optimizer:
        _C = config
        param_groups = []
        for name, param in named_parameters:
            lr, wd = param_group_hparams(_C, name)
            param_groups.append({"params": [param], "lr": lr, "weight_decay": wd})
        kwargs = {"momentum": _C.OPTIM.SGD_MOMENTUM} if _C.OPTIM.OPTIMIZER_NAME == "sgd" else {}
        optimizer = cls.create(_C.OPTIM.OPTIMIZER_NAME, param_groups, **kwargs)
        if _C.OPTIM.LOOKAHEAD.USE:
            optimizer = voptim.Lookahead(optimizer, k=_C.OPTIM.LOOKAHEAD.STEPS, alpha=_C.OPTIM.LOOKAHEAD.ALPHA)
        return optimizer


class LRSchedulerFactory(Factory):
    PRODUCTS: Dict[str, Callable] = {
        "none": voptim.LinearWarmupNoDecayLR,
        "multistep": voptim.LinearWarmupMultiStepLR,
        "linear": voptim.LinearWarmupLinearDecayLR,
        "cosine": voptim.LinearWarmupCosineAnnealingLR,
    }

    @classmethod
    def from_config(cls, config: Config, optimizer: optim.Optimizer) -> optim.lr_scheduler.LambdaLR:
        _C = config
        kwargs = {"total_steps": _C.OPTIM.NUM_ITERATIONS, "warmup_steps": _C.OPTIM.WARMUP_STEPS}
        if _C.OPTIM.LR_DECAY_NAME == "multistep":
            kwargs.update(gamma=_C.OPTIM.LR_GAMMA, milestones=_C.OPTIM.LR_STEPS)
        return cls.create(_C.OPTIM.LR_DECAY_NAME, optimizer, **kwargs)
