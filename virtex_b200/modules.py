"""Parameter-owning modules that mirror the reference's module tree for the bicaptioning path.

Same constructor signatures, attribute names, parameter/buffer names and state_dict keys as
`virtex/modules/visual_backbones.py:34-74`, `virtex/modules/textual_heads.py:46-95,146-214` and
`virtex/modules/embedding.py:25-44`, so reference checkpoints load with `strict=True` and the name-based optimiser
grouping of `virtex/factories.py:529-533` applies unchanged.  Unlike the reference these modules do not compute with
torch / torchvision kernels: the arithmetic is executed by `virtex_b200.engine.Engine` through the C-ABI library.
torch.nn containers (Conv2d, BatchNorm2d, Linear, Embedding, LayerNorm) are used ONLY as named parameter holders.
"""
import math
from typing import List, Optional

import torch
from torch import nn

_RESNET_BLOCKS = {"resnet50": [3, 4, 6, 3], "resnet101": [3, 4, 23, 3], "resnet152": [3, 8, 36, 3]}


class _NoForward(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError(f"{type(self).__name__} only owns parameters; run the model through virtex_b200.engine")


class Bottleneck(_NoForward):
    """Parameters of torchvision's Bottleneck (torchvision/models/resnet.py:108-163): 1x1 -> 3x3(stride) -> 1x1."""
    expansion = 4

    def __init__(self, inplanes: int, planes: int, stride: int = 1, downsample: bool = False):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, stride=stride, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.stride = stride
        self.downsample = None
        if downsample:
            self.downsample = nn.Sequential(nn.Conv2d(inplanes, planes * 4, 1, stride=stride, bias=False),
                                            nn.BatchNorm2d(planes * 4))


class ResNetParams(_NoForward):
    """Parameter tree of torchvision ResNet-50/101/152 up to layer4 (`fc` replaced by Identity as in the reference)."""

    def __init__(self, name: str = "resnet50", zero_init_residual: bool = True):
        super().__init__()
        if name not in _RESNET_BLOCKS:
            raise KeyError(f"unsupported torchvision backbone '{name}' (supported: {sorted(_RESNET_BLOCKS)})")
        self.blocks_per_layer: List[int] = list(_RESNET_BLOCKS[name])
        self.conv1 = nn.Conv2d(3, 64, 7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        inplanes = 64
        for li, (planes, n) in enumerate(zip([64, 128, 256, 512], self.blocks_per_layer), start=1):
            blocks = []
            for bi in range(n):
                stride = 2 if (bi == 0 and li > 1) else 1
                blocks.append(Bottleneck(inplanes, planes, stride, downsample=(stride != 1 or inplanes != planes * 4)))
                inplanes = planes * 4
            setattr(self, f"layer{li}", nn.Sequential(*blocks))
        self.fc = nn.Identity()
        # torchvision/models/resnet.py:208-223
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
        if zero_init_residual:
            for m in self.modules():
                if isinstance(m, Bottleneck):
                    nn.init.constant_(m.bn3.weight, 0)


class VisualBackbone(nn.Module):
    def __init__(self, visual_feature_size: int):
        super().__init__()
        self.visual_feature_size = visual_feature_size


class TorchvisionVisualBackbone(VisualBackbone):
    """Drop-in for virtex/modules/visual_backbones.py:16-74: `forward(image (B,3,H,W) f32) -> (B,C,H/32,W/32)`."""

    def __init__(self, name: str = "resnet50", visual_feature_size: int = 2048, pretrained: bool = False,
                 frozen: bool = False):
        super().__init__(visual_feature_size)
        if pretrained:
            raise RuntimeError("pretrained torchvision weights need a download; load a state_dict instead (no network)")
        self.cnn = ResNetParams(name, zero_init_residual=True)
        self.frozen = frozen
        if frozen:
            for p in self.cnn.parameters():
                p.requires_grad = False
            self.cnn.eval()

    def forward(self, image: torch.Tensor) -> torch.Tensor:
        from .engine import backbone_features
        return backbone_features(self, image)

    def detectron2_backbone_state_dict(self):
        raise NotImplementedError("Detectron2 export is outside the bicaptioning hot path (SURVEY.md section 2.1 #5)")


class WordAndPositionalEmbedding(_NoForward):
    """Parameters of virtex/modules/embedding.py:25-44 (words with padding_idx, positions, LayerNorm eps=1e-8)."""

    def __init__(self, vocab_size: int, hidden_size: int, dropout: float = 0.0, max_caption_length: int = 30,
                 padding_idx: int = 0):
        super().__init__()
        self.vocab_size = vocab_size
        self.padding_idx = padding_idx
        self.words = nn.Embedding(vocab_size, hidden_size, padding_idx=padding_idx)
        self.positions = nn.Embedding(max_caption_length, hidden_size)
        self.layer_norm = nn.LayerNorm(hidden_size, eps=1e-8, elementwise_affine=True)
        self.dropout = nn.Dropout(p=dropout)


class MultiheadAttentionParams(_NoForward):
    """Parameter layout of nn.MultiheadAttention with packed in-projection."""

    def __init__(self, embed_dim: int, num_heads: int):
        super().__init__()
        self.embed_dim, self.num_heads = embed_dim, num_heads
        self.in_proj_weight = nn.Parameter(torch.empty(3 * embed_dim, embed_dim))
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * embed_dim))
        self.out_proj = nn.Linear(embed_dim, embed_dim)
        nn.init.xavier_uniform_(self.in_proj_weight)
        nn.init.constant_(self.out_proj.bias, 0.0)


class TransformerDecoderLayerParams(_NoForward):
    def __init__(self, d_model: int, nhead: int, dim_feedforward: int, norm_first: bool):
        super().__init__()
        self.self_attn = MultiheadAttentionParams(d_model, nhead)
        self.multihead_attn = MultiheadAttentionParams(d_model, nhead)
        self.linear1 = nn.Linear(d_model, dim_feedforward)
        self.linear2 = nn.Linear(dim_feedforward, d_model)
        self.norm_first = norm_first
        self.norm1 = nn.LayerNorm(d_model, eps=1e-5)
        self.norm2 = nn.LayerNorm(d_model, eps=1e-5)
        self.norm3 = nn.LayerNorm(d_model, eps=1e-5)


class TransformerDecoderParams(_NoForward):
    def __init__(self, d_model, nhead, dim_feedforward, num_layers, norm_first):
        super().__init__()
        self.layers = nn.ModuleList(
            [TransformerDecoderLayerParams(d_model, nhead, dim_feedforward, norm_first) for _ in range(num_layers)])
        self.num_layers = num_layers
        self.norm = nn.LayerNorm(d_model) if norm_first else None


class TextualHead(nn.Module):
    def __init__(self, visual_feature_size: int, vocab_size: int, hidden_size: int):
        super().__init__()
        self.visual_feature_size = visual_feature_size
        self.vocab_size = vocab_size
        self.hidden_size = hidden_size

    @property
    def textual_feature_size(self):
        return self.hidden_size


class LinearTextualHead(TextualHead):
    """Drop-in for virtex/modules/textual_heads.py:46-95: global average pooling of the visual features, then one
    linear layer to the vocabulary (`output`, torch's default initialisation).  The classification pretext models use
    it; `caption_tokens` / `caption_lengths` are accepted and ignored, as in the reference."""

    def __init__(self, visual_feature_size: int, vocab_size: int, **kwargs):
        super().__init__(visual_feature_size, vocab_size, visual_feature_size)
        self.output = nn.Linear(visual_feature_size, vocab_size)

    def forward(self, visual_features: torch.Tensor, caption_tokens: Optional[torch.Tensor] = None,
                caption_lengths: Optional[torch.Tensor] = None) -> torch.Tensor:
        from .engine import head_logits
        return head_logits(self, visual_features, caption_tokens, caption_lengths)


class TransformerDecoderTextualHead(TextualHead):
    """Drop-in for virtex/modules/textual_heads.py:98-292 (same kwargs, attributes and initialisation)."""

    def __init__(self, visual_feature_size: int, vocab_size: int, hidden_size: int, num_layers: int,
                 attention_heads: int, feedforward_size: int, dropout: float = 0.1, norm_first: bool = False,
                 mask_future_positions: bool = True, max_caption_length: int = 30, padding_idx: int = 0):
        super().__init__(visual_feature_size, vocab_size, hidden_size)
        if hidden_size != 64 * attention_heads:
            raise ValueError("the B200 attention kernel is specialised for head_dim 64 (A = H/64 in every VirTex config)")
        self.num_layers = num_layers
        self.attention_heads = attention_heads
        self.feedforward_size = feedforward_size
        self.dropout = dropout
        self.norm_first = norm_first
        self.mask_future_positions = mask_future_positions
        self.padding_idx = padding_idx
        self.max_caption_length = max_caption_length

        self.visual_projection = nn.Linear(visual_feature_size, self.textual_feature_size)
        self.embedding = WordAndPositionalEmbedding(self.vocab_size, self.textual_feature_size, dropout=dropout,
                                                    max_caption_length=max_caption_length, padding_idx=padding_idx)
        self.transformer = TransformerDecoderParams(self.textual_feature_size, attention_heads, feedforward_size,
                                                    num_layers, norm_first)
        self.apply(self._init_weights)
        # created after the init sweep, tied to the word embedding (textual_heads.py:197-200)
        self.output = nn.Linear(self.textual_feature_size, vocab_size)
        self.output.weight = self.embedding.words.weight

    @staticmethod
    def _init_weights(module):
        """BERT-style N(0, 0.02) for Linear / MHA / Embedding weights; biases keep torch defaults (textual_heads.py:202-214)."""
        if isinstance(module, nn.Linear):
            module.weight.data.normal_(mean=0.0, std=0.02)
        elif isinstance(module, MultiheadAttentionParams):
            module.in_proj_weight.data.normal_(mean=0.0, std=0.02)
            module.out_proj.weight.data.normal_(mean=0.0, std=0.02)
        elif isinstance(module, nn.Embedding):
            module.weight.data.normal_(mean=0.0, std=0.02)
            if module.padding_idx is not None:
                module.weight.data[module.padding_idx].zero_()

    def forward(self, visual_features: torch.Tensor, caption_tokens: torch.Tensor,
                caption_lengths: torch.Tensor) -> torch.Tensor:
        from .engine import head_logits
        return head_logits(self, visual_features, caption_tokens, caption_lengths)
