"""Execution engine of the bicaptioning step: schedules the C-ABI kernels over pre-allocated HBM buffers.

This replaces, for the hot path, what autograd + cuDNN + cuBLASLt + ATen do for the reference
(`virtex/models/captioning.py:99-143` forward; its autograd backward).  One `Engine` owns

  * a flat fp32 parameter arena (the modules' nn.Parameters are re-pointed to views of it), a flat fp32 gradient arena
    of identical layout (what the data-parallel all-reduce and the fused optimiser consume), and a flat bf16 mirror of
    the parameters (the GEMM B operands) plus packed bf16 layouts for the 3x3 / 7x7 convolution weights;
  * every activation / workspace buffer, allocated once per (batch, caption length) shape -- no allocation, no host
    synchronisation and no Python-side tensor math inside a step (the step is launch-ahead of the GPU by design; it is
    NOT captured in a CUDA graph today -- the GPU is 99 % busy without one, and the tensor maps are re-encoded per launch).

Data layout in HBM: backbone activations NHWC bf16 (a conv output is a row-major [N*H*W, C] matrix: 1x1 convs are
GEMMs as-is, 3x3/stride-1 convs are implicit GEMMs through 4-D TMA boxes), BN statistics / affine parameters fp32,
decoder residual stream fp32 with bf16 shadows feeding the GEMMs, logits bf16 (fp32 only for eval argmax).
"""
from __future__ import annotations

import math
import os
import struct
from typing import Dict, List, Optional, Tuple

import torch
from torch import nn

from . import ops
from .beam_search import BeamState
from .modules import LinearTextualHead
from .ops import call, gemm, _p, _stream

BF16, F32 = torch.bfloat16, torch.float32
_ALIGN = 64  # arena alignment in elements (256 B for fp32, 128 B for bf16: TMA base pointers need 16 B)


def _round_up(x, m):
    return (x + m - 1) // m * m


class Arena:
    """Flat fp32 parameter / gradient storage with a bf16 mirror; parameters become views into it."""

    def __init__(self, named_params: List[Tuple[str, nn.Parameter]], device):
        self.device = device
        self.names: List[str] = []
        self.offsets: Dict[str, int] = {}
        self.numels: Dict[str, int] = {}
        self.shapes: Dict[str, torch.Size] = {}
        off = 0
        seen = {}
        for name, p in named_params:
            if id(p) in seen:
                continue
            seen[id(p)] = name
            self.names.append(name)
            self.offsets[name] = off
            self.numels[name] = p.numel()
            self.shapes[name] = p.shape
            off = _round_up(off + p.numel(), _ALIGN)
        self.total = off
        self.params = torch.zeros(off, dtype=F32, device=device)
        self.grads = torch.zeros(off, dtype=F32, device=device)
        self.mirror = torch.zeros(off, dtype=BF16, device=device)
        self._param_objs = {seen[id(p)]: p for _, p in named_params}
        with torch.no_grad():
            for name in self.names:
                p = self._param_objs[name]
                v = self.view(self.params, name)
                v.copy_(p.data.to(device=device, dtype=F32))
                p.data = v
                p.grad = None

    def view(self, flat, name):
        o = self.offsets[name]
        return flat[o:o + self.numels[name]].view(self.shapes[name])

    def p(self, name):
        return self.view(self.params, name)

    def g(self, name):
        return self.view(self.grads, name)

    def w(self, name):
        return self.view(self.mirror, name)

    def intact(self):
        """True while every parameter still aliases the arena (a `.to()` / `.half()` on the module breaks it)."""
        base, end = self.params.data_ptr(), self.params.data_ptr() + self.total * 4
        for name in (self.names[0], self.names[-1]):
            ptr = self._param_objs[name].data_ptr()
            if not (base <= ptr < end):
                return False
        return True

    def refresh_mirror(self):
        call("vtx_cast_bf16", self.params.data_ptr(), self.mirror.data_ptr(), self.total, _stream())


class _Workspace:
    """Named device buffers that only ever grow: after the first step of a given shape nothing is allocated."""

    def __init__(self, device):
        self.device = device
        self.flat: Dict[str, torch.Tensor] = {}

    def get(self, name, shape, dtype):
        shape = tuple(int(s) for s in shape)
        n = 1
        for s in shape:
            n *= s
        t = self.flat.get(name)
        if t is None or t.dtype != dtype or t.numel() < n:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self.flat[name] = t
        return t[:n].view(shape)

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in self.flat.values())


def _require_cuda(dev):
    if dev is None or dev.type != "cuda":
        raise RuntimeError("virtex_b200 has no CPU path: move the model to a CUDA device first (model.cuda())")


class Engine:
    """Forward/backward of (backbone) + (forward head) + (backward head) on one GPU.  Any part may be absent."""

    def __init__(self, visual=None, textual=None, backward_textual=None, prefix_map=None, ignore_indices=()):
        self.visual, self.textual, self.backward_textual = visual, textual, backward_textual
        # classification pretext heads (pool + linear + K-hot loss) instead of a transformer decoder
        self.classification = isinstance(textual, LinearTextualHead)
        named: List[Tuple[str, nn.Parameter]] = []
        if visual is not None:
            named += [("visual." + n, p) for n, p in visual.named_parameters()]
        if textual is not None:
            named += [("textual." + n, p) for n, p in textual.named_parameters()]
        if backward_textual is not None:
            named += [("backward_textual." + n, p) for n, p in backward_textual.named_parameters()]
        dev = None
        for _, p in named:
            dev = p.device
            break
        _require_cuda(dev)
        self.device = dev
        self.arena = Arena(named, dev)
        self.ws = _Workspace(dev)
        self.buffers: Dict[str, torch.Tensor] = {}
        if visual is not None:
            self.buffers.update({"visual." + n: b for n, b in visual.named_buffers()})
        head = textual if textual is not None else backward_textual
        self.pad = getattr(head, "padding_idx", 0) if head is not None else 0
        # label ids the K-hot loss leaves out of every image's label set (ClassificationModel.ignore_indices)
        self.ignore = torch.tensor([int(i) for i in ignore_indices], dtype=torch.int64, device=dev)
        self.seed = torch.zeros(1, dtype=torch.int64, device=dev)
        self.loss = torch.zeros(2, dtype=F32, device=dev)       # per-direction mean NLL
        self.count = torch.zeros(2, dtype=F32, device=dev)      # per-direction number of valid targets
        self._packed: Dict[str, torch.Tensor] = {}
        self._tape = None
        self.generation = 0  # bumped by every forward(): a backward must match the forward that filled the tape
        self._weights_fresh = False
        # BN-backward reductions (sum dz, sum dz * xhat) accumulated by the epilogue of the GEMM that produces the
        # gradient (bn1 / bn2 of every block, bn3 of blocks followed by an identity block) instead of a separate pass;
        # VTX_BNR_FUSE=0 is the measurement knob for the A/B against the standalone vtx_bn_bwd_reduce launches
        self.fuse_bn_reduce = os.environ.get("VTX_BNR_FUSE", "1") != "0"
        self.fuse_bn3_min_rows = int(os.environ.get("VTX_BNR_BN3_MIN_ROWS", "100000"))  # (env: measurement knob)
        self._build_backbone_plan()

    # ------------------------------------------------------------------------------------------------ parameters
    def P(self, name):
        return self.arena.p(name)

    def W(self, name):
        return self.arena.w(name)

    def G(self, name):
        return self.arena.g(name)

    def mark_weights_dirty(self):
        self._weights_fresh = False

    def _build_backbone_plan(self):
        self.blocks = []
        self._jobs: Dict[str, tuple] = {}
        if self.visual is None:
            return
        cnn = self.visual.cnn
        for li in range(1, 5):
            layer = getattr(cnn, f"layer{li}")
            for bi, blk in enumerate(layer):
                self.blocks.append((f"visual.cnn.layer{li}.{bi}", blk))
        # fp32 weight-gradient scratch of every k > 1 convolution (GEMM output layout), one flat buffer zeroed once per
        # backward; the batched unpack jobs fold it into the OIHW gradient arena per all-reduce bucket
        sizes = [("visual.cnn.conv1", 64 * 256)]
        sizes += [(name + ".conv2", 9 * blk.conv2.weight.shape[0] ** 2) for name, blk in self.blocks]
        total = sum(_round_up(n, _ALIGN) for _, n in sizes)
        self._dwp_flat = torch.zeros(total, dtype=F32, device=self.device)
        self._dwp, off = {}, 0
        for key, n in sizes:
            self._dwp[key] = self._dwp_flat[off:off + n]
            off += _round_up(n, _ALIGN)

    # ------------------------------------------------------------------------------------ batched weight-layout jobs
    def _job_table(self, key, make):
        """Device-resident VtxWeightJob table, built once per key: (src, dst, total, O, I, KH, KW, ldk, kind) rows."""
        tab = self._jobs.get(key)
        if tab is None:
            rows = make()
            blk = ops.L.load().vtx_weight_job_block_elems()
            blob, b0 = b"", 0
            for src, dst, total, O, I, KH, KW, ldk, kind in rows:
                blob += struct.pack("<QQq8i", src.data_ptr(), dst.data_ptr(), total, O, I, KH, KW, ldk, kind, b0, 0)
                b0 += (total + blk - 1) // blk
            dev = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(self.device) if rows else None
            tab = self._jobs[key] = (dev, len(rows), b0)
        return tab

    def _run_jobs(self, key, make):
        dev, n, blocks = self._job_table(key, make)
        if n:
            call("vtx_conv_w_jobs", dev.data_ptr(), n, blocks, _stream())

    def _pack_rows(self):
        w = self.P("visual.cnn.conv1.weight")
        rows = [(w, self._pack_buf("visual.cnn.conv1.weight", (64, 160)), 64 * 160, 64, 3, 7, 7, 160, 0),
                (w, self._pack_buf("visual.cnn.conv1.weight#s2d", (64, 256)), 64 * 256, 64, 3, 7, 7, 256, 4)]
        for name, blk in self.blocks:
            w = self.P(name + ".conv2.weight")
            pl = w.shape[0]
            rows.append((w, self._pack_buf(name + ".conv2.weight", (pl, 9 * pl)), 9 * pl * pl, pl, pl, 3, 3, 9 * pl, 0))
            if blk.stride == 1:
                rows.append((w, self._pack_buf(name + ".conv2.weight#dgrad", (pl, 9 * pl)), 9 * pl * pl, pl, pl, 3, 3,
                             9 * pl, 1))
            if blk.stride == 2 and blk.downsample is not None:
                wdn = self.P(name + ".downsample.0.weight")
                C4, Cin = wdn.shape[0], wdn.shape[1]
                if Cin % 64 == 0:  # transposed copy: K-major B operand of the downsample's (implicit, strided-store) dgrad
                    rows.append((wdn, self._pack_buf(name + ".downsample.0.weight#t", (Cin, C4)), C4 * Cin, C4, Cin, 1, 1,
                                 C4, 7))
            if blk.stride != 1:  # stride-2 dgrad: one weight slice per parity class (ph, pw) of the input gradient
                for ph in (0, 1):
                    for pw in (0, 1):
                        nt = (1 + ph) * (1 + pw)
                        rows.append((w, self._pack_buf(f"{name}.conv2.weight#dgrad_s2_{ph}{pw}", (pl, nt * pl)),
                                     nt * pl * pl, pl, pl, ph, pw, nt * pl, 6))
        return rows

    def _unpack_rows(self, layer, stem_s2d):
        """Unpack-accumulate jobs of one gradient bucket: 'layer4' / 'layer3' / 'layer2' / 'rest' (layer1 + stem)."""
        rows = []
        want = "layer1" if layer == "rest" else layer
        for name, blk in self.blocks:
            if name.split(".")[2] != want:
                continue
            pl = blk.conv2.weight.shape[0]
            transposed = blk.stride == 1 and pl == 64  # halo-reuse wgrad writes [(tap, cin), cout]
            rows.append((self._dwp[name + ".conv2"], self.G(name + ".conv2.weight"), 9 * pl * pl, pl, pl, 3, 3, 9 * pl,
                         3 if transposed else 2))
        if layer == "rest":
            g = self.G("visual.cnn.conv1.weight")
            if stem_s2d:
                rows.append((self._dwp["visual.cnn.conv1"], g, 64 * 147, 64, 3, 7, 7, 256, 5))
            else:
                rows.append((self._dwp["visual.cnn.conv1"], g, 64 * 147, 64, 3, 7, 7, 160, 2))
        return rows

    def prepare_weights(self, mirror=True):
        """bf16 mirror of all parameters + packed GEMM layouts of the k>1 convolution weights."""
        if mirror:
            self.arena.refresh_mirror()
        if self.visual is not None:
            self._run_jobs("pack", self._pack_rows)  # every packed conv-weight layout in one launch
        self._weights_fresh = True

    def _pack_buf(self, key, shape):
        t = self._packed.get(key)
        if t is None:
            t = torch.empty(shape, dtype=BF16, device=self.device)
            self._packed[key] = t
        return t

    # ------------------------------------------------------------------------------------------------ backbone fwd
    def _bn_fwd(self, y, bn_name, M, C, training, stats):
        bnp = self.ws.get("bnp:" + bn_name, (4, C), F32)
        nbt = self.buffers[bn_name + ".num_batches_tracked"]
        call("vtx_bn_finalize", _p(stats), float(M), self.P(bn_name + ".weight").data_ptr(),
             self.P(bn_name + ".bias").data_ptr(), self.buffers[bn_name + ".running_mean"].data_ptr(),
             self.buffers[bn_name + ".running_var"].data_ptr(), nbt.data_ptr(), 0.1, 1e-5, int(training),
             bnp.data_ptr(), C, _stream())
        return bnp

    def _bn_act_fwd(self, y, bn_name, M, C, training, stats, out, res=None, bnp_res=None, relu=1, mask=None):
        """BN finalize (batch or running statistics -> bnp, running-stat update) + apply + ReLU (+ residual), one launch.
        `mask`: uint8 [M, C/8] ReLU sign bits for backward (block outputs, whose pre-activation includes the shortcut)."""
        bnp = self.ws.get("bnp:" + bn_name, (4, C), F32)
        call("vtx_bn_finalize_act", _p(stats), float(M), self.P(bn_name + ".weight").data_ptr(),
             self.P(bn_name + ".bias").data_ptr(), self.buffers[bn_name + ".running_mean"].data_ptr(),
             self.buffers[bn_name + ".running_var"].data_ptr(),
             self.buffers[bn_name + ".num_batches_tracked"].data_ptr(), 0.1, 1e-5, int(training), bnp.data_ptr(),
             y.data_ptr(), _p(res), _p(bnp_res), out.data_ptr(), _p(mask), M, C, relu, _stream())
        return bnp

    def _stats_slab(self, training):
        """One zeroed fp32 slab per step holding every BN's [2,C] sum/sumsq (fwd) and [2,C] dz sums (bwd)."""
        total = 2 * 64 * 2
        for name, blk in self.blocks:
            planes = blk.conv1.weight.shape[0]
            total += 2 * 2 * (planes + planes + 4 * planes + (4 * planes if blk.downsample is not None else 0))
        slab = self.ws.get("bn_slab", (total,), F32)
        slab.zero_()
        self._slab, self._slab_off = slab, 0
        return slab

    def _slab_take(self, n):
        t = self._slab[self._slab_off:self._slab_off + n]
        self._slab_off += n
        return t

    def backbone_forward(self, image: torch.Tensor, training: bool):
        """image fp32 NCHW [B,3,H,W] -> NHWC bf16 feature matrix [B*h*w, 2048]; fills the tape used by backward."""
        if not self._weights_fresh:
            self.prepare_weights()
        B, _, H, W = image.shape
        s = _stream()
        ws = self.ws
        self._stats_slab(training)
        tape = {"B": B, "blocks": [], "training": training}
        # ---- stem: im2col -> GEMM(+stats) -> BN finalize -> BN+ReLU+maxpool
        Ho, Wo = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
        M0 = B * Ho * Wo
        y0 = ws.get("stem.y", (M0, 64), BF16)
        st = self._slab_take(128) if training else None
        cols = s2d = None
        if H % 2 == 0 and W % 4 == 0 and Ho % 8 == 0 and Wo % 16 == 0:  # the 16 x 8 TMA boxes tile the output exactly
            # 4-tap implicit GEMM over the space-to-depth view of the image (csrc/stem_s2d.cu)
            s2d = ws.get("stem.s2d", (B, H // 2 + 3, W // 2 + 3, 16), BF16)
            call("vtx_stem_s2d", image.data_ptr(), s2d.data_ptr(), B, H, W, s)
            gemm(s2d, self._packed["visual.cnn.conv1.weight#s2d"], y0, M0, 64, 256, lda=64, ldb=256, stats=st,
                 conv=(B, Ho, Wo, 64), conv_mode=5)
        else:  # other image sizes: im2col + plain GEMM
            cols = ws.get("stem.cols", (M0, 160), BF16)
            call("vtx_stem_im2col", image.data_ptr(), cols.data_ptr(), B, H, W, 160, s)
            gemm(cols, self._packed["visual.cnn.conv1.weight"], y0, M0, 64, 160, stats=st)
        bnp0 = self._bn_fwd(y0, "visual.cnn.bn1", M0, 64, training, st)
        Hp, Wp = (Ho - 1) // 2 + 1, (Wo - 1) // 2 + 1
        x = ws.get("stem.pool", (B * Hp * Wp, 64), BF16)
        idx = ws.get("stem.idx", (B * Hp * Wp, 64), torch.uint8)
        call("vtx_bn_relu_maxpool", y0.data_ptr(), bnp0.data_ptr(), x.data_ptr(), idx.data_ptr(), B, Ho, Wo, 64, s)
        tape["stem"] = dict(cols=cols, s2d=s2d, y=y0, bnp=bnp0, idx=idx, Ho=Ho, Wo=Wo, Hp=Hp, Wp=Wp, M=M0)
        Hc, Wc, Cin = Hp, Wp, 64
        # ---- bottleneck blocks
        for name, blk in self.blocks:
            planes = blk.conv1.weight.shape[0]
            stride = blk.stride
            Hn, Wn = (Hc - 1) // stride + 1, (Wc - 1) // stride + 1
            Min, Mout = B * Hc * Wc, B * Hn * Wn
            rec = dict(name=name, x=x, Hin=Hc, Win=Wc, Hout=Hn, Wout=Wn, Cin=Cin, planes=planes, stride=stride,
                       Min=Min, Mout=Mout, has_ds=blk.downsample is not None)
            # conv1 1x1
            y1 = ws.get(name + ".y1", (Min, planes), BF16)
            st1 = self._slab_take(2 * planes) if training else None
            gemm(x, self.W(name + ".conv1.weight").view(planes, Cin), y1, Min, planes, Cin, stats=st1)
            a1 = ws.get(name + ".a1", (Min, planes), BF16)
            bnp1 = self._bn_act_fwd(y1, name + ".bn1", Min, planes, training, st1, a1)
            # conv2 3x3 (stride)
            y2 = ws.get(name + ".y2", (Mout, planes), BF16)
            st2 = self._slab_take(2 * planes) if training else None
            w2 = self._packed[name + ".conv2.weight"]
            if planes % 64 == 0:
                # implicit GEMM: 4-D TMA boxes gather the taps (zero fill = padding); stride 2 through TMA traversal strides
                gemm(a1, w2, y2, Mout, planes, 9 * planes, lda=planes, stats=st2, conv=(B, Hc, Wc, planes), conv_mode=1,
                     conv_stride=stride)
                rec["cols2"] = None
            else:
                cols2 = ws.get(name + ".cols2", (Mout, 9 * planes), BF16)
                call("vtx_im2col3x3", a1.data_ptr(), cols2.data_ptr(), B, Hc, Wc, planes, stride, s)
                gemm(cols2, w2, y2, Mout, planes, 9 * planes, stats=st2)
                rec["cols2"] = cols2
            a2 = ws.get(name + ".a2", (Mout, planes), BF16)
            bnp2 = self._bn_act_fwd(y2, name + ".bn2", Mout, planes, training, st2, a2)
            # conv3 1x1
            C4 = 4 * planes
            y3 = ws.get(name + ".y3", (Mout, C4), BF16)
            st3 = self._slab_take(2 * C4) if training else None
            gemm(a2, self.W(name + ".conv3.weight").view(C4, planes), y3, Mout, C4, planes, stats=st3)
            out = ws.get(name + ".out", (Mout, C4), BF16)
            # backward needs only the SIGN of the block output's pre-activation: one bit per element instead of re-reading
            # the bf16 output twice (bn_bwd_reduce and bn_bwd_apply)
            m3 = ws.get(name + ".m3", (Mout, C4 // 8), torch.uint8) if training else None
            if blk.downsample is not None:
                yd = ws.get(name + ".yd", (Mout, C4), BF16)
                std = self._slab_take(2 * C4) if training else None
                wd = self.W(name + ".downsample.0.weight").view(C4, Cin)
                if stride == 1:
                    xs = x
                    gemm(xs, wd, yd, Mout, C4, Cin, stats=std)
                elif Cin % 64 == 0:
                    xs = None  # strided 1x1 conv = one-tap implicit GEMM over x (no subsampled copy)
                    gemm(x, wd, yd, Mout, C4, Cin, lda=Cin, stats=std, conv=(B, Hc, Wc, Cin), conv_mode=1,
                         conv_stride=stride, conv_taps=1)
                else:
                    xs = ws.get(name + ".xs", (Mout, Cin), BF16)
                    call("vtx_subsample", x.data_ptr(), xs.data_ptr(), B, Hc, Wc, Cin, stride, s)
                    gemm(xs, wd, yd, Mout, C4, Cin, stats=std)
                bnpd = self._bn_fwd(yd, name + ".downsample.1", Mout, C4, training, std)
                bnp3 = self._bn_act_fwd(y3, name + ".bn3", Mout, C4, training, st3, out, res=yd, bnp_res=bnpd, mask=m3)
                rec.update(xs=xs, yd=yd, bnpd=bnpd)
            else:
                bnp3 = self._bn_act_fwd(y3, name + ".bn3", Mout, C4, training, st3, out, res=x, mask=m3)
            rec.update(y1=y1, bnp1=bnp1, a1=a1, y2=y2, bnp2=bnp2, a2=a2, y3=y3, bnp3=bnp3, out=out, m3=m3)
            tape["blocks"].append(rec)
            x, Hc, Wc, Cin = out, Hn, Wn, C4
        tape["feat"] = x
        tape["hw"] = (Hc, Wc)
        tape["C"] = Cin
        self._tape = tape
        return x, Hc, Wc

    # ------------------------------------------------------------------------------------------------ backbone bwd
    def _wgrad(self, dY, X, dW, n_out, k_in, m_rows):
        """dW[n_out, k_in] (fp32, += ) = dY[m_rows, n_out]^T . X[m_rows, k_in]   (both operands MN-major, split-K)."""
        tiles = ((n_out + 127) // 128) * ((k_in + 255) // 256)
        sk = ops.split_k_for(tiles, (m_rows + 63) // 64)
        gemm(dY, X, dW, n_out, k_in, m_rows, a_mn=1, b_mn=1, atomic=True, split_k=sk, ldd=k_in, out_f32=True)

    def _bn_bwd(self, dA, a, y, bnp, bn_name, M, C, dy, two=None, dz_out=None, mask_from_y=0, sums=None):
        """dA -> dy through (ReLU from the bit mask `a`, or recomputed from y when mask_from_y) + train-mode BN;
        two = (y2, bnp2, bn2_name, dy2) shares dz.  `sums`: the [2, C] reduction already accumulated by the epilogue of
        the GEMM that produced dA (VtxGemm.bnr_*), so only the apply pass is left."""
        s = _stream()
        fused = sums is not None
        if not fused:
            sums = self._slab_take(2 * C)
        if two is None:
            if not fused:
                call("vtx_bn_bwd_reduce", dA.data_ptr(), _p(a), y.data_ptr(), bnp.data_ptr(), 0, 0, sums.data_ptr(), 0,
                     M, C, mask_from_y, s)
            call("vtx_bn_bwd_finalize_apply", sums.data_ptr(), 0, float(M), self.G(bn_name + ".weight").data_ptr(),
                 self.G(bn_name + ".bias").data_ptr(), 0, 0, dA.data_ptr(), _p(a), y.data_ptr(), bnp.data_ptr(),
                 dy.data_ptr(), 0, 0, 0, _p(dz_out), M, C, mask_from_y, s)
        else:
            y2, bnp2, bn2_name, dy2 = two
            sums2 = self._slab_take(2 * C)
            call("vtx_bn_bwd_reduce", dA.data_ptr(), _p(a), y.data_ptr(), bnp.data_ptr(), y2.data_ptr(),
                 bnp2.data_ptr(), sums.data_ptr(), sums2.data_ptr(), M, C, mask_from_y, s)
            call("vtx_bn_bwd_finalize_apply", sums.data_ptr(), sums2.data_ptr(), float(M),
                 self.G(bn_name + ".weight").data_ptr(), self.G(bn_name + ".bias").data_ptr(),
                 self.G(bn2_name + ".weight").data_ptr(), self.G(bn2_name + ".bias").data_ptr(), dA.data_ptr(), _p(a),
                 y.data_ptr(), bnp.data_ptr(), dy.data_ptr(), y2.data_ptr(), bnp2.data_ptr(), dy2.data_ptr(),
                 _p(dz_out), M, C, mask_from_y, s)

    def backbone_backward(self, dfeat: torch.Tensor, bucket_cb=None):
        """dfeat bf16 [B*h*w, C]: gradient w.r.t. the backbone output.  Accumulates into the gradient arena.
        `bucket_cb(tag)` is called when every gradient of 'layer4' / 'layer3' / 'layer2' has been enqueued."""
        tape = self._tape
        if getattr(self.visual, "frozen", False):
            return  # frozen backbone: no parameter gradients, nothing below the visual projection
        if not tape["training"]:
            raise RuntimeError("backward through eval-mode BatchNorm (running statistics) is not implemented")
        B = tape["B"]
        s = _stream()
        ws = self.ws
        dOut = dfeat
        scratch_i = 0
        prev_layer = None
        self._dwp_flat.zero_()
        stem_s2d = tape["stem"]["s2d"] is not None
        blocks = tape["blocks"]
        fuse = self.fuse_bn_reduce
        sums3 = None  # bn3 sums of the current block when the GEMM that produced dOut already accumulated them
        for bi in range(len(blocks) - 1, -1, -1):
            rec = blocks[bi]
            name, planes, Cin, stride = rec["name"], rec["planes"], rec["Cin"], rec["stride"]
            layer = name.split(".")[2]
            if prev_layer is not None and layer != prev_layer:
                self._run_jobs("unpack:" + prev_layer, lambda: self._unpack_rows(prev_layer, stem_s2d))
                if bucket_cb is not None:
                    bucket_cb(prev_layer)
            prev_layer = layer
            Min, Mout, C4 = rec["Min"], rec["Mout"], 4 * rec["planes"]
            Hc, Wc, Hn, Wn = rec["Hin"], rec["Win"], rec["Hout"], rec["Wout"]
            # ---- block output: ReLU mask + bn3 (+ downsample BN) backward
            dy3 = ws.get("bwd.dy3", (Mout, C4), BF16)
            if rec["has_ds"]:
                dyd = ws.get("bwd.dyd", (Mout, C4), BF16)
                self._bn_bwd(dOut, rec["m3"], rec["y3"], rec["bnp3"], name + ".bn3", Mout, C4, dy3,
                             two=(rec["yd"], rec["bnpd"], name + ".downsample.1", dyd))
                dz = None
            else:
                # the shortcut gradient dz = dOut * [block output > 0] is never written: conv1's dgrad epilogue adds
                # dOut under the same bit mask (VtxGemm.residual_mask)
                dz = None
                self._bn_bwd(dOut, rec["m3"], rec["y3"], rec["bnp3"], name + ".bn3", Mout, C4, dy3, sums=sums3)
            sums3 = None
            # ---- conv3 (1x1): wgrad + dgrad; the dgrad epilogue accumulates bn2's backward sums (ReLU mask from y2)
            self._wgrad(dy3, rec["a2"], self.G(name + ".conv3.weight"), C4, planes, Mout)
            da2 = ws.get("bwd.da2", (Mout, planes), BF16)
            sums2 = self._slab_take(2 * planes) if fuse else None
            gemm(dy3, self.W(name + ".conv3.weight").view(C4, planes), da2, Mout, planes, C4, b_mn=1,
                 bnr=(rec["y2"], rec["bnp2"], sums2, None) if fuse else None)
            # ---- bn2 + ReLU backward
            dy2 = ws.get("bwd.dy2", (Mout, planes), BF16)
            self._bn_bwd(da2, None, rec["y2"], rec["bnp2"], name + ".bn2", Mout, planes, dy2, mask_from_y=1, sums=sums2)
            # ---- conv2 (3x3): wgrad + dgrad
            dwp = self._dwp[name + ".conv2"].view(planes, 9 * planes)
            da1 = ws.get("bwd.da1", (Min, planes), BF16)
            sums1 = None
            if rec["cols2"] is None:
                if planes == 64 and stride == 1:
                    # halo-reuse wgrad: D[(tap, cin), cout], accumulated in TMEM over all spatial tiles of a CTA
                    gemm(dy2, rec["a1"], dwp, 9 * planes, planes, Mout, atomic=True, lda=planes, ldb=planes, ldd=planes,
                         conv=(B, Hc, Wc, planes), conv_mode=4, out_f32=True)
                else:
                    tiles = ((planes + 127) // 128) * ((9 * planes + 255) // 256)
                    sk = ops.split_k_for(tiles, (Mout + 63) // 64)
                    gemm(dy2, rec["a1"], dwp, planes, 9 * planes, Mout, atomic=True, split_k=sk, lda=planes,
                         ldb=planes, conv=(B, Hc, Wc, planes), conv_mode=2, out_f32=True, conv_stride=stride)
                if fuse and stride in (1, 2):
                    sums1 = self._slab_take(2 * planes)  # bn1's backward sums, accumulated by the conv2-dgrad epilogue(s)
                if stride == 1:
                    gemm(dy2, self._packed[name + ".conv2.weight#dgrad"], da1, Min, planes, 9 * planes, lda=planes,
                         conv=(B, Hc, Wc, planes), conv_mode=1,
                         bnr=(rec["y1"], rec["bnp1"], sums1, None) if fuse else None)
                elif stride == 2:
                    # strided dgrad as four implicit GEMMs, one per parity class (ph, pw) of the input position: row
                    # 2i+ph of da1 gathers dy rows i+a, a < 1+ph, through kernel rows ph+1-2a (same along w); each class
                    # writes its own strided sub-grid of da1, so every element is written exactly once -- no per-tap
                    # gradient matrix, no col2im scatter
                    for ph in (0, 1):
                        for pw in (0, 1):
                            th, tw = 1 + ph, 1 + pw
                            Hs, Ws = (Hc - ph + 1) // 2, (Wc - pw + 1) // 2
                            if Hs <= 0 or Ws <= 0:
                                continue
                            voff = (ph * Wc + pw) * planes * 2
                            gemm(dy2, self._packed[f"{name}.conv2.weight#dgrad_s2_{ph}{pw}"], da1, Mout, planes,
                                 th * tw * planes, lda=planes, conv=(B, Hn, Wn, planes), conv_mode=1, tap_grid=(th, tw, 0),
                                 d_ptr=da1.data_ptr() + voff,
                                 out_view=(Hs, Ws, 2 * planes, 2 * Wc * planes, Hc * Wc * planes),
                                 bnr=(rec["y1"], rec["bnp1"], sums1, None, rec["y1"].data_ptr() + voff) if fuse else None)
                else:  # other strides: per-tap gradients by a plain GEMM, scattered back by col2im
                    dcols = ws.get("bwd.dcols", (Mout, 9 * planes), BF16)
                    gemm(dy2, self._packed[name + ".conv2.weight"], dcols, Mout, 9 * planes, planes, b_mn=1)
                    call("vtx_col2im3x3", dcols.data_ptr(), da1.data_ptr(), B, Hc, Wc, planes, stride, s)
            else:
                self._wgrad(dy2, rec["cols2"], dwp, planes, 9 * planes, Mout)
                dcols = ws.get("bwd.dcols", (Mout, 9 * planes), BF16)
                gemm(dy2, self._packed[name + ".conv2.weight"], dcols, Mout, 9 * planes, planes, b_mn=1)
                call("vtx_col2im3x3", dcols.data_ptr(), da1.data_ptr(), B, Hc, Wc, planes, stride, s)
            # ---- bn1 + ReLU backward
            dy1 = ws.get("bwd.dy1", (Min, planes), BF16)
            self._bn_bwd(da1, None, rec["y1"], rec["bnp1"], name + ".bn1", Min, planes, dy1, mask_from_y=1, sums=sums1)
            # ---- conv1 (1x1): wgrad + dgrad (+ shortcut gradient)
            self._wgrad(dy1, rec["x"], self.G(name + ".conv1.weight"), planes, Cin, Min)
            dx = ws.get(f"bwd.dx{scratch_i & 1}", (Min, Cin), BF16)
            scratch_i += 1
            w1 = self.W(name + ".conv1.weight").view(planes, Cin)
            if rec["has_ds"]:
                wd = self.W(name + ".downsample.0.weight").view(C4, Cin)
                if rec["xs"] is not None:
                    self._wgrad(dyd, rec["xs"], self.G(name + ".downsample.0.weight"), C4, Cin, Mout)
                else:  # one-tap implicit wgrad over the strided view of x, straight into the [C4, Cin, 1, 1] gradient
                    tiles = ((C4 + 127) // 128) * ((Cin + 255) // 256)
                    gemm(dyd, rec["x"], self.G(name + ".downsample.0.weight").view(C4, Cin), C4, Cin, Mout, atomic=True,
                         split_k=ops.split_k_for(tiles, (Mout + 63) // 64), lda=C4, ldb=Cin, conv=(B, Hc, Wc, Cin),
                         conv_mode=2, conv_stride=stride, conv_taps=1, out_f32=True)
                gemm(dy1, w1, dx, Min, Cin, planes, b_mn=1)
                if stride == 1:
                    gemm(dyd, wd, dx, Min, Cin, C4, b_mn=1, residual=dx)
                elif stride == 2 and rec["xs"] is None:
                    # dx[:, ::2, ::2] += dyd . Wd: one-tap implicit GEMM over the dyd grid whose output (and residual) is
                    # the even-position sub-grid of dx -- in-place accumulation, no dxs buffer, no upsample_add pass
                    gemm(dyd, self._packed[name + ".downsample.0.weight#t"], dx, Mout, Cin, C4, lda=C4,
                         conv=(B, Hn, Wn, C4), conv_mode=1, conv_taps=1, residual=dx, d_ptr=dx.data_ptr(),
                         out_view=((Hc + 1) // 2, (Wc + 1) // 2, 2 * Cin, 2 * Wc * Cin, Hc * Wc * Cin))
                else:
                    dxs = ws.get("bwd.dxs", (Mout, Cin), BF16)
                    gemm(dyd, wd, dxs, Mout, Cin, C4, b_mn=1)
                    call("vtx_upsample_add", dxs.data_ptr(), dx.data_ptr(), B, Hc, Wc, Cin, stride, s)
            else:
                # dx is the output gradient of the previous block: when that block has a single-branch bn3, its backward
                # sums (ReLU bit mask m3 of THAT block) are accumulated here, over the staged dx tiles
                prev = blocks[bi - 1] if bi > 0 else None
                bnr3 = None
                # (only for the large early-layer tensors: at layer3 / layer4 sizes the longer epilogue costs what the
                # stand-alone pass costs -- +42 us vs 44 us per launch at 50176 x 1024, profiles/r02n_*)
                if fuse and prev is not None and not prev["has_ds"] and Cin % 32 == 0 and Min >= self.fuse_bn3_min_rows:
                    sums3 = self._slab_take(2 * Cin)
                    bnr3 = (prev["y3"], prev["bnp3"], sums3, prev["m3"])
                gemm(dy1, w1, dx, Min, Cin, planes, b_mn=1, residual=dOut, residual_mask=rec["m3"], bnr=bnr3)
            dOut = dx
        # ---- stem: maxpool bwd -> ReLU/BN bwd -> wgrad
        st = tape["stem"]
        M0 = st["M"]
        da0 = ws.get("bwd.da0", (M0, 64), BF16)
        call("vtx_maxpool_bwd", dOut.data_ptr(), st["idx"].data_ptr(), da0.data_ptr(), B, st["Ho"], st["Wo"], 64, s)
        dy0 = ws.get("bwd.dy0", (M0, 64), BF16)
        self._bn_bwd(da0, None, st["y"], st["bnp"], "visual.cnn.bn1", M0, 64, dy0, mask_from_y=1)
        if stem_s2d:  # implicit wgrad over the space-to-depth view
            dwx = self._dwp["visual.cnn.conv1"].view(64, 256)
            gemm(dy0, st["s2d"], dwx, 64, 256, M0, lda=64, ldb=64, atomic=True, out_f32=True,
                 split_k=ops.split_k_for(1, M0 // 64), conv=(B, st["Ho"], st["Wo"], 64), conv_mode=6)
        else:
            dwp0 = self._dwp["visual.cnn.conv1"][:64 * 160].view(64, 160)
            self._wgrad(dy0, st["cols"], dwp0, 64, 160, M0)
        # layer1's 3x3 weight gradients + the stem's, in one launch (the 'rest' all-reduce bucket follows)
        self._run_jobs("unpack:rest:" + ("s2d" if stem_s2d else "cols"), lambda: self._unpack_rows("rest", stem_s2d))

    # ------------------------------------------------------------------------------------------------ head
    def _head_modules(self, direction):
        return self.textual if direction == "textual" else self.backward_textual

    def visual_projection_forward(self, feat, S):
        """mem[S,H] = feat[S,Cv] . Wvp^T + b   (computed once, shared by both directions)."""
        H = self.textual.hidden_size
        mem = self.ws.get("head.mem", (S, H), BF16)
        gemm(feat, self.W("textual.visual_projection.weight"), mem, S, H, feat.shape[1],
             bias=self.P("textual.visual_projection.bias"))
        return mem

    def head_forward(self, direction, mem, tokens, lengths, training, want_logits_f32=False):
        """tokens int64 [B,T] -> bf16 logits [B*T, V] (and the tape for backward)."""
        mod = self._head_modules(direction)
        B, T = tokens.shape
        M, H, Fd, V, A = B * T, mod.hidden_size, mod.feedforward_size, mod.vocab_size, mod.attention_heads
        S = mem.shape[0]
        Sk = S // B
        p = float(mod.dropout) if training else 0.0
        d = direction
        di = 0 if d == "textual" else 1
        # self-attention mask: 1 = future + key padding (captioning), 2 = key padding only (masked language modelling)
        self._mask_mode = mm = 1 if mod.mask_future_positions else 2
        s = _stream()
        ws = self.ws
        seed = self.seed.data_ptr()
        site = di * 1000
        rec = dict(direction=d, B=B, T=T, M=M, S=S, Sk=Sk, p=p, layers=[], tokens=tokens, lengths=lengths, mem=mem,
                   mask_mode=mm)
        emb = "textual.embedding."
        z0 = ws.get(d + ".z0", (M, H), F32)
        st0 = ws.get(d + ".st0", (M, 2), F32)
        x = ws.get(d + ".x0", (M, H), F32)
        xb = ws.get(d + ".x0b", (M, H), BF16)
        call("vtx_embed_fwd", tokens.data_ptr(), self.P(emb + "words.weight").data_ptr(),
             self.P(emb + "positions.weight").data_ptr(), self.P(emb + "layer_norm.weight").data_ptr(),
             self.P(emb + "layer_norm.bias").data_ptr(), z0.data_ptr(), st0.data_ptr(), x.data_ptr(), xb.data_ptr(),
             M, T, H, self.pad, 1e-8, p, seed, site, s)
        rec.update(z0=z0, st0=st0)
        for l in range(mod.num_layers):
            q = f"{d}.transformer.layers.{l}."
            k = f"{d}.L{l}."
            sb = site + 10 * (l + 1)
            if mod.norm_first:
                x = self._prenorm_layer_forward(rec, q, k, sb, x, mem, lengths, p, B, T, A, H, Fd, S, Sk)
                continue
            lr = dict(q=q, x_in=x, x_inb=xb)
            # self-attention block
            qkv = ws.get(k + "qkv", (M, 3 * H), BF16)
            gemm(xb, self.W(q + "self_attn.in_proj_weight"), qkv, M, 3 * H, H, bias=self.P(q + "self_attn.in_proj_bias"))
            o_s = ws.get(k + "o_s", (M, H), BF16)
            lse_s = ws.get(k + "lse_s", (B * A * 32,), F32)
            e = qkv.element_size()
            call("vtx_attn_fwd", qkv.data_ptr(), 3 * H, qkv.data_ptr() + H * e, 3 * H, qkv.data_ptr() + 2 * H * e,
                 3 * H, o_s.data_ptr(), H, lse_s.data_ptr(), B, A, T, T, lengths.data_ptr(), mm, p, seed, sb + 0, s)
            pr = ws.get(k + "proj", (M, H), BF16)
            gemm(o_s, self.W(q + "self_attn.out_proj.weight"), pr, M, H, H, bias=self.P(q + "self_attn.out_proj.bias"))
            z1, st1 = ws.get(k + "z1", (M, H), F32), ws.get(k + "st1", (M, 2), F32)
            x1, x1b = ws.get(k + "x1", (M, H), F32), ws.get(k + "x1b", (M, H), BF16)
            call("vtx_add_ln_fwd", x.data_ptr(), pr.data_ptr(), self.P(q + "norm1.weight").data_ptr(),
                 self.P(q + "norm1.bias").data_ptr(), z1.data_ptr(), st1.data_ptr(), x1.data_ptr(), x1b.data_ptr(), M,
                 H, 1e-5, p, seed, sb + 1, 1, s)
            # cross-attention block
            wc, bc = self.W(q + "multihead_attn.in_proj_weight"), self.P(q + "multihead_attn.in_proj_bias")
            qc = ws.get(k + "qc", (M, H), BF16)
            gemm(x1b, wc[:H], qc, M, H, H, bias=bc[:H])
            kv = ws.get(k + "kv", (S, 2 * H), BF16)
            gemm(mem, wc[H:], kv, S, 2 * H, H, bias=bc[H:])
            o_c = ws.get(k + "o_c", (M, H), BF16)
            lse_c = ws.get(k + "lse_c", (B * A * 32,), F32)
            call("vtx_attn_fwd", qc.data_ptr(), H, kv.data_ptr(), 2 * H, kv.data_ptr() + H * e, 2 * H, o_c.data_ptr(),
                 H, lse_c.data_ptr(), B, A, T, Sk, 0, 0, p, seed, sb + 2, s)
            gemm(o_c, self.W(q + "multihead_attn.out_proj.weight"), pr, M, H, H,
                 bias=self.P(q + "multihead_attn.out_proj.bias"))
            z2, st2 = ws.get(k + "z2", (M, H), F32), ws.get(k + "st2", (M, 2), F32)
            x2, x2b = ws.get(k + "x2", (M, H), F32), ws.get(k + "x2b", (M, H), BF16)
            call("vtx_add_ln_fwd", x1.data_ptr(), pr.data_ptr(), self.P(q + "norm2.weight").data_ptr(),
                 self.P(q + "norm2.bias").data_ptr(), z2.data_ptr(), st2.data_ptr(), x2.data_ptr(), x2b.data_ptr(), M,
                 H, 1e-5, p, seed, sb + 3, 1, s)
            # feed-forward block
            u = ws.get(k + "u", (M, Fd), BF16)
            gemm(x2b, self.W(q + "linear1.weight"), u, M, Fd, H, bias=self.P(q + "linear1.bias"))
            h = ws.get(k + "h", (M, Fd), BF16)
            call("vtx_gelu_dropout_fwd", u.data_ptr(), h.data_ptr(), M * Fd, p, seed, sb + 4, s)
            gemm(h, self.W(q + "linear2.weight"), pr, M, H, Fd, bias=self.P(q + "linear2.bias"))
            z3, st3 = ws.get(k + "z3", (M, H), F32), ws.get(k + "st3", (M, 2), F32)
            x3, x3b = ws.get(k + "x3", (M, H), F32), ws.get(k + "x3b", (M, H), BF16)
            call("vtx_add_ln_fwd", x2.data_ptr(), pr.data_ptr(), self.P(q + "norm3.weight").data_ptr(),
                 self.P(q + "norm3.bias").data_ptr(), z3.data_ptr(), st3.data_ptr(), x3.data_ptr(), x3b.data_ptr(), M,
                 H, 1e-5, p, seed, sb + 5, 1, s)
            lr.update(qkv=qkv, o_s=o_s, lse_s=lse_s, z1=z1, st1=st1, x1b=x1b, qc=qc, kv=kv, o_c=o_c, lse_c=lse_c,
                      z2=z2, st2=st2, x2b=x2b, u=u, h=h, z3=z3, st3=st3, sb=sb)
            rec["layers"].append(lr)
            x, xb = x3, x3b
        if mod.norm_first:  # final LayerNorm of pre-norm decoders (textual_heads.py:192-193)
            qn = f"{d}.transformer.norm."
            zf, stf = ws.get(d + ".zf", (M, H), F32), ws.get(d + ".stf", (M, 2), F32)
            xb = ws.get(d + ".xfb", (M, H), BF16)
            call("vtx_add_ln_fwd", x.data_ptr(), 0, self.P(qn + "weight").data_ptr(), self.P(qn + "bias").data_ptr(),
                 zf.data_ptr(), stf.data_ptr(), 0, xb.data_ptr(), M, H, 1e-5, 0.0, seed, 0, 1, s)
            rec.update(zf=zf, stf=stf)
        rec["x_out_b"] = xb
        # tied output projection
        wv = self.W("textual.embedding.words.weight")
        bo = self.P("textual.output.bias")
        if want_logits_f32:
            lf = ws.get(d + ".logits_f32", (M, V), F32)
            gemm(xb, wv, lf, M, V, H, bias=bo)
            rec["logits_f32"] = lf
        logits = ws.get(d + ".logits", (M, V), BF16)
        gemm(xb, wv, logits, M, V, H, bias=bo)
        rec["logits"] = logits
        return rec

    def _prenorm_layer_forward(self, rec, q, k, sb, x, mem, lengths, p, B, T, A, H, Fd, S, Sk):
        """x + f(LN(x)) for the three blocks (torch/nn/modules/transformer.py:1131-1143); returns the new fp32 x."""
        s, ws, seed = _stream(), self.ws, self.seed.data_ptr()
        M = B * T
        e = 2
        lr = dict(q=q, sb=sb, x0=x)

        def norm(name, xin, tag):
            z, st = ws.get(k + "z" + tag, (M, H), F32), ws.get(k + "st" + tag, (M, 2), F32)
            nb = ws.get(k + "n" + tag + "b", (M, H), BF16)
            call("vtx_add_ln_fwd", xin.data_ptr(), 0, self.P(q + name + ".weight").data_ptr(),
                 self.P(q + name + ".bias").data_ptr(), z.data_ptr(), st.data_ptr(), 0, nb.data_ptr(), M, H, 1e-5, 0.0,
                 seed, 0, 1, s)
            return z, st, nb

        def residual(xin, branch, tag, site):
            xo = ws.get(k + "x" + tag, (M, H), F32)
            call("vtx_add_ln_fwd", xin.data_ptr(), branch.data_ptr(), 0, 0, xo.data_ptr(), 0, 0, 0, M, H, 0.0, p, seed,
                 site, 0, s)
            return xo

        pr = ws.get(k + "proj", (M, H), BF16)
        # self attention
        z1, st1, n1b = norm("norm1", x, "1")
        qkv = ws.get(k + "qkv", (M, 3 * H), BF16)
        gemm(n1b, self.W(q + "self_attn.in_proj_weight"), qkv, M, 3 * H, H, bias=self.P(q + "self_attn.in_proj_bias"))
        o_s = ws.get(k + "o_s", (M, H), BF16)
        lse_s = ws.get(k + "lse_s", (B * A * 32,), F32)
        call("vtx_attn_fwd", qkv.data_ptr(), 3 * H, qkv.data_ptr() + H * e, 3 * H, qkv.data_ptr() + 2 * H * e, 3 * H,
             o_s.data_ptr(), H, lse_s.data_ptr(), B, A, T, T, lengths.data_ptr(), rec["mask_mode"], p, seed, sb + 0, s)
        gemm(o_s, self.W(q + "self_attn.out_proj.weight"), pr, M, H, H, bias=self.P(q + "self_attn.out_proj.bias"))
        x1 = residual(x, pr, "1", sb + 1)
        # cross attention
        z2, st2, n2b = norm("norm2", x1, "2")
        wc, bc = self.W(q + "multihead_attn.in_proj_weight"), self.P(q + "multihead_attn.in_proj_bias")
        qc = ws.get(k + "qc", (M, H), BF16)
        gemm(n2b, wc[:H], qc, M, H, H, bias=bc[:H])
        kv = ws.get(k + "kv", (S, 2 * H), BF16)
        gemm(mem, wc[H:], kv, S, 2 * H, H, bias=bc[H:])
        o_c = ws.get(k + "o_c", (M, H), BF16)
        lse_c = ws.get(k + "lse_c", (B * A * 32,), F32)
        call("vtx_attn_fwd", qc.data_ptr(), H, kv.data_ptr(), 2 * H, kv.data_ptr() + H * e, 2 * H, o_c.data_ptr(), H,
             lse_c.data_ptr(), B, A, T, Sk, 0, 0, p, seed, sb + 2, s)
        gemm(o_c, self.W(q + "multihead_attn.out_proj.weight"), pr, M, H, H,
             bias=self.P(q + "multihead_attn.out_proj.bias"))
        x2 = residual(x1, pr, "2", sb + 3)
        # feed forward
        z3, st3, n3b = norm("norm3", x2, "3")
        u = ws.get(k + "u", (M, Fd), BF16)
        gemm(n3b, self.W(q + "linear1.weight"), u, M, Fd, H, bias=self.P(q + "linear1.bias"))
        h = ws.get(k + "h", (M, Fd), BF16)
        call("vtx_gelu_dropout_fwd", u.data_ptr(), h.data_ptr(), M * Fd, p, seed, sb + 4, s)
        gemm(h, self.W(q + "linear2.weight"), pr, M, H, Fd, bias=self.P(q + "linear2.bias"))
        x3 = residual(x2, pr, "3", sb + 5)
        lr.update(z1=z1, st1=st1, n1b=n1b, qkv=qkv, o_s=o_s, lse_s=lse_s, z2=z2, st2=st2, n2b=n2b, qc=qc, kv=kv, o_c=o_c,
                  lse_c=lse_c, z3=z3, st3=st3, n3b=n3b, u=u, h=h)
        rec["layers"].append(lr)
        return x3

    def _prenorm_layer_backward(self, rec, lr, g, dmem, dmem_started, mod):
        """g = dL/dx_out (fp32 [M,H], updated in place to dL/dx_in)."""
        B, T, M, S, Sk, p = rec["B"], rec["T"], rec["M"], rec["S"], rec["Sk"], rec["p"]
        H, Fd, A = mod.hidden_size, mod.feedforward_size, mod.attention_heads
        s, ws, seed = _stream(), self.ws, self.seed.data_ptr()
        q, sb = lr["q"], lr["sb"]
        e = 2
        dbr = ws.get("hb.dbr", (M, H), BF16)
        dxb = ws.get("hb.dxb", (M, H), BF16)
        do = ws.get("hb.do", (M, H), BF16)

        def branch_grad(site):  # d(branch) = g * dropout mask (bf16); g itself keeps flowing through the skip path
            call("vtx_ln_bwd", g.data_ptr(), 0, 0, 0, 0, 0, 0, dbr.data_ptr(), 0, 0, M, H, p, seed, site, 0, s)

        def norm_bwd(name, z, st, dn):  # g += LN_backward(dn)
            call("vtx_ln_bwd", 0, dn.data_ptr(), z.data_ptr(), st.data_ptr(), self.P(q + name + ".weight").data_ptr(),
                 g.data_ptr(), g.data_ptr(), 0, self.G(q + name + ".weight").data_ptr(),
                 self.G(q + name + ".bias").data_ptr(), M, H, 0.0, seed, 0, 1, s)

        # feed forward
        branch_grad(sb + 5)
        dh = ws.get("hb.dh", (M, Fd), BF16)
        self._linear_bwd(dbr, lr["h"], q + "linear2.weight", q + "linear2.bias", dh, M, H, Fd)
        call("vtx_gelu_dropout_bwd", dh.data_ptr(), lr["u"].data_ptr(), dh.data_ptr(), M * Fd, p, seed, sb + 4, s)
        self._linear_bwd(dh, lr["n3b"], q + "linear1.weight", q + "linear1.bias", dxb, M, Fd, H)
        norm_bwd("norm3", lr["z3"], lr["st3"], dxb)
        # cross attention
        branch_grad(sb + 3)
        self._linear_bwd(dbr, lr["o_c"], q + "multihead_attn.out_proj.weight", q + "multihead_attn.out_proj.bias", do,
                         M, H, H)
        dqc = ws.get("hb.dqc", (M, H), BF16)
        dkv = ws.get("hb.dkv", (S, 2 * H), BF16)
        kv = lr["kv"]
        call("vtx_attn_bwd", lr["qc"].data_ptr(), H, kv.data_ptr(), 2 * H, kv.data_ptr() + H * e, 2 * H, do.data_ptr(),
             H, lr["lse_c"].data_ptr(), dqc.data_ptr(), H, dkv.data_ptr(), 2 * H, dkv.data_ptr() + H * e, 2 * H, B, A, T,
             Sk, 0, 0, p, seed, sb + 2, s)
        wn, bn = q + "multihead_attn.in_proj_weight", q + "multihead_attn.in_proj_bias"
        self._linear_bwd(dqc, lr["n2b"], wn, bn, dxb, M, H, H, w_rows=slice(0, H))
        self._linear_bwd(dkv, rec["mem"], wn, bn, dmem, S, 2 * H, H, w_rows=slice(H, 3 * H),
                         residual=dmem if dmem_started else None)
        norm_bwd("norm2", lr["z2"], lr["st2"], dxb)
        # self attention
        branch_grad(sb + 1)
        self._linear_bwd(dbr, lr["o_s"], q + "self_attn.out_proj.weight", q + "self_attn.out_proj.bias", do, M, H, H)
        dqkv = ws.get("hb.dqkv", (M, 3 * H), BF16)
        qkv = lr["qkv"]
        call("vtx_attn_bwd", qkv.data_ptr(), 3 * H, qkv.data_ptr() + H * e, 3 * H, qkv.data_ptr() + 2 * H * e, 3 * H,
             do.data_ptr(), H, lr["lse_s"].data_ptr(), dqkv.data_ptr(), 3 * H, dqkv.data_ptr() + H * e, 3 * H,
             dqkv.data_ptr() + 2 * H * e, 3 * H, B, A, T, T, rec["lengths"].data_ptr(), rec["mask_mode"], p, seed, sb + 0,
             s)
        self._linear_bwd(dqkv, lr["n1b"], q + "self_attn.in_proj_weight", q + "self_attn.in_proj_bias", dxb, M, 3 * H, H)
        norm_bwd("norm1", lr["z1"], lr["st1"], dxb)

    def head_loss(self, rec, write_grad, labels=None):
        """Token-mean cross entropy (ignore_index = pad).  labels None: next-token targets tokens[:, 1:] against
        logits[:, :-1] (captioning.py:111-114); labels [B,T]: one label per position (masked_lm.py:68-72)."""
        di = 0 if rec["direction"] == "textual" else 1
        s = _stream()
        V = rec["logits"].shape[1]
        tgt, shift = (rec["tokens"], 1) if labels is None else (labels, 0)
        call("vtx_count_valid", tgt.data_ptr(), rec["B"], rec["T"], self.pad, shift, self.count[di:].data_ptr(), s)
        call("vtx_cross_entropy", rec["logits"].data_ptr(), V, tgt.data_ptr(), rec["B"], rec["T"], V, self.pad, shift,
             self.count[di:].data_ptr(), self.loss[di:].data_ptr(), int(write_grad), s)

    def _linear_bwd(self, dY, X, wname, bname, dX, M, n_out, k_in, w_rows=None, residual=None):
        """Backward of Y = X W^T + b for W [n_out, k_in] (optionally the row slice `w_rows` of a packed weight)."""
        W, dW, db = self.W(wname), self.G(wname), self.G(bname)
        if w_rows is not None:
            W, dW, db = W[w_rows], dW[w_rows], db[w_rows]
        call("vtx_colsum", dY.data_ptr(), dY.stride(0), M, n_out, db.data_ptr(), _stream())
        self._wgrad(dY, X, dW, n_out, k_in, M)
        if dX is not None:
            gemm(dY, W, dX, M, k_in, n_out, b_mn=1, residual=residual)

    def head_backward(self, rec, dmem, dmem_started):
        """Backward of one direction from the dlogits already written in place of rec['logits'].
        Accumulates parameter gradients; adds this direction's contribution to dmem [S,H]."""
        d = rec["direction"]
        mod = self._head_modules(d)
        B, T, M, S, Sk, p = rec["B"], rec["T"], rec["M"], rec["S"], rec["Sk"], rec["p"]
        H, Fd, V, A = mod.hidden_size, mod.feedforward_size, mod.vocab_size, mod.attention_heads
        s = _stream()
        ws = self.ws
        seed = self.seed.data_ptr()
        dlog = rec["logits"]
        # tied output projection: d_bias, d_words (vocab-projection part), dx
        call("vtx_colsum", dlog.data_ptr(), V, M, V, self.G("textual.output.bias").data_ptr(), s)
        self._wgrad(dlog, rec["x_out_b"], self.G("textual.embedding.words.weight"), V, H, M)
        dxb = ws.get("hb.dxb", (M, H), BF16)
        gemm(dlog, self.W("textual.embedding.words.weight"), dxb, M, H, V, b_mn=1)
        dres_a = ws.get("hb.dres_a", (M, H), F32)
        dres_b = ws.get("hb.dres_b", (M, H), F32)
        dbr = ws.get("hb.dbr", (M, H), BF16)
        dy_a, dy_b = None, dxb
        e = 2
        if mod.norm_first:
            qn = f"{d}.transformer.norm."
            g = dres_a
            call("vtx_ln_bwd", 0, dxb.data_ptr(), rec["zf"].data_ptr(), rec["stf"].data_ptr(),
                 self.P(qn + "weight").data_ptr(), 0, g.data_ptr(), 0, self.G(qn + "weight").data_ptr(),
                 self.G(qn + "bias").data_ptr(), M, H, 0.0, seed, 0, 1, s)
            for l in reversed(range(mod.num_layers)):
                self._prenorm_layer_backward(rec, rec["layers"][l], g, dmem, dmem_started, mod)
                dmem_started = True
            dy_a, dy_b = g, None
        for l in (reversed(range(mod.num_layers)) if not mod.norm_first else ()):
            lr = rec["layers"][l]
            q, sb = lr["q"], lr["sb"]
            # LN3 / FFN
            call("vtx_ln_bwd", _p(dy_a), _p(dy_b), lr["z3"].data_ptr(), lr["st3"].data_ptr(),
                 self.P(q + "norm3.weight").data_ptr(), 0, dres_a.data_ptr(), dbr.data_ptr(),
                 self.G(q + "norm3.weight").data_ptr(), self.G(q + "norm3.bias").data_ptr(), M, H, p, seed, sb + 5, 1, s)
            dh = ws.get("hb.dh", (M, Fd), BF16)
            self._linear_bwd(dbr, lr["h"], q + "linear2.weight", q + "linear2.bias", dh, M, H, Fd)
            call("vtx_gelu_dropout_bwd", dh.data_ptr(), lr["u"].data_ptr(), dh.data_ptr(), M * Fd, p, seed, sb + 4, s)
            self._linear_bwd(dh, lr["x2b"], q + "linear1.weight", q + "linear1.bias", dxb, M, Fd, H)
            # LN2 / cross attention
            call("vtx_ln_bwd", dres_a.data_ptr(), dxb.data_ptr(), lr["z2"].data_ptr(), lr["st2"].data_ptr(),
                 self.P(q + "norm2.weight").data_ptr(), 0, dres_b.data_ptr(), dbr.data_ptr(),
                 self.G(q + "norm2.weight").data_ptr(), self.G(q + "norm2.bias").data_ptr(), M, H, p, seed, sb + 3, 1, s)
            do = ws.get("hb.do", (M, H), BF16)
            self._linear_bwd(dbr, lr["o_c"], q + "multihead_attn.out_proj.weight", q + "multihead_attn.out_proj.bias",
                             do, M, H, H)
            dqc = ws.get("hb.dqc", (M, H), BF16)
            dkv = ws.get("hb.dkv", (S, 2 * H), BF16)
            kv = lr["kv"]
            call("vtx_attn_bwd", lr["qc"].data_ptr(), H, kv.data_ptr(), 2 * H, kv.data_ptr() + H * e, 2 * H,
                 do.data_ptr(), H, lr["lse_c"].data_ptr(), dqc.data_ptr(), H, dkv.data_ptr(), 2 * H,
                 dkv.data_ptr() + H * e, 2 * H, B, A, T, Sk, 0, 0, p, seed, sb + 2, s)
            wn, bn = q + "multihead_attn.in_proj_weight", q + "multihead_attn.in_proj_bias"
            self._linear_bwd(dqc, lr["x1b"], wn, bn, dxb, M, H, H, w_rows=slice(0, H))
            self._linear_bwd(dkv, rec["mem"], wn, bn, dmem, S, 2 * H, H, w_rows=slice(H, 3 * H),
                             residual=dmem if dmem_started else None)
            dmem_started = True
            # LN1 / self attention
            call("vtx_ln_bwd", dres_b.data_ptr(), dxb.data_ptr(), lr["z1"].data_ptr(), lr["st1"].data_ptr(),
                 self.P(q + "norm1.weight").data_ptr(), 0, dres_a.data_ptr(), dbr.data_ptr(),
                 self.G(q + "norm1.weight").data_ptr(), self.G(q + "norm1.bias").data_ptr(), M, H, p, seed, sb + 1, 1, s)
            self._linear_bwd(dbr, lr["o_s"], q + "self_attn.out_proj.weight", q + "self_attn.out_proj.bias", do, M, H, H)
            dqkv = ws.get("hb.dqkv", (M, 3 * H), BF16)
            qkv = lr["qkv"]
            call("vtx_attn_bwd", qkv.data_ptr(), 3 * H, qkv.data_ptr() + H * e, 3 * H, qkv.data_ptr() + 2 * H * e,
                 3 * H, do.data_ptr(), H, lr["lse_s"].data_ptr(), dqkv.data_ptr(), 3 * H, dqkv.data_ptr() + H * e,
                 3 * H, dqkv.data_ptr() + 2 * H * e, 3 * H, B, A, T, T, rec["lengths"].data_ptr(), rec["mask_mode"], p, seed,
                 sb + 0, s)
            self._linear_bwd(dqkv, lr["x_inb"], q + "self_attn.in_proj_weight", q + "self_attn.in_proj_bias", dxb, M,
                             3 * H, H)
            dy_a, dy_b = dres_a, dxb
        emb = "textual.embedding."
        di = 0 if d == "textual" else 1
        call("vtx_embed_bwd", _p(dy_a), _p(dy_b), rec["tokens"].data_ptr(), rec["z0"].data_ptr(),
             rec["st0"].data_ptr(), self.P(emb + "layer_norm.weight").data_ptr(),
             self.G(emb + "words.weight").data_ptr(), self.G(emb + "positions.weight").data_ptr(),
             self.G(emb + "layer_norm.weight").data_ptr(), self.G(emb + "layer_norm.bias").data_ptr(), M, T, H,
             self.pad, p, seed, di * 1000, s)
        return dmem_started

    # ------------------------------------------------------------------------------------------------ classification
    def _pool_linear(self, feat, B, S):
        """feat bf16 [B*S, C] -> pooled bf16 [B, C] (global average pooling) -> fp32 logits [B, ldl], ldl = V rounded up
        to 8 (16-byte rows for the fp32 logits and for the bf16 dlogits that share the width)."""
        C, V = feat.shape[1], self.textual.vocab_size
        ldl = _round_up(V, 8)
        pooled = self.ws.get("clf.pooled", (B, C), BF16)
        call("vtx_avgpool_fwd", feat.data_ptr(), pooled.data_ptr(), B, S, C, _stream())
        logits = self.ws.get("clf.logits", (B, ldl), F32)
        gemm(pooled, self.W("textual.output.weight"), logits, B, V, C, ldd=ldl, bias=self.P("textual.output.bias"))
        return pooled, logits, ldl

    def _classify(self, feat, B, S, labels, with_grad):
        """Pool + linear + K-hot loss (virtex/models/classification.py:69-100) into self.loss[0]; leaves the bf16
        dlogits for backward when `with_grad`."""
        if labels is None or labels.dim() != 2 or labels.shape[0] != B or labels.dtype != torch.int64:
            raise ValueError("a classification batch needs 'labels', int64 (B, L)")
        if labels.device != self.device:
            raise RuntimeError("virtex_b200 has no CPU path: the labels must live on the model's CUDA device")
        V = self.textual.vocab_size
        pooled, logits, ldl = self._pool_linear(feat, B, S)
        dlog = self.ws.get("clf.dlogits", (B, ldl), BF16) if with_grad else None
        labels = labels.contiguous()
        L = labels.shape[1]
        call("vtx_khot_xent", logits.data_ptr(), ldl, labels.data_ptr(), L, _p(self.ignore), self.ignore.numel(), B, V,
             self.loss.data_ptr(), _p(dlog), ldl, _stream())
        return dict(B=B, S=S, V=V, ldl=ldl, feat=feat, pooled=pooled, logits=logits, dlog=dlog)

    def _classify_backward(self, bucket_cb):
        """Output layer (db by column sums, dW, dpooled fp32) -> pool backward -> backbone backward."""
        c = self._clf
        B, S, V = c["B"], c["S"], c["V"]
        C = c["pooled"].shape[1]
        frozen = getattr(self.visual, "frozen", False)
        dpooled = None if frozen else self.ws.get("clf.dpooled", (B, C), F32)
        self._linear_bwd(c["dlog"][:, :V], c["pooled"], "textual.output.weight", "textual.output.bias", dpooled, B, V, C)
        if bucket_cb is not None:
            bucket_cb("head")
        if not frozen:
            dfeat = self.ws.get("hb.dfeat", (B * S, C), BF16)
            call("vtx_avgpool_bwd", dpooled.data_ptr(), dfeat.data_ptr(), B, S, C, _stream())
            self.backbone_backward(dfeat, bucket_cb)
        if bucket_cb is not None:
            bucket_cb("rest")

    def linear_logits(self, visual_features):
        """`LinearTextualHead.forward`: (B,C,h,w) -> fp32 logits view (B,V)."""
        B, C, h, w = visual_features.shape
        feat = visual_features.permute(0, 2, 3, 1).reshape(B * h * w, C).to(BF16).contiguous()
        _, logits, _ = self._pool_linear(feat, B, h * w)
        return logits[:, :self.textual.vocab_size]

    # ------------------------------------------------------------------------------------------------ full model
    def forward(self, image, tokens, noitpac, lengths, training=True, with_grad=True, labels=None):
        """Loss of the bicaptioning model (labels None) or of the masked-LM sibling (labels = masked_labels [B,T], single
        direction).  Leaves dlogits in the logits buffers when `with_grad`.  With a LinearTextualHead: the K-hot loss of
        labels [B, L] (tokens / noitpac / lengths unused) in loss[0]."""
        if not self.arena.intact():
            raise RuntimeError("model parameters were moved after the engine adopted them; rebuild the engine")
        self.generation += 1
        self.loss.zero_()
        self.count.zero_()
        # BatchNorm follows the backbone's OWN mode flag, like the reference's nn.BatchNorm2d: `model.train()` puts a
        # frozen backbone's BN back into batch-statistics mode (visual_backbones.py:48-52 only calls .eval() once)
        bn_training = bool(self.visual.cnn.training) if self.visual is not None else training
        feat, h, w = self.backbone_forward(image, bn_training)
        if self.classification:
            self._clf = self._classify(feat, image.shape[0], h * w, labels, with_grad)
            return self.loss
        B = image.shape[0]
        S = B * h * w
        mem = self.visual_projection_forward(feat, S)
        recs = [self.head_forward("textual", mem, tokens, lengths, training, want_logits_f32=not training)]
        self.head_loss(recs[0], with_grad, labels)
        if self.backward_textual is not None:
            recs.append(self.head_forward("backward_textual", mem, noitpac, lengths, training))
            self.head_loss(recs[1], with_grad)
        self._recs, self._mem, self._feat = recs, mem, feat
        return self.loss

    def backward(self, zero_grads=True, bucket_cb=None):
        """Gradients of (loss_fwd + loss_bwd) w.r.t. every parameter into the flat gradient arena.
        `bucket_cb(tag)`, tag in {'head_b','head','layer4','layer3','layer2','rest'}, fires as gradient ranges complete (in
        backward order) so a data-parallel all-reduce can overlap the remaining backward."""
        if zero_grads:
            self.arena.grads.zero_()
        if self.classification:
            self._classify_backward(bucket_cb)
            return
        feat, mem = self._feat, self._mem
        S, H = mem.shape
        dmem = self.ws.get("hb.dmem", (S, H), BF16)
        started = False
        for rec in reversed(self._recs):
            started = self.head_backward(rec, dmem, started)
            if bucket_cb is not None and rec["direction"] == "backward_textual":
                bucket_cb("head_b")  # only this direction writes the backward_textual.* gradients
        Cv = feat.shape[1]
        dfeat = self.ws.get("hb.dfeat", (S, Cv), BF16)
        frozen = getattr(self.visual, "frozen", False)
        self._linear_bwd(dmem, feat, "textual.visual_projection.weight", "textual.visual_projection.bias",
                         None if frozen else dfeat, S, H, Cv)
        if bucket_cb is not None:
            bucket_cb("head")
        if not frozen:
            self.backbone_backward(dfeat, bucket_cb)
        if bucket_cb is not None:
            bucket_cb("rest")

    def predictions(self):
        """argmax over the fp32 forward-direction logits of the last eval-mode forward -> int64 [B,T]; for a
        classification head the top 10 of the logits, best first -> int64 [B, 10]."""
        if self.classification:
            c = self._clf
            out = self.ws.get("clf.top10", (c["B"], 10), torch.int64)
            call("vtx_topk_rows", c["logits"].data_ptr(), c["ldl"], c["B"], c["V"], 10, out.data_ptr(), _stream())
            return out
        rec = self._recs[0]
        lf = rec["logits_f32"]
        out = self.ws.get("pred", (rec["M"],), torch.int64)
        call("vtx_argmax_rows", lf.data_ptr(), lf.stride(0), rec["M"], lf.shape[1], out.data_ptr(), _stream())
        return out.view(rec["B"], rec["T"])

    # ------------------------------------------------------------------------------------------------ decoding
    def visual_features(self, image):
        """Backbone forward in the backbone's own BN mode -> (B, C, h, w) fp32, the reference's `visual(image)`."""
        feat, h, w = self.backbone_forward(image.contiguous().float(), bool(self.visual.cnn.training))
        B, C = image.shape[0], feat.shape[1]
        out = torch.empty(B, C, h, w, dtype=F32, device=image.device)
        call("vtx_nhwc_to_nchw_f32", feat.data_ptr(), out.data_ptr(), B, h * w, C, _stream())
        return out

    def head_logits(self, visual_features, tokens, lengths, training=False):
        """Forward-direction textual head over whole captions: (B,C,h,w), (B,T), (B,) -> fp32 logits view (B,T,V)."""
        B, C, h, w = visual_features.shape
        feat = visual_features.permute(0, 2, 3, 1).reshape(B * h * w, C).to(BF16).contiguous()
        mem = self.visual_projection_forward(feat, B * h * w)
        rec = self.head_forward("textual", mem, tokens.contiguous(), lengths.contiguous(), training=training,
                                want_logits_f32=True)
        return rec["logits_f32"].view(B, tokens.shape[1], -1)

    def decode(self, image, sos, eos, beam_size=5, per_node=2, max_steps=30, only_return_best=True, training=False):
        """Beam-search captions of `image` (virtex/models/captioning.py:144-163 with utils/beam_search.py).

        The backbone and the visual projection run once, the cross-attention keys / values once per layer for the B
        images (never repeated per beam).  Step 1 runs the head on B rows of [SOS]; steps 2... run it on the B * beam
        rows for ONE new position each (the reference re-runs the whole prefix, without [SOS]): the keys / values of
        earlier positions come from a position-major cache written by the QKV GEMM, and a per-row index table that
        follows the selected parents decides whose history each row attends to.  Moving that int32 index costs
        rows * t * 4 bytes per step; gathering the caches themselves would read and write rows * t * 3H * 2 bytes per
        layer (450 MB at t = 29, H = 1024, 1280 rows).  One host synchronisation per step (the ended flag).
        Returns (predictions, scores) like AutoRegressiveBeamSearch.search."""
        if training:
            raise RuntimeError("beam-search decoding runs in eval mode only (call model.eval()): the reference would "
                               "decode with dropout active, which cannot be reproduced")
        mod = self.textual
        if mod is None or not mod.mask_future_positions:
            raise RuntimeError("decoding needs a forward-direction captioning head (mask_future_positions=True)")
        B = image.shape[0]
        per_node = per_node or beam_size
        T_cache = max(max_steps - 1, 1)  # positions 0 .. max_steps - 2 (step 1's [SOS] is not reused)
        max_pos = self.P("textual.embedding.positions.weight").shape[0]
        # the limits of vtx_decode_attn / vtx_beam_step, checked before the backbone runs
        if max_steps < 1 or T_cache > min(max_pos, 64):
            raise ValueError(f"max_steps = {max_steps} needs {T_cache} positions; the decoder has {max_pos} (at most 64)")
        if not 1 <= beam_size <= 8:
            raise ValueError(f"beam_size = {beam_size}: the beam-selection kernel handles 1 to 8 beams")
        if not 1 <= per_node <= min(16, mod.vocab_size):
            raise ValueError(f"per_node_beam_size = {per_node}: the beam-selection kernel takes 1 to 16 per beam")
        h, w = image.shape[2], image.shape[3]
        for _ in range(5):  # stem conv (7x7/2, pad 3), max-pool (3x3/2, pad 1), layer2..4 (stride 2)
            h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
        if h * w > 64:
            raise ValueError(f"{image.shape[2]}x{image.shape[3]} images give {h * w} visual tokens; cross attention "
                             "while decoding takes at most 64 (8x8, images up to 256x256)")
        ws = self.ws
        rows_max = B * beam_size
        kvs, caches, Sk = self.decode_setup(image, rows_max, T_cache)
        st = BeamState(self.device, B, beam_size, per_node, eos, max_steps, with_table=True, ws=ws)
        start = ws.get("dec.start", (B,), torch.int64)
        start.fill_(sos)
        st.first(self._decode_logits(start, B, 0, 1, None, kvs, caches, Sk, T_cache))
        if beam_size == 1 and st.all_ended():
            return st.empty_result()
        for t in range(1, max_steps):
            if st.all_ended():
                break
            # position t - 1 holds each beam's newest token; positions < t - 1 are cached
            st.step(self._decode_logits(st.last_tokens, rows_max, t - 1, beam_size, st.cache_table, kvs, caches, Sk,
                                        T_cache))
        return st.result(only_return_best)

    def decode_setup(self, image, rows_max, T_cache):
        """Eval backbone + visual projection, then the cross-attention keys / values of every layer for the B images
        ([B * h * w, 2H] each) and empty self-attention caches [T_cache, rows_max, 3H] -> (kvs, caches, h * w)."""
        mod = self.textual
        H = mod.hidden_size
        feat, h, w = self.backbone_forward(image.contiguous().float(), bool(self.visual.cnn.training))
        S = image.shape[0] * h * w
        mem = self.visual_projection_forward(feat, S)
        kvs, caches = [], []
        for l in range(mod.num_layers):
            q = f"textual.transformer.layers.{l}."
            wc, bc = self.W(q + "multihead_attn.in_proj_weight"), self.P(q + "multihead_attn.in_proj_bias")
            kv = self.ws.get(f"dec.kv{l}", (S, 2 * H), BF16)
            gemm(mem, wc[H:], kv, S, 2 * H, H, bias=bc[H:])
            kvs.append(kv)
            caches.append(self.ws.get(f"dec.cache{l}", (T_cache, rows_max, 3 * H), BF16))
        return kvs, caches, h * w

    def _decode_logits(self, tokens, rows, pos, group, table, kvs, caches, Sk, T_cache):
        """fp32 logits [rows, V] of position `pos` of every row, whose token is tokens[row]; writes the position's
        Q/K/V into the caches.  group = rows per image."""
        mod = self.textual
        H, Fd, V, A = mod.hidden_size, mod.feedforward_size, mod.vocab_size, mod.attention_heads
        s, ws, seed = _stream(), self.ws, self.seed.data_ptr()
        M = rows
        emb = "textual.embedding."
        z, st_ = ws.get("dec.z", (M, H), F32), ws.get("dec.st", (M, 2), F32)
        x, xb = ws.get("dec.x0", (M, H), F32), ws.get("dec.x0b", (M, H), BF16)
        pos_ptr = self.P(emb + "positions.weight").data_ptr() + pos * H * 4  # T = 1: every row reads position `pos`
        call("vtx_embed_fwd", tokens.data_ptr(), self.P(emb + "words.weight").data_ptr(), pos_ptr,
             self.P(emb + "layer_norm.weight").data_ptr(), self.P(emb + "layer_norm.bias").data_ptr(), z.data_ptr(),
             st_.data_ptr(), x.data_ptr(), xb.data_ptr(), M, 1, H, self.pad, 1e-8, 0.0, seed, 0, s)
        pr = ws.get("dec.proj", (M, H), BF16)
        o = ws.get("dec.o", (M, H), BF16)
        qc = ws.get("dec.qc", (M, H), BF16)
        u = ws.get("dec.u", (M, Fd), BF16)
        hh = ws.get("dec.h", (M, Fd), BF16)
        nb = ws.get("dec.nb", (M, H), BF16)
        # residual stream: a layer reading buffer i writes x1 -> i+1, x2 -> i+2 and its output x3 -> i+1 (mod 3)
        bufs = [(x, xb), (ws.get("dec.xa", (M, H), F32), ws.get("dec.xab", (M, H), BF16)),
                (ws.get("dec.xc", (M, H), F32), ws.get("dec.xcb", (M, H), BF16))]
        ldt = table.stride(0) if table is not None else 0
        e = 2

        def add_ln(res, branch, name, out, out_b):
            """post-norm: out = LN(res + branch); branch None: out_b = LN(res) (pre-norm's normalised input);
            name None: out = res + branch (pre-norm residual)."""
            if name is None:
                call("vtx_add_ln_fwd", res.data_ptr(), branch.data_ptr(), 0, 0, out.data_ptr(), 0, 0, 0, M, H, 0.0, 0.0,
                     seed, 0, 0, s)
                return
            call("vtx_add_ln_fwd", res.data_ptr(), _p(branch), self.P(name + ".weight").data_ptr(),
                 self.P(name + ".bias").data_ptr(), z.data_ptr(), st_.data_ptr(), _p(out), out_b.data_ptr(), M, H,
                 1e-5, 0.0, seed, 0, 1, s)

        i = 0
        pre = mod.norm_first
        for l in range(mod.num_layers):
            q = f"textual.transformer.layers.{l}."
            cache = caches[l]
            slot = cache[pos, :M]  # [M, 3H] view, row stride 3H
            x, xb = bufs[i]
            x1, x1b = bufs[(i + 1) % 3]
            x2, x2b = bufs[(i + 2) % 3]
            # ---- self attention over the cached positions 0 .. pos
            if pre:
                add_ln(x, None, q + "norm1", None, nb)
            gemm(nb if pre else xb, self.W(q + "self_attn.in_proj_weight"), slot, M, 3 * H, H,
                 bias=self.P(q + "self_attn.in_proj_bias"))
            base = cache.data_ptr()
            call("vtx_decode_attn", slot.data_ptr(), 3 * H, base + H * e, base + 2 * H * e, 3 * H,
                 cache.stride(0), _p(table), ldt, 1, o.data_ptr(), H, M, A, pos + 1, T_cache, s)
            gemm(o, self.W(q + "self_attn.out_proj.weight"), pr, M, H, H, bias=self.P(q + "self_attn.out_proj.bias"))
            if pre:
                add_ln(x, pr, None, x1, None)
                add_ln(x1, None, q + "norm2", None, nb)
            else:
                add_ln(x, pr, q + "norm1", x1, x1b)
            # ---- cross attention over the row's image (row // group)
            wc, bc = self.W(q + "multihead_attn.in_proj_weight"), self.P(q + "multihead_attn.in_proj_bias")
            gemm(nb if pre else x1b, wc[:H], qc, M, H, H, bias=bc[:H])
            kv = kvs[l]
            call("vtx_decode_attn", qc.data_ptr(), H, kv.data_ptr(), kv.data_ptr() + H * e, Sk * 2 * H, 2 * H, 0, 0,
                 group, o.data_ptr(), H, M, A, Sk, Sk, s)
            gemm(o, self.W(q + "multihead_attn.out_proj.weight"), pr, M, H, H,
                 bias=self.P(q + "multihead_attn.out_proj.bias"))
            if pre:
                add_ln(x1, pr, None, x2, None)
                add_ln(x2, None, q + "norm3", None, nb)
            else:
                add_ln(x1, pr, q + "norm2", x2, x2b)
            # ---- feed forward
            gemm(nb if pre else x2b, self.W(q + "linear1.weight"), u, M, Fd, H, bias=self.P(q + "linear1.bias"))
            call("vtx_gelu_dropout_fwd", u.data_ptr(), hh.data_ptr(), M * Fd, 0.0, seed, 0, s)
            gemm(hh, self.W(q + "linear2.weight"), pr, M, H, Fd, bias=self.P(q + "linear2.bias"))
            if pre:
                add_ln(x2, pr, None, x1, None)
            else:
                add_ln(x2, pr, q + "norm3", x1, x1b)
            i = (i + 1) % 3
        x, xb = bufs[i]
        if pre:  # final LayerNorm of pre-norm decoders
            add_ln(x, None, "textual.transformer.norm", None, nb)
            xb = nb
        lf = ws.get("dec.logits", (M, V), F32)
        gemm(xb, self.W("textual.embedding.words.weight"), lf, M, V, H, bias=self.P("textual.output.bias"))
        return lf


# ---------------------------------------------------------------------------------------------------- module-level API
def _module_engine(mod, **kw):
    eng = getattr(mod, "_vtx_engine", None)
    if eng is None or not eng.arena.intact():
        eng = Engine(**kw)
        object.__setattr__(mod, "_vtx_engine", eng)
    return eng


@torch.no_grad()
def backbone_features(backbone, image: torch.Tensor) -> torch.Tensor:
    """`TorchvisionVisualBackbone.forward`: (B,3,H,W) fp32 -> (B,C,H/32,W/32) fp32, NCHW-shaped like the reference.
    Module-level calls are inference-style (no autograd); training goes through the model-level engine."""
    eng = _module_engine(backbone, visual=backbone)
    eng.mark_weights_dirty()
    return eng.visual_features(image)


@torch.no_grad()
def head_logits(head, visual_features, caption_tokens, caption_lengths) -> torch.Tensor:
    """`TransformerDecoderTextualHead.forward`: (B,C,h,w), (B,T), (B,) -> fp32 logits (B,T,V);
    `LinearTextualHead.forward`: (B,C,h,w) -> fp32 logits (B,V) (the captions are ignored)."""
    eng = _module_engine(head, textual=head)
    eng.mark_weights_dirty()
    eng.prepare_weights()
    if eng.classification:
        return eng.linear_logits(visual_features.contiguous().float()).clone()
    return eng.head_logits(visual_features, caption_tokens, caption_lengths, training=head.training).clone()
