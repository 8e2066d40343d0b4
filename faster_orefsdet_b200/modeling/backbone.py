"""VoVNet-19-slim-eSE + FPN feature extractor (the caller side of the hot path, SURVEY 8f#4).

On CUDA every convolution runs on the tensor-core kernel (csrc/conv_tc.cu via modeling/tcconv.py), pooling, eSE gate
and stem on csrc/glue.cu; on CPU tensors the same module runs through ATen - that is the CPU baseline of bench.py.

Restates d2!/modeling/backbone/vovnet.py:50-58,205-489,527-555 and
d2!/modeling/backbone/fpn.py:17-155 with the same module / state_dict key names
(log:549-697), so reference checkpoints load.  Runs in ``channels_last`` so the
feature maps it hands to the head are already in the NHWC layout the kernels read.
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, List

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops
from ..compat import Backbone, register, resolve, BACKBONE_REGISTRY, ShapeSpec
from . import tcconv

_STAGE_SPECS = {
    # name: (stem, stage_conv_ch, stage_out_ch, layers_per_block, blocks_per_stage)   vovnet.py:50-97
    "V-19-slim-eSE": ([64, 64, 128], [64, 80, 96, 112], [112, 256, 384, 512], 3, [1, 1, 1, 1]),
    "V-19-eSE": ([64, 64, 128], [128, 160, 192, 224], [256, 512, 768, 1024], 3, [1, 1, 1, 1]),
    "V-39-eSE": ([64, 64, 128], [128, 160, 192, 224], [256, 512, 768, 1024], 5, [1, 1, 2, 2]),
}


class FrozenBatchNorm2d(nn.Module):
    """BatchNorm with fixed statistics and affine parameters (d2!/layers/batch_norm.py)."""

    def __init__(self, num_features: int, eps: float = 1e-5):
        super().__init__()
        self.num_features, self.eps = num_features, eps
        self.register_buffer("weight", torch.ones(num_features))
        self.register_buffer("bias", torch.zeros(num_features))
        self.register_buffer("running_mean", torch.zeros(num_features))
        self.register_buffer("running_var", torch.ones(num_features) - eps)

    def forward(self, x):
        scale = self.weight * (self.running_var + self.eps).rsqrt()
        bias = self.bias - self.running_mean * scale
        return x * scale.reshape(1, -1, 1, 1).to(x.dtype) + bias.reshape(1, -1, 1, 1).to(x.dtype)


class ConvNormReLUSeq(nn.Sequential):
    """Sequential of (conv, FrozenBN, ReLU) triples, named like the reference (``X/conv``, ``X/norm``,
    ``X/relu``).  At inference the frozen BN is folded into the convolution (weight * scale, bias through
    cuDNN's fused epilogue) and the ReLU is in place, so a triple costs one conv and one vectorised
    elementwise pass instead of a broadcast multiply-add over the whole activation."""

    def __init__(self, *args):
        super().__init__(*args)
        self._fold_cache = {}

    def _folded(self, i, conv, norm):
        key = (conv.weight.data_ptr(), conv.weight._version, norm.weight._version, norm.bias._version,
               norm.running_mean._version, norm.running_var._version, conv.weight.device, conv.weight.stride())
        hit = self._fold_cache.get(i)
        if hit is None or hit[0] != key:
            scale = norm.weight * (norm.running_var + norm.eps).rsqrt()
            w = (conv.weight * scale.reshape(-1, 1, 1, 1)).contiguous(memory_format=torch.channels_last)
            b = norm.bias - norm.running_mean * scale
            hit = (key, w.detach(), b.detach())
            self._fold_cache[i] = hit
        return hit[1], hit[2]

    def forward(self, x):
        mods = list(self.children())
        if self.training or len(mods) % 3 != 0:
            for m in mods:
                x = m(x)
            return x
        for i in range(0, len(mods), 3):
            conv, norm, _ = mods[i:i + 3]
            if tcconv.supported(conv, x):          # tcgen05 3xTF32 kernel (csrc/conv_tc.cu)
                x = tcconv.conv(x, conv, norm, relu=True)
                continue
            w, b = self._folded(i, conv, norm)     # CPU tensors (the CPU baseline), shapes outside the kernel: ATen
            with torch.backends.cudnn.flags(allow_tf32=False):      # the reference computes in fp32 (log:490-491)
                x = F.relu_(F.conv2d(x, w, b, conv.stride, conv.padding, conv.dilation, conv.groups))
        return x


def _conv_norm_relu(cin, cout, name, postfix, stride=1, k=3, pad=1):
    return [
        (f"{name}_{postfix}/conv", nn.Conv2d(cin, cout, kernel_size=k, stride=stride, padding=pad, bias=False)),
        (f"{name}_{postfix}/norm", FrozenBatchNorm2d(cout)),
        (f"{name}_{postfix}/relu", nn.ReLU(inplace=True)),
    ]


class _ESE(nn.Module):
    def __init__(self, channel):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.fc = nn.Conv2d(channel, channel, kernel_size=1, padding=0)

    def gate(self, x):
        """hsigmoid(fc(avg(x))) as [N, C, 1, 1].  On CUDA the 1x1 convolution over the pooled [N, C, 1, 1] vector is a
        plain [N, C] x [C, C] product (cuDNN serves it with a 200 us grouped-convolution kernel)."""
        if x.is_cuda:
            n, c = x.shape[0], x.shape[1]
            z = torch.addmm(self.fc.bias, x.mean((2, 3)), self.fc.weight.view(c, c).t())
            return (F.relu6(z + 3.0) / 6.0).view(n, c, 1, 1)
        return F.relu6(self.fc(self.avg_pool(x)) + 3.0) / 6.0

    def forward(self, x):
        return x * self.gate(x)


class _OSAModule(nn.Module):
    def __init__(self, in_ch, stage_ch, concat_ch, layers, name, identity=False):
        super().__init__()
        self.identity = identity
        self.layers = nn.ModuleList()
        c = in_ch
        for i in range(layers):
            self.layers.append(ConvNormReLUSeq(OrderedDict(_conv_norm_relu(c, stage_ch, name, i))))
            c = stage_ch
        self.concat = ConvNormReLUSeq(OrderedDict(_conv_norm_relu(in_ch + layers * stage_ch, concat_ch, name, "concat", k=1, pad=0)))
        self.ese = _ESE(concat_ch)

    def forward(self, x):
        if not self.training and all(tcconv.supported(layer[0], x) for layer in self.layers):
            buf, amax = self._layers_in_place(x)
            y = self.ese(tcconv.conv(buf, self.concat[0], self.concat[1], relu=True, x_amax=amax[:len(self.layers) + 1]))
            return y + x if self.identity else y
        outs = [x]
        y = x
        for layer in self.layers:
            y = layer(y)
            outs.append(y)
        y = self.ese(self.concat(torch.cat(outs, dim=1)))
        return y + x if self.identity else y

    @property
    def concat_channels(self) -> int:
        return self.layers[0][0].in_channels + sum(layer[0].out_channels for layer in self.layers)

    def new_buffer(self, n, h, w, device):
        """NHWC buffer [x | y0 | y1 | y2] of this module, its first slice (written by the producer of x) and the bounds
        max|.| per slice AND image, [slices, N] (the operand bounds of the tensor-core convolutions, ops.conv2d_nhwc: every
        image is scaled by its own bounds, so its result does not depend on its batch mates)."""
        buf = torch.empty((n, h, w, self.concat_channels), dtype=torch.float32, device=device).permute(0, 3, 1, 2)
        # one more row than slices: the actual max|x| of a first slice that arrives pre-split (row 0 then holds ITS bound)
        return buf, buf[:, :self.layers[0][0].in_channels], ops.new_amax(device, (len(self.layers) + 2) * n).view(len(self.layers) + 2, n)

    def _layers_in_place(self, x, buf=None, amax=None):
        """The 3x3 layers write their outputs straight into channel slices of one NHWC buffer
        [x | y0 | y1 | y2] and read their inputs from it: torch.cat never runs."""
        n, c, h, w = x.shape
        if buf is None:
            buf, first, amax = self.new_buffer(n, h, w, x.device)
            first.copy_(x)
            amax[0].copy_(x.detach().abs().amax((1, 2, 3)))
        src, off = buf[:, :c], c
        for i, layer in enumerate(self.layers):
            cw = layer[0].out_channels
            dst = buf[:, off:off + cw]
            tcconv.conv(src, layer[0], layer[1], relu=True, out=dst, x_amax=amax[i:i + 1], y_amax=amax[i + 1])
            src, off = dst, off + cw
        return buf, amax

    def _split_eligible(self) -> bool:
        """Whole 16-channel groups everywhere (the split format packs 16 channels into 64 bytes) and plain 3x3 layers."""
        convs = [layer[0] for layer in self.layers]
        return (all(cv.kernel_size == (3, 3) and cv.stride == (1, 1) and cv.out_channels % 16 == 0 for cv in convs)
                and convs[0].in_channels % 16 == 0 and len({cv.out_channels for cv in convs}) == 1 and len(convs) + 1 <= 8
                and self.concat[0].out_channels % 4 == 0)

    def forward_buffer(self, buf, amax, in_presplit: bool = False, in_bound_is_actual: bool = False):
        """Tensor-core path with x already sitting in the first slice of ``buf`` (and its bound in amax[0]): returns the
        concat-conv output BEFORE the eSE gate, the gate [N,C,1,1] (the consumer fuses the multiplication) and the
        bound of the output.  ``in_presplit``: the producer wrote x in the split operand format at the scale of the bound
        in amax[0]; the actual max|x| is in the last row of amax, unless ``in_bound_is_actual`` (amax[0] is it: the pooling's
        bound is the maximum of its source)."""
        c = self.layers[0][0].in_channels
        n, _, h, w = buf.shape
        a_y = ops.new_amax(buf.device, n)
        cout = self.concat[0].out_channels
        # the eSE average comes out of the concat convolution's epilogue as per-tile channel sums: no pass over y
        colsum = torch.empty((n, ops.conv2d_tiles_per_image(h, w), cout), dtype=torch.float32, device=buf.device)
        nl = len(self.layers)
        if in_presplit and not self._split_eligible():
            raise RuntimeError("a pre-split first slice needs the split hand-off of this module")
        if self._split_eligible():
            # Split hand-off: every 3x3 layer writes its slice in the operand format of its readers (fp16 hi / lo of
            # y * 2^e, e from the bound l1 * max|x| + beta that it publishes into amax[i + 1]); the next 3x3 layer reads it
            # without its conversion pass, the concat convolution rescales each slice to its common scale by a power of
            # two.  The actual maxima (``act``) only feed the next layer's bound, so the bounds do not compound.
            act = ops.new_amax(buf.device, nl * n).view(nl, n)
            src, off = buf[:, :c], c
            for i, layer in enumerate(self.layers):
                cw = layer[0].out_channels
                dst = buf[:, off:off + cw]
                pk, b, cw4 = tcconv.packed(layer[0], layer[1])
                l1, beta = tcconv.bound_consts(layer[0], layer[1])
                ops.conv2d_nhwc_split(src, pk, b, cw4, 3, dst, amax[i:i + 1], y_amax=act[i], x_presplit=i > 0 or in_presplit,
                                      x_actual=act[i - 1] if i > 0 else (amax[nl + 1] if in_presplit and not in_bound_is_actual else None),
                                      y_bound=amax[i + 1], y_l1=l1, y_beta=beta)
                src, off = dst, off + cw
            pk, b, co4 = tcconv.packed(self.concat[0], self.concat[1])
            starts = [0] + [c + i * self.layers[0][0].out_channels for i in range(nl)]
            y = torch.empty((n, h, w, co4), dtype=torch.float32, device=buf.device).permute(0, 3, 1, 2)
            ops.conv2d_nhwc_split(buf, pk, b, co4, 1, y, amax[:nl + 1], y_amax=a_y, x_presplit_from=0 if in_presplit else c,
                                  slice_ch=starts, colsum=colsum)
        else:
            amax[1:nl + 1].zero_()
            self._layers_in_place(buf[:, :c], buf, amax)
            y = tcconv.conv(buf, self.concat[0], self.concat[1], relu=True, x_amax=amax[:nl + 1], y_amax=a_y, colsum=colsum)
        gate = ops.ese_gate(colsum, h * w, self.ese.fc.weight, self.ese.fc.bias)
        return y, gate.view(n, cout, 1, 1), a_y


class _OSAStage(nn.Sequential):
    def __init__(self, in_ch, stage_ch, concat_ch, blocks, layers, stage_num):
        super().__init__()
        if stage_num != 2:
            self.add_module("Pooling", nn.MaxPool2d(kernel_size=3, stride=2, ceil_mode=True))
        self.add_module(f"OSA{stage_num}_1", _OSAModule(in_ch, stage_ch, concat_ch, layers, f"OSA{stage_num}_1"))
        for i in range(blocks - 1):
            n = f"OSA{stage_num}_{i + 2}"
            self.add_module(n, _OSAModule(concat_ch, stage_ch, concat_ch, layers, n, identity=True))


class VoVNet(Backbone):     # detectron2's build_backbone asserts isinstance(backbone, Backbone) (d2!/modeling/backbone/build.py:32)
    def __init__(self, cfg, input_ch: int, out_features: List[str]):
        super().__init__()
        stem_ch, conv_ch, out_ch, layers, blocks = _STAGE_SPECS[cfg.MODEL.VOVNET.CONV_BODY]
        if cfg.MODEL.VOVNET.NORM != "FrozenBN":
            raise NotImplementedError("only MODEL.VOVNET.NORM=FrozenBN (the inference configuration) is built")
        self._out_features = list(out_features)
        stem = _conv_norm_relu(input_ch, stem_ch[0], "stem", "1", 2)
        stem += _conv_norm_relu(stem_ch[0], stem_ch[1], "stem", "2", 1)
        stem += _conv_norm_relu(stem_ch[1], stem_ch[2], "stem", "3", 2)
        self.add_module("stem", ConvNormReLUSeq(OrderedDict(stem)))
        stride = 4
        self._out_feature_strides = {"stem": stride, "stage2": stride}
        self._out_feature_channels = {"stem": stem_ch[2]}
        in_list = [stem_ch[2]] + out_ch[:-1]
        self.stage_names = []
        for i in range(4):
            name = f"stage{i + 2}"
            self.stage_names.append(name)
            self.add_module(name, _OSAStage(in_list[i], conv_ch[i], out_ch[i], blocks[i], layers, i + 2))
            self._out_feature_channels[name] = out_ch[i]
            if i != 0:
                stride *= 2
                self._out_feature_strides[name] = stride

    def _tc_path(self, x) -> bool:
        return (x.is_cuda and x.dtype == torch.float32 and not self.training and x.shape[1] == 3
                and all(len([m for m in getattr(self, n) if isinstance(m, _OSAModule)]) == 1 for n in self.stage_names))

    def _stem1_packed(self):
        """stem_1 (3x3, stride 2, 3 input channels) as a 1x1 convolution over 32-wide im2col rows (ops.stem_patches)."""
        conv, norm = self.stem[0], self.stem[1]
        key = tcconv._versions(conv.weight, *norm.buffers())
        hit = getattr(self, "_stem1_cache", None)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                w, b = tcconv.folded(conv, norm)
                w = w.permute(0, 2, 3, 1).reshape(w.shape[0], 27)                      # k = (ky*3 + kx)*3 + c
                w = torch.cat((w, w.new_zeros(w.shape[0], 5)), 1).reshape(-1, 32, 1, 1).contiguous()
                hit = (key, ops.conv2d_pack(w), b.detach().float().contiguous())
            self._stem1_cache = hit
        return hit[1], hit[2]

    def _tc_modules(self):
        return [[m for m in getattr(self, name) if isinstance(m, _OSAModule)][0] for name in self.stage_names]

    def tc_new_input_buffer(self, n, h, w, device):
        """Concat buffer of the first OSA stage for n images of h x w pixels, its first slice (where stem_3 writes) and
        its per-slice bounds."""
        h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1       # stem_1
        h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1       # stem_3
        return self._tc_modules()[0].new_buffer(n, h, w, device)

    def _stem1_folded(self):
        conv, norm = self.stem[0], self.stem[1]
        key = tcconv._versions(conv.weight, *norm.buffers())
        hit = getattr(self, "_stem1_folded_cache", None)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                w, b = tcconv.folded(conv, norm)
                hit = (key, w.detach().float().contiguous(), b.detach().float().contiguous())
            self._stem1_folded_cache = hit
        return hit[1], hit[2]

    def _stem1_bound(self, mean, std):
        """One device float >= every output of stem_1 (ReLU of the folded convolution) for ANY uint8 image: the absolute
        row sums of the folded weight times the largest normalised pixel magnitude per colour plane, plus |bias|."""
        conv, norm = self.stem[0], self.stem[1]
        key = (tcconv._versions(conv.weight, *norm.buffers()), tuple(mean), tuple(std))
        hit = getattr(self, "_stem1_bound_cache", None)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                w, b = self._stem1_folded()
                xmax = torch.tensor([max(abs(0.0 - m), abs(255.0 - m)) / abs(sd) for m, sd in zip(mean, std)],
                                    dtype=torch.float64, device=w.device)
                rows = (w.double().abs().sum((2, 3)) * xmax.view(1, 3)).sum(1) + (b.double().abs() if b is not None else 0.0)
                bound = (rows.max() * 1.001).clamp_min(1e-30).float().reshape(1).contiguous()
            hit = (key, bound, {})
            self._stem1_bound_cache = hit
        return hit[1]

    def _stem1_bound_rows(self, mean, std, n):
        """The same bound as a [1, n] row (one column per image), cached per batch size."""
        bound = self._stem1_bound(mean, std)
        rows = self._stem1_bound_cache[2]
        if n not in rows:
            rows[n] = bound.expand(n).contiguous().view(1, n)
        return rows[n]

    def stem_u8_writes_split(self) -> bool:
        """tc_stem_u8 leaves its output (the first slice of the stage-2 concat buffer) in the split operand format."""
        return ("stem" not in self._out_features and self.stem[0].out_channels == 64
                and tuple(self.stem[0].weight.shape[1:]) == (3, 3, 3) and self.stem[6].out_channels % 16 == 0
                and self._tc_modules()[0]._split_eligible())

    def tc_stem_u8(self, x_u8, mean, std, out, out_amax, out_act=None, scratch=None):
        """Raw uint8 images -> stem_1 (normalisation fused; tensor-core kernel ops.stem1_u8_tc, the im2col gathered into
        tensor memory) -> stem_2 -> stem_3 into ``out``; same contract as tc_stem.  With ``out_act`` (when
        stem_u8_writes_split()) ``out`` is left in the split operand format of the first OSA module."""
        if self.stem[0].out_channels != 64 or tuple(self.stem[0].weight.shape[1:]) != (3, 3, 3):
            return self.tc_stem(ops.stem_patches_u8(x_u8, mean, std), None, out, out_amax)
        n = x_u8.shape[0]
        if scratch is not None:      # [2, n] zeroed floats of the caller (one fill per batch instead of two per chunk)
            a1, a2 = scratch[0], scratch[1]
        else:
            a1, a2 = ops.new_amax(x_u8.device, n), ops.new_amax(x_u8.device, n)          # per image
        # stem_1 writes the operand format of stem_2 (fp16 hi / lo of y * 2^e) instead of fp32: its output bound follows
        # from the weights and the pixel range alone, so the scale is known before the layer runs and stem_2 skips
        # the conversion pass of every staged tile
        pk, b = self._stem1_packed()
        bound = self._stem1_bound(mean, std)
        if out_act is None:
            y = ops.stem1_u8_tc(x_u8, mean, std, pk, b, y_bound=bound)
            y = tcconv.conv(y, self.stem[3], self.stem[4], relu=True, x_amax=bound, y_amax=a2, x_presplit=True)
            tcconv.conv(y, self.stem[6], self.stem[7], relu=True, out=out, x_amax=a2.view(1, n), y_amax=out_amax)
            return
        # split hand-off all the way: stem_2 -> stem_3 -> the first OSA module
        y = ops.stem1_u8_tc(x_u8, mean, std, pk, b, y_amax=a1, y_bound=bound)
        pk2, b2, c2 = tcconv.packed(self.stem[3], self.stem[4])
        l1, beta = tcconv.bound_consts(self.stem[3], self.stem[4])
        b2nd = torch.empty((n,), dtype=torch.float32, device=x_u8.device)          # stem_2's published bound, per image (a plain store)
        y2 = torch.empty((n, y.shape[2], y.shape[3], c2), dtype=torch.float32, device=y.device).permute(0, 3, 1, 2)
        ops.conv2d_nhwc_split(y, pk2, b2, c2, 3, y2, self._stem1_bound_rows(mean, std, n),
                              y_amax=a2, x_presplit=True, x_actual=a1, y_bound=b2nd, y_l1=l1, y_beta=beta)
        pk3, b3, c3 = tcconv.packed(self.stem[6], self.stem[7])
        l1, beta = tcconv.bound_consts(self.stem[6], self.stem[7])
        # out_amax receives stem_3's bound, out_act its max(y)
        ops.conv2d_nhwc_split(y2, pk3, b3, c3, 3, out, b2nd.view(1, n), y_amax=out_act, x_actual=a2, y_bound=out_amax,
                              y_l1=l1, y_beta=beta, x_presplit_from=0, slice_ch=[0], stride=2)

    def tc_stem(self, patches, patches_amax, out, out_amax):
        """stem_1 (as a 1x1 convolution over im2col rows) -> stem_2 -> stem_3 into ``out`` (a batch slice of the first
        slice of the stage-2 concat buffer; ``out_amax`` is only ever raised).  Works on any sub-batch, so a caller can
        overlap host-to-device copies of later images with the stem of earlier ones."""
        pk, b = self._stem1_packed()
        n = patches.shape[0]
        if patches_amax is None:
            patches_amax = patches.detach().abs().amax((1, 2, 3)).view(1, n)           # per image
        a1, a2 = ops.new_amax(patches.device, n), ops.new_amax(patches.device, n)
        y = ops.conv2d_nhwc(patches, pk, b, self.stem[0].out_channels, 1, relu=True, x_amax=patches_amax, y_amax=a1)
        y = tcconv.conv(y, self.stem[3], self.stem[4], relu=True, x_amax=a1.view(1, n), y_amax=a2)
        tcconv.conv(y, self.stem[6], self.stem[7], relu=True, out=out, x_amax=a2.view(1, n), y_amax=out_amax)

    def tc_body(self, buf, amax, want_amax: bool = False, fuse_gates: bool = False, in_presplit: bool = False):
        """OSA stages from a filled stage-2 concat buffer.  The stage poolings write straight into the first slice of
        the next stage's buffer; the eSE gate of a stage (<= 1, so the bound of the ungated map still holds) is applied
        inside the pooling that consumes it.  For the stages that are FPN inputs the gated map is materialised, unless
        ``fuse_gates``: then the UNGATED map is returned together with its gate (third result, {name: [N,C,1,1]}) and the
        consumer multiplies it in (FPN.top_down passes it to the lateral convolution)."""
        outputs, bounds, gates = {}, {}, {}
        mods = self._tc_modules()
        n = buf.shape[0]
        if "stem" in self._out_features:
            outputs["stem"], bounds["stem"] = buf[:, :mods[0].layers[0][0].in_channels], amax[0]
        for i, (name, mod) in enumerate(zip(self.stage_names, mods)):
            y, gate, a_y = mod.forward_buffer(buf, amax, in_presplit=in_presplit, in_bound_is_actual=i > 0)
            if name in self._out_features:
                if fuse_gates:
                    outputs[name], bounds[name], gates[name] = y, a_y, gate
                else:
                    y = y.mul_(gate)
                    outputs[name], bounds[name] = y, a_y
                    gate = None
            if i + 1 < len(mods):
                h, w = (y.shape[2] - 2) // 2 + 1, (y.shape[3] - 2) // 2 + 1
                buf, first, amax = mods[i + 1].new_buffer(n, h, w, y.device)
                # the pooling hands the next stage its first slice in the split format when that stage reads it that way:
                # the bound is the actual maximum of the pooled map's source (the gate is <= 1)
                in_presplit = mods[i + 1]._split_eligible() and a_y.numel() == n
                ops.maxpool3x3s2_nhwc(y, gate, out=first, y_bound=a_y if in_presplit else None)
                amax[0].copy_(a_y)
        if fuse_gates:
            return outputs, bounds, gates
        return (outputs, bounds) if want_amax else outputs

    def _forward_tc(self, x):
        """Inference on CUDA: every convolution on the tensor cores (csrc/conv_tc.cu), no torch.cat, no layout copies."""
        buf, first, amax = self.tc_new_input_buffer(x.shape[0], x.shape[2], x.shape[3], x.device)
        patches = ops.stem_patches(x)
        self.tc_stem(patches, None, first, amax[0])
        return self.tc_body(buf, amax)

    def forward(self, x):
        if self._tc_path(x):
            return self._forward_tc(x)
        outputs = {}
        x = self.stem(x)
        if "stem" in self._out_features:
            outputs["stem"] = x
        for name in self.stage_names:
            x = getattr(self, name)(x)
            if name in self._out_features:
                outputs[name] = x
        return outputs

    def output_shape(self):
        return {n: ShapeSpec(channels=self._out_feature_channels[n], stride=self._out_feature_strides[n])
                for n in self._out_features}


class FPN(Backbone):
    """Top-down pathway with lateral 1x1 and output 3x3 convs, "sum" fusion, no top block
    (MODEL.FCOS.TOP_LEVELS = 0, log:264)."""

    def __init__(self, bottom_up: VoVNet, in_features: List[str], out_channels: int, fuse_type: str = "sum"):
        super().__init__()
        shapes = bottom_up.output_shape()
        strides = [shapes[f].stride for f in in_features]
        laterals, outputs = [], []
        for f in in_features:
            stage = int(math.log2(shapes[f].stride))
            lat = nn.Conv2d(shapes[f].channels, out_channels, kernel_size=1)
            out = nn.Conv2d(out_channels, out_channels, kernel_size=3, padding=1)
            for m in (lat, out):      # c2_xavier_fill (fvcore): kaiming_uniform(a=1), zero bias
                nn.init.kaiming_uniform_(m.weight, a=1)
                nn.init.constant_(m.bias, 0)
            self.add_module(f"fpn_lateral{stage}", lat)
            self.add_module(f"fpn_output{stage}", out)
            laterals.append(lat)
            outputs.append(out)
        self._laterals, self._outputs = laterals[::-1], outputs[::-1]
        self.in_features = tuple(in_features)
        self.bottom_up = bottom_up
        self._out_feature_strides = {f"p{int(math.log2(s))}": s for s in strides}
        self._out_features = list(self._out_feature_strides)
        self._out_feature_channels = {k: out_channels for k in self._out_features}
        self._size_divisibility = strides[-1]
        assert fuse_type in ("sum", "avg")
        self._fuse_type = fuse_type

    @property
    def size_divisibility(self) -> int:
        return self._size_divisibility

    def forward(self, x) -> Dict[str, torch.Tensor]:
        return self.top_down(self.bottom_up(x))

    def top_down(self, feats, bounds=None, gates=None) -> Dict[str, torch.Tensor]:
        """Lateral 1x1 + nearest 2x upsampling + sum + output 3x3.  ``bounds[name]``: device scalar bounding
        max|feats[name]| when the producer knows it (the tensor-core convolutions need one; computed otherwise).
        ``gates[name]``: [N,C,1,1] factor still to be multiplied into feats[name] (the eSE gate, VoVNet.tc_body)."""
        bounds, gates = bounds or {}, gates or {}

        def per_image(a, t):      # a bound per image [N] -> the [1, N] operand-bound layout of ops.conv2d_nhwc
            return a.reshape(1, -1) if a is not None and a.dim() == 1 and a.numel() == t.shape[0] and t.shape[0] > 1 else a

        def run(m, t, a_in=None, a_out=None, gate=None):
            if tcconv.supported(m, t) and (gate is None or m.in_channels % 32 == 0):
                return tcconv.conv(t, m, x_amax=per_image(a_in, t), y_amax=a_out, a_gate=gate)
            y = m(t if gate is None else t * gate)
            if a_out is not None:
                a_out.copy_(y.detach().abs().max().reshape(1))
            return y

        def bound(t):
            return ops.new_amax(t.device, t.shape[0]) if t.is_cuda else None      # [N]: one bound per image

        top = self.in_features[-1]
        a_prev = bound(feats[top])
        prev = run(self._laterals[0], feats[top], bounds.get(top), a_prev, gates.get(top))
        out_bounds = []      # max|output map| per level (device scalars), reported by the output convolutions' epilogues

        def out_bound(t):
            b = ops.new_amax(t.device, t.shape[0]) if t.is_cuda else None      # [N]: one bound per image
            out_bounds.insert(0, b)
            return b

        results = [run(self._outputs[0], prev, a_prev, out_bound(prev))]
        for idx in range(1, len(self._laterals)):
            name = self.in_features[-idx - 1]
            f, lat = feats[name], self._laterals[idx]
            gate = gates.get(name)
            if (tcconv.supported(lat, f) and self._fuse_type == "sum" and lat.out_channels % 4 == 0
                    and (gate is None or lat.in_channels % 32 == 0)
                    and tuple(prev.shape[2:]) == ((f.shape[2] + 1) // 2, (f.shape[3] + 1) // 2)):
                # nearest 2x upsampling + sum inside the lateral convolution's epilogue; its bound is that of the sum
                a_prev = bound(f)
                prev = tcconv.conv(f, lat, x_amax=per_image(bounds.get(name), f), y_amax=a_prev, residual=prev,
                                   residual_upsample2=True, a_gate=gate)
            else:
                top_down = F.interpolate(prev, scale_factor=2.0, mode="nearest")
                a_lat = bound(f)
                prev = run(lat, f, bounds.get(name), a_lat, gate) + top_down
                if a_lat is not None:
                    a_prev = a_lat + a_prev            # |lateral + upsampled| <= bound + bound
                if self._fuse_type == "avg":
                    prev = prev / 2
            results.insert(0, run(self._outputs[idx], prev, a_prev, out_bound(prev)))
        self.last_output_bounds = dict(zip(self._out_features, out_bounds))
        return dict(zip(self._out_features, results))

    def output_shape(self):
        return {n: ShapeSpec(channels=self._out_feature_channels[n], stride=self._out_feature_strides[n])
                for n in self._out_features}


@register(BACKBONE_REGISTRY)
def build_fcos_vovnet_fpn_backbone(cfg, input_shape: ShapeSpec):
    if cfg.MODEL.FCOS.TOP_LEVELS != 0:
        raise NotImplementedError("MODEL.FCOS.TOP_LEVELS != 0 (P6/P7) is not used by finetune_vovnet.yaml")
    bottom_up = VoVNet(cfg, input_shape.channels, cfg.MODEL.VOVNET.OUT_FEATURES)
    return FPN(bottom_up, cfg.MODEL.FPN.IN_FEATURES, cfg.MODEL.FPN.OUT_CHANNELS, cfg.MODEL.FPN.FUSE_TYPE)


def build_backbone(cfg, input_shape: ShapeSpec = None):
    if input_shape is None:
        input_shape = ShapeSpec(channels=len(cfg.MODEL.PIXEL_MEAN))
    return resolve(BACKBONE_REGISTRY, cfg.MODEL.BACKBONE.NAME)(cfg, input_shape)
