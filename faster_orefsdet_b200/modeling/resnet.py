"""ResNet-50 C4 feature extractor of the FsodRCNN path (caller side of the hot path; SURVEY 8f#3).

Restates d2!/modeling/backbone/resnet.py (BasicStem, BottleneckBlock, ResNet, build_resnet_backbone) with the same module
/ state_dict key names (``backbone.stem.conv1.norm.weight``, ``backbone.res3.0.shortcut.weight`` ...), FrozenBN only.
On CUDA the 1x1 / 3x3 convolutions the tensor-core kernel supports run through it (FrozenBN folded, ReLU and the
residual sum fused into its epilogue); the 7x7 stem and the strided 1x1 convolutions go through ATen.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
import torch.nn.functional as F
from torch import nn

from .. import ops
from ..compat import BACKBONE_REGISTRY, Backbone, ShapeSpec, register
from . import tcconv
from .backbone import FrozenBatchNorm2d


class ConvNorm(nn.Conv2d):
    """``detectron2.layers.Conv2d`` with a FrozenBN ``norm`` child and an optional fused ReLU / residual."""

    def __init__(self, cin, cout, k, stride=1, padding=0):
        super().__init__(cin, cout, k, stride=stride, padding=padding, bias=False)
        self.norm = FrozenBatchNorm2d(cout)
        nn.init.kaiming_normal_(self.weight, mode="fan_out", nonlinearity="relu")    # c2_msra_fill

    def forward(self, x, relu: bool = False, residual: Optional[torch.Tensor] = None):
        """On CUDA every image (every ROI row in res5) is scaled by its own operand bound, so that its result depends
        neither on the other images of the batch nor on rows nobody wrote (the padding rows of a ragged ROI batch)."""
        if x.is_cuda:       # the kernels read NHWC memory; ATen ops (stem, pooling) may hand over NCHW
            x = x.contiguous(memory_format=torch.channels_last)
        if tcconv.supported(self, x) and not self.training:
            return tcconv.conv(x, self, self.norm, relu=relu, residual=residual, x_amax=ops.absmax(x, per_image=True).reshape(1, -1))
        if x.is_cuda and self.kernel_size == (1, 1) and self.stride == (2, 2) and self.in_channels % 4 == 0 and not self.training:
            # a strided 1x1 convolution = the 1x1 convolution of the subsampled map
            xs = x[:, :, ::2, ::2].contiguous(memory_format=torch.channels_last)
            pk, b, cout = tcconv.packed(self, self.norm)
            return ops.conv2d_nhwc(xs, pk, b, cout, 1, relu, residual=residual, x_amax=ops.absmax(xs, per_image=True).reshape(1, -1))
        with torch.backends.cudnn.flags(allow_tf32=False):
            y = self.norm(F.conv2d(x, self.weight, None, self.stride, self.padding))
        if residual is not None:
            y = y + residual
        return F.relu_(y) if relu else y


class BasicStem(nn.Module):
    def __init__(self, cin=3, cout=64):
        super().__init__()
        self.conv1 = ConvNorm(cin, cout, 7, stride=2, padding=3)
        self.out_channels, self.stride = cout, 4

    def forward(self, x):
        return F.max_pool2d(self.conv1(x, relu=True), kernel_size=3, stride=2, padding=1)


class BottleneckBlock(nn.Module):
    def __init__(self, cin, cout, *, bottleneck_channels, stride=1, stride_in_1x1=True):
        super().__init__()
        self.in_channels, self.out_channels, self.stride = cin, cout, stride
        self.shortcut = ConvNorm(cin, cout, 1, stride=stride) if cin != cout else None
        s1, s3 = (stride, 1) if stride_in_1x1 else (1, stride)
        self.conv1 = ConvNorm(cin, bottleneck_channels, 1, stride=s1)
        self.conv2 = ConvNorm(bottleneck_channels, bottleneck_channels, 3, stride=s3, padding=1)
        self.conv3 = ConvNorm(bottleneck_channels, cout, 1)

    def forward(self, x):
        out = self.conv2(self.conv1(x, relu=True), relu=True)
        shortcut = self.shortcut(x) if self.shortcut is not None else x
        return self.conv3(out, relu=True, residual=shortcut)         # relu(conv3 + shortcut)


def make_stage(num_blocks, stride_per_block, cin, cout, bottleneck_channels, stride_in_1x1=True) -> List[nn.Module]:
    blocks = []
    for i in range(num_blocks):
        blocks.append(BottleneckBlock(cin, cout, bottleneck_channels=bottleneck_channels, stride=stride_per_block[i],
                                      stride_in_1x1=stride_in_1x1))
        cin = cout
    return blocks


class ResNet(Backbone):
    def __init__(self, stem, stages: List[List[nn.Module]], out_features: List[str]):
        super().__init__()
        self.stem = stem
        self.stage_names, self._out_features = [], list(out_features)
        self._out_feature_strides, self._out_feature_channels = {"stem": stem.stride}, {"stem": stem.out_channels}
        stride = stem.stride
        for i, blocks in enumerate(stages):
            name = f"res{i + 2}"
            self.add_module(name, nn.Sequential(*blocks))
            self.stage_names.append(name)
            stride *= int(torch.tensor([b.stride for b in blocks]).prod())
            self._out_feature_strides[name], self._out_feature_channels[name] = stride, blocks[-1].out_channels

    @property
    def size_divisibility(self) -> int:
        return 0

    def forward(self, x) -> Dict[str, torch.Tensor]:
        out = {}
        if x.is_cuda:
            x = x.contiguous(memory_format=torch.channels_last)
        x = self.stem(x)
        for name in self.stage_names:
            x = getattr(self, name)(x)
            if name in self._out_features:
                out[name] = x
        return out

    def output_shape(self):
        return {n: ShapeSpec(channels=self._out_feature_channels[n], stride=self._out_feature_strides[n]) for n in self._out_features}


@register(BACKBONE_REGISTRY)
def build_resnet_backbone(cfg, input_shape: ShapeSpec):
    """d2!/modeling/backbone/resnet.py build_resnet_backbone for the configurations of the reference (depth 50 / 101,
    FrozenBN, no deformable convolutions, stages up to the last requested output feature)."""
    r = cfg.MODEL.RESNETS
    if r.NORM != "FrozenBN" or r.NUM_GROUPS != 1 or any(r.DEFORM_ON_PER_STAGE) or r.RES5_DILATION != 1:
        raise NotImplementedError("build_resnet_backbone: FrozenBN, one group, no deformable / dilated stages (Base-FSOD-C4.yaml)")
    depth = {50: [3, 4, 6, 3], 101: [3, 4, 23, 3]}[r.DEPTH]
    out_features = list(r.OUT_FEATURES)
    last = max({"res2": 2, "res3": 3, "res4": 4, "res5": 5}[f] for f in out_features)
    stem = BasicStem(input_shape.channels, r.STEM_OUT_CHANNELS)
    cin, cout, bott = r.STEM_OUT_CHANNELS, r.RES2_OUT_CHANNELS, r.NUM_GROUPS * r.WIDTH_PER_GROUP
    stages = []
    for idx in range(2, last + 1):
        first = 1 if idx == 2 else 2
        stages.append(make_stage(depth[idx - 2], [first] + [1] * (depth[idx - 2] - 1), cin, cout, bott, r.STRIDE_IN_1X1))
        cin, cout, bott = cout, cout * 2, bott * 2
    return ResNet(stem, stages, out_features)
