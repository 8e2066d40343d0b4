"""Attention-RPN proposal generator of the FsodRCNN path (SURVEY 8f#3).

``FsodRPN`` mirrors fewx/modeling/fsod/fsod_rpn.py:149-490 at inference: ``StandardRPNHead`` (the fork's 192-channel
hidden layer, :75-147), ``DefaultAnchorGenerator`` (d2!/modeling/anchor_generator.py) and ``find_top_rpn_proposals``
(d2!/modeling/proposal_generator/proposal_utils.py:19-119).  B200 path: the 3x3 hidden convolution runs on the
tensor-core kernel with the support correlation of FsodRCNN fused into its A operand (``a_gate``), objectness and
anchor deltas are one stacked 1x1 convolution, the NMS is ``fod_batched_nms``.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F
from torch import nn

from .. import ops
from ..compat import PROPOSAL_GENERATOR_REGISTRY, Boxes, Instances, ShapeSpec, register
from . import tcconv

_SCALE_CLAMP = math.log(1000.0 / 16)


def apply_deltas(deltas: torch.Tensor, boxes: torch.Tensor, weights: Sequence[float]) -> torch.Tensor:
    """Box2BoxTransform.apply_deltas (d2!/modeling/box_regression.py:77-115), class-agnostic [N,4]."""
    boxes = boxes.to(deltas.dtype)
    widths, heights = boxes[:, 2] - boxes[:, 0], boxes[:, 3] - boxes[:, 1]
    ctr_x, ctr_y = boxes[:, 0] + 0.5 * widths, boxes[:, 1] + 0.5 * heights
    wx, wy, ww, wh = weights
    dx, dy = deltas[:, 0] / wx, deltas[:, 1] / wy
    dw, dh = torch.clamp(deltas[:, 2] / ww, max=_SCALE_CLAMP), torch.clamp(deltas[:, 3] / wh, max=_SCALE_CLAMP)
    pcx, pcy = dx * widths + ctr_x, dy * heights + ctr_y
    pw, ph = torch.exp(dw) * widths, torch.exp(dh) * heights
    return torch.stack((pcx - 0.5 * pw, pcy - 0.5 * ph, pcx + 0.5 * pw, pcy + 0.5 * ph), 1)


class StandardRPNHead(nn.Module):
    def __init__(self, in_channels: int, num_anchors: int, box_dim: int = 4):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, 192, kernel_size=3, stride=1, padding=1)      # fsod_rpn.py:101
        self.objectness_logits = nn.Conv2d(192, num_anchors, kernel_size=1)
        self.anchor_deltas = nn.Conv2d(192, num_anchors * box_dim, kernel_size=1)
        for l in (self.conv, self.objectness_logits, self.anchor_deltas):
            nn.init.normal_(l.weight, std=0.01)
            nn.init.constant_(l.bias, 0)

    def forward(self, features: List[torch.Tensor], gates: Optional[List[torch.Tensor]] = None,
                bounds: Optional[List[torch.Tensor]] = None):
        """``gates[l]`` [N, C]: per-(image, channel) factors multiplied into features[l] first (the support correlation
        of FsodRCNN); ``bounds[l]``: device floats [1, N], bound of max|features[l] * gate| per image.  Each image is
        scaled by its own bound in both convolutions: its outputs do not depend on its batch mates."""
        logits, deltas = [], []
        A = self.objectness_logits.out_channels
        for l, x in enumerate(features):
            g = gates[l] if gates is not None else None
            if tcconv.supported(self.conv, x) and (g is None or x.shape[1] % 32 == 0):
                x_amax = bounds[l] if bounds is not None else ops.absmax(ops.nhwc(x), per_image=True).reshape(1, -1)
                t_amax = ops.new_amax(x.device, x.shape[0])
                t = tcconv.conv(x, self.conv, relu=True, a_gate=g, x_amax=x_amax, y_amax=t_amax)
                y = tcconv.conv(t, self.objectness_logits, extra=self.anchor_deltas,       # [N, A + 4A (+pad), H, W]
                                x_amax=t_amax.reshape(1, -1))
                logits.append(y[:, :A])
                deltas.append(y[:, A:A + self.anchor_deltas.out_channels])
            else:                                                                          # CPU tensors
                if g is not None:
                    x = x * g.reshape(x.shape[0], -1, 1, 1)
                t = F.relu(self.conv(x))
                logits.append(self.objectness_logits(t))
                deltas.append(self.anchor_deltas(t))
        return logits, deltas


class DefaultAnchorGenerator(nn.Module):
    """d2!/modeling/anchor_generator.py DefaultAnchorGenerator: (H, W, A)-ordered XYXY anchors per level."""

    def __init__(self, sizes, aspect_ratios, strides, offset: float = 0.0):
        super().__init__()
        n = len(strides)
        sizes = list(sizes) * n if len(sizes) == 1 else sizes
        aspect_ratios = list(aspect_ratios) * n if len(aspect_ratios) == 1 else aspect_ratios
        self.strides, self.offset = list(strides), offset
        self.cell_anchors = []
        for s, a in zip(sizes, aspect_ratios):
            anchors = []
            for size in s:
                area = size ** 2.0
                for ar in a:
                    w = math.sqrt(area / ar)
                    h = ar * w
                    anchors.append([-w / 2.0, -h / 2.0, w / 2.0, h / 2.0])
            self.cell_anchors.append(torch.tensor(anchors))
        self.num_anchors = [len(c) for c in self.cell_anchors]
        self.box_dim = 4

    def forward(self, features: List[torch.Tensor]) -> List[torch.Tensor]:
        out = []
        for f, stride, base in zip(features, self.strides, self.cell_anchors):
            h, w = f.shape[-2:]
            sx = torch.arange(self.offset * stride, w * stride, step=stride, dtype=torch.float32, device=f.device)
            sy = torch.arange(self.offset * stride, h * stride, step=stride, dtype=torch.float32, device=f.device)
            yy, xx = torch.meshgrid(sy, sx, indexing="ij")
            shifts = torch.stack((xx.reshape(-1), yy.reshape(-1), xx.reshape(-1), yy.reshape(-1)), 1)
            out.append((shifts.view(-1, 1, 4) + base.to(f.device).view(1, -1, 4)).reshape(-1, 4))
        return out


@register(PROPOSAL_GENERATOR_REGISTRY)
class FsodRPN(nn.Module):
    def __init__(self, cfg, input_shape: Dict[str, ShapeSpec]):
        super().__init__()
        r = cfg.MODEL.RPN
        self.in_features = list(r.IN_FEATURES)
        shapes = [input_shape[f] for f in self.in_features]
        a = cfg.MODEL.ANCHOR_GENERATOR
        self.anchor_generator = DefaultAnchorGenerator(a.SIZES, a.ASPECT_RATIOS, [s.stride for s in shapes], a.OFFSET)
        if len({s.channels for s in shapes}) != 1 or len(set(self.anchor_generator.num_anchors)) != 1:
            raise NotImplementedError("FsodRPN: one channel count and one anchor count over the levels")
        self.rpn_head = StandardRPNHead(shapes[0].channels, self.anchor_generator.num_anchors[0])
        self.box_weights = tuple(float(x) for x in r.BBOX_REG_WEIGHTS)
        self.pre_nms_topk, self.post_nms_topk = r.PRE_NMS_TOPK_TEST, r.POST_NMS_TOPK_TEST
        self.nms_thresh, self.min_box_size = r.NMS_THRESH, cfg.MODEL.PROPOSAL_GENERATOR.MIN_SIZE

    def forward(self, images, features: Dict[str, torch.Tensor], gt_instances=None, gates=None, bounds=None):
        if self.training:
            raise NotImplementedError("FsodRPN: training (anchor labelling / losses) is outside the inference hot path")
        feats = [features[f] for f in self.in_features]
        anchors = self.anchor_generator(feats)
        logits, deltas = self.rpn_head(feats, gates, bounds)
        logits = [s.permute(0, 2, 3, 1).flatten(1) for s in logits]                     # (N, Hi*Wi*A)
        deltas = [x.reshape(x.shape[0], -1, 4, x.shape[-2], x.shape[-1]).permute(0, 3, 4, 1, 2).flatten(1, -2) for x in deltas]
        return self.predict_proposals(anchors, logits, deltas, images.image_sizes), {}

    @torch.no_grad()
    def predict_proposals(self, anchors, logits, deltas, image_sizes) -> List[Instances]:
        """find_top_rpn_proposals (proposal_utils.py:19-119): per level top-k by objectness, decode, clip, drop empty,
        level-wise NMS (fod_batched_nms), first post_nms_topk."""
        n_img = len(image_sizes)
        top_scores, top_boxes, level_ids = [], [], []
        for lvl, (anc, lg, dl) in enumerate(zip(anchors, logits, deltas)):
            k = min(lg.shape[1], self.pre_nms_topk)
            s, idx = lg.sort(descending=True, dim=1)
            s, idx = s[:, :k], idx[:, :k]
            boxes = []
            for n in range(n_img):       # only the selected anchors are decoded
                boxes.append(apply_deltas(dl[n][idx[n]].float(), anc[idx[n]], self.box_weights))
            top_scores.append(s)
            top_boxes.append(torch.stack(boxes))
            level_ids.append(torch.full((k,), lvl, dtype=torch.int64, device=lg.device))
        top_scores, top_boxes, level_ids = torch.cat(top_scores, 1), torch.cat(top_boxes, 1), torch.cat(level_ids)
        results = []
        for n, size in enumerate(image_sizes):
            b, s, lv = top_boxes[n], top_scores[n], level_ids
            valid = torch.isfinite(b).all(1) & torch.isfinite(s)
            b, s, lv = b[valid], s[valid], lv[valid]
            boxes = Boxes(b.contiguous())
            boxes.clip(size)
            keep = boxes.nonempty(threshold=self.min_box_size)
            b, s, lv = boxes.tensor[keep], s[keep], lv[keep]
            if b.is_cuda:
                keep = ops.batched_nms(b.contiguous(), s.contiguous(), lv if len(anchors) > 1 else None, self.nms_thresh)
            else:
                from torchvision.ops import boxes as box_ops
                keep = box_ops.batched_nms(b, s, lv, self.nms_thresh)
            keep = keep[: self.post_nms_topk]
            inst = Instances(tuple(size))
            inst.proposal_boxes = Boxes(b[keep])
            inst.objectness_logits = s[keep]
            results.append(inst)
        return results
