"""ROI heads of the FsodRCNN path (SURVEY 8f#3): ``FsodRes5ROIHeads`` (fewx/modeling/fsod/fsod_roi_heads.py:53-215) and
``FsodFastRCNNOutputLayers`` (fewx/modeling/fsod/fsod_fast_rcnn.py:392-589) at inference, under the same parameter names.

B200 path: the 14x14 ROIAlign over the 1024-channel res4 map is ``fod_roi_align_wide``, the res5 bottlenecks and
``conv_1`` run on the tensor-core convolution (FrozenBN folded, residual sum fused), scoring + box decoding + class-wise
NMS + top-k + rescale is ``fod_final_detect`` - the same kernel that closes the CenterNet2 path.  The three relation
terms after ``conv_1`` (global average + fc, depthwise 7x7 correlation, 49x49 patch attention) are a few small ATen
calls per class on [R, 1024, 49] tensors.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F
from torch import nn

from .. import ops
from ..compat import Boxes, Instances, ShapeSpec, register
from . import tcconv
from .resnet import make_stage
from .roi_heads import ROI_HEADS_REGISTRY
from .rpn import apply_deltas


def positional_encoding(d_model: int, max_len: int) -> torch.Tensor:
    """PositionalEncoding.pe (fsod_fast_rcnn.py:687-697, fsod_rcnn.py:535-545): [1, max_len, d_model]."""
    pe = torch.zeros(max_len, d_model)
    position = torch.arange(0.0, max_len).unsqueeze(1)
    div_term = torch.exp(torch.arange(0.0, d_model, 2) * -(math.log(10000.0) / float(d_model)))
    pe[:, 0::2] = torch.sin(position * div_term)
    pe[:, 1::2] = torch.cos(position * div_term)
    return pe.unsqueeze(0)


class FsodFastRCNNOutputLayers(nn.Module):
    def __init__(self, cfg, input_shape: ShapeSpec):
        super().__init__()
        dim_in = input_shape.channels                                     # 2048
        h = cfg.MODEL.ROI_BOX_HEAD
        if not h.CLS_AGNOSTIC_BBOX_REG or cfg.MODEL.ROI_HEADS.NUM_CLASSES != 1:
            raise NotImplementedError("FsodFastRCNNOutputLayers: class-agnostic boxes, one foreground class")
        self.conv_1 = nn.Conv2d(dim_in, dim_in // 2, 1, padding=0, bias=False)
        self.bbox_pred_all = nn.Linear(dim_in, 4)                         # present in checkpoints, unused at inference
        self.rcnn_reduce_dim = 256
        self.cls_score_pr = nn.Linear(49 * 49, 2)
        self.rcnn_adapt_k_layer = nn.Linear(dim_in // 2, self.rcnn_reduce_dim)
        self.rcnn_adapt_q_layer = nn.Linear(dim_in // 2, self.rcnn_reduce_dim)
        self.rcnn_unary_layer = nn.Linear(dim_in // 2, 1)                 # unused at inference
        self.bbox_pred_cor = nn.Linear(dim_in // 2, 4)
        self.cls_score_cor = nn.Linear(dim_in // 2, 2)
        self.cls_score_fc = nn.Linear(dim_in, 2)
        self.register_buffer("_pe", positional_encoding(dim_in // 2, 49), persistent=False)
        self.box_weights = tuple(float(x) for x in h.BBOX_REG_WEIGHTS)
        self.test_score_thresh = cfg.MODEL.ROI_HEADS.SCORE_THRESH_TEST
        self.test_nms_thresh = cfg.MODEL.ROI_HEADS.NMS_THRESH_TEST
        self.test_topk_per_image = cfg.TEST.DETECTIONS_PER_IMAGE

    def _conv1(self, x):
        if tcconv.supported(self.conv_1, x):      # one operand bound per ROI row (see resnet.ConvNorm)
            return tcconv.conv(x, self.conv_1, relu=True, x_amax=ops.absmax(x, per_image=True).reshape(1, -1))
        return F.relu(self.conv_1(x))

    def embed_support(self, x_support: torch.Tensor) -> Dict[str, torch.Tensor]:
        """Everything of ``forward`` that depends on the support features only (once per class and episode)."""
        s = self._conv1(x_support.contiguous(memory_format=torch.channels_last) if x_support.is_cuda else x_support)
        sup = s.reshape(1, s.shape[1], -1).transpose(1, 2) + self._pe           # [1, 49, 1024]
        k = self.rcnn_adapt_k_layer(sup)
        k = k - k.mean(1, keepdim=True)
        return {"map": s, "pooled": s.mean((2, 3)), "k": k}

    def forward(self, x_query: torch.Tensor, x_support, embedded: Optional[Dict[str, torch.Tensor]] = None):
        """x_query [R, 2048, 7, 7]; x_support [1, 2048, 7, 7] (or its ``embed_support``) -> (logits [R, 2], deltas [R, 4])
        (fsod_fast_rcnn.py:518-589)."""
        e = embedded if embedded is not None else self.embed_support(x_support)
        q = self._conv1(x_query)                                                # [R, 1024, 7, 7]
        R = q.shape[0]
        # global relation: avgpool(cat(query, support)) -> fc
        cls_fc = self.cls_score_fc(torch.cat((q.mean((2, 3)), e["pooled"].expand(R, -1)), 1))
        # local correlation: depthwise 7x7 cross-correlation = per-channel dot product over the 49 positions
        x_cor = F.relu((q * e["map"]).sum((2, 3)))
        bbox_cor, cls_cor = self.bbox_pred_cor(x_cor), self.cls_score_cor(x_cor)
        # patch relation: 49 x 49 attention between query and support positions
        query = q.reshape(R, q.shape[1], -1).transpose(1, 2) + self._pe
        qm = self.rcnn_adapt_q_layer(query)
        qm = qm - qm.mean(1, keepdim=True)
        attn = torch.matmul(qm, e["k"].transpose(1, 2)) / math.sqrt(self.rcnn_reduce_dim)
        cls_pr = self.cls_score_pr(F.softmax(attn, dim=2).reshape(R, -1))
        return cls_cor / 0.1 + cls_fc + cls_pr, bbox_cor / 0.1


@register(ROI_HEADS_REGISTRY)
class FsodRes5ROIHeads(nn.Module):
    def __init__(self, cfg, input_shape: Dict[str, ShapeSpec]):
        super().__init__()
        self.in_features = list(cfg.MODEL.ROI_HEADS.IN_FEATURES)
        h, r = cfg.MODEL.ROI_BOX_HEAD, cfg.MODEL.RESNETS
        if len(self.in_features) != 1 or h.POOLER_TYPE != "ROIAlignV2" or h.POOLER_SAMPLING_RATIO != 0 or cfg.MODEL.MASK_ON:
            raise NotImplementedError("FsodRes5ROIHeads: one input level, ROIAlignV2 with adaptive sampling, no mask head")
        self.pooler_resolution = h.POOLER_RESOLUTION
        self.stride = input_shape[self.in_features[0]].stride
        out_channels = r.RES2_OUT_CHANNELS * 8
        self.res5 = nn.Sequential(*make_stage(3, [2, 1, 1], out_channels // 2, out_channels, r.NUM_GROUPS * r.WIDTH_PER_GROUP * 8,
                                              r.STRIDE_IN_1X1))
        self.box_predictor = FsodFastRCNNOutputLayers(cfg, ShapeSpec(channels=out_channels, height=1, width=1))

    def roi_pooling(self, features: Dict[str, torch.Tensor], boxes: torch.Tensor, counts: Optional[torch.Tensor],
                    problems_per_image: int) -> torch.Tensor:
        """boxes [P, cap, 4] -> [P, cap, C, R, R] view in NHWC memory (d2 poolers.py:190-250 with one level)."""
        f = features[self.in_features[0]]
        if not f.is_cuda:
            from torchvision.ops import roi_align
            P, cap = boxes.shape[:2]
            img = torch.arange(P, device=boxes.device).div(problems_per_image, rounding_mode="floor").repeat_interleave(cap)
            rois = torch.cat((img[:, None].to(boxes.dtype), boxes.reshape(-1, 4)), 1)
            y = roi_align(f, rois, self.pooler_resolution, 1.0 / self.stride, 0, True)
            return y.reshape(P, cap, f.shape[1], self.pooler_resolution, self.pooler_resolution)
        R = self.pooler_resolution
        pooled = ops.roi_align([f], [self.stride], boxes, counts, problems_per_image, R)              # [P, cap, R*R, C]
        return pooled.reshape(boxes.shape[0], boxes.shape[1], R, R, f.shape[1]).permute(0, 1, 4, 2, 3)

    def _shared_roi_transform(self, features, boxes, counts=None, problems_per_image: int = 1):
        x = self.roi_pooling(features, boxes, counts, problems_per_image)
        P, cap = x.shape[:2]
        return self.res5(x.reshape(P * cap, *x.shape[2:]))

    @torch.no_grad()
    def eval_with_support(self, image_sizes, out_sizes, features, proposals: torch.Tensor, counts: torch.Tensor,
                          support_embedded: List[Dict[str, torch.Tensor]], class_ids: Sequence[int]):
        """fsod_roi_heads.py:143-191 for a batch: proposals [B*C, cap, 4] (problem = image-major, class-minor), counts
        [B*C]; returns padded detections (boxes [B,K,4], scores [B,K], class ids [B,K] i64, count [B] i32)."""
        C = len(class_ids)
        P, cap = proposals.shape[:2]
        box_features = self._shared_roi_transform(features, proposals, counts, C)                      # [P*cap, 2048, 7, 7]
        box_features = box_features.reshape(P, cap, *box_features.shape[1:])
        det_boxes = torch.zeros((P, cap, 4), dtype=torch.float32, device=proposals.device)
        det_scores = torch.zeros((P, cap), dtype=torch.float32, device=proposals.device)
        raw = []
        for p in range(P):
            logits, deltas = self.box_predictor(box_features[p], None, support_embedded[p % C])
            det_boxes[p] = apply_deltas(deltas.float(), proposals[p], self.box_predictor.box_weights)
            det_scores[p] = F.softmax(logits, dim=-1)[:, 0]
            raw.append((logits, deltas))
        bp = self.box_predictor
        if proposals.is_cuda:
            status = ops.new_status(proposals.device)
            hw = torch.tensor([list(s) for s in image_sizes], dtype=torch.int32, device=proposals.device)
            ohw = torch.tensor([list(s) for s in out_sizes], dtype=torch.int32, device=proposals.device)
            ob, os_, ocls, _, oc = ops.final_detect(det_boxes, det_scores, counts, C, bp.test_score_thresh, bp.test_nms_thresh,
                                                    bp.test_topk_per_image, hw, ohw, status)
            ops.check_status(status)
            ids = torch.tensor(list(class_ids), dtype=torch.int64, device=ocls.device)
            return (ob, os_, ids[ocls], oc), raw
        raise NotImplementedError("FsodRes5ROIHeads: the final class-wise NMS exists only as a CUDA kernel")
