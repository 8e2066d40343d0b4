"""``FsodRCNN`` meta-architecture: the R50-C4 Attention-RPN path of the reference (SURVEY 8f#3).

Drop-in for fewx/modeling/fsod/fsod_rcnn.py:36-616 at inference: same registry name, ``cls(cfg)`` construction,
parameter names (tests/golden/fsodrcnn_param_shapes.txt is the reference's own ``state_dict``), the
``./support_dir/support_feature.pkl`` side channel with its ``res4_avg`` / ``res5_avg`` schema (:344,420-428) including
the build-then-``sys.exit(0)`` branch, and ``forward(batched_inputs) -> [{"instances": Instances}]``.

What the reference computes per class c (fsod_rcnn.py:472-513), and where it runs here:

  channel_weight = sigmoid(LN(ch_wz(ch_wv(avgpool14(res4)) . softmax(ch_wq(res4_avg_c)))))      polarized channel attention
  correlation    = channel_weight * res4 + depthwise_conv1x1(res4, mean_hw(res4_avg_c))        1024-channel correlation
                 = (channel_weight + k_c) (.) res4                                              -> a per-channel gate
  proposals_c    = FsodRPN(correlation)                      3x3 conv with the gate fused into its A operand (tcgen05),
                                                             stacked 1x1 heads, fod_batched_nms
  box features   = res5(ROIAlign14(res4, proposals))         fod_roi_align_wide + tensor-core bottlenecks
  logits, deltas = FsodFastRCNNOutputLayers(box features, res5_avg_c)
  detections     = class-wise NMS over the union, top-k, rescale                               fod_final_detect

Serving: ``submit(batch)`` enqueues the whole forward without a host synchronisation - the RPN proposals of each class
are selected on the device (``FsodRPN.propose_device``, fod_rpn_proposals) - and ``model(pending)`` returns exactly what
``model(batch)`` returns, as for CenterNet2Detector.

Differences to the reference (as for CenterNet2Detector): B >= 1 query images per call, any number of proposals per
class (the reference slices ``box_features[cnt*100:(cnt+1)*100]``, fsod_roi_heads.py:172), the pickle is read once per
file version, ``MODEL.DEVICE=cpu`` is refused.
"""
from __future__ import annotations

import logging
import os
import pickle
import sys
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F
from torch import nn

from .. import _lib, ops
from ..compat import META_ARCH_REGISTRY, PROPOSAL_GENERATOR_REGISTRY, Boxes, ImageList, Instances, register, resolve
from .backbone import build_backbone
from .fsod_heads import positional_encoding
from .fsod_cen import PendingBatch
from .roi_heads import build_roi_heads, instances_from_block, pack_block, pack_instances
from . import fsod_heads, rpn  # noqa: F401  (register FsodRes5ROIHeads / FsodRPN)

__all__ = ["FsodRCNN", "ParallelPolarizedSelfAttention"]


class ParallelPolarizedSelfAttention(nn.Module):
    """fsod_rcnn.py:548-588: only the channel branch reaches the output; sp_wv / sp_wq are parameters only."""

    def __init__(self, channel: int = 1024):
        super().__init__()
        self.ch_wv = nn.Conv2d(channel, channel // 2, kernel_size=1)
        self.ch_wq = nn.Conv2d(channel, 1, kernel_size=1)
        self.ch_wz = nn.Conv2d(channel // 2, channel, kernel_size=1)
        self.ln = nn.LayerNorm(channel)
        self.sp_wv = nn.Conv2d(channel, channel // 2, kernel_size=1)
        self.sp_wq = nn.Conv2d(channel, channel // 2, kernel_size=1)

    @staticmethod
    def _conv1x1(m: nn.Conv2d, x: torch.Tensor) -> torch.Tensor:
        """A 1x1 convolution as a plain fp32 matrix product ([b, Cin, n] -> [b, Cout, n]): these maps have 196 or 1
        positions, and cuDNN would be free to use TF32 (the reference computes in fp32)."""
        return torch.matmul(m.weight.reshape(m.out_channels, -1), x.flatten(2)) + m.bias.reshape(1, -1, 1)

    def support_query(self, q: torch.Tensor) -> torch.Tensor:
        """softmax over the 14x14 positions of ch_wq(support): [1, 196, 1] (depends on the support only)."""
        return F.softmax(self._conv1x1(self.ch_wq, q).reshape(q.shape[0], -1, 1), dim=1)

    def forward(self, x: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
        b, c, _, _ = x.shape
        wv = self._conv1x1(self.ch_wv, x)                                        # [b, c/2, h*w]
        wz = torch.matmul(wv, self.support_query(q))                             # [b, c/2, 1]
        z = self._conv1x1(self.ch_wz, wz)                                        # [b, c, 1]
        return torch.sigmoid(self.ln(z.permute(0, 2, 1))).permute(0, 2, 1).reshape(b, c, 1, 1)

    def gates(self, x: torch.Tensor, wq: torch.Tensor, k: torch.Tensor) -> torch.Tensor:
        """forward for all classes at once, plus the depthwise kernel of each class: x [B, c, 14, 14] (avgpool14 of the
        query), wq [h*w, C] (support_query of every class), k [C, c] -> gates [C, B, c].  One image at a time, so that
        every matrix product has the same shape whatever the batch: cuBLAS may pick another algorithm (another
        summation order) for another shape, and an image's gates must not depend on its batch mates."""
        x = x.contiguous()
        cv, cz = self.ch_wv, self.ch_wz
        wv_w, wz_w = cv.weight.reshape(cv.out_channels, -1), cz.weight.reshape(cz.out_channels, -1)
        out = []
        for b in range(x.shape[0]):
            wv = torch.addmm(cv.bias[:, None], wv_w, x[b].reshape(x.shape[1], -1))         # [c/2, h*w]
            z = torch.addmm(cz.bias[:, None], wz_w, wv @ wq)                               # [c, C]
            out.append(torch.sigmoid(self.ln(z.t())) + k)                                 # [C, c]
        return torch.stack(out, 1)


@register(META_ARCH_REGISTRY)
class FsodRCNN(nn.Module):
    def __init__(self, cfg, pos_encoding=True):
        super().__init__()
        self.backbone = build_backbone(cfg)
        self.proposal_generator = resolve(PROPOSAL_GENERATOR_REGISTRY, cfg.MODEL.PROPOSAL_GENERATOR.NAME)(cfg, self.backbone.output_shape())
        self.roi_heads = build_roi_heads(cfg, self.backbone.output_shape())
        self.vis_period = cfg.VIS_PERIOD
        self.input_format = cfg.INPUT.FORMAT
        self.register_buffer("pixel_mean", torch.Tensor(cfg.MODEL.PIXEL_MEAN).view(-1, 1, 1))
        self.register_buffer("pixel_std", torch.Tensor(cfg.MODEL.PIXEL_STD).view(-1, 1, 1))
        self.in_features = cfg.MODEL.ROI_HEADS.IN_FEATURES
        self.support_way = cfg.INPUT.FS.SUPPORT_WAY
        self.support_shot = cfg.INPUT.FS.SUPPORT_SHOT
        self.logger = logging.getLogger(__name__)
        self.rpn_channel_k_layer = nn.Linear(1024, 1)
        self.rcnn_channel_k_layer = nn.Linear(2048, 1)
        self.pos_encoding = pos_encoding
        self.channel_attention = ParallelPolarizedSelfAttention()
        self.agp = nn.AdaptiveAvgPool2d((14, 14))
        self.register_buffer("_rpn_pe", positional_encoding(1024, 196), persistent=False)     # PositionalEncoding(max_len=196)
        self.register_buffer("_rcnn_pe", positional_encoding(2048, 49), persistent=False)
        self._episode = None
        self._episode_key = None
        self.support_path = os.path.join("support_dir", "support_feature.pkl")
        if str(cfg.MODEL.DEVICE).startswith("cpu"):
            raise _lib.FodError("MODEL.DEVICE=cpu: the detection head exists only as sm_100a CUDA kernels")

    @property
    def device(self):
        return self.pixel_mean.device

    def forward(self, batched_inputs):
        """``batched_inputs``: list[dict] like the reference, or a ``PendingBatch`` from ``submit``."""
        if self.training:
            raise NotImplementedError("FsodRCNN: training (fsod_rcnn.py:141-335) is outside the inference hot path")
        if isinstance(batched_inputs, PendingBatch):
            return self.collect(batched_inputs)
        with torch.cuda.device(self.device):
            self.init_model()
            return self.inference(batched_inputs)

    # ------------------------------------------------------------------ episode (support side)
    @torch.no_grad()
    def set_prototypes(self, support_dict: Dict[str, Dict[int, torch.Tensor]]):
        """Install an episode from a pkl-schema dict {'res4_avg': {cls: [1,1024,14,14]}, 'res5_avg': {cls: [1,2048,7,7]}}:
        everything that depends on the support only is reduced here, once."""
        class_ids = list(support_dict["res4_avg"].keys())
        dev = self.device
        k, wq, emb = [], [], []
        for c in class_ids:
            r4 = support_dict["res4_avg"][c].to(dev, torch.float32)
            k.append(r4.mean((2, 3)).reshape(1, -1))                                      # depthwise 1x1 kernel, :487
            wq.append(self.channel_attention.support_query(r4).reshape(-1, 1))
            emb.append(self.roi_heads.box_predictor.embed_support(support_dict["res5_avg"][c].to(dev, torch.float32)))
        self._episode = {"class_ids": class_ids, "k": torch.cat(k, 0), "wq": torch.cat(wq, 1), "emb": emb,
                         "weights": tuple((p.data_ptr(), p._version) for p in self.parameters())}
        self._episode_src = support_dict
        self._episode_key = ("memory", id(support_dict))

    def init_model(self):
        """fsod_rcnn.py:337-460: load the cached support features (once per file version), or build them from
        ./datasets/coco/10_shot_support_df.pkl, write the pickle and ``sys.exit(0)`` like the reference."""
        if self._episode is not None and self._episode_key[0] == "memory":
            if self._episode["weights"] != tuple((p.data_ptr(), p._version) for p in self.parameters()):
                self.set_prototypes(self._episode_src)           # the reduced episode depends on the weights
            return
        os.makedirs(os.path.dirname(self.support_path) or ".", exist_ok=True)
        if not os.path.exists(self.support_path):
            self._build_support_cache()
            self.logger.info("=========== Offline support features are generated. ===========")
            self.logger.info("============ Few-shot object detetion will start. =============")
            sys.exit(0)
        st = os.stat(self.support_path)
        key = (os.path.abspath(self.support_path), st.st_mtime_ns, st.st_size, tuple((p.data_ptr(), p._version) for p in self.parameters()))
        if self._episode_key != key:
            with open(self.support_path, "rb") as f:
                d = pickle.load(f, encoding="latin1")
            self.set_prototypes(d)
            self._episode_key = key

    @torch.no_grad()
    def build_support_dict(self, images_per_class: Dict[int, List[torch.Tensor]], boxes_per_class: Dict[int, List[List[float]]]):
        """fsod_rcnn.py:350-428: support images -> res4 -> ROIAlign 14x14 of the support box (+ res5) -> positional
        encoding, channel enhancement, shot mean -> {'res4_avg', 'res5_avg'} entries (CPU tensors)."""
        out = {"res4_avg": {}, "res5_avg": {}}
        for cls, imgs in images_per_class.items():
            ims = [(x.to(self.device).float() - self.pixel_mean) / self.pixel_std for x in imgs]
            il = ImageList.from_tensors(ims, self.backbone.size_divisibility)
            feats = self.backbone(il.tensor)
            S = len(imgs)
            rois = torch.tensor(boxes_per_class[cls], dtype=torch.float32, device=self.device).reshape(S, 1, 4)
            res4_pooled = self.roi_heads.roi_pooling(feats, rois, None, 1).reshape(S, 1024, 14, 14)
            res5 = self.roi_heads.res5(res4_pooled.contiguous(memory_format=torch.channels_last))          # [S, 2048, 7, 7]
            s_mat = res4_pooled.reshape(S, 1024, -1).transpose(1, 2).unsqueeze(1)                          # [S, 1, 196, 1024]
            q_mat = res5.reshape(S, 2048, -1).transpose(1, 2).unsqueeze(1)                                 # [S, 1, 49, 2048]
            sums, dense = [], []
            for j in range(S):
                s = s_mat[j] + self._rpn_pe if self.pos_encoding else s_mat[j]
                q = q_mat[j] + self._rcnn_pe if self.pos_encoding else q_mat[j]
                w = F.softmax(self.rpn_channel_k_layer(s), 1)
                sums.append(s + 0.5 * F.leaky_relu(torch.bmm(w.transpose(1, 2), s)))
                w2 = F.softmax(self.rcnn_channel_k_layer(q), 1)
                dense.append(q + 0.5 * F.leaky_relu(torch.bmm(w2.transpose(1, 2), q)))
            r4 = torch.stack(sums, 0).mean(0).reshape(1, -1, 14, 1024).transpose(1, 3)
            r5 = torch.stack(dense, 0).mean(0).reshape(1, -1, 7, 2048).transpose(1, 3)
            out["res4_avg"][cls] = r4.contiguous().cpu()
            out["res5_avg"][cls] = r5.contiguous().cpu()
        return out

    def _build_support_cache(self):
        import pandas as pd
        from .fsod_cen import _read_image_bgr
        df = pd.read_pickle("./datasets/coco/10_shot_support_df.pkl")
        try:        # the reference maps dataset ids to contiguous ids through detectron2's catalogue (:345-348)
            from detectron2.data import MetadataCatalog
            mapping = MetadataCatalog.get("coco_2017_train_stone").thing_dataset_id_to_contiguous_id
            df["category_id"] = df["category_id"].map(lambda i: mapping[i])
        except Exception:
            pass
        images, boxes = {}, {}
        for cls in df["category_id"].unique():
            rows = df.loc[df["category_id"] == cls, :].reset_index()
            images[cls], boxes[cls] = [], []
            for index, row in rows.iterrows():
                if index >= self.support_shot:
                    break
                images[cls].append(_read_image_bgr(os.path.join("./datasets/coco", row["file_path"])))
                boxes[cls].append([float(v) for v in row["support_box"]])
        with open(self.support_path, "wb") as f:
            pickle.dump(self.build_support_dict(images, boxes), f)

    # ------------------------------------------------------------------ inference (query side)
    def preprocess_image(self, batched_inputs, non_blocking: bool = False) -> ImageList:
        images = [(x["image"].to(self.device, non_blocking=non_blocking).float() - self.pixel_mean) / self.pixel_std
                  for x in batched_inputs]
        return ImageList.from_tensors(images, self.backbone.size_divisibility)

    @torch.no_grad()
    def inference(self, batched_inputs, detected_instances=None, do_postprocess: bool = True, want_trace: bool = False):
        if self._episode is None:
            raise _lib.FodError("no support features installed: call init_model() / set_prototypes() first")
        images = self.preprocess_image(batched_inputs)
        features = self.backbone(images.tensor)
        sizes = [tuple(s) for s in images.image_sizes]
        out_sizes = [(int(inp.get("height", s[0])), int(inp.get("width", s[1]))) if do_postprocess else s
                     for inp, s in zip(batched_inputs, sizes)]
        (ob, os_, ocls, oc), trace = self.head(features, sizes, out_sizes)
        results = pack_instances(ob, os_, ocls, oc, out_sizes)
        for r in results:       # the reference emits the support class ids as int8 (fsod_roi_heads.py:176)
            r.pred_classes = r.pred_classes.to(torch.int8)
        out = [{"instances": r} for r in results] if do_postprocess else results
        return (out, trace) if want_trace else out

    @torch.no_grad()
    def head(self, features: Dict[str, torch.Tensor], image_sizes, out_sizes):
        """res4 maps [B, 1024, H, W] -> padded detections + a trace of the per-class intermediates."""
        ep = self._episode
        res4, gates, bounds = self._rpn_gates(features)
        B, C = res4.shape[0], len(ep["class_ids"])
        trace = {"gate": [], "proposals": []}
        cap = self.proposal_generator.post_nms_topk
        props = torch.zeros((B, C, cap, 4), dtype=torch.float32, device=res4.device)
        counts = torch.zeros((B, C), dtype=torch.int32, device=res4.device)
        fake_images = type("Sizes", (), {"image_sizes": image_sizes})()
        for ci in range(C):
            gate = gates[ci]                                                        # channel_att + spatial_att = gate (.) res4
            plist, _ = self.proposal_generator(fake_images, {self.proposal_generator.in_features[0]: res4}, None,
                                               gates=[gate], bounds=[bounds[ci]])
            trace["gate"].append(gate)
            trace["proposals"].append(plist)
            for b, p in enumerate(plist):
                n = len(p)
                props[b, ci, :n] = p.proposal_boxes.tensor
                counts[b, ci] = n
        res, raw = self.roi_heads.eval_with_support(image_sizes, out_sizes, {self.in_features[0]: res4}, props.reshape(B * C, cap, 4),
                                                    counts.reshape(-1), ep["emb"], ep["class_ids"])
        trace["raw"] = raw
        return res, trace

    def _rpn_gates(self, features: Dict[str, torch.Tensor]):
        """The preamble of ``head``: res4 (NHWC), the correlation gate of every class [C, B, 1024] and, per class, the
        per-image bound [1, B] of the gated map that the RPN's 3x3 convolution reads."""
        ep = self._episode
        res4 = features["res4"]
        if res4.is_cuda:
            res4 = ops.nhwc(res4, "res4")
        B = res4.shape[0]
        gates = self.channel_attention.gates(self.agp(res4), ep["wq"], ep["k"])      # [C, B, 1024]: (:480-488)
        amax = ops.absmax(res4, per_image=True)                                     # per image: no batch-mate coupling
        return res4, gates, [(amax * gate.abs().amax(1)).reshape(1, B) for gate in gates]

    # ------------------------------------------------------------------ serving (submit / collect)
    def submit(self, batched_inputs: List[dict], do_postprocess: bool = True) -> PendingBatch:
        """Asynchronous half of ``forward``, as CenterNet2Detector.submit: enqueue everything a batch needs - non-blocking
        host-to-device copies of the images, the backbone, the RPN of every class with its proposals selected on the
        device (``FsodRPN.propose_device``), the ROI head, one device-to-host copy of the padded detections and of the
        status word - and return at once.  A serving loop submits batch k+1 before it collects batch k
        (``model(pending_k)``), so the host work of one batch runs under the kernels of the other.  ``model(pending)``
        returns what ``model(batched_inputs)`` returns.

        Contract for the caller: pinned host images are read by the copy engine after this call returns - do not modify
        or free them until the batch has been collected or abandoned (``abandon``)."""
        if self.training:
            raise NotImplementedError("FsodRCNN: training (fsod_rcnn.py:141-335) is outside the inference hot path")
        with torch.cuda.device(self.device):
            self.init_model()
            return self._submit(batched_inputs, do_postprocess)

    @torch.no_grad()
    def _submit(self, batched_inputs, do_postprocess):
        ep = self._episode
        if ep is None:
            raise _lib.FodError("no support features installed: call init_model() / set_prototypes() first")
        images = self.preprocess_image(batched_inputs, non_blocking=True)
        features = self.backbone(images.tensor)
        sizes = [tuple(s) for s in images.image_sizes]
        out_sizes = [(int(inp.get("height", s[0])), int(inp.get("width", s[1]))) if do_postprocess else s
                     for inp, s in zip(batched_inputs, sizes)]
        res4, gates, bounds = self._rpn_gates(features)
        B, C = res4.shape[0], len(ep["class_ids"])
        rpn = self.proposal_generator
        cap, dev = rpn.post_nms_topk, res4.device
        # class-major here, so that each class's outputs are contiguous; the ROI head takes them image-major like head's
        props = torch.zeros((C, B, cap, 4), dtype=torch.float32, device=dev)
        logits = torch.empty((C, B, cap), dtype=torch.float32, device=dev)
        counts = torch.zeros((C, B), dtype=torch.int32, device=dev)
        image_hw = fsod_heads.upload([list(s) for s in sizes], torch.int32, dev)
        for ci in range(C):
            rpn.propose_device([res4], image_hw, [gates[ci]], [bounds[ci]], props[ci], logits[ci], counts[ci])
        (ob, os_, ocls, oc), _, status = self.roi_heads.launch_with_support(
            sizes, out_sizes, {self.in_features[0]: res4}, props.transpose(0, 1).reshape(B * C, cap, 4),
            counts.t().reshape(-1), ep["emb"], ep["class_ids"])
        block = pack_block(ob, os_, ocls, oc)
        host = torch.empty(block.shape, dtype=torch.float32, pin_memory=True)
        status_host = torch.empty((1,), dtype=status.dtype, pin_memory=True)
        host.copy_(block, non_blocking=True)
        status_host.copy_(status.view(-1)[:1], non_blocking=True)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(dev))
        return PendingBatch(batched_inputs, images.tensor, sizes, out_sizes, block, host, status_host, done)

    def collect(self, pending: PendingBatch, do_postprocess: bool = True):
        """Wait for a submitted batch and build its results (what ``forward`` returns)."""
        if pending.done is None:
            raise _lib.FodError("collect: this PendingBatch was already collected or abandoned")
        pending.done.synchronize()
        pending.done = None
        ops.check_status(pending.status_host)
        results = instances_from_block(pending.block, pending.host, pending.out_sizes)
        for r in results:       # the reference emits the support class ids as int8 (fsod_roi_heads.py:176)
            r.pred_classes = r.pred_classes.to(torch.int8)
        return [{"instances": r} for r in results] if do_postprocess else results

    def abandon(self, pending: PendingBatch) -> None:
        """Give up a submitted batch without building its results (its kernels still run to completion)."""
        if pending.done is not None:
            pending.done.synchronize()
            pending.done = None
