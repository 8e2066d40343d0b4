"""``CenterNet2Detector`` meta-architecture (host side of the hot path).

Drop-in for fewx/modeling/fsod/fsod_cen.py:38-571: same registry name, ``cls(cfg)``
construction, parameter names, ``forward(batched_inputs) -> [{"instances": Instances}]``
and the ``./support_dir/support_feature.pkl`` side channel.  Differences (recorded in
DESIGN.md):

  * B >= 1 query images per call (the reference asserts B == 1, :438); results equal B
    separate calls.
  * N-way episodes: every class of the pickle is scored (SURVEY section 8a row N1); the
    reference's three per-level loops keep only the last class (:454-509).
  * the pickle is read once (cached on mtime) and reduced to a device-resident
    ``PrototypeBank``; the reference reloads and re-uploads it per forward (:152-153,410-415).
  * ``MODEL.DEVICE=cpu`` is refused: the head exists only as sm_100a kernels.
"""
from __future__ import annotations

import logging
import os
import pickle
import sys
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
from torch import nn
from torch.nn import functional as F

from .. import _lib, ops
from ..compat import register, resolve, META_ARCH_REGISTRY, Boxes, ImageList, Instances
from .backbone import build_backbone
from .centernet import CenterNet, RawProposals  # noqa: F401  (registers "CenterNet")
from .prototypes import (LEVELS, PrototypeBank, SM_Block, SupportCache, bank_from_support_dict, broadcast_bank, load_bank,
                         save_bank)
from .roi_heads import build_roi_heads, instances_from_block, pack_block, pack_instances
from ..compat import PROPOSAL_GENERATOR_REGISTRY

__all__ = ["CenterNet2Detector"]


class PendingBatch:
    """A query batch that ``submit`` (CenterNet2Detector or FsodRCNN) has put on the device: its host-to-device copies,
    the forward and the device-to-host copy of the padded detections are all enqueued; ``model(pending)`` (or
    ``collect``) waits for the one event and builds the ``Instances``.  Equivalent to calling ``model(inputs)``.
    ``x_u8`` holds the device image batch (CenterNet2Detector: raw uint8; FsodRCNN: normalised and padded)."""

    __slots__ = ("inputs", "x_u8", "image_sizes", "out_sizes", "block", "host", "status_host", "done")

    def __init__(self, inputs, x_u8, image_sizes, out_sizes, block, host, status_host, done):
        self.inputs, self.x_u8, self.image_sizes, self.out_sizes = inputs, x_u8, image_sizes, out_sizes
        self.block, self.host, self.status_host, self.done = block, host, status_host, done

    def __len__(self):
        return len(self.inputs)


def build_proposal_generator(cfg, input_shape):
    return resolve(PROPOSAL_GENERATOR_REGISTRY, cfg.MODEL.PROPOSAL_GENERATOR.NAME)(cfg, input_shape)


@register(META_ARCH_REGISTRY)
class CenterNet2Detector(nn.Module):
    def __init__(self, cfg, pos_encoding=True):
        super().__init__()
        self.backbone = build_backbone(cfg)
        self.proposal_generator = build_proposal_generator(cfg, self.backbone.output_shape())
        self.roi_heads = build_roi_heads(cfg, self.backbone.output_shape())
        self.vis_period = cfg.VIS_PERIOD
        self.input_format = cfg.INPUT.FORMAT
        assert len(cfg.MODEL.PIXEL_MEAN) == len(cfg.MODEL.PIXEL_STD)
        self.register_buffer("pixel_mean", torch.Tensor(cfg.MODEL.PIXEL_MEAN).view(-1, 1, 1))
        self.register_buffer("pixel_std", torch.Tensor(cfg.MODEL.PIXEL_STD).view(-1, 1, 1))
        self.in_features = cfg.MODEL.ROI_HEADS.IN_FEATURES
        self.support_way = cfg.INPUT.FS.SUPPORT_WAY
        self.support_shot = cfg.INPUT.FS.SUPPORT_SHOT
        self.logger = logging.getLogger(__name__)
        # dense-head prototype builder (fsod_cen.py:66-75) and the relation conv on maps (:76-78)
        self.vip_p3 = SM_Block(128, 32)
        self.vip_p4 = SM_Block(128, 16)
        self.vip_p5 = SM_Block(128, 8)
        self.conv1 = nn.Conv2d(128, 64, 1)     # present in checkpoints, unused at inference (:470)
        self.conv2 = nn.Conv2d(128, 64, 1)
        self.conv3 = nn.Conv2d(256, 128, 1)
        self._support = SupportCache()
        self._bank: Optional[PrototypeBank] = None
        self._bank_key = None
        if str(cfg.MODEL.DEVICE).startswith("cpu"):
            raise _lib.FodError("MODEL.DEVICE=cpu: the detection head exists only as sm_100a CUDA kernels; "
                                "the CPU restatement lives in oracle/ and is test infrastructure")

    @property
    def device(self):
        return self.pixel_mean.device

    # ------------------------------------------------------------------ forward
    def submit(self, batched_inputs: List[dict], do_postprocess: bool = True):
        """Asynchronous half of ``forward`` (the role of the reference's DataLoader prefetch + ``.to(device)``,
        fsod_cen.py:540-555, and of its evaluator's per-image ``.to(cpu)``, fewx/evaluation/coco_evaluation.py:119-126):
        enqueue everything a batch needs - chunked host-to-device copies on the copy stream, the stem behind them, the
        graph replay, one device-to-host copy of the padded detections and of the status word - and return at once.
        A serving loop submits batch k+1 before it collects batch k (``model(pending_k)``), so the PCIe transfers and the
        host-side construction of the ``Instances`` ride under the kernels of the neighbouring batches.  Returns a
        ``PendingBatch``, or ``batched_inputs`` itself when the uint8 fast path or the CUDA graph does not apply (then
        nothing is enqueued and ``model(...)`` runs the batch synchronously).

        Contract for the caller: pinned host images are read by the copy engine AFTER this call returns - do not
        modify or free them until the batch has been collected (``model(pending)``) or abandoned (``abandon``).  Every
        PendingBatch must be collected or abandoned: the input ring holds ``U8_RING`` device buffers."""
        if self.training or not self.USE_CUDA_GRAPH:
            return batched_inputs
        with torch.cuda.device(self.device):
            return self._submit(batched_inputs, do_postprocess)

    def _submit(self, batched_inputs, do_postprocess):
        self.init_model()
        if self._bank is None:
            raise _lib.FodError("no support prototypes installed: call init_model() / set_prototypes() first")
        if getattr(self, "_in_flight", 0) >= self.U8_RING - 1:
            raise _lib.FodError(f"submit: {self._in_flight} batches are already in flight; collect one first "
                                f"(the input ring holds {self.U8_RING} buffers)")
        staged = self._stage_uint8(batched_inputs)
        if staged is None:
            return batched_inputs
        x_u8, events, chunk = staged
        n, _, h, w = x_u8.shape
        image_sizes = [(int(h), int(w))] * n
        out_sizes = [(int(inp.get("height", h)), int(inp.get("width", w))) if do_postprocess else (int(h), int(w))
                     for inp in batched_inputs]
        g = self._graph_for(n, h, w)
        self._stem_from_uint8(x_u8, events, chunk, into=(g["buf"], g["first"], g["amax"]))
        self._graph_launch(g, image_sizes, out_sizes)
        (ob, os_, ocls, orow, oc), per_roi, props, attn, status = g["res"]
        block = pack_block(ob, os_, ocls, oc)        # a fresh tensor per batch: the graph's buffers belong to the next replay
        host = torch.empty(block.shape, dtype=torch.float32, pin_memory=True)
        status_host = torch.empty((1,), dtype=status.dtype, pin_memory=True)
        host.copy_(block, non_blocking=True)
        status_host.copy_(status.view(-1)[:1], non_blocking=True)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(self.device))
        # counted only once everything is enqueued: an exception above leaves the counter untouched
        self._in_flight = getattr(self, "_in_flight", 0) + 1
        return PendingBatch(batched_inputs, x_u8, image_sizes, out_sizes, block, host, status_host, done)

    def abandon(self, pending: "PendingBatch") -> None:
        """Give up a submitted batch without building its results (its kernels still run to completion)."""
        if isinstance(pending, PendingBatch) and pending.done is not None:
            pending.done.synchronize()
            pending.done = None
            self._in_flight = max(getattr(self, "_in_flight", 0) - 1, 0)

    def collect(self, pending: "PendingBatch", do_postprocess: bool = True):
        """Wait for a submitted batch and build its results (what ``forward`` returns)."""
        if pending.done is None:
            raise _lib.FodError("collect: this PendingBatch was already collected or abandoned")
        pending.done.synchronize()
        pending.done = None
        self._in_flight = max(getattr(self, "_in_flight", 0) - 1, 0)
        st = int(pending.status_host[0]) & 0xFFFFFFFF
        if st:
            # ties above the reserved proposal slack (or an error): redo this batch eagerly with fresh buffers, stream
            # ordered behind whatever has been submitted since
            ob, os_, ocls, oc = self.head(self.features_from_uint8(pending.x_u8), pending.image_sizes, pending.out_sizes)
            results = pack_instances(ob, os_, ocls, oc, pending.out_sizes)
        else:
            results = instances_from_block(pending.block, pending.host, pending.out_sizes)
        return [{"instances": r} for r in results] if do_postprocess else results

    def forward(self, batched_inputs):
        """``batched_inputs``: list[dict] like the reference (fsod_cen.py:417), or a ``PendingBatch`` from ``submit``."""
        if not self.training:
            with torch.cuda.device(self.device):      # launches go to the model's device whatever the caller's current one
                self.init_model()
                return self.inference(batched_inputs)
        raise NotImplementedError("CenterNet2Detector: training (fsod_cen.py:156-308) is outside the inference hot path")

    # ------------------------------------------------------------------ prototypes
    def set_prototypes(self, support_dict: Dict[str, Dict[int, torch.Tensor]]) -> PrototypeBank:
        """Install an episode from an in-memory pkl-schema dict (what init_model does from disk)."""
        self._bank = bank_from_support_dict(support_dict, self.roi_heads, self.device)
        self._bank_key = ("memory", id(support_dict))
        return self._bank

    def set_bank(self, bank: PrototypeBank) -> None:
        self._bank, self._bank_key = bank, ("bank", id(bank))

    def sync_prototypes(self, src: int = 0) -> PrototypeBank:
        """Multi-GPU: rank ``src`` owns the episode, everyone else receives it over NCCL."""
        self.set_bank(broadcast_bank(self._bank, self.device, src))
        return self._bank

    def _refresh_bank_bias(self):
        """The folded per-class bias depends on the relation-head weights: recompute it when they changed (any path:
        load_state_dict on the model or on a sub-module, in-place edits, .to()), also for banks installed through
        set_prototypes / set_bank / sync_prototypes."""
        bank = self._bank
        if bank is None:
            return
        fk = self.roi_heads.fold_key()
        if bank.__dict__.get("_bias_key") != fk:
            bank.bias_cls = self.roi_heads.class_bias(bank.support_mean)
            bank.__dict__["_bias_key"] = fk

    def init_model(self):
        """fsod_cen.py:313-415.  Cache present: load it (once per file version).  Cache missing:
        build it from ./datasets/coco/10_shot_support_df.pkl, write it, and ``sys.exit(0)`` exactly
        like the reference (README.md:74 tells users to delete the cache before fine-tuning)."""
        if self._bank is not None and self._bank_key is not None and self._bank_key[0] in ("memory", "bank"):
            self._refresh_bank_bias()
            return
        os.makedirs(os.path.dirname(self._support.path) or ".", exist_ok=True)
        if not self._support.exists():
            self._build_support_cache()
            self.logger.info("=========== Offline support features are generated. ===========")
            self.logger.info("============ Few-shot object detetion will start. =============")
            sys.exit(0)
        # The pickle stays the source of truth (README.md:74: users delete it to rebuild), but it is only unpickled when it
        # changed: its (mtime, size) is checked per call, and the reduced episode (taps, support mean, folded bias) is kept
        # next to it as a binary, mmap-able file that a fresh process uploads with one copy (SURVEY 8f#2).
        src = self._support.stat_key()
        key = (os.path.abspath(self._support.path),) + tuple(src)
        if self._bank is not None and self._bank_key == key:
            self._refresh_bank_bias()
            return
        bank = None
        if os.environ.get("FOD_BINARY_PROTOTYPES", "1") == "1":
            bank = load_bank(self._support.binary_path, self.device, src)
            if bank is not None:     # taps and support mean depend on the pickle only; the folded bias on this model's weights
                bank.bias_cls = self.roi_heads.class_bias(bank.support_mean)
        if bank is None:
            bank = bank_from_support_dict(self._support.load(), self.roi_heads, self.device)
            try:
                save_bank(bank, self._support.binary_path, src)
            except OSError:
                pass
        self._bank, self._bank_key = bank, key
        self._refresh_bank_bias()

    @torch.no_grad()
    def build_support_dict(self, images_per_class: Dict[int, List[torch.Tensor]],
                           boxes_per_class: Dict[int, List[List[float]]]) -> Dict[str, Dict[int, torch.Tensor]]:
        """Rows P1+P2 (fsod_cen.py:348-389): support images -> backbone -> ROIAlign of the support
        box (CUDA kernel) + SM_Block dense prototypes -> pkl-schema dict of CPU tensors."""
        out = {k: {} for k in ("p3", "p4", "p5", "rcnn_8", "rcnn_4")}
        for cls, imgs in images_per_class.items():
            ims = [(x.to(self.device).float() - self.pixel_mean) / self.pixel_std for x in imgs]
            il = ImageList.from_tensors(ims, self.backbone.size_divisibility)
            feats = self.backbone(il.tensor.contiguous(memory_format=torch.channels_last))
            fl = [feats[f] for f in self.in_features]
            S = len(imgs)
            rois = torch.tensor(boxes_per_class[cls], dtype=torch.float32, device=self.device).reshape(S, 1, 4)
            for res, key in ((self.roi_heads.pooler_resolution, "rcnn_8"), (self.roi_heads.pooler_resolution2, "rcnn_4")):
                pooled = ops.roi_align(fl, self.roi_heads.strides, rois, None, 1, res)       # [S,1,res*res,128]
                out[key][cls] = pooled.reshape(S, res, res, 128).permute(0, 3, 1, 2).contiguous().cpu()
            for l, size, blk in (("p3", 32, self.vip_p3), ("p4", 16, self.vip_p4), ("p5", 8, self.vip_p5)):
                x = F.adaptive_avg_pool2d(feats[l], (size, size)).permute(0, 2, 3, 1)
                y = blk(x).permute(0, 3, 2, 1)                     # note the H/W swap of the reference (:371-373)
                out[l][cls] = y.mean(0, True).contiguous().cpu()
        return out

    def _build_support_cache(self):
        import pandas as pd
        df = pd.read_pickle("./datasets/coco/10_shot_support_df.pkl")
        images, boxes = {}, {}
        for cls in df["category_id"].unique():
            rows = df.loc[df["category_id"] == cls, :].reset_index()
            images[cls], boxes[cls] = [], []
            for index, row in rows.iterrows():
                if index >= self.support_shot:
                    break
                images[cls].append(_read_image_bgr(os.path.join("./datasets/coco", row["file_path"])))
                boxes[cls].append([float(v) for v in row["support_box"]])
        d = self.build_support_dict(images, boxes)
        with open(self._support.path, "wb") as f:
            pickle.dump(d, f)

    # ------------------------------------------------------------------ inference
    @torch.no_grad()
    def inference(self, batched_inputs: List[dict], detected_instances=None, do_postprocess: bool = True):
        assert not self.training
        if self._bank is None:
            raise _lib.FodError("no support prototypes installed: call init_model() / set_prototypes() first")
        if isinstance(batched_inputs, PendingBatch):
            return self.collect(batched_inputs, do_postprocess)
        staged = self._stage_uint8(batched_inputs)
        if staged is not None:
            x_u8, events, chunk = staged
            image_sizes = [(int(x_u8.shape[2]), int(x_u8.shape[3]))] * x_u8.shape[0]
        else:
            images = self.preprocess_image(batched_inputs)
            image_sizes = images.image_sizes
        out_sizes = []
        for inp, size in zip(batched_inputs, image_sizes):
            out_sizes.append((int(inp.get("height", size[0])), int(inp.get("width", size[1]))) if do_postprocess else tuple(size))
        if staged is not None:
            ob, os_, ocls, oc = self.detect_from_uint8(x_u8, image_sizes, out_sizes, events, chunk)
        else:
            ob, os_, ocls, oc = self.head(self.backbone(images.tensor), image_sizes, out_sizes)
        results = pack_instances(ob, os_, ocls, oc, out_sizes)
        return [{"instances": r} for r in results] if do_postprocess else results

    # ------------------------------------------------------------------ input staging (SURVEY 8f#4)
    PIPELINE_CHUNK = 16      # images per host-to-device chunk (measured against 32: +4 % on the synchronous path, -1 % pipelined)
    U8_RING = 3              # device input buffers per batch shape (batches in flight + 1)

    def features_from_uint8(self, x_u8: torch.Tensor, events=None, chunk: int = 0) -> Dict[str, torch.Tensor]:
        """Raw uint8 image batch [N,3,H,W] already on the device (H, W multiples of the backbone's size divisibility)
        -> FPN maps.  Normalisation is fused into the im2col kernel of stem_1.  With ``events`` (one CUDA event per
        chunk of ``chunk`` images, recorded by the stream that fills ``x_u8``) the stem of chunk k starts as soon as
        chunk k has landed, overlapping the copies of the later chunks."""
        buf, amax = self._stem_from_uint8(x_u8, events, chunk)
        vov = self.backbone.bottom_up
        return self.backbone.top_down(*vov.tc_body(buf, amax, fuse_gates=True, in_presplit=vov.stem_u8_writes_split()))

    def _stem_from_uint8(self, x_u8, events=None, chunk: int = 0, into=None):
        """stem_1..3 of a raw uint8 batch into the first slice of a stage-2 concat buffer (``into`` = (buf, first) of a
        captured graph, or a fresh one); returns the buffer."""
        vov = self.backbone.bottom_up
        n, _, h, w = x_u8.shape
        buf, first, amax = into if into is not None else vov.tc_new_input_buffer(n, h, w, x_u8.device)
        mean, std = self._mean_std_host()
        split = vov.stem_u8_writes_split()     # row 0 then receives stem_3's bound (a plain store), the last row max(y)
        amax[-1 if split else 0].zero_()
        chunk = chunk or n
        scratch = torch.zeros((2, n), dtype=torch.float32, device=x_u8.device)     # max(y) of stem_1 / stem_2 per image
        main = torch.cuda.current_stream(x_u8.device)
        for k, c0 in enumerate(range(0, n, chunk)):
            c1 = min(c0 + chunk, n)
            if events is not None:
                main.wait_event(events[k])
            vov.tc_stem_u8(x_u8[c0:c1], mean, std, first[c0:c1], amax[0, c0:c1], amax[-1, c0:c1] if split else None,
                           scratch=scratch[:, c0:c1])
        last = getattr(self, "_u8_last", None)
        if last is not None and last[2] is x_u8:     # the ring slot may be refilled once this stem has read it
            ev = torch.cuda.Event()
            ev.record(main)
            last[0]["consumed"][last[1]] = ev
        return buf, amax

    def detect_from_uint8(self, x_u8: torch.Tensor, image_sizes, out_sizes, events=None, chunk: int = 0):
        """Raw uint8 batch on the device -> padded detections (boxes, scores, classes, count): the stem eagerly (chunk by
        chunk behind the copy events), everything else as one CUDA-graph replay."""
        n, _, h, w = x_u8.shape
        if not self.USE_CUDA_GRAPH:
            return self.head(self.features_from_uint8(x_u8, events, chunk), image_sizes, out_sizes)
        g = self._graph_for(n, h, w)
        self._stem_from_uint8(x_u8, events, chunk, into=(g["buf"], g["first"], g["amax"]))
        return self._graph_replay(g, image_sizes, out_sizes)

    def _mean_std_host(self):
        key = (self.pixel_mean._version, self.pixel_std._version, self.pixel_mean.data_ptr())
        hit = getattr(self, "_mean_std_cache", None)
        if hit is None or hit[0] != key:
            hit = (key, [float(v) for v in self.pixel_mean.flatten().tolist()], [float(v) for v in self.pixel_std.flatten().tolist()])
            self._mean_std_cache = hit
        return hit[1], hit[2]

    def _features_pipelined(self, batched_inputs: List[dict]):
        """(features, image sizes) through the staged uint8 path, or (None, None) when it does not apply."""
        staged = self._stage_uint8(batched_inputs)
        if staged is None:
            return None, None
        x_u8, events, chunk = staged
        return self.features_from_uint8(x_u8, events, chunk), [(int(x_u8.shape[2]), int(x_u8.shape[3]))] * x_u8.shape[0]

    def _stage_uint8(self, batched_inputs: List[dict]):
        """Fast path of preprocess_image for the common serving case: equally sized uint8 CHW images whose size needs no
        padding.  The images are copied chunk by chunk on a side stream into one device batch; the caller runs the stem
        of chunk k behind event k while the later chunks are still in flight.  Returns (x_u8, events, chunk) or None."""
        from . import tcconv
        imgs = [x["image"] for x in batched_inputs]
        d = self.backbone.size_divisibility
        vov = getattr(self.backbone, "bottom_up", None)
        if (vov is None or not imgs or any(im.dtype != torch.uint8 or im.dim() != 3 or im.shape != imgs[0].shape
                                                                 for im in imgs)
                or imgs[0].shape[0] != 3 or imgs[0].shape[1] % d or imgs[0].shape[2] % d or self.device.type != "cuda"
                or not vov._tc_path(torch.empty((1, 3, 1, 1), device=self.device))):
            return None
        n, (c, h, w) = len(imgs), imgs[0].shape
        main = torch.cuda.current_stream(self.device)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(self.device)
        side = self._copy_stream
        # The device batch comes from a ring of U8_RING persistent buffers per batch shape: the copy stream must not wait
        # for the main stream as a whole (a submitted batch may still be running there), only for the stem that last
        # read this slot (event recorded by _stem_from_uint8).
        rings = self.__dict__.setdefault("_u8_rings", {})
        ring = rings.get((n, c, h, w))
        if ring is None:
            ring = {"bufs": [torch.empty((n, c, h, w), dtype=torch.uint8, device=self.device) for _ in range(self.U8_RING)],
                    "consumed": [None] * self.U8_RING, "next": 0}
            rings.clear()                      # one batch shape at a time
            rings[(n, c, h, w)] = ring
            side.wait_stream(main)             # the buffers were allocated on the main stream
        if any(im.is_cuda for im in imgs):
            side.wait_stream(main)             # device-resident inputs: whatever produced them on the current stream first
        j = ring["next"]
        ring["next"] = (j + 1) % self.U8_RING
        x_u8 = ring["bufs"][j]
        if ring["consumed"][j] is not None:
            side.wait_event(ring["consumed"][j])
        self._u8_last = (ring, j, x_u8)
        events, chunk = [], self.PIPELINE_CHUNK
        with torch.cuda.stream(side):
            for c0 in range(0, n, chunk):
                for i in range(c0, min(c0 + chunk, n)):
                    x_u8[i].copy_(imgs[i], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(side)
                events.append(ev)
        return x_u8, events, chunk

    @torch.no_grad()
    def head(self, features: Dict[str, torch.Tensor], image_sizes, out_sizes, want_trace: bool = False):
        """The hot path on device tensors: features[l] [B,128,H,W] -> padded detections
        (boxes [B,K,4], scores [B,K], classes [B,K] i64, count [B] i32).  No host sync except the
        final status check."""
        dev = features[self.in_features[0]].device
        image_hw = torch.tensor([list(s) for s in image_sizes], dtype=torch.int32).to(dev, non_blocking=True)
        out_hw = torch.tensor([list(s) for s in out_sizes], dtype=torch.int32).to(dev, non_blocking=True)
        with ops.zero_arena(dev, self._arena_bytes(len(image_sizes))):
            res = self._head_launch(features, image_hw, out_hw, None)
        return self._head_finish(res, features, image_hw, out_hw, want_trace)

    def _arena_bytes(self, n_images: int) -> int:
        P = n_images * max(self._bank.num_classes if self._bank is not None else 1, 1)
        return P * self.proposal_generator.roi_cap * 64 + n_images * 100 * 64 + (1 << 20)

    def _head_launch(self, features, image_hw, out_hw, cap, feature_bounds=None):
        """Kernel launches of the head only (stream-ordered, no host sync: CUDA-graph capturable).  ``feature_bounds``:
        {level: device scalar >= max|features[level]|} when the feature extractor reported them."""
        bank = self._bank
        raw = [features[f] for f in self.in_features]
        status = ops.new_status(raw[0].device)
        attn, attn_amax = ops.correlate_levels(raw, bank.taps_host, self.conv3.weight, self.conv3.bias, want_amax=True)
        props = self.proposal_generator.propose_raw(attn, status, cap, bounds=attn_amax)
        fb = None if feature_bounds is None else [feature_bounds.get(f) for f in self.in_features]
        out, per_roi = self.roi_heads.detect_raw(raw, bank.bias_cls, props.boxes, props.count, bank.num_classes, image_hw, out_hw,
                                                 status, feature_bounds=fb)
        return out, per_roi, props, attn, status

    def _head_finish(self, res, features, image_hw, out_hw, want_trace: bool = False):
        """The single sync of the head: read the status word; ties above the reserved proposal slack redo the head
        once with full capacity."""
        (ob, os_, ocls, orow, oc), per_roi, props, attn, status = res
        st = int(status.item()) & 0xFFFFFFFF
        if st & _lib.FOD_STATUS_PROPOSAL_OVERFLOW:
            res = self._head_launch(features, image_hw, out_hw, props.cand_boxes.shape[1])
            (ob, os_, ocls, orow, oc), per_roi, props, attn, status = res
            st = int(status.item()) & 0xFFFFFFFF
        if st:
            ops.check_status(status)
        if want_trace:
            return (ob, os_, ocls, oc), dict(attn=attn, proposals=props, det_boxes=per_roi[0], det_scores=per_roi[1], rows=orow)
        return ob, os_, ocls, oc

    # ------------------------------------------------------------------ CUDA graph of everything behind the stem
    USE_CUDA_GRAPH = os.environ.get("FOD_CUDA_GRAPH", "1") == "1"

    def _weights_fingerprint(self):
        """(data_ptr, version) of every parameter and buffer: changes on load_state_dict (of the model or of any
        sub-module), in-place edits, .to() / .float().  The tensor list is cached per epoch (``_apply`` and
        ``load_state_dict`` bump it; code that REPLACES Parameter objects must call ``_bump_weights_epoch``)."""
        ep = getattr(self, "_weights_epoch", 0)
        hit = self.__dict__.get("_fp_tensors")
        if hit is None or hit[0] != ep:
            hit = (ep, list(self.parameters()) + list(self.buffers()))
            self.__dict__["_fp_tensors"] = hit
        return tuple((t.data_ptr(), t._version) for t in hit[1])

    def _graph_key(self, n, h, w):
        # weights enter the captured graph as packed copies (tcconv cache, folded relation matrix, folded bias): the key
        # carries the identity and version of every parameter, so no path that changes a weight can leave a stale graph
        return (n, h, w, self._bank_key, id(self._bank), self._weights_fingerprint(), str(self.device))

    def _bump_weights_epoch(self, *args, **kwargs):
        self._weights_epoch = getattr(self, "_weights_epoch", 0) + 1

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self._bump_weights_epoch()
        return out

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._bump_weights_epoch()
        return out

    def _graph_for(self, n, h, w):
        """Captured once per (batch, image size, episode, weights): OSA stages + FPN + CenterNetHead + the head kernels
        (~140 launches, many of them a few microseconds long) replay as one graph launch.  The stem stays outside so
        that it can start on the first images while the later ones are still being copied."""
        key = self._graph_key(n, h, w)
        hit = getattr(self, "_graph", None)
        if hit is not None and hit["key"] == key:
            return hit
        dev = self.device
        vov = self.backbone.bottom_up
        buf, first, amax = vov.tc_new_input_buffer(n, h, w, dev)
        g = {"key": key, "buf": buf, "first": first, "amax": amax,
             "image_hw": torch.zeros((n, 2), dtype=torch.int32, device=dev), "out_hw": torch.zeros((n, 2), dtype=torch.int32, device=dev)}
        g["image_hw"][:] = torch.tensor([h, w], dtype=torch.int32, device=dev)
        g["out_hw"][:] = g["image_hw"]
        first.zero_()

        def run():
            with ops.zero_arena(dev, self._arena_bytes(n)):      # every counter / bound / padded output: one fill
                feats = self.backbone.top_down(*vov.tc_body(buf, amax, fuse_gates=True, in_presplit=vov.stem_u8_writes_split()))
                return feats, self._head_launch(feats, g["image_hw"], g["out_hw"], None, self.backbone.last_output_bounds)

        main = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(dev)
        side.wait_stream(main)
        with torch.cuda.stream(side):          # warm-up outside capture: weight packing, cuDNN/cuBLAS handles and plans
            for _ in range(2):
                run()
        main.wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            g["feats"], g["res"] = run()
        g["graph"] = graph
        # the graph's kernel nodes hold raw pointers into the packed weight copies and the episode tensors: keep those
        # alive for as long as the graph, whatever an eager call re-packs in the meantime
        from . import tcconv
        g["keepalive"] = ([v for v in tcconv._cache.values()], self.roi_heads._fold_cache, self._bank,
                          self._bank.bias_cls, list(self._bank.taps))
        self._graph = g
        return g

    def _graph_launch(self, g, image_sizes, out_sizes):
        # a fresh pinned block per launch: an earlier submitted batch may not have read its sizes yet
        sh = torch.tensor([[list(s) for s in image_sizes], [list(s) for s in out_sizes]], dtype=torch.int32).pin_memory()
        g["image_hw"].copy_(sh[0], non_blocking=True)
        g["out_hw"].copy_(sh[1], non_blocking=True)
        g["graph"].replay()

    def _graph_replay(self, g, image_sizes, out_sizes, want_trace: bool = False):
        self._graph_launch(g, image_sizes, out_sizes)
        return self._head_finish(g["res"], g["feats"], g["image_hw"], g["out_hw"], want_trace)

    def preprocess_image(self, batched_inputs: List[dict]) -> ImageList:
        """Normalise, pad to a multiple of 32, batch (fsod_cen.py:540-555); channels_last for cuDNN."""
        imgs = [x["image"].to(self.device, non_blocking=True) for x in batched_inputs]
        sizes = [(int(im.shape[-2]), int(im.shape[-1])) for im in imgs]
        d = self.backbone.size_divisibility
        H = (max(s[0] for s in sizes) + d - 1) // d * d
        W = (max(s[1] for s in sizes) + d - 1) // d * d
        if all(s == sizes[0] for s in sizes):
            x = (torch.stack(imgs).float() - self.pixel_mean) / self.pixel_std
            if (H, W) != sizes[0]:
                x = F.pad(x, [0, W - sizes[0][1], 0, H - sizes[0][0]], value=0.0)
        else:
            x = torch.zeros((len(imgs), imgs[0].shape[0], H, W), dtype=torch.float32, device=self.device)
            for i, im in enumerate(imgs):
                x[i, :, : sizes[i][0], : sizes[i][1]] = (im.float() - self.pixel_mean) / self.pixel_std
        return ImageList(x.contiguous(memory_format=torch.channels_last), sizes)

    @staticmethod
    def _postprocess(instances, batched_inputs, image_sizes):
        """Kept for API parity (fsod_cen.py:557-571); the rescale itself runs inside fod_final_detect."""
        return [{"instances": r} for r in instances]


def _read_image_bgr(path: str) -> torch.Tensor:
    from PIL import Image
    img = np.asarray(Image.open(path).convert("RGB"))[:, :, ::-1]
    return torch.as_tensor(np.ascontiguousarray(img.transpose(2, 0, 1)))
