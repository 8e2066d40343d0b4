"""Operator-level host wrappers: torch CUDA tensors in, C-ABI kernels underneath.

Every function here launches hand-written sm_100a kernels from ``libfod_b200.so``
on torch's current stream.  There is no PyTorch / CPU fallback: a CPU tensor or a
missing library is an error.

Layout: feature maps are passed as ordinary NCHW-shaped tensors but must be (or
are made) ``torch.channels_last`` in memory, which is the NHWC layout the kernels
read (include/fod_b200.h).
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import fod_level_t

Tensor = torch.Tensor
_vp = ctypes.c_void_p


def _stream() -> _vp:
    """torch's current stream of the CURRENT device; ``_chk`` makes sure the tensors live there."""
    return _vp(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[Tensor]) -> _vp:
    return _vp(0) if t is None else _vp(t.data_ptr())


def _chk(t: Tensor, dtype, name: str) -> Tensor:
    if not t.is_cuda:
        raise _lib.FodError(f"{name}: expected a CUDA tensor (the detection head has no CPU path)")
    if t.dtype != dtype:
        raise _lib.FodError(f"{name}: expected {dtype}, got {t.dtype}")
    if t.device.index != torch.cuda.current_device():
        # the launch goes to the current device's stream and the library sizes its grids from the current device
        raise _lib.FodError(f"{name}: tensor on {t.device} but the current CUDA device is {torch.cuda.current_device()}; "
                            f"wrap the call in torch.cuda.device({t.device.index})")
    return t


def nhwc(t: Tensor, name: str = "map") -> Tensor:
    """Return ``t`` ([N,C,H,W] logical) with NHWC memory (no copy if already channels_last)."""
    _chk(t, torch.float32, name)
    if t.dim() != 4:
        raise _lib.FodError(f"{name}: expected [N,C,H,W]")
    # channels_last contiguity test that also works for N==1 / C==1 corner cases
    n, c, h, w = t.shape
    if t.stride() != (h * w * c, 1, w * c, c):
        t = t.contiguous(memory_format=torch.channels_last)
        if t.stride() != (h * w * c, 1, w * c, c):   # ambiguous strides (size-1 dims): force
            t = t.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    return t


def _levels(maps: Sequence[Tensor], strides: Sequence[int]):
    arr = (fod_level_t * len(maps))()
    for i, (m, s) in enumerate(zip(maps, strides)):
        arr[i].height, arr[i].width, arr[i].stride = int(m.shape[-2]), int(m.shape[-1]), int(s)
    return arr


def _ptr_array(ts: Sequence[Tensor]):
    return (_vp * len(ts))(*[t.data_ptr() for t in ts])


# ---- zero-initialised scratch: counters, bounds and padded outputs of one pass come out of ONE pre-zeroed buffer (one
# fill kernel instead of ~30 small ones per step; profiles/r2_ncu_summary.md)
_ARENA = None


class zero_arena:
    """``with ops.zero_arena(device, nbytes):`` - inside, every zero-filled buffer the wrappers need is a 256-byte-aligned
    view of one zeroed allocation (falling back to ``torch.zeros`` when it is used up)."""

    def __init__(self, device, nbytes: int):
        self.device, self.nbytes = torch.device(device), int(nbytes)

    def __enter__(self):
        global _ARENA
        self.prev = _ARENA
        _ARENA = [torch.zeros((self.nbytes,), dtype=torch.uint8, device=self.device), 0]
        return self

    def __exit__(self, *exc):
        global _ARENA
        _ARENA = self.prev
        return False


def _zeros(shape, dtype, device) -> Tensor:
    a = _ARENA
    if a is not None and a[0].device == torch.device(device):
        n = 1
        for d in shape:
            n *= int(d)
        nbytes = n * torch.empty((), dtype=dtype).element_size()
        if a[1] + nbytes <= a[0].numel():
            off = a[1]
            a[1] = (off + nbytes + 255) // 256 * 256
            return a[0][off:off + nbytes].view(dtype).view(tuple(shape))
    return torch.zeros(tuple(shape), dtype=dtype, device=device)


def new_status(device) -> Tensor:
    return _zeros((1,), torch.int32, device)


def check_status(status: Tensor) -> None:
    """Synchronising read of the device status word; raises on any overflow bit."""
    v = int(status.item()) & 0xFFFFFFFF
    if v:
        names = [n for b, n in ((1, "candidate list overflow"), (2, "proposal capacity overflow (ties above roi_cap)"),
                                (4, "final-NMS row overflow")) if v & b]
        raise _lib.FodError("device status: " + ", ".join(names))


# --------------------------------------------------------------------------- Q1
def support_taps(proto: Tensor) -> Tensor:
    """proto [C,128,h,w] (one level, all classes) -> taps [C,7,128] (fsod_cen.py:458-460)."""
    proto = nhwc(proto, "proto")
    C, ch, h, w = proto.shape
    if ch != 128:
        raise _lib.FodError("support_taps: 128 channels expected")
    taps = torch.empty((C, 7, 128), dtype=torch.float32, device=proto.device)
    _lib.check(_lib.lib().fod_support_taps(_ptr(proto), C, h, w, _ptr(taps), _stream()), "fod_support_taps")
    return taps


# --------------------------------------------------------------------------- Q2+Q3
def correlate(q: Tensor, taps: Tensor, w3: Tensor, b3: Tensor) -> Tensor:
    """One level: q [B,128,H,W], taps [C,7,128] -> attn [B*C,128,H,W] (see correlate_levels)."""
    return correlate_levels([q], [taps], w3, b3)[0]


def _empty_nhwc(n: int, h: int, w: int, device) -> Tensor:
    """[n,128,h,w] logical, NHWC memory (explicit strides also for size-1 dims)."""
    return torch.empty((n, h, w, 128), dtype=torch.float32, device=device).permute(0, 3, 1, 2)


def correlate_levels(q: Sequence[Tensor], taps: Sequence[Tensor], w3: Tensor, b3: Tensor, want_amax: bool = False):
    """All FPN levels in one persistent tensor-core launch.
    q[l] [B,128,H_l,W_l], taps[l] [C,7,128] -> attn[l] [B*C,128,H_l,W_l] (NHWC memory), problem-major
    (fsod_cen.py:463-470, 482-491, 502-509).  ``taps`` are episode constants and travel to the kernel as launch
    parameters: pass HOST tensors (``PrototypeBank.taps_host``); CUDA tensors are copied to the host first, which
    synchronises (tests / interop only - not allowed inside a graph capture).  With ``want_amax`` also returns, per
    level, max(attn[l][p]) for every problem p as device floats [B*C] (the per-image operand bounds of the tower
    convolutions), tracked in the kernel's epilogue."""
    L = len(q)
    if L < 1 or L > 3 or len(taps) != L:
        raise _lib.FodError("correlate_levels: 1..3 levels with one taps tensor each")
    q = [nhwc(t, f"q[{i}]") for i, t in enumerate(q)]
    B, C = q[0].shape[0], taps[0].shape[0]
    taps = [t.detach().to("cpu", torch.float32).contiguous() for t in taps]
    for t, qq in zip(taps, q):
        if tuple(t.shape) != (C, 7, 128) or qq.shape[0] != B or qq.shape[1] != 128:
            raise _lib.FodError("correlate_levels: bad shapes")
    w3 = _chk(w3, torch.float32, "w3").reshape(128, 256).contiguous()
    b3 = _chk(b3, torch.float32, "b3").contiguous()
    attn = [_empty_nhwc(B * C, t.shape[2], t.shape[3], t.device) for t in q]
    lv = _levels(q, [0] * L)
    out_amax = _zeros((L, B * C), torch.float32, q[0].device) if want_amax else None
    am_ptrs = (_vp * L)(*[out_amax[i].data_ptr() for i in range(L)]) if want_amax else None
    _lib.check(_lib.lib().fod_correlate_levels(_ptr_array(q), _ptr_array(taps), lv, L, _ptr(w3), _ptr(b3),
                                               _ptr_array(attn), am_ptrs, B, C, _stream()), "fod_correlate_levels")
    if want_amax:
        return attn, [out_amax[i] for i in range(L)]       # per level: [B*C] bounds, one per problem
    return attn


# --------------------------------------------------------------------------- D1-D3
def decode_topk(hm: Sequence[Tensor], reg: Sequence[Tensor], strides: Sequence[int], score_thresh: float,
                pre_topk: int, status: Tensor, hm_is_logit: bool = True, cand_cap: Optional[int] = None,
                reg_scale: Optional[Sequence[float]] = None):
    """hm[l] [P,1,H,W], reg[l] [P,4,H,W] (either memory format; with ``reg_scale`` the raw bbox_pred output, the
    kernel applies relu(reg_scale[l] * x) = the Scale + ReLU of centernet_head.py:157-160 as it reads it) ->
    (boxes [P,cap,4], scores [P,cap], loc [P,cap] i64, level_count [P,L] i32, cand_count [P] i32)
    (fsod_rpn.py:1071-1181)."""
    L = len(hm)
    P = hm[0].shape[0]
    dev = hm[0].device
    # heat-maps: dense [P,H,W], or channel 0 of a wider NHWC buffer read in place through its pixel stride
    hms, hm_ps = [], []
    for h in hm:
        _chk(h, torch.float32, "hm")
        _, _, H, W = h.shape
        s = h.stride()
        ps = s[3] if W > 1 else (s[2] if H > 1 else 1)
        if not ((W == 1 or s[3] == ps) and (H == 1 or s[2] == W * ps) and (P == 1 or s[0] == H * W * ps) and ps >= 1):
            h, ps = h.reshape(P, H, W).contiguous(), 1
        hms.append(h)
        hm_ps.append(int(ps))
    hm = hms
    regs, cl, reg_ps = [], None, []
    for r in reg:
        _chk(r, torch.float32, "reg")
        n, c, h, w = r.shape
        try:
            ps = _pixel_stride(r, "reg")          # NHWC view, possibly a channel slice of a wider buffer
            is_cl = c > 1 and ps >= 4
        except _lib.FodError:
            ps, is_cl = 4, False
        if cl is None:
            cl = is_cl
        if is_cl != cl:
            r = nhwc(r) if cl else r.contiguous()
            ps = 4
        elif not is_cl:
            r = r.contiguous()
        regs.append(r)
        reg_ps.append(int(ps))
    cap = cand_cap if cand_cap is not None else L * pre_topk
    boxes = torch.empty((P, cap, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((P, cap), dtype=torch.float32, device=dev)
    loc = torch.empty((P, cap), dtype=torch.int64, device=dev)
    level_count = torch.empty((P, L), dtype=torch.int32, device=dev)
    cand_count = torch.empty((P,), dtype=torch.int32, device=dev)
    lv = _levels(hm, strides)
    rs = None if reg_scale is None else (ctypes.c_float * L)(*[float(v) for v in reg_scale])
    hps = (ctypes.c_int * L)(*hm_ps)
    rps = (ctypes.c_int * L)(*reg_ps) if cl else None
    _lib.check(_lib.lib().fod_decode_topk(_ptr_array(hm), _ptr_array(regs), lv, L, P, int(hm_is_logit), int(bool(cl)), hps, rps, rs,
                                          float(score_thresh), int(pre_topk), cap, _ptr(boxes), _ptr(scores), _ptr(loc),
                                          _ptr(level_count), _ptr(cand_count), _ptr(status), _stream()),
               "fod_decode_topk")
    return boxes, scores, loc, level_count, cand_count


def decode_topk_taps(taps: Sequence[Tensor], bias5: Sequence[float], strides: Sequence[int], score_thresh: float,
                     pre_topk: int, status: Tensor, reg_scale: Optional[Sequence[float]] = None,
                     cand_cap: Optional[int] = None):
    """decode_topk with the 3x3 output convolutions folded in: taps[l] [P,48,H,W] NHWC = the per-tap products of the
    stacked agn_hm | bbox_pred filter with the tower output (one 1x1 contraction; column tap = heat-map, 12 + tap*4 + j =
    regression output j); the kernel forms
    bias + the nine shifted sums as it reads (centernet_head.py:152-160, fsod_rpn.py:1071-1181).  Same outputs as
    decode_topk."""
    L = len(taps)
    P, dev = taps[0].shape[0], taps[0].device
    ps = []
    for t in taps:
        s_ = _pixel_stride(t, "taps")
        if t.shape[1] < 48 or s_ % 4:
            raise _lib.FodError("decode_topk_taps: 48 tap columns per pixel expected")
        ps.append(int(s_))
    cap = cand_cap if cand_cap is not None else L * pre_topk
    boxes = torch.empty((P, cap, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((P, cap), dtype=torch.float32, device=dev)
    loc = torch.empty((P, cap), dtype=torch.int64, device=dev)
    level_count = torch.empty((P, L), dtype=torch.int32, device=dev)
    cand_count = torch.empty((P,), dtype=torch.int32, device=dev)
    lv = _levels(taps, strides)
    rs = None if reg_scale is None else (ctypes.c_float * L)(*[float(v) for v in reg_scale])
    b5 = (ctypes.c_float * 5)(*[float(v) for v in bias5])
    ws = torch.empty((max(int(_lib.lib().fod_decode_topk_taps_workspace_bytes(lv, L, P)), 4),), dtype=torch.uint8, device=dev)
    _lib.check(_lib.lib().fod_decode_topk_taps(_ptr_array(taps), (ctypes.c_int * L)(*ps), b5, lv, L, P, rs, float(score_thresh),
                                               int(pre_topk), cap, _ptr(boxes), _ptr(scores), _ptr(loc), _ptr(level_count),
                                               _ptr(cand_count), _ptr(status), _ptr(ws), _stream()), "fod_decode_topk_taps")
    return boxes, scores, loc, level_count, cand_count


# --------------------------------------------------------------------------- N0
def nms_proposals(boxes: Tensor, scores: Tensor, count: Optional[Tensor], iou_thresh: float, post_topk: int,
                  roi_cap: int, status: Tensor):
    """-> (keep [P,roi_cap] i64, out_boxes [P,roi_cap,4], out_scores [P,roi_cap], out_count [P] i32)
    (fsod_rpn.py:1184-1210)."""
    _chk(boxes, torch.float32, "boxes"), _chk(scores, torch.float32, "scores")
    P, cap = scores.shape
    dev = boxes.device
    boxes, scores = boxes.contiguous(), scores.contiguous()
    keep = _zeros((P, roi_cap), torch.int64, dev)
    ob = _zeros((P, roi_cap, 4), torch.float32, dev)
    os_ = _zeros((P, roi_cap), torch.float32, dev)
    oc = torch.empty((P,), dtype=torch.int32, device=dev)
    _lib.check(_lib.lib().fod_nms_proposals(_ptr(boxes), _ptr(scores), _ptr(count), P, cap, float(iou_thresh),
                                            int(post_topk), int(roi_cap), _ptr(keep), _ptr(ob), _ptr(os_), _ptr(oc),
                                            _ptr(status), _stream()), "fod_nms_proposals")
    return keep, ob, os_, oc


# --------------------------------------------------------------------------- N2
def rpn_proposals(logits: Sequence[Tensor], deltas: Sequence[Tensor], anchors: Sequence[Tensor], image_hw: Tensor,
                  pre_topk: int, box_weights: Sequence[float], min_size: float, iou_thresh: float, post_topk: int,
                  out: Optional[Tuple[Tensor, Tensor, Tensor]] = None):
    """find_top_rpn_proposals (proposal_utils.py:19-119) of P problems, problem p = image p of every level ->
    (boxes [P,post_topk,4], objectness logits [P,post_topk], count [P] i32), proposals in NMS visit order.  Rows at or
    beyond count are not written: zeros in fresh outputs, untouched in ``out`` (preallocated, written in place).
    logits[l] [P,A,H,W] / deltas[l] [P,4A,H,W]: the channels of the stacked StandardRPNHead output; read in place when
    deltas[l] directly follows logits[l] in one NHWC buffer (StandardRPNHead.forward's views), stacked into one first
    otherwise.  anchors[l] [H*W*A,4] (DefaultAnchorGenerator); image_hw [P,2] int32 (height, width) on the device."""
    L = len(logits)
    if L < 1 or L > 3 or len(deltas) != L or len(anchors) != L:
        raise _lib.FodError("rpn_proposals: 1..3 levels with logits, deltas and anchors each")
    P, A = logits[0].shape[0], logits[0].shape[1]
    dev = logits[0].device
    maps, ps, ancs, slots = [], [], [], 0
    for lg, dl, an in zip(logits, deltas, anchors):
        _chk(lg, torch.float32, "logits"), _chk(dl, torch.float32, "deltas"), _chk(an, torch.float32, "anchors")
        n, a, h, w = lg.shape
        if (n, a) != (P, A) or tuple(dl.shape) != (P, 4 * A, h, w) or tuple(an.shape) != (h * w * A, 4):
            raise _lib.FodError("rpn_proposals: logits [P,A,H,W], deltas [P,4A,H,W] and anchors [H*W*A,4] per level")
        try:
            s = _pixel_stride(lg, "logits")
            in_place = dl.data_ptr() == lg.data_ptr() + 4 * A and _pixel_stride(dl, "deltas") == s
        except _lib.FodError:
            in_place = False
        if not in_place:
            lg = nhwc(torch.cat((lg, dl), 1))
            s = 5 * A
        if not an.is_contiguous() or an.data_ptr() % 16:
            an = an.clone()
        maps.append(lg)
        ps.append(int(s))
        ancs.append(an)
        slots += min(h * w * A, int(pre_topk))
    if slots > _lib.FOD_NMS_MAX_BOXES:
        raise _lib.FodError(f"rpn_proposals: {slots} candidates per problem > FOD_NMS_MAX_BOXES ({_lib.FOD_NMS_MAX_BOXES})")
    image_hw = _chk(image_hw, torch.int32, "image_hw")
    if tuple(image_hw.shape) != (P, 2) or not image_hw.is_contiguous():
        raise _lib.FodError("rpn_proposals: image_hw must be a contiguous [P, 2] int32 tensor")
    if out is None:
        out = (torch.zeros((P, post_topk, 4), dtype=torch.float32, device=dev),
               torch.zeros((P, post_topk), dtype=torch.float32, device=dev),
               torch.zeros((P,), dtype=torch.int32, device=dev))
    ob, ol, oc = out
    for t_, dt, shape, name in ((ob, torch.float32, (P, post_topk, 4), "boxes"), (ol, torch.float32, (P, post_topk), "logits"),
                                (oc, torch.int32, (P,), "count")):
        if tuple(_chk(t_, dt, name).shape) != shape or not t_.is_contiguous():
            raise _lib.FodError(f"rpn_proposals: out {name} must be a contiguous {shape} tensor")
    lv = _levels(maps, [0] * L)
    L_ = _lib.lib()
    ws = torch.empty((max(int(L_.fod_rpn_proposals_workspace_bytes(lv, L, P, A, int(pre_topk))), 16),), dtype=torch.uint8,
                     device=dev)
    bw = (ctypes.c_float * 4)(*[float(v) for v in box_weights])
    _lib.check(L_.fod_rpn_proposals(_ptr_array(maps), (ctypes.c_int * L)(*ps), _ptr_array(ancs), lv, L, P, A, _ptr(image_hw),
                                    int(pre_topk), bw, float(min_size), float(iou_thresh), int(post_topk), _ptr(ob), _ptr(ol),
                                    _ptr(oc), _ptr(ws), _stream()), "fod_rpn_proposals")
    return ob, ol, oc


# --------------------------------------------------------------------------- R1 / P1
def tile_pooled(x: Tensor) -> Tensor:
    """[P,cap,64,128] ROI rows -> the tiled operand layout [P,U,256,128,32] of relation_head (U = ceil(cap/128);
    unit u = rows 128u..128u+127, k-chunk = bin*4 + channel//32).  Test / interop helper (torch ops)."""
    P, cap = x.shape[0], x.shape[1]
    U = (cap + 127) // 128
    rows = torch.zeros((P, U * 128, 8192), dtype=x.dtype, device=x.device)
    rows[:, :cap] = x.reshape(P, cap, 8192)
    return rows.reshape(P, U, 128, 256, 32).permute(0, 1, 3, 2, 4).contiguous()


def untile_pooled(t: Tensor, cap: int) -> Tensor:
    """Inverse of tile_pooled: [P,U,256,128,32] -> [P,cap,64,128]."""
    P, U = t.shape[0], t.shape[1]
    return t.permute(0, 1, 3, 2, 4).reshape(P, U * 128, 64, 128)[:, :cap]


def roi_align(feats: Sequence[Tensor], strides: Sequence[int], rois: Tensor, roi_count: Optional[Tensor],
              problems_per_image: int, resolution: int, out: Optional[Tensor] = None, want_levels: bool = False,
              tiled: bool = False, per_roi: bool = False):
    """feats[l] [B,C,H,W] (C a multiple of 128); rois [P,cap,4] -> pooled [P,cap,R*R,C] (bin-major, channel innermost;
    R = 4, 8 or 14), or with tiled=True (R == 8, C == 128) the relation-head operand layout [P,U,256,128,32] (see
    tile_pooled) (d2 poolers.py:190-250).  R == 8 over 128-channel maps runs the tile-stationary kernel; per_roi=True
    forces the one-CTA-per-ROI kernel (fod_roi_align_per_roi: bit-identical results, kept for comparison)."""
    feats = [nhwc(f, "feat") for f in feats]
    B, ch = feats[0].shape[0], feats[0].shape[1]
    _chk(rois, torch.float32, "rois")
    rois = rois.contiguous()
    P, cap = rois.shape[0], rois.shape[1]
    if P != B * problems_per_image:
        raise _lib.FodError("roi_align: rois.shape[0] must be batch * problems_per_image")
    if ch % 128 or any(f.shape[1] != ch for f in feats):
        raise _lib.FodError("roi_align: maps with a multiple of 128 channels expected")
    dev = rois.device
    if out is None:
        shape = (P, (cap + 127) // 128, 256, 128, 32) if tiled else (P, cap, resolution * resolution, ch)
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    lvl = torch.zeros((P, cap), dtype=torch.int32, device=dev) if want_levels else None
    lv = _levels(feats, strides)
    L = _lib.lib()
    ws = torch.empty((L.fod_roi_align_workspace_bytes(P, cap, int(resolution)) // 16, 4), dtype=torch.int32, device=dev)
    fn = L.fod_roi_align_per_roi if per_roi else L.fod_roi_align_wide
    _lib.check(fn(_ptr_array(feats), lv, len(feats), B, int(problems_per_image), _ptr(rois), _ptr(roi_count), cap,
                  int(resolution), int(ch), int(bool(tiled)), _ptr(out), _ptr(lvl), _ptr(ws), _stream()), "fod_roi_align")
    return (out, lvl) if want_levels else out


# --------------------------------------------------------------------------- R2+R3
def relation_pack(w_fold: Tensor) -> Tensor:
    """Folded relation matrix [128, 8192] -> the packed operand of relation_head: scaled fp16 hi / lo planes + the scale
    (fod_conv2d_pack_weights of the matrix seen as a 1x1 convolution weight; once per weight load)."""
    w = _chk(w_fold, torch.float32, "w_fold")
    if tuple(w.shape) != (128, 8192):
        raise _lib.FodError("relation_pack: folded matrix [128, 8192] expected")
    return conv2d_pack(w.reshape(128, 8192, 1, 1))


def relation_head(pooled: Tensor, w_fold: Tensor, bias_cls: Tensor, w_out: Tensor, b_out: Tensor, rois: Tensor,
                  roi_count: Optional[Tensor], problems_per_image: int, reg_weights: Sequence[float],
                  want_raw: bool = False, x_amax: Optional[Tensor] = None):
    """-> (det_boxes [P,cap,4] unclipped, det_scores [P,cap][, logits [P,cap,2], deltas [P,cap,4]])
    (fsod_roi_heads.py:482-520, custom_fast_rcnn.py:160-170, d2 box_regression.py:77-115).
    pooled: the tiled layout [P,U,256,128,32] written by roi_align(tiled=True) (a [P,cap,64,128] tensor is
    re-tiled with torch ops first - tests only).  w_fold: the folded matrix [128,8192] or, preferably, its packed form
    (relation_pack).  x_amax: device floats bounding max|pooled| = the bounds of the feature maps the ROIAlign read:
    [k] (k = 1..8, one scale for the call) or [k, B] (per image: the rows of image b are scaled by column b, so its
    scores do not depend on its batch mates); computed from ``pooled`` when omitted, which needs the dense
    [P,cap,64,128] form."""
    P, cap = rois.shape[0], rois.shape[1]
    dev = rois.device
    if w_fold.dim() == 2:
        w_fold = relation_pack(w_fold)
    if x_amax is None:
        if pooled.dim() != 4:
            raise _lib.FodError("relation_head: x_amax (bounds of the pooled features) is required with the tiled layout")
        x_amax = absmax(pooled.contiguous())
    if pooled.dim() == 4:
        pooled = tile_pooled(pooled)
    if tuple(pooled.shape) != (P, (cap + 127) // 128, 256, 128, 32):
        raise _lib.FodError("relation_head: pooled must be [P,U,256,128,32]")
    for t, n in ((pooled, "pooled"), (w_fold, "w_fold"), (bias_cls, "bias_cls"), (w_out, "w_out"), (b_out, "b_out"),
                 (rois, "rois"), (x_amax, "x_amax")):
        _chk(t, torch.float32, n)
        if not t.is_contiguous():
            raise _lib.FodError(f"relation_head: {n} must be contiguous")
    if w_fold.numel() != _lib.lib().fod_conv2d_packed_floats(128, 8192, 1) or tuple(w_out.shape) != (6, 128) or bias_cls.shape[-1] != 128:
        raise _lib.FodError("relation_head: bad weight shapes")
    per_image = x_amax.dim() == 2
    n_amax = x_amax.shape[0] if per_image else x_amax.numel()
    if not 1 <= n_amax <= 8 or (per_image and x_amax.shape[1] * problems_per_image != P):
        raise _lib.FodError("relation_head: x_amax must be [k] or [k, B] with k = 1..8")
    det_boxes = _zeros((P, cap, 4), torch.float32, dev)
    det_scores = _zeros((P, cap), torch.float32, dev)
    logits = torch.zeros((P, cap, 2), dtype=torch.float32, device=dev) if want_raw else None
    deltas = torch.zeros((P, cap, 4), dtype=torch.float32, device=dev) if want_raw else None
    rw = (ctypes.c_float * 4)(*[float(x) for x in reg_weights])
    _lib.check(_lib.lib().fod_relation_head(_ptr(pooled), _ptr(x_amax), int(n_amax), int(per_image), _ptr(w_fold), _ptr(bias_cls),
                                            _ptr(w_out), _ptr(b_out), _ptr(rois), _ptr(roi_count), P, int(problems_per_image),
                                            cap, rw, _ptr(det_boxes), _ptr(det_scores), _ptr(logits), _ptr(deltas), _stream()),
               "fod_relation_head")
    return (det_boxes, det_scores, logits, deltas) if want_raw else (det_boxes, det_scores)


# --------------------------------------------------------------------------- R4 / N1 / O1
def final_detect(det_boxes: Tensor, det_scores: Tensor, roi_count: Optional[Tensor], problems_per_image: int,
                 score_thresh: float, iou_thresh: float, max_det: int, image_hw: Tensor, out_hw: Optional[Tensor],
                 status: Tensor):
    """-> (boxes [B,max_det,4], scores [B,max_det], classes [B,max_det] i64, rows [B,max_det] i64, count [B] i32)
    (d2 fast_rcnn.py:118-171, fsod_fast_rcnn.py:84-145, d2 postprocessing.py:9-75)."""
    P, cap = det_scores.shape
    B = P // problems_per_image
    dev = det_boxes.device
    _chk(det_boxes, torch.float32, "det_boxes"), _chk(det_scores, torch.float32, "det_scores")
    det_boxes, det_scores = det_boxes.contiguous(), det_scores.contiguous()
    ob = _zeros((B, max_det, 4), torch.float32, dev)
    os_ = _zeros((B, max_det), torch.float32, dev)
    ocls = _zeros((B, max_det), torch.int64, dev)
    orow = _zeros((B, max_det), torch.int64, dev)
    oc = torch.empty((B,), dtype=torch.int32, device=dev)
    _lib.check(_lib.lib().fod_final_detect(_ptr(det_boxes), _ptr(det_scores), _ptr(roi_count), B,
                                           int(problems_per_image), cap, float(score_thresh), float(iou_thresh),
                                           int(max_det), _ptr(image_hw), _ptr(out_hw), _ptr(ob), _ptr(os_), _ptr(ocls),
                                           _ptr(orow), _ptr(oc), _ptr(status), _stream()), "fod_final_detect")
    return ob, os_, ocls, orow, oc


# --------------------------------------------------------------------------- operator boundary
def batched_nms(boxes: Tensor, scores: Tensor, idxs: Optional[Tensor], iou_threshold: float) -> Tensor:
    """Drop-in for detectron2.layers.batched_nms (d2 nms.py:10-30): returns kept indices,
    score-descending.  Synchronises once to size the result, like the reference op."""
    _chk(boxes, torch.float32, "boxes"), _chk(scores, torch.float32, "scores")
    n = boxes.shape[0]
    dev = boxes.device
    boxes, scores = boxes.contiguous(), scores.contiguous()
    if idxs is not None:
        idxs = _chk(idxs, torch.int64, "idxs").contiguous()
    keep = torch.empty((max(n, 1),), dtype=torch.int64, device=dev)
    cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    _lib.check(_lib.lib().fod_batched_nms(_ptr(boxes), _ptr(scores), _ptr(idxs), n, float(iou_threshold), _ptr(keep),
                                          _ptr(cnt), _stream()), "fod_batched_nms")
    return keep[: int(cnt.item())]


# --------------------------------------------------------------------------- H0 (convolutions)
def _pixel_stride(t: Tensor, name: str) -> int:
    """Pixel stride (in floats) of an [N,C,H,W]-shaped NHWC view; C may be a slice of a wider buffer."""
    _chk(t, torch.float32, name)
    if t.dim() != 4:
        raise _lib.FodError(f"{name}: expected [N,C,H,W]")
    n, c, h, w = t.shape
    sn, sc, sh, sw = t.stride()
    ps = sw if w > 1 else (sh if h > 1 else c)
    ok = (c == 1 or sc == 1) and (w == 1 or sw == ps) and (h == 1 or sh == w * ps) and (n == 1 or sn == h * w * ps) and ps >= c
    if not ok:
        raise _lib.FodError(f"{name}: not an NHWC (channels_last) view: shape {tuple(t.shape)} stride {t.stride()}")
    return int(ps)


def conv2d_pack(weight: Tensor) -> Tensor:
    """PyTorch conv weight [Cout,Cin,k,k] -> tf32 hi/lo planes for conv2d_nhwc (fod_conv2d_pack_weights)."""
    weight = _chk(weight, torch.float32, "weight").contiguous()
    cout, cin, k, k2 = weight.shape
    if k != k2 or k not in (1, 3):
        raise _lib.FodError("conv2d_pack: 1x1 or 3x3 kernels")
    L = _lib.lib()
    packed = torch.empty((L.fod_conv2d_packed_floats(cout, cin, k),), dtype=torch.float32, device=weight.device)
    _lib.check(L.fod_conv2d_pack_weights(_ptr(weight), cout, cin, k, _ptr(packed), _stream()), "fod_conv2d_pack_weights")
    return packed


def absmax(x: Tensor, per_image: bool = False) -> Tensor:
    """max |x| of a dense fp32 tensor as a device float[1] (no host sync): the operand bound conv2d_nhwc needs.
    ``per_image``: one maximum per index of dim 0 instead, as device floats [N] (x_amax.reshape(1, N) of conv2d_nhwc)."""
    _chk(x, torch.float32, "x")
    if not (x.is_contiguous() or x.is_contiguous(memory_format=torch.channels_last)):
        raise _lib.FodError("absmax: dense tensor expected")
    rows = x.shape[0] if per_image else 1
    out = torch.empty((rows,), dtype=torch.float32, device=x.device)
    if rows:
        _lib.check(_lib.lib().fod_absmax_rows(_ptr(x), rows, x.numel() // rows, _ptr(out), _stream()), "fod_absmax_rows")
    return out


def new_amax(device, n: int = 1) -> Tensor:
    return _zeros((n,), torch.float32, device)


def conv2d_nhwc(x: Tensor, packed: Tensor, bias: Optional[Tensor], cout: int, ksize: int, relu: bool = False,
                out: Optional[Tensor] = None, stride: int = 1, x_amax: Optional[Tensor] = None,
                y_amax: Optional[Tensor] = None, residual: Optional[Tensor] = None, residual_upsample2: bool = False,
                a_gate: Optional[Tensor] = None, colsum: Optional[Tensor] = None, a_shift: Optional[Tensor] = None,
                a_relu: bool = False, colsumsq: Optional[Tensor] = None, x_presplit: bool = False) -> Tensor:
    """Convolution with padding ksize//2 on the tensor cores (fp16-split operands, fp32 accuracy), bias + optional
    ReLU fused.  ``x_presplit``: x is not fp32 but the kernel's own operand format, written by a producer that was given
    the bound in ``x_amax`` (stem1_u8_tc(y_bound=...)): per pixel and 16 channels [16 x fp16 hi | 16 x fp16 lo] of
    x * 2^e - the 3x3 layer then skips its conversion pass.  x [N,Cin,H,W] NHWC view (may be a channel slice of a wider channels_last buffer); ``out`` likewise.
    ``x_amax``: device floats bounding max|x|: [k] (k = 1..8 values, one scale for the batch; computed with ``absmax`` when
    omitted, which needs a dense x) or [k, N] (image n is scaled by the maximum of column n: its result does not depend
    on its batch mates); ``y_amax``: zeroed device floats that receive max|y|: [1], or [N] for one bound per image."""
    ps_x = _pixel_stride(x, "x")
    n, cin, h, w = x.shape
    pad = ksize // 2
    ho, wo = (h + 2 * pad - ksize) // stride + 1, (w + 2 * pad - ksize) // stride + 1
    if out is None:
        out = torch.empty((n, ho, wo, cout), dtype=torch.float32, device=x.device).permute(0, 3, 1, 2)
    ps_y = _pixel_stride(out, "out")
    if tuple(out.shape) != (n, cout, ho, wo):
        raise _lib.FodError("conv2d_nhwc: bad output shape")
    if bias is not None:
        bias = _chk(bias, torch.float32, "bias").contiguous()
    if x_amax is None:
        if ps_x != cin:
            raise _lib.FodError("conv2d_nhwc: x_amax is required for a channel-slice input")
        x_amax = absmax(x)
    _chk(x_amax, torch.float32, "x_amax")
    x_pi = x_amax.dim() == 2
    if x_pi and (x_amax.shape[1] != n or not x_amax.is_contiguous()):
        raise _lib.FodError("conv2d_nhwc: per-image x_amax must be a contiguous [k, N] tensor")
    n_amax = x_amax.shape[0] if x_pi else x_amax.numel()
    y_pi = False
    if y_amax is not None:
        _chk(y_amax, torch.float32, "y_amax")
        if y_amax.numel() not in (1, n):
            raise _lib.FodError("conv2d_nhwc: y_amax must hold 1 or N floats")
        y_pi = y_amax.numel() == n and n > 1
    if residual is not None:     # added before the activation; with residual_upsample2 read at (oy // 2, ox // 2)
        residual = nhwc(residual, "residual")
        rh, rw = ((ho + 1) // 2, (wo + 1) // 2) if residual_upsample2 else (ho, wo)
        if tuple(residual.shape) != (n, cout, rh, rw):
            raise _lib.FodError(f"conv2d_nhwc: residual shape {tuple(residual.shape)}, expected {(n, cout, rh, rw)}")
    if a_gate is not None:       # [N, Cin] factors multiplied into x (the eSE gate of the stage that produced x)
        a_gate = _chk(a_gate, torch.float32, "a_gate").reshape(n, cin).contiguous()
    if a_shift is not None:      # x' = act(x * a_gate + a_shift) inside the image (group_norm_affine)
        a_shift = _chk(a_shift, torch.float32, "a_shift").reshape(n, cin).contiguous()
    for name, cs in (("colsum", colsum), ("colsumsq", colsumsq)):   # [N, tiles per image, Cout] per-tile channel sums
        if cs is not None:
            _chk(cs, torch.float32, name)
            if tuple(cs.shape) != (n, conv2d_tiles_per_image(ho, wo), cout) or not cs.is_contiguous():
                raise _lib.FodError(f"conv2d_nhwc: bad {name} buffer")
    _lib.check(_lib.lib().fod_conv2d_nhwc(_ptr(x), n, h, w, cin, ps_x, _ptr(x_amax), int(n_amax), int(x_pi) | (int(y_pi) << 1) | (int(bool(x_presplit)) << 2),
                                          _ptr(packed), _ptr(bias),
                                          cout, ksize, int(stride), int(relu), _ptr(out), ps_y, _ptr(y_amax), _ptr(residual),
                                          int(residual_upsample2), _ptr(a_gate), _ptr(a_shift), int(a_relu), _ptr(colsum),
                                          _ptr(colsumsq), _stream()), "fod_conv2d_nhwc")
    return out


def conv2d_nhwc_split(x: Tensor, packed: Tensor, bias: Optional[Tensor], cout: int, ksize: int, out: Tensor,
                      x_amax: Tensor, y_amax: Optional[Tensor] = None, x_presplit: bool = False,
                      x_actual: Optional[Tensor] = None, y_bound: Optional[Tensor] = None, y_l1: float = 0.0, y_beta: float = 0.0,
                      x_presplit_from: int = -1, slice_ch: Optional[Sequence[int]] = None, colsum: Optional[Tensor] = None,
                      stride: int = 1) -> Tensor:
    """conv2d_nhwc (+ ReLU) with the split hand-off of fod_conv2d_nhwc_split: ``y_bound`` ([1, N] or [1]) makes the output
    leave in the operand format of its consumer and receives the bound that fixes its scale; ``x_presplit`` (3x3) /
    ``x_presplit_from`` + ``slice_ch`` (1x1 over a concat buffer) say which input channels arrive in that format;
    ``x_actual``: the actual max|x| per image when ``x_amax`` is such a published bound."""
    ps_x, ps_y = _pixel_stride(x, "x"), _pixel_stride(out, "out")
    n, cin, h, w = x.shape
    _chk(x_amax, torch.float32, "x_amax")
    x_pi = x_amax.dim() == 2
    if x_pi and (x_amax.shape[1] != n or not x_amax.is_contiguous()):
        raise _lib.FodError("conv2d_nhwc_split: per-image x_amax must be a contiguous [k, N] tensor")
    n_amax = x_amax.shape[0] if x_pi else x_amax.numel()
    want = n if x_pi else 1
    for name, t in (("x_actual", x_actual), ("y_bound", y_bound)):
        if t is not None and (_chk(t, torch.float32, name).numel() != want or not t.is_contiguous()):
            raise _lib.FodError(f"conv2d_nhwc_split: {name} must hold {want} float(s) like a row of x_amax")
    y_pi = y_amax is not None and y_amax.numel() == n and n > 1
    if bias is not None:
        bias = _chk(bias, torch.float32, "bias").contiguous()
    sl = None
    if slice_ch is not None:
        if len(slice_ch) != n_amax:
            raise _lib.FodError("conv2d_nhwc_split: one slice start per x_amax row")
        sl = (ctypes.c_int * len(slice_ch))(*[int(v) for v in slice_ch])
    _lib.check(_lib.lib().fod_conv2d_nhwc_split(
        _ptr(x), n, h, w, cin, ps_x, _ptr(x_amax), int(n_amax), int(x_pi) | (int(y_pi) << 1) | (int(bool(x_presplit)) << 2),
        _ptr(packed), _ptr(bias), cout, ksize, int(stride), 1, _ptr(out), ps_y, _ptr(y_amax), _ptr(colsum), _ptr(x_actual),
        _ptr(y_bound), float(y_l1), float(y_beta), int(x_presplit_from), sl, _stream()), "fod_conv2d_nhwc_split")
    return out


def conv2d_tiles_per_image(ho: int, wo: int) -> int:
    return int(_lib.lib().fod_conv2d_tiles_per_image(int(ho), int(wo)))


def ese_gate(colsum: Tensor, hw: int, fc_weight: Tensor, fc_bias: Tensor) -> Tensor:
    """Per-tile channel sums of a convolution output (conv2d_nhwc colsum) -> eSE gate [N, C]
    = relu6(fc(mean over H*W) + 3) / 6  (vovnet.py eSEModule)."""
    n, tiles, c = colsum.shape
    w = _chk(fc_weight, torch.float32, "fc_weight").reshape(c, c).contiguous()
    b = _chk(fc_bias, torch.float32, "fc_bias").contiguous()
    gate = torch.empty((n, c), dtype=torch.float32, device=colsum.device)
    _lib.check(_lib.lib().fod_ese_gate(_ptr(colsum), n, tiles, c, int(hw), _ptr(w), _ptr(b), _ptr(gate), _stream()), "fod_ese_gate")
    return gate


def group_norm_affine(colsum: Tensor, colsumsq: Tensor, hw: int, groups: int, gamma: Optional[Tensor], beta: Optional[Tensor],
                      eps: float, x_amax: Optional[Tensor] = None):
    """GroupNorm statistics from the per-tile channel sums of the producing convolution -> (scale [N,C], shift [N,C],
    bound of the normalised map as a device float): the consumer applies act(x * scale + shift) to its operand
    (conv2d_nhwc a_gate / a_shift / a_relu)."""
    n, tiles, c = colsum.shape
    dev = colsum.device
    scale = torch.empty((n, c), dtype=torch.float32, device=dev)
    shift = torch.empty((n, c), dtype=torch.float32, device=dev)
    per_map = x_amax is not None and x_amax.numel() == n and n > 1      # one bound per map in, one per map out
    bound = _zeros((n if per_map else 1,), torch.float32, dev)
    g = None if gamma is None else _chk(gamma, torch.float32, "gamma").contiguous()
    b = None if beta is None else _chk(beta, torch.float32, "beta").contiguous()
    _lib.check(_lib.lib().fod_group_norm_affine(_ptr(colsum), _ptr(colsumsq), n, tiles, c, groups, int(hw), _ptr(g), _ptr(b),
                                                float(eps), _ptr(x_amax), _ptr(scale), _ptr(shift), _ptr(bound), int(per_map),
                                                _stream()),
               "fod_group_norm_affine")
    return scale, shift, bound


def group_norm_nhwc(x: Tensor, groups: int, gamma: Optional[Tensor], beta: Optional[Tensor], eps: float,
                    relu: bool = False, inplace: bool = False, y_amax: Optional[Tensor] = None) -> Tensor:
    """GroupNorm (+ ReLU) of a dense NHWC map [N,C,H,W] (centernet_head.py:61-72); output NHWC."""
    x = nhwc(x, "x")
    n, c, h, w = x.shape
    y = x if inplace else torch.empty((n, h, w, c), dtype=torch.float32, device=x.device).permute(0, 3, 1, 2)
    L = _lib.lib()
    ws = torch.empty((L.fod_group_norm_workspace_bytes(n, groups) // 8,), dtype=torch.float64, device=x.device)
    g = None if gamma is None else _chk(gamma, torch.float32, "gamma").contiguous()
    b = None if beta is None else _chk(beta, torch.float32, "beta").contiguous()
    per_map = y_amax is not None and y_amax.numel() == n and n > 1       # [N]: one bound per map
    if y_amax is not None and y_amax.numel() not in (1, n):
        raise _lib.FodError("group_norm_nhwc: y_amax must hold 1 or N floats")
    _lib.check(L.fod_group_norm_nhwc(_ptr(x), n, h * w, c, groups, _ptr(g), _ptr(b), float(eps), int(relu), _ptr(y),
                                     _ptr(y_amax), int(per_map), _ptr(ws), _stream()), "fod_group_norm_nhwc")
    return y


# --------------------------------------------------------------------------- feature-extractor glue
def stem_patches(x: Tensor) -> Tensor:
    """x [N,3,H,W] NHWC normalised image -> [N,32,ceil(H/2),ceil(W/2)] NHWC rows of the 27 values a 3x3 / stride-2 /
    pad-1 convolution reads (k = (ky*3+kx)*3 + c, 5 zeros)."""
    x = nhwc(x, "x")
    n, c, h, w = x.shape
    if c != 3:
        raise _lib.FodError("stem_patches: 3 input channels")
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    out = torch.empty((n, ho, wo, 32), dtype=torch.float32, device=x.device).permute(0, 3, 1, 2)
    _lib.check(_lib.lib().fod_stem_patches(_ptr(x), n, h, w, _ptr(out), _stream()), "fod_stem_patches")
    return out


def stem_patches_u8(x: Tensor, mean: Sequence[float], std: Sequence[float], out: Optional[Tensor] = None) -> Tensor:
    """x [N,3,H,W] uint8 (planar, contiguous) -> normalised im2col rows [N,32,ceil(H/2),ceil(W/2)] (NHWC memory)."""
    _chk(x, torch.uint8, "x")
    if x.dim() != 4 or x.shape[1] != 3 or not x.is_contiguous():
        raise _lib.FodError("stem_patches_u8: contiguous [N,3,H,W] uint8 expected")
    n, _, h, w = x.shape
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    if out is None:
        out = torch.empty((n, ho, wo, 32), dtype=torch.float32, device=x.device).permute(0, 3, 1, 2)
    if tuple(out.shape) != (n, 32, ho, wo) or _pixel_stride(out, "out") != 32:
        raise _lib.FodError("stem_patches_u8: bad output")
    m3, s3 = (ctypes.c_float * 3)(*[float(v) for v in mean]), (ctypes.c_float * 3)(*[float(v) for v in std])
    _lib.check(_lib.lib().fod_stem_patches_u8(_ptr(x), n, h, w, m3, s3, _ptr(out), _stream()), "fod_stem_patches_u8")
    return out


def stem1_u8(x: Tensor, mean: Sequence[float], std: Sequence[float], weight: Tensor, bias: Optional[Tensor],
             y_amax: Optional[Tensor] = None) -> Tensor:
    """Raw uint8 batch [N,3,H,W] -> normalise -> stem_1 (3x3 / 2, 64 channels, BN folded into weight / bias) -> ReLU,
    one CUDA-core pass; returns [N,64,ceil(H/2),ceil(W/2)] (NHWC memory)."""
    _chk(x, torch.uint8, "x")
    if x.dim() != 4 or x.shape[1] != 3 or not x.is_contiguous():
        raise _lib.FodError("stem1_u8: contiguous [N,3,H,W] uint8 expected")
    weight = _chk(weight, torch.float32, "weight").contiguous()
    if tuple(weight.shape) != (64, 3, 3, 3):
        raise _lib.FodError("stem1_u8: weight [64,3,3,3] expected")
    if bias is not None:
        bias = _chk(bias, torch.float32, "bias").contiguous()
    n, _, h, w = x.shape
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    out = torch.empty((n, ho, wo, 64), dtype=torch.float32, device=x.device).permute(0, 3, 1, 2)
    m3, s3 = (ctypes.c_float * 3)(*[float(v) for v in mean]), (ctypes.c_float * 3)(*[float(v) for v in std])
    per_image = y_amax is not None and y_amax.numel() == n and n > 1
    if y_amax is not None and y_amax.numel() not in (1, n):
        raise _lib.FodError("stem1_u8: y_amax must hold 1 or N floats")
    _lib.check(_lib.lib().fod_stem1_u8(_ptr(x), n, h, w, m3, s3, _ptr(weight), _ptr(bias), _ptr(out), _ptr(y_amax),
                                       int(per_image), _stream()), "fod_stem1_u8")
    return out


def stem1_u8_tc(x: Tensor, mean: Sequence[float], std: Sequence[float], packed: Tensor, bias: Optional[Tensor],
                y_amax: Optional[Tensor] = None, y_bound: Optional[Tensor] = None) -> Tensor:
    """stem1_u8 on the tensor cores (fod_stem1_u8_tc): ``packed`` = conv2d_pack of the [64,32,1,1] im2col matrix with
    columns (ky*3 + kx)*3 + c (27..31 zero).  With ``y_bound`` (one device float >= every output, e.g. from the weights'
    absolute row sums and the pixel range) the output is written in the operand format of the next 3x3 convolution
    (conv2d_nhwc(..., x_amax=y_bound, x_presplit=True)) instead of fp32: same bytes, no conversion pass downstream."""
    _chk(x, torch.uint8, "x")
    if x.dim() != 4 or x.shape[1] != 3 or not x.is_contiguous():
        raise _lib.FodError("stem1_u8_tc: contiguous [N,3,H,W] uint8 expected")
    _chk(packed, torch.float32, "packed")
    if packed.numel() != 64 * 32 + 4:
        raise _lib.FodError("stem1_u8_tc: packed weights of a [64,32,1,1] matrix expected")
    if bias is not None:
        bias = _chk(bias, torch.float32, "bias").contiguous()
        if bias.numel() != 64:
            raise _lib.FodError("stem1_u8_tc: 64 bias values expected")
    n, _, h, w = x.shape
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    out = torch.empty((n, ho, wo, 64), dtype=torch.float32, device=x.device).permute(0, 3, 1, 2)
    m3, s3 = (ctypes.c_float * 3)(*[float(v) for v in mean]), (ctypes.c_float * 3)(*[float(v) for v in std])
    if y_amax is not None and y_amax.numel() not in (1, n):
        raise _lib.FodError("stem1_u8_tc: y_amax must hold 1 or N floats")
    per_image = y_amax is not None and y_amax.numel() == n and n > 1
    if y_bound is not None:
        _chk(y_bound, torch.float32, "y_bound")
        if y_bound.numel() != 1:
            raise _lib.FodError("stem1_u8_tc: y_bound must hold one float")
        _lib.check(_lib.lib().fod_stem1_u8_tc_split(_ptr(x), n, h, w, m3, s3, _ptr(packed), _ptr(bias), _ptr(out), 64, _ptr(y_amax),
                                                    int(per_image), _ptr(y_bound), _stream()), "fod_stem1_u8_tc_split")
        return out
    _lib.check(_lib.lib().fod_stem1_u8_tc(_ptr(x), n, h, w, m3, s3, _ptr(packed), _ptr(bias), _ptr(out), 64, _ptr(y_amax),
                                          int(per_image), _stream()), "fod_stem1_u8_tc")
    return out


def maxpool3x3s2_nhwc(x: Tensor, gate: Optional[Tensor] = None, out: Optional[Tensor] = None,
                      y_bound: Optional[Tensor] = None) -> Tensor:
    """nn.MaxPool2d(3, 2, ceil_mode=True) of an NHWC view, times an optional per-(image, channel) gate [N,C] (<= 1);
    ``out`` may be a channel slice of a wider NHWC buffer.  ``y_bound`` [N] (>= max|x| per image): the output leaves in
    the split hand-off format of conv2d_nhwc_split instead of fp32."""
    ps_x = _pixel_stride(x, "x")
    n, c, h, w = x.shape
    ho, wo = (h - 2) // 2 + 1, (w - 2) // 2 + 1
    if out is None:
        out = torch.empty((n, ho, wo, c), dtype=torch.float32, device=x.device).permute(0, 3, 1, 2)
    if tuple(out.shape) != (n, c, ho, wo):
        raise _lib.FodError("maxpool3x3s2_nhwc: bad output shape")
    ps_y = _pixel_stride(out, "out")
    if gate is not None:
        gate = _chk(gate, torch.float32, "gate").reshape(n, c).contiguous()
    if y_bound is not None:
        if _chk(y_bound, torch.float32, "y_bound").numel() != n or not y_bound.is_contiguous():
            raise _lib.FodError("maxpool3x3s2_nhwc: y_bound must hold N floats")
        _lib.check(_lib.lib().fod_maxpool3x3s2_nhwc_split(_ptr(x), n, h, w, c, ps_x, _ptr(gate), _ptr(out), ps_y, _ptr(y_bound),
                                                          _stream()), "fod_maxpool3x3s2_nhwc_split")
        return out
    _lib.check(_lib.lib().fod_maxpool3x3s2_nhwc(_ptr(x), n, h, w, c, ps_x, _ptr(gate), _ptr(out), ps_y, _stream()),
               "fod_maxpool3x3s2_nhwc")
    return out
