"""FsodRCNN served through submit / collect: the device RPN proposal selection (ops.rpn_proposals, fod_rpn_proposals)
bit for bit against FsodRPN.predict_proposals and against a stable CPU-sorted reference, its writes, and
model(model.submit(batch)) against model(batch)."""
import math

import numpy as np
import pytest
import torch

from faster_orefsdet_b200 import _lib, ops, synth
from faster_orefsdet_b200.compat import Boxes, ShapeSpec
from faster_orefsdet_b200.modeling.rpn import FsodRPN, apply_deltas
from oracle import head_oracle as O
from tests.test_fsodrcnn_cpu import build, param_shapes
from tests.test_fsodrcnn_gpu import fsodrcnn_support
from tests.test_guards_gpu import GuardedTorch

pytestmark = pytest.mark.gpu
DEV = "cuda"


# ---------------------------------------------------------------------------------------------- the op
def _rpn(levels=1, pre=6000, post=100, min_size=0):
    from faster_orefsdet_b200.config import get_cfg
    import faster_orefsdet_b200.modeling  # noqa: F401
    import os
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(os.path.dirname(os.path.dirname(__file__)), "configs/fsod/Base-FSOD-C4.yaml"))
    cfg.MODEL.RPN.IN_FEATURES = ["res4", "res5"][:levels]
    cfg.MODEL.RPN.PRE_NMS_TOPK_TEST, cfg.MODEL.RPN.POST_NMS_TOPK_TEST = pre, post
    cfg.MODEL.PROPOSAL_GENERATOR.MIN_SIZE = min_size
    shapes = {"res4": ShapeSpec(channels=1024, stride=16), "res5": ShapeSpec(channels=1024, stride=32)}
    return FsodRPN(cfg, shapes).to(DEV).eval()


def _head_out(P, H, W, A, seed, delta_scale=0.3, pad=3):
    """A stacked StandardRPNHead output [P, 5A + pad, H, W] in NHWC memory: logits in channels 0..A-1, deltas after."""
    g = torch.Generator().manual_seed(seed)
    y = torch.randn((P, H, W, 5 * A + pad), generator=g)
    y[..., A:5 * A] *= delta_scale
    return y.to(DEV).permute(0, 3, 1, 2)


def _A(rpn):
    return rpn.anchor_generator.num_anchors[0]


def _eager(rpn, ys, sizes):
    """FsodRPN.forward after its rpn_head call."""
    A = _A(rpn)
    lg = [y[:, :A].permute(0, 2, 3, 1).flatten(1) for y in ys]
    dl = [y[:, A:5 * A].reshape(y.shape[0], -1, 4, y.shape[-2], y.shape[-1]).permute(0, 3, 4, 1, 2).flatten(1, -2) for y in ys]
    return rpn.predict_proposals(rpn.anchor_generator(ys), lg, dl, sizes)


def _device(rpn, ys, sizes, out=None):
    A = _A(rpn)
    hw = torch.tensor(sizes, dtype=torch.int32, device=DEV)
    return ops.rpn_proposals([y[:, :A] for y in ys], [y[:, A:5 * A] for y in ys], rpn.anchor_generator(ys), hw,
                             rpn.pre_nms_topk, rpn.box_weights, rpn.min_box_size, rpn.nms_thresh, rpn.post_nms_topk, out=out)


def _assert_same(ref, got):
    """ref: per problem (boxes, logits); got: the op's padded outputs."""
    ob, ol, oc = got
    assert oc.shape[0] == len(ref)
    for p, (b, s) in enumerate(ref):
        n = b.shape[0]
        assert int(oc[p]) == n, f"problem {p}: {int(oc[p])} proposals, the reference has {n}"
        assert torch.equal(ob[p, :n], b), f"problem {p}: boxes differ"
        assert torch.equal(ol[p, :n], s), f"problem {p}: logits differ"


def _instances(ref):
    return [(i.proposal_boxes.tensor, i.objectness_logits) for i in ref]


# name: (levels [(H, W)], image sizes, pre, post, min_size, modification of the head output)
CASES = {
    "small_1200_anchors": ([(8, 10)], [(128, 160), (100, 150)], 1000, 100, 0, None),
    "all_anchors_selected": ([(8, 10)], [(128, 160)], 6000, 1000, 0, None),
    "tiny_fewer_than_post_topk": ([(3, 4)], [(48, 64), (40, 60)], 6000, 1000, 0, None),
    "over_6000_anchors": ([(24, 20)], [(384, 320), (300, 250), (384, 200)], 6000, 100, 0, None),
    "res4_of_1333x800": ([(50, 84)], [(800, 1333), (760, 1300)], 6000, 1000, 0, None),
    "classes_stacked": ([(24, 20)], [(384, 320), (384, 320), (300, 250), (300, 250)], 6000, 100, 0, None),
    "deltas_beyond_clamp": ([(24, 20)], [(384, 320), (300, 250)], 6000, 100, 0, "clamp"),
    "boxes_outside_image": ([(24, 20)], [(384, 320), (200, 150)], 6000, 100, 0, "outside"),
    "min_size": ([(24, 20)], [(384, 320), (300, 250)], 6000, 100, 16, None),
    "zero_survivors": ([(8, 10)], [(128, 160), (128, 160)], 1000, 100, 0, "empty1"),
    "two_levels": ([(16, 20), (8, 10)], [(256, 320), (250, 300)], 1000, 100, 0, None),
}


def _modify(y, A, how):
    d = y[:, A:5 * A]                    # a view: writes go into y
    if how == "clamp":                   # dw, dh up to ~12, beyond log(1000/16)
        d[:, 2::4] *= 40.0
        d[:, 3::4] *= 40.0
    elif how == "outside":               # centres moved far out of the image
        d[:, 0::4] *= 60.0
        d[:, 1::4] *= 60.0
    elif how == "empty1":                # image 1: every box right of the image, width 0 after the clip
        d[1, 0::4] = 1e4


@pytest.mark.parametrize("name", list(CASES))
def test_rpn_proposals_equal_predict_proposals(name):
    levels, sizes, pre, post, min_size, how = CASES[name]
    rpn = _rpn(len(levels), pre, post, min_size)
    A = _A(rpn)
    ys = [_head_out(len(sizes), H, W, A, 100 + 7 * l + len(name)) for l, (H, W) in enumerate(levels)]
    if how:
        _modify(ys[0], A, how)
    ref = _instances(_eager(rpn, ys, sizes))
    got = _device(rpn, ys, sizes)
    _assert_same(ref, got)
    if how == "empty1":
        assert int(got[2][1]) == 0 and int(got[2][0]) > 0
    if name.startswith("tiny"):
        assert int(got[2].max()) < post


def _stable_reference(rpn, ys, sizes):
    """find_top_rpn_proposals with the top-k of a stable CPU sort (NumPy), then the eager decode / filter / clip and the
    oracle's coordinate-trick NMS (torchvision's CPU kernel)."""
    A, L = _A(rpn), len(ys)
    anchors = rpn.anchor_generator(ys)
    out = []
    for p, size in enumerate(sizes):
        bs, ss, lvs = [], [], []
        for l, (y, anc) in enumerate(zip(ys, anchors)):
            H, W = y.shape[-2:]
            lg = y[p, :A].permute(1, 2, 0).reshape(-1)
            dl = y[p, A:5 * A].reshape(A, 4, H, W).permute(2, 3, 0, 1).reshape(-1, 4)
            k = min(lg.numel(), rpn.pre_nms_topk)
            order = torch.from_numpy(np.argsort(-lg.cpu().numpy(), kind="stable")[:k]).to(DEV)
            bs.append(apply_deltas(dl[order], anc[order], rpn.box_weights))
            ss.append(lg[order])
            lvs.append(torch.full((k,), l, dtype=torch.int64, device=DEV))
        b, s, lv = torch.cat(bs), torch.cat(ss), torch.cat(lvs)
        valid = torch.isfinite(b).all(1) & torch.isfinite(s)
        b, s, lv = b[valid], s[valid], lv[valid]
        boxes = Boxes(b.contiguous())
        boxes.clip(size)
        keep = boxes.nonempty(threshold=rpn.min_box_size)
        b, s, lv = boxes.tensor[keep], s[keep], lv[keep]
        idx = lv.cpu() if L > 1 else torch.zeros(len(s), dtype=torch.int64)
        keep = O.batched_nms_coordinate_trick(b.cpu(), s.cpu(), idx, rpn.nms_thresh)[: rpn.post_nms_topk].to(DEV)
        out.append((b[keep], s[keep]))
    return out


@pytest.mark.parametrize("levels,pre", [([(8, 10)], 1000), ([(24, 20)], 6000), ([(16, 20), (8, 10)], 1000)])
def test_rpn_proposals_ties_follow_a_stable_sort(levels, pre):
    """Logits on a coarse grid (hundreds of equal values, also across the top-k cut) and signed zeros: the selection, the
    NMS visit order and the cut follow a stable descending sort (lower anchor index first, lower level first)."""
    rpn = _rpn(len(levels), pre, 100)
    A = _A(rpn)
    sizes = [(16 * levels[0][0], 16 * levels[0][1]), (16 * levels[0][0] - 20, 16 * levels[0][1] - 30)]
    ys = [_head_out(len(sizes), H, W, A, 300 + l) for l, (H, W) in enumerate(levels)]
    for y in ys:
        lg = y[:, :A]
        lg.copy_(torch.round(lg * 2.0) / 2.0)
        lg[lg == 0] = torch.where(torch.arange(int((lg == 0).sum()), device=DEV) % 2 == 0, 0.0, -0.0)
    _assert_same(_stable_reference(rpn, ys, sizes), _device(rpn, ys, sizes))


@pytest.mark.parametrize("H,W", [(8, 10), (24, 20)])
def test_rpn_proposals_nan_and_inf_like_the_eager_path(H, W):
    """NaN ranks above +inf in the selection and takes a slot; rows with a non-finite logit or box are dropped
    afterwards; NaN / inf deltas make non-finite boxes (the clamp lets NaN through)."""
    rpn = _rpn(1, 1000, 100)
    A = _A(rpn)
    sizes = [(16 * H, 16 * W), (16 * H - 10, 16 * W - 20)]
    y = _head_out(2, H, W, A, 500 + H)
    g = torch.Generator().manual_seed(H)
    flat = y.permute(0, 2, 3, 1)                      # [P, H, W, C] view of the same memory
    for val, ch in ((float("nan"), 0), (float("inf"), 0), (-float("inf"), 0), (float("nan"), 1), (float("inf"), 1),
                    (-float("inf"), 1)):
        for _ in range(40):
            p, yy, xx = [int(torch.randint(0, m, (1,), generator=g)) for m in (2, H, W)]
            a = int(torch.randint(0, A, (1,), generator=g))
            c = a if ch == 0 else A + 4 * a + int(torch.randint(0, 4, (1,), generator=g))
            flat[p, yy, xx, c] = val
    _assert_same(_instances(_eager(rpn, [y], sizes)), _device(rpn, [y], sizes))


def test_rpn_proposals_write_nothing_outside_their_outputs(monkeypatch):
    """Guard bands around the outputs and the workspace stay intact, the inputs are not written, rows at or beyond the
    count keep the fill of the output buffers, and the valid rows do not depend on the fill of outputs or workspace."""
    rpn = _rpn(2, 1000, 1000)
    A = _A(rpn)
    sizes = [(256, 320), (250, 300), (200, 160)]
    ys = [_head_out(3, H, W, A, 700 + H) for H, W in ((16, 20), (8, 10))]
    _modify(ys[0], A, "outside")
    before = [y.clone() for y in ys]
    P, post, G = len(sizes), rpn.post_nms_topk, 4096
    results = []
    for fill in (0xA5, 0xFF, 0x00):
        bufs, outs = [], []
        for shape, dt in (((P, post, 4), torch.float32), ((P, post), torch.float32), ((P,), torch.int32)):
            n = math.prod(shape)
            buf = torch.empty(n + 2 * G, dtype=dt, device=DEV)
            buf.view(torch.uint8).fill_(fill)
            bufs.append((buf, n))
            outs.append(buf[G:G + n].view(shape))
        g = GuardedTorch(fill)
        monkeypatch.setattr(ops, "torch", g)
        ob, ol, oc = _device(rpn, ys, sizes, out=tuple(outs))
        g.check()
        monkeypatch.undo()
        torch.cuda.synchronize()
        for buf, n in bufs:
            b = buf.view(torch.uint8)
            es = buf.element_size()
            assert bool((b[:G * es] == fill).all()) and bool((b[(G + n) * es:] == fill).all()), "a guard band was written"
        for p in range(P):
            n = int(oc[p])
            assert n < post, "the case must leave unused rows"
            assert bool((ob[p, n:].view(torch.uint8) == fill).all()) and bool((ol[p, n:].view(torch.uint8) == fill).all())
        for y, y0 in zip(ys, before):
            assert torch.equal(y.contiguous().view(torch.uint8), y0.contiguous().view(torch.uint8)), "an input was written"
        results.append([(ob[p, :int(oc[p])].clone(), ol[p, :int(oc[p])].clone()) for p in range(P)])
    for other in results[1:]:
        for (b0, s0), (b1, s1) in zip(results[0], other):
            assert torch.equal(b0.view(torch.uint8), b1.view(torch.uint8)) and torch.equal(s0.view(torch.uint8), s1.view(torch.uint8))
    _assert_same(_instances(_eager(rpn, ys, sizes)), (ob, ol, oc))


def test_rpn_proposals_capacity_is_checked_from_shapes():
    rpn = _rpn(2, 6000, 100)
    A = _A(rpn)
    ys = [_head_out(1, 24, 20, A, 1), _head_out(1, 12, 10, A, 2)]     # 6000 + 1800 fits, one more level would not
    _device(rpn, ys, [(384, 320)])
    ys = [_head_out(1, 24, 20, A, 1), _head_out(1, 24, 20, A, 2)]     # 12000 candidates > FOD_NMS_MAX_BOXES
    with pytest.raises(_lib.FodError):
        _device(rpn, ys, [(384, 320)])


# ---------------------------------------------------------------------------------------------- submit / collect
@pytest.fixture(scope="module")
def model():
    m = build().cuda()
    m.load_state_dict(synth.state_dict(param_shapes()))
    return m


def _batch(specs, seed):
    """specs: (h, w) or (h, w, out_h, out_w); pinned uint8 images"""
    out = []
    for i, s in enumerate(specs):
        d = {"image": synth.ore_image(s[0], s[1], seed + i).pin_memory()}
        if len(s) == 4:
            d["height"], d["width"] = s[2], s[3]
        out.append(d)
    return out


def _assert_results_equal(got, ref):
    assert len(got) == len(ref)
    for g, r in zip(got, ref):
        gi, ri = g["instances"], r["instances"]
        assert gi.image_size == ri.image_size and len(gi) == len(ri)
        assert torch.equal(gi.pred_boxes.tensor, ri.pred_boxes.tensor) and torch.equal(gi.scores, ri.scores)
        assert gi.pred_classes.dtype == torch.int8 and torch.equal(gi.pred_classes, ri.pred_classes)
        gc, rc = gi.to("cpu"), ri.to("cpu")
        assert torch.equal(gc.pred_boxes.tensor, rc.pred_boxes.tensor) and torch.equal(gc.scores, rc.scores)
        assert gc.pred_classes.dtype == torch.int8 and torch.equal(gc.pred_classes, rc.pred_classes)


SUBMIT_CASES = {
    "batch1_2way": ([3, 9], [(160, 192)]),
    "batch2_2way": ([3, 9], [(160, 192), (160, 192)]),
    "batch5_mixed_sizes": ([3, 9], [(160, 192), (128, 160, 256, 320), (192, 160), (48, 64), (160, 192, 100, 120)]),
    "batch2_1way": ([5], [(160, 192), (128, 128, 200, 200)]),
    "small_query": ([3, 9], [(48, 64)]),
}


@pytest.mark.parametrize("name", list(SUBMIT_CASES))
def test_submit_equals_the_plain_call(model, name):
    classes, specs = SUBMIT_CASES[name]
    model.set_prototypes(fsodrcnn_support(classes, 11))
    b = _batch(specs, 4000 + len(name))
    ref = model(b)
    _assert_results_equal(model(model.submit(b)), ref)
    if name == "small_query":
        _, trace = model.inference(b, want_trace=True)
        assert min(len(p[0]) for p in trace["proposals"]) < model.proposal_generator.post_nms_topk


def test_submit_ahead_of_collect(model):
    """Batch k+1 is submitted before batch k is collected; every result equals its plain call."""
    model.set_prototypes(fsodrcnn_support([3, 9], 11))
    batches = [_batch([(160, 192), (128, 160)], 5000 + 10 * k) for k in range(3)]
    refs = [model(b) for b in batches]
    pend = [model.submit(batches[0]), model.submit(batches[1])]
    got = [model(pend[0])]
    pend.append(model.submit(batches[2]))
    got += [model(pend[1]), model(pend[2])]
    for g, r in zip(got, refs):
        _assert_results_equal(g, r)


def test_abandon_and_second_collect_raise(model):
    model.set_prototypes(fsodrcnn_support([3, 9], 11))
    b = _batch([(160, 192)], 6000)
    p = model.submit(b)
    model.abandon(p)
    with pytest.raises(_lib.FodError):
        model(p)
    p = model.submit(b)
    _assert_results_equal(model(p), model(b))
    with pytest.raises(_lib.FodError):
        model.collect(p)


def test_submit_does_not_synchronise(model):
    """After one warm-up, submit enqueues the whole batch without a host synchronisation (the C ABI never synchronises;
    this covers the torch side)."""
    model.set_prototypes(fsodrcnn_support([3, 9], 11))
    b = _batch([(160, 192), (160, 192)], 7000)
    ref = model(model.submit(b))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        p = model.submit(b)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    _assert_results_equal(model(p), ref)
