"""Stage-by-stage parity of the FsodRCNN CUDA path (SURVEY 8f#3) against what the UNMODIFIED reference recorded
(tests/golden/make_golden_fsodrcnn.py -> fsodrcnn.npz), cases a (1-way) and b (2-way).

Every stage is teacher-forced: it gets the reference's recorded input (or, where only a subsample was recorded, the
output of the previous CUDA stage after that stage has been checked), so an error of one stage cannot hide behind
another.  The index stages (RPN NMS, class-wise NMS + top-k + rescale) are compared bit for bit with the oracle on the
CUDA path's own inputs.  Order differences of proposals / detections are accepted only between entries whose recorded
scores are closer than the score error measured on the same call.

Padding rows and batch mates: per-problem ROI batches are padded to POST_NMS_TOPK rows; what the ROI head computes for
the valid rows must not depend on the padding (filled here with 2.98e29, 3.39e38 and NaN bytes), and an image's
detections must not depend on the other images of the batch.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from faster_orefsdet_b200 import ops, synth
from faster_orefsdet_b200.modeling.rpn import apply_deltas
from oracle import head_oracle as O
from tests.test_fsodrcnn_cpu import build, param_shapes, teacher_forced_inputs
from tests.test_fsodrcnn_gpu import fsodrcnn_support
from tests.test_guards_gpu import GuardedTorch
from tests.util import golden, t

pytestmark = pytest.mark.gpu
DEV = "cuda"
TAGS = ["a", "b"]


def _model():
    model = build().cuda()
    model.load_state_dict(synth.state_dict(param_shapes()))
    return model


def _case(tag):
    g = golden("fsodrcnn")
    class_ids = [int(c) for c in g[f"{tag}_class_ids"]]
    h, w, oh, ow, feat_seed, sup_seed = [int(v) for v in g[f"{tag}_size"]]
    return g, class_ids, (h, w), (oh, ow), fsodrcnn_support(class_ids, sup_seed)


def _max_err(got, ref):
    return float((got.detach().cpu().double() - ref.double()).abs().max())


def _assert_order_with_ties(what, got_rows, got_scores, ref_rows, ref_scores, row_tol):
    """got_rows / ref_rows [n, k], scores [n].  Same count; row i must match ref row i within row_tol, except where two
    entries changed places: then the recorded scores of the pair must differ by less than the score error measured on
    the matched entries (the order of the pair is decided below the accuracy of the scores)."""
    assert got_rows.shape == ref_rows.shape, f"{what}: {tuple(got_rows.shape)} vs {tuple(ref_rows.shape)}"
    n = ref_rows.shape[0]
    d = (got_rows[:, None, :].double() - ref_rows[None, :, :].double()).abs().amax(-1)       # [got, ref]
    perm = torch.where(d[torch.arange(n), torch.arange(n)] <= row_tol[torch.arange(n)], torch.arange(n), d.argmin(1))
    assert bool((d[torch.arange(n), perm] <= row_tol[perm]).all()), f"{what}: a row has no counterpart in the reference"
    assert perm.unique().numel() == n, f"{what}: two rows matched the same reference row"
    score_err = float((got_scores.double() - ref_scores[perm].double()).abs().max())
    for i in torch.nonzero(perm != torch.arange(n)).flatten().tolist():
        j = int(perm[i])
        gap = abs(float(ref_scores[i]) - float(ref_scores[j]))
        assert gap <= score_err, f"{what}: rows {i} and {j} swapped although their scores differ by {gap:.3e} > {score_err:.3e}"
    return perm


def _rpn_inputs(model, tag):
    """Synthetic res4 of the case and the correlation gate of each class, as the CUDA head forms them."""
    g, class_ids, (h, w), _, sup = _case(tag)
    model.set_prototypes(sup)
    res4 = synth.tensor((1, 1024, (h + 15) // 16, (w + 15) // 16), int(g[f"{tag}_size"][4]), 0.0, 2.0).to(DEV)
    res4 = ops.nhwc(res4)
    ep = model._episode
    gates = model.channel_attention.gates(model.agp(res4), ep["wq"], ep["k"])
    return g, class_ids, res4, list(gates)


@pytest.mark.parametrize("tag", TAGS)
def test_rpn_head_on_cuda_matches_reference(tag):
    """The gated 3x3 convolution (gate fused into the A operand, tcgen05) and the stacked 1x1 objectness / delta heads
    against the reference's recorded RPN outputs.  Measured on a B200: within 8.9e-6 absolute of values up to 3.6."""
    model = _model()
    g, class_ids, res4, gates = _rpn_inputs(model, tag)
    for ci, gate in enumerate(gates):
        corr = (res4 * gate.reshape(1, -1, 1, 1)).reshape(-1)[::53].cpu()
        ref = t(g[f"{tag}_corr{ci}"])
        assert bool(((corr - ref).abs() <= 1e-4 * ref.abs() + 1e-5).all()), "correlation gate"
        bound = (ops.absmax(res4, per_image=True) * gate.abs().amax(1)).reshape(1, 1)
        logits, deltas = model.proposal_generator.rpn_head([res4], [gate], [bound])
        for got, name, step in ((logits[0], "rpn_logits", 7), (deltas[0], "rpn_deltas", 29)):
            got = got.contiguous().reshape(-1)[::step].cpu()
            ref = t(g[f"{tag}_{name}{ci}"])
            err = (got - ref).abs()
            assert bool((err <= 1e-4 * ref.abs() + 1e-5).all()), f"{name}{ci}: max err {float(err.max()):.3e}"


@pytest.mark.parametrize("tag", TAGS)
def test_rpn_nms_indices_and_proposals_match_reference(tag, monkeypatch):
    """fod_batched_nms on the CUDA path's own decoded, clipped candidates is bit-exact against the oracle's coordinate
    trick NMS; the proposals after it match the reference's in count and order (ties per _assert_order_with_ties),
    boxes within 1e-4 relative + 1e-4 px, objectness logits within 1e-4 relative + 1e-5."""
    model = _model()
    g, class_ids, (h, w), (oh, ow), sup = _case(tag)
    model.set_prototypes(sup)
    res4 = synth.tensor((1, 1024, (h + 15) // 16, (w + 15) // 16), int(g[f"{tag}_size"][4]), 0.0, 2.0).to(DEV)
    calls = []
    real = ops.batched_nms

    def recording_nms(boxes, scores, idxs, thr):
        keep = real(boxes, scores, idxs, thr)
        calls.append((boxes.cpu(), scores.cpu(), idxs, thr, keep.cpu()))
        return keep

    monkeypatch.setattr(ops, "batched_nms", recording_nms)
    _, trace = model.head({"res4": res4}, [(h, w)], [(oh, ow)])
    monkeypatch.undo()
    assert len(calls) == len(class_ids)
    for ci, (boxes, scores, idxs, thr, keep) in enumerate(calls):
        assert idxs is None                                       # one level: one NMS group
        ref_keep = O.batched_nms_coordinate_trick(boxes, scores, torch.zeros(len(scores), dtype=torch.long), thr)
        assert torch.equal(keep, ref_keep), f"class {ci}: RPN NMS keeps differ"
        p = trace["proposals"][ci][0]
        gb, gl = p.proposal_boxes.tensor.cpu(), p.objectness_logits.cpu()
        rb, rl = t(g[f"{tag}_prop_boxes{ci}"]), t(g[f"{tag}_prop_logits{ci}"])
        assert gb.shape == rb.shape, f"class {ci}: {len(gb)} proposals, the reference has {len(rb)}"
        perm = _assert_order_with_ties(f"proposals {ci}", gb, gl, rb, rl, 1e-4 * rb.abs().amax(1) + 1e-4)
        err = (gl - rl[perm]).abs()
        assert bool((err <= 1e-4 * rl[perm].abs() + 1e-5).all()), f"objectness {ci}: max err {float(err.max()):.3e}"


@pytest.mark.parametrize("tag", TAGS)
def test_roi_align_res5_box_predictor_from_recorded_proposals(tag):
    """Teacher-forced ROI head: the reference's recorded proposals (classes concatenated in class order, the rows its res5
    ran on) -> fod_roi_align_wide 14x14 -> res5 (tensor-core bottlenecks) -> box predictor per class.
    Bars: pooled within 1e-5 of max|ref| (measured on a B200: 2.4e-7 of a maximum of 2.0), res5 within 1e-4 * max|ref|
    (measured 3.4e-5 of a maximum of 8.3), logits / deltas |err| <= 1e-4 |ref| + 1e-4 max|ref| on all 100 rows
    (measured at most 2.2e-5 of a maximum of 2.6 - 3.2)."""
    model = _model()
    g, class_ids, _, _, sup = _case(tag)
    model.set_prototypes(sup)
    res4, boxes = teacher_forced_inputs(g, tag, DEV)
    rh = model.roi_heads
    with torch.no_grad():
        pooled = rh.roi_pooling({"res4": ops.nhwc(res4)}, boxes, None, 1)[0]                  # [C*100, 1024, 14, 14]
        ref = t(g[f"{tag}_pooled"])
        assert _max_err(pooled.contiguous().reshape(-1)[::1009], ref) <= 1e-5 * float(ref.abs().max()), "pooled"
        feat = rh.res5(pooled.contiguous(memory_format=torch.channels_last))
        ref = t(g[f"{tag}_boxfeat"])
        assert _max_err(feat.contiguous().reshape(-1)[::211], ref) <= 1e-4 * float(ref.abs().max()), "res5"
        for ci in range(len(class_ids)):
            logits, deltas = rh.box_predictor(feat[ci * 100:(ci + 1) * 100], None, model._episode["emb"][ci])
            for got, name in ((logits, "cls_logits"), (deltas, "deltas")):
                ref = t(g[f"{tag}_{name}{ci}"])
                err = (got.cpu().double() - ref.double()).abs()
                tol = 1e-4 * ref.double().abs() + 1e-4 * float(ref.abs().max())
                assert bool((err <= tol).all()), f"{name}{ci}: max err {float(err.max()):.3e}"


@pytest.mark.parametrize("tag", TAGS)
def test_final_detect_bit_exact_and_detections_match_reference(tag):
    """Scores and decoded boxes formed on the device from the GPU's own logits / deltas of the recorded proposals; the
    class-wise NMS + top-k + rescale (fod_final_detect) is bit-exact against the oracle's final_detect + postprocess on
    the same tensors, and its detections match the reference's: same count, classes exact, boxes within 1e-4 relative
    + 1e-4 px, scores within 1e-4, order per _assert_order_with_ties."""
    model = _model()
    g, class_ids, (h, w), (oh, ow), sup = _case(tag)
    model.set_prototypes(sup)
    res4, boxes = teacher_forced_inputs(g, tag, DEV)
    rh, bp = model.roi_heads, model.roi_heads.box_predictor
    C = len(class_ids)
    with torch.no_grad():
        pooled = rh.roi_pooling({"res4": ops.nhwc(res4)}, boxes, None, 1)[0]
        feat = rh.res5(pooled.contiguous(memory_format=torch.channels_last))
        props = boxes.reshape(C, 100, 4)
        det_boxes, det_scores = [], []
        for ci in range(C):
            logits, deltas = bp(feat[ci * 100:(ci + 1) * 100], None, model._episode["emb"][ci])
            det_boxes.append(apply_deltas(deltas.float(), props[ci], bp.box_weights))
            det_scores.append(F.softmax(logits, dim=-1)[:, 0])
        det_boxes, det_scores = torch.stack(det_boxes).contiguous(), torch.stack(det_scores).contiguous()
    counts = torch.full((C,), 100, dtype=torch.int32, device=DEV)
    hw = torch.tensor([[h, w]], dtype=torch.int32, device=DEV)
    ohw = torch.tensor([[oh, ow]], dtype=torch.int32, device=DEV)
    status = ops.new_status(DEV)
    ob, os_, ocls, _, oc = ops.final_detect(det_boxes, det_scores, counts, C, bp.test_score_thresh, bp.test_nms_thresh,
                                            bp.test_topk_per_image, hw, ohw, status)
    ops.check_status(status)
    m = int(oc[0])
    cfg = O.HeadConfig(score_thresh_test=bp.test_score_thresh, nms_thresh_test=bp.test_nms_thresh,
                       detections_per_image=bp.test_topk_per_image)
    cls_idx = torch.arange(C).repeat_interleave(100)
    fb, fs, fc, _ = O.final_detect(det_boxes.cpu().reshape(-1, 4), det_scores.cpu().reshape(-1), cls_idx, (h, w), cfg)
    pb, ps, pc = O.postprocess(fb, fs, fc, (h, w), oh, ow)
    assert m == pb.shape[0]
    assert np.array_equal(ob[0, :m].cpu().numpy(), pb.numpy())
    assert np.array_equal(os_[0, :m].cpu().numpy(), ps.numpy())
    assert np.array_equal(ocls[0, :m].cpu().numpy(), pc.numpy())
    rb, rs, rc = t(g[f"{tag}_out_boxes"]), t(g[f"{tag}_out_scores"]), t(g[f"{tag}_out_classes"])
    ids = torch.tensor(class_ids)
    gb, gs, gc = ob[0, :m].cpu(), os_[0, :m].cpu(), ids[ocls[0, :m].cpu()]
    assert m == rb.shape[0], f"{m} detections, the reference has {rb.shape[0]}"
    # a row = (class, box): a detection can only stand for a reference detection of the same class
    got_rows = torch.cat((gc[:, None].double() * 1e6, gb.double()), 1)
    ref_rows = torch.cat((rc[:, None].double() * 1e6, rb.double()), 1)
    perm = _assert_order_with_ties("detections", got_rows, gs, ref_rows, rs, 1e-4 * rb.abs().amax(1) + 1e-4)
    assert float((gs - rs[perm]).abs().max()) <= 1e-4


# ------------------------------------------------------------------------------------------- padding rows, batch mates
def _poisoned(monkeypatch, fill, fn):
    g = GuardedTorch(fill)
    monkeypatch.setattr(ops, "torch", g)
    try:
        out = fn()
        g.check()
    finally:
        monkeypatch.undo()
    return out


def test_padding_rows_do_not_change_valid_rows(monkeypatch):
    """eval_with_support over B=2 x C=2 problems with counts [100, 37, 0, 1]: the boxes of the padding rows are
    arbitrary and every buffer the operator wrappers leave uninitialised (the pooled ROI rows beyond each count among
    them) is filled with 0x70 (2.98e29 as fp32), 0x7F (3.39e38) or 0xFF (NaN).  Logits, deltas and detections of the
    valid rows must be bit-identical across fills, and logits / deltas within the bars of
    test_roi_align_res5_box_predictor_from_recorded_proposals of the float64 CPU run of the same modules."""
    model = _model()
    _, class_ids, _, _, sup = _case("b")
    model.set_prototypes(sup)
    B, C, cap = 2, 2, 100
    res4 = synth.tensor((B, 1024, 10, 13), 4242, 0.0, 2.0)
    wh = synth.tensor((B * C * cap, 2), 4244, 12.0, 150.0)
    ctr = synth.tensor((B * C * cap, 2), 4243, 0.0, 200.0)
    boxes = torch.cat((ctr - wh / 2, ctr + wh / 2), 1).reshape(B * C, cap, 4)
    counts = torch.tensor([100, 37, 0, 1], dtype=torch.int32)
    junk = synth.tensor((B * C, cap, 4), 4245, -5e4, 5e4)
    valid = torch.arange(cap)[None, :] < counts[:, None].long()
    boxes = torch.where(valid[..., None], boxes, junk)
    sizes, outs = [(160, 208)] * B, [(160, 208)] * B
    rh = model.roi_heads
    res4_d = ops.nhwc(res4.to(DEV))

    def run():
        (ob, os_, ocls, oc), raw = rh.eval_with_support(sizes, outs, {"res4": res4_d}, boxes.to(DEV), counts.to(DEV),
                                                        model._episode["emb"], class_ids)
        torch.cuda.synchronize()
        return ob, os_, ocls, oc, raw

    def valid_parts(o):
        ob, os_, ocls, oc, raw = o
        parts = [oc.cpu()]
        for b in range(B):
            m = int(oc[b])
            parts += [ob[b, :m].cpu(), os_[b, :m].cpu(), ocls[b, :m].cpu()]
        for p in range(B * C):
            n = int(counts[p])
            parts += [raw[p][0][:n].cpu(), raw[p][1][:n].cpu()]
        return parts

    results = [valid_parts(_poisoned(monkeypatch, fill, run)) for fill in (0x70, 0x7F, 0xFF)]
    for other, fill in zip(results[1:], ("0x7F", "0xFF")):
        for k, (a, b) in enumerate(zip(results[0], other)):
            assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), f"part {k} differs between fills 0x70 and {fill}"
    # the CPU float64 run of the same modules on the valid rows (the first 20 of each problem)
    cpu = build("cuda")
    cpu.load_state_dict(synth.state_dict(param_shapes()))
    cpu = cpu.double()
    with torch.no_grad():
        for p in range(B * C):
            n = min(int(counts[p]), 20)
            if n == 0:
                continue
            x = cpu.roi_heads.roi_pooling({"res4": res4.double()[p // C:p // C + 1]}, boxes[p:p + 1, :n].double(), None, 1)
            feat = cpu.roi_heads.res5(x[0])
            logits, deltas = cpu.roi_heads.box_predictor(feat, sup["res5_avg"][class_ids[p % C]].double())
            got_l, got_d = results[0][1 + 3 * B + 2 * p], results[0][2 + 3 * B + 2 * p]
            for got, ref, name in ((got_l[:n], logits, "logits"), (got_d[:n], deltas, "deltas")):
                err = (got.double() - ref).abs()
                tol = 1e-4 * ref.abs() + 1e-4 * float(ref.abs().max())
                assert bool((err <= tol).all()), f"problem {p} {name}: max err {float(err.max()):.3e}"


def test_small_query_with_fewer_proposals_than_the_cap_is_fill_independent(monkeypatch):
    """A query small enough that the RPN returns fewer than POST_NMS_TOPK proposals for some class (asserted: the
    padding rows exist), through model.head: detections bit-identical across fills of the uninitialised buffers."""
    model = _model()
    _, class_ids, _, _, sup = _case("b")
    model.set_prototypes(sup)
    res4 = synth.tensor((1, 1024, 3, 4), 4300, 0.0, 2.0).to(DEV)
    cap = model.proposal_generator.post_nms_topk

    def run():
        (ob, os_, ocls, oc), tr = model.head({"res4": res4}, [(48, 64)], [(48, 64)])
        m = int(oc[0])
        return [len(p[0]) for p in tr["proposals"]], [ob[0, :m].cpu(), os_[0, :m].cpu(), ocls[0, :m].cpu()]

    results = [_poisoned(monkeypatch, fill, run) for fill in (0x70, 0x7F, 0xFF)]
    assert min(results[0][0]) < cap, f"every class got {cap} proposals: no padding rows to test"
    for n_props, parts in results[1:]:
        assert n_props == results[0][0]
        for a, b in zip(results[0][1], parts):
            assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), "detections depend on the padding rows"


def test_head_batch_equals_separate_calls():
    """model.head over two res4 maps whose magnitudes differ by 1000x gives each image exactly what it gets alone."""
    model = _model()
    _, class_ids, _, _, sup = _case("b")
    model.set_prototypes(sup)
    maps = [synth.tensor((1, 1024, 10, 13), 4400, 0.0, 2.0), synth.tensor((1, 1024, 10, 13), 4401, 0.0, 2.0) * 1000.0]
    size = [(160, 208)]
    (ob, os_, ocls, oc), tr = model.head({"res4": torch.cat(maps).to(DEV)}, size * 2, size * 2)
    for b in range(2):
        (sb, ss, sc, sn), st = model.head({"res4": maps[b].to(DEV)}, size, size)
        for ci in range(len(class_ids)):
            assert torch.equal(tr["gate"][ci][b], st["gate"][ci][0]), f"image {b}: correlation gate of class {ci}"
            assert torch.equal(tr["proposals"][ci][b].proposal_boxes.tensor, st["proposals"][ci][0].proposal_boxes.tensor), \
                f"image {b}: proposals of class {ci}"
        m = int(sn[0])
        assert int(oc[b]) == m
        assert torch.equal(ob[b, :m], sb[0, :m]) and torch.equal(os_[b, :m], ss[0, :m]) and torch.equal(ocls[b, :m], sc[0, :m])

