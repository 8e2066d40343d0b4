"""Pin the CPU oracle against golden vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py ran the real fewx / detectron2 code in the build
container).  Index outputs must be bit-exact, floating point within 1e-4 relative
(BASELINE.json north_star)."""
import numpy as np
import torch

from faster_orefsdet_b200 import synth
from oracle import head_oracle as O
from tests.util import assert_close, golden, head_state_dict, t

CFG = O.HeadConfig()


def _nms_inputs():
    n = 700
    ctr = synth.tensor((n, 2), 11, 20.0, 300.0)
    wh = synth.tensor((n, 2), 12, 8.0, 90.0)
    boxes = torch.cat((ctr - wh / 2, ctr + wh / 2), 1)
    scores = torch.round(synth.tensor((n,), 13, 0.0, 1.0) * 64) / 64
    boxes[100:140] = boxes[60:100]
    idxs = (synth.tensor((n,), 14, 0.0, 1.0) * 3).long()
    return boxes, scores, idxs


def test_batched_nms_matches_reference_bit_exact():
    g = golden("ops")
    boxes, scores, idxs = _nms_inputs()
    for thr in (0.6, 0.9):
        k1 = O.batched_nms_coordinate_trick(boxes, scores, torch.zeros_like(idxs), thr)
        k3 = O.batched_nms_coordinate_trick(boxes, scores, idxs, thr)
        assert np.array_equal(k1.numpy(), g[f"nms1_keep_{thr}"])
        assert np.array_equal(k3.numpy(), g[f"nms3_keep_{thr}"])
    eb = torch.tensor([[0, 0, 10, 10], [0, 0, 10, 6], [0, 0, 5, 9], [0, 0, 9, 10.0]])
    es = torch.tensor([0.9, 0.8, 0.7, 0.6])
    for thr in (0.6, 0.9, 0.45):
        k = O.batched_nms_coordinate_trick(eb, es, torch.zeros(4, dtype=torch.long), thr)
        assert np.array_equal(k.numpy(), g[f"nms_edge_keep_{thr}"])


def test_decode_level_matches_reference():
    g = golden("ops")
    H, W, stride = 40, 48, 8
    reg = synth.tensor((1, 4, H, W), 22, 0.0, 9.0)
    # tie-free heat-map: exact candidate set, exact boxes/scores
    hm2 = synth.tensor((1, 1, H, W), 23, -9.0, 3.0)
    loc, boxes, scores = O.decode_level(hm2[0, 0], reg[0], stride, CFG)
    assert loc.numel() == 1000 and torch.all(loc[1:] > loc[:-1])
    b = boxes.numpy()
    order = np.lexsort(b.T[::-1])
    assert np.array_equal(b[order], g["psl2_boxes_lexsorted"])
    assert np.array_equal(scores.numpy()[order], g["psl2_scores_lexsorted"])
    # NMS(0.6) + post-NMS top-256 on that level alone (fsod_rpn.py:1184-1210)
    keep = O.proposal_nms_topk(boxes, scores, CFG)
    assert np.array_equal(boxes[keep].numpy(), g["psl2_post_boxes"])
    assert np.array_equal(scores[keep].numpy(), g["psl2_post_scores"])
    # heat-map with ties (also at the k-th value): the multiset of selected scores is defined
    hm = torch.round(synth.tensor((1, 1, H, W), 21, -9.0, 3.0) * 8) / 8
    hm[0, 0, :2] = -20.0
    loc, boxes, scores = O.decode_level(hm[0, 0], reg[0], stride, CFG)
    assert int(g["psl_count"]) == loc.numel()
    assert np.array_equal(np.sort(scores.numpy())[::-1], g["psl_scores_sorted"])


def _pool_inputs(g):
    feats = synth.features(2, 256, 320, 31)
    return [feats["p3"], feats["p4"], feats["p5"]], t(g["pool_boxes"])


def test_roi_pool_matches_reference():
    g = golden("ops")
    fl, bx = _pool_inputs(g)
    for res in (8, 4):
        out = O.roi_pool(fl, [bx[0], bx[1]], res)
        assert_close(out[:, ::8], t(golden("roi_pool")[f"pool_out{res}"]), what=f"roi_pool{res}")


def test_relation_head_matches_reference():
    g = golden("ops")
    sd = head_state_dict()
    fl, bx = _pool_inputs(g)
    x = O.roi_pool(fl, [bx[0], bx[1]], 8)
    sup = synth.tensor((5, 128, 8, 8), 41, -1.0, 1.0)
    logits, deltas = O.relation_head(x, sup, sd)
    assert_close(logits, t(g["rel_logits"]), what="logits")
    assert_close(deltas, t(g["rel_deltas"]), what="deltas")


def test_apply_deltas_matches_reference():
    g = golden("ops")
    _, bx = _pool_inputs(g)
    out = O.apply_deltas(t(g["deltas_in"]), bx[0])
    assert_close(out, t(g["deltas_out"]), rtol=1e-6, atol=1e-4, what="apply_deltas")


def test_final_detect_matches_reference():
    g = golden("ops")
    pb, pr = t(g["frcnn_in_boxes"]), t(g["frcnn_in_probs"])
    for tag, sthr, nthr, topk in (("frcnn", 0.0, 0.9, 100), ("frcnn2", 0.3, 0.5, 10)):
        cfg = O.HeadConfig(score_thresh_test=sthr, nms_thresh_test=nthr, detections_per_image=topk)
        b, s, c, rows = O.final_detect(pb, pr[:, 0], torch.zeros(pb.shape[0], dtype=torch.long), (256, 320), cfg)
        assert np.array_equal(rows.numpy(), _rows_after_valid(pb, pr, g[f"{tag}_kept"]))
        assert np.array_equal(b.numpy(), g[f"{tag}_boxes"])
        assert np.array_equal(s.numpy(), g[f"{tag}_scores"])


def _rows_after_valid(pb, pr, kept):
    # the reference reports kept indices relative to the rows that survived the
    # isfinite filter (d2 fast_rcnn.py:137-140); the oracle reports original rows.
    valid = torch.isfinite(pb).all(1) & torch.isfinite(pr).all(1)
    return torch.nonzero(valid).squeeze(1).numpy()[kept]


def test_nway_classwise_nms_matches_reference():
    g = golden("ops")
    C, R = 3, 32
    boxes, probs = t(g["nway_in_boxes"]), t(g["nway_in_probs"])
    cls_idx = torch.arange(C).repeat_interleave(R)
    cfg = O.HeadConfig(nms_thresh_test=0.5)
    b, s, c, _ = O.final_detect(boxes, probs[:, 0], cls_idx, (256, 320), cfg)
    assert np.array_equal(b.numpy(), g["nway_boxes"])
    assert np.array_equal(s.numpy(), g["nway_scores"])
    assert np.array_equal((c + 5).numpy(), g["nway_classes"])


def test_postprocess_matches_reference():
    g = golden("ops")
    nb = g["post_in_boxes"].shape[0]
    b, s, _ = O.postprocess(t(g["post_in_boxes"]), synth.tensor((nb,), 71, 0.0, 1.0),
                            torch.zeros(nb, dtype=torch.long), (256, 320), 300, 500)
    assert np.array_equal(b.numpy(), g["post_boxes"])
    assert np.array_equal(s.numpy(), g["post_scores"])


def test_sm_block_matches_reference():
    g = golden("ops")
    sd = head_state_dict()
    x = synth.tensor((3, 16, 16, 128), 81, -1.0, 1.0)
    assert_close(O.sm_block(x, sd, "vip_p4.", 16), t(g["sm_p4"]), what="sm_block")


def test_prototype_build_matches_reference():
    g = golden("prototypes")
    sd = head_state_dict()
    feats = synth.features(3, 256, 320, 900)
    boxes = [t(g["support_boxes"][i:i + 1]) for i in range(3)]
    out = O.build_prototypes(feats, boxes, sd, CFG)
    for k in ("p3", "p4", "p5", "rcnn_8", "rcnn_4"):
        assert_close(out[k], t(g[k]), what=k)


def _run_full(name):
    g = golden(name)
    sd = head_state_dict()
    protos = synth.prototypes(list(g["class_ids"]), int(g["shots"]), int(g["proto_seed"]))
    for i, ((h, w), (oh, ow)) in enumerate(zip(g["sizes"], g["out_sizes"])):
        feats = synth.features(1, int(h), int(w), int(g["feat_seed"]) + i)
        tr = {}
        b, s, c = O.detect_image(feats, protos, sd, (int(h), int(w)), CFG, (int(oh), int(ow)), tr)
        pc = tr["per_class"][0]
        for l in range(3):
            ga = g[f"img{i}_attn{l}"]
            a = pc["attn"][l][0]
            assert_close(a if ga.ndim == 3 else a.reshape(-1)[::97], t(ga), what=f"attn{l}")
            assert_close(pc["hm"][l][0, 0], t(g[f"img{i}_hm{l}"]), what=f"hm{l}")
            assert_close(pc["reg"][l][0], t(g[f"img{i}_reg{l}"]), what=f"reg{l}")
        assert_close(pc["proposals"], t(g[f"img{i}_proposal_boxes"]), atol=1e-3, what="proposals")
        assert_close(pc["objectness"], t(g[f"img{i}_objectness"]), what="objectness")
        assert_close(pc["logits"], t(g[f"img{i}_logits"]), what="logits")
        assert_close(pc["deltas"], t(g[f"img{i}_deltas"]), what="deltas")
        assert_close(b, t(g[f"img{i}_out_boxes"]), atol=1e-3, what="out boxes")
        assert_close(s, t(g[f"img{i}_out_scores"]), what="out scores")
        assert np.array_equal(c.numpy(), g[f"img{i}_out_classes"])


def test_full_forward_small_matches_reference():
    _run_full("full_small")


def test_full_forward_640_matches_reference():
    _run_full("full_640")


def test_c_restatement_of_nms_equals_torchvision_and_reference():
    from oracle import nms_c
    g = golden("ops")
    boxes, scores, idxs = _nms_inputs()
    for thr in (0.6, 0.9):
        assert np.array_equal(nms_c.batched_nms(boxes, scores, None, thr).numpy(), g[f"nms1_keep_{thr}"])
        assert np.array_equal(nms_c.batched_nms(boxes, scores, idxs, thr).numpy(), g[f"nms3_keep_{thr}"])
    for n, seed in ((0, 1), (1, 2), (3000, 3)):
        ctr = synth.tensor((n, 2), seed, 20.0, 600.0)
        wh = synth.tensor((n, 2), seed + 50, 8.0, 190.0)
        b = torch.cat((ctr - wh / 2, ctr + wh / 2), 1)
        s = torch.round(synth.tensor((n,), seed + 99, 0.0, 1.0) * 100) / 100
        ref = O.batched_nms_coordinate_trick(b, s, torch.zeros(n, dtype=torch.long), 0.6)
        assert np.array_equal(nms_c.batched_nms(b, s, None, 0.6).numpy(), ref.numpy())
