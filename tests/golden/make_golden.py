"""Generate golden vectors by running the UNMODIFIED reference in the build container.

    python tests/golden/make_golden.py            # writes tests/golden/*.npz

Needs FOD_REFERENCE_DIR (a read-only checkout of the reference); the tests only
read the committed ``.npz`` files.  The reference modules are imported from
where they lie through ``refshim`` (stand-ins for the missing third-party
packages only; see its docstring).  Harness-level substitutions, none of which
touches the arithmetic of the hot path:

  * ``model.backbone`` is replaced by a stub returning ``synth.features`` (the
    backbone is outside the path; the head sees ordinary fp32 NCHW maps);
  * ``torch.Tensor.cuda`` is made the identity so ``init_model`` (fsod_cen.py:415)
    runs with MODEL.DEVICE=cpu;
  * weights are ``synth.state_dict`` values loaded into the real modules, inputs
    are ``synth.*`` tensors, so fixtures hold OUTPUTS and seeds only.
"""
from __future__ import annotations

import os
import pickle
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import refshim  # noqa: E402

refshim.install()

from faster_orefsdet_b200 import synth  # noqa: E402

torch.set_num_threads(4)
torch.Tensor.cuda = lambda self, *a, **k: self  # MODEL.DEVICE=cpu harness (see docstring)

from fewx.config import get_cfg  # noqa: E402
from detectron2.modeling import build_model  # noqa: E402
import fewx.modeling  # noqa: E402,F401
from detectron2.structures import Boxes, Instances  # noqa: E402
from detectron2.layers import batched_nms  # noqa: E402
from detectron2.modeling.poolers import ROIPooler  # noqa: E402
from detectron2.modeling.box_regression import Box2BoxTransform  # noqa: E402
from detectron2.modeling.roi_heads.fast_rcnn import fast_rcnn_inference_single_image  # noqa: E402
from detectron2.modeling.postprocessing import detector_postprocess  # noqa: E402
from fewx.modeling.fsod.fsod_fast_rcnn import fsod_fast_rcnn_inference_single_image  # noqa: E402
from fewx.modeling.fsod.fsod_cen import SM_Block  # noqa: E402

YAML = os.path.join(refshim.REFERENCE, "configs/fsod/finetune_vovnet.yaml")


class StubBackbone(torch.nn.Module):
    size_divisibility = 32

    def __init__(self):
        super().__init__()
        self.seed = 0

    def forward(self, x):
        return synth.features(x.shape[0], x.shape[2], x.shape[3], self.seed)


def build_reference(opts=()):
    cfg = get_cfg()
    cfg.merge_from_file(YAML)
    cfg.merge_from_list(["MODEL.DEVICE", "cpu"] + list(opts))
    model = build_model(cfg).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items() if not k.startswith("backbone.")}
    model.backbone = StubBackbone()
    model.load_state_dict(synth.state_dict(shapes), strict=True)
    return cfg, model, shapes


def np_(t):
    return t.detach().cpu().numpy()


def run_full(model, name, sizes, out_sizes, feat_seed, class_ids, shots, proto_seed, store_attn):
    """Real CenterNet2Detector.forward, one image per call (fsod_cen.py:438)."""
    rec = {"sizes": np.array(sizes), "out_sizes": np.array(out_sizes), "feat_seed": np.array(feat_seed),
           "class_ids": np.array(class_ids), "shots": np.array(shots), "proto_seed": np.array(proto_seed)}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)
        os.makedirs("support_dir")
        with open("support_dir/support_feature.pkl", "wb") as f:
            pickle.dump(synth.prototypes(class_ids, shots, proto_seed), f)
        try:
            for i, ((h, w), (oh, ow)) in enumerate(zip(sizes, out_sizes)):
                cap = {}
                head = model.proposal_generator.centernet_head
                h1 = head.register_forward_hook(lambda m, inp, out: cap.update(attn=inp[0], hm=out[2], reg=out[1]))
                h2 = model.proposal_generator.register_forward_hook(lambda m, inp, out: cap.update(props=out[0]))
                h3 = model.roi_heads.register_forward_hook(lambda m, inp, out: cap.update(dets=out[0]))
                bp = model.roi_heads.box_predictor[0]
                h4 = bp.register_forward_hook(lambda m, inp, out: cap.update(logits=out[0], deltas=out[1]))
                model.backbone.seed = feat_seed + i
                img = synth.ore_image(h, w, feat_seed + i)
                with torch.no_grad():
                    out = model([{"image": img, "height": oh, "width": ow}])[0]["instances"]
                for hh in (h1, h2, h3, h4):
                    hh.remove()
                for l in range(3):
                    a = cap["attn"][l][0]
                    rec[f"img{i}_attn{l}"] = np_(a) if store_attn else np_(a.reshape(-1)[::97])
                    rec[f"img{i}_hm{l}"] = np_(cap["hm"][l][0, 0])
                    rec[f"img{i}_reg{l}"] = np_(cap["reg"][l][0])
                p = cap["props"][0]
                rec[f"img{i}_proposal_boxes"] = np_(p.proposal_boxes.tensor)
                rec[f"img{i}_objectness"] = np_(p.objectness_logits)
                rec[f"img{i}_logits"] = np_(cap["logits"])
                rec[f"img{i}_deltas"] = np_(cap["deltas"])
                d = cap["dets"][0]
                rec[f"img{i}_det_boxes"] = np_(d.pred_boxes.tensor)
                rec[f"img{i}_det_scores"] = np_(d.scores)
                rec[f"img{i}_out_boxes"] = np_(out.pred_boxes.tensor)
                rec[f"img{i}_out_scores"] = np_(out.scores)
                rec[f"img{i}_out_classes"] = np_(out.pred_classes)
                print(name, i, (h, w), "proposals", len(p), "dets", len(d), "out", len(out),
                      "score range", float(out.scores.min()), float(out.scores.max()))
        finally:
            os.chdir(cwd)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **rec)


def run_ops(model, cfg):
    rec = {}
    # ---- batched_nms / ml_nms semantic (d2!/layers/nms.py:10-30), incl. engineered ties ----
    n = 700
    ctr = synth.tensor((n, 2), 11, 20.0, 300.0)
    wh = synth.tensor((n, 2), 12, 8.0, 90.0)
    boxes = torch.cat((ctr - wh / 2, ctr + wh / 2), 1)
    scores = synth.tensor((n,), 13, 0.0, 1.0)
    scores = torch.round(scores * 64) / 64          # many exact ties
    boxes[100:140] = boxes[60:100]                  # duplicates: IoU exactly 1
    idxs = (synth.tensor((n,), 14, 0.0, 1.0) * 3).long()
    for thr in (0.6, 0.9):
        rec[f"nms1_keep_{thr}"] = np_(batched_nms(boxes, scores, torch.zeros(n, dtype=torch.long), thr))
        rec[f"nms3_keep_{thr}"] = np_(batched_nms(boxes, scores, idxs, thr))
    # IoU exactly at the threshold: boxes [0,0,10,10] and [0,0,10,6] -> 0.6 in fp32 arithmetic
    eb = torch.tensor([[0, 0, 10, 10], [0, 0, 10, 6], [0, 0, 5, 9], [0, 0, 9, 10.0]])
    es = torch.tensor([0.9, 0.8, 0.7, 0.6])
    for thr in (0.6, 0.9, 0.45):
        rec[f"nms_edge_keep_{thr}"] = np_(batched_nms(eb, es, torch.zeros(4, dtype=torch.long), thr))

    # ---- predict_single_level + nms_and_topK on the real CenterNet (fsod_rpn.py:1116-1210) ----
    pg = model.proposal_generator
    H, W, stride = 40, 48, 8
    hm = synth.tensor((1, 1, H, W), 21, -9.0, 3.0)
    hm = torch.round(hm * 8) / 8                    # ties in the heat-map, also at the k-th value
    hm[0, 0, :2] = -20.0                            # below INFERENCE_TH after sigmoid
    reg = synth.tensor((1, 4, H, W), 22, 0.0, 9.0)
    grids = pg.compute_grids([hm])
    res = pg.predict_single_level(grids[0], hm.sigmoid(), reg * stride, [(H * stride, W * stride)], None, 0)[0]
    rec["psl_scores_sorted"] = np.sort(np_(res.scores))[::-1].copy()
    rec["psl_count"] = np.array(len(res))
    # (set comparison: topk(sorted=False) order / choice among ties is implementation-defined)
    key = np_(res.pred_boxes.tensor)
    rec["psl_boxes_lexsorted"] = key[np.lexsort(key.T[::-1])]
    # tie-free version for an exact set + NMS comparison
    hm2 = synth.tensor((1, 1, H, W), 23, -9.0, 3.0)
    res2 = pg.predict_single_level(grids[0], hm2.sigmoid(), reg * stride, [(H * stride, W * stride)], None, 0)[0]
    k2 = np_(res2.pred_boxes.tensor)
    order = np.lexsort(k2.T[::-1])
    rec["psl2_boxes_lexsorted"] = k2[order]
    rec["psl2_scores_lexsorted"] = np_(res2.scores)[order]
    out2 = pg.nms_and_topK([res2])[0]
    rec["psl2_post_boxes"] = np_(out2.pred_boxes.tensor)
    rec["psl2_post_scores"] = np_(out2.scores)

    # ---- ROIPooler 8x8 and 4x4 (d2!/modeling/poolers.py:190-250) ----
    feats = synth.features(2, 256, 320, 31)
    fl = [feats["p3"], feats["p4"], feats["p5"]]
    nb = 96
    c = synth.tensor((2, nb, 2), 32, 0.0, 1.0) * torch.tensor([320.0, 256.0])
    sz = torch.exp(synth.tensor((2, nb, 2), 33, math_log(0.02), math_log(400.0)))
    bx = torch.cat((c - sz / 2, c + sz / 2), 2)
    bx[0, 0] = torch.tensor([10.0, 10.0, 10.01, 10.01])          # min-size box of fsod_rpn.py:1172
    bx[0, 1] = torch.tensor([-50.0, -30.0, 400.0, 300.0])        # beyond the map on every side
    bx[0, 2] = torch.tensor([0.0, 0.0, 112.0, 112.0])            # exactly on the level-3/level-4 edge (size 112)
    bx[0, 3] = torch.tensor([0.0, 0.0, 224.0, 224.0])
    bx[0, 4] = torch.tensor([0.0, 0.0, 448.0, 448.0])
    rec["pool_boxes"] = np_(bx)
    for res_, pooler in ((8, model.roi_heads.box_pooler), (4, model.roi_heads.box_pooler2)):
        rec[f"pool_out{res_}"] = np_(pooler(fl, [Boxes(bx[0]), Boxes(bx[1])])[:, ::8])  # every 8th channel

    # ---- relation head through the real roi_heads._run_stage (fsod_roi_heads.py:459-520) ----
    props = [Instances((256, 320), proposal_boxes=Boxes(bx[0])), Instances((256, 320), proposal_boxes=Boxes(bx[1]))]
    sup = [synth.tensor((5, 128, 8, 8), 41, -1.0, 1.0), synth.tensor((5, 128, 4, 4), 42, -1.0, 1.0)]
    with torch.no_grad():
        logits, deltas = model.roi_heads._run_stage(fl, sup, props, 0)
    rec["rel_logits"], rec["rel_deltas"] = np_(logits), np_(deltas)

    # ---- apply_deltas (d2!/modeling/box_regression.py:77-115) ----
    t = Box2BoxTransform(weights=(10.0, 10.0, 5.0, 5.0))
    dl = synth.tensor((nb, 4), 51, -6.0, 25.0)        # includes dw,dh above the clamp
    rec["deltas_in"] = np_(dl)
    rec["deltas_out"] = np_(t.apply_deltas(dl, bx[0]))

    # ---- fast_rcnn_inference_single_image (d2!/modeling/roi_heads/fast_rcnn.py:118-171) ----
    pb = t.apply_deltas(synth.tensor((nb, 4), 52, -1.0, 1.0), bx[0])
    pr = torch.softmax(synth.tensor((nb, 2), 53, -3.0, 3.0), 1)
    pb[7, 2] = float("nan")
    pr[9, 0] = float("inf")
    r, kept = fast_rcnn_inference_single_image(pb, pr, (256, 320), 0.0, 0.9, 100)
    rec["frcnn_in_boxes"], rec["frcnn_in_probs"] = np_(pb), np_(pr)
    rec["frcnn_boxes"], rec["frcnn_scores"], rec["frcnn_kept"] = np_(r.pred_boxes.tensor), np_(r.scores), np_(kept)
    r, kept = fast_rcnn_inference_single_image(pb, pr, (256, 320), 0.3, 0.5, 10)
    rec["frcnn2_boxes"], rec["frcnn2_scores"], rec["frcnn2_kept"] = np_(r.pred_boxes.tensor), np_(r.scores), np_(kept)

    # ---- N-way class-wise inference (fsod_fast_rcnn.py:84-145), 3 classes x 32 boxes ----
    C, R = 3, 32
    nb_boxes = t.apply_deltas(synth.tensor((C * R, 4), 61, -1.0, 1.0), bx[0][: C * R])
    nb_probs = torch.softmax(synth.tensor((C * R, 2), 62, -3.0, 3.0), 1)
    pred_cls = torch.arange(C).repeat_interleave(R).to(torch.int8) + 5
    r, kept = fsod_fast_rcnn_inference_single_image(pred_cls, nb_boxes, nb_probs, (256, 320), 0.0, 0.5, 100)
    rec["nway_in_boxes"], rec["nway_in_probs"], rec["nway_in_cls"] = np_(nb_boxes), np_(nb_probs), np_(pred_cls)
    rec["nway_boxes"], rec["nway_scores"] = np_(r.pred_boxes.tensor), np_(r.scores)
    rec["nway_classes"] = np_(r.pred_classes).astype(np.int64)

    # ---- detector_postprocess (d2!/modeling/postprocessing.py:9-75) ----
    inst = Instances((256, 320), pred_boxes=Boxes(clip(bx[1], 256, 320)), scores=synth.tensor((nb,), 71, 0.0, 1.0),
                     pred_classes=torch.zeros(nb, dtype=torch.long))
    pp = detector_postprocess(inst, 300, 500)
    rec["post_in_boxes"] = np_(clip(bx[1], 256, 320))
    rec["post_boxes"], rec["post_scores"] = np_(pp.pred_boxes.tensor), np_(pp.scores)

    # ---- SM_Block on the real module with synthetic weights (fsod_cen.py:584-630) ----
    x = synth.tensor((3, 16, 16, 128), 81, -1.0, 1.0)
    with torch.no_grad():
        rec["sm_p4"] = np_(model.vip_p4(x))
    # the pooled maps in a file of their own keep every fixture under 1 MB
    np.savez_compressed(os.path.join(HERE, "roi_pool.npz"), **{k: rec.pop(k) for k in ("pool_out8", "pool_out4")})
    np.savez_compressed(os.path.join(HERE, "ops.npz"), **rec)
    print("ops:", {k: v.shape for k, v in rec.items()})


def math_log(x):
    import math
    return math.log(x)


def clip(b, h, w):
    b = b.clone()
    b[:, 0::2] = b[:, 0::2].clamp(0, w)
    b[:, 1::2] = b[:, 1::2].clamp(0, h)
    return b


def run_prototype_build(model):
    """The reference's own cache-build branch of init_model (fsod_cen.py:321-408) on a
    synthetic 3-shot support set written to a temp ./datasets/coco."""
    import pandas as pd
    from PIL import Image
    rec = {}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)
        os.makedirs("datasets/coco/img")
        rows = []
        boxes = [[40.0, 30.0, 200.0, 180.0], [10.0, 60.0, 120.0, 250.0], [100.0, 100.0, 300.0, 240.0]]
        for s in range(3):
            img = synth.ore_image(256, 320, 500 + s).permute(1, 2, 0).numpy()
            Image.fromarray(img[:, :, ::-1].copy()).save(f"datasets/coco/img/s{s}.png")
            rows.append({"category_id": 1, "file_path": f"img/s{s}.png", "support_box": boxes[s]})
        pd.DataFrame(rows).to_pickle("datasets/coco/10_shot_support_df.pkl")
        model.backbone.seed = 900
        model.support_shot = 3
        try:
            with torch.no_grad():
                model.init_model()
        except SystemExit:
            pass
        with open("support_dir/support_feature.pkl", "rb") as f:
            d = pickle.load(f)
        os.chdir(cwd)
    rec["support_boxes"] = np.array(boxes, dtype=np.float32)
    for k in ("p3", "p4", "p5", "rcnn_8", "rcnn_4"):
        rec[k] = np_(d[k][1])
    np.savez_compressed(os.path.join(HERE, "prototypes.npz"), **rec)
    print("prototypes:", {k: v.shape for k, v in rec.items()})


def run_backbone():
    """The reference's own VoVNet-19-slim-eSE + FPN (d2 vovnet.py / fpn.py) on a small image."""
    cfg = get_cfg()
    cfg.merge_from_file(YAML)
    cfg.merge_from_list(["MODEL.DEVICE", "cpu"])
    model = build_model(cfg).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items() if k.startswith("backbone.")}
    model.load_state_dict(synth.state_dict(shapes), strict=False)
    with open(os.path.join(HERE, "backbone_param_shapes.txt"), "w") as f:
        for k, v in shapes.items():
            f.write(f"{k} {' '.join(map(str, v))}\n")
    x = synth.tensor((2, 3, 96, 160), 601, -120.0, 130.0)
    with torch.no_grad():
        out = model.backbone(x)
    np.savez_compressed(os.path.join(HERE, "backbone.npz"), **{k: np_(v) for k, v in out.items()})
    print("backbone:", {k: tuple(v.shape) for k, v in out.items()})


def main():
    run_backbone()
    cfg, model, shapes = build_reference()
    with open(os.path.join(HERE, "head_param_shapes.txt"), "w") as f:
        for k, v in shapes.items():
            f.write(f"{k} {' '.join(map(str, v))}\n")
    run_ops(model, cfg)
    run_prototype_build(model)
    # full forward, 1-way 5-shot: small maps, everything stored
    run_full(model, "full_small", [(256, 320), (224, 288)], [(300, 375), (224, 288)], 101, [1], 5, 7, True)
    # full forward at the headline size 640x640, 1-way 25-shot
    run_full(model, "full_640", [(640, 640)], [(640, 640)], 201, [3], 25, 8, False)


if __name__ == "__main__":
    main()
