"""Golden vectors of the reference's FsodRCNN (R50-C4 Attention-RPN path, fewx/modeling/fsod/fsod_rcnn.py) by running
the UNMODIFIED reference in the build container (CPU):

    python tests/golden/make_golden_fsodrcnn.py        # writes tests/golden/fsodrcnn.npz, fsodrcnn_param_shapes.txt

Same rules as make_golden.py (refshim stand-ins for missing third-party packages only; synthetic hash weights; fixtures
hold OUTPUTS and seeds).  Harness-level substitutions:
  * ``model.backbone`` is a stub returning ``synth.tensor`` res4 maps for the head fixtures (the real ResNet is recorded
    separately on a small image: ``backbone_*``);
  * ``torch.Tensor.cuda`` is the identity (fsod_rcnn.py:457 moves the pickle to the GPU);
  * ``fsod_rcnn.Have_a_Look`` (a debugging visualiser that opens a hard-coded image path of the authors' machine,
    fsod_rcnn.py:491 -> demo_visualizer.py:108) is a no-op.
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

torch.set_num_threads(8)
torch.Tensor.cuda = lambda self, *a, **k: self

from fewx.config import get_cfg  # noqa: E402
from detectron2.modeling import build_model  # noqa: E402
import fewx.modeling  # noqa: E402,F401
import fewx.modeling.fsod.fsod_rcnn as ref_rcnn  # noqa: E402

ref_rcnn.Have_a_Look = lambda *a, **k: None
YAML = os.path.join(refshim.REFERENCE, "configs/fsod/Base-FSOD-C4.yaml")


def fsodrcnn_support(class_ids, seed):
    """pkl of FsodRCNN.init_model (fsod_rcnn.py:344,420-428): {'res4_avg': {cls: [1,1024,14,14]}, 'res5_avg': {cls: [1,2048,7,7]}}"""
    d = {"res4_avg": {}, "res5_avg": {}}
    for j, c in enumerate(class_ids):
        d["res4_avg"][c] = synth.tensor((1, 1024, 14, 14), seed * 31 + 2 * j, 0.0, 1.2)
        d["res5_avg"][c] = synth.tensor((1, 2048, 7, 7), seed * 31 + 2 * j + 1, 0.0, 1.0)
    return d


class StubBackbone(torch.nn.Module):
    size_divisibility = 0

    def __init__(self):
        super().__init__()
        self.seed = 0

    def forward(self, x):
        return {"res4": synth.tensor((x.shape[0], 1024, (x.shape[2] + 15) // 16, (x.shape[3] + 15) // 16), self.seed, 0.0, 2.0)}


def np_(t):
    return t.detach().cpu().numpy()


def main():
    cfg = get_cfg()
    cfg.merge_from_file(YAML)
    cfg.merge_from_list(["MODEL.DEVICE", "cpu", "INPUT.FS.SUPPORT_WAY", 2, "INPUT.FS.SUPPORT_SHOT", 3])
    model = build_model(cfg).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    with open(os.path.join(HERE, "fsodrcnn_param_shapes.txt"), "w") as f:
        for k, s in shapes.items():
            f.write(k + " " + " ".join(str(x) for x in s) + "\n")
    model.load_state_dict(synth.state_dict(shapes), strict=True)
    rec = {}
    # the reference's own ResNet-50 C4 on a small image
    x = synth.tensor((2, 3, 96, 128), 811, -120.0, 130.0)
    with torch.no_grad():
        rec["backbone_res4"] = np_(model.backbone(x)["res4"])
    real_backbone = model.backbone
    model.backbone = StubBackbone()
    cases = [("a", [5], (192, 256), (192, 256), 41, 7), ("b", [3, 9], (160, 208), (300, 400), 43, 11)]
    rec["cases"] = np.array([c[0] for c in cases])
    cwd = os.getcwd()
    for tag, class_ids, (h, w), (oh, ow), feat_seed, sup_seed in cases:
        with tempfile.TemporaryDirectory() as td:
            os.chdir(td)
            os.makedirs("support_dir")
            with open("support_dir/support_feature.pkl", "wb") as f:
                pickle.dump(fsodrcnn_support(class_ids, sup_seed), f)
            cap = {"corr": [], "rpn_logits": [], "rpn_deltas": [], "props": [], "bp": []}
            def h_pg(m, inp, out):
                cap["corr"].append(inp[1]["res4"])
                cap["props"].append(out[0][0])

            def h_rpn(m, inp, out):
                cap["rpn_logits"].append(out[0][0])
                cap["rpn_deltas"].append(out[1][0])

            def h_res5(m, inp, out):
                cap.update(pooled=inp[0], boxfeat=out)

            def h_bp(m, inp, out):
                cap["bp"].append(out)

            hooks = [model.proposal_generator.register_forward_hook(h_pg),
                     model.proposal_generator.rpn_head.register_forward_hook(h_rpn),
                     model.roi_heads.res5.register_forward_hook(h_res5),
                     model.roi_heads.box_predictor.register_forward_hook(h_bp)]
            model.backbone.seed = feat_seed
            img = synth.ore_image(h, w, feat_seed)
            try:
                with torch.no_grad():
                    out = model([{"image": img, "height": oh, "width": ow}])[0]["instances"]
            finally:
                for hk in hooks:
                    hk.remove()
                os.chdir(cwd)
            rec[f"{tag}_class_ids"] = np.array(class_ids)
            rec[f"{tag}_size"] = np.array([h, w, oh, ow, feat_seed, sup_seed])
            for ci in range(len(class_ids)):
                rec[f"{tag}_corr{ci}"] = np_(cap["corr"][ci].reshape(-1)[::53])
                rec[f"{tag}_rpn_logits{ci}"] = np_(cap["rpn_logits"][ci].reshape(-1)[::7])
                rec[f"{tag}_rpn_deltas{ci}"] = np_(cap["rpn_deltas"][ci].reshape(-1)[::29])
                rec[f"{tag}_prop_boxes{ci}"] = np_(cap["props"][ci].proposal_boxes.tensor)
                rec[f"{tag}_prop_logits{ci}"] = np_(cap["props"][ci].objectness_logits)
                rec[f"{tag}_cls_logits{ci}"] = np_(cap["bp"][ci][0])
                rec[f"{tag}_deltas{ci}"] = np_(cap["bp"][ci][1])
            rec[f"{tag}_pooled"] = np_(cap["pooled"].reshape(-1)[::1009])
            rec[f"{tag}_boxfeat"] = np_(cap["boxfeat"].reshape(-1)[::211])
            rec[f"{tag}_out_boxes"] = np_(out.pred_boxes.tensor)
            rec[f"{tag}_out_scores"] = np_(out.scores)
            rec[f"{tag}_out_classes"] = np_(out.pred_classes).astype(np.int64)
            print(tag, class_ids, "proposals", [len(p) for p in cap["props"]], "detections", len(out))
    model.backbone = real_backbone
    np.savez_compressed(os.path.join(HERE, "fsodrcnn.npz"), **rec)
    print("wrote fsodrcnn.npz", sum(v.nbytes for v in rec.values()) // 1024, "KiB")


if __name__ == "__main__":
    main()
