"""Subprocess body of tests/test_dropin_cpu.py (needs FOD_REFERENCE_DIR, see tests/golden/refshim.py).

Plays `fsod_train_net.py --eval-only` / `demo.py` up to the model construction with the UNMODIFIED reference imported
the way those scripts import it, then installs this package over the reference's registry names and builds the model
through detectron2's own `build_model(cfg)` (d2!/modeling/meta_arch/build.py:16-25) from the reference's own config
object (`fewx.config.get_cfg()` + configs/fsod/finetune_vovnet.yaml).  Prints one JSON line.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
sys.path.insert(0, ROOT)

import refshim  # noqa: E402

refshim.install()
import torch  # noqa: E402

out = {}
# --- what fsod_train_net.py:18-30 / demo.py:14-17 import
from fewx.config import get_cfg  # noqa: E402   (pulls in fewx/__init__.py -> fewx.modeling registrations)
import fewx.modeling  # noqa: E402,F401
from detectron2.modeling import BACKBONE_REGISTRY, META_ARCH_REGISTRY, PROPOSAL_GENERATOR_REGISTRY, build_model  # noqa: E402
import fewx.modeling.fsod.fsod_roi_heads as ref_roi  # noqa: E402

ref_cls = {"meta": META_ARCH_REGISTRY.get("CenterNet2Detector"), "pg": PROPOSAL_GENERATOR_REGISTRY.get("CenterNet"),
           "roi": ref_roi.ROI_HEADS_REGISTRY.get("CustomCascadeROIHeads"),
           "bb": BACKBONE_REGISTRY.get("build_fcos_vovnet_fpn_backbone")}
out["reference_registered_first"] = all(c.__module__.startswith(("fewx.", "detectron2.")) for c in ref_cls.values())

# --- importing this package next to the reference must not raise and must not steal the names
import faster_orefsdet_b200  # noqa: E402
import faster_orefsdet_b200.modeling as ours  # noqa: E402
from faster_orefsdet_b200 import compat  # noqa: E402

out["bound_to_real_detectron2"] = bool(compat.HAVE_DETECTRON2) and compat.META_ARCH_REGISTRY is META_ARCH_REGISTRY
out["import_keeps_reference"] = META_ARCH_REGISTRY.get("CenterNet2Detector") is ref_cls["meta"]
rep = faster_orefsdet_b200.install(override=False)
out["install_without_override_keeps_reference"] = (META_ARCH_REGISTRY.get("CenterNet2Detector") is ref_cls["meta"]
                                                   and rep["META_ARCH"]["CenterNet2Detector"] == "kept foreign")

# --- explicit override, then the scripts' own construction path
rep = faster_orefsdet_b200.install(override=True)
out["report"] = rep
out["override_replaces"] = (META_ARCH_REGISTRY.get("CenterNet2Detector") is ours.CenterNet2Detector
                            and META_ARCH_REGISTRY.get("FsodRCNN") is ours.FsodRCNN
                            and PROPOSAL_GENERATOR_REGISTRY.get("CenterNet") is ours.CenterNet
                            and ref_roi.ROI_HEADS_REGISTRY.get("CustomCascadeROIHeads") is ours.CustomCascadeROIHeads)

cfg = get_cfg()                                                   # the REFERENCE's config object and defaults
cfg.merge_from_file(os.path.join(refshim.REFERENCE, "configs/fsod/finetune_vovnet.yaml"))
cfg.merge_from_list(["MODEL.DEVICE", "cuda"])
moved = []
_to = torch.nn.Module.to
torch.nn.Module.to = lambda self, *a, **k: (moved.append(a), self)[1]     # the test needs no GPU
try:
    model = build_model(cfg)                                      # fsod_train_net.py:95 -> Trainer.build_model -> this
finally:
    torch.nn.Module.to = _to
out["built_class"] = type(model).__module__ + "." + type(model).__name__
out["moved_to"] = [str(a[0]) for a in moved]
out["submodules"] = {"proposal_generator": type(model.proposal_generator).__module__,
                     "roi_heads": type(model.roi_heads).__module__, "backbone": type(model.backbone).__module__}

# --- the reference's own entry script, executed unchanged up to (not including) its __main__ block: its module-level
# imports must survive the override, and ITS Trainer.build_model(cfg) (fsod_train_net.py:95 for --eval-only) must build
# this package's detector
import runpy  # noqa: E402

try:
    ns = runpy.run_path(os.path.join(refshim.REFERENCE, "fsod_train_net.py"), run_name="fsod_train_net_not_main")
    torch.nn.Module.to = lambda self, *a, **k: self
    try:
        m2 = ns["Trainer"].build_model(cfg)
    finally:
        torch.nn.Module.to = _to
    out["trainer_build_model"] = type(m2).__module__ + "." + type(m2).__name__
except Exception as e:   # reported, asserted by the test
    out["trainer_build_model"] = f"{type(e).__name__}: {e}"

# --- the reference's own model from the same cfg (its classes, fetched before the override): checkpoints must fit both
cfg_cpu = cfg.clone()
cfg_cpu.merge_from_list(["MODEL.DEVICE", "cpu"])
PROPOSAL_GENERATOR_REGISTRY._obj_map["CenterNet"] = ref_cls["pg"]
ref_roi.ROI_HEADS_REGISTRY._obj_map["CustomCascadeROIHeads"] = ref_cls["roi"]
BACKBONE_REGISTRY._obj_map["build_fcos_vovnet_fpn_backbone"] = ref_cls["bb"]
ref_model = ref_cls["meta"](cfg_cpu)
faster_orefsdet_b200.install(override=True)
a = {k: tuple(v.shape) for k, v in ref_model.state_dict().items()}
b = {k: tuple(v.shape) for k, v in model.state_dict().items()}
out["state_dict_equal"] = a == b
out["n_params"] = len(a)
out["missing_in_ours"] = sorted(set(a) - set(b))[:5]
out["extra_in_ours"] = sorted(set(b) - set(a))[:5]
sd = ref_model.state_dict()
res = model.load_state_dict(sd, strict=True)                      # DetectionCheckpointer.resume_or_load ends here
out["strict_load_ok"] = not res.missing_keys and not res.unexpected_keys

# --- demo.py -> predictor.py:16-37 -> DefaultPredictor: build_model(cfg) + eval(); its call is model([{image,height,width}])
from detectron2.structures import Instances  # noqa: E402
from faster_orefsdet_b200.modeling.roi_heads import DetectionInstances  # noqa: E402

out["instances_is_detectron2s"] = issubclass(DetectionInstances, Instances) and compat.Instances is Instances
print(json.dumps(out))
