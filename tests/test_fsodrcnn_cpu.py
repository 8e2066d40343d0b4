"""FsodRCNN (R50-C4 Attention-RPN path, SURVEY 8f#3): host-side checks that need no GPU."""
import os

import pytest
import torch

from faster_orefsdet_b200 import synth
from faster_orefsdet_b200.config import get_cfg
from faster_orefsdet_b200.compat import META_ARCH_REGISTRY
from tests.util import GOLDEN, golden, t

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def param_shapes():
    shapes = {}
    with open(os.path.join(GOLDEN, "fsodrcnn_param_shapes.txt")) as f:
        for line in f:
            parts = line.split()
            shapes[parts[0]] = tuple(int(x) for x in parts[1:])
    return shapes


def build(device="cuda"):
    import faster_orefsdet_b200.modeling  # noqa: F401
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(ROOT, "configs/fsod/Base-FSOD-C4.yaml"))
    cfg.merge_from_list(["MODEL.DEVICE", device, "INPUT.FS.SUPPORT_WAY", 2, "INPUT.FS.SUPPORT_SHOT", 3])
    return META_ARCH_REGISTRY.get("FsodRCNN")(cfg).eval()


def test_state_dict_names_and_shapes_match_the_reference_fsodrcnn():
    """tests/golden/fsodrcnn_param_shapes.txt is the state_dict of the reference's own FsodRCNN built from
    configs/fsod/Base-FSOD-C4.yaml (make_golden_fsodrcnn.py): reference checkpoints must load with strict=True."""
    model = build()
    ours = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    ref = param_shapes()
    assert set(ours) == set(ref), (sorted(set(ref) - set(ours))[:5], sorted(set(ours) - set(ref))[:5])
    assert ours == ref
    res = model.load_state_dict(synth.state_dict(ref), strict=True)
    assert not res.missing_keys and not res.unexpected_keys


def test_cpu_device_is_refused():
    with pytest.raises(Exception, match="cpu"):
        build("cpu")


def test_resnet_c4_matches_the_reference_backbone_on_cpu():
    """The feature extractor module through ATen against the reference's own R50-C4 output (fsodrcnn.npz backbone_res4)."""
    model = build()
    model.load_state_dict(synth.state_dict(param_shapes()))
    x = synth.tensor((2, 3, 96, 128), 811, -120.0, 130.0)
    with torch.no_grad():
        y = model.backbone(x)["res4"]
    ref = t(golden("fsodrcnn")["backbone_res4"])
    assert y.shape == ref.shape
    assert float((y - ref).abs().max()) <= 2e-4 * float(ref.abs().max())


def test_rpn_and_output_layers_match_reference_on_cpu_tensors():
    """The ATen side of FsodRPN.rpn_head and FsodFastRCNNOutputLayers against the reference's recorded logits / deltas
    (the CUDA path of the same modules is compared in tests/test_fsodrcnn_gpu.py)."""
    g = golden("fsodrcnn")
    model = build()
    model.load_state_dict(synth.state_dict(param_shapes()))
    h, w, oh, ow, feat_seed, sup_seed = [int(v) for v in g["a_size"]]
    res4 = synth.tensor((1, 1024, (h + 15) // 16, (w + 15) // 16), feat_seed, 0.0, 2.0)
    from tests.test_fsodrcnn_gpu import fsodrcnn_support
    sup = fsodrcnn_support([int(c) for c in g["a_class_ids"]], sup_seed)
    r4 = sup["res4_avg"][5]
    with torch.no_grad():
        weight = model.channel_attention(model.agp(res4), r4)
        gate = weight.reshape(1, -1) + r4.mean((2, 3)).reshape(1, -1)
        corr = res4 * gate.reshape(1, -1, 1, 1)
        assert torch.allclose(corr.reshape(-1)[::53], t(g["a_corr0"]), rtol=1e-4, atol=1e-5)
        logits, deltas = model.proposal_generator.rpn_head([res4], [gate])
        assert torch.allclose(logits[0].reshape(-1)[::7], t(g["a_rpn_logits0"]), rtol=1e-4, atol=2e-5)
        assert torch.allclose(deltas[0].reshape(-1)[::29], t(g["a_rpn_deltas0"]), rtol=1e-4, atol=2e-5)


def teacher_forced_inputs(g, tag, device="cpu"):
    """res4 of case ``tag`` and the reference's recorded proposals of every class, concatenated in class order: the rows
    the reference's res5 ran on (fsod_roi_heads.py:165-172), [1, C * 100, 4]."""
    h, w, oh, ow, feat_seed, sup_seed = [int(v) for v in g[f"{tag}_size"]]
    C = len(g[f"{tag}_class_ids"])
    res4 = synth.tensor((1, 1024, (h + 15) // 16, (w + 15) // 16), feat_seed, 0.0, 2.0).to(device)
    boxes = torch.cat([t(g[f"{tag}_prop_boxes{ci}"]) for ci in range(C)]).reshape(1, -1, 4).to(device)
    return res4, boxes


@pytest.mark.parametrize("tag", ["a", "b"])
def test_roi_heads_from_recorded_proposals_match_reference_on_cpu(tag):
    """Teacher-forced: the reference's own proposals through the ATen side of roi_pooling (torchvision ROIAlign), res5 and
    box_predictor, each stage against what the reference recorded at that stage (fsodrcnn.npz {tag}_pooled every 1009th
    element of the NCHW [C*100, 1024, 14, 14] input of res5, {tag}_boxfeat every 211th of its output, all 100 rows of
    logits / deltas per class).  Pins the fixture layout the CUDA stage tests in test_fsodrcnn_parity_gpu.py rely on.
    Measured: pooled bit-exact, boxfeat within 2.1e-6 of a maximum of 8.3, logits / deltas within 3e-6."""
    from tests.test_fsodrcnn_gpu import fsodrcnn_support
    g = golden("fsodrcnn")
    model = build()
    model.load_state_dict(synth.state_dict(param_shapes()))
    class_ids = [int(c) for c in g[f"{tag}_class_ids"]]
    sup = fsodrcnn_support(class_ids, int(g[f"{tag}_size"][5]))
    res4, boxes = teacher_forced_inputs(g, tag)
    rh = model.roi_heads
    with torch.no_grad():
        pooled = rh.roi_pooling({"res4": res4}, boxes, None, 1).reshape(-1, 1024, 14, 14)
        ref = t(g[f"{tag}_pooled"])
        assert float((pooled.reshape(-1)[::1009] - ref).abs().max()) <= 1e-6 * float(ref.abs().max())
        feat = rh.res5(pooled)
        ref = t(g[f"{tag}_boxfeat"])
        assert float((feat.reshape(-1)[::211] - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
        for ci, c in enumerate(class_ids):
            logits, deltas = rh.box_predictor(feat[ci * 100:(ci + 1) * 100], sup["res5_avg"][c])
            for got, name in ((logits, "cls_logits"), (deltas, "deltas")):
                ref = t(g[f"{tag}_{name}{ci}"])
                assert float((got - ref).abs().max()) <= 1e-5 * float(ref.abs().max()), name
