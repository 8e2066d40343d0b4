"""FsodRCNN path (SURVEY 8f#3) end to end through model(batched_inputs) with the support pickle; the stage-by-stage
parity against the reference's recorded outputs is tests/test_fsodrcnn_parity_gpu.py."""
import pytest
import torch

from faster_orefsdet_b200 import synth


def fsodrcnn_support(class_ids, seed):
    """Same generator as tests/golden/make_golden_fsodrcnn.py::fsodrcnn_support."""
    d = {"res4_avg": {}, "res5_avg": {}}
    for j, c in enumerate(class_ids):
        d["res4_avg"][c] = synth.tensor((1, 1024, 14, 14), seed * 31 + 2 * j, 0.0, 1.2)
        d["res5_avg"][c] = synth.tensor((1, 2048, 7, 7), seed * 31 + 2 * j + 1, 0.0, 1.0)
    return d


@pytest.mark.gpu
def test_fsodrcnn_full_forward_batch_and_pkl(tmp_path, monkeypatch):
    """model(batched_inputs) through the real ResNet, support features from ./support_dir/support_feature.pkl; a batch of
    two images gives exactly what two single-image calls give; pred_classes carry the support class ids as int8."""
    import os
    import pickle
    from tests.test_fsodrcnn_cpu import build, param_shapes
    monkeypatch.chdir(tmp_path)
    os.makedirs("support_dir")
    with open("support_dir/support_feature.pkl", "wb") as f:
        pickle.dump(fsodrcnn_support([3, 9], 11), f)
    model = build().cuda()
    model.load_state_dict(synth.state_dict(param_shapes()))
    imgs = [synth.ore_image(160, 192, 1000), synth.ore_image(160, 192, 1001)]
    out = model([{"image": imgs[0], "height": 200, "width": 240}, {"image": imgs[1]}])
    assert out[0]["instances"].image_size == (200, 240) and out[1]["instances"].image_size == (160, 192)
    assert out[0]["instances"].pred_classes.dtype == torch.int8
    assert set(out[0]["instances"].pred_classes.tolist()) <= {3, 9}
    for i, inp in enumerate(({"image": imgs[0], "height": 200, "width": 240}, {"image": imgs[1]})):
        single = model([inp])[0]["instances"]
        both = out[i]["instances"]
        assert len(single) == len(both)
        assert torch.equal(single.pred_boxes.tensor, both.pred_boxes.tensor)
        assert torch.equal(single.scores, both.scores) and torch.equal(single.pred_classes, both.pred_classes)
