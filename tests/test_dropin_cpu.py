"""Drop-in under the reference's own construction path (VERDICT r1 item 3): with the unmodified reference imported the
way fsod_train_net.py / demo.py import it, `faster_orefsdet_b200.install(override=True)` must make
`detectron2.modeling.build_model(cfg)` build this package's detector from the reference's own config object, with a
state_dict the reference's checkpoints fit.  Needs FOD_REFERENCE_DIR (a checkout of the reference project); runs in a
fresh interpreter so that the compat layer binds to the real (vendored) detectron2."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = os.environ.get("FOD_REFERENCE_DIR", "")


@pytest.mark.skipif(not REFERENCE or not os.path.exists(os.path.join(REFERENCE, "fsod_train_net.py")),
                    reason="needs FOD_REFERENCE_DIR: a checkout of the reference project")
def test_install_override_builds_this_detector_through_detectron2_build_model():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin", "check_dropin.py")], capture_output=True,
                       text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["reference_registered_first"] and out["bound_to_real_detectron2"]
    assert out["import_keeps_reference"] and out["install_without_override_keeps_reference"]
    assert out["override_replaces"], out["report"]
    assert out["built_class"] == "faster_orefsdet_b200.modeling.fsod_cen.CenterNet2Detector"
    assert out["moved_to"] == ["cuda"]                      # d2!/modeling/meta_arch/build.py:23 model.to(cfg.MODEL.DEVICE)
    assert all(m.startswith("faster_orefsdet_b200.") for m in out["submodules"].values()), out["submodules"]
    assert out["state_dict_equal"] and out["strict_load_ok"], (out["missing_in_ours"], out["extra_in_ours"])
    assert out["n_params"] > 150
    assert out["trainer_build_model"] == "faster_orefsdet_b200.modeling.fsod_cen.CenterNet2Detector"
    assert out["instances_is_detectron2s"]


def test_launcher_runs_a_script_as_main_with_its_own_arguments(tmp_path):
    """python -m faster_orefsdet_b200.run script.py args...: the script sees its own argv, runs as __main__, and the
    registries already hold this package's classes (no reference needed: only free names are taken)."""
    script = tmp_path / "probe.py"
    script.write_text(
        "import sys, json\n"
        "from faster_orefsdet_b200.compat import META_ARCH_REGISTRY\n"
        "print(json.dumps({'main': __name__, 'argv': sys.argv[1:], 'cls': META_ARCH_REGISTRY.get('CenterNet2Detector').__module__}))\n")
    r = subprocess.run([sys.executable, "-m", "faster_orefsdet_b200.run", str(script), "--eval-only", "MODEL.WEIGHTS", "x.pth"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out == {"main": "__main__", "argv": ["--eval-only", "MODEL.WEIGHTS", "x.pth"],
                   "cls": "faster_orefsdet_b200.modeling.fsod_cen"}
