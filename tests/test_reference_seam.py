"""The drop-in boundary (SURVEY.md 8(b)) against the reference's recorded contract (tests/golden/reference_seam.json, recorded from the
unmodified reference by tests/golden/make_golden_seam.py): `plugin.install_into_reference()` into a registry holding the reference's
names, construction through that registry from an EasyDict config for all five detectors, the reference module's state_dict layout and
parameter count, strict `load_state_dict`.  The worker runs in its own process: it puts a stand-in registry module into sys.modules."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_worker(name, timeout=900):
    env = dict(os.environ)
    env.pop("VD3D_CONV_ENGINE", None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "workers", name)], capture_output=True, text=True, timeout=timeout, env=env)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("SEAM_JSON ")]
    assert r.returncode == 0 and lines, f"worker {name} failed (rc {r.returncode}):\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    return json.loads(lines[-1][len("SEAM_JSON "):])


def test_install_into_reference_and_strict_state_dicts():
    out = run_worker("seam_cpu.py")
    assert out["installed"] == sorted(["Stereo3D", "Yolo3D", "GroundAwareYolo3D", "MonoFlex", "KM3D"])
    assert out["pipelines_kept"]
    assert set(out["reference_detectors_left"]) >= {"RetinaNet", "MonoDepth"}            # untouched: out of scope, still the reference's
    for name, rec in out["detectors"].items():
        assert rec["class_module"].startswith("visualdet3d_b200."), (name, rec)
        assert rec["is_nn_module"] and rec["keys_equal"] and rec["shapes_equal"], (name, rec)
        assert rec["missing"] == [] and rec["unexpected"] == [] and rec["values_loaded"], (name, rec)
        assert rec["n_params"] == rec["n_params_reference"] > 1_000_000, (name, rec)
        assert rec["cpu_forward"] != "ran", (name, rec)                                  # the B200 classes have no CPU path
    print({k: v["n_params"] for k, v in out["detectors"].items()})
