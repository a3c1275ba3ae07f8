"""Worker of tests/test_reference_seam.py (own process: it puts a stand-in `visualDet3D` registry module into sys.modules).  CPU only.

Executes the drop-in boundary against the reference's recorded contract (tests/golden/reference_seam.json, written by
tests/golden/make_golden_seam.py from the unmodified reference): `plugin.install_into_reference()` puts the B200 detector classes into
a registry holding the names the reference registers; `DETECTOR_DICT[cfg.detector.name](cfg.detector)` -- the exact expression of
scripts/eval.py:37 / train.py:87 -- then builds OUR class from an EasyDict config, and its state_dict must carry the reference module's
keys, in order, with its shapes and parameter count, and load a state_dict of that layout with strict key equality.  Prints one JSON line.

The stand-in registry is this project's own `plugin.Registry`, which restates the reference's registry contract (plugin.py docstring,
pinned by tests/test_abi.py::test_registry_contract): `install_into_reference()` is exercised against that restatement, not against the
reference's own `_register_module(force=...)` code, which cannot run without the reference package."""
import hashlib
import json
import os
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import torch  # noqa: E402
import refload  # noqa: E402

NAMES = ["Stereo3D", "Yolo3D", "GroundAwareYolo3D", "MonoFlex", "KM3D"]


def configs(tmp):
    """The detector configs of the seam: synthetic anchor priors written under `tmp`."""
    from visualdet3d_b200 import synth
    from visualdet3d_b200.detectors.centernet import km3d_cfg, monoflex_cfg
    cfgs = {}
    pm, ps = synth.synth_priors(16, 3, ["Car", "Pedestrian"])
    d = os.path.join(tmp, "s"); os.makedirs(d)
    synth.write_priors(d, pm, ps, ["Car", "Pedestrian"])
    cfgs["Stereo3D"] = synth.stereo3d_cfg(d, ["Car", "Pedestrian"])
    pm, ps = synth.synth_priors(16, 2, ["Car"])
    d = os.path.join(tmp, "m"); os.makedirs(d)
    synth.write_priors(d, pm, ps, ["Car"])
    cfgs["Yolo3D"] = synth.mono3d_cfg(d, "Yolo3D", ["Car"], None)
    cfgs["GroundAwareYolo3D"] = synth.mono3d_cfg(d, "GroundAwareYolo3D", ["Car"], None)
    cfgs["MonoFlex"], cfgs["KM3D"] = monoflex_cfg(), km3d_cfg()
    return cfgs


def layout_digest(state_dict):
    """sha256 of the ordered `key:shape` list of a state_dict: what a checkpoint's layout is."""
    txt = "\n".join(f"{k}:{tuple(v.shape)}" for k, v in state_dict.items())
    return hashlib.sha256(txt.encode()).hexdigest()


def stand_in_registry(golden):
    """A `visualDet3D.networks.utils.registry` holding placeholders under the names the reference registers."""
    from visualdet3d_b200.plugin import Registry
    reg = types.ModuleType("visualDet3D.networks.utils.registry")
    reg.DETECTOR_DICT, reg.PIPELINE_DICT = Registry("detectors"), Registry("pipelines")
    for n in golden["detectors_registered"]:
        reg.DETECTOR_DICT._register_module(type(n, (torch.nn.Module,), {}))
    for n in golden["pipelines_registered"]:
        f = lambda *a, **k: None
        f.__name__ = n
        reg.PIPELINE_DICT._register_module(f)
    for name in ("visualDet3D", "visualDet3D.networks", "visualDet3D.networks.utils"):
        sys.modules[name] = types.ModuleType(name)
    sys.modules["visualDet3D.networks.utils"].registry = reg
    sys.modules["visualDet3D.networks.utils.registry"] = reg
    return reg


def main():
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_seam.json")))
    from visualdet3d_b200 import plugin, synth
    import visualdet3d_b200.detectors as D  # noqa: F401  (registers the B200 detectors in plugin.DETECTOR_DICT)
    ref_pipelines = dict(stand_in_registry(golden).PIPELINE_DICT.module_dict)
    cfgs = configs(tempfile.mkdtemp())
    ref = plugin.install_into_reference()
    out = {"installed": sorted(k for k in ref.DETECTOR_DICT.module_dict if ref.DETECTOR_DICT[k].__module__.startswith("visualdet3d_b200")),
           "reference_detectors_left": sorted(k for k in ref.DETECTOR_DICT.module_dict if not ref.DETECTOR_DICT[k].__module__.startswith("visualdet3d_b200")),
           "pipelines_kept": sorted(ref_pipelines) == sorted(ref.PIPELINE_DICT.module_dict), "detectors": {}}
    for n in NAMES:
        want = golden["detectors"][n]
        cfg = refload.to_edict(cfgs[n])                     # an EasyDict, like cfg.detector of the reference's config files
        det = ref.DETECTOR_DICT[cfg.name](cfg)              # scripts/eval.py:37
        rec = {"class_module": type(det).__module__, "is_nn_module": isinstance(det, torch.nn.Module)}
        ours = det.state_dict()
        rec["keys_equal"] = len(ours) == want["n_entries"] and layout_digest(ours) == want["layout_sha256"]
        rec["shapes_equal"] = rec["keys_equal"]             # the digest covers names, order and shapes
        sd = synth.synth_state_dict({k: tuple(v.shape) for k, v in ours.items()}, 0)
        sd = {k: sd[k].to(v.dtype) if k in sd else v.clone() + 1 for k, v in ours.items()}
        res = det.load_state_dict(sd, strict=True)          # scripts/eval.py:42 uses strict=False; strict proves the key contract
        rec["missing"], rec["unexpected"] = list(res.missing_keys), list(res.unexpected_keys)
        rec["n_params"] = int(sum(p.numel() for p in det.parameters()))
        rec["n_params_reference"] = want["n_params"]
        rec["values_loaded"] = all(torch.equal(det.state_dict()[k], v) for k, v in sd.items())
        det.eval(); det.train(); str(det)                   # the calls scripts/train.py / eval.py make on the object
        try:
            det([torch.zeros(1, 3, 32, 32), torch.zeros(1, 3, 4)])
            rec["cpu_forward"] = "ran"
        except Exception as e:                              # no CPU fallback: must fail loudly
            rec["cpu_forward"] = type(e).__name__
        out["detectors"][n] = rec
    print("SEAM_JSON " + json.dumps(out))


if __name__ == "__main__":
    main()
