"""Golden contract of the drop-in boundary (tests/golden/reference_seam.json) from the UNMODIFIED reference (CPU, needs the reference tree):
the names its registries hold, and for each of the five detectors the parameter count and the ordered `key:shape` layout of the state_dict
its own module produces from the seam's configs (tests/workers/seam_cpu.py).

    VISUALDET3D_REF=<reference checkout> python tests/golden/make_golden_seam.py
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests", "workers"))

import torch  # noqa: E402
import refload  # noqa: E402
import seam_cpu  # noqa: E402


def main():
    refload.load_reference()
    from visualDet3D.networks.utils import registry as ref
    cfgs = seam_cpu.configs(tempfile.mkdtemp())
    out = {"detectors_registered": sorted(ref.DETECTOR_DICT.module_dict), "pipelines_registered": sorted(ref.PIPELINE_DICT.module_dict),
           "detectors": {}}
    for n in seam_cpu.NAMES:
        torch.manual_seed(0)
        m = ref.DETECTOR_DICT[n](refload.to_edict(cfgs[n]))
        sd = m.state_dict()
        out["detectors"][n] = {"n_params": int(sum(p.numel() for p in m.parameters())), "n_entries": len(sd),
                               "layout_sha256": seam_cpu.layout_digest(sd)}
    with open(os.path.join(HERE, "reference_seam.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["detectors"], indent=1))


if __name__ == "__main__":
    main()
