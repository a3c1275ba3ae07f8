"""ORACLE infrastructure (not product code): builds the REFERENCE's own two compiled extensions — DCN (v1 + v2) and
iou3d — from the sources where they lie under /root/reference, into oracle/_ref/ (git-ignored, travels to the GPU box).

They are the GPU-side oracle for SURVEY.md section 8 rows a12/a13/a16 (the reference has no CPU path for either op:
deform_conv.py:174-175, iou3d.cpp:7-9).  The reference's own build system (setup.py / make.sh) is not run; this is a
plain torch.utils.cpp_extension.load() on its three + two source files.  No reference source is copied into the repo.

    build()            in the build container (needs /root/reference)
    load(name)         on any box: imports the prebuilt oracle/_ref/<name>/<name>.so   (name: ref_deform_conv_ext | ref_iou3d_cuda)
"""
from __future__ import annotations

import importlib.machinery
import importlib.util
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
REF = os.environ.get("VISUALDET3D_REF", "/root/reference")
OPS = os.path.join(REF, "visualDet3D", "networks", "lib", "ops")

SOURCES = {
    "ref_deform_conv_ext": [os.path.join(OPS, "dcn", "src", f) for f in
                            ("deform_conv_ext.cpp", os.path.join("cuda", "deform_conv_cuda.cpp"), os.path.join("cuda", "deform_conv_cuda_kernel.cu"))],
    "ref_iou3d_cuda": [os.path.join(OPS, "iou3d", "src", f) for f in ("iou3d.cpp", "iou3d_kernel.cu")],
}


def _so_path(name: str) -> str:
    return os.path.join(OUT, name, name + ".so")


def build(verbose: bool = False) -> None:
    """No-op when the reference tree is absent (GPU box) or the outputs are already there."""
    if not os.path.isdir(OPS):
        return
    todo = [n for n in SOURCES if not os.path.exists(_so_path(n))]
    if not todo:
        return
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    os.environ.setdefault("CUDA_HOME", "/usr/local/cuda")
    from torch.utils import cpp_extension
    for name in todo:
        bdir = os.path.join(OUT, name)
        os.makedirs(bdir, exist_ok=True)
        cpp_extension.load(name=name, sources=SOURCES[name], build_directory=bdir, verbose=verbose,
                           extra_cflags=["-DWITH_CUDA", "-O2"],
                           extra_cuda_cflags=["-DWITH_CUDA", "-D__CUDA_NO_HALF_OPERATORS__", "-D__CUDA_NO_HALF_CONVERSIONS__",
                                              "-D__CUDA_NO_HALF2_OPERATORS__"],
                           is_python_module=False)


def load(name: str):
    """Import a prebuilt reference extension; raises FileNotFoundError if build() never ran for it."""
    if name in sys.modules:
        return sys.modules[name]
    p = _so_path(name)
    if not os.path.exists(p):
        raise FileNotFoundError(f"{p} missing: run oracle/build_ref.py in the build container (needs {REF})")
    import torch  # noqa: F401  (libtorch symbols must be loaded first)
    spec = importlib.util.spec_from_file_location(name, p, loader=importlib.machinery.ExtensionFileLoader(name, p))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.modules[name] = mod
    return mod


if __name__ == "__main__":
    build(verbose=True)
    for n in SOURCES:
        print(n, "->", _so_path(n), os.path.exists(_so_path(n)))
