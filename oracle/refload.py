"""ORACLE infrastructure (not product code): import the UNMODIFIED reference package.

    load_reference()                      CPU (build container or GPU box): the reference runs on the host cores
    load_reference(device="cuda", ...)    GPU box: the reference runs on the GPU, its two compiled extensions replaced by the modules
                                          passed in (`visualdet3d_b200.ops.dcn` / `.ops.iou3d` = the drop-in test, or the reference's own
                                          extensions built by oracle/build_ref.py)

Where the package comes from: the reference checkout `oracle/build_ref.py` compiles the extensions from ($VISUALDET3D_REF or its
default).  No reference source is edited or copied: the recipe of SURVEY.md section 8(c) is environmental shims only (easydict / skimage / matplotlib stand-ins, the numba CUDA simulator,
and -- CPU mode only -- `Tensor.cuda` as the identity because the reference hard-codes `.cuda()` calls, PSM_cost_volume.py:51,83).

Used by: tests/golden/make_golden*.py (fixture generation), bench.py --impl reference (the CPU arm); `to_edict` by tests/workers/seam_cpu.py.
"""
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))


def ref_root() -> str:
    sys.path.insert(0, HERE)
    try:
        import build_ref
    finally:
        sys.path.remove(HERE)
    return build_ref.REF


def available() -> bool:
    return os.path.isdir(os.path.join(ref_root(), "visualDet3D"))


class EasyDict(dict):
    """Minimal stand-in for the uninstalled `easydict` package."""

    def __init__(self, d=None, **kw):
        super().__init__()
        d = dict(d or {})
        d.update(kw)
        for k, v in d.items():
            self[k] = v

    def __setitem__(self, k, v):
        if isinstance(v, dict) and not isinstance(v, EasyDict):
            v = EasyDict(v)
        super().__setitem__(k, v)

    __setattr__ = __setitem__

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)

    def copy(self):
        return EasyDict(dict.copy(self))


def to_edict(d):
    if isinstance(d, dict):
        return EasyDict({k: to_edict(v) for k, v in d.items()})
    return d


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


DCN_EXT = "visualDet3D.networks.lib.ops.dcn.deform_conv_ext"
IOU3D_EXT = "visualDet3D.networks.lib.ops.iou3d.iou3d_cuda"


def load_reference(device: str = "cpu", dcn_ext=None, iou3d_ext=None):
    """Returns the imported `visualDet3D` reference package.  One mode per process (the import is global)."""
    if "visualDet3D" in sys.modules and getattr(sys.modules["visualDet3D"], "_b200_ref", None):
        have = sys.modules["visualDet3D"]._b200_ref
        if have != device:
            raise RuntimeError(f"the reference is already imported in {have} mode in this process")
        if device == "cuda":                      # the extension modules may be swapped between tests
            _install_ext(dcn_ext, iou3d_ext)
        return sys.modules["visualDet3D"]
    import torch
    import torchvision

    os.environ.setdefault("NUMBA_ENABLE_CUDASIM", "1")     # evaluator/kitti/rotate_iou.py jit-compiles CUDA kernels at import
    sys.dont_write_bytecode = True
    if "easydict" not in sys.modules:
        try:
            __import__("easydict")
        except Exception:
            _stub("easydict", EasyDict=EasyDict)
    for n in ("skimage", "skimage.io", "skimage.measure", "matplotlib", "matplotlib.pyplot"):
        if n not in sys.modules:
            try:
                __import__(n)
            except Exception:
                _stub(n)
    if device == "cpu":
        # compiled extensions are import-time dependencies only: stub the two pybind modules
        notimpl = lambda *a, **k: (_ for _ in ()).throw(NotImplementedError("reference CUDA extension stub"))
        _stub(DCN_EXT, deform_conv_forward=notimpl, deform_conv_backward_input=notimpl,
              deform_conv_backward_parameters=notimpl, modulated_deform_conv_forward=notimpl, modulated_deform_conv_backward=notimpl)
        _stub(IOU3D_EXT, boxes_iou_bev_gpu=notimpl, boxes_overlap_bev_gpu=notimpl, nms_normal_gpu=notimpl, nms_gpu=notimpl)
        # hard-coded .cuda() / cuda.synchronize() in the reference -> no-ops: the model stays on the host
        torch.Tensor.cuda = lambda self, *a, **k: self
        torch.cuda.synchronize = lambda *a, **k: None
    else:
        if dcn_ext is None or iou3d_ext is None:
            raise ValueError("device='cuda' needs the two extension modules (ours or the reference's compiled ones)")
        _install_ext(dcn_ext, iou3d_ext)
    root = ref_root()
    if not os.path.isdir(os.path.join(root, "visualDet3D")):
        raise FileNotFoundError(f"no reference package under {root} (set VISUALDET3D_REF to a reference checkout)")
    sys.path.insert(0, root)
    import visualDet3D
    import visualDet3D.networks  # registers detectors
    if device == "cpu":
        # DCNv2 has no CPU path in the reference (deform_conv.py:174-175): torchvision stand-in, same mmcv lineage
        from visualDet3D.networks.lib.ops.dcn import deform_conv as _dc

        def _mdcn_cpu(x, off, m, w, b, s=1, p=0, d=1, g=1, dg=1):
            return torchvision.ops.deform_conv2d(x, off, w, b, stride=s, padding=p, dilation=d, mask=m)

        def _dcn_cpu(x, off, w, s=1, p=0, d=1, g=1, dg=1):
            return torchvision.ops.deform_conv2d(x, off, w, None, stride=s, padding=p, dilation=d)

        _dc.modulated_deform_conv = _mdcn_cpu
        _dc.deform_conv = _dcn_cpu
    visualDet3D._b200_ref = device
    return visualDet3D


def _install_ext(dcn_ext, iou3d_ext):
    """THE substitution: the reference's `from . import deform_conv_ext` / `from . import iou3d_cuda` resolve to these modules."""
    if dcn_ext is not None:
        sys.modules[DCN_EXT] = dcn_ext
        pkg = sys.modules.get("visualDet3D.networks.lib.ops.dcn")
        if pkg is not None:
            pkg.deform_conv_ext = dcn_ext
            dc = sys.modules.get("visualDet3D.networks.lib.ops.dcn.deform_conv")
            if dc is not None:
                dc.deform_conv_ext = dcn_ext
    if iou3d_ext is not None:
        sys.modules[IOU3D_EXT] = iou3d_ext
        pkg = sys.modules.get("visualDet3D.networks.lib.ops.iou3d")
        if pkg is not None:
            pkg.iou3d_cuda = iou3d_ext
            m = sys.modules.get("visualDet3D.networks.lib.ops.iou3d.iou3d")
            if m is not None:
                m.iou3d_cuda = iou3d_ext
