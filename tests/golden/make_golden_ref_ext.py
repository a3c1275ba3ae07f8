"""Golden outputs of the reference's own compiled DCN / iou3d extensions (tests/golden/ref_ext.npz) on the seeded inputs of
tests/test_dcn_iou3d_gpu.py.  Needs a B200 and the extensions oracle/build_ref.py compiles from the reference sources:

    python tests/golden/make_golden_ref_ext.py

A DCN output or gradient is stored as the values at a seeded random set of flat indices (`<key>_idx`, sorted; every index when the tensor
is small), with the full tensor's max |value| where the test scales its error by it.
"""
import os
import sys
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import build_ref  # noqa: E402
import test_dcn_iou3d_gpu as T  # noqa: E402


FWD_SAMPLES, BWD_SAMPLES = 1024, 512


def keep(out, key, t, cap):
    """Store the entries of `t` at `cap` flat indices drawn without replacement from a generator seeded by `key`."""
    f = t.detach().reshape(-1).cpu().numpy()
    idx = np.arange(f.size) if f.size <= cap else np.sort(np.random.default_rng(zlib.crc32(key.encode())).choice(f.size, cap, replace=False))
    out[key], out[key + "_idx"] = f[idx], idx.astype(np.int32)


def main():
    iou, dcn = build_ref.load("ref_iou3d_cuda"), build_ref.load("ref_deform_conv_ext")
    out = {}
    a, b = T.iou_pair_inputs()
    for key, fn in (("iou_pair/overlap", iou.boxes_overlap_bev_gpu), ("iou_pair/iou", iou.boxes_iou_bev_gpu)):
        o = torch.zeros(70, 45, device="cuda")
        assert fn(a, b, o) == 1
        out[key] = o.cpu().numpy()
    for n in T.NMS_SIZES:
        boxes = T.nms_inputs(n)
        for key, fn in ((f"nms{n}/rotated", iou.nms_gpu), (f"nms{n}/normal", iou.nms_normal_gpu)):
            k = torch.zeros(n, dtype=torch.int64)
            out[key] = k[:fn(boxes, k, 0.3)].numpy()
    for i, case in enumerate(T.DCN_CASES):
        B, C, H, W, Co, k, s, p, d, dg = case
        x, w, bias, off, mask = [t.cuda() for t in T.dcn_forward_inputs(case)]
        e = x.new_empty(0)
        o = torch.empty(B, Co, *off.shape[2:], device="cuda")
        dcn.modulated_deform_conv_forward(x, w, bias, e, off, mask, o, e, k, k, s, s, p, p, d, d, 1, dg, True)
        keep(out, f"dcn_fwd{i}/v2", o, FWD_SAMPLES)
        o = torch.empty(B, Co, *off.shape[2:], device="cuda")
        dcn.deform_conv_forward(x, w, off, o, e, e, k, k, s, s, p, p, d, d, 1, dg, B)
        keep(out, f"dcn_fwd{i}/v1", o, FWD_SAMPLES)
        grads = T.dcn_backward(dcn, case, *T.dcn_backward_inputs(case))
        for name, gr in zip(T.V2_GRADS + T.V1_GRADS, grads):
            keep(out, f"dcn_bwd{i}/{name}", gr, BWD_SAMPLES)
            out[f"dcn_bwd{i}/{name}_absmax"] = np.float32(gr.abs().max().item())
    for i, case in enumerate(T.FUSED_CASES):
        B, C, H, W, Co, s, d, _ = case
        x, w, bias, ow, ob, _ = T.fused_inputs(case)
        off, mask = T.offsets_and_mask(x, ow, ob, s, d)
        xc = x.cuda()
        o = torch.empty(B, Co, *off.shape[2:], device="cuda")
        dcn.modulated_deform_conv_forward(xc, w.cuda(), bias.cuda(), xc.new_empty(0), off, mask, o, xc.new_empty(0), 3, 3, s, s, d, d, d, d, 1, 1, True)
        keep(out, f"fused{i}", o, BWD_SAMPLES)
    torch.cuda.synchronize()
    np.savez_compressed(os.path.join(HERE, "ref_ext.npz"), **out)
    print("wrote", len(out), "arrays,", sum(v.nbytes for v in out.values()), "bytes")


if __name__ == "__main__":
    main()
