"""-m gpu: the two op families the reference builds under make.sh (DCN v1/v2, iou3d) against (a) the outputs of the reference's OWN
compiled extensions on the same seeded inputs, recorded on a B200 (tests/golden/ref_ext.npz, tests/golden/make_golden_ref_ext.py;
large tensors as a seeded random sample of entries, stored with their flat indices) and (b) CPU restatements (oracle/torch_port.py,
torchvision's deform_conv2d and its autograd backward) over whole tensors."""
import os

import numpy as np
import pytest
import torch

import torch_port as tp
from conftest import GOLDEN

pytestmark = pytest.mark.gpu


_GOLD = {}


def ref_out(key):
    """What the reference's compiled extension returned for the inputs the test builds (`key` names the call)."""
    if not _GOLD:
        z = np.load(os.path.join(GOLDEN, "ref_ext.npz"))
        _GOLD.update({k: z[k] for k in z.files})
    return _GOLD[key]


def at(t, key):
    """The entries of `t` (flattened in its logical order) at the flat indices the stored reference values `key` were taken at."""
    return t.detach().reshape(-1).cpu().numpy()[ref_out(key + "_idx")]


def rand_boxes(n, g, spread=10.0):
    c = torch.rand(n, 2, generator=g) * spread
    wh = torch.rand(n, 2, generator=g) * 4 + 0.5
    ry = (torch.rand(n, generator=g) - 0.5) * 2 * np.pi
    return torch.cat([c - wh / 2, c + wh / 2, ry[:, None]], dim=1).contiguous()


def iou_pair_inputs():
    g = torch.Generator().manual_seed(0)
    return rand_boxes(70, g).cuda(), rand_boxes(45, g).cuda()


def test_iou3d_pairwise_vs_reference_extension_and_clipping():
    from visualdet3d_b200.ops import iou3d
    a, b = iou_pair_inputs()
    for mine, key in ((iou3d.boxes_overlap_bev_gpu, "iou_pair/overlap"), (iou3d.boxes_iou_bev_gpu, "iou_pair/iou")):
        o1 = torch.zeros(70, 45, device="cuda")
        assert mine(a, b, o1) == 1
        torch.cuda.synchronize()
        np.testing.assert_allclose(o1.cpu().numpy(), ref_out(key), rtol=1e-4, atol=1e-5)
    ov = torch.zeros(70, 45, device="cuda")
    iou3d.boxes_overlap_bev_gpu(a, b, ov)
    ac, bc, ovc = a.cpu().numpy(), b.cpu().numpy(), ov.cpu().numpy()
    for i in range(0, 70, 7):
        for j in range(0, 45, 5):
            assert abs(ovc[i, j] - tp.rotated_overlap_bev(ac[i], bc[j])) < 2e-3, (i, j)
    # identical boxes: overlap == area, IoU == 1
    io = torch.zeros(70, 70, device="cuda")
    iou3d.boxes_iou_bev_gpu(a, a, io)
    np.testing.assert_allclose(torch.diagonal(io).cpu().numpy(), 1.0, atol=1e-3)


NMS_SIZES = [1, 63, 64, 65, 300]


def nms_inputs(n):
    g = torch.Generator().manual_seed(n)
    return rand_boxes(n, g, spread=8.0).cuda()


@pytest.mark.parametrize("n", NMS_SIZES)
def test_iou3d_nms_vs_reference_extension(n):
    from visualdet3d_b200.ops import iou3d
    boxes = nms_inputs(n)
    for mine, key in ((iou3d.nms_gpu, f"nms{n}/rotated"), (iou3d.nms_normal_gpu, f"nms{n}/normal")):
        k1 = torch.zeros(n, dtype=torch.int64)
        n1 = mine(boxes, k1, 0.3)
        assert torch.equal(k1[:n1], torch.from_numpy(ref_out(key)))           # same count, bit-exact keep indices
    assert iou3d.nms_gpu(boxes[:0], torch.zeros(0, dtype=torch.int64), 0.3) == 0
    with pytest.raises(RuntimeError):
        iou3d.nms_gpu(boxes.cpu(), torch.zeros(n, dtype=torch.int64), 0.3)


def test_boxes_iou3d_wrapper():
    from visualdet3d_b200.ops import iou3d
    g = torch.Generator().manual_seed(2)
    b = torch.rand(9, 7, generator=g) * 3 + 1
    b[:, 6] = (torch.rand(9, generator=g) - 0.5) * 3
    b = b.cuda()
    iou = iou3d.boxes_iou3d_gpu(b, b)
    np.testing.assert_allclose(torch.diagonal(iou).cpu().numpy(), 1.0, atol=1e-3)
    assert float(iou.max()) <= 1.0 + 1e-3 and float(iou.min()) >= 0.0


DCN_CASES = [  # B, C, H, W, Cout, k, stride, pad, dil, dg
    (2, 64, 20, 30, 64, 3, 1, 1, 1, 1),
    (1, 32, 17, 23, 48, 3, 1, 1, 1, 1),
    (2, 64, 12, 16, 32, 3, 2, 1, 1, 1),
    (1, 64, 10, 14, 64, 3, 1, 2, 2, 2),
    (1, 16, 9, 11, 24, 1, 1, 0, 1, 1),
]


def dcn_forward_inputs(case):
    B, C, H, W, Co, k, s, p, d, dg = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(B, C, H, W, generator=g)
    w = torch.randn(Co, C, k, k, generator=g) / np.sqrt(C * k * k)
    bias = torch.randn(Co, generator=g)
    Ho, Wo = (H + 2 * p - (d * (k - 1) + 1)) // s + 1, (W + 2 * p - (d * (k - 1) + 1)) // s + 1
    off = torch.randn(B, 2 * k * k * dg, Ho, Wo, generator=g) * 2.0
    off[0, :, 0, 0] = 50.0                 # far outside -> contributes zero
    off[0, :, 1, 1] = -0.999               # the `> -1` knife edge
    mask = torch.sigmoid(torch.randn(B, k * k * dg, Ho, Wo, generator=g))
    return x, w, bias, off, mask


@pytest.mark.parametrize("case", DCN_CASES)
def test_modulated_deform_conv_vs_reference_extension(case):
    from visualdet3d_b200.ops import dcn
    B, C, H, W, Co, k, s, p, d, dg = case
    i = DCN_CASES.index(case)
    x, w, bias, off, mask = dcn_forward_inputs(case)
    Ho, Wo = off.shape[2:]
    xc, wc, bc, oc, mc = x.cuda(), w.cuda(), bias.cuda(), off.cuda(), mask.cuda()
    out = torch.empty(B, Co, Ho, Wo, device="cuda")
    dcn.modulated_deform_conv_forward(xc, wc, bc, xc.new_empty(0), oc, mc, out, xc.new_empty(0), k, k, s, s, p, p, d, d, 1, dg, True)
    torch.cuda.synchronize()
    np.testing.assert_allclose(at(out, f"dcn_fwd{i}/v2"), ref_out(f"dcn_fwd{i}/v2"), rtol=1e-4, atol=2e-5)
    cpu = tp.modulated_deform_conv(x, off, mask, w, bias, s, p, d)
    np.testing.assert_allclose(out.cpu().numpy(), cpu.numpy(), rtol=1e-4, atol=2e-5)
    # DCN v1 (no mask, no bias)
    o1 = torch.empty(B, Co, Ho, Wo, device="cuda")
    assert dcn.deform_conv_forward(xc, wc, oc, o1, xc.new_empty(0), xc.new_empty(0), k, k, s, s, p, p, d, d, 1, dg, B) == 1
    torch.cuda.synchronize()
    np.testing.assert_allclose(at(o1, f"dcn_fwd{i}/v1"), ref_out(f"dcn_fwd{i}/v1"), rtol=1e-4, atol=2e-5)
    cpu = tp.modulated_deform_conv(x, off, None, w, None, s, p, d)
    np.testing.assert_allclose(o1.cpu().numpy(), cpu.numpy(), rtol=1e-4, atol=2e-5)


V2_GRADS = ("grad_input", "grad_weight", "grad_bias", "grad_offset", "grad_mask")
V1_GRADS = ("v1_grad_input", "v1_grad_offset", "v1_grad_weight")


def dcn_backward_inputs(case):
    B, C, H, W, Co, k, s, p, d, dg = case
    g = torch.Generator().manual_seed(1000 + sum(case))
    x = torch.randn(B, C, H, W, generator=g)
    w = torch.randn(Co, C, k, k, generator=g) / np.sqrt(C * k * k)
    bias = torch.randn(Co, generator=g)
    Ho, Wo = (H + 2 * p - (d * (k - 1) + 1)) // s + 1, (W + 2 * p - (d * (k - 1) + 1)) // s + 1
    off = torch.randn(B, 2 * k * k * dg, Ho, Wo, generator=g) * 2.0
    off[0, :, 0, 0] = 50.0
    mask = torch.sigmoid(torch.randn(B, k * k * dg, Ho, Wo, generator=g))
    gout = torch.randn(B, Co, Ho, Wo, generator=g)
    return [t.cuda() for t in (x, w, bias, off, mask, gout)]


def dcn_backward(ext, case, xc, wc, bc, oc, mc, gc):
    """The three backward entries of `ext` on zero-initialised gradients: the DCNv2 and the DCNv1 gradients, in V2_GRADS + V1_GRADS order."""
    B, C, H, W, Co, k, s, p, d, dg = case
    e = lambda: xc.new_empty(0)
    gi, gw, gb = torch.zeros_like(xc), torch.zeros_like(wc), torch.zeros_like(bc)
    go, gm = torch.zeros_like(oc), torch.zeros_like(mc)
    ext.modulated_deform_conv_backward(xc, wc, bc, e(), oc, mc, e(), gi, gw, gb, go, gm, gc, k, k, s, s, p, p, d, d, 1, dg, True)
    g1i, g1o, g1w = torch.zeros_like(xc), torch.zeros_like(oc), torch.zeros_like(wc)
    assert ext.deform_conv_backward_input(xc, oc, gc, g1i, g1o, wc, e(), k, k, s, s, p, p, d, d, 1, dg, B) == 1
    assert ext.deform_conv_backward_parameters(xc, oc, gc, g1w, e(), e(), k, k, s, s, p, p, d, d, 1, dg, 0.5, B) == 1
    torch.cuda.synchronize()
    return [gi, gw, gb, go, gm, g1i, g1o, g1w]


def cpu_backward(case, xc, wc, bc, oc, mc, gc):
    """The same gradients, in the same order, from torchvision's deform_conv2d autograd on the host (v1 grad_weight scaled by 0.5)."""
    B, C, H, W, Co, k, s, p, d, dg = case
    out = []
    for modulated in (True, False):
        x, w, b, o, m = [t.detach().cpu().clone().requires_grad_(True) for t in (xc, wc, bc, oc, mc)]
        y = tp.modulated_deform_conv(x, o, m if modulated else None, w, b if modulated else None, s, p, d)
        y.backward(gc.cpu())
        out += [x.grad, w.grad, b.grad, o.grad, m.grad] if modulated else [x.grad, o.grad, 0.5 * w.grad]
    return out


@pytest.mark.parametrize("case", DCN_CASES)
def test_deform_conv_backward_vs_reference_extension(case):
    """SURVEY.md 8(f) rank 4: the three backward entries of `deform_conv_ext` against the reference's own compiled kernels
    (modulated col2im / col2im_coord, deform_conv_cuda_kernel.cu:635-767; DCNv1 :279-436) on the same tensors: grad_input, grad_offset,
    grad_mask, grad_weight, grad_bias (v1 grad_weight with scale 0.5).  Sums run in a different order (one fused pass, fp32 atomics):
    rtol 1e-4 of the tensor's scale."""
    from visualdet3d_b200.ops import dcn
    B, C, H, W, Co, k, s, p, d, dg = case
    i = DCN_CASES.index(case)
    xc, wc, bc, oc, mc, gc = dcn_backward_inputs(case)

    def close(a, what, factor=1.0):
        key = f"dcn_bwd{i}/{what}"
        want = factor * ref_out(key)
        scale = factor * float(ref_out(key + "_absmax")) + 1e-12
        err = float(np.abs(at(a, key) - want).max()) / scale
        assert err < 1e-4, (what, err)
        return err

    res = dcn_backward(dcn, case, xc, wc, bc, oc, mc, gc)
    errs = [close(a, n) for a, n in zip(res, V2_GRADS + V1_GRADS)]
    for a, b, n in zip(res, cpu_backward(case, xc, wc, bc, oc, mc, gc), V2_GRADS + V1_GRADS):      # every entry, against the host restatement
        err = float((a.cpu() - b).abs().max()) / (float(b.abs().max()) + 1e-12)
        assert err < 1e-4, (n, "vs host", err)
    # accumulate-into contracts: a second call doubles grad_input / grad_weight / grad_bias, re-assigns grad_offset / grad_mask
    gi, gw, gb, go, gm = [t.clone() for t in res[:5]]
    e = lambda: xc.new_empty(0)
    dcn.modulated_deform_conv_backward(xc, wc, bc, e(), oc, mc, e(), gi, gw, gb, go, gm, gc, k, k, s, s, p, p, d, d, 1, dg, True)
    close(gi, "grad_input", 2.0), close(gw, "grad_weight", 2.0), close(go, "grad_offset")
    print(case, "max relative errors", ["%.1e" % v for v in errs])


FUSED_CASES = [(2, 64, 24, 40, 64, 1, 1, 0.5), (1, 128, 20, 28, 64, 1, 1, 0.5), (2, 64, 17, 23, 256, 1, 1, 0.5), (1, 64, 21, 30, 128, 2, 1, 0.5),
               (1, 192, 9, 50, 96, 1, 2, 0.5), (2, 64, 33, 47, 64, 1, 1, 5.0), (1, 256, 13, 21, 128, 1, 1, 2.0)]


def fused_inputs(case):
    """x, w, bias, offset-conv weight / bias, and the generator the residual is drawn from next."""
    B, C, H, W, Co, s, d, off_scale = case
    g = torch.Generator().manual_seed(int(sum(case)))
    x = torch.randn(B, C, H, W, generator=g)
    w = torch.randn(Co, C, 3, 3, generator=g) / np.sqrt(C * 9)
    bias = torch.randn(Co, generator=g)
    ow = torch.randn(27, C, 3, 3, generator=g) * 0.03
    ob = torch.randn(27, generator=g) * off_scale
    return x, w, bias, ow, ob, g


def offsets_and_mask(x, ow, ob, s, d):
    """The offset conv of the module, computed by torch on the host: offsets and sigmoid mask on the device."""
    om = torch.nn.functional.conv2d(x, ow, ob, stride=s, padding=d, dilation=d)
    return om[:, :18].contiguous().cuda(), torch.sigmoid(om[:, 18:]).contiguous().cuda()


@pytest.mark.parametrize("case", FUSED_CASES)
def test_fused_deform_conv_matches_unfused_and_reference(case, monkeypatch):
    """csrc/dcn_fused.cu (bilinear gather written straight into the swizzled shared-memory operand of the tcgen05 GEMM) against
    (a) the unfused path (fp16 column planes in HBM + 1x1 conv): bit-identical, same K order and gather arithmetic;
    (b) the reference's own compiled extension on the same tensors: rtol 1e-4."""
    from visualdet3d_b200 import engine as E
    B, C, H, W, Co, s, d, off_scale = case          # off_scale: spread of the offsets in pixels (5.0: most samples leave the staged halo -> global fallback)
    x, w, bias, ow, ob, g = fused_inputs(case)
    layer = E.DeformConvLayer(w, bias, ow, ob, None, stride=s, pad=d, dil=d, relu=True, device="cuda")
    assert layer.k_order == (1 if (s == 1 and d == 1) else 0)
    Ho, Wo = layer.out_hw(H, W)
    planes = lambda *sh: torch.zeros(2, *sh, device="cuda", dtype=torch.float16)
    xa = E.split_lo(E.Act(x.permute(0, 2, 3, 1).contiguous().cuda(), 0, None, planes(B, H, W, C)))
    res = E.Act(torch.randn(B, Ho, Wo, Co, generator=g).cuda())
    outs = []
    variants = [("1", "1"), ("0", "1")] + ([("1", "0")] if C == 64 else [])       # (fused, staged): staged fused / unfused / global-gather fused
    for fused, staged_env in variants:
        monkeypatch.setenv("VD3D_DCN_FUSED", fused)
        monkeypatch.setenv("VD3D_DCN_STAGED", staged_env)
        assert layer.fused_ok() == (fused == "1")
        ar = E.Arena()
        out = E.Act(torch.full((B, Ho, Wo, Co + 8), 7.0, device="cuda"), 4, Co, planes(B, Ho, Wo, Co + 8))
        layer(xa, out, ar, "t", res=res)
        torch.cuda.synchronize()
        outs.append((out.t.clone(), out.lo.clone(), ar))
    for o in outs[1:]:
        assert torch.equal(outs[0][0], o[0]) and torch.equal(outs[0][1], o[1])                    # fp32 output and its fp16 planes, bit for bit
    assert "dcn.cols" not in {k[0] for k in outs[0][2]._bufs} and "dcn.cols" in {k[0] for k in outs[1][2]._bufs}      # no column tensor in the fused path
    assert float(outs[0][0][..., :4].min()) == 7.0 and float(outs[0][0][..., 4 + Co:].min()) == 7.0   # channel slice respected
    # the reference extension on offsets / mask from the same offset conv (offsets_and_mask), + the residual, ReLU
    key = f"fused{FUSED_CASES.index(case)}"
    resid = res.t.permute(0, 3, 1, 2)
    want = np.maximum(ref_out(key) + at(resid, key), 0)
    got = outs[0][0][..., 4:4 + Co].permute(0, 3, 1, 2)
    np.testing.assert_allclose(at(got, key), want, rtol=1e-4, atol=5e-5)
    # every entry, against the host restatement on the same offsets / mask
    off, mask = offsets_and_mask(x, ow, ob, s, d)
    want = torch.relu(tp.modulated_deform_conv(x, off.cpu(), mask.cpu(), w, bias, s, d, d) + resid.cpu())
    np.testing.assert_allclose(got.cpu().numpy(), want.numpy(), rtol=1e-4, atol=5e-5)


def test_dcn_error_behaviour_and_pack_module():
    from visualdet3d_b200.ops import dcn
    x = torch.randn(1, 32, 8, 8)
    w = torch.randn(16, 32, 3, 3)
    with pytest.raises(RuntimeError):
        dcn.modulated_deform_conv_forward(x, w, None, x, torch.zeros(1, 18, 8, 8), torch.ones(1, 9, 8, 8), torch.empty(1, 16, 8, 8), x,
                                          3, 3, 1, 1, 1, 1, 1, 1, 1, 1, False)
    with pytest.raises(RuntimeError):       # backward entries mirror the forward's checks (CPU tensors are refused, not computed on the host)
        dcn.modulated_deform_conv_backward(x, w, None, x, torch.zeros(1, 18, 8, 8), torch.ones(1, 9, 8, 8), x, torch.zeros_like(x), torch.zeros_like(w),
                                           None, torch.zeros(1, 18, 8, 8), torch.zeros(1, 9, 8, 8), torch.zeros(1, 16, 8, 8),
                                           3, 3, 1, 1, 1, 1, 1, 1, 1, 1, False)
    # module mirror vs the CPU restatement, conv_offset re-randomised (the reference zero-fills it)
    m = dcn.ModulatedDeformConvPack(64, 64, 3, padding=1)
    g = torch.Generator().manual_seed(0)
    m.conv_offset.weight.data = torch.randn(m.conv_offset.weight.shape, generator=g) * 0.05
    m.conv_offset.bias.data = torch.randn(27, generator=g) * 0.1
    sd = {"d." + k: v.detach().clone() for k, v in m.state_dict().items()}
    assert sorted(sd) == ["d.bias", "d.conv_offset.bias", "d.conv_offset.weight", "d.weight"]
    xin = torch.randn(2, 64, 14, 18, generator=g)
    ref = tp.modulated_deform_conv_pack(sd, "d", xin, 1, 1, 1)
    got = m.cuda()(xin.cuda()).cpu()
    np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=1e-4, atol=5e-5)
