"""GPU parity of the convolution front end (ResNet-C4 + RoIAlign + res5 head), through the C ABI.

Operator level: each op is compared with a plain fp32 torch restatement evaluated on the SAME bf16-rounded operands, so
the only differences are fp32 accumulation order and the final bf16 rounding of the output: |diff| <= 1e-2 of the output's
max for bf16 outputs (half an ulp of bf16 is 2^-9 = 2e-3 of the value; the bound leaves room for cancellation in sums of
~5k products), relative L2 <= 3e-3.  Pure data movement (layout changes, max-pool, im2col/col2im round trip) is bit-exact.

End to end (33 bottlenecks + head), two bounds (measured values are printed by the test and recorded in DESIGN.md):
  * against the reference fixture (fp32): outputs relative L2 <= 3e-2 (random walk of one bf16 rounding per stored
    activation).  Gradients: a ReLU whose pre-activation lies within rounding distance of 0 flips its mask and changes
    that element's gradient by 100%, so forward error eps becomes gradient error ~ sqrt(eps) (10-20% at the bottom of a
    100-layer bf16 network, for ANY bf16 implementation: oracle/frontend_oracle.py reproduces it in fp32 arithmetic with
    bf16-rounded storage).  Asserted: gradient norm within 5%, relative L2 <= 0.3.
  * rounding to bf16 also makes a deep network diverge from ANY other evaluation of itself: a difference delta << ulp in a
    layer's input flips a fraction ~delta/ulp of the output roundings, i.e. becomes sqrt(delta * ulp) >> delta one layer
    later (measured with tools/frontend_diag.py against the oracle's bf16-storage graph: 2e-5 after the stem, 1e-3 after
    7 blocks, 1e-2 after 33), so no oracle can pin the end-to-end gradients tighter than the bound above.  The backward
    kernels are therefore pinned per Bottleneck with identical inputs (test_bottleneck_against_bf16_storage_oracle: same
    masks, forward <= 2e-3, gradients <= 1.5e-2, measured ~6e-3) and per operator (test_conv_bn_act_forward_backward)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import frontend_oracle as fo
from synth import E2E_GRAD_SLICES, frontend_config, frontend_shapes, synth_frontend_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def maxrel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def bf(x):
    return x.to(torch.bfloat16).float()


def nhwc(x):  # NCHW f32 -> NHWC bf16
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def nchw(x):  # NHWC bf16 -> NCHW f32
    return x.float().permute(0, 3, 1, 2).contiguous()


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = old


CONV_CASES = [
    # (N, H, W, Cin, Cout, k, stride, pad, dil, relu_mode, resid)
    (2, 9, 11, 64, 128, 1, 1, 0, 1, 1, False),      # 1x1 (direct GEMM, no lowering)
    (2, 10, 12, 64, 256, 1, 2, 0, 1, 0, False),     # 1x1 stride 2 (stride_in_1x1 / downsample)
    (2, 9, 11, 64, 64, 3, 1, 1, 1, 1, False),       # 3x3
    (3, 14, 14, 128, 128, 3, 1, 2, 2, 1, False),    # 3x3 dilation 2 (res5 head)
    (2, 13, 10, 64, 64, 3, 2, 1, 1, 1, False),      # 3x3 stride 2 (stride_in_1x1 = False)
    (2, 37, 45, 3, 64, 7, 2, 3, 1, 1, False),       # stem 7x7/2, Cin = 3 (scalar im2col, K padded 147 -> 152)
    (2, 9, 11, 64, 256, 1, 1, 0, 1, 2, True),       # conv3 + residual + ReLU
    (1, 5, 7, 256, 64, 1, 1, 0, 1, 1, False),       # P = 35 rows (ragged tile)
    (4, 19, 23, 64, 64, 3, 1, 1, 1, 1, False),      # P = 1748 (ragged last tile), tensor > 128 KiB
    (2, 21, 17, 128, 64, 3, 1, 1, 1, 2, True),      # 3x3 + residual
    (5, 14, 14, 512, 512, 3, 1, 2, 2, 1, False),    # the res5 head's 3x3 at full width (K = 4608)
    (2, 30, 22, 256, 128, 1, 2, 0, 1, 1, False),    # layer2.0.conv1 geometry (stride_in_1x1)
]


@pytest.mark.parametrize("implicit", [True, False], ids=["tma_im2col", "explicit_im2col"])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_bn_act_forward_backward(case, implicit, monkeypatch):
    from vlbert_b200 import functional as VF
    monkeypatch.setattr(VF, "IMPLICIT_CONV", implicit)
    N, H, W, Cin, Cout, k, stride, pad, dil, relu_mode, has_res = case
    g = torch.Generator().manual_seed(hash(case) % 1000)
    x = bf(torch.randn(N, Cin, H, W, generator=g)).to(DEV)
    w = (torch.randn(Cout, Cin, k, k, generator=g) * (2.0 / (Cin * k * k)) ** 0.5).to(DEV)
    scale = (0.5 + torch.rand(Cout, generator=g)).to(DEV)
    shift = (0.2 * torch.randn(Cout, generator=g)).to(DEV)
    Ho = (H + 2 * pad - dil * (k - 1) - 1) // stride + 1
    Wo = (W + 2 * pad - dil * (k - 1) - 1) // stride + 1
    r = bf(torch.randn(N, Cout, Ho, Wo, generator=g)).to(DEV) if has_res else None
    gy = bf(torch.randn(N, Cout, Ho, Wo, generator=g)).to(DEV)

    # fp32 restatement on the bf16-rounded operands
    xr = x.clone().requires_grad_(True)
    wr = bf(w).clone().requires_grad_(True)
    rr = r.clone().requires_grad_(True) if has_res else None
    y_ref = F.conv2d(xr, wr, stride=stride, padding=pad, dilation=dil) * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1)
    if has_res:
        y_ref = y_ref + rr
    if relu_mode:
        y_ref = torch.relu(y_ref)
    y_ref.backward(gy)

    need_dx = Cin % 8 == 0          # the stem (Cin = 3) is frozen in every reference cfg: col2im needs C % 8 == 0
    xo = nhwc(x).requires_grad_(need_dx)
    wo = w.clone().requires_grad_(True)
    ro = nhwc(r).requires_grad_(True) if has_res else None
    y = VF.conv_bn_act(xo, wo, scale, shift, resid=ro, stride=stride, pad=pad, dil=dil, relu_mode=relu_mode)
    assert y.shape == (N, Ho, Wo, Cout) and y.dtype == torch.bfloat16
    y.backward(nhwc(gy))
    assert maxrel(nchw(y), y_ref) <= 1e-2 and rel(nchw(y), y_ref) <= 3e-3, (maxrel(nchw(y), y_ref), rel(nchw(y), y_ref))
    # the backward masks with the bf16 output's sign: identical to the fp32 mask except where |pre-activation| < 1 bf16 ulp
    if need_dx:
        assert rel(nchw(xo.grad), xr.grad) <= 6e-3, rel(nchw(xo.grad), xr.grad)
    assert rel(wo.grad, wr.grad) <= 6e-3, rel(wo.grad, wr.grad)
    if has_res:
        assert rel(nchw(ro.grad), rr.grad) <= 6e-3


def test_layout_changes_and_pools_are_exact():
    from vlbert_b200 import functional as VF
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 3, 21, 30, generator=g).to(DEV)
    xh = VF.nchw_to_nhwc_bf16(x)
    assert torch.equal(xh, nhwc(x))
    assert torch.equal(VF.nhwc_to_nchw_f32(xh), nchw(xh))
    f = bf(torch.randn(2, 64, 23, 31, generator=g)).to(DEV)
    mp = VF.maxpool3x3s2(nhwc(f))
    assert torch.equal(nchw(mp), F.max_pool2d(f, 3, 2, 1))
    # mean pool (AvgPool2d(14) + flatten, common/fast_rcnn.py:80-84): fp32 sum of 196 bf16 values
    h = bf(torch.randn(5, 2048, 14, 14, generator=g)).to(DEV).requires_grad_(True)
    ho = nhwc(h.detach()).requires_grad_(True)
    a = VF.AvgPoolFn.apply(ho)
    a_ref = F.avg_pool2d(h, 14).flatten(1)
    assert maxrel(a, a_ref) <= 1e-5
    ga = torch.randn(5, 2048, generator=g).to(DEV)
    a.backward(ga)
    a_ref.backward(ga)
    assert maxrel(nchw(ho.grad), bf(h.grad)) <= 1e-6


def test_im2col_col2im_adjoint():
    """<im2col(x), c> == <x, col2im(c)> (the property that makes dx = col2im(dcol) the true gradient); exact in fp64 on
    bf16-representable integers."""
    from vlbert_b200 import _lib, functional as VF
    g = torch.Generator().manual_seed(6)
    for (N, H, W, C, k, s, p, d) in ((2, 9, 8, 16, 3, 1, 1, 1), (1, 14, 14, 8, 3, 1, 2, 2), (2, 11, 9, 8, 3, 2, 1, 1), (1, 12, 10, 8, 1, 2, 0, 1)):
        Ho, Wo = VF._conv_out(H, k, s, p, d), VF._conv_out(W, k, s, p, d)
        Kp = k * k * C
        x = torch.randint(-4, 5, (N, H, W, C), generator=g).to(DEV).to(torch.bfloat16)
        c = torch.randint(-4, 5, (N * Ho * Wo, Kp), generator=g).to(DEV).to(torch.bfloat16)
        col = VF._im2col(x, k, k, s, p, d, Ho, Wo, Kp)
        dx = torch.empty_like(x)
        VF._chk(_lib.lib().vlb_col2im_nhwc(c.data_ptr(), None, dx.data_ptr(), N, H, W, C, k, k, s, p, d, Ho, Wo, Kp, VF._stream()))
        assert (col.double() * c.double()).sum().item() == (x.double() * dx.double()).sum().item()
        # and im2col agrees with torch's unfold (channel-major there, tap-major here)
        u = F.unfold(x.float().permute(0, 3, 1, 2), k, dilation=d, padding=p, stride=s)          # [N, C*k*k, L]
        u = u.view(N, C, k * k, Ho * Wo).permute(0, 3, 2, 1).reshape(N * Ho * Wo, Kp)
        assert torch.equal(col.float(), u)


def test_roi_align_nhwc_matches_the_oracle():
    """same sampling rules as the NCHW op (bit-exact there); here the feature map is bf16 and the output is rounded to bf16."""
    from vlbert_b200 import functional as VF
    import roi_align as ro
    g = torch.Generator().manual_seed(9)
    N, C, H, W = 2, 256, 38, 63
    f = bf(torch.randn(N, C, H, W, generator=g))
    K = 37
    b = torch.randint(0, N, (K,), generator=g).float()
    x1 = torch.rand(K, generator=g) * 800
    y1 = torch.rand(K, generator=g) * 450
    rois = torch.stack((b, x1, y1, x1 + 5 + torch.rand(K, generator=g) * 190, y1 + 5 + torch.rand(K, generator=g) * 140), 1)
    rois[0, 1:] = torch.tensor([-20.0, -20.0, 1100.0, 700.0])       # hangs over every edge
    ref = torch.from_numpy(ro.roi_align_forward(f.numpy(), rois.numpy(), 1 / 16.0, 14, 14, 1))
    fo_ = nhwc(f.to(DEV)).requires_grad_(True)
    out = VF.RoIAlignNHWCFn.apply(fo_, rois.to(DEV), 14, 14, 1 / 16.0, 1)
    assert maxrel(out.float().permute(0, 3, 1, 2), ref) <= 4e-3          # one bf16 rounding of the output
    gy = bf(torch.randn(K, C, 14, 14, generator=g))
    gref = torch.from_numpy(ro.roi_align_backward(gy.numpy(), rois.numpy(), 1 / 16.0, 14, 14, N, C, H, W, 1))
    out.backward(nhwc(gy.to(DEV)))
    assert rel(nchw(fo_.grad), gref) <= 3e-3


def _load_e2e(final_dim=64):
    import vlbert_b200
    m = vlbert_b200.FastRCNN(frontend_config(101), average_pool=True, final_dim=final_dim, enable_cnn_reg_loss=False)
    sd = fo.synth_frontend_state({k: v.shape for k, v in m.state_dict().items()}, 77)
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval(), sd


def test_state_dict_shapes_match_the_reference_layout():
    m, _ = _load_e2e()
    ours = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert ours == {k: tuple(v) for k, v in frontend_shapes().items()}


BLOCK_CASES = [
    # (inplanes, planes, stride, dilation, stride_in_1x1, N, H, W)
    (256, 128, 2, 1, True, 2, 18, 22),     # layer2.0 / layer3.0: stride 2 in conv1 + strided downsample
    (512, 128, 1, 1, False, 2, 9, 11),     # identity block
    (1024, 512, 1, 2, True, 3, 14, 14),    # res5 head block 0: dilation 2, 1x1 downsample, stride 1 (IMAGE_C5_DILATED)
    (256, 64, 2, 1, False, 2, 12, 10),     # stride in the 3x3 (stride_in_1x1 = False)
]


@pytest.mark.parametrize("case", BLOCK_CASES)
def test_bottleneck_against_bf16_storage_oracle(case):
    """One Bottleneck (resnet.py:98-118), forward + backward, on identical bf16 inputs against the oracle graph with the
    same bf16 storage points: the ReLU masks agree, so the comparison is tight."""
    from vlbert_b200.resnet import Bottleneck, make_layer
    inpl, planes, stride, dil, s11, N, H, W = case
    torch.manual_seed(sum(case))
    layer, _ = make_layer(inpl, planes, 1, stride=stride, dilation=dil, stride_in_1x1=s11)
    blk = layer[0]
    sd = fo.synth_frontend_state({"blk." + k: v.shape for k, v in blk.state_dict().items()}, 5)
    blk.load_state_dict({k[4:]: v for k, v in sd.items()})
    blk = blk.to(DEV).eval()
    g = torch.Generator().manual_seed(1)
    x = bf(torch.randn(N, inpl, H, W, generator=g))
    names = [k for k in sd if k.endswith("conv1.weight") or k.endswith("conv2.weight") or k.endswith("conv3.weight") or k.endswith("downsample.0.weight")]
    for k in names:
        sd[k] = sd[k].clone().requires_grad_(True)
    xr = x.clone().requires_grad_(True)
    y_ref = fo.bottleneck(sd, "blk", xr, stride, dil, s11, storage="bf16")
    gy = bf(torch.randn(y_ref.shape, generator=g))
    y_ref.backward(gy)
    xo = nhwc(x.to(DEV)).requires_grad_(True)
    y = blk(xo)
    y.backward(nhwc(gy.to(DEV)))
    assert rel(nchw(y), y_ref) <= 2e-3, rel(nchw(y), y_ref)
    assert rel(nchw(xo.grad), xr.grad) <= 1.5e-2, rel(nchw(xo.grad), xr.grad)     # measured 5e-3 .. 7e-3
    for k in names:
        mine = dict(blk.named_parameters())[k[4:]].grad
        assert rel(mine, sd[k].grad) <= 1.5e-2, (k, rel(mine, sd[k].grad))


@pytest.mark.parametrize("compact", [True, False])
def test_fastrcnn_end_to_end_against_reference_fixture(golden_dir, compact):
    G = np.load(os.path.join(golden_dir, "fastrcnn_e2e.npz"))
    m, sd = _load_e2e()
    m.compact_rois = compact
    images, boxes, box_mask, im_info, gw = [t.to(DEV) for t in synth_frontend_inputs(78)]
    from vlbert_b200 import functional as VF
    body4 = VF.nhwc_to_nchw_f32(m.backbone(images)["body4"])
    e = {"body4": rel(body4[:, ::8], torch.from_numpy(G["body4_slice"]))}
    out = m(images=images, boxes=boxes, box_mask=box_mask, im_info=im_info)
    e["obj_reps"] = rel(out["obj_reps"], torch.from_numpy(G["obj_reps"]))
    e["obj_reps_raw"] = rel(out["obj_reps_raw"], torch.from_numpy(G["obj_reps_raw"]))
    pad = ~torch.from_numpy(G["obj_reps"]).abs().sum(-1).bool()
    assert bool((out["obj_reps"].cpu()[pad] == 0).all())
    m.zero_grad()
    (out["obj_reps"] * gw).sum().backward()
    params = dict(m.named_parameters())
    for name, rows in E2E_GRAD_SLICES:
        gfull = params[name].grad
        e["grad:" + name] = rel(gfull if rows is None else gfull[:rows], torch.from_numpy(G["grad:" + name]))
        a, b = (gfull if rows is None else gfull[:rows]).double().cpu().flatten(), torch.from_numpy(G["grad:" + name]).double().flatten()
        e["cos:" + name] = float(a @ b / (a.norm() * b.norm()))
        assert abs(float(gfull.double().norm()) / float(G["gnorm:" + name]) - 1) < 5e-2, name
    print("fastrcnn_e2e vs reference fixture (fp32), relative L2:", {k: "%.2e" % v for k, v in e.items()})
    assert e["body4"] <= 3e-2 and e["obj_reps"] <= 3e-2 and e["obj_reps_raw"] <= 3e-2, e
    # Gradients of a 100-layer ReLU network cannot be pinned to the fp32 run tighter than the ReLU-mask flips allow (DESIGN.md 3):
    # the yardstick is the bf16 comparator -- the oracle graph with the SAME bf16 storage points as the CUDA path
    # (frontend_oracle storage="bf16") -- measured against the same reference fixture.  The CUDA path has to be within
    # 1.25x of the comparator's error on average (RMS over the checked tensors) and within 2x on every single tensor
    # (single tensors are noisy: a flipped mask moves one tensor's gradient by percents on either side).
    # The comparator computes in fp64 between the bf16 storage points.  In fp32, the host's convolutions sum in an order
    # that depends on its thread count and instruction set, which flips bf16 roundings and ReLU masks and so moves the
    # yardstick from host to host; fp64 sums leave every bf16 rounding, and with it the yardstick, the same on any host.
    sdc = {k: (v.clone().double().requires_grad_(v.is_floating_point() and "running" not in k) if v.is_floating_point() else v)
           for k, v in sd.items()}
    ci, cb, cm, cinfo, cgw = synth_frontend_inputs(78)
    c_obj, _ = fo.fast_rcnn_end2end(sdc, ci.double(), cb.double(), cm, cinfo.double(), storage="bf16")
    (c_obj * cgw.double()).sum().backward()
    ratios = {}
    for name, rows in E2E_GRAD_SLICES:
        gc = sdc[name].grad
        ec = rel(gc if rows is None else gc[:rows], torch.from_numpy(G["grad:" + name]))
        ratios[name] = (e["grad:" + name], ec)
    rms = lambda xs: (sum(x * x for x in xs) / len(xs)) ** 0.5  # noqa: E731
    ours_rms, cmp_rms = rms([a for a, _ in ratios.values()]), rms([b for _, b in ratios.values()])
    print("front-end gradient errors vs fixture, ours (bf16-storage comparator):", {k: "%.2e (%.2e)" % v for k, v in ratios.items()},
          "RMS %.3e (%.3e)" % (ours_rms, cmp_rms))
    assert ours_rms <= 1.25 * cmp_rms, (ours_rms, cmp_rms, ratios)
    assert all(a <= 2.0 * b + 1e-3 for a, b in ratios.values()), ratios
    assert all(v >= 0.95 for k, v in e.items() if k.startswith("cos:")), e
    # frozen parts get no gradient (IMAGE_FROZEN_BACKBONE_STAGES [1, 2], IMAGE_FROZEN_BN)
    assert all(p.grad is None for n, p in params.items() if n.startswith("backbone.layer1") or ".bn" in n or n.startswith("backbone.conv1"))
    assert all(p.grad is not None for n, p in params.items() if p.requires_grad)


def test_fastrcnn_end_to_end_against_the_oracle_other_shape():
    """a second geometry (odd sizes, 3 images, every box valid) against the CPU oracle directly"""
    m, sd = _load_e2e()
    images, boxes, box_mask, im_info, gw = synth_frontend_inputs(91, B=3, R=3, H=112, W=176)
    box_mask[:] = True
    boxes = boxes.abs() + 3.0
    boxes[..., 2:] = boxes[..., :2] + 30
    ref_obj, ref_raw = fo.fast_rcnn_end2end(sd, images, boxes, box_mask, im_info)
    out = m(images=images.to(DEV), boxes=boxes.to(DEV), box_mask=box_mask.to(DEV), im_info=im_info.to(DEV))
    assert rel(out["obj_reps_raw"], ref_raw) <= 3e-2 and rel(out["obj_reps"], ref_obj) <= 3e-2


def test_cnn_reg_loss_outputs():
    import vlbert_b200
    m = vlbert_b200.FastRCNN(frontend_config(50), average_pool=True, final_dim=64, enable_cnn_reg_loss=True).to(DEV).eval()
    images, boxes, box_mask, im_info, _ = [t.to(DEV) for t in synth_frontend_inputs(3)]
    classes = torch.randint(0, 81, box_mask.shape, device=DEV)
    out = m(images=images, boxes=boxes, box_mask=box_mask, im_info=im_info, classes=classes)
    K = int(box_mask.sum())
    assert out["obj_logits"].shape == (K, 81) and out["obj_labels"].shape == (K,) and out["cnn_regularization_loss"].shape == (1,)
    assert torch.isfinite(out["cnn_regularization_loss"]).all()


def test_fastrcnn_with_instance_masks_against_the_oracle():
    """`segms` (VCR): mask-weighted mean pool of the res5 map, common/fast_rcnn.py:151-156"""
    m, sd = _load_e2e()
    images, boxes, box_mask, im_info, gw = synth_frontend_inputs(11, B=2, R=3, H=96, W=128)
    box_mask[1, 2] = False
    segms = (torch.rand(2, 3, 14, 14, generator=torch.Generator().manual_seed(4)) > 0.4).float()
    ref_obj, ref_raw = fo.fast_rcnn_end2end(sd, images, boxes, box_mask, im_info, segms=segms)
    for compact in (True, False):
        m.compact_rois = compact
        out = m(images=images.to(DEV), boxes=boxes.to(DEV), box_mask=box_mask.to(DEV), im_info=im_info.to(DEV), segms=segms.to(DEV))
        assert rel(out["obj_reps_raw"], ref_raw) <= 3e-2 and rel(out["obj_reps"], ref_obj) <= 3e-2
        m.zero_grad()
        (out["obj_reps"] * gw.to(DEV)).sum().backward()
        assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in m.parameters() if p.requires_grad)
