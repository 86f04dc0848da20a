"""TEST INFRASTRUCTURE ONLY -- fp32 CPU restatement of the end-to-end region-feature front end.

Follows (reference file:line):
  Bottleneck.forward            common/backbone/resnet/resnet.py:98-118
  ResNet.forward (body4)        common/backbone/resnet/resnet.py:175-199  (expose_stages=[4], stride_in_1x1)
  res5 head + AvgPool + flatten common/fast_rcnn.py:74-86
  FastRCNN.forward, conv path   common/fast_rcnn.py:128-193
  _ROIAlign                     common/lib/roi_pooling/roi_align.py:11-43  (via oracle/roi_align_oracle.c)

It is a function of a reference-format state_dict (keys `backbone.*`, `roi_head_feature_extractor.*`,
`obj_downsample.1.*`), so it is pinned two ways: against the reference module's outputs with instance masks
(tests/test_oracle_vs_reference.py, tests/golden/reference_parity.npz) and by the committed fixture tests/golden/fastrcnn_e2e.npz that
oracle/make_golden.py wrote from the reference.  BatchNorm is the eval-mode (frozen statistics) map, the
only mode the reference runs the backbone in (common/fast_rcnn.py:122-126, FastRCNN.bn_eval).

`storage="bf16"` evaluates the same fp32 graph but rounds every tensor the CUDA path keeps in bf16 (images, conv
weights, each conv+BN(+ReLU) output, RoIAlign output, the region operand and the projection) to bf16, forward and
backward (straight-through).  ReLU networks amplify forward rounding into gradient error (a pre-activation within
rounding distance of 0 flips its mask and moves that element's gradient by 100%: relative L2 error ~ sqrt(fraction
flipped)), so the fp32 graph bounds the CUDA path's gradients only loosely; the bf16-storage graph has the same masks
and bounds them tightly.  tests/test_gpu_frontend.py uses both.  The graph computes in the dtype of its inputs (fp32, or
fp64 between the bf16 storage points for a comparator that does not depend on the host's summation order).

Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may import this module.
"""
import numpy as np
import torch
import torch.nn.functional as F

try:
    from . import roi_align as _roi
    from .vlbert_oracle import coordinate_embeddings
except ImportError:  # tests put oracle/ itself on sys.path
    import roi_align as _roi
    from vlbert_oracle import coordinate_embeddings

LAYERS = {50: (3, 4, 6), 101: (3, 4, 23), 152: (3, 8, 36)}


class _RoundBF16(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(g.dtype)


def _q(storage):
    if storage is None:
        return lambda t: t
    assert storage == "bf16"
    return _RoundBF16.apply


def _bn(sd, prefix, x, eps=1e-5):
    return F.batch_norm(x, sd[prefix + ".running_mean"], sd[prefix + ".running_var"], sd[prefix + ".weight"], sd[prefix + ".bias"],
                        False, 0.0, eps)


def bottleneck(sd, prefix, x, stride, dilation, stride_in_1x1, storage=None):
    """resnet.py:79-118.  `stride` applies to conv1 when stride_in_1x1 else to conv2; the downsample conv takes it too."""
    q = _q(storage)
    s1, s2 = (stride, 1) if stride_in_1x1 else (1, stride)
    o = q(torch.relu(_bn(sd, prefix + ".bn1", F.conv2d(x, q(sd[prefix + ".conv1.weight"]), stride=s1))))
    o = q(torch.relu(_bn(sd, prefix + ".bn2", F.conv2d(o, q(sd[prefix + ".conv2.weight"]), stride=s2, padding=dilation, dilation=dilation))))
    o = _bn(sd, prefix + ".bn3", F.conv2d(o, q(sd[prefix + ".conv3.weight"])))
    if prefix + ".downsample.0.weight" in sd:
        x = q(_bn(sd, prefix + ".downsample.1", F.conv2d(x, q(sd[prefix + ".downsample.0.weight"]), stride=stride)))
    return q(torch.relu(o + x))


def res_layer(sd, prefix, x, blocks, stride, dilation, stride_in_1x1, storage=None):
    """resnet.py:158-173: the first block carries the stride (and stride_in_1x1); the rest are stride 1."""
    x = bottleneck(sd, prefix + ".0", x, stride, dilation, stride_in_1x1, storage)
    for i in range(1, blocks):
        x = bottleneck(sd, "%s.%d" % (prefix, i), x, 1, dilation, False, storage)
    return x


def resnet_c4(sd, images, layers=(3, 4, 23), stride_in_1x1=True, prefix="backbone", storage=None):
    """resnet.py:175-186 up to body4."""
    q = _q(storage)
    x = q(torch.relu(_bn(sd, prefix + ".bn1", F.conv2d(q(images), q(sd[prefix + ".conv1.weight"]), stride=2, padding=3))))
    x = F.max_pool2d(x, kernel_size=3, stride=2, padding=1)
    for i, (blocks, stride) in enumerate(zip(layers, (1, 2, 2))):
        x = res_layer(sd, "%s.layer%d" % (prefix, i + 1), x, blocks, stride, 1, stride_in_1x1, storage)
    return x


class _RoIAlign(torch.autograd.Function):
    """roi_align.py:11-43 on the C restatement of ROIAlign_cpu.cpp / ROIAlign_cuda.cu."""

    @staticmethod
    def forward(ctx, feat, rois, ph, pw, scale, sr):
        ctx.save_for_backward(rois)
        ctx.cfg = (ph, pw, scale, sr, tuple(feat.shape))
        return torch.from_numpy(_roi.roi_align_forward(feat.detach().numpy(), rois.numpy(), scale, ph, pw, sr)).to(feat.dtype)

    @staticmethod
    def backward(ctx, g):
        (rois,) = ctx.saved_tensors
        ph, pw, scale, sr, (N, C, H, W) = ctx.cfg
        return torch.from_numpy(_roi.roi_align_backward(g.contiguous().numpy(), rois.numpy(), scale, ph, pw, N, C, H, W, sr)).to(g.dtype), \
            None, None, None, None, None


def fast_rcnn_end2end(sd, images, boxes, box_mask, im_info, layers=(3, 4, 23), stride_in_1x1=True, c5_dilated=True,
                      mvrc_ops=None, mask_visual_embed=None, storage=None, segms=None):
    """common/fast_rcnn.py:128-193 (no classes / segms, dropout p = 0).  Returns obj_reps [B,R,D], obj_reps_raw [B,R,2048]."""
    q = _q(storage)
    B, R = box_mask.shape
    idx = box_mask.nonzero()
    feat = resnet_c4(sd, images, layers, stride_in_1x1, storage=storage)
    rois = torch.cat((idx[:, 0, None].to(boxes.dtype), boxes[idx[:, 0], idx[:, 1]][:, :4]), 1)
    pooled = q(_RoIAlign.apply(feat, rois, 14, 14, 1.0 / 16, 1))
    x = res_layer(sd, "roi_head_feature_extractor", pooled, 3, 1 if c5_dilated else 2, 2 if c5_dilated else 1, stride_in_1x1, storage)
    if segms is not None:                      # common/fast_rcnn.py:151-156 (VCR instance masks)
        x = q(x * segms[idx[:, 0], None, idx[:, 1]].to(x.dtype))
    post = F.avg_pool2d(x, 14 if c5_dilated else 7, stride=1).flatten(1)
    feats = post
    if mvrc_ops is not None and mask_visual_embed is not None:
        feats = feats.clone()
        feats[(mvrc_ops == 1)[idx[:, 0], idx[:, 1]]] = mask_visual_embed
    ce = coordinate_embeddings(torch.cat((boxes[idx[:, 0], idx[:, 1]][:, :4], im_info[idx[:, 0], :2]), 1), 256)
    operand = q(torch.cat((ce.reshape(ce.shape[0], -1), feats), -1))
    final = q(torch.relu(F.linear(operand, q(sd["obj_downsample.1.weight"]), sd["obj_downsample.1.bias"])))
    slot = torch.cumsum(box_mask.long(), 1) - 1
    obj_reps = final.new_zeros((B, R, final.shape[1]))
    raw = post.new_zeros((B, R, post.shape[1]))
    obj_reps[idx[:, 0], slot[idx[:, 0], idx[:, 1]]] = final
    raw[idx[:, 0], slot[idx[:, 0], idx[:, 1]]] = post
    return obj_reps, raw


def synth_frontend_state(shapes, seed):
    """Deterministic weights for a FastRCNN state_dict ({name: shape}); numpy's legacy RandomState is stable across
    versions, so make_golden.py (reference side) and the tests (library side) regenerate identical tensors."""
    rs = np.random.RandomState(seed)
    sd = {}
    for k, shp in shapes.items():
        shp = tuple(shp)
        if k.startswith("head."):
            continue
        if k.endswith("num_batches_tracked"):
            v = np.zeros(shp, np.int64)
        elif k.endswith("running_mean"):
            v = 0.1 * rs.standard_normal(shp)
        elif k.endswith("running_var"):
            v = rs.uniform(0.5, 1.5, shp)
        elif ".bn" in k or k.startswith("backbone.bn1") or ".downsample.1." in k:
            if k.endswith("weight"):
                v = rs.uniform(0.25, 0.45, shp) if ".bn3." in k else rs.uniform(0.6, 1.0, shp)
            else:
                v = 0.1 * rs.standard_normal(shp)
        elif k.endswith("conv1.weight") or k.endswith("conv2.weight") or k.endswith("conv3.weight") or ".downsample.0." in k:
            fan_in = shp[1] * shp[2] * shp[3]
            v = rs.standard_normal(shp) * np.sqrt(2.0 / fan_in)
        elif k.endswith("bias"):
            v = 0.02 * rs.standard_normal(shp)
        else:
            v = 0.02 * rs.standard_normal(shp)
        sd[k] = torch.from_numpy(np.asarray(v)).to(torch.int64 if k.endswith("num_batches_tracked") else torch.float32)
    for k in shapes:                       # `head.0.*` aliases `roi_head_feature_extractor.*` (same module object)
        if k.startswith("head.0."):
            sd[k] = sd["roi_head_feature_extractor." + k[len("head.0."):]]
    return sd
