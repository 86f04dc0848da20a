"""Seeded synthetic inputs / weights shared by the tests, bench.py and smoke().

`synth_vlbert_inputs` and `seeded_state_dict` must stay call-for-call identical to
oracle/make_golden.py (which produced tests/golden/*.npz from the real reference)."""
import torch


def synth_vlbert_inputs(B, T, R, H, vocab, seed, ragged=True):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(min(1000, vocab // 2), vocab, (B, T), generator=g)
    types = torch.randint(0, 2, (B, T), generator=g)
    tvis = torch.randn(B, T, H, generator=g)
    ovl = torch.randn(B, R, 2 * H, generator=g)
    tmask = torch.ones(B, T, dtype=torch.bool)
    omask = torch.ones(B, R, dtype=torch.bool)
    if ragged:
        for b in range(B):
            tl = int(torch.randint(max(1, T // 2), T + 1, (1,), generator=g))
            ol = int(torch.randint(1, R + 1, (1,), generator=g))
            if b == 0:
                tl, ol = T, R
            tmask[b, tl:] = False
            omask[b, ol:] = False
        ids = ids * tmask
    return ids, types, tvis, tmask, ovl, omask


def seeded_state_dict(model, seed, std=0.02):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, v in model.state_dict().items():
        if "LayerNorm.weight" in k or k.startswith("visual_ln") and k.endswith("weight"):
            sd[k] = 1.0 + 0.1 * torch.randn(v.shape, generator=g)
        elif k.endswith("bias"):
            sd[k] = 0.02 * torch.randn(v.shape, generator=g)
        else:
            sd[k] = std * torch.randn(v.shape, generator=g)
    return sd


def vlbert_loss(layers, pooled, seed):
    """The scalar the golden gradients were taken of (oracle/make_golden.py:run_vlbert)."""
    g = torch.Generator().manual_seed(seed + 1)
    gw = [torch.randn(l.shape, generator=g).to(l.device) for l in layers]
    gp = torch.randn(pooled.shape, generator=g).to(pooled.device)
    loss = sum((l.float() * w).sum() for l, w in zip(layers, gw)) * 0.5 + (pooled.float() * gp).sum()
    return loss + (layers[-1].float() * gw[-1]).sum() * 0.5


E2E_GRAD_SLICES = (("obj_downsample.1.bias", None), ("obj_downsample.1.weight", 8),
                   ("roi_head_feature_extractor.2.conv3.weight", 32), ("roi_head_feature_extractor.0.conv2.weight", 4),
                   ("roi_head_feature_extractor.0.downsample.0.weight", 16), ("backbone.layer3.22.conv3.weight", 32),
                   ("backbone.layer3.0.conv2.weight", 8), ("backbone.layer2.0.conv1.weight", None),
                   ("backbone.layer2.0.conv2.weight", 8), ("backbone.layer2.0.downsample.0.weight", 16))


def synth_frontend_inputs(seed, B=2, R=4, H=128, W=160):
    """call-for-call identical to oracle/make_golden.py:synth_frontend_inputs"""
    g = torch.Generator().manual_seed(seed)
    images = torch.randn(B, 3, H, W, generator=g)
    im_info = torch.tensor([[float(W), float(H), 1.0, 1.0]] * B)
    x1 = torch.rand(B, R, generator=g) * W * 0.55
    y1 = torch.rand(B, R, generator=g) * H * 0.55
    x2 = x1 + 12 + torch.rand(B, R, generator=g) * W * 0.4
    y2 = y1 + 12 + torch.rand(B, R, generator=g) * H * 0.4
    boxes = torch.stack((x1, y1, x2.clamp(max=W - 1), y2.clamp(max=H - 1)), -1)
    box_mask = torch.ones(B, R, dtype=torch.bool)
    box_mask[1, R - 1:] = False
    boxes[~box_mask] = -2.0
    grad_out = torch.randn(B, R, 64, generator=g)
    return images, boxes, box_mask, im_info, grad_out


def frontend_config(num_layers=101):
    import types
    return types.SimpleNamespace(NETWORK=types.SimpleNamespace(
        IMAGE_FEAT_PRECOMPUTED=False, IMAGE_SEMANTIC=False, IMAGE_STRIDE_IN_1x1=True, IMAGE_C5_DILATED=True, IMAGE_NUM_LAYERS=num_layers,
        IMAGE_PRETRAINED="", IMAGE_PRETRAINED_EPOCH=0, OUTPUT_CONV5=False, IMAGE_FROZEN_BN=True, IMAGE_FROZEN_BACKBONE_STAGES=[1, 2]))


def frontend_shapes(num_layers=101, final_dim=64):
    """{state_dict key: shape} of the reference's end-to-end FastRCNN (common/fast_rcnn.py:36-109), written out from the
    module definitions so the oracle needs no nn.Module."""
    shapes = {}

    def bn(p, c):
        shapes[p + ".weight"] = shapes[p + ".bias"] = shapes[p + ".running_mean"] = shapes[p + ".running_var"] = (c,)
        shapes[p + ".num_batches_tracked"] = ()

    def layer(p, inpl, planes, blocks, first_has_ds=True):
        for i in range(blocks):
            q = "%s.%d" % (p, i)
            cin = inpl if i == 0 else planes * 4
            shapes[q + ".conv1.weight"] = (planes, cin, 1, 1); bn(q + ".bn1", planes)
            shapes[q + ".conv2.weight"] = (planes, planes, 3, 3); bn(q + ".bn2", planes)
            shapes[q + ".conv3.weight"] = (planes * 4, planes, 1, 1); bn(q + ".bn3", planes * 4)
            if i == 0:
                shapes[q + ".downsample.0.weight"] = (planes * 4, cin, 1, 1); bn(q + ".downsample.1", planes * 4)
    shapes["backbone.conv1.weight"] = (64, 3, 7, 7); bn("backbone.bn1", 64)
    inpl = 64
    for i, (planes, blocks) in enumerate(zip((64, 128, 256), {50: (3, 4, 6), 101: (3, 4, 23), 152: (3, 8, 36)}[num_layers])):
        layer("backbone.layer%d" % (i + 1), inpl, planes, blocks)
        inpl = planes * 4
    layer("roi_head_feature_extractor", inpl, 512, 3)
    for k in [k for k in shapes if k.startswith("roi_head_feature_extractor.")]:
        shapes["head.0." + k[len("roi_head_feature_extractor."):]] = shapes[k]
    shapes["obj_downsample.1.weight"] = (final_dim, 4096)
    shapes["obj_downsample.1.bias"] = (final_dim,)
    return shapes


def adamw_case(seed=5):
    """call-for-call identical to oracle/make_golden.py:adamw_case"""
    g = torch.Generator().manual_seed(seed)
    shapes = [(37, 19), (19,), (8, 3, 5)]
    params = [torch.randn(s, generator=g) for s in shapes]
    grads = [[torch.randn(s, generator=g) * (0.5 + k) for s in shapes] for k in range(4)]
    groups = [dict(idx=[0, 2], lr=2e-3, weight_decay=0.01), dict(idx=[1], lr=1e-3, weight_decay=0.0)]
    lr_scale = [0.25, 0.5, 0.75, 1.0]
    return params, grads, groups, lr_scale


def fake_hf_checkpoint(kind, H=64, L=2, I=128, vocab=120, max_pos=40):
    """a state_dict with HuggingFace BERT (old TF-style gamma/beta names, cls.* heads) or RoBERTa (roberta.*, lm_head.*, one
    token type) key names, random values"""
    g = torch.Generator().manual_seed(7 if kind == "bert" else 8)
    r = lambda *s: torch.randn(*s, generator=g)
    pre = "bert." if kind == "bert" else "roberta."
    ln_w, ln_b = ("gamma", "beta") if kind == "bert" else ("weight", "bias")
    sd = {pre + "embeddings.word_embeddings.weight": r(vocab, H), pre + "embeddings.position_embeddings.weight": r(max_pos, H),
          pre + "embeddings.token_type_embeddings.weight": r(2 if kind == "bert" else 1, H),
          pre + "embeddings.LayerNorm." + ln_w: r(H), pre + "embeddings.LayerNorm." + ln_b: r(H),
          pre + "embeddings.position_ids": torch.arange(max_pos)[None],                       # unexpected key
          pre + "pooler.dense.weight": r(H, H), pre + "pooler.dense.bias": r(H)}
    for l in range(L):
        q = pre + "encoder.layer.%d." % l
        for n, shp in (("attention.self.query", (H, H)), ("attention.self.key", (H, H)), ("attention.self.value", (H, H)),
                       ("attention.output.dense", (H, H)), ("intermediate.dense", (I, H)), ("output.dense", (H, I))):
            sd[q + n + ".weight"], sd[q + n + ".bias"] = r(*shp), r(shp[0])
        for n in ("attention.output.LayerNorm", "output.LayerNorm"):
            sd[q + n + "." + ln_w], sd[q + n + "." + ln_b] = r(H), r(H)
    if kind == "bert":
        sd.update({"cls.seq_relationship.weight": r(2, H), "cls.seq_relationship.bias": r(2),
                   "cls.predictions.bias": r(vocab), "cls.predictions.transform.dense.weight": r(H, H),
                   "cls.predictions.transform.dense.bias": r(H), "cls.predictions.transform.LayerNorm.gamma": r(H),
                   "cls.predictions.transform.LayerNorm.beta": r(H), "cls.predictions.decoder.weight": r(vocab, H)})
    else:
        sd.update({"lm_head.bias": r(vocab), "lm_head.dense.weight": r(H, H), "lm_head.dense.bias": r(H),
                   "lm_head.layer_norm.weight": r(H), "lm_head.layer_norm.bias": r(H), "lm_head.decoder.weight": r(vocab, H)})
    sd["some.other.tensor"] = r(3)
    return sd
