"""CPU: the oracle and the drop-in modules against the unmodified reference.  Most tests compare with what the reference
computed on the same seeded inputs, stored in tests/golden/reference_parity.{npz,json} by oracle/make_golden_reference.py;
the tests that run the reference's own task modules on top of the drop-in need the reference tree itself and are skipped
where it is absent."""
import json
import os
import sys

import numpy as np
import pytest
import torch

import ref_shim
import vlbert_oracle as vo
from make_golden_reference import (ABI_KW, E2E_CFG, LOADER_KW, ORACLE_KW, compared_rows, digest, digest_json, loaded_keys,
                                   masks_inputs, roialign_inputs, sample_index)
from synth import fake_hf_checkpoint, seeded_state_dict, synth_vlbert_inputs

needs_reference = pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")


@pytest.fixture(scope="module")
def gold(golden_dir):
    with open(os.path.join(golden_dir, "reference_parity.json")) as f:
        return np.load(os.path.join(golden_dir, "reference_parity.npz")), json.load(f)


def _close_to_sample(got, arrays, key, atol, rtol):
    """`got` against the reference's stored sample of the same tensor: |got - want| <= atol + rtol |want| elementwise"""
    assert tuple(got.shape) == tuple(arrays[key + "_shape"]), (key, tuple(got.shape), tuple(arrays[key + "_shape"]))
    want = arrays[key]
    g = got.detach().reshape(-1).numpy()[sample_index(got.numel())]
    assert g.shape == want.shape and np.allclose(g, want, atol=atol, rtol=rtol), (key, np.abs(g - want).max())


@pytest.mark.parametrize("ragged", [False, True])
def test_oracle_equals_reference_module(gold, ragged):
    arrays, _ = gold
    ora = vo.VisualLinguisticBertOracle(vo.default_config(**ORACLE_KW)).eval()
    ora.load_state_dict(seeded_state_dict(ora, 5, std=0.05), strict=True)
    inputs = synth_vlbert_inputs(B=4, T=12, R=7, H=128, vocab=300, seed=9, ragged=ragged)
    with torch.no_grad():
        text, obj, pooled = ora(*inputs, output_all_encoded_layers=True, output_text_and_object_separately=True)
    assert len(text) == len(obj) == ORACLE_KW["num_hidden_layers"]
    for name, ts in (("text", text), ("object", obj), ("pooled", [pooled])):
        for i, t in enumerate(ts):
            key = "vlbert_ragged%d_%s%d" % (ragged, name, i)
            _close_to_sample(t, arrays, key, atol=2e-5, rtol=1e-5)
            assert abs(float(t.abs().max()) - float(arrays[key + "_absmax"])) <= 2e-5 + 1e-5 * float(arrays[key + "_absmax"]), key


def test_reference_cpu_roialign_equals_c_oracle(gold):
    import roi_align as ro
    _, meta = gold
    f, rois = roialign_inputs()
    for sr in (1, 2, 0):
        b = ro.roi_align_forward(f.numpy(), rois.numpy(), 1 / 16.0, 14, 14, sr)
        assert digest(b) == meta["roialign_sha256"][str(sr)], sr           # bit-exact


def test_dropin_classes_have_the_reference_checkpoint_abi(gold):
    """state_dict keys + shapes of the drop-in modules == the reference modules (SURVEY 8b.2)."""
    import vlbert_b200
    _, meta = gold
    for our_cls, args in ((vlbert_b200.VisualLinguisticBert, ()),
                          (vlbert_b200.VisualLinguisticBertForPretraining, (None, True, True, True))):
        b = our_cls(vo.default_config(**ABI_KW), *args).state_dict()
        assert digest_json([[k, list(v.shape)] for k, v in b.items()]) == meta["vlbert_state_dict"][our_cls.__name__], \
            [(k, tuple(v.shape)) for k, v in b.items()]


@needs_reference
def test_dropin_install_patches_the_reference_modules():
    ref_shim.install()
    import vlbert_b200
    assert vlbert_b200.dropin.install()
    import common.fast_rcnn
    import common.visual_linguistic_bert as m
    assert m.VisualLinguisticBert is vlbert_b200.VisualLinguisticBert
    assert m.VisualLinguisticBertForPretraining is vlbert_b200.VisualLinguisticBertForPretraining
    from easydict import EasyDict
    frcnn = common.fast_rcnn.FastRCNN(EasyDict({"NETWORK": {"IMAGE_FEAT_PRECOMPUTED": True, "IMAGE_SEMANTIC": False}}), True, 768)
    assert isinstance(frcnn, vlbert_b200.FastRCNN)
    assert list(frcnn.state_dict().keys()) == ["obj_downsample.1.weight", "obj_downsample.1.bias"]
    # the task module builds on the patched classes (construction only: forward needs a GPU)
    import importlib
    import pretrain.modules.resnet_vlbert_for_pretraining as tm
    importlib.reload(tm)
    assert tm.VisualLinguisticBertForPretraining is vlbert_b200.VisualLinguisticBertForPretraining


def test_end_to_end_fastrcnn_has_the_reference_checkpoint_abi(gold):
    """ResNet-101 C4 + res5 head (common/fast_rcnn.py:36-102): same state_dict keys/shapes/dtypes and the same trainable set."""
    import types
    import warnings
    import vlbert_b200
    _, meta = gold
    cfg = types.SimpleNamespace(NETWORK=types.SimpleNamespace(**E2E_CFG))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ours = vlbert_b200.FastRCNN(cfg, True, 768, True)
    b = ours.state_dict()
    assert digest_json([[k, list(v.shape), str(v.dtype)] for k, v in b.items()]) == meta["fastrcnn_e2e_state_dict"]
    tb = [n for n, p in ours.named_parameters() if p.requires_grad]
    assert digest_json(tb) == meta["fastrcnn_e2e_trainable"] and len(tb) > 0


@pytest.mark.parametrize("kind", ["bert", "roberta"])
@pytest.mark.parametrize("pretraining", [False, True])
def test_language_checkpoint_loader_equals_the_reference(gold, tmp_path, kind, pretraining, capsys):
    """load_language_pretrained_model (common/visual_linguistic_bert.py:243-309 and :382-470): same tensors end up in the same
    parameters, including the relationship / MLM heads of the pre-training class and the RoBERTa renames."""
    import vlbert_b200
    want = gold[1]["language_loader"]["%s_%d" % (kind, pretraining)]
    path = str(tmp_path / "lm.bin")
    torch.save(fake_hf_checkpoint(kind), path)
    cls = vlbert_b200.VisualLinguisticBertForPretraining if pretraining else vlbert_b200.VisualLinguisticBert
    ours = cls(vo.default_config(**LOADER_KW), path)
    capsys.readouterr()
    b = ours.state_dict()
    assert digest_json(list(b.keys())) == want["keys"], list(b.keys())
    compared = {}
    for k in loaded_keys(list(b), kind):
        rows = compared_rows(k, kind, pretraining)
        if rows != 0:
            compared[k] = digest(b[k] if rows is None else b[k][:rows])
    assert sorted(compared) == sorted(want["sha256"])
    assert [k for k in compared if compared[k] != want["sha256"][k]] == []          # bit-exact
    assert torch.equal(b["mlm_head.predictions.decoder.weight"], b["word_embeddings.weight"]) if pretraining else True


def test_frontend_oracle_with_instance_masks_equals_the_reference(gold):
    """FastRCNN end to end with `segms` (the VCR path): oracle/frontend_oracle.py against the reference module's outputs."""
    import frontend_oracle as fo
    from synth import frontend_shapes
    arrays, _ = gold
    sd = fo.synth_frontend_state(frontend_shapes(50, 32), 21)
    images, boxes, box_mask, im_info, segms = masks_inputs()
    torch.set_num_threads(8)
    with torch.no_grad():
        got = dict(zip(("obj_reps", "obj_reps_raw"),
                       fo.fast_rcnn_end2end(sd, images, boxes, box_mask, im_info, layers=fo.LAYERS[50], segms=segms)))
    for k, t in got.items():
        absmax = float(arrays["masks_%s_absmax" % k])
        _close_to_sample(t, arrays, "masks_" + k, atol=1e-4 * absmax, rtol=0.0)
        assert abs(float(t.abs().max()) - absmax) <= 1e-4 * absmax, k


@needs_reference
def test_reference_pretraining_task_module_runs_unchanged_on_the_dropin(tmp_path, monkeypatch, capsys):
    """The boundary itself (SURVEY 8b): pretrain/modules/resnet_vlbert_for_pretraining.py built from the reference's own
    cfgs/pretrain/base_prec_4x16G_fp32.yaml (2 layers), once untouched and once after vlbert_b200.dropin.install() -- same
    state_dict keys, and on the same weights and inputs the same logits, losses and parameter gradients.  The kernels are
    replaced by fp32 torch stand-ins (tests/cpu_shim.py), so this checks everything the Python layer of the drop-in decides."""
    import importlib
    import warnings
    ref_shim.install()
    import cpu_shim
    import vlbert_b200
    vocab_dir = tmp_path / "bert-base-uncased"
    vocab_dir.mkdir()
    (vocab_dir / "vocab.txt").write_text("\n".join(["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + ["tok%d" % i for i in range(30517)]) + "\n")
    import pretrain.function.config as cfgmod
    cfgmod = importlib.reload(cfgmod)               # update_config() is not idempotent on the module-level singleton
    config, update_config = cfgmod.config, cfgmod.update_config
    update_config(os.path.join(ref_shim.REFERENCE_ROOT, "cfgs", "pretrain", "base_prec_4x16G_fp32.yaml"))
    config.NETWORK.VLBERT.num_hidden_layers = 2
    config.NETWORK.VLBERT.hidden_dropout_prob = 0.0
    config.NETWORK.VLBERT.attention_probs_dropout_prob = 0.0
    config.NETWORK.BERT_MODEL_NAME = str(vocab_dir)
    config.NETWORK.BERT_PRETRAINED = ""
    import common.fast_rcnn
    import common.visual_linguistic_bert
    import pretrain.modules.resnet_vlbert_for_pretraining as tm

    def fresh():
        importlib.reload(common.fast_rcnn)
        importlib.reload(common.visual_linguistic_bert)
        return importlib.reload(tm)

    g = torch.Generator().manual_seed(3)
    B, R, T, C = 2, 4, 8, config.NETWORK.VLBERT.visual_region_classes
    x1, y1 = torch.rand(B, R, generator=g) * 300, torch.rand(B, R, generator=g) * 200
    boxes = torch.cat((torch.stack((x1, y1, x1 + 20 + torch.rand(B, R, generator=g) * 250, y1 + 20 + torch.rand(B, R, generator=g) * 150), -1),
                       torch.randn(B, R, 2048, generator=g)), -1)
    boxes[1, 3] = -2.0                                                       # pretrain/data/collate_batch.py:39
    im_info = torch.tensor([[600., 400., 1., 1., 0.], [600., 400., 1., 1., 1.]])
    text = torch.randint(1000, 30522, (B, T), generator=g)
    text[1, 6:] = 0
    rel_label = torch.ones(B, dtype=torch.long)
    mlm_labels = torch.full((B, T), -1, dtype=torch.long)
    mlm_labels[0, 2], mlm_labels[1, 4] = 1234, 4321
    mvrc_ops = torch.tensor([[0, 1, 0, 0], [1, 0, 0, 0]])
    mvrc_labels = torch.zeros(B, R, C)
    mvrc_labels[mvrc_ops == 1] = torch.softmax(torch.randn(2, C, generator=g), -1)

    def run(model):
        model.zero_grad()
        out, loss = model(None, boxes.clone(), im_info, text, rel_label, mlm_labels, mvrc_ops, mvrc_labels.clone())
        loss.backward()
        return out, loss, {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}

    try:
        torch.manual_seed(0)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = fresh().ResNetVLBERTForPretraining(config)
            ref.eval()          # (the reference's train() override returns None)
            sd = {k: v.clone() for k, v in ref.state_dict().items()}
            o1, l1, g1 = run(ref)                 # the untouched reference first: install() rebinds the names its super() calls use
            assert vlbert_b200.dropin.install()
            cpu_shim.install(monkeypatch)
            cpu_shim.install_encoder(monkeypatch)
            ours = importlib.reload(tm).ResNetVLBERTForPretraining(config)
            ours.eval()
            assert isinstance(ours.vlbert, vlbert_b200.VisualLinguisticBertForPretraining)
            assert isinstance(ours.image_feature_extractor, vlbert_b200.FastRCNN)
            assert list(ours.state_dict().keys()) == list(sd.keys())
            ours.load_state_dict(sd, strict=True)
            o2, l2, g2 = run(ours)
        capsys.readouterr()
        assert abs(float(l1.detach()) - float(l2.detach())) <= 1e-5 * abs(float(l1.detach())), (float(l1.detach()), float(l2.detach()))
        for k in ("relationship_logits", "mlm_logits", "mvrc_logits", "relationship_loss", "mlm_loss", "mvrc_loss"):
            assert (o1[k] is None) == (o2[k] is None), k
            if o1[k] is not None:
                assert (o1[k] - o2[k]).abs().max() <= 2e-4 * o1[k].abs().max().clamp_min(1e-6), k
        assert set(g1.keys()) == set(g2.keys())
        for k in g1:
            assert (g1[k] - g2[k]).abs().max() <= 5e-4 * g1[k].abs().max().clamp_min(1e-9), k
    finally:
        fresh()


def _task_module_parity(monkeypatch, capsys, task, yaml_name, cls_name, tweak, build_inputs, call, vocab_dir, tol_out=2e-4, tol_grad=5e-4, zoo=None, after_build=None):
    """Build `<task>.modules.<cls_name>` from the reference's own yaml twice -- untouched, then with vlbert_b200.dropin installed
    and the kernels replaced by the fp32 stand-ins of tests/cpu_shim.py -- load the same weights, run the same inputs, and compare
    every tensor output, the loss and every parameter gradient."""
    import importlib
    import warnings
    import cpu_shim
    import vlbert_b200
    import torch.utils.model_zoo as model_zoo
    monkeypatch.setattr(model_zoo, "load_url", lambda *a, **k: (zoo if zoo is not None else {}))   # no network: the "model zoo"
    cfgmod = importlib.reload(importlib.import_module(task + ".function.config"))   # update_config() is not idempotent on the singleton
    config = cfgmod.config
    cfgmod.update_config(os.path.join(ref_shim.REFERENCE_ROOT, "cfgs", task, yaml_name))
    config.NETWORK.VLBERT.hidden_dropout_prob = 0.0
    config.NETWORK.VLBERT.attention_probs_dropout_prob = 0.0
    config.NETWORK.BERT_MODEL_NAME = str(vocab_dir)
    config.NETWORK.BERT_PRETRAINED = ""
    tweak(config)
    import common.fast_rcnn
    import common.visual_linguistic_bert
    import common.lib.roi_pooling.roi_align as ref_roi
    f, b = ref_shim.cpu_roi_functions()
    monkeypatch.setattr(ref_roi.C_ROIPooling, "roi_align_forward", f, raising=False)
    monkeypatch.setattr(ref_roi.C_ROIPooling, "roi_align_backward", b, raising=False)
    tm = importlib.import_module(task + ".modules")

    def fresh():
        importlib.reload(common.fast_rcnn)
        importlib.reload(common.visual_linguistic_bert)
        for name in sorted(k for k in sys.modules if k.startswith(task + ".modules.")):
            importlib.reload(sys.modules[name])
        return importlib.reload(tm)

    inputs = build_inputs(config)

    def run(model):
        model.zero_grad()
        out, loss = call(model, [t.clone() if torch.is_tensor(t) else t for t in inputs])
        loss.backward()
        return out, loss.detach(), {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}

    try:
        torch.manual_seed(0)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = getattr(fresh(), cls_name)(config)
            ref.eval()
            sd = {k: v.clone() for k, v in ref.state_dict().items()}
            o1, l1, g1 = run(ref)                 # the untouched reference first: install() rebinds the names its super() calls use
            assert vlbert_b200.dropin.install()
            cpu_shim.install(monkeypatch)
            cpu_shim.install_encoder(monkeypatch)
            for name in sorted(k for k in sys.modules if k.startswith(task + ".modules.")):
                importlib.reload(sys.modules[name])
            ours = getattr(importlib.reload(tm), cls_name)(config)
            ours.eval()
            assert isinstance(ours.image_feature_extractor, vlbert_b200.FastRCNN)
            assert list(ours.state_dict().keys()) == list(sd.keys())
            if after_build is not None:
                after_build(sd, ours)
            ours.load_state_dict(sd, strict=True)
            o2, l2, g2 = run(ours)
        capsys.readouterr()
        assert abs(float(l1) - float(l2)) <= 1e-5 * max(1e-6, abs(float(l1))), (float(l1), float(l2))
        for k in o1:
            if torch.is_tensor(o1[k]) and o1[k].is_floating_point():
                assert (o1[k] - o2[k]).abs().max() <= tol_out * o1[k].abs().max().clamp_min(1e-6), k
        assert set(g1.keys()) == set(g2.keys())
        for k in g1:
            assert (g1[k] - g2[k]).abs().max() <= tol_grad * g1[k].abs().max().clamp_min(1e-9), k
        return ours
    finally:
        fresh()


def _vocab_dir(tmp_path, n, with_checkpoint=None):
    d = tmp_path / "bert-base-uncased"
    d.mkdir()
    (d / "vocab.txt").write_text("\n".join(["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + ["tok%d" % i for i in range(n - 5)]) + "\n")
    if with_checkpoint is not None:
        torch.save(with_checkpoint, str(d / "pytorch_model.bin"))
    return d


@needs_reference
def test_reference_vqa_task_module_runs_unchanged_on_the_dropin(tmp_path, monkeypatch, capsys):
    """vqa/modules/resnet_vlbert_for_vqa.py from cfgs/vqa/base_4x16G_fp32.yaml (BASELINE config 3's module; 2 layers, vocabulary cut to
    1000): `mlm` classifier initialised from a BERT checkpoint through the module's own loader, uint8 text masks from
    prepare_text_from_qa, precomputed region features."""
    ref_shim.install()
    vocab = 1000
    d = _vocab_dir(tmp_path, vocab, fake_hf_checkpoint("bert", H=768, L=2, I=3072, vocab=vocab, max_pos=512))

    def tweak(config):
        config.NETWORK.VLBERT.num_hidden_layers = 2
        config.NETWORK.VLBERT.vocab_size = vocab
        config.NETWORK.CLASSIFIER_DROPOUT = 0.0
        config.DATASET.ANSWER_VOCAB_SIZE = 37

    def build_inputs(config):
        g = torch.Generator().manual_seed(5)
        B, R, T = 3, 5, 7
        x1, y1 = torch.rand(B, R, generator=g) * 300, torch.rand(B, R, generator=g) * 200
        boxes = torch.cat((torch.stack((x1, y1, x1 + 20 + torch.rand(B, R, generator=g) * 250, y1 + 20 + torch.rand(B, R, generator=g) * 150), -1),
                           torch.randn(B, R, 2048, generator=g)), -1)
        boxes[1, 3:] = -2.0
        boxes[2, 4:] = -2.0
        im_info = torch.tensor([[600., 400., 1., 1.]] * B)
        question = torch.randint(5, vocab, (B, T), generator=g)
        question[0, 5:] = 0
        question[2, 3:] = 0
        label = torch.rand(B, 37, generator=g)
        return [None, boxes, im_info, question, label]

    _task_module_parity(monkeypatch, capsys, "vqa", "base_4x16G_fp32.yaml", "ResNetVLBERT", tweak, build_inputs,
                        lambda m, ins: m.train_forward(*ins), d)


@needs_reference
def test_reference_vcr_task_module_runs_unchanged_on_the_dropin(tmp_path, monkeypatch, capsys):
    """vcr/modules/resnet_vlbert_for_vcr.py from cfgs/vcr/base_q2a_4x16G_fp32.yaml (BASELINE config 4's module at base width; 2 layers):
    images through the END-TO-END FastRCNN (ResNet-101 C4 + RoIAlign + dilated res5) with instance masks (`segms`) and object classes,
    TimeDistributed VL-BERT over the four answer choices, text/object outputs returned separately, the CNN regularisation head on
    the object outputs.  Exercises the drop-in's end-to-end front end under its real caller."""
    ref_shim.install()
    import torch.utils.model_zoo as model_zoo
    from common.backbone.resnet.resnet import Bottleneck, ResNet
    vocab = 600
    d = _vocab_dir(tmp_path, vocab)
    torch.manual_seed(1)
    zoo = ResNet(Bottleneck, [3, 4, 23, 3], num_classes=None, expose_stages=[5]).state_dict()      # what the model zoo would return
    for k, v in zoo.items():                                                                      # non-trivial frozen statistics
        if k.endswith("running_var"):
            v.uniform_(0.5, 1.5)
        elif k.endswith("running_mean"):
            v.normal_(0, 0.1)
        elif ".bn" in k and k.endswith("weight") or "downsample.1.weight" in k:
            v.uniform_(0.3, 0.6)

    torch.save(zoo, str(tmp_path / "resnet101-0000.model"))                                       # NETWORK.IMAGE_PRETRAINED checkpoint

    def tweak(config):
        config.NETWORK.VLBERT.num_hidden_layers = 2
        config.NETWORK.VLBERT.vocab_size = vocab
        config.NETWORK.CLASSIFIER_DROPOUT = 0.0
        config.NETWORK.IMAGE_PRETRAINED = str(tmp_path / "resnet101")
        config.NETWORK.IMAGE_PRETRAINED_EPOCH = 0
        assert config.NETWORK.IMAGE_FEAT_PRECOMPUTED is False and config.NETWORK.ENABLE_CNN_REG_LOSS and config.NETWORK.CNN_LOSS_TOP

    def after_build(ref_sd, ours):
        # both sides initialise the backbone and the res5 head (layer4.*) from the same IMAGE_PRETRAINED file (common/fast_rcnn.py:41-63,111-120)
        mine = ours.state_dict()
        for k in ref_sd:
            if k.startswith(("image_feature_extractor.backbone.", "image_feature_extractor.roi_head_feature_extractor.", "image_feature_extractor.head.")):
                assert torch.equal(mine[k], ref_sd[k]), k

    def build_inputs(config):
        g = torch.Generator().manual_seed(9)
        B, R, NC, Lq, La, H, W = 2, 3, 4, 5, 4, 64, 96
        image = torch.randn(B, 3, H, W, generator=g)
        x1, y1 = torch.rand(B, R, generator=g) * 40, torch.rand(B, R, generator=g) * 25
        boxes = torch.stack((x1, y1, x1 + 16 + torch.rand(B, R, generator=g) * 38, y1 + 16 + torch.rand(B, R, generator=g) * 20,
                             torch.randint(1, 81, (B, R), generator=g).float()), -1)
        boxes[:, 0, :4] = torch.tensor([0.0, 0.0, W - 1.0, H - 1.0])          # the whole image as the first box (ADD_IMAGE_AS_A_BOX)
        boxes[:, 0, 4] = 0
        boxes[1, 2] = -1.0                                                     # padded box
        masks = (torch.rand(B, R, 14, 14, generator=g) > 0.35).float()
        masks[:, 0] = 1.0
        question = torch.stack((torch.randint(5, vocab, (B, Lq), generator=g), torch.randint(-1, 2, (B, Lq), generator=g)), -1)
        question[1, 3:] = 0
        answers = torch.stack((torch.randint(5, vocab, (B, NC, La), generator=g), torch.randint(-1, 2, (B, NC, La), generator=g)), -1)
        answers[0, 1, 2:] = 0
        answers[1, 3, 3:] = 0
        answer_label = torch.tensor([2, 0])
        im_info = torch.tensor([[float(W), float(H), 1.0, 1.0]] * B)
        return [image, boxes, masks, question, None, answers, None, answer_label, im_info]

    torch.set_num_threads(8)
    _task_module_parity(monkeypatch, capsys, "vcr", "base_q2a_4x16G_fp32.yaml", "ResNetVLBERT", tweak, build_inputs,
                        lambda m, ins: m.train_forward(*ins), d, zoo=zoo, after_build=after_build)


@needs_reference
def test_reference_refcoco_task_module_runs_unchanged_on_the_dropin(tmp_path, monkeypatch, capsys):
    """refcoco/modules/resnet_vlbert_for_refcoco.py from cfgs/refcoco/base_detected_regions_4x16G.yaml (2 layers): end-to-end FastRCNN
    without masks, `with_pooler: false`, per-region classifier on the object outputs."""
    ref_shim.install()
    from common.backbone.resnet.resnet import Bottleneck, ResNet
    vocab = 500
    d = _vocab_dir(tmp_path, vocab)
    torch.manual_seed(2)
    zoo = ResNet(Bottleneck, [3, 4, 23, 3], num_classes=None, expose_stages=[5]).state_dict()
    for k, v in zoo.items():
        if k.endswith("running_var"):
            v.uniform_(0.5, 1.5)
        elif ".bn" in k and k.endswith("weight") or "downsample.1.weight" in k:
            v.uniform_(0.3, 0.6)
    torch.save(zoo, str(tmp_path / "resnet101-0000.model"))

    def tweak(config):
        config.NETWORK.VLBERT.num_hidden_layers = 2
        config.NETWORK.VLBERT.vocab_size = vocab
        config.NETWORK.IMAGE_PRETRAINED = str(tmp_path / "resnet101")
        config.NETWORK.IMAGE_PRETRAINED_EPOCH = 0

    def build_inputs(config):
        g = torch.Generator().manual_seed(13)
        B, R, T, H, W = 2, 4, 6, 64, 80
        image = torch.randn(B, 3, H, W, generator=g)
        x1, y1 = torch.rand(B, R, generator=g) * 30, torch.rand(B, R, generator=g) * 25
        boxes = torch.stack((x1, y1, x1 + 16 + torch.rand(B, R, generator=g) * 30, y1 + 16 + torch.rand(B, R, generator=g) * 20), -1)
        boxes[0, 3] = -2.0
        im_info = torch.tensor([[float(W), float(H), 1.0, 1.0]] * B)
        expression = torch.randint(5, vocab, (B, T), generator=g)
        expression[1, 4:] = 0
        label = (torch.rand(B, R, generator=g) > 0.5).float()
        return [image, boxes, im_info, expression, label]

    torch.set_num_threads(8)
    _task_module_parity(monkeypatch, capsys, "refcoco", "base_detected_regions_4x16G.yaml", "ResNetVLBERT", tweak, build_inputs,
                        lambda m, ins: m.train_forward(*ins), d, zoo=zoo)


@needs_reference
@pytest.mark.parametrize("yaml_name", ["base_e2e_16x16G_fp16.yaml", "base_prec_4x16G_fp32.yaml"])
def test_reference_multitask_pretraining_module_runs_unchanged_on_the_dropin(tmp_path, monkeypatch, capsys, yaml_name):
    """pretrain/modules/resnet_vlbert_for_pretraining_multitask.py -- the MODULE both pre-training yamls name, i.e. the real caller of
    BASELINE config 2 (precomputed features) and config 5 (end to end).  It appends text-only samples (no boxes at all: box_mask
    all False) to the batch, masks region features with `mask_visual_embed` on the end-to-end path, and uses all three heads."""
    ref_shim.install()
    from common.backbone.resnet.resnet import Bottleneck, ResNet
    e2e = "e2e" in yaml_name
    vocab = 700
    d = _vocab_dir(tmp_path, vocab)
    zoo = None
    if e2e:
        torch.manual_seed(4)
        zoo = ResNet(Bottleneck, [3, 4, 23, 3], num_classes=None, expose_stages=[5]).state_dict()
        for k, v in zoo.items():
            if k.endswith("running_var"):
                v.uniform_(0.5, 1.5)
            elif ".bn" in k and k.endswith("weight") or "downsample.1.weight" in k:
                v.uniform_(0.3, 0.6)
        torch.save(zoo, str(tmp_path / "resnet101-0000.model"))

    def tweak(config):
        config.NETWORK.VLBERT.num_hidden_layers = 2
        config.NETWORK.VLBERT.vocab_size = vocab
        config.NETWORK.VLBERT.visual_region_classes = 23
        if e2e:
            config.NETWORK.IMAGE_PRETRAINED = str(tmp_path / "resnet101")
            config.NETWORK.IMAGE_PRETRAINED_EPOCH = 0

    def build_inputs(config):
        g = torch.Generator().manual_seed(17)
        B, R, T, C, H, W = 2, 4, 7, 23, 64, 96
        x1, y1 = torch.rand(B, R, generator=g) * 40, torch.rand(B, R, generator=g) * 25
        box4 = torch.stack((x1, y1, x1 + 16 + torch.rand(B, R, generator=g) * 38, y1 + 16 + torch.rand(B, R, generator=g) * 20), -1)
        if e2e:
            image, boxes = torch.randn(B, 3, H, W, generator=g), box4
        else:
            image, boxes = None, torch.cat((box4, torch.randn(B, R, 2048, generator=g)), -1)
        boxes[1, 3] = -2.0
        im_info = torch.tensor([[float(W), float(H), 1.0, 1.0, 0.0], [float(W), float(H), 1.0, 1.0, 1.0]])
        text = torch.randint(5, vocab, (B, T), generator=g)
        text[1, 5:] = 0
        rel = torch.ones(B, dtype=torch.long)
        mlm = torch.full((B, T), -1, dtype=torch.long)
        mlm[0, 2], mlm[1, 3] = 77, 88
        mvrc_ops = torch.tensor([[0, 1, 0, 0], [1, 0, 0, 0]])
        mvrc_labels = torch.zeros(B, R, C)
        mvrc_labels[mvrc_ops == 1] = torch.softmax(torch.randn(2, C, generator=g), -1)
        aux_text = torch.randint(5, vocab, (3, 9), generator=g)            # three text-only samples, longer than the captions
        aux_text[0, 6:] = 0
        aux_mlm = torch.full((3, 9), -1, dtype=torch.long)
        aux_mlm[0, 1], aux_mlm[2, 8] = 99, 111
        return [image, boxes, im_info, text, rel, mlm, mvrc_ops, mvrc_labels, aux_text, aux_mlm]

    torch.set_num_threads(8)
    _task_module_parity(monkeypatch, capsys, "pretrain", yaml_name, "ResNetVLBERTForPretrainingMultitask", tweak, build_inputs,
                        lambda m, ins: m(*ins), d, zoo=zoo)
