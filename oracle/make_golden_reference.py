"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/reference_parity.{npz,json}: what tests/test_oracle_vs_reference.py and
tests/test_task_glue.py compare the oracle and the library against, computed by the UNMODIFIED reference (via
oracle/ref_shim.py and oracle/build_ref.py) on the seeded inputs the tests regenerate.  Run where the reference tree exists:

    python oracle/make_golden_reference.py

Float tensors larger than SAMPLE elements are stored as a fixed seeded sample (`sample_index`) plus their shape and max |value|;
outputs the tests compare bit for bit are stored as SHA-256 digests of their bytes (`digest`).
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "..", "tests"))
import ref_shim  # noqa: E402

GOLD = os.path.join(HERE, "..", "tests", "golden")
SAMPLE = 1024


def sample_index(n, seed=0):
    """Flat indices of the stored sample of an n-element tensor (all of them when n <= SAMPLE)."""
    if n <= SAMPLE:
        return np.arange(n)
    return np.sort(np.random.RandomState(seed).choice(n, SAMPLE, replace=False))


def store_sampled(arrays, key, t):
    """the sample of `t` at arrays[key], with its shape and max |value|"""
    a = t.detach().reshape(-1).numpy()
    arrays[key] = a[sample_index(a.size)]
    arrays[key + "_shape"] = np.asarray(t.shape, np.int64)
    arrays[key + "_absmax"] = np.float32(t.abs().max())


def digest(t):
    a = np.ascontiguousarray(t.detach().numpy() if torch.is_tensor(t) else t)
    return hashlib.sha256(str(a.dtype).encode() + str(a.shape).encode() + a.tobytes()).hexdigest()


def digest_json(obj):
    return hashlib.sha256(json.dumps(obj).encode()).hexdigest()


def roialign_inputs():
    """tests/test_oracle_vs_reference.py:test_reference_cpu_roialign_equals_c_oracle"""
    g = torch.Generator().manual_seed(3)
    f = torch.randn(2, 8, 38, 63, generator=g)
    K = 40
    x1 = torch.rand(K, generator=g) * 900
    y1 = torch.rand(K, generator=g) * 550
    rois = torch.stack([torch.randint(0, 2, (K,), generator=g).float(), x1, y1, x1 + torch.rand(K, generator=g) * 300,
                        y1 + torch.rand(K, generator=g) * 300], 1)
    return f, rois


ORACLE_KW = dict(vocab_size=300, hidden_size=128, num_hidden_layers=3, num_attention_heads=2, intermediate_size=512,
                 max_position_embeddings=80, visual_size=128, with_pooler=True)
ABI_KW = dict(vocab_size=300, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
              max_position_embeddings=80, visual_size=128, visual_region_classes=11, pos_embedding_frozen=False)
LOADER_KW = dict(vocab_size=120, hidden_size=64, num_hidden_layers=2, num_attention_heads=1, intermediate_size=128,
                 max_position_embeddings=40, visual_size=64, visual_region_classes=7, pos_embedding_frozen=False)
E2E_CFG = dict(IMAGE_FEAT_PRECOMPUTED=False, IMAGE_SEMANTIC=False, IMAGE_STRIDE_IN_1x1=True, IMAGE_C5_DILATED=True,
               IMAGE_NUM_LAYERS=101, IMAGE_PRETRAINED="", IMAGE_PRETRAINED_EPOCH=0, OUTPUT_CONV5=False,
               IMAGE_FROZEN_BN=True, IMAGE_FROZEN_BACKBONE_STAGES=[1, 2])


def masks_inputs():
    """tests/test_oracle_vs_reference.py:test_frontend_oracle_with_instance_masks_equals_the_reference"""
    from synth import synth_frontend_inputs
    images, boxes, box_mask, im_info, _ = synth_frontend_inputs(12, B=2, R=3, H=80, W=112)
    box_mask[0, 2] = False
    segms = (torch.rand(2, 3, 14, 14, generator=torch.Generator().manual_seed(2)) > 0.5).float()
    return images, boxes, box_mask, im_info, segms


def loaded_keys(keys, kind):
    heads = ("relationsip_head.", "mlm_head.") if kind == "bert" else ("mlm_head.",)
    return [k for k in keys if k.startswith(("encoder.", "embedding_LayerNorm.", "word_embeddings.", "position_embeddings.",
                                             "pooler.") + heads)] + ["token_type_embeddings.weight"]


def compared_rows(k, kind, pretraining):
    """rows of token_type_embeddings the loader writes (the rest keep their random init); None = the whole tensor; 0 = not compared
    (the MLM decoder weight is tied to the word embeddings)"""
    if k == "token_type_embeddings.weight":
        return 2 if (kind == "bert" or pretraining) else 3
    if k.startswith("mlm_head.") and "decoder.weight" in k:
        return 0
    return None


def main():
    import warnings
    import torch.utils.model_zoo as model_zoo
    import vlbert_oracle as vo
    from synth import seeded_state_dict, synth_vlbert_inputs
    from frontend_oracle import synth_frontend_state
    ref_shim.install()
    from easydict import EasyDict
    arrays, meta = {}, {}

    # the oracle's VL-BERT against common/visual_linguistic_bert.py
    from common.visual_linguistic_bert import VisualLinguisticBert, VisualLinguisticBertForPretraining
    for ragged in (False, True):
        torch.manual_seed(0)
        ref = VisualLinguisticBert(ref_shim.vlbert_config(**ORACLE_KW)).eval()
        sd = seeded_state_dict(ref, 5, std=0.05)
        sd_o = seeded_state_dict(vo.VisualLinguisticBertOracle(vo.default_config(**ORACLE_KW)), 5, std=0.05)
        assert list(sd) == list(sd_o) and all(torch.equal(sd[k], sd_o[k]) for k in sd)   # the test seeds the oracle
        ref.load_state_dict(sd)
        inputs = synth_vlbert_inputs(B=4, T=12, R=7, H=128, vocab=300, seed=9, ragged=ragged)
        with torch.no_grad():
            text, obj, pooled = ref(*inputs, output_all_encoded_layers=True, output_text_and_object_separately=True)
        for name, ts in (("text", text), ("object", obj), ("pooled", [pooled])):
            for i, t in enumerate(ts):
                key = "vlbert_ragged%d_%s%d" % (ragged, name, i)
                store_sampled(arrays, key, t)

    # the reference's own CPU RoIAlign kernel (bit-exact comparison)
    import build_ref
    ext = build_ref.load()
    f, rois = roialign_inputs()
    meta["roialign_sha256"] = {str(sr): digest(ext.roi_align_forward(f, rois, 1 / 16.0, 14, 14, sr)) for sr in (1, 2, 0)}

    # checkpoint ABI: state_dict keys and shapes
    meta["vlbert_state_dict"] = {}
    for cls, args in ((VisualLinguisticBert, ()), (VisualLinguisticBertForPretraining, (None, True, True, True))):
        sd = cls(ref_shim.vlbert_config(**ABI_KW), *args).state_dict()
        meta["vlbert_state_dict"][cls.__name__] = digest_json([[k, list(v.shape)] for k, v in sd.items()])
    model_zoo.load_url = lambda *a, **k: {}                  # no network: the zoo download returns no tensors
    import common.fast_rcnn
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        frcnn = common.fast_rcnn.FastRCNN(EasyDict({"NETWORK": dict(E2E_CFG)}), True, 768, True)
    meta["fastrcnn_e2e_state_dict"] = digest_json([[k, list(v.shape), str(v.dtype)] for k, v in frcnn.state_dict().items()])
    meta["fastrcnn_e2e_trainable"] = digest_json([n for n, p in frcnn.named_parameters() if p.requires_grad])

    # load_language_pretrained_model: which tensors end up where
    import tempfile
    from synth import fake_hf_checkpoint
    import common.visual_linguistic_bert as ref_mod
    meta["language_loader"] = {}
    with tempfile.TemporaryDirectory() as tmp:
        for kind in ("bert", "roberta"):
            path = os.path.join(tmp, kind + ".bin")
            torch.save(fake_hf_checkpoint(kind), path)
            for pretraining in (False, True):
                cls = ref_mod.VisualLinguisticBertForPretraining if pretraining else ref_mod.VisualLinguisticBert
                sd = cls(ref_shim.vlbert_config(**LOADER_KW), path).state_dict()
                tensors = {}
                for k in loaded_keys(list(sd), kind):
                    rows = compared_rows(k, kind, pretraining)
                    if rows != 0:
                        tensors[k] = digest(sd[k] if rows is None else sd[k][:rows])
                meta["language_loader"]["%s_%d" % (kind, pretraining)] = {"keys": digest_json(list(sd)), "sha256": tensors}

    # FastRCNN end to end with instance masks (ResNet-50, final_dim 32), CPU RoIAlign of the reference's lineage
    import common.lib.roi_pooling.roi_align as ref_roi
    fwd, bwd = ref_shim.cpu_roi_functions()
    ref_roi.C_ROIPooling.roi_align_forward, ref_roi.C_ROIPooling.roi_align_backward = fwd, bwd
    from synth import frontend_config, frontend_shapes
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = common.fast_rcnn.FastRCNN(EasyDict({"NETWORK": dict(vars(frontend_config(50).NETWORK))}), True, 32, False)
    shapes = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    assert list(shapes.items()) == list(frontend_shapes(50, 32).items())      # the test builds the weights from frontend_shapes
    sd = synth_frontend_state(shapes, 21)
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    images, boxes, box_mask, im_info, segms = masks_inputs()
    torch.set_num_threads(8)
    with torch.no_grad():
        want = ref(images=images, boxes=boxes, box_mask=box_mask, im_info=im_info, segms=segms)
    for k in ("obj_reps", "obj_reps_raw"):
        store_sampled(arrays, "masks_" + k, want[k])

    # the VQA / VCR task-module text packing and pad_sequence
    import importlib
    from make_golden_glue import _Self, glue_inputs
    vqa = importlib.import_module("vqa.modules.resnet_vlbert_for_vqa")
    vcr = importlib.import_module("vcr.modules.resnet_vlbert_for_vcr")
    from common.utils.pad_sequence import pad_sequence
    for seed in (1, 2, 3):
        q, qt, qm, a, at, am = glue_inputs(100 + seed, B=7, C=3, Lq=12, La=10)
        qt3 = qt.repeat(1, a.shape[1]).view(qt.shape[0], a.shape[1], -1)
        outs = {"vqa1": vqa.ResNetVLBERT.prepare_text_from_qa(_Self(), q, qt, qm, a[:, 1], at[:, 1], am[:, 1]),
                "vqa0": vqa.ResNetVLBERT.prepare_text_from_qa(_Self(), q, qt, qm, a[:, 0], at[:, 0], am[:, 0]),
                "qa": vcr.ResNetVLBERT.prepare_text_from_qa(_Self(), q, qt3, qm, a, at, am),
                "aq": vcr.ResNetVLBERT.prepare_text_from_aq(_Self(), q, qt3, qm, a, at, am),
                "qa_onesent": vcr.ResNetVLBERT.prepare_text_from_qa_onesent(_Self(), q, qt3, qm, a, at, am)}
        for name, ts in outs.items():
            for i, t in enumerate(ts):
                arrays["glue%d_%s_%d" % (seed, name, i)] = t.numpy()
        g = torch.Generator().manual_seed(seed)
        lengths = torch.randint(0, 6, (9,), generator=g).tolist()
        seq = torch.randn(sum(lengths), 4, generator=g)
        if max(lengths) > 0:
            arrays["glue%d_pad" % seed] = pad_sequence(seq, lengths).numpy()

    np.savez_compressed(os.path.join(GOLD, "reference_parity.npz"), **arrays)
    with open(os.path.join(GOLD, "reference_parity.json"), "w") as fh:
        json.dump(meta, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print("wrote reference_parity.npz (%d arrays) and reference_parity.json" % len(arrays))


if __name__ == "__main__":
    main()
