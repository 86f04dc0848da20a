"""CPU.  The first test needs the reference tree (it is skipped where the tree is absent): the reference's OWN training loop --
common/trainer.py:train (:56-197: net.train(), forward, loss.mean(), backward, LR-scheduler step, clip_grad_norm_,
optimizer.step(), zero_grad, metrics.update) -- driven for several optimisation steps on
pretrain.modules.ResNetVLBERTForPretraining built from cfgs/pretrain/base_prec_4x16G_fp32.yaml (2 layers, synthetic
loader: BASELINE config 1, "plumbing"), once untouched and once after vlbert_b200.dropin.install().  The loss trajectory,
the metrics the loop accumulates and the final weights have to agree.

What is a stand-in here and why: the reference tree and a GPU are not expected on the same machine, so the two cannot meet
in one process.  The kernels are therefore replaced by the fp32 torch stand-ins of tests/cpu_shim.py (this
checks every decision of the Python layer under the real loop: train()/eval() switching, parameter registration seen by the
optimizer and by clip_grad_norm_, in-place updates of the weights the fused path caches, gradient accumulation), `to_cuda`
(common/trainer.py:42-53) is replaced by the identity, and dropout probabilities are 0 (the stand-ins have no Philox masks;
the masks are pinned on the GPU in tests/test_gpu_dropout.py).  The GPU half -- the same loop semantics on the CUDA path with
FusedAdamW against the oracle + the reference's AdamW restatement -- is tests/test_gpu_training_loop.py."""
import importlib
import os
import sys
import warnings

import pytest
import torch

import ref_shim


STEPS_PER_EPOCH, EPOCHS = 3, 2


def _loader(config, seed=3):
    g = torch.Generator().manual_seed(seed)
    B, R, T, C = 2, 4, 8, config.NETWORK.VLBERT.visual_region_classes
    batches = []
    for _ in range(STEPS_PER_EPOCH):
        x1, y1 = torch.rand(B, R, generator=g) * 300, torch.rand(B, R, generator=g) * 200
        boxes = torch.cat((torch.stack((x1, y1, x1 + 20 + torch.rand(B, R, generator=g) * 250, y1 + 20 + torch.rand(B, R, generator=g) * 150), -1),
                           torch.randn(B, R, 2048, generator=g)), -1)
        boxes[1, 3] = -2.0                                                       # pretrain/data/collate_batch.py:39
        im_info = torch.tensor([[600., 400., 1., 1., 0.], [600., 400., 1., 1., 1.]])
        text = torch.randint(1000, 30522, (B, T), generator=g)
        text[1, 6:] = 0
        rel_label = torch.randint(0, 2, (B,), generator=g)
        mlm_labels = torch.full((B, T), -1, dtype=torch.long)
        mlm_labels[0, 2], mlm_labels[1, 4] = int(text[0, 2]), int(text[1, 4])
        mvrc_ops = torch.tensor([[0, 1, 0, 0], [1, 0, 0, 0]])
        mvrc_labels = torch.zeros(B, R, C)
        mvrc_labels[mvrc_ops == 1] = torch.softmax(torch.randn(2, C, generator=g), -1)
        batches.append((None, boxes, im_info, text, rel_label, mlm_labels, mvrc_ops, mvrc_labels))

    class Loader(object):
        """what the trainer needs of a DataLoader: len() and fresh tensors on every pass (the task module writes into `boxes`)"""

        def __len__(self):
            return len(batches)

        def __iter__(self):
            for b in batches:
                yield tuple(t.clone() if torch.is_tensor(t) else t for t in b)

    return Loader()


class _Recorder(object):
    """batch_end_callback of the loop: records the loss the trainer computed for every batch"""

    def __init__(self):
        self.losses = []

    def __call__(self, p):
        self.losses.append(float(p.locals["loss"].detach()))


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present")
@pytest.mark.parametrize("accumulate", [1, 2])
def test_reference_trainer_loop_runs_identically_on_the_dropin(tmp_path, monkeypatch, capsys, accumulate):
    ref_shim.install()
    import cpu_shim
    import vlbert_b200
    vocab_dir = tmp_path / "bert-base-uncased"
    vocab_dir.mkdir()
    (vocab_dir / "vocab.txt").write_text("\n".join(["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + ["tok%d" % i for i in range(30517)]) + "\n")
    import pretrain.function.config as cfgmod
    cfgmod = importlib.reload(cfgmod)               # update_config() is not idempotent on the module-level singleton
    config = cfgmod.config
    cfgmod.update_config(os.path.join(ref_shim.REFERENCE_ROOT, "cfgs", "pretrain", "base_prec_4x16G_fp32.yaml"))
    config.NETWORK.VLBERT.num_hidden_layers = 2
    config.NETWORK.VLBERT.hidden_dropout_prob = 0.0
    config.NETWORK.VLBERT.attention_probs_dropout_prob = 0.0
    config.NETWORK.BERT_MODEL_NAME = str(vocab_dir)
    config.NETWORK.BERT_PRETRAINED = ""
    import common.fast_rcnn
    import common.trainer as trainer
    import common.visual_linguistic_bert
    import pretrain.modules.resnet_vlbert_for_pretraining as tm
    from common.metrics.composite_eval_metric import CompositeEvalMetric
    from common.metrics import pretrain_metrics
    from common.nlp.bert.optimization import AdamW, WarmupLinearSchedule
    monkeypatch.setattr(trainer, "to_cuda", lambda batch: list(batch))     # the CPU device shim of BASELINE config 1

    def fresh():
        importlib.reload(common.fast_rcnn)
        importlib.reload(common.visual_linguistic_bert)
        return importlib.reload(tm)

    def drive(model):
        """pretrain/function/train.py:139-160,318-360 in miniature: per-name weight-decay groups, AdamW, triangle schedule,
        CLIP_GRAD_NORM from the yaml, the pre-training metrics, then common.trainer.train"""
        model.image_feature_extractor.obj_downsample[0].p = 0.0
        no_decay = ("bias", "LayerNorm.weight")
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
        groups = [{"params": [p for n, p in named if not any(k in n for k in no_decay)], "weight_decay": 0.01},
                  {"params": [p for n, p in named if any(k in n for k in no_decay)], "weight_decay": 0.0}]
        opt = AdamW(groups, lr=2e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.01, correct_bias=True)
        total = EPOCHS * STEPS_PER_EPOCH // accumulate
        sched = WarmupLinearSchedule(opt, 1, t_total=total, last_epoch=-1)
        metrics = CompositeEvalMetric()
        chosen = []                                                  # pretrain/function/train.py:226-242
        if config.NETWORK.WITH_REL_LOSS:
            chosen += [pretrain_metrics.RelationshipAccuracy(), pretrain_metrics.LossLogger("relationship_loss")]
        if config.NETWORK.WITH_MLM_LOSS:
            chosen += [pretrain_metrics.MLMAccuracy(), pretrain_metrics.LossLogger("mlm_loss")]
        if config.NETWORK.WITH_MVRC_LOSS:
            chosen += [pretrain_metrics.MVRCAccuracy(), pretrain_metrics.LossLogger("mvrc_loss")]
        assert chosen
        for m in chosen:
            metrics.add(m)
        rec = _Recorder()
        import logging
        trainer.train(model, opt, sched, _loader(config), None, metrics, 0, EPOCHS, logging.getLogger("t"), rank=0,
                      batch_end_callbacks=[rec], clip_grad_norm=float(config.TRAIN.CLIP_GRAD_NORM) if config.TRAIN.CLIP_GRAD_NORM > 0 else 1.0,
                      gradient_accumulate_steps=accumulate)
        names, values = metrics.get()
        return rec.losses, dict(zip(names, values)), {k: v.detach().clone() for k, v in model.state_dict().items()}

    try:
        torch.manual_seed(0)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = fresh().ResNetVLBERTForPretraining(config)
            sd0 = {k: v.clone() for k, v in ref.state_dict().items()}
            l1, m1, w1 = drive(ref)               # the untouched reference first: install() rebinds the names its super() calls use
            assert vlbert_b200.dropin.install()
            cpu_shim.install(monkeypatch)
            cpu_shim.install_encoder(monkeypatch)
            ours = importlib.reload(tm).ResNetVLBERTForPretraining(config)
            assert isinstance(ours.vlbert, vlbert_b200.VisualLinguisticBertForPretraining)
            assert isinstance(ours.image_feature_extractor, vlbert_b200.FastRCNN)
            ours.load_state_dict(sd0, strict=True)
            l2, m2, w2 = drive(ours)
        capsys.readouterr()
        assert len(l1) == len(l2) == EPOCHS * STEPS_PER_EPOCH
        assert l1[0] != l1[-1]                                    # the loop really optimised something
        for a, b in zip(l1, l2):
            assert abs(a - b) <= 2e-4 * abs(a), (l1, l2)
        assert set(m1) == set(m2)
        for k in m1:
            assert abs(m1[k] - m2[k]) <= 1e-3 * max(1e-6, abs(m1[k])), (k, m1[k], m2[k])
        moved = 0
        for k in w1:
            if w1[k].is_floating_point():
                assert (w1[k] - w2[k]).abs().max() <= 5e-4 * w1[k].abs().max().clamp_min(1e-6), k
                moved += int(not torch.equal(w1[k], sd0[k]))
        assert moved > 20                                         # weights moved away from the initial state_dict
    finally:
        fresh()


def test_dropin_module_survives_torch_ddp_wrapper_and_the_native_reducer(monkeypatch):
    """pretrain/function/train.py:90 wraps the task module in torch.nn.parallel.DistributedDataParallel.  The drop-in must
    not break inside that wrapper (vlbert_b200.ddp.attach is the fast path, not a requirement): single-process gloo group,
    the encoder on the fp32 stand-ins, two wrapped steps give the gradients of the unwrapped module."""
    import torch.distributed as dist
    import cpu_shim
    import vlbert_b200
    import vlbert_oracle as vo
    from synth import seeded_state_dict, synth_vlbert_inputs
    cpu_shim.install_encoder(monkeypatch)
    cfg = vo.default_config(num_hidden_layers=2, vocab_size=300, max_position_embeddings=64)
    model = vlbert_b200.VisualLinguisticBert(cfg)
    model.load_state_dict(seeded_state_dict(vo.VisualLinguisticBertOracle(cfg), 5), strict=True)
    inputs = synth_vlbert_inputs(B=2, T=8, R=4, H=768, vocab=300, seed=6)

    def grads(m):
        m.zero_grad()
        out, pooled = m(*inputs, output_all_encoded_layers=False)
        (out.float().pow(2).mean() + pooled.sum()).backward()
        mod = m.module if hasattr(m, "module") else m
        return {k: p.grad.clone() for k, p in mod.named_parameters() if p.grad is not None}

    g0 = grads(model)
    dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)      # in-process store: no TCP port to collide on
    try:
        wrapped = torch.nn.parallel.DistributedDataParallel(model)
        for _ in range(2):
            g1 = grads(wrapped)
        assert set(g0) == set(g1)
        for k in g0:
            assert torch.allclose(g0[k], g1[k], rtol=1e-5, atol=1e-7), k
        assert "_rng_state" not in model.state_dict()         # the dropout state buffer is not a checkpoint key
    finally:
        dist.destroy_process_group()
