"""GPU parity of the fused masked-region-classification loss head (csrc/heads.cu soft_target_rows / soft_ce_* +
functional.MVRCLossFn) against the torch head of the same module (VisualLinguisticBertMVRCHead + soft_cross_entropy, restated
in oracle/mvrc_oracle.py and pinned to the reference by tests/golden/mvrc_loss.npz) and against the reference-generated
fixture tests/golden/vlbert_tiny_pretrain_heads.npz.  Index work (valid rows, compaction order, counts, target arg-max)
bit-exact; loss within 2e-3 (bf16 logits); gradients within 3e-2 relative L2 (the logits, hence S softmax - t, are
bf16-rounded before the GEMMs) -- the bounds of the masked-LM head."""
import os

import numpy as np
import pytest
import torch

import mvrc_oracle as mo
import vlbert_oracle as vo
from synth import synth_vlbert_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _targets(B, R, C, seed):
    """15 % soft-target rows, plus rows summing to 0.95 / 1.05 (valid) and 0.5 / 2.0 (invalid)"""
    g = torch.Generator().manual_seed(seed)
    sums = {(0, 1): 0.95, (B - 1, R - 1): 1.05, (0, 2): 0.5, (B // 2, 0): 2.0}
    return mo.synth_targets(B, R, C, 0.15, g, sums)


def _compact(t2d, cap):
    import vlbert_b200
    L = vlbert_b200._lib
    n, C = t2d.shape
    st = torch.cuda.current_stream().cuda_stream
    t = t2d.to(DEV)
    assert t.is_contiguous()
    arg = torch.full((n,), 7, dtype=torch.int64, device=DEV)
    idx = torch.full((cap,), 7, dtype=torch.int32, device=DEV)
    lab = torch.full((cap,), 7, dtype=torch.int32, device=DEV)
    cnt = torch.zeros(1, dtype=torch.int32, device=DEV)
    L.check(L.lib().vlb_soft_target_rows(t.data_ptr(), n, C, C, arg.data_ptr(), st))
    L.check(L.lib().vlb_label_compact(arg.data_ptr(), n, -1, idx.data_ptr(), lab.data_ptr(), cap, cnt.data_ptr(), st))
    return arg.cpu(), idx.cpu(), lab.cpu(), int(cnt)


def test_valid_rows_and_compaction_are_exact(golden_dir):
    G = np.load(os.path.join(golden_dir, "mvrc_loss.npz"))
    cases = [torch.from_numpy(G["a_targets"]).view(-1, 17), torch.from_numpy(G["b_targets"]).view(-1, 17),
             _targets(64, 100, 1601, 3).view(-1, 1601)]
    for t in cases:
        valid = mo.valid_rows(t)
        pos = valid.nonzero().flatten()
        am = t.argmax(1)
        for cap in sorted({max(1, pos.numel() // 2), max(1, pos.numel()), pos.numel() + 40}):
            arg, idx, lab, cnt = _compact(t, cap)
            assert torch.equal(arg, torch.where(valid, am, torch.full_like(am, -1)))
            assert cnt == pos.numel()
            k = min(cap, pos.numel())
            assert torch.equal(idx[:k].long(), pos[:k]) and torch.equal(lab[:k].long(), am[pos[:k]])
            assert bool((idx[k:] == -1).all()) and bool((lab[k:] == -1).all())


def test_target_rows_at_any_alignment():
    """row stride of C = 1601 fp32 leaves every row at a different 4-byte offset; an offset base pointer shifts them again"""
    t = _targets(4, 40, 1601, 4).view(-1, 1601)
    t[3, 1600] = 5.0                                     # a maximum in the tail
    t[5, 0] = 5.0                                        # ... and in the head
    t[3] /= t[3].sum()
    t[5] /= t[5].sum()
    buf = torch.zeros(t.numel() + 3, device=DEV)
    for off in range(4):
        arg, _, _, _ = _compact(buf[off: off + t.numel()].copy_(t.view(-1).to(DEV)).view_as(t), 8)
        assert torch.equal(arg, torch.where(mo.valid_rows(t), t.argmax(1), torch.full((t.shape[0],), -1)))


def _build(B, R, H, C, seed):
    import vlbert_b200
    cfg = vo.default_config(vocab_size=200, hidden_size=H, num_hidden_layers=1, num_attention_heads=max(1, H // 64),
                            intermediate_size=2 * H, max_position_embeddings=128, visual_size=H, visual_region_classes=C)
    torch.manual_seed(seed)
    m = vlbert_b200.VisualLinguisticBertForPretraining(cfg, None, False, False, True).to(DEV)
    with torch.no_grad():
        m.mvrc_head.transform.dense.bias.normal_(0, 0.02)
        m.mvrc_head.region_cls_pred.bias.normal_(0, 0.02)
    return m


def _torch_reference(m, object_out, targets, bf):
    o = object_out.clone().requires_grad_(True)
    logits = m.mvrc_head(o)
    loss = mo.soft_cross_entropy_loss(logits, targets, norm_in_batch_first=bf)
    m.zero_grad()
    loss.backward()
    grads = {k: p.grad.clone() for k, p in m.named_parameters() if k.startswith("mvrc_head")}
    return float(loss.detach()), grads, o.grad, mo.mvrc_correct(logits.detach(), targets)[0]


def _fused(m, object_out, targets, bf, max_valid):
    o = object_out.clone().requires_grad_(True)
    m.zero_grad()
    loss, correct, count = m.mvrc_loss(o, targets, max_valid=max_valid, norm_in_batch_first=bf)
    (loss * 1.0).backward()
    grads = {k: p.grad.clone() for k, p in m.named_parameters() if k.startswith("mvrc_head")}
    return float(loss.detach()), grads, o.grad, int(correct), int(count)


@pytest.mark.parametrize("shape", [(3, 5, 128, 17), (64, 100, 768, 1601)])
@pytest.mark.parametrize("bf", [False, True])
@pytest.mark.parametrize("hint", [False, True])
def test_fused_mvrc_loss_against_the_torch_head(shape, bf, hint):
    B, R, H, C = shape
    m = _build(B, R, H, C, 5)
    g = torch.Generator().manual_seed(6)
    object_out = torch.randn(B, R, H, generator=g).to(DEV)
    targets = _targets(B, R, C, 7).to(DEV)
    if B * R < 64:
        targets[1, 3] = torch.softmax(torch.randn(C, generator=g), -1).to(DEV)   # at least a few valid rows at the tiny shape
    valid = mo.valid_rows(targets).view(-1)
    loss_ref, g_ref, o_ref, acc_ref = _torch_reference(m, object_out, targets, bf)
    loss, grads, o_grad, correct, count = _fused(m, object_out, targets, bf, B * R if hint else None)
    assert count == int(valid.sum())
    assert abs(loss - loss_ref) <= 2e-3 * abs(loss_ref), (loss, loss_ref)
    assert abs(correct - acc_ref) <= max(1, int(0.02 * count))
    errs = {k: rel(grads[k], g_ref[k]) for k in g_ref}
    errs["object_out"] = rel(o_grad, o_ref)
    print("fused MVRC loss %s bf=%s hint=%s: loss %.6f (ref %.6f) correct %d (ref %d) grad errors %s" % (
        shape, bf, hint, loss, loss_ref, correct, acc_ref, {k: "%.2e" % v for k, v in errs.items()}))
    assert all(v <= 3e-2 for v in errs.values()), errs
    assert bool((o_grad.view(-1, H)[~valid] == 0).all())                          # invalid regions get no gradient


def test_fused_mvrc_loss_against_the_reference_fixture(golden_dir):
    """the reference's own mvrc logits (tests/golden/vlbert_tiny_pretrain_heads.npz) -> soft cross-entropy on the host, against
    the fused loss computed from the library encoder's object output with the fixture's weights"""
    import vlbert_b200
    G = np.load(os.path.join(golden_dir, "vlbert_tiny_pretrain_heads.npz"))
    cfg = vo.default_config(vocab_size=200, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256,
                            max_position_embeddings=64, visual_size=128, visual_region_classes=17, pos_embedding_frozen=False)
    model = vlbert_b200.VisualLinguisticBertForPretraining(cfg, None, True, True, True).to(DEV)
    model.load_state_dict({k[3:]: torch.from_numpy(G[k]) for k in G.files if k.startswith("sd.")}, strict=True)
    inputs = [t.to(DEV) for t in synth_vlbert_inputs(B=3, T=9, R=5, H=128, vocab=200, seed=62)]
    with torch.no_grad():
        _, object_out, _ = vlbert_b200.VisualLinguisticBert.forward(model, *inputs, output_all_encoded_layers=False,
                                                                    output_text_and_object_separately=True)
    ref_logits = torch.from_numpy(G["mvrc"])
    g = torch.Generator().manual_seed(9)
    targets = mo.synth_targets(3, 5, 17, 0.5, g, {(2, 4): 1.05, (1, 1): 0.5})
    targets[1, 0] = torch.softmax(torch.randn(17, generator=g), -1)
    targets *= inputs[5].cpu().unsqueeze(-1)              # no target on a padding region slot
    for bf in (False, True):
        loss_ref = float(mo.soft_cross_entropy_loss(ref_logits, targets, norm_in_batch_first=bf))
        loss, correct, count = model.mvrc_loss(object_out, targets.to(DEV), norm_in_batch_first=bf)
        assert int(count) == int(mo.valid_rows(targets).sum())
        assert abs(float(loss) - loss_ref) <= 1e-2 * abs(loss_ref), (bf, float(loss), loss_ref)


@pytest.mark.parametrize("bf", [False, True])
def test_no_valid_row_gives_zero_loss_and_gradients(bf):
    B, R, H, C = 4, 6, 128, 17
    m = _build(B, R, H, C, 8)
    g = torch.Generator().manual_seed(10)
    object_out = torch.randn(B, R, H, generator=g).to(DEV)
    targets = mo.synth_targets(B, R, C, 0.0, g, {(0, 0): 0.5, (1, 2): 2.0}).to(DEV)
    for hint in (None, 16):
        loss, grads, o_grad, correct, count = _fused(m, object_out, targets, bf, hint)
        assert loss == 0.0 and correct == 0 and count == 0
        assert bool((o_grad == 0).all()) and all(bool((v == 0).all()) for v in grads.values())


@pytest.mark.parametrize("bf", [False, True])
def test_overflow_normalises_by_the_rows_used(bf):
    """max_valid below the number of valid rows: the first max_valid rows (ascending) enter the loss, normalised by the rows
    used (per sample in batch-first mode), and n_valid reports the true count"""
    B, R, H, C = 4, 10, 128, 17
    m = _build(B, R, H, C, 11)
    g = torch.Generator().manual_seed(12)
    object_out = torch.randn(B, R, H, generator=g).to(DEV)
    targets = mo.synth_targets(B, R, C, 0.6, g).to(DEV)
    valid = mo.valid_rows(targets).view(-1)
    pos = valid.nonzero().flatten()
    cap = 8
    assert pos.numel() > cap + 4
    used = torch.zeros_like(valid)
    used[pos[:cap]] = True
    t_used = targets * used.view(B, R, 1)                 # the rows beyond the first `cap` made invalid (all-zero)
    loss_ref, g_ref, o_ref, _ = _torch_reference(m, object_out, t_used, bf)
    loss, grads, o_grad, _, count = _fused(m, object_out, targets, bf, cap)
    assert count == pos.numel()
    assert abs(loss - loss_ref) <= 2e-3 * abs(loss_ref), (loss, loss_ref)
    errs = {k: rel(grads[k], g_ref[k]) for k in g_ref}
    errs["object_out"] = rel(o_grad, o_ref)
    assert all(v <= 3e-2 for v in errs.values()), errs
    assert bool((o_grad.view(-1, H)[~used] == 0).all())


def test_static_max_valid_is_sync_free():
    B, R, H, C = 8, 36, 256, 1601
    m = _build(B, R, H, C, 13)
    g = torch.Generator().manual_seed(14)
    object_out = torch.randn(B, R, H, generator=g).to(DEV).requires_grad_(True)
    targets = _targets(B, R, C, 15).to(DEV)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for bf in (False, True):
            loss, correct, count = m.mvrc_loss(object_out, targets, max_valid=B * R, norm_in_batch_first=bf)
            loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(loss).all() and int(count) == int(mo.valid_rows(targets).sum())


def test_pretraining_objective_in_a_cuda_graph():
    """mlm_loss + mvrc_loss with static bounds captured in GraphedStep and replayed on two label batches: the loss and every
    gradient equal those of eager steps on the same batches (dropout off)"""
    import vlbert_b200
    B, T, R, H, V, C = 4, 12, 8, 128, 200, 17
    cfg = vo.default_config(vocab_size=V, hidden_size=H, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256,
                            max_position_embeddings=64, visual_size=H, visual_region_classes=C, hidden_dropout_prob=0.0,
                            attention_probs_dropout_prob=0.0)
    torch.manual_seed(16)
    model = vlbert_b200.VisualLinguisticBertForPretraining(cfg, None, False, True, True).to(DEV)
    model.train()
    model.max_length_hint = T + R + 1

    def loss_fn(m, ids, types, tvis, tmask, ovl, omask, mlm_labels, mvrc_labels):
        text_out, object_out, _ = vlbert_b200.VisualLinguisticBert.forward(m, ids, types, tvis, tmask, ovl, omask,
                                                                           output_all_encoded_layers=False,
                                                                           output_text_and_object_separately=True)
        l_mlm, _, _ = m.mlm_loss(text_out, mlm_labels, max_labelled=B * T)
        l_mvrc, _, _ = m.mvrc_loss(object_out, mvrc_labels, max_valid=B * R)
        return l_mlm + l_mvrc

    def batch(seed):
        g = torch.Generator().manual_seed(seed)
        ins = list(synth_vlbert_inputs(B=B, T=T, R=R, H=H, vocab=V, seed=seed, ragged=False))
        mlm = torch.where(torch.rand(B, T, generator=g) < 0.3, torch.randint(0, V, (B, T), generator=g), torch.full((B, T), -1))
        return [t.to(DEV) for t in ins + [mlm, mo.synth_targets(B, R, C, 0.3, g)]]

    b1, b2 = batch(21), batch(22)
    eager = []
    for b in (b1, b2):
        model.zero_grad(set_to_none=True)
        loss = loss_fn(model, *b)
        loss.backward()
        eager.append((float(loss.detach()), {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}))
        del loss                                          # no autograd node of the eager steps may outlive them into the capture
    step = vlbert_b200.GraphedStep(model, loss_fn, b1)
    for b, (l_e, g_e) in zip((b2, b1), (eager[1], eager[0])):
        loss = float(step(*b))
        assert abs(loss - l_e) <= 1e-5 * abs(l_e), (loss, l_e)
        for k, ge in g_e.items():
            if k.endswith("attention.self.key.bias"):     # exactly zero in exact arithmetic (softmax shift invariance)
                continue
            p = dict(model.named_parameters())[k]
            assert rel(p.grad, ge) <= 1e-5, k
