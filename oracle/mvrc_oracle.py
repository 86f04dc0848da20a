"""Portable restatement of the masked visual region classification (MVRC) loss and metric of the pre-training task, in fp32
torch on any device.  Pinned against the reference by tests/golden/mvrc_loss.npz (oracle/make_golden_mvrc.py)."""
import torch
import torch.nn.functional as F

VALID_EPS = 0.1        # common/utils/misc.py:132-133: a target row is valid when |sum - 1| < 0.1


def valid_rows(targets):
    """[..., C] soft targets -> bool [...] (common/utils/misc.py:133; common/metrics/pretrain_metrics.py:81)"""
    return (targets.sum(-1) - 1).abs() < VALID_EPS


def soft_cross_entropy_loss(logits, targets, norm_in_batch_first=False):
    """logits, targets [B, R, C] -> scalar loss.
    False: soft_cross_entropy(logits.view(-1, C), targets.view(-1, C)) -- mean over the valid rows of
           -sum_c t_c log_softmax(x)_c, and 0 when no row is valid (common/utils/misc.py:124-144).
    True : MVRC_LOSS_NORM_IN_BATCH_FIRST -- the per-row losses (reduction='none', 0 on invalid rows) divided by the valid rows
           of their sample + 1e-4, summed, divided by the samples with a valid row + 1e-4
           (pretrain/modules/resnet_vlbert_for_pretraining.py:191-197)."""
    B, R, C = logits.shape
    valid = valid_rows(targets)
    row = -(F.log_softmax(logits, -1) * targets).sum(-1)
    row = torch.where(valid, row, torch.zeros_like(row))
    if norm_in_batch_first:
        nv = valid.sum(1, keepdim=True).to(row.dtype)
        return (row / (nv + 1e-4)).sum() / ((nv != 0).sum().to(row.dtype) + 1e-4)
    return row.sum() / valid.sum().clamp(min=1).to(row.dtype)


def mvrc_correct(logits, targets):
    """what MVRCAccuracy.update adds to sum_metric / num_inst (common/metrics/pretrain_metrics.py:74-85): valid rows whose logit
    arg-max equals the target arg-max, and the number of valid rows"""
    C = logits.shape[-1]
    valid = valid_rows(targets).view(-1)
    x, t = logits.reshape(-1, C)[valid], targets.reshape(-1, C)[valid]
    return int((x.argmax(1) == t.argmax(1)).sum()), int(valid.sum())


def synth_targets(B, R, C, frac, generator, sums=None):
    """seeded soft targets [B, R, C]: a fraction `frac` of the regions carries a softmax row (sum 1), the rest zeros; `sums`
    optionally rescales chosen rows {(b, r): row sum}"""
    t = torch.zeros(B, R, C)
    on = torch.rand(B, R, generator=generator) < frac
    t[on] = torch.softmax(torch.randn(int(on.sum()), C, generator=generator) * 3.0, -1)
    for (b, r), s in (sums or {}).items():
        t[b, r] = torch.softmax(torch.randn(C, generator=generator) * 3.0, -1) * s
    return t
