"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/mvrc_loss.npz by executing the UNMODIFIED reference loss and metric
(/root/reference via oracle/ref_shim.py) on seeded logits and soft targets.  Run in the build container:

    python oracle/make_golden_mvrc.py

  a_*  batch of 4 samples x 6 regions x 17 classes: valid softmax rows, all-zero rows, rows summing to 0.95 / 1.05 (valid)
       and 0.5 / 2.0 (invalid); sample 2 has no valid row
  b_*  batch with no valid row at all
  *_mean  soft_cross_entropy(x, t)                                  common/utils/misc.py:124-144 (reduction='mean')
  *_none  soft_cross_entropy(x, t, reduction='none')                common/utils/misc.py:145-148
  *_bf    the MVRC_LOSS_NORM_IN_BATCH_FIRST formula on *_none       pretrain/modules/resnet_vlbert_for_pretraining.py:191-197
  *_correct, *_ninst  MVRCAccuracy.update                          common/metrics/pretrain_metrics.py:74-85
  *_grad_mean, *_grad_bf  d loss / d logits of *_mean and *_bf
Every row sum is at least 1e-3 away from the 0.9 / 1.1 validity thresholds, so fp32 summation order cannot flip a row.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import mvrc_oracle  # noqa: E402
import ref_shim  # noqa: E402

GOLD = os.path.join(HERE, "..", "tests", "golden")
B, R, C = 4, 6, 17


def batch_a(g):
    sums = {(0, 1): 0.95, (0, 2): 1.05, (0, 3): 0.5, (0, 4): 2.0, (1, 0): 0.95, (2, 0): 0.5, (2, 1): 2.0, (3, 5): 1.05}
    t = mvrc_oracle.synth_targets(B, R, C, 0.5, g, sums)
    t[2, 2:] = 0.0                                         # sample 2: no valid row
    t[0, 5] = 0.0                                          # an all-zero row next to valid ones
    t[3, 0] = 0.0
    t[3, 0, 3] = 1.0                                       # a one-hot target
    return t


def batch_b(g):
    return mvrc_oracle.synth_targets(B, R, C, 0.0, g, {(0, 0): 0.5, (1, 3): 2.0, (3, 2): 0.85})


def main():
    ref_shim.install()
    from common.utils.misc import soft_cross_entropy
    from common.metrics.pretrain_metrics import MVRCAccuracy
    g = torch.Generator().manual_seed(2024)
    out = {}
    for name, make in (("a", batch_a), ("b", batch_b)):
        t = make(g)
        x = torch.randn(B, R, C, generator=g) * 2.0
        s = t.sum(-1)
        assert bool(((s - 0.9).abs() > 1e-3).all() and ((s - 1.1).abs() > 1e-3).all())
        out[name + "_logits"], out[name + "_targets"] = x.numpy(), t.numpy()
        xm = x.clone().requires_grad_(True)
        loss = soft_cross_entropy(xm.view(-1, C), t.view(-1, C))
        if loss.requires_grad:
            loss.backward()
            out[name + "_grad_mean"] = xm.grad.numpy()
        else:                                              # no valid row: input.new_zeros(()), no graph to the logits
            out[name + "_grad_mean"] = np.zeros((B, R, C), np.float32)
        out[name + "_mean"] = loss.detach().numpy()
        xb = x.clone().requires_grad_(True)
        none = soft_cross_entropy(xb.view(-1, C), t.view(-1, C), reduction="none")
        valid = (t.sum(-1) - 1).abs() < 1.0e-1
        # resnet_vlbert_for_pretraining.py:193-197; with no valid row `none` is the 0-dim zero and broadcasts
        none_br = none.view(B, R) if none.dim() else none
        bf = (none_br / (valid.sum(1, keepdim=True).to(dtype=none.dtype) + 1e-4)).sum() / \
            ((valid.sum(1) != 0).sum().to(dtype=none.dtype) + 1e-4)
        if bf.requires_grad:
            bf.backward()
            out[name + "_grad_bf"] = xb.grad.numpy()
        else:
            out[name + "_grad_bf"] = np.zeros((B, R, C), np.float32)
        out[name + "_none"] = (none.detach() if none.dim() else torch.zeros(B * R)).numpy()
        out[name + "_bf"] = bf.detach().numpy()
        metric = MVRCAccuracy()
        metric.update({"mvrc_logits": x, "mvrc_label": t})
        out[name + "_correct"] = np.asarray(metric.sum_metric)
        out[name + "_ninst"] = np.asarray(metric.num_inst)
    np.savez_compressed(os.path.join(GOLD, "mvrc_loss.npz"), **out)
    print("wrote mvrc_loss.npz:", {k: (v.shape, float(v.ravel()[0]) if v.size else None) for k, v in out.items()})


if __name__ == "__main__":
    main()
