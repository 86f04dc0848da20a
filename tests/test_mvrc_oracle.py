"""CPU: pins the MVRC loss restatement (oracle/mvrc_oracle.py) against tests/golden/mvrc_loss.npz, which
oracle/make_golden_mvrc.py produced by executing the reference's soft_cross_entropy, its batch-first normalisation and
MVRCAccuracy.  Losses within 1e-6 relative, gradients within 1e-6 of the largest, counts exact."""
import os

import numpy as np
import pytest
import torch

import mvrc_oracle as mo


@pytest.fixture(scope="module")
def G(golden_dir):
    return np.load(os.path.join(golden_dir, "mvrc_loss.npz"))


def _loss_and_grad(G, b, bf):
    x = torch.from_numpy(G[b + "_logits"]).requires_grad_(True)
    loss = mo.soft_cross_entropy_loss(x, torch.from_numpy(G[b + "_targets"]), norm_in_batch_first=bf)
    loss.backward()
    return float(loss.detach()), x.grad.numpy()


@pytest.mark.parametrize("batch", ["a", "b"])
@pytest.mark.parametrize("bf", [False, True])
def test_loss_and_gradient_match_the_reference(G, batch, bf):
    key = "_bf" if bf else "_mean"
    loss, grad = _loss_and_grad(G, batch, bf)
    ref = float(G[batch + key])
    assert abs(loss - ref) <= 1e-6 * max(abs(ref), 1e-30) or (ref == 0.0 and loss == 0.0), (loss, ref)
    gref = G[batch + "_grad" + key]
    assert np.abs(grad - gref).max() <= 1e-6 * max(np.abs(gref).max(), 1e-30) or not gref.any() and not grad.any()


@pytest.mark.parametrize("batch", ["a", "b"])
def test_per_row_losses_and_metric_counts(G, batch):
    x, t = torch.from_numpy(G[batch + "_logits"]), torch.from_numpy(G[batch + "_targets"])
    valid = mo.valid_rows(t).view(-1)
    row = -(torch.log_softmax(x, -1) * t).sum(-1).view(-1)
    row = torch.where(valid, row, torch.zeros_like(row)).numpy()
    ref = G[batch + "_none"]
    assert np.abs(row - ref).max() <= 1e-6 * max(np.abs(ref).max(), 1e-30) or not ref.any() and not row.any()
    correct, ninst = mo.mvrc_correct(x, t)
    assert correct == int(G[batch + "_correct"]) and ninst == int(G[batch + "_ninst"])


def test_fixture_covers_the_edge_rows(G):
    s = G["a_targets"].sum(-1)
    for target in (0.0, 0.5, 0.95, 1.05, 2.0):
        assert np.isclose(s, target, atol=1e-5).any(), target
    assert not mo.valid_rows(torch.from_numpy(G["a_targets"]))[2].any()          # a sample with no valid row
    assert not mo.valid_rows(torch.from_numpy(G["b_targets"])).any()             # a batch with no valid row
    assert float(G["b_mean"]) == 0.0 and float(G["b_bf"]) == 0.0
