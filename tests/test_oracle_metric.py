"""Pins oracle/oracle_metric.py against hand-computed known answers; checks the product's host-side Dice rule against the
oracle."""
import pytest
import torch

import diff_unet_amos_b200.engine as eng
from oracle import oracle_metric


def _cases():
    torch.manual_seed(5)
    a = (torch.rand(2, 3, 6, 7, 5) > 0.5).float()
    b = (torch.rand(2, 3, 6, 7, 5) > 0.4).float()
    return a, b


def test_known_answers():
    r = torch.tensor([1, 1, 0, 0, 1, 0]).float()
    l = torch.tensor([1, 0, 0, 1, 1, 0]).float()
    assert oracle_metric.dice_coeff(r, l) == pytest.approx(2 * 2 / (3 + 3))
    z = torch.zeros(6)
    assert oracle_metric.dice_coeff(z, z) == 0.0  # ZeroDivisionError branch, metric.py:44-47
    assert oracle_metric.per_class_dice(r.view(1, 1, 6), z.view(1, 1, 6)) == [1.0]  # test.py:146-147
    assert oracle_metric.per_class_dice(z.view(1, 1, 6), l.view(1, 1, 6)) == [0.0]


def test_host_rule_matches_oracle():
    a, b = _cases()
    b[:, 2] = 0  # empty label, non-empty prediction -> 1
    counts = [[int((a[:, c].bool() & b[:, c].bool()).sum()), int(a[:, c].sum()), int(b[:, c].sum())] for c in range(3)]
    assert eng.dice_from_counts(counts) == pytest.approx(oracle_metric.per_class_dice(a, b))
    assert eng.dice_from_counts([[0, 0, 0]]) == [0.0]
