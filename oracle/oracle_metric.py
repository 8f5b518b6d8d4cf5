"""CPU restatement of the evaluation metric on the inference path.  TEST INFRASTRUCTURE ONLY (oracle).

Follows the reference's ``dice_coeff`` (metric.py:3-49) and the per-class rule of ``Tester.validation_step``
(test.py:143-151).  PARITY PIN: tests/test_oracle_metric.py checks this restatement against hand-computed known answers.
"""
from __future__ import annotations

import torch


def dice_coeff(result: torch.Tensor, reference: torch.Tensor) -> float:
    """metric.py:38-47: 2 |A & B| / (|A| + |B|) on binary masks, 0.0 when both are empty."""
    inter = int(torch.sum(result.bool() & reference.bool()).item())
    s1 = int(torch.sum(result.bool()).item())
    s2 = int(torch.sum(reference.bool()).item())
    if s1 + s2 == 0:
        return 0.0
    return 2.0 * inter / float(s1 + s2)


def per_class_dice(outputs: torch.Tensor, labels: torch.Tensor) -> list:
    """test.py:143-151: outputs/labels [N, C, ...] binary; prediction non-empty and label empty -> 1."""
    res = []
    for i in range(outputs.shape[1]):
        o, l = outputs[:, i], labels[:, i]
        if o.sum() > 0 and l.sum() == 0:
            res.append(1.0)
        else:
            res.append(dice_coeff(o, l))
    return res
