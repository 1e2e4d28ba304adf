"""ORACLE — dense restatement of ``uibk/deep_preconditioning/metrics.py`` (test infrastructure), on plain tensors.

Inputs are the dense batches the reference gets from ``.dense()[:, 0]``: ``lower [B,N,N]`` (the CNN output ``L``) and
``tril [B,N,N]`` (the stored lower triangle of ``A``). Pinned to the values the reference module produced
(``tests/golden/metrics_golden.json``, ``tests/test_oracle.py::test_metrics_oracle_matches_golden``): the reference
only needs ``SparseConvTensor`` objects with ``dense()`` / ``replace_feature``, which the stand-in in
``deeppreconditioning_b200.model`` provides.
"""

from __future__ import annotations

import torch


def systems_from_tril(tril: torch.Tensor) -> torch.Tensor:
    return tril + torch.tril(tril, -1).transpose(-1, -2)  # metrics.py:46-47


def frobenius_loss(lower, solution, right_hand_side):
    """metrics.py:13-31: ``sum_b || L (L^T x) - b ||_2``."""
    interim = torch.bmm(lower.transpose(-1, -2), solution.unsqueeze(-1))
    interim = torch.bmm(lower, interim).squeeze(-1)
    return torch.linalg.vector_norm(interim - right_hand_side, ord=2, dim=1).sum()


def inverse_loss(tril, lower):
    """metrics.py:34-55: ``mean_b || L L^T A - I ||_F``."""
    preconditioners = torch.matmul(lower, lower.transpose(-1, -2))
    preconditioned = torch.matmul(preconditioners, systems_from_tril(tril))
    identity = torch.eye(tril.shape[1]).unsqueeze(0).expand((tril.shape[0], -1, -1))
    return torch.linalg.matrix_norm(preconditioned - identity).mean()


def hutchinson_trace(tril, lower, vector):
    """metrics.py:58-77 with the probe given: ``mean_b || L (L^T v) - A v ||_2``."""
    v = vector.unsqueeze(-1)
    interim = torch.bmm(lower, torch.bmm(lower.transpose(-1, -2), v))
    interim = interim - torch.bmm(systems_from_tril(tril), v)
    return torch.linalg.vector_norm(interim.squeeze(-1), ord=2, dim=1).mean()
