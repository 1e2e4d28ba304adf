"""Sparse forms of the reference's training losses (``uibk/deep_preconditioning/metrics.py``), SURVEY §8f-3.

The reference evaluates them on dense ``n x n`` tensors (``metrics.py:44-50,66-75``), which is what confines its pipeline
to n ~ 2.4 k (SURVEY D4). Here every product is the batched COO SpMV kernel (``utils.sparse_matvec_mul`` ->
``dp_coo_spmv_batch_f32``), differentiable with respect to the CNN output, so the same quantities are available at the
BASELINE sizes:

* :func:`frobenius_loss`   ``metrics.py:13-31`` - literally two ``sparse_matvec_mul`` calls and a norm; same value.
* :func:`hutchinson_trace` ``metrics.py:58-77`` - ``mean_b || L L^T v - A v ||_2`` for a random probe ``v`` per system; same
  value for the same probes (pass ``vector=``), ``A v`` formed from the stored lower triangle as ``T v + T^T v - diag(T) v``.
* :func:`inverse_loss`     ``metrics.py:34-55`` - ``mean_b || L L^T A - I ||_F``; the Frobenius norm is taken through
  probes, ``||M||_F^2 = sum_k ||M e_k||^2``: with ``probes=None`` all ``n`` unit vectors (exact, the reference's value; small
  systems), else that many Rademacher probes (an unbiased estimate of ``||M||_F^2``, Hutchinson).
``condition_loss`` (``metrics.py:80-100``, dense SVD) is out of scope; the solve-side estimate is ``spectrum.kappa_estimate``.

Under ``torch.use_deterministic_algorithms(True)`` (the reference's ``train.py`` sets it) the three losses and
:func:`system_matvec` run on the sorted-site kernels instead (``dp_llt_residual_f32`` and its gradient,
``dp_system_matvec_f32``): values and gradients are the same bits on every run, for any order of the input's sites, and a
system's term is the same alone and in a batch. That path differentiates with respect to the features of ``L`` only
(``ValueError`` if the vectors or ``T`` require grad), and refuses a repeated ``(batch, row, col)`` site or a site outside
``spatial_shape`` (``DpcgError``), which the default path accepts.
"""

from __future__ import annotations

import torch

from . import utils
from .utils import sparse_matvec_mul


def _deterministic() -> bool:
    return torch.are_deterministic_algorithms_enabled()


def _refuse_grad(what: str, *tensors) -> None:
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        raise ValueError(f"under torch.use_deterministic_algorithms the losses differentiate with respect to the features "
                         f"of L only; {what} requires grad")


class _LltLoss(torch.autograd.Function):
    """``(loss, terms)`` of ``sum_p || L L^T x_p - b_p ||`` per system (``utils.llt_residual``); the gradient reaches the
    features of ``L`` only (``utils.llt_residual_grad``)."""

    @staticmethod
    def forward(ctx, feats, sites, x, b, divisor, mean):
        loss, terms, t, r = utils.llt_residual(sites, feats, x, b, divisor, mean)
        ctx.save_for_backward(feats, x, t, r, terms)
        ctx.sites, ctx.divisor, ctx.mean = sites, divisor, mean
        ctx.mark_non_differentiable(terms)
        return loss, terms

    @staticmethod
    def backward(ctx, grad_loss, _grad_terms):
        feats, x, t, r, terms = ctx.saved_tensors
        grad = utils.llt_residual_grad(ctx.sites, feats, x, t, r, terms, grad_loss, ctx.divisor, ctx.mean)
        return grad, None, None, None, None, None


def llt_loss(lower_triangular, x: torch.Tensor, b: torch.Tensor, divisor: int = 1, mean: bool = False):
    """``(loss, terms)`` on the deterministic path: ``terms[s] = sqrt(sum_p || L L^T x[s, p] - b[s, p] ||^2 / divisor)``
    for ``x, b [B, P, N]``, ``loss`` their sum (``mean``: mean) in system order; differentiable in ``L``'s features."""
    _refuse_grad("a vector", x, b)
    sites = utils.SortedSites(lower_triangular)
    feats = utils.site_features(lower_triangular, sites.device)
    return _LltLoss.apply(feats, sites, x.detach(), b.detach(), int(divisor), bool(mean))


def _system_matvec_sorted(systems_tril, vectors: torch.Tensor) -> torch.Tensor:
    """``A v`` for ``vectors [B, P, N]`` on the sorted sites (no gradient)."""
    _refuse_grad("the system matrix or the vector", systems_tril.features, vectors)
    sites = utils.SortedSites(systems_tril)
    return utils.system_matvec_sorted(sites, utils.site_features(systems_tril, sites.device).detach(), vectors)


def frobenius_loss(lower_triangular, solution: torch.Tensor, right_hand_side: torch.Tensor) -> torch.Tensor:
    """Frobenius norm of the error, arXiv 2305.16432 eq. (11) (``metrics.py:13-31``): ``sum_b || L L^T x_b - b_b ||_2``."""
    if _deterministic():
        return llt_loss(lower_triangular, solution[:, None], right_hand_side[:, None])[0]
    interim = sparse_matvec_mul(lower_triangular, solution, transpose=True)
    interim = sparse_matvec_mul(lower_triangular, interim, transpose=False)
    return torch.linalg.vector_norm(interim - right_hand_side.to(interim.device), ord=2, dim=1).sum()


def _diagonal_part(tensor):
    """The same tensor restricted to its diagonal sites (for ``A v = T v + T^T v - diag(T) v``)."""
    keep = tensor.indices[:, 1] == tensor.indices[:, 2]
    return type(tensor)(tensor.features[keep], tensor.indices[keep], tensor.spatial_shape, tensor.batch_size)


def system_matvec(systems_tril, vector_batch: torch.Tensor) -> torch.Tensor:
    """``A v`` per batch element from the stored lower triangle ``T`` (``systems += tril(systems, -1)^T``, metrics.py:47,70)."""
    if _deterministic():
        return _system_matvec_sorted(systems_tril, vector_batch[:, None])[:, 0].to(vector_batch.device)
    return (sparse_matvec_mul(systems_tril, vector_batch, False) + sparse_matvec_mul(systems_tril, vector_batch, True)
            - sparse_matvec_mul(_diagonal_part(systems_tril), vector_batch, False))


def hutchinson_trace(systems_tril, preconditioners_tril, vector: torch.Tensor | None = None) -> torch.Tensor:
    """``mean_b || L (L^T v) - A v ||_2`` (``metrics.py:58-77``); ``vector`` ``[B, N]`` fixes the probes (default: randn)."""
    batch, dof = systems_tril.batch_size, systems_tril.spatial_shape[0]
    if vector is None:
        vector = torch.randn(batch, dof, device=systems_tril.features.device)
    if _deterministic():
        av = _system_matvec_sorted(systems_tril, vector[:, None])
        return llt_loss(preconditioners_tril, vector[:, None], av, mean=True)[0]
    interim = sparse_matvec_mul(preconditioners_tril, sparse_matvec_mul(preconditioners_tril, vector, True), False)
    interim = interim - system_matvec(systems_tril, vector)
    return torch.linalg.vector_norm(interim, ord=2, dim=1).mean()


def inverse_loss(systems_tril, preconditioners_tril, probes: int | None = None, generator=None) -> torch.Tensor:
    """``mean_b || L L^T A - I ||_F`` (``metrics.py:34-55``) without dense matrices: ``sum_k || (L L^T A - I) v_k ||^2`` over
    unit vectors (``probes=None``: exact) or ``probes`` Rademacher vectors (scaled: unbiased for the squared norm)."""
    batch, dof = systems_tril.batch_size, systems_tril.spatial_shape[0]
    device = systems_tril.features.device if systems_tril.features.is_cuda else torch.device("cuda")
    if _deterministic():
        device = systems_tril.features.device  # a CPU system is refused below, not moved
        if probes is None:
            v, divisor = torch.eye(dof, device=device).expand(batch, dof, dof), 1
        else:  # the same generator calls, in the same order, as the loop below
            v = torch.stack([torch.randint(0, 2, (batch, dof), device=device, generator=generator).float() * 2 - 1
                             for _ in range(int(probes))], dim=1)
            divisor = int(probes)
        av = _system_matvec_sorted(systems_tril, v)
        return llt_loss(preconditioners_tril, av, v, divisor, mean=True)[0]
    total = torch.zeros(batch, device=device)

    def residual(v):  # (L L^T A - I) v
        w = system_matvec(systems_tril, v)
        w = sparse_matvec_mul(preconditioners_tril, sparse_matvec_mul(preconditioners_tril, w, True), False)
        return w - v

    if probes is None:
        for k in range(dof):
            v = torch.zeros(batch, dof, device=device)
            v[:, k] = 1.0
            total = total + residual(v).square().sum(dim=1)
    else:
        for _ in range(int(probes)):
            v = torch.randint(0, 2, (batch, dof), device=device, generator=generator).float() * 2 - 1
            total = total + residual(v).square().sum(dim=1) / probes
    return total.sqrt().mean()
