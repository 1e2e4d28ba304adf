"""Drop-in for the hot-path-adjacent part of ``uibk/deep_preconditioning/utils.py``."""

from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .sparse import _workspace


def _coo_spmv(indices: torch.Tensor, feats: torch.Tensor, vec: torch.Tensor, transpose: bool) -> torch.Tensor:
    """``dp_coo_spmv_batch_f32`` on prepared device tensors (int32 ``[nnz,3]``, fp32 ``[nnz]``, fp32 ``[B,N]``)."""
    out = torch.empty_like(vec)
    with torch.cuda.device(vec.device):
        _lib.check(_lib.lib().dp_coo_spmv_batch_f32(_lib.ptr(indices), _lib.ptr(feats), indices.shape[0], vec.shape[0],
                                                    vec.shape[1], _lib.ptr(vec), int(bool(transpose)), _lib.ptr(out),
                                                    _lib.stream_ptr(vec.device)), "dp_coo_spmv_batch_f32")
    return out


def _site_products(indices, grad, vec, transpose):
    """``d/d feat[e] = grad[b_e, row_e] * vec[b_e, col_e]`` (0 for sites outside the vectors): one product per site."""
    b = indices[:, 0].long()
    r = indices[:, 2 if transpose else 1].long()
    c = indices[:, 1 if transpose else 2].long()
    inside = (r < vec.shape[1]) & (c < vec.shape[1]) & (b < vec.shape[0])
    return torch.where(inside, grad[b.clamp_max(vec.shape[0] - 1), r.clamp_max(vec.shape[1] - 1)]
                       * vec[b.clamp_max(vec.shape[0] - 1), c.clamp_max(vec.shape[1] - 1)], 0.0)


class SortedSites:
    """The sites of a batch of sparse matrices sorted by (batch, row, col) and by (batch, col, row): the row and column
    CSRs of ``dp_factor_sites_t``, each one ``dp_spconv_sort_sites`` call, made on first use. The deterministic products
    read them; they refuse a repeated ``(batch, row, col)`` site or one outside ``spatial_shape`` (:class:`DpcgError`)."""

    def __init__(self, tensor):
        if not tensor.indices.is_cuda:
            raise _lib.DpcgError("the deterministic loss products take CUDA tensors (no CPU fallback)")
        self.device = tensor.indices.device
        self.indices = tensor.indices.to(torch.int32).contiguous()
        self.batch_size = int(tensor.batch_size)
        self.h, self.w = (int(s) for s in tensor.spatial_shape)
        self._csr = {}

    def csr(self, transpose: bool):
        """``(rowptr, col, perm)`` over rows (``transpose`` False) or columns."""
        if transpose not in self._csr:
            from .spconv import sort_sites

            if transpose:
                self._csr[True] = sort_sites(self.indices[:, [0, 2, 1]], self.batch_size, self.w, self.h)
            else:
                self._csr[False] = sort_sites(self.indices, self.batch_size, self.h, self.w)
        return self._csr[transpose]

    def struct(self, feats: torch.Tensor, rows: bool = True, cols: bool = True):
        """``dp_factor_sites_t`` over ``feats`` (fp32 ``[nnz]`` on the device, kept alive by the caller)."""
        rp, cl, pm = self.csr(False) if rows else (None, None, None)
        rpt, clt, pmt = self.csr(True) if cols else (None, None, None)
        return _lib.FactorSites(nnz=int(self.indices.shape[0]), nbatch=self.batch_size, h=self.h, w=self.w, reserved=0,
                                features=_lib.ptr(feats), rowptr=_lib.ptr(rp), col=_lib.ptr(cl), perm=_lib.ptr(pm),
                                rowptr_t=_lib.ptr(rpt), col_t=_lib.ptr(clt), perm_t=_lib.ptr(pmt))


def site_features(tensor, device) -> torch.Tensor:
    """Channel 0 of a sparse tensor's features as fp32 ``[nnz]`` on ``device`` (autograd follows the conversion)."""
    feats = tensor.features.to(device=device, dtype=torch.float32)
    return (feats[:, 0] if feats.dim() == 2 else feats).contiguous()


def _batched(sites: SortedSites, vec: torch.Tensor) -> torch.Tensor:
    """``[nbatch, nvec, n]`` fp32 on the sites' device; the batch must match the sparse tensor's."""
    vec = vec.to(device=sites.device, dtype=torch.float32).contiguous()
    if vec.dim() != 3 or vec.shape[0] != sites.batch_size:
        raise ValueError(f"vectors of shape {tuple(vec.shape)} do not fit a batch of {sites.batch_size} matrices")
    return vec


def _sorted_spmv(sites: SortedSites, feats: torch.Tensor, vec: torch.Tensor, transpose: bool) -> torch.Tensor:
    """``dp_sorted_spmv_f32``: ``T x`` or ``T^T x`` for ``vec [nbatch, nvec, n]``, sequential sums in index order."""
    vec = _batched(sites, vec)
    out = torch.empty_like(vec)
    s = sites.struct(feats, rows=not transpose, cols=bool(transpose))
    with torch.cuda.device(sites.device):
        _lib.check(_lib.lib().dp_sorted_spmv_f32(C.byref(s), int(bool(transpose)), vec.shape[1], vec.shape[2],
                                                 _lib.ptr(vec), _lib.ptr(out), _lib.stream_ptr(sites.device)),
                   "dp_sorted_spmv_f32")
    return out


def system_matvec_sorted(sites: SortedSites, feats: torch.Tensor, vec: torch.Tensor) -> torch.Tensor:
    """``dp_system_matvec_f32``: ``A v = (T v + T^T v) - diag(T) v`` from the stored lower triangle, ``vec [nbatch, nvec,
    n]``."""
    vec = _batched(sites, vec)
    out = torch.empty_like(vec)
    s = sites.struct(feats)
    with torch.cuda.device(sites.device):
        _lib.check(_lib.lib().dp_system_matvec_f32(C.byref(s), vec.shape[1], vec.shape[2], _lib.ptr(vec), _lib.ptr(out),
                                                   _lib.stream_ptr(sites.device)), "dp_system_matvec_f32")
    return out


def llt_residual(sites: SortedSites, feats: torch.Tensor, x: torch.Tensor, b: torch.Tensor, divisor: int = 1,
                 mean: bool = False):
    """``dp_llt_residual_f32``: ``(loss, terms [nbatch], t, r)`` with ``t = L^T x``, ``r = L t - b`` (``[nbatch, nvec,
    n]``), ``terms[b] = sqrt(sum_p ||r_bp||^2 / divisor)`` and ``loss`` their sum (or mean) in system order."""
    x, b = _batched(sites, x), _batched(sites, b)
    if b.shape != x.shape:
        raise ValueError(f"x {tuple(x.shape)} and b {tuple(b.shape)} differ in shape")
    nbatch, nvec, n = x.shape
    t, r = torch.empty_like(x), torch.empty_like(x)
    terms = torch.zeros(nbatch, dtype=torch.float32, device=sites.device)
    loss = torch.zeros((), dtype=torch.float32, device=sites.device)
    s = sites.struct(feats)
    lib = _lib.lib()
    ws = _workspace(lib.dp_llt_residual_workspace_bytes(nbatch, nvec, n), sites.device)
    with torch.cuda.device(sites.device):
        _lib.check(lib.dp_llt_residual_f32(C.byref(s), nvec, n, int(divisor), int(bool(mean)), _lib.ptr(x), _lib.ptr(b),
                                           _lib.ptr(t), _lib.ptr(r), _lib.ptr(terms), _lib.ptr(loss), _lib.ptr(ws),
                                           ws.numel(), _lib.stream_ptr(sites.device)), "dp_llt_residual_f32")
    return loss, terms, t, r


def llt_residual_grad(sites: SortedSites, feats, x, t, r, terms, grad_loss, divisor: int = 1, mean: bool = False):
    """``dp_llt_residual_grad_f32``: the gradient of :func:`llt_residual`'s loss with respect to ``feats``, in the input's
    site order, for the upstream gradient ``grad_loss`` (a device scalar)."""
    nbatch, nvec, n = x.shape
    grad = torch.empty_like(feats)
    grad_loss = grad_loss.to(device=sites.device, dtype=torch.float32).reshape(()).contiguous()
    s = sites.struct(feats)
    lib = _lib.lib()
    ws = _workspace(lib.dp_llt_residual_workspace_bytes(nbatch, nvec, n), sites.device)
    with torch.cuda.device(sites.device):
        _lib.check(lib.dp_llt_residual_grad_f32(C.byref(s), nvec, n, int(divisor), int(bool(mean)), _lib.ptr(x),
                                                _lib.ptr(t), _lib.ptr(r), _lib.ptr(terms), _lib.ptr(grad_loss),
                                                _lib.ptr(grad), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(sites.device)),
                   "dp_llt_residual_grad_f32")
    return grad


class _SortedMatvecMul(torch.autograd.Function):
    """:class:`_SparseMatvecMul` on the sorted sites: the forward and the vector gradient are ``dp_sorted_spmv_f32``
    (the gradient is the transposed product), the feature gradient the same per-site products."""

    @staticmethod
    def forward(ctx, feats, vec, sites, transpose):
        ctx.save_for_backward(feats, vec)
        ctx.sites, ctx.transpose = sites, bool(transpose)
        return _sorted_spmv(sites, feats, vec[:, None], transpose)[:, 0]

    @staticmethod
    def backward(ctx, grad):
        feats, vec = ctx.saved_tensors
        grad = grad.contiguous()
        grad_feats = grad_vec = None
        if ctx.needs_input_grad[0]:
            grad_feats = _site_products(ctx.sites.indices, grad, vec, ctx.transpose)
        if ctx.needs_input_grad[1]:
            grad_vec = _sorted_spmv(ctx.sites, feats, grad[:, None], not ctx.transpose)[:, 0]
        return grad_feats, grad_vec, None, None


class _SparseMatvecMul(torch.autograd.Function):
    """``out[b, row] = sum feat * vec[b, col]`` with the gradients the training losses need (``metrics.py:28-29``):
    ``d/d vec`` is the transposed product (the same kernel), ``d/d feat[e] = grad[b_e, row_e] * vec[b_e, col_e]``."""

    @staticmethod
    def forward(ctx, feats, vec, indices, transpose):
        ctx.save_for_backward(feats, vec, indices)
        ctx.transpose = bool(transpose)
        return _coo_spmv(indices, feats, vec, transpose)

    @staticmethod
    def backward(ctx, grad):
        feats, vec, indices = ctx.saved_tensors
        grad = grad.contiguous()
        grad_feats = grad_vec = None
        if ctx.needs_input_grad[0]:
            grad_feats = _site_products(indices, grad, vec, ctx.transpose)
        if ctx.needs_input_grad[1]:
            grad_vec = _coo_spmv(indices, feats, grad, not ctx.transpose)
        return grad_feats, grad_vec, None, None


def sparse_matvec_mul(spconv_batch, vector_batch: torch.Tensor, transpose: bool) -> torch.Tensor:
    """Batched COO sparse matrix-vector product (utils.py:15-43), fp32, on the GPU (``dp_coo_spmv_batch_f32``).

    Differentiable with respect to the features and the vectors, like the reference's gather / ``scatter_reduce`` form
    (its callers are the training losses, ``metrics.py:28-29``).

    Args:
        spconv_batch: a batch as a ``SparseConvTensor``-like object (``features [nnz,1]``, ``indices [nnz,3]``).
        vector_batch: ``[B, N]`` vectors to multiply with the matrices.
        transpose: multiply with the transposed matrices instead.

    Under ``torch.use_deterministic_algorithms(True)`` the products run on the sorted sites (``dp_sorted_spmv_f32``):
    every output value, and the vector gradient, is a sequential sum in index order, the same bits on every run and for
    any order of the input's sites. That path refuses a repeated ``(batch, row, col)`` site and a site outside
    ``spatial_shape`` (:class:`DpcgError`; the default path accepts both), needs the sparse tensor on the GPU, and
    vectors with one row per matrix of the batch.
    """
    if torch.are_deterministic_algorithms_enabled():
        return _deterministic_matvec(spconv_batch, vector_batch, transpose)
    device = vector_batch.device if vector_batch.is_cuda else torch.device("cuda")
    indices = spconv_batch.indices.to(device=device, dtype=torch.int32).contiguous()
    feats = spconv_batch.features.to(device=device, dtype=torch.float32)
    feats = (feats[:, 0] if feats.dim() == 2 else feats).contiguous()
    vec = vector_batch.to(device=device, dtype=torch.float32).contiguous()
    if torch.is_grad_enabled() and (feats.requires_grad or vec.requires_grad):
        out = _SparseMatvecMul.apply(feats, vec, indices, bool(transpose))
    else:
        out = _coo_spmv(indices, feats.detach(), vec.detach(), transpose)
    return out if vector_batch.is_cuda else out.to(vector_batch.device)


def _deterministic_matvec(spconv_batch, vector_batch: torch.Tensor, transpose: bool) -> torch.Tensor:
    sites = SortedSites(spconv_batch)
    feats = site_features(spconv_batch, sites.device)
    vec = vector_batch.to(device=sites.device, dtype=torch.float32).contiguous()
    if torch.is_grad_enabled() and (feats.requires_grad or vec.requires_grad):
        out = _SortedMatvecMul.apply(feats, vec, sites, bool(transpose))
    else:
        out = _sorted_spmv(sites, feats.detach(), vec[:, None], transpose)[:, 0]
    return out if vector_batch.is_cuda else out.to(vector_batch.device)
