"""CPU tests of the deterministic loss path (dp_sorted_spmv_f32, dp_system_matvec_f32, dp_llt_residual_*): argument
checks before any launch, workspace queries, empty inputs, and the choice of path from
torch.are_deterministic_algorithms_enabled()."""
import contextlib
import ctypes

import pytest
import torch

from deeppreconditioning_b200 import _lib, build, metrics, utils
from deeppreconditioning_b200 import model as models

OK, INVALID, ALIGNMENT, WORKSPACE = 0, 1, 2, 3
FAKE = 4096  # a non-null, 16-byte aligned address: never dereferenced by a call that is rejected or has nothing to do


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.lib()


@contextlib.contextmanager
def flag(enabled):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(enabled, warn_only=False)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def sites(nnz=10, nbatch=2, h=5, w=5, **overrides):
    fields = dict(nnz=nnz, nbatch=nbatch, h=h, w=w, reserved=0, features=FAKE, rowptr=FAKE, col=FAKE, perm=FAKE,
                  rowptr_t=FAKE, col_t=FAKE, perm_t=FAKE)
    fields.update(overrides)
    return _lib.FactorSites(**fields)


def spmv(lib, s, transpose=0, nvec=1, n=5, x=FAKE, y=FAKE):
    return lib.dp_sorted_spmv_f32(None if s is None else ctypes.byref(s), transpose, nvec, n, x, y, None)


def matvec(lib, s, nvec=1, n=5, v=FAKE, y=FAKE):
    return lib.dp_system_matvec_f32(None if s is None else ctypes.byref(s), nvec, n, v, y, None)


def residual(lib, s, nvec=1, n=5, divisor=1, mean=0, ptrs=FAKE, ws=FAKE, ws_bytes=1 << 30):
    return lib.dp_llt_residual_f32(None if s is None else ctypes.byref(s), nvec, n, divisor, mean, ptrs, ptrs, ptrs, ptrs,
                                   ptrs, ptrs, ws, ws_bytes, None)


def residual_grad(lib, s, nvec=1, n=5, divisor=1, mean=0, ptrs=FAKE, grad=FAKE, ws=FAKE, ws_bytes=1 << 30):
    return lib.dp_llt_residual_grad_f32(None if s is None else ctypes.byref(s), nvec, n, divisor, mean, ptrs, ptrs, ptrs,
                                        ptrs, ptrs, grad, ws, ws_bytes, None)


def test_bad_arguments_are_rejected(lib):
    for call in (spmv, matvec, residual, residual_grad):
        assert call(lib, None) == INVALID
        assert call(lib, sites(nnz=-1)) == INVALID
        assert call(lib, sites(nnz=1 << 31)) == INVALID
        assert call(lib, sites(nbatch=-1)) == INVALID
        assert call(lib, sites(h=-1)) == INVALID
        assert call(lib, sites(w=-1)) == INVALID
        assert call(lib, sites(nbatch=1 << 16, h=1 << 16)) == INVALID
        assert call(lib, sites(features=None)) == INVALID
        assert call(lib, sites(), nvec=-1) == INVALID
        assert call(lib, sites(), n=-1) == INVALID
    # the CSRs a call reads must be there
    assert spmv(lib, sites(rowptr=None)) == INVALID
    assert spmv(lib, sites(col=None)) == INVALID
    assert spmv(lib, sites(perm_t=None), transpose=1) == INVALID
    assert spmv(lib, sites(), transpose=2) == INVALID
    for call in (matvec, residual, residual_grad):
        assert call(lib, sites(rowptr_t=None)) == INVALID
        assert call(lib, sites(perm=None)) == INVALID
    assert spmv(lib, sites(), y=None) == INVALID
    assert matvec(lib, sites(), v=None) == INVALID
    for call in (residual, residual_grad):
        assert call(lib, sites(), divisor=0) == INVALID
        assert call(lib, sites(), mean=2) == INVALID
        assert call(lib, sites(), ptrs=None) == INVALID
        assert call(lib, sites(), ws=None) == INVALID
        assert call(lib, sites(), ws=FAKE + 8) == ALIGNMENT
        assert call(lib, sites(), ws_bytes=16) == WORKSPACE
    assert residual_grad(lib, sites(), grad=None) == INVALID


def test_empty_inputs_do_nothing(lib):
    for call in (spmv, matvec, residual):
        assert call(lib, sites(nbatch=0, nnz=0)) == OK
        assert call(lib, sites(), nvec=0) == OK
        assert call(lib, sites(), n=0) == OK
    # zero sites: no feature array, no columns, no gradient to write
    empty = sites(nnz=0, features=None, col=None, perm=None, col_t=None, perm_t=None)
    assert residual_grad(lib, empty, ptrs=None, grad=None, ws=None) == OK
    assert residual(lib, sites(nnz=0, nbatch=0, features=None), ptrs=None, ws=None) == OK


def test_workspace_query(lib):
    chunk = lib.dp_llt_residual_chunk_rows()
    assert chunk > 0 and chunk % 512 == 0
    for nbatch, nvec, n in ((1, 1, 81), (8, 1, 316 * 316), (3, 256, 450), (2, 1, chunk), (2, 1, chunk + 1)):
        need = lib.dp_llt_residual_workspace_bytes(nbatch, nvec, n)
        assert need % 256 == 0
        assert need >= 8 * nbatch * nvec * -(-n // chunk)  # the fp64 chunk partials of the forward
        assert need >= 2 * 4 * nbatch * nvec * n            # rho and s of the backward
    assert lib.dp_llt_residual_workspace_bytes(-1, 1, 5) == 0
    assert lib.dp_llt_residual_workspace_bytes(1, -1, 5) == 0
    assert lib.dp_llt_residual_workspace_bytes(1, 1, -5) == 0


def _tiny():
    ind = torch.tensor([[0, 0, 0], [0, 1, 0], [0, 1, 1]], dtype=torch.int32)
    return models.SparseConvTensor(torch.ones(3, 1), ind, [2, 2], 1)


def _spy(monkeypatch, module, name, result):
    calls = []

    def fake(*args, **kwargs):
        calls.append(args)
        return result(*args, **kwargs)

    monkeypatch.setattr(module, name, fake)
    return calls


def test_losses_follow_the_flag(monkeypatch):
    new = _spy(monkeypatch, metrics, "llt_loss", lambda *a: (torch.zeros(()), torch.zeros(1)))
    old = _spy(monkeypatch, metrics, "sparse_matvec_mul", lambda st, v, transpose: v)
    x, b = torch.ones(1, 2), torch.zeros(1, 2)
    metrics.frobenius_loss(_tiny(), x, b)
    assert len(old) == 2 and not new
    with flag(True):
        metrics.frobenius_loss(_tiny(), x, b)
    assert len(old) == 2 and len(new) == 1
    assert new[0][1].shape == (1, 1, 2) and new[0][2].shape == (1, 1, 2)  # one probe per system


def test_matvec_follows_the_flag(monkeypatch):
    new = _spy(monkeypatch, utils, "_deterministic_matvec", lambda st, v, transpose: v)
    with flag(True):
        utils.sparse_matvec_mul(_tiny(), torch.ones(1, 2), transpose=False)
    assert len(new) == 1
    with contextlib.suppress(RuntimeError, AssertionError):  # without a GPU the default path cannot move to the device
        utils.sparse_matvec_mul(_tiny(), torch.ones(1, 2), transpose=False)
    assert len(new) == 1


def test_cpu_tensors_raise_under_the_flag():
    x = torch.ones(1, 2)
    with flag(True):
        with pytest.raises(_lib.DpcgError):
            utils.sparse_matvec_mul(_tiny(), x, transpose=False)
        with pytest.raises(_lib.DpcgError):
            metrics.frobenius_loss(_tiny(), x, x)
        with pytest.raises(_lib.DpcgError):
            metrics.system_matvec(_tiny(), x)
        with pytest.raises(_lib.DpcgError):
            metrics.hutchinson_trace(_tiny(), _tiny(), x)
        with pytest.raises(_lib.DpcgError):
            metrics.inverse_loss(_tiny(), _tiny(), probes=2)


def test_gradients_of_vectors_or_the_system_are_refused_under_the_flag():
    x = torch.ones(1, 2)
    with flag(True):
        with pytest.raises(ValueError):
            metrics.frobenius_loss(_tiny(), x.clone().requires_grad_(True), x)
        with pytest.raises(ValueError):
            metrics.frobenius_loss(_tiny(), x, x.clone().requires_grad_(True))
        system = _tiny().replace_feature(torch.ones(3, 1, requires_grad=True))
        with pytest.raises(ValueError):
            metrics.system_matvec(system, x)
        with pytest.raises(ValueError):
            metrics.hutchinson_trace(system, _tiny(), x)
        with torch.no_grad(), pytest.raises(_lib.DpcgError):  # without autograd only the device is missing
            metrics.system_matvec(system, x)
