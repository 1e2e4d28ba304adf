"""Device path of the factor network's forward (inference only): ``libdpcg``'s sparse-convolution kernels (``dp_spconv_*``).

:class:`model.InferenceNet` is the public interface; this module holds the bindings it is built from, each usable on
its own (the tests compare every layer's pattern and values with the PyTorch module):

* :func:`sort_sites` - the input's sites as a per-(batch, row) CSR with sorted columns, plus the permutation;
* :func:`conv_rules` - output sites and per-tap source sites of a 2x2 layer (padding ``(1, 0)`` or ``(0, 1)``);
* :func:`conv_layer` - one layer's gather-GEMM, bias and activation, optionally with the final 1x1 and the output tail.
"""

from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .sparse import _workspace

MAX_CHANNELS = 64
PADDINGS_2X2 = ((1, 0), (0, 1))


def _launch(name: str, *args) -> None:
    _lib.check(getattr(_lib.lib(), name)(*args), name)


def sort_sites(indices: torch.Tensor, batch_size: int, h: int, w: int):
    """``(rowptr int32[batch_size*h + 1], col int32[nnz], perm int32[nnz])``: sites sorted by (batch, row, col), ``perm[i]``
    the input row of sorted site ``i``. Raises :class:`DpcgError` for a repeated site or one outside the image."""
    device = indices.device
    indices = indices.to(torch.int32).contiguous()
    nnz, rows = int(indices.shape[0]), int(batch_size) * int(h)
    rowptr = torch.empty(rows + 1, dtype=torch.int32, device=device)
    col = torch.empty(nnz, dtype=torch.int32, device=device)
    perm = torch.empty(nnz, dtype=torch.int32, device=device)
    flag = torch.zeros(1, dtype=torch.int32, device=device)
    lib = _lib.lib()
    ws = _workspace(lib.dp_spconv_sort_workspace_bytes(int(batch_size), int(h)), device)
    with torch.cuda.device(device):
        _launch("dp_spconv_sort_sites", _lib.ptr(indices), nnz, int(batch_size), int(h), int(w), _lib.ptr(rowptr),
                _lib.ptr(col), _lib.ptr(perm), _lib.ptr(flag), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(device))
    _lib.raise_on_flag(flag, "dp_spconv_sort_sites (a site repeats or lies outside the spatial shape)")
    return rowptr, col, perm


def conv_rules(rowptr: torch.Tensor, col: torch.Tensor, batch_size: int, h: int, w: int, padding, perm=None,
               with_indices: bool = False):
    """Pattern of a 2x2 layer on sorted sites: ``(rowptr_out, col_out, rules int32[nout, 4], indices int32[nout, 3] | None)``.

    ``rules[s, 2 ky + kx]`` is the input site of tap ``(ky, kx)`` (-1: inactive), numbered as the sorted sites or, with
    ``perm``, as ``perm`` maps them. One device synchronisation (the output count sizes the arrays)."""
    ph, pw = (int(p) for p in padding)
    device = rowptr.device
    ho = int(h) + 2 * ph - 1
    rows_out = int(batch_size) * ho
    rowptr_out = torch.empty(rows_out + 1, dtype=torch.int32, device=device)
    lib = _lib.lib()
    ws = _workspace(lib.dp_spconv_rules_workspace_bytes(int(batch_size), int(h), ph), device)
    stream = _lib.stream_ptr(device)
    with torch.cuda.device(device):
        _launch("dp_spconv_rules_count", _lib.ptr(rowptr), _lib.ptr(col), int(batch_size), int(h), int(w), ph, pw,
                _lib.ptr(rowptr_out), _lib.ptr(ws), ws.numel(), stream)
        nout = int(rowptr_out[-1].item())
        col_out = torch.empty(nout, dtype=torch.int32, device=device)
        rules = torch.empty((nout, 4), dtype=torch.int32, device=device)
        indices = torch.empty((nout, 3), dtype=torch.int32, device=device) if with_indices else None
        _launch("dp_spconv_rules_fill", _lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(perm), int(batch_size), int(h), int(w),
                ph, pw, _lib.ptr(rowptr_out), _lib.ptr(col_out), _lib.ptr(rules), _lib.ptr(indices), stream)
    return rowptr_out, col_out, rules, indices


def conv_layer(features: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor | None, src: torch.Tensor | None = None,
               nout: int | None = None, slope: torch.Tensor | None = None, head_weight: torch.Tensor | None = None,
               head_bias: torch.Tensor | None = None, indices: torch.Tensor | None = None) -> torch.Tensor:
    """One layer on the device (``dp_spconv_layer_f32``): ``weight [cout, k, k, cin]`` (spconv layout), ``src [nout, k*k]``
    the source site of every tap (``None``: a 1x1 layer in the input's own site order), ``slope`` a device scalar (PReLU
    weight / LeakyReLU slope, ``None``: no activation). ``head_weight [1, 1, 1, cout]`` applies the final 1x1 layer in the
    epilogue; ``indices`` the output tail (strict upper triangle times 0, softplus on the diagonal). Returns fp32
    ``[nout, cout]``, or ``[nout, 1]`` with a head."""
    device = features.device
    cout, ntaps, cin = weight.shape[0], weight.shape[1] * weight.shape[2], weight.shape[3]
    if nout is None:
        nout = int(src.shape[0]) if src is not None else int(features.shape[0])
    out = torch.empty((nout, 1 if head_weight is not None else cout), dtype=torch.float32, device=device)

    def param(t):
        return None if t is None else t.detach().to(torch.float32).contiguous()

    keep = [features.contiguous(), param(weight), param(bias), param(slope), param(head_weight), param(head_bias),
            None if src is None else src.contiguous(), None if indices is None else indices.to(torch.int32).contiguous()]
    feats, w, b, sl, hw, hb, src_, ind = keep
    layer = _lib.SpconvLayer(nout=nout, ntaps=ntaps, cin=cin, cout=cout, reserved=0, src=_lib.ptr(src_),
                             in_=_lib.ptr(feats), weight=_lib.ptr(w), bias=_lib.ptr(b), slope=_lib.ptr(sl),
                             head_weight=_lib.ptr(hw), head_bias=_lib.ptr(hb), indices=_lib.ptr(ind), out=_lib.ptr(out))
    with torch.cuda.device(device):
        _launch("dp_spconv_layer_f32", C.byref(layer), _lib.stream_ptr(device))
    return out
