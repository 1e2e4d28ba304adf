"""Device path of the factor network: ``libdpcg``'s sparse-convolution kernels (``dp_spconv_*``), forward and backward.

:class:`model.InferenceNet` and :class:`model.TrainableNet` are the public interface; this module holds the bindings they
are built from, each usable on its own (the tests compare every layer's pattern, values and gradients with the PyTorch
module and with fp64):

* :func:`sort_sites` - the input's sites as a per-(batch, row) CSR with sorted columns, plus the permutation;
* :func:`conv_rules` - output sites and per-tap source sites of a 2x2 layer (padding ``(1, 0)`` or ``(0, 1)``);
* :func:`conv_layer` - one layer's gather-GEMM, bias and activation, optionally with the final 1x1 and the output tail;
* :func:`layer_train` - :func:`conv_layer` that also returns what the backward reads;
* :func:`invert_rules` - per tap, the output site that reads each input site;
* :func:`wgrad` - one layer's activation (or tail) backward and its weight, bias and slope gradients.
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


def _param(t):
    return None if t is None else t.detach().to(torch.float32).contiguous()


def _layer_struct(features, weight, bias, src, nout, slope, head_weight, head_bias, indices, out):
    """``(dp_spconv_layer_t, tensors it points to)``: the tensors must outlive the launch."""
    cout, ntaps, cin = weight.shape[0], weight.shape[1] * weight.shape[2], weight.shape[3]
    keep = [features.contiguous(), _param(weight), _param(bias), _param(slope), _param(head_weight), _param(head_bias),
            None if src is None else src.contiguous(), None if indices is None else indices.to(torch.int32).contiguous()]
    feats, w, b, sl, hw, hb, src_, ind = keep
    layer = _lib.SpconvLayer(nout=nout, ntaps=ntaps, cin=cin, cout=cout, reserved=0, src=_lib.ptr(src_),
                             in_=_lib.ptr(feats), weight=_lib.ptr(w), bias=_lib.ptr(b), slope=_lib.ptr(sl),
                             head_weight=_lib.ptr(hw), head_bias=_lib.ptr(hb), indices=_lib.ptr(ind), out=_lib.ptr(out))
    return layer, keep


def _nout(features, src, nout):
    if nout is not None:
        return int(nout)
    return int(src.shape[0]) if src is not None else int(features.shape[0])


def conv_layer(features: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor | None, src: torch.Tensor | None = None,
               nout: int | None = None, slope: torch.Tensor | None = None, head_weight: torch.Tensor | None = None,
               head_bias: torch.Tensor | None = None, indices: torch.Tensor | None = None) -> torch.Tensor:
    """One layer on the device (``dp_spconv_layer_f32``): ``weight [cout, k, k, cin]`` (spconv layout), ``src [nout, k*k]``
    the source site of every tap (``None``: a 1x1 layer in the input's own site order), ``slope`` a device scalar (PReLU
    weight / LeakyReLU slope, ``None``: no activation). ``head_weight [1, 1, 1, cout]`` applies the final 1x1 layer in the
    epilogue; ``indices`` the output tail (strict upper triangle times 0, softplus on the diagonal). Returns fp32
    ``[nout, cout]``, or ``[nout, 1]`` with a head."""
    device = features.device
    nout = _nout(features, src, nout)
    out = torch.empty((nout, 1 if head_weight is not None else weight.shape[0]), dtype=torch.float32, device=device)
    layer, _keep = _layer_struct(features, weight, bias, src, nout, slope, head_weight, head_bias, indices, out)
    with torch.cuda.device(device):
        _launch("dp_spconv_layer_f32", C.byref(layer), _lib.stream_ptr(device))
    return out


def layer_train(features: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor | None, src: torch.Tensor | None = None,
                nout: int | None = None, slope: torch.Tensor | None = None, head_weight: torch.Tensor | None = None,
                head_bias: torch.Tensor | None = None, indices: torch.Tensor | None = None):
    """:func:`conv_layer` as a training forward (``dp_spconv_layer_train_f32``): ``(out, pre, hidden, head_pre)``. ``out``
    is bitwise :func:`conv_layer`'s; ``pre [nout, cout]`` is the value before the activation (``None`` without one);
    with a head, ``hidden [nout, cout]`` holds the activated rows the head reads and ``head_pre [nout]`` the head's value
    before the tail; with a tail and no head, ``head_pre`` is the layer's value before it."""
    device = features.device
    nout = _nout(features, src, nout)
    cout = weight.shape[0]
    head = head_weight is not None
    out = torch.empty((nout, 1 if head else cout), dtype=torch.float32, device=device)
    pre = torch.empty((nout, cout), dtype=torch.float32, device=device) if slope is not None else None
    hidden = torch.empty((nout, cout), dtype=torch.float32, device=device) if head else None
    head_pre = torch.empty(nout, dtype=torch.float32, device=device) if (head or indices is not None) else None
    layer, _keep = _layer_struct(features, weight, bias, src, nout, slope, head_weight, head_bias, indices, out)
    with torch.cuda.device(device):
        _launch("dp_spconv_layer_train_f32", C.byref(layer), _lib.ptr(pre), _lib.ptr(hidden), _lib.ptr(head_pre),
                _lib.stream_ptr(device))
    return out, pre, hidden, head_pre


def invert_rules(rules: torch.Tensor, nin: int) -> torch.Tensor:
    """``inv int32[nin, ntaps]`` with ``inv[rules[s, t], t] = s`` and -1 where no output site reads that input site
    (``dp_spconv_rules_invert``). Raises :class:`DpcgError` when a slot is claimed twice or a source is out of range."""
    device = rules.device
    rules = rules.to(torch.int32).contiguous()
    nout, ntaps = int(rules.shape[0]), int(rules.shape[1])
    inv = torch.empty((int(nin), ntaps), dtype=torch.int32, device=device)
    flag = torch.zeros(1, dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        _launch("dp_spconv_rules_invert", _lib.ptr(rules), nout, ntaps, int(nin), _lib.ptr(inv), _lib.ptr(flag),
                _lib.stream_ptr(device))
    _lib.raise_on_flag(flag, "dp_spconv_rules_invert (two output sites read one input site through the same tap)")
    return inv


def wgrad(features: torch.Tensor, grad_out: torch.Tensor, weight_shape, src: torch.Tensor | None = None,
          pre: torch.Tensor | None = None, slope: torch.Tensor | None = None, tail_indices: torch.Tensor | None = None,
          slope_grad: bool = False):
    """Backward of one layer's activation (or, with ``tail_indices``, of the output tail) and its parameter gradients
    (``dp_spconv_wgrad_f32``): ``(grad_pre [nout, cout], grad_weight weight_shape, grad_bias [cout], grad_slope [1] |
    None)``. ``features`` is the layer's input, ``grad_out [nout, cout]`` the upstream gradient, ``pre`` what
    :func:`layer_train` kept; ``src`` as for :func:`conv_layer`. Deterministic: fixed chunks of
    ``dp_spconv_wgrad_chunk_sites()`` sites, partials added in chunk order in fp64."""
    device = grad_out.device
    cout, kh, kw, cin = (int(d) for d in weight_shape)
    ntaps = kh * kw
    grad_out = grad_out.to(torch.float32).contiguous()
    nout = int(grad_out.shape[0])
    grad_pre = torch.empty((nout, cout), dtype=torch.float32, device=device)
    grad_weight = torch.zeros((cout, kh, kw, cin), dtype=torch.float32, device=device)
    grad_bias = torch.zeros(cout, dtype=torch.float32, device=device)
    grad_slope = torch.zeros(1, dtype=torch.float32, device=device) if slope_grad else None
    keep = [features.contiguous(), None if src is None else src.contiguous(),
            None if pre is None else pre.contiguous(), _param(slope),
            None if tail_indices is None else tail_indices.to(torch.int32).contiguous()]
    feats, src_, pre_, sl, ind = keep
    lib = _lib.lib()
    ws = _workspace(lib.dp_spconv_wgrad_workspace_bytes(nout, ntaps, cin, cout), device)
    g = _lib.SpconvGrad(nout=nout, ntaps=ntaps, cin=cin, cout=cout, reserved=0, src=_lib.ptr(src_), in_=_lib.ptr(feats),
                        grad_out=_lib.ptr(grad_out), pre=_lib.ptr(pre_), slope=_lib.ptr(sl),
                        tail_indices=_lib.ptr(ind), grad_pre=_lib.ptr(grad_pre), grad_weight=_lib.ptr(grad_weight),
                        grad_bias=_lib.ptr(grad_bias), grad_slope=_lib.ptr(grad_slope))
    with torch.cuda.device(device):
        _launch("dp_spconv_wgrad_f32", C.byref(g), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(device))
    return grad_pre, grad_weight, grad_bias, grad_slope
