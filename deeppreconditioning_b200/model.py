"""spconv-free stand-ins for the CNN side of the path (input producers, not the optimisation target).

The reference builds its factor ``L`` with ``spconv`` (``uibk/deep_preconditioning/model.py:13-59``),
a CUDA-12.4 wheel that does not exist in this image. ``north_star`` keeps the CNN forward in PyTorch, so
this module provides

* :class:`SparseConvTensor` — the four fields of ``spconv.pytorch.SparseConvTensor`` the hot path touches
  (``features``, ``indices``, ``spatial_shape``, ``batch_size``) plus ``dense()`` / ``replace_feature``;
* :class:`SparseConv2d` — regular (pattern-dilating) sparse convolution, stride 1, in plain PyTorch
  (gather - GEMM - scatter over coordinate keys);
* :class:`PreconditionerNet` — same layer stack and the same output post-processing as the reference
  (``model.py:27-40`` and ``model.py:53-57``): strict upper triangle zeroed *by value*, softplus on the diagonal.

Weights are random-init (the checkpoint ``best.pt`` is not shipped), so values are "parity unpinned"
against spconv; what is pinned are the structural properties the reference tests
(``tests/test_model.py:31-42``): non-zero diagonal, zero strict upper triangle, ``L @ L.T`` SPD.
"""

from __future__ import annotations

import torch
from torch import nn
from torch.autograd.function import once_differentiable


class SparseConvTensor:
    """Minimal ``spconv.pytorch.SparseConvTensor``: COO sites ``(batch, row, col)`` with channel features."""

    def __init__(self, features: torch.Tensor, indices: torch.Tensor, spatial_shape, batch_size: int) -> None:
        assert features.dim() == 2 and indices.dim() == 2 and indices.shape[1] == 3
        assert features.shape[0] == indices.shape[0]
        self.features = features
        self.indices = indices
        self.spatial_shape = list(spatial_shape)
        self.batch_size = int(batch_size)

    def replace_feature(self, features: torch.Tensor) -> "SparseConvTensor":
        return SparseConvTensor(features, self.indices, self.spatial_shape, self.batch_size)

    def dense(self) -> torch.Tensor:
        """``[B, C, H, W]`` like spconv's ``dense()`` (channels first). O(B*H*W): small systems only."""
        h, w = self.spatial_shape
        c = self.features.shape[1]
        out = torch.zeros(self.batch_size, h, w, c, dtype=self.features.dtype, device=self.features.device)
        idx = self.indices.long()
        out[idx[:, 0], idx[:, 1], idx[:, 2]] = self.features
        return out.permute(0, 3, 1, 2).contiguous()

    @classmethod
    def from_dense(cls, x: torch.Tensor) -> "SparseConvTensor":
        """From ``[B, H, W, C]`` (the layout ``SparseConvTensor.from_dense`` takes, ``tests/test_model.py:22``)."""
        mask = (x != 0).any(dim=-1)
        idx = mask.nonzero()
        return cls(x[mask], idx.int(), list(x.shape[1:3]), x.shape[0])


class SparseConv2d(nn.Module):
    """Regular sparse convolution (stride 1): an output site is active iff its window holds an active input.

    ``out[y, x] = bias + sum_{ky,kx} in[y + ky - ph, x + kx - pw] @ W[:, ky, kx, :].T`` - the dense ``conv2d``
    (cross-correlation) restricted to the active output sites (``tests/test_host.py::test_sparse_conv_is_the_dense_conv``).
    Output spatial shape is ``(H + 2*ph - k + 1, W + 2*pw - k + 1)``. ``weight`` has spconv 2.x's layout
    ``[out, k, k, in]`` and the parameter names are spconv's (``weight``, ``bias``), so a state dict saved from the
    reference's ``spconv.SparseConv2d`` layers loads unchanged (``test.py:216``).
    """

    def __init__(self, in_channels: int, out_channels: int, kernel_size: int, padding=(0, 0), bias: bool = True) -> None:
        super().__init__()
        self.k = int(kernel_size)
        self.padding = (padding, padding) if isinstance(padding, int) else tuple(padding)
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None
        fan_in = in_channels * self.k * self.k
        bound = (1.0 / fan_in) ** 0.5
        # drawn in (k, k, in, out) order, stored in spconv's [out, k, k, in]: the random-init factors of the committed
        # golden vectors (tests/golden) were made with this draw order
        drawn = nn.init.uniform_(torch.empty(self.k, self.k, in_channels, out_channels), -bound * 3**0.5, bound * 3**0.5)
        self.weight = nn.Parameter(drawn.permute(3, 0, 1, 2).contiguous())
        if bias:
            nn.init.uniform_(self.bias, -bound, bound)

    def forward(self, x: SparseConvTensor) -> SparseConvTensor:
        k, (ph, pw) = self.k, self.padding
        h, w = x.spatial_shape
        ho, wo = h + 2 * ph - k + 1, w + 2 * pw - k + 1
        if k == 1 and ph == 0 and pw == 0:
            out = x.features @ self.weight[:, 0, 0, :].t()
            if self.bias is not None:
                out = out + self.bias
            return SparseConvTensor(out, x.indices, [ho, wo], x.batch_size)
        b, r, c = (x.indices[:, i].long() for i in range(3))
        keys, srcs, taps = [], [], []
        for ky in range(k):
            for kx in range(k):
                ro, co = r - ky + ph, c - kx + pw
                ok = (ro >= 0) & (ro < ho) & (co >= 0) & (co < wo)
                keys.append(((b * ho + ro) * wo + co)[ok])
                srcs.append(ok.nonzero().squeeze(1))
                taps.append((ky, kx))
        uniq, inverse = torch.unique(torch.cat(keys), return_inverse=True)
        out = x.features.new_zeros(uniq.shape[0], self.weight.shape[0])
        start = 0
        for key, src, (ky, kx) in zip(keys, srcs, taps):
            dst = inverse[start:start + key.shape[0]]
            start += key.shape[0]
            out.index_add_(0, dst, x.features[src] @ self.weight[:, ky, kx, :].t())
        if self.bias is not None:
            out = out + self.bias
        indices = torch.stack((uniq // (ho * wo), (uniq // wo) % ho, uniq % wo), dim=1).int()
        return SparseConvTensor(out, indices, [ho, wo], x.batch_size)


class PReLU(nn.PReLU):
    """``nn.PReLU`` on the features of a sparse tensor. A subclass, not a wrapper: inside ``nn.Sequential`` its parameter is
    ``layers.N.weight`` exactly as in the reference's ``spconv.SparseSequential(..., nn.PReLU())`` (``model.py:27-37``)."""

    def forward(self, x: SparseConvTensor) -> SparseConvTensor:  # type: ignore[override]
        return x.replace_feature(super().forward(x.features))


class LeakyReLU(nn.LeakyReLU):
    def forward(self, x: SparseConvTensor) -> SparseConvTensor:  # type: ignore[override]
        return x.replace_feature(super().forward(x.features))


def _lower_triangular_tail(interim: SparseConvTensor) -> SparseConvTensor:
    """The output post-processing of ``model.py:53-57`` / ``model.py:173-177``."""
    feats = interim.features.clone()
    upper = interim.indices[:, 1] < interim.indices[:, 2]  # (batch, row, col)
    feats[upper] = feats[upper] * 0  # make the matrix lower triangular (by value, sites stay active)
    diag = interim.indices[:, 1] == interim.indices[:, 2]
    feats[diag] = nn.functional.softplus(feats[diag])  # enforce positive diagonal
    return interim.replace_feature(feats)


class PreconditionerNet(nn.Module):
    """Fully convolutional network mapping ``tril(A)`` to a lower-triangular ``L`` (``model.py:13-59``).

    Same module tree as the reference (``self.layers``: conv, PReLU, 4 x (2x2 conv, PReLU), conv), hence the same
    ``state_dict`` keys and tensor shapes: ``load_state_dict(torch.load("best.pt"))`` of a reference checkpoint works
    (``test.py:216``; ``tests/test_host.py::test_reference_checkpoint_layout_loads``)."""

    def __init__(self, channels: list[int]) -> None:
        super().__init__()
        assert len(channels) % 2
        layers: list[nn.Module] = [SparseConv2d(channels[0], channels[1], 1), PReLU()]
        for index, (cin, cout) in enumerate(zip(channels[1:-2], channels[2:-1], strict=True)):
            padding = (1, 0) if index < (len(channels) - 2) // 2 else (0, 1)
            layers += [SparseConv2d(cin, cout, 2, padding=padding), PReLU()]
        layers.append(SparseConv2d(channels[-2], channels[-1], 1))
        self.layers = nn.Sequential(*layers)

    def forward(self, input_: SparseConvTensor) -> SparseConvTensor:
        return _lower_triangular_tail(self.layers(input_))


class PreconditionerTrilNet(nn.Module):
    """Pattern-preserving variant: 1x1 convolutions only, so ``L`` keeps ``tril(A)``'s sparsity.

    Stands in for the submanifold ``PreconditionerSparseUNet`` (``model.py:62-179``, first/last layers share
    ``indice_key="subm1"``), whose output pattern equals its input pattern; the U-Net body itself is out of scope.
    """

    def __init__(self, channels: list[int]) -> None:
        super().__init__()
        layers: list[nn.Module] = []
        for cin, cout in zip(channels[:-2], channels[1:-1], strict=True):
            layers += [SparseConv2d(cin, cout, 1), LeakyReLU()]
        layers.append(SparseConv2d(channels[-2], channels[-1], 1))
        self.layers = nn.Sequential(*layers)

    def forward(self, input_: SparseConvTensor) -> SparseConvTensor:
        return _lower_triangular_tail(self.layers(input_))


DEFAULT_CHANNELS = [1, 16, 32, 64, 32, 16, 1]  # params.yaml:6-13


class InferenceNet:
    """Inference-only forward of a :class:`PreconditionerNet` or :class:`PreconditionerTrilNet` on ``libdpcg``'s sparse
    convolution kernels (``dp_spconv_*``, sm_100a): site sort, per-row rule merge of the 2x2 layers, one gather-GEMM
    launch per layer with bias and activation in its epilogue, and the final 1x1 layer and output tail fused into the
    layer before it.

    The module's contract: ``SparseConvTensor -> SparseConvTensor`` for any ``batch_size``, same ``indices`` (sorted by
    (batch, row, col) after a 2x2 layer, the input's own order for an all-1x1 network), ``spatial_shape`` and
    ``batch_size`` as ``net(input)``, features fp32 ``[nnz, 1]``. CUDA tensors only, no autograd. The values are the fp32
    forward in a fixed summation order (one fma chain per tap, taps added in (ky, kx) order, bias last), so they do not
    depend on the batch a system is in. The parameters are read at every call: a later ``load_state_dict`` applies.
    Usable wherever the module is called, e.g. ``BenchmarkSuite(data_set, InferenceNet(net))``.

    Supported (checked here, without a GPU; anything else raises ``ValueError``): layers ``SparseConv2d`` with
    ``kernel_size`` 1 (no padding) or 2 (padding ``(1, 0)`` or ``(0, 1)``) and 1..64 channels, each but the last
    followed by at most one scalar ``PReLU`` / ``LeakyReLU``, the last with one output channel.
    """

    def __init__(self, net: nn.Module) -> None:
        if not isinstance(net, (PreconditionerNet, PreconditionerTrilNet)):
            raise ValueError(f"InferenceNet runs PreconditionerNet or PreconditionerTrilNet, not {type(net).__name__}")
        steps: list[list] = []
        for layer in net.layers:
            if isinstance(layer, SparseConv2d):
                _check_conv(layer)
                if steps and steps[-1][0].weight.shape[0] != layer.weight.shape[3]:
                    raise ValueError("consecutive layers disagree on the channel count")
                steps.append([layer, None])
            elif isinstance(layer, (PReLU, LeakyReLU)):
                if not steps or steps[-1][1] is not None:
                    raise ValueError("an activation must follow a convolution")
                if isinstance(layer, PReLU) and layer.weight.numel() != 1:
                    raise ValueError("only a scalar PReLU (num_parameters=1) is supported")
                steps[-1][1] = layer
            else:
                raise ValueError(f"unsupported layer {type(layer).__name__}")
        if not steps or steps[-1][1] is not None or steps[-1][0].weight.shape[0] != 1:
            raise ValueError("the network must end with a convolution to one channel")
        self.net = net
        self.steps = [tuple(s) for s in steps]
        self._slopes: dict = {}

    def _slope(self, act, device) -> torch.Tensor | None:
        if act is None:
            return None
        if isinstance(act, PReLU):
            return act.weight
        key = (float(act.negative_slope), device)
        if key not in self._slopes:
            self._slopes[key] = torch.tensor([key[0]], dtype=torch.float32, device=device)
        return self._slopes[key]

    def _check_input(self, input_: SparseConvTensor) -> torch.device:
        from . import _lib

        feats, indices = input_.features, input_.indices
        if not (feats.is_cuda and indices.is_cuda):
            raise _lib.DpcgError(f"{type(self).__name__} runs on CUDA tensors only (no CPU fallback)")
        if feats.dtype != torch.float32 or feats.dim() != 2 or feats.shape[1] != self.steps[0][0].weight.shape[3]:
            raise _lib.DpcgError(f"{type(self).__name__} needs fp32 features [nnz, {self.steps[0][0].weight.shape[3]}]")
        device = feats.device
        for conv, act in self.steps:
            for p in [conv.weight, conv.bias] + ([act.weight] if isinstance(act, PReLU) else []):
                if p is not None and p.device != device:
                    raise _lib.DpcgError(f"{type(self).__name__}: the network's parameters are not on the input's device")
        return device

    def _plan(self, input_: SparseConvTensor):
        """The launches of a forward: ``(layers, out_indices, spatial_shape)``, ``layers`` a list of ``(conv, act, rules
        or None, head or None)``: one launch each, the final 1x1 fused as ``head`` into the last. All patterns are built
        here, before the first GEMM (their sizes are read back once per 2x2 layer)."""
        from . import spconv

        indices = input_.indices
        batch, (h, w) = input_.batch_size, input_.spatial_shape
        rules: dict[int, torch.Tensor] = {}
        out_indices = indices
        last_k2 = max((i for i, (conv, _) in enumerate(self.steps) if conv.k == 2), default=None)
        if last_k2 is not None:
            rowptr, col, perm = spconv.sort_sites(indices, batch, h, w)
            for i, (conv, _) in enumerate(self.steps):
                if conv.k == 2:
                    rowptr, col, rules[i], ind = spconv.conv_rules(rowptr, col, batch, h, w, conv.padding, perm,
                                                                   with_indices=i == last_k2)
                    perm = None  # later layers read features in sorted site order
                    if ind is not None:
                        out_indices = ind
                h, w = h + 2 * conv.padding[0] - conv.k + 1, w + 2 * conv.padding[1] - conv.k + 1
        steps = self.steps
        head = None
        if len(steps) > 1 and steps[-1][0].k == 1:
            head, steps = steps[-1][0], steps[:-1]
        layers = [(conv, act, rules.get(i), head if i == len(steps) - 1 else None) for i, (conv, act) in enumerate(steps)]
        return layers, out_indices, [h, w]

    def __call__(self, input_: SparseConvTensor) -> SparseConvTensor:
        from . import spconv

        device = self._check_input(input_)
        layers, out_indices, shape = self._plan(input_)
        x = input_.features
        for i, (conv, act, src, head) in enumerate(layers):
            last = i == len(layers) - 1
            nout = int(src.shape[0]) if src is not None else int(x.shape[0])
            x = spconv.conv_layer(x, conv.weight, conv.bias, src, nout, self._slope(act, device),
                                  head.weight if head is not None else None, head.bias if head is not None else None,
                                  out_indices if last else None)
        return SparseConvTensor(x, out_indices, shape, input_.batch_size)


class TrainableNet(InferenceNet):
    """:class:`InferenceNet` with a backward on the device kernels: training of the factor network without the PyTorch
    layers.

    When autograd is enabled and a parameter of ``net`` requires grad, the call runs a ``torch.autograd.Function``: the
    training forward (``dp_spconv_layer_train_f32``, output bitwise :class:`InferenceNet`'s) keeps every layer's input,
    its value before the activation, the fused head's input and value before the tail, and each 2x2 layer's inverse
    rules; its backward walks the layers in reverse, one weight-gradient launch (``dp_spconv_wgrad_f32``) and one
    input-gradient launch (the forward kernel on the transposed weights and inverse rules) per layer. Gradients go to
    ``net``'s own parameters (conv weights, biases, PReLU weights), so ``loss.backward()`` accumulates into their
    ``.grad`` and ``torch.optim.*(net.parameters())`` works unchanged. They are deterministic: the same bits on every
    run, and a system's input gradient at every layer does not depend on its batch.

    Otherwise (``torch.no_grad()``, or no parameter requires grad) the call is exactly :class:`InferenceNet`'s. Input
    features that require grad raise ``ValueError``: the first layer's input gradient is not computed.
    """

    def _parameters(self) -> list:
        params = []
        for conv, act in self.steps:
            params += [conv.weight] + ([conv.bias] if conv.bias is not None else [])
            if isinstance(act, PReLU):
                params.append(act.weight)
        return params

    def __call__(self, input_: SparseConvTensor) -> SparseConvTensor:
        params = self._parameters()
        if not (torch.is_grad_enabled() and any(p.requires_grad for p in params)):
            return super().__call__(input_)
        if input_.features.requires_grad:
            raise ValueError("TrainableNet does not compute the gradient of its input features")
        self._check_input(input_)
        layers, out_indices, shape = self._plan(input_)
        feats = _DeviceTraining.apply(self, layers, out_indices, input_.features, *params)
        return SparseConvTensor(feats, out_indices, shape, input_.batch_size)


class _DeviceTraining(torch.autograd.Function):
    """Forward and backward of :class:`TrainableNet` (inputs after ``out_indices``: the features, then the parameters in
    ``TrainableNet._parameters`` order)."""

    @staticmethod
    def forward(ctx, inet, layers, out_indices, feats, *params):
        from . import spconv

        device = feats.device
        saved = []
        x = feats
        for i, (conv, act, src, head) in enumerate(layers):
            last = i == len(layers) - 1
            nout = int(src.shape[0]) if src is not None else int(x.shape[0])
            out, pre, hidden, head_pre = spconv.layer_train(
                x, conv.weight, conv.bias, src, nout, inet._slope(act, device),
                head.weight if head is not None else None, head.bias if head is not None else None,
                out_indices if last else None)
            inv = spconv.invert_rules(src, x.shape[0]) if (src is not None and i > 0) else None
            saved.append((x, pre, hidden, head_pre, inv))
            x = out
        ctx.inet, ctx.layers, ctx.out_indices, ctx.saved = inet, layers, out_indices, saved
        ctx.param_ids = [id(p) for p in params]
        ctx.param_dtypes = [p.dtype for p in params]
        return x

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_features):
        from . import spconv

        inet, layers, out_indices = ctx.inet, ctx.layers, ctx.out_indices
        device = grad_features.device
        grads: dict[int, torch.Tensor] = {}
        g = grad_features.to(torch.float32).contiguous()
        for i in reversed(range(len(layers))):
            conv, act, src, head = layers[i]
            x, pre, hidden, head_pre, inv = ctx.saved[i]
            tail = None
            if head is not None:  # the fused final 1x1 and the tail: its gradients, then g at the hidden rows
                g_u, grads[id(head.weight)], db, _ = spconv.wgrad(hidden, g, head.weight.shape, pre=head_pre,
                                                                  tail_indices=out_indices)
                if head.bias is not None:
                    grads[id(head.bias)] = db
                g = spconv.conv_layer(g_u, head.weight.detach().permute(3, 1, 2, 0), None)
            elif i == len(layers) - 1:
                tail, pre = out_indices, head_pre
            prelu = isinstance(act, PReLU)
            slope = None if tail is not None else inet._slope(act, device)
            g_z, grads[id(conv.weight)], db, dslope = spconv.wgrad(x, g, conv.weight.shape, src, pre, slope, tail,
                                                                   slope_grad=prelu)
            if conv.bias is not None:
                grads[id(conv.bias)] = db
            if prelu:
                grads[id(act.weight)] = dslope.reshape(act.weight.shape)
            if i > 0:  # dX: the layer on g_z with the transposed weights and the inverse rules
                g = spconv.conv_layer(g_z, conv.weight.detach().permute(3, 1, 2, 0), None, inv, int(x.shape[0]))
        ctx.saved = None
        out = [grads[k].to(dt) for k, dt in zip(ctx.param_ids, ctx.param_dtypes)]
        return (None, None, None, None, *out)


def _check_conv(conv: SparseConv2d) -> None:
    cout, k, _, cin = conv.weight.shape
    if conv.k not in (1, 2):
        raise ValueError(f"kernel_size {conv.k} is not supported (1 or 2)")
    if conv.k == 1 and tuple(conv.padding) != (0, 0):
        raise ValueError("a 1x1 layer must not pad")
    if conv.k == 2 and tuple(conv.padding) not in ((1, 0), (0, 1)):
        raise ValueError(f"padding {tuple(conv.padding)} of a 2x2 layer is not supported ((1, 0) or (0, 1))")
    if not (1 <= cin <= 64 and 1 <= cout <= 64):
        raise ValueError(f"{cin} -> {cout} channels: at most 64 are supported")
