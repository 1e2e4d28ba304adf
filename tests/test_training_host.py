"""CPU tests of TrainableNet and the backward entry points (dp_spconv_layer_train_f32, dp_spconv_rules_invert,
dp_spconv_wgrad_*): what is accepted, what is rejected before any launch."""
import ctypes

import pytest
import torch
from torch import nn

from deeppreconditioning_b200 import _lib, build
from deeppreconditioning_b200 import model as models


def _net_with(mutate):
    torch.manual_seed(0)
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS)
    mutate(net)
    return net


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.lib()


def _tiny_input(requires_grad=False):
    feats = torch.ones(3, 1, requires_grad=requires_grad)
    return models.SparseConvTensor(feats, torch.tensor([[0, 0, 0], [0, 1, 0], [0, 1, 1]], dtype=torch.int32), [2, 2], 1)


def test_trainable_net_accepts_what_inference_net_accepts():
    torch.manual_seed(0)
    for net in (models.PreconditionerNet(models.DEFAULT_CHANNELS), models.PreconditionerTrilNet(models.DEFAULT_CHANNELS),
                models.PreconditionerTrilNet([1, 1]), models.PreconditionerNet([1, 64, 64, 64, 1])):
        t, i = models.TrainableNet(net), models.InferenceNet(net)
        assert isinstance(t, models.InferenceNet)
        assert t.steps == i.steps
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS)
    # conv weights and biases of every layer, then the PReLU weights: every parameter of the module, once
    assert {id(p) for p in models.TrainableNet(net)._parameters()} == {id(p) for p in net.parameters()}
    assert len(models.TrainableNet(net)._parameters()) == len(list(net.parameters()))
    tril = models.PreconditionerTrilNet(models.DEFAULT_CHANNELS)  # LeakyReLU: no parameter of its own
    assert {id(p) for p in models.TrainableNet(tril)._parameters()} == {id(p) for p in tril.parameters()}


@pytest.mark.parametrize("mutate", [
    lambda n: setattr(n.layers[2], "padding", (1, 1)),
    lambda n: n.layers.__setitem__(2, models.SparseConv2d(16, 32, 3, padding=(1, 1))),
    lambda n: n.layers.__setitem__(1, models.PReLU(16)),
    lambda n: n.layers.__setitem__(1, nn.ReLU()),
    lambda n: n.layers.append(models.PReLU()),
    lambda n: n.layers.__setitem__(len(n.layers) - 1, models.SparseConv2d(16, 2, 1)),
], ids=["pad11", "k3", "prelu16", "relu", "trailing_act", "two_out"])
def test_trainable_net_rejects_what_inference_net_rejects(mutate):
    with pytest.raises(ValueError):
        models.TrainableNet(_net_with(mutate))


def test_trainable_net_rejects_other_modules_and_wide_layers():
    with pytest.raises(ValueError):
        models.TrainableNet(nn.Sequential(models.SparseConv2d(1, 1, 1)))
    with pytest.raises(ValueError):
        models.TrainableNet(models.PreconditionerNet([1, 65, 1]))


def test_cpu_inputs_and_inputs_that_require_grad_raise():
    torch.manual_seed(0)
    net = models.TrainableNet(models.PreconditionerNet(models.DEFAULT_CHANNELS))
    with pytest.raises(_lib.DpcgError):
        net(_tiny_input())  # the autograd path
    with torch.no_grad(), pytest.raises(_lib.DpcgError):
        net(_tiny_input())  # the inference path
    with pytest.raises(ValueError):
        net(_tiny_input(requires_grad=True))


def test_backward_argument_validation_without_a_gpu(lib):
    L = _lib.SpconvLayer
    layer = L(nout=10, ntaps=3, cin=4, cout=4, in_=16, weight=16, out=16)
    assert lib.dp_spconv_layer_train_f32(ctypes.byref(layer), 16, 16, 16, None) == 1  # 3 taps
    layer = L(nout=10, ntaps=4, cin=65, cout=4, src=16, in_=16, weight=16, out=16)
    assert lib.dp_spconv_layer_train_f32(ctypes.byref(layer), 16, 16, 16, None) == 1  # 65 channels
    layer = L(nout=10, ntaps=1, cin=4, cout=4, in_=16, weight=16, out=16, slope=16)
    assert lib.dp_spconv_layer_train_f32(ctypes.byref(layer), None, None, None, None) == 1  # activation without pre
    layer = L(nout=10, ntaps=1, cin=4, cout=4, in_=16, weight=16, out=16, slope=16, head_weight=16)
    assert lib.dp_spconv_layer_train_f32(ctypes.byref(layer), 16, None, 16, None) == 1  # head without hidden
    layer = L(nout=10, ntaps=1, cin=4, cout=1, in_=16, weight=16, out=16, indices=16)
    assert lib.dp_spconv_layer_train_f32(ctypes.byref(layer), None, None, None, None) == 1  # tail without head_pre
    layer = L(nout=10, ntaps=1, cin=4, cout=4, slope=16)
    assert lib.dp_spconv_layer_train_f32(ctypes.byref(layer), 16, None, None, None) == 1  # no input / weight / out
    assert lib.dp_spconv_layer_train_f32(None, None, None, None, None) == 1

    assert lib.dp_spconv_rules_invert(16, 10, 2, 10, 16, 16, None) == 1  # 2 taps
    assert lib.dp_spconv_rules_invert(None, 10, 4, 10, 16, 16, None) == 1  # no rules
    assert lib.dp_spconv_rules_invert(16, 10, 4, 10, None, 16, None) == 1  # no inverse
    assert lib.dp_spconv_rules_invert(16, 10, 4, 10, 16, None, None) == 1  # no flag
    assert lib.dp_spconv_rules_invert(16, -1, 4, 10, 16, 16, None) == 1
    assert lib.dp_spconv_rules_invert(16, 10, 4, 1 << 31, 16, 16, None) == 1

    G = _lib.SpconvGrad
    full = dict(in_=16, grad_out=16, grad_pre=16, grad_weight=16)
    ws_bytes = lib.dp_spconv_wgrad_workspace_bytes(10, 4, 4, 4)

    def wgrad(g, ws=256, nbytes=ws_bytes):
        return lib.dp_spconv_wgrad_f32(ctypes.byref(g), ws, nbytes, None)

    assert wgrad(G(nout=10, ntaps=2, cin=4, cout=4, src=16, **full)) == 1  # 2 taps
    assert wgrad(G(nout=10, ntaps=4, cin=0, cout=4, src=16, **full)) == 1  # no channels
    assert wgrad(G(nout=10, ntaps=4, cin=4, cout=65, src=16, **full)) == 1  # 65 channels
    assert wgrad(G(nout=10, ntaps=4, cin=4, cout=4, **full)) == 1  # a 2x2 layer needs its rules
    assert wgrad(G(nout=10, ntaps=4, cin=4, cout=4, src=16, slope=16, **full)) == 1  # activation without pre
    assert wgrad(G(nout=10, ntaps=1, cin=4, cout=2, pre=16, tail_indices=16, **full)) == 1  # the tail is one channel
    assert wgrad(G(nout=10, ntaps=1, cin=4, cout=1, pre=16, slope=16, tail_indices=16, **full)) == 1  # tail and slope
    assert wgrad(G(nout=10, ntaps=1, cin=4, cout=4, grad_slope=16, **full)) == 1  # slope gradient without a slope
    assert wgrad(G(nout=10, ntaps=4, cin=4, cout=4, src=16, in_=16, grad_out=16, grad_pre=16)) == 1  # no grad_weight
    assert wgrad(G(nout=10, ntaps=4, cin=4, cout=4, src=16, **full), ws=None) == 1  # no workspace
    assert wgrad(G(nout=10, ntaps=4, cin=4, cout=4, src=16, **full), ws=264) == 2  # unaligned workspace
    assert wgrad(G(nout=10, ntaps=4, cin=4, cout=4, src=16, **full), nbytes=ws_bytes - 1) == 3  # short workspace
    assert lib.dp_spconv_wgrad_f32(None, 256, 1 << 20, None) == 1


def test_empty_layers_do_nothing(lib):
    layer = _lib.SpconvLayer(nout=0, ntaps=4, cin=4, cout=4, src=16, slope=16)
    assert lib.dp_spconv_layer_train_f32(ctypes.byref(layer), None, None, None, None) == 0
    assert lib.dp_spconv_rules_invert(None, 0, 4, 0, None, None, None) == 0
    g = _lib.SpconvGrad(nout=0, ntaps=4, cin=4, cout=4, src=16)
    assert lib.dp_spconv_wgrad_f32(ctypes.byref(g), None, 0, None) == 0


def test_chunk_size_and_workspace_query(lib):
    c = lib.dp_spconv_wgrad_chunk_sites()
    assert c > 0
    row = 4 * 32 * (4 * 64 + 2)  # bytes of one chunk partial of a 64 -> 32 2x2 layer
    assert lib.dp_spconv_wgrad_workspace_bytes(c, 4, 64, 32) >= row
    assert lib.dp_spconv_wgrad_workspace_bytes(c + 1, 4, 64, 32) >= 2 * row
    sizes = [lib.dp_spconv_wgrad_workspace_bytes(n, 4, 64, 32) for n in (1, c, c + 1, 10 * c, 4_000_000)]
    assert sizes == sorted(sizes) and sizes[-1] > sizes[0]
    assert lib.dp_spconv_wgrad_workspace_bytes(0, 4, 64, 32) == 0
    assert lib.dp_spconv_wgrad_workspace_bytes(10, 3, 64, 32) == 0
    assert lib.dp_spconv_wgrad_workspace_bytes(10, 4, 65, 32) == 0
    assert lib.dp_spconv_wgrad_workspace_bytes(-1, 4, 64, 32) == 0
