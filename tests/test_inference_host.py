"""CPU tests of InferenceNet and the dp_spconv_* entry points: what is accepted, what is rejected before any launch."""
import ctypes

import pytest
import torch
from torch import nn

from deeppreconditioning_b200 import _lib, build
from deeppreconditioning_b200 import model as models


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.lib()


def test_both_module_trees_are_accepted():
    torch.manual_seed(0)
    net = models.InferenceNet(models.PreconditionerNet(models.DEFAULT_CHANNELS))
    assert [(c.k, tuple(c.padding)) for c, _ in net.steps] == [(1, (0, 0)), (2, (1, 0)), (2, (1, 0)), (2, (0, 1)),
                                                               (2, (0, 1)), (1, (0, 0))]
    assert all(isinstance(a, models.PReLU) for _, a in net.steps[:-1]) and net.steps[-1][1] is None
    tril = models.InferenceNet(models.PreconditionerTrilNet(models.DEFAULT_CHANNELS))
    assert all(c.k == 1 for c, _ in tril.steps) and all(isinstance(a, models.LeakyReLU) for _, a in tril.steps[:-1])
    models.InferenceNet(models.PreconditionerTrilNet([1, 1]))  # a single 1x1 layer
    models.InferenceNet(models.PreconditionerNet([1, 64, 64, 64, 1]))


def _net_with(mutate):
    torch.manual_seed(0)
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS)
    mutate(net)
    return net


@pytest.mark.parametrize("mutate", [
    lambda n: setattr(n.layers[2], "padding", (1, 1)),
    lambda n: setattr(n.layers[2], "padding", (0, 0)),
    lambda n: setattr(n.layers[0], "padding", (1, 0)),
    lambda n: n.layers.__setitem__(2, models.SparseConv2d(16, 32, 3, padding=(1, 1))),
    lambda n: n.layers.__setitem__(1, models.PReLU(16)),
    lambda n: n.layers.__setitem__(1, nn.ReLU()),
    lambda n: n.layers.append(models.PReLU()),
    lambda n: n.layers.__setitem__(len(n.layers) - 1, models.SparseConv2d(16, 2, 1)),
    lambda n: n.layers.__setitem__(len(n.layers) - 1, models.SparseConv2d(8, 1, 1)),
], ids=["pad11", "pad00", "pad1x1", "k3", "prelu16", "relu", "trailing_act", "two_out", "channel_mismatch"])
def test_unsupported_trees_raise_at_construction(mutate):
    with pytest.raises(ValueError):
        models.InferenceNet(_net_with(mutate))


def test_other_modules_and_wide_layers_raise():
    with pytest.raises(ValueError):
        models.InferenceNet(nn.Sequential(models.SparseConv2d(1, 1, 1)))
    with pytest.raises(ValueError):
        models.InferenceNet(models.PreconditionerNet([1, 65, 1]))


def test_cpu_input_raises():
    torch.manual_seed(0)
    net = models.InferenceNet(models.PreconditionerNet(models.DEFAULT_CHANNELS))
    st = models.SparseConvTensor(torch.ones(3, 1), torch.tensor([[0, 0, 0], [0, 1, 0], [0, 1, 1]], dtype=torch.int32),
                                 [2, 2], 1)
    with pytest.raises(_lib.DpcgError):
        net(st)


def test_spconv_argument_validation_without_a_gpu(lib):
    layer = _lib.SpconvLayer(nout=10, ntaps=3, cin=4, cout=4)
    assert lib.dp_spconv_layer_f32(ctypes.byref(layer), None) == 1  # 3 taps
    layer = _lib.SpconvLayer(nout=10, ntaps=4, cin=65, cout=4, src=16)
    assert lib.dp_spconv_layer_f32(ctypes.byref(layer), None) == 1  # 65 channels
    layer = _lib.SpconvLayer(nout=10, ntaps=4, cin=4, cout=4)
    assert lib.dp_spconv_layer_f32(ctypes.byref(layer), None) == 1  # a 2x2 layer needs its rules
    layer = _lib.SpconvLayer(nout=10, ntaps=1, cin=4, cout=2, indices=16)
    assert lib.dp_spconv_layer_f32(ctypes.byref(layer), None) == 1  # the tail acts on one channel
    layer = _lib.SpconvLayer(nout=0, ntaps=1, cin=4, cout=4)
    assert lib.dp_spconv_layer_f32(ctypes.byref(layer), None) == 0  # nothing to do
    assert lib.dp_spconv_rules_count(16, 32, 1, 8, 8, 1, 1, 48, 64, 1 << 20, None) == 1  # padding (1, 1)
    assert lib.dp_spconv_rules_fill(16, 32, None, 1, 8, 8, 1, 0, 48, 64, 72, None, None) == 2  # rules not 16-byte aligned
    assert lib.dp_spconv_sort_sites(None, 5, 1, 4, 4, None, None, None, None, None, 0, None) == 1
    assert lib.dp_spconv_sort_workspace_bytes(2, 100) >= 4 * 201
