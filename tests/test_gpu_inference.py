"""InferenceNet: the factor network's forward on the device kernels (dp_spconv_*) against the PyTorch module.

Patterns (site sets and per-tap rules of every layer) must be the module's bit for bit. Values are held to the a-priori
bound of an fp32 recursive sum against an fp64 evaluation of the same layer on the same fp32 inputs:
|y - y64| <= (K + 2) 2^-24 sum|terms|, K the number of terms; scaled by max(1, |slope|) after the activation.
"""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

import helpers
import deeppreconditioning_b200 as dp
from deeppreconditioning_b200 import _lib, model as models, spconv, synthetic
from deeppreconditioning_b200.sparse import CsrMatrix
from deeppreconditioning_b200.test import BenchmarkSuite
from oracle import sparse as osp

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
SPREAD = json.loads((Path(__file__).parent / "golden" / "pcg_spread.json").read_text())["cases"]


def seeded_net(cls=models.PreconditionerNet, seed=69, device=None):
    torch.manual_seed(seed)  # test.py:205, the seed tests/helpers.py gives the factors of the golden vectors
    net = cls(models.DEFAULT_CHANNELS)
    return net.to(device) if device is not None else net


def on(st, device):
    return helpers.to_device(st, device)


def module_rules(conv, x):
    """Output indices and per-tap rules of a 2x2 layer exactly as model.SparseConv2d.forward derives them."""
    k, (ph, pw) = conv.k, conv.padding
    h, w = x.spatial_shape
    ho, wo = h + 2 * ph - k + 1, w + 2 * pw - k + 1
    b, r, c = (x.indices[:, i].long() for i in range(3))
    keys, srcs = [], []
    for ky in range(k):
        for kx in range(k):
            ro, co = r - ky + ph, c - kx + pw
            ok = (ro >= 0) & (ro < ho) & (co >= 0) & (co < wo)
            keys.append(((b * ho + ro) * wo + co)[ok])
            srcs.append(ok.nonzero().squeeze(1))
    uniq, inverse = torch.unique(torch.cat(keys), return_inverse=True)
    rules = torch.full((uniq.shape[0], 4), -1, dtype=torch.int64, device=uniq.device)
    start = 0
    for t, (key, src) in enumerate(zip(keys, srcs)):
        rules[inverse[start:start + key.shape[0]], t] = src
        start += key.shape[0]
    indices = torch.stack((uniq // (ho * wo), (uniq // wo) % ho, uniq % wo), dim=1).int()
    return indices, rules


def module_trace(net, st):
    """The module's input to every convolution, and its output."""
    inputs, x = [], st
    with torch.no_grad():
        for layer in net.layers:
            if isinstance(layer, models.SparseConv2d):
                inputs.append(x)
            x = layer(x)
        return inputs, net(st)


def device_patterns(inet, st):
    """Per-layer (indices, rules) of the device path: what InferenceNet computes before its first GEMM."""
    batch, (h, w) = st.batch_size, st.spatial_shape
    rowptr, col, perm = spconv.sort_sites(st.indices, batch, h, w)
    out = []
    for conv, _ in inet.steps:
        if conv.k == 2:
            rowptr, col, rules, ind = spconv.conv_rules(rowptr, col, batch, h, w, conv.padding, perm, with_indices=True)
            perm = None
            out.append((ind, rules))
        else:
            out.append(None)
        h, w = h + 2 * conv.padding[0] - conv.k + 1, w + 2 * conv.padding[1] - conv.k + 1
    return out


def assert_patterns(net, st):
    inet = models.InferenceNet(net)
    inputs, want = module_trace(net, st)
    got = inet(st)
    for (conv, _), x, pat in zip(inet.steps, inputs, device_patterns(inet, st)):
        if pat is None:
            continue
        ind, rules = module_rules(conv, x)
        assert torch.equal(pat[0], ind), "site set differs"
        assert torch.equal(pat[1].long(), rules), "rules differ"
    assert torch.equal(got.indices, want.indices) and got.indices.dtype == want.indices.dtype
    assert got.spatial_shape == want.spatial_shape and got.batch_size == want.batch_size
    assert got.features.dtype == torch.float32 and got.features.shape == (want.indices.shape[0], 1)
    return got, want


def fp64_layer(x32, conv, rules, slope):
    """fp64 evaluation of one layer on fp32 inputs: (y64 after the activation, bound of the fp32 result)."""
    cout, k, _, cin = conv.weight.shape
    W = conv.weight.detach().double().reshape(cout, k * k, cin)
    x = x32.double()
    if rules is None:
        rules = torch.arange(x.shape[0], device=x.device)[:, None]
    rules = rules.long()
    y = torch.zeros(rules.shape[0], cout, dtype=torch.float64, device=x.device)
    terms = torch.zeros_like(y)
    for t in range(k * k):
        active = rules[:, t] >= 0
        xs = x[rules[active, t]]
        y[active] += xs @ W[:, t, :].T
        terms[active] += xs.abs() @ W[:, t, :].abs().T
    nterms = (rules >= 0).sum(1, keepdim=True).double() * cin
    if conv.bias is not None:
        b = conv.bias.detach().double()
        y, terms, nterms = y + b, terms + b.abs(), nterms + 1
    bound = (nterms + 2) * U * terms
    if slope is not None:
        a = float(slope)
        y = torch.where(y > 0, y, a * y)
        bound = bound * max(1.0, abs(a))
    return y, bound


def slope_of(act):
    if act is None:
        return None
    return float(act.weight) if isinstance(act, models.PReLU) else float(act.negative_slope)


def check_values(net, st):
    """Every layer on the module's fp32 inputs against fp64; the fused last layer (1x1 head and tail included) too."""
    inet = models.InferenceNet(net)
    inputs, want = module_trace(net, st)
    pats = device_patterns(inet, st)
    steps = inet.steps
    for i, ((conv, act), x, pat) in enumerate(zip(steps, inputs, pats)):
        rules = None if pat is None else pat[1]
        slope = None if act is None else inet._slope(act, x.features.device)
        if i == len(steps) - 1:
            continue  # the head: checked fused below
        got = spconv.conv_layer(x.features, conv.weight, conv.bias, rules, slope=slope)
        y64, bound = fp64_layer(x.features, conv, rules, slope_of(act))
        err = (got.double() - y64).abs()
        assert bool((err <= bound).all()), f"layer {i}: worst excess {float((err - bound).max())}"
    # fused: last hidden layer, its activation, the final 1x1 and the tail
    (conv, act), (head, _) = steps[-2], steps[-1]
    x, pat = inputs[-2], pats[-2]
    rules = None if pat is None else pat[1]
    h64, hbound = fp64_layer(x.features, conv, rules, slope_of(act))
    w1 = head.weight.detach().double().reshape(-1)
    b1 = head.bias.detach().double()
    y64 = h64 @ w1 + b1
    ybound = hbound @ w1.abs() + (w1.numel() + 3) * U * ((h64.abs() + hbound) @ w1.abs() + b1.abs())
    ind = want.indices.long()
    got = inet(st).features[:, 0].double()
    upper, diag = ind[:, 1] < ind[:, 2], ind[:, 1] == ind[:, 2]
    assert bool((got[upper] == 0).all())
    sp64 = torch.nn.functional.softplus(y64[diag])
    err = (got[diag] - sp64).abs()
    assert bool((err <= ybound[diag] + 4 * U * sp64.abs()).all())
    lower = ~upper & ~diag
    assert bool(((got[lower] - y64[lower]).abs() <= ybound[lower]).all())
    rel = float(torch.linalg.vector_norm(inet(st).features.double() - want.features.double())
                / torch.linalg.vector_norm(want.features.double()))
    assert rel <= 1e-5, rel
    return rel


def padded_batch(cuda):
    st, _, _, sizes = synthetic.make_batch("poisson2d", 24, [0, 1, 2], pad_to=24 * 24 + 50)
    return on(st, cuda)


def batch_with_empty_system(cuda):
    st, _, _, _ = synthetic.make_batch("poisson2d", 20, [3, 4])
    ind = st.indices.clone()
    ind[ind[:, 0] == 1, 0] = 2  # systems 0 and 2 hold sites, system 1 none
    return models.SparseConvTensor(st.features.to(cuda), ind.to(cuda), st.spatial_shape, 3)


def edge_sites(cuda):
    """Sites on the first and last rows and columns of a 40 x 30 image, where the paddings clip, in random order."""
    g = torch.Generator().manual_seed(5)
    h, w = 40, 30
    dense = torch.rand(h, w, generator=g) < 0.15
    dense[0, :] = dense[-1, :] = dense[:, 0] = dense[:, -1] = True
    idx = dense.nonzero()
    idx = idx[torch.randperm(idx.shape[0], generator=g)]
    ind = torch.cat([torch.zeros(idx.shape[0], 1, dtype=torch.long), idx], 1).int()
    feats = torch.randn(ind.shape[0], 1, generator=g)
    return models.SparseConvTensor(feats.to(cuda), ind.to(cuda), [h, w], 1)


def shuffled(st, seed=3):
    g = torch.Generator().manual_seed(seed)
    order = torch.randperm(st.indices.shape[0], generator=g).to(st.indices.device)
    return models.SparseConvTensor(st.features[order], st.indices[order], st.spatial_shape, st.batch_size)


def with_zero_entries(cuda):
    p = helpers.problem("poisson2d", 32, 2)
    st = on(p.systems_tril, cuda)
    feats = st.features.clone()
    feats[::7] = 0.0  # stored zeros stay active sites
    return models.SparseConvTensor(feats, st.indices, st.spatial_shape, 1)


CASES = {
    "2d64": lambda cuda: on(helpers.problem("poisson2d", 64, 0).systems_tril, cuda),
    "2d316": lambda cuda: on(helpers.problem("poisson2d", 316, 0).systems_tril, cuda),
    "padded_batch": padded_batch,
    "3d32": lambda cuda: on(helpers.problem("poisson3d", 32, 0).systems_tril, cuda),
    "shuffled": lambda cuda: shuffled(on(helpers.problem("poisson2d", 48, 1).systems_tril, cuda)),
    "zero_entries": with_zero_entries,
    "edges": edge_sites,
    "empty_system": batch_with_empty_system,
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_patterns_are_the_modules(cuda, case):
    st = CASES[case](cuda)
    assert_patterns(seeded_net(device=cuda), st)


@pytest.mark.parametrize("case", ["2d64", "2d316", "padded_batch", "edges", "empty_system"])
def test_values_within_fp32_bound_of_fp64(cuda, case):
    rel = check_values(seeded_net(device=cuda), CASES[case](cuda))
    print(f"{case}: normwise relative difference to the PyTorch forward {rel:.3e}")


@pytest.mark.parametrize("case", ["2d64", "3d32"])
def test_tril_net_pattern_and_values(cuda, case):
    net = seeded_net(models.PreconditionerTrilNet, device=cuda)
    st = shuffled(CASES[case](cuda))
    got, want = assert_patterns(net, st)
    assert got.indices is st.indices  # all-1x1: the input's own sites, in its order
    check_values(net, st)


def test_deterministic_and_batch_independent(cuda):
    net = models.InferenceNet(seeded_net(device=cuda))
    st, _, _, _ = synthetic.make_batch("poisson2d", 40, [0, 1, 2])
    batch = net(on(st, cuda))
    again = net(on(st, cuda))
    assert torch.equal(batch.indices, again.indices)
    assert torch.equal(batch.features.view(torch.int32), again.features.view(torch.int32))
    for k in range(3):
        single, _, _, _ = synthetic.make_batch("poisson2d", 40, [k])
        alone = net(on(single, cuda))
        mine = batch.indices[:, 0] == k
        assert torch.equal(batch.indices[mine, 1:], alone.indices[:, 1:])
        assert torch.equal(batch.features[mine].view(torch.int32), alone.features.view(torch.int32))


def test_downstream_parity_316(cuda):
    p = helpers.problem("poisson2d", 316, 0, 0.5, "net")
    case = next(c for c in SPREAD if c["kind"] == "poisson2d" and c["side"] == 316 and c["net"] == "net"
                and c["precond"] == "multiply" and c["index"] == 0)
    out = models.InferenceNet(seeded_net(device=cuda))(on(p.systems_tril, cuda))
    L, Lt = CsrMatrix.from_spconv(out, p.n, "tril"), CsrMatrix.from_spconv(out, p.n, "tril_t")
    rowptr, col, _ = L.to_host()
    assert np.array_equal(rowptr, p.L[0]) and np.array_equal(col, p.L[1])
    A = CsrMatrix.from_spconv(on(p.systems_tril, cuda), p.n, "symmetrise")
    result = dp.pcg_solve(A, p.b.to(cuda), dp.FactoredMultiply(L, Lt), max_iter=case["max_iter"])
    lo, hi = case["iterations_min"], case["iterations_max"]
    margin = max(1, hi - lo)  # test_gpu_parity.spread_margin
    assert lo - margin <= result.iterations <= hi + margin, (result.iterations, lo, hi)
    a, bn = osp.to_scipy(*p.A), p.b.numpy()
    true_rel = np.linalg.norm(a @ result.x_hat.cpu().numpy() - bn) / np.linalg.norm(bn)
    assert true_rel < 2e-4, true_rel
    print(f"316^2 multiply-mode PCG on the device factor: {result.iterations} iterations (reference {lo}..{hi}), "
          f"true residual {true_rel:.2e}")


def test_load_state_dict_applies(cuda):
    net = seeded_net(device=cuda)
    inet = models.InferenceNet(net)
    st = on(helpers.problem("poisson2d", 24, 0).systems_tril, cuda)
    before = inet(st).features.clone()
    other = seeded_net(seed=7, device=cuda)
    net.load_state_dict(other.state_dict())
    after = inet(st).features
    assert not torch.equal(before, after)
    assert torch.equal(after.view(torch.int32), models.InferenceNet(other)(st).features.view(torch.int32))
    with torch.no_grad():
        want = other(st).features
    assert float(torch.linalg.vector_norm(after - want) / torch.linalg.vector_norm(want)) <= 1e-5


def test_benchmark_suite_with_inference_net(cuda):
    net = seeded_net(device=cuda)
    data = synthetic.SyntheticPressureDataSet("poisson2d", 24, number_samples=3, batch_size=1, device=cuda)
    ref = BenchmarkSuite(data, net, techniques=("learned",), max_iter=5000)
    ref.run()
    dev = BenchmarkSuite(data, models.InferenceNet(net), techniques=("learned",), max_iter=5000)
    dev.run()
    assert dev.densities["learned"] == ref.densities["learned"]
    assert len(dev.iterations["learned"]) == 3 and all(0 < i < 5000 for i in dev.iterations["learned"])
    assert all(s == 100 for s in dev.successes["learned"]) and all(r < 1e-8 for r in dev.residuals["learned"])


def test_duplicate_sites_raise(cuda):
    st = on(helpers.problem("poisson2d", 16, 0).systems_tril, cuda)
    dup = models.SparseConvTensor(torch.cat([st.features, st.features[5:6]]), torch.cat([st.indices, st.indices[5:6]]),
                                  st.spatial_shape, 1)
    with pytest.raises(_lib.DpcgError):
        models.InferenceNet(seeded_net(device=cuda))(dup)
