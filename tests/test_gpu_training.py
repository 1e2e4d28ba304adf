"""TrainableNet: the factor network's backward on the device kernels (dp_spconv_layer_train_f32, dp_spconv_rules_invert,
dp_spconv_wgrad_f32, and dp_spconv_layer_f32 for the input gradient) against fp64 and against the PyTorch module.

Per layer, every device result is held to the a-priori bound of its fp32 summation order against an fp64 evaluation on
the device path's own fp32 inputs (u = 2^-24): the weight, bias and slope gradients (chunked fma chains of at most
C = dp_spconv_wgrad_chunk_sites() terms, chunk partials added in fp64) within (C + 2) u sum|terms|, the input gradient
(the forward kernel) within (K + 2) u sum|terms| with K = ntaps cout. End to end, the parameter gradients must be at
least as close to fp64 as the fp32 module's autograd, within a factor of two.
"""
import copy

import pytest
import torch

from deeppreconditioning_b200 import _lib, metrics, model as models, spconv, synthetic

from test_gpu_inference import CASES, device_patterns, on, seeded_net, shuffled

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
CHUNK = None


def chunk_sites():
    global CHUNK
    if CHUNK is None:
        CHUNK = int(_lib.lib().dp_spconv_wgrad_chunk_sites())
    return CHUNK


def site_wave(st, seed=0):
    """A deterministic function of each site's (row, col): the same value for a system alone and in a batch."""
    ind = st.indices.double()
    return torch.sin(0.37 * ind[:, 1] + 0.11 * ind[:, 2] + seed).float()


def loss_vectors(st, seed=11):
    g = torch.Generator().manual_seed(seed)
    n = st.spatial_shape[0]
    x = torch.randn(st.batch_size, n, generator=g, dtype=torch.float64)
    b = torch.randn(st.batch_size, n, generator=g, dtype=torch.float64)
    return x.to(st.features.device), b.to(st.features.device)


def frobenius64(out, x, b):
    """metrics.frobenius_loss in fp64 with torch ops (the device loss kernels are fp32)."""
    ind = out.indices.long()
    v = out.features[:, 0]
    bb, r, c = ind[:, 0], ind[:, 1], ind[:, 2]

    def mv(vec, transpose):
        src, dst = (r, c) if transpose else (c, r)
        y = torch.zeros_like(vec)
        y.index_put_((bb, dst), v * vec[bb, src], accumulate=True)
        return y

    return torch.linalg.vector_norm(mv(mv(x, True), False) - b, dim=1).sum()


# ---- per-layer walk of the device path --------------------------------------------------------------------------------
def device_walk(inet, st, upstream):
    """Forward with layer_train and backward one primitive at a time, exactly as TrainableNet runs them. Returns the
    per-layer records (inputs, kept values, gradients) and the launch plan. ``upstream`` gives the output gradient."""
    device = st.features.device
    layers, out_indices, _ = inet._plan(st)
    recs, x = [], st.features
    for i, (conv, act, src, head) in enumerate(layers):
        last = i == len(layers) - 1
        nout = int(src.shape[0]) if src is not None else int(x.shape[0])
        out, pre, hidden, head_pre = spconv.layer_train(
            x, conv.weight, conv.bias, src, nout, inet._slope(act, device), head.weight if head is not None else None,
            head.bias if head is not None else None, out_indices if last else None)
        recs.append(dict(conv=conv, act=act, src=src, head=head, x=x, pre=pre, hidden=hidden, head_pre=head_pre,
                         out=out, inv=spconv.invert_rules(src, x.shape[0]) if src is not None else None))
        x = out
    g = upstream(x, out_indices)
    for i in reversed(range(len(recs))):
        r = recs[i]
        conv, act, head = r["conv"], r["act"], r["head"]
        tail, pre = None, r["pre"]
        if head is not None:
            r["g_head"] = g
            r["g_u"], r["dhw"], r["dhb"], _ = spconv.wgrad(r["hidden"], g, head.weight.shape, pre=r["head_pre"],
                                                           tail_indices=out_indices)
            g = spconv.conv_layer(r["g_u"], head.weight.detach().permute(3, 1, 2, 0), None)
            r["g_hidden"] = g
        elif i == len(recs) - 1:
            tail, pre = out_indices, r["head_pre"]
        slope = None if tail is not None else inet._slope(act, device)
        r["g_y"] = g
        r["g_z"], r["dW"], r["db"], r["dslope"] = spconv.wgrad(r["x"], g, conv.weight.shape, r["src"], pre, slope, tail,
                                                               slope_grad=isinstance(act, models.PReLU))
        r["tail"] = tail
        if i > 0:
            g = spconv.conv_layer(r["g_z"], conv.weight.detach().permute(3, 1, 2, 0), None, r["inv"], int(r["x"].shape[0]))
            r["dX"] = g
    return recs, out_indices


def slope_value(act):
    """The slope as the kernels see it (an fp32 scalar)."""
    if act is None:
        return None
    if isinstance(act, models.PReLU):
        return float(act.weight.detach())
    return float(torch.tensor(act.negative_slope, dtype=torch.float32))


def tail_grad64(g, u, ind):
    g, u = g.double(), u.double()
    r, c = ind[:, 1].long(), ind[:, 2].long()
    want = torch.where(r > c, g, torch.where(r < c, torch.zeros_like(g), g * torch.sigmoid(u)))
    return want, r < c, r == c


def wgrad64(x, g_z, rules, cout, ntaps, cin):
    """dW, db in fp64 from the device's fp32 g_z and inputs, with sum|terms|."""
    x, g = x.double(), g_z.double()
    nout = g.shape[0]
    if rules is None:
        rules = torch.arange(nout, device=g.device)[:, None]
    rules = rules.long()
    dW = torch.zeros(cout, ntaps, cin, dtype=torch.float64, device=g.device)
    terms = torch.zeros_like(dW)
    for t in range(ntaps):
        act = rules[:, t] >= 0
        xs = x[rules[act, t]]
        dW[:, t] = g[act].T @ xs
        terms[:, t] = g[act].abs().T @ xs.abs()
    return dW, terms, g.sum(0), g.abs().sum(0)


def dx64(g_z, weight, inv, nin):
    """The input gradient in fp64 from the device's g_z, with sum|terms|."""
    cout, k, _, cin = weight.shape
    W = weight.detach().double().reshape(cout, k * k, cin)
    g = g_z.double()
    if inv is None:
        inv = torch.arange(nin, device=g.device)[:, None]
    inv = inv.long()
    y = torch.zeros(nin, cin, dtype=torch.float64, device=g.device)
    terms = torch.zeros_like(y)
    for t in range(k * k):
        act = inv[:, t] >= 0
        gs = g[inv[act, t]]
        y[act] += gs @ W[:, t, :]
        terms[act] += gs.abs() @ W[:, t, :].abs()
    nterms = (inv >= 0).sum(1, keepdim=True).double() * cout
    return y, (nterms + 2) * U * terms


def within(got, want, bound, what):
    err = (got.double() - want).abs()
    assert bool((err <= bound).all()), f"{what}: worst excess {float((err - bound).max()):.3e}"


def check_layers(net, st, only_widest=False):
    """Check 3: every layer's g_z, dW, db, dslope and dX against fp64 on the device path's own fp32 inputs."""
    inet = models.TrainableNet(net)
    recs, out_indices = device_walk(inet, st, lambda y, ind: site_wave(models.SparseConvTensor(y, ind, [1, 1], 1))[:, None])
    cb = (chunk_sites() + 2) * U
    widest = max(range(len(recs)), key=lambda i: recs[i]["conv"].weight.numel() * int(recs[i]["g_z"].shape[0]))
    for i, r in enumerate(recs):
        if only_widest and i != widest:
            continue
        conv, act = r["conv"], r["act"]
        cout, k, _, cin = conv.weight.shape
        if r["head"] is not None:  # the tail and the head's own gradients
            want, upper, diag = tail_grad64(r["g_head"][:, 0], r["head_pre"], out_indices)
            gu = r["g_u"][:, 0]
            assert bool((gu[upper] == 0).all())
            lower = ~upper & ~diag
            assert torch.equal(gu[lower], r["g_head"][lower, 0])
            within(gu[diag], want[diag], 8 * U * want[diag].abs(), "tail (diagonal)")
            dhw, hterms, dhb, bterms = wgrad64(r["hidden"], r["g_u"], None, 1, 1, r["hidden"].shape[1])
            within(r["dhw"].reshape(1, 1, -1), dhw, cb * hterms, "head dW")
            within(r["dhb"], dhb, cb * bterms, "head db")
            hw = r["head"].weight.detach().double().reshape(-1)
            within(r["g_hidden"], r["g_u"].double() @ hw[None, :], U * (r["g_u"].double().abs() @ hw.abs()[None, :]),
                   "g_hidden")
        g_y = r["g_y"].double()
        if r["tail"] is not None:
            want, upper, diag = tail_grad64(r["g_y"][:, 0], r["head_pre"], out_indices)
            gz = r["g_z"][:, 0]
            assert bool((gz[upper] == 0).all())
            within(gz[diag], want[diag], 8 * U * want[diag].abs(), "tail (diagonal)")
        elif act is not None:
            a = slope_value(act)
            pre = r["pre"].double()
            gz64 = torch.where(pre > 0, g_y, a * g_y)
            within(r["g_z"], gz64, U * gz64.abs(), f"layer {i} g_z")
            assert torch.equal(r["g_z"][pre > 0], r["g_y"][pre > 0])  # exact where the derivative is 1
            if isinstance(act, models.PReLU):
                neg = pre <= 0
                ds = (g_y * pre)[neg].sum()
                within(r["dslope"], ds, cb * (g_y * pre)[neg].abs().sum(), f"layer {i} dslope")
        else:
            assert torch.equal(r["g_z"], r["g_y"])
        dW, terms, db, bterms = wgrad64(r["x"], r["g_z"], r["src"], cout, k * k, cin)
        within(r["dW"].reshape(cout, k * k, cin), dW, cb * terms, f"layer {i} dW")
        within(r["db"], db, cb * bterms, f"layer {i} db")
        if i > 0:
            y, bound = dx64(r["g_z"], conv.weight, r["inv"], int(r["x"].shape[0]))
            within(r["dX"], y, bound, f"layer {i} dX")
    return recs, widest


def grads_of(net):
    return [p.grad.detach().clone() for p in net.parameters()]


def check_end_to_end(net, st):
    """Check 4: per parameter tensor, ||g_dev - g64|| <= max(2 ||g_mod32 - g64||, 1e-5 ||g64||). Returns the ratios."""
    x, b = loss_vectors(st)
    dev_net, mod_net, net64 = copy.deepcopy(net), copy.deepcopy(net), copy.deepcopy(net).double()
    metrics.frobenius_loss(models.TrainableNet(dev_net)(st), x.float(), b.float()).backward()
    metrics.frobenius_loss(mod_net(st), x.float(), b.float()).backward()
    st64 = models.SparseConvTensor(st.features.double(), st.indices, st.spatial_shape, st.batch_size)
    frobenius64(net64(st64), x, b).backward()
    ratios = {}
    for (name, _), gd, gm, g64 in zip(net.named_parameters(), grads_of(dev_net), grads_of(mod_net), grads_of(net64)):
        e_dev = float(torch.linalg.vector_norm(gd.double() - g64))
        e_mod = float(torch.linalg.vector_norm(gm.double() - g64))
        ref = float(torch.linalg.vector_norm(g64))
        ratios[name] = e_dev / max(e_mod, 1e-300)
        assert e_dev <= max(2 * e_mod, 1e-5 * ref), (name, e_dev, e_mod, ref)
    return ratios


LAYER_CASES = ["2d64", "padded_batch", "edges", "empty_system", "shuffled", "3d32"]
LOSS_CASES = ["2d64", "padded_batch", "empty_system", "shuffled", "3d32"]  # square matrix images


# ---- 1. forward unchanged ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", LAYER_CASES)
def test_training_forward_is_the_inference_forward(cuda, case):
    st = CASES[case](cuda)
    net = seeded_net(device=cuda)
    got = models.TrainableNet(net)(st)
    want = models.InferenceNet(net)(st)
    assert got.features.grad_fn is not None
    assert torch.equal(got.indices, want.indices)
    assert got.spatial_shape == want.spatial_shape and got.batch_size == want.batch_size
    assert torch.equal(got.features.detach().view(torch.int32), want.features.view(torch.int32))
    with torch.no_grad():
        plain = models.TrainableNet(net)(st)
    assert plain.features.grad_fn is None
    assert torch.equal(plain.features.view(torch.int32), want.features.view(torch.int32))
    for p in net.parameters():
        p.requires_grad_(False)
    assert models.TrainableNet(net)(st).features.grad_fn is None


# ---- 2. inverse rules -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["2d64", "padded_batch", "edges", "empty_system", "shuffled", "3d32"])
def test_inverse_rules_are_the_scatter(cuda, case):
    st = CASES[case](cuda)
    inet = models.InferenceNet(seeded_net(device=cuda))
    nin = int(st.indices.shape[0])
    for pat in device_patterns(inet, st):
        if pat is None:
            continue
        ind, rules = pat
        inv = spconv.invert_rules(rules, nin)
        want = torch.full((nin, 4), -1, dtype=torch.int32, device=cuda)
        s = torch.arange(rules.shape[0], dtype=torch.int32, device=cuda)
        for t in range(4):
            act = rules[:, t] >= 0
            want[rules[act, t].long(), t] = s[act]
        assert torch.equal(inv, want)
        nin = int(rules.shape[0])


def test_duplicated_rules_raise(cuda):
    rules = torch.tensor([[0, -1, 1, -1], [2, 0, -1, -1], [0, -1, -1, -1]], dtype=torch.int32, device=cuda)
    with pytest.raises(_lib.DpcgError):
        spconv.invert_rules(rules, 3)  # sites 0 and 2 both read input 0 through tap 0
    with pytest.raises(_lib.DpcgError):
        spconv.invert_rules(rules[:2], 2)  # input 2 is out of range
    assert spconv.invert_rules(rules[:2], 3).shape == (3, 4)


# ---- 3. per layer against fp64 ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", LAYER_CASES)
def test_layer_gradients_within_fp32_bound_of_fp64(cuda, case):
    check_layers(seeded_net(device=cuda), CASES[case](cuda))


# ---- 4. end to end against the module ---------------------------------------------------------------------------------
@pytest.mark.parametrize("case", LOSS_CASES)
def test_parameter_gradients_as_close_to_fp64_as_the_module(cuda, case):
    ratios = check_end_to_end(seeded_net(device=cuda), CASES[case](cuda))
    print(f"{case}: ||g_dev - g64|| / ||g_mod32 - g64|| per parameter: "
          + ", ".join(f"{k} {v:.2f}" for k, v in ratios.items()))


# ---- 5. benchmark scale -----------------------------------------------------------------------------------------------
def test_gradients_at_benchmark_scale(cuda):
    st, _, _, _ = synthetic.make_batch("poisson2d", 316, [0, 1], device=cuda)
    net = seeded_net(device=cuda)
    recs, widest = check_layers(net, st, only_widest=True)
    nout = int(recs[widest]["g_z"].shape[0])
    props = torch.cuda.get_device_properties(cuda)
    resident_max = props.multi_processor_count * (props.max_threads_per_multi_processor // 256)
    chunks = -(-nout // chunk_sites())
    # bite guard: more chunks than CTAs of 256 threads can be resident, so the partials cross several waves
    assert chunks > resident_max, (chunks, resident_max)
    ratios = check_end_to_end(net, st)
    print(f"2 x 316^2: widest layer {widest} with {nout} sites in {chunks} chunks (resident CTAs <= {resident_max}); "
          + "ratios " + ", ".join(f"{k} {v:.2f}" for k, v in ratios.items()))


# ---- 6. determinism ---------------------------------------------------------------------------------------------------
def loss_gradient(tnet, st):
    """The gradient of frobenius_loss with respect to the network's output features, evaluated once. The loss's own
    COO products accumulate with fp32 atomics, so its value and this gradient may differ in the last bits between
    evaluations; the network's backward is checked on one fixed upstream gradient."""
    x, b = loss_vectors(st)
    with torch.no_grad():
        out = tnet(st)
    feats = out.features.clone().requires_grad_(True)
    loss = metrics.frobenius_loss(models.SparseConvTensor(feats, out.indices, out.spatial_shape, out.batch_size),
                                  x.float(), b.float())
    (g,) = torch.autograd.grad(loss, feats)
    return g


def test_backward_is_deterministic(cuda):
    st = CASES["padded_batch"](cuda)
    net = seeded_net(device=cuda)
    tnet = models.TrainableNet(net)
    g = loss_gradient(tnet, st)
    runs = []
    for _ in range(2):
        net.zero_grad(set_to_none=True)
        out = tnet(st)
        out.features.backward(g)
        runs.append(grads_of(net))
    for a, c in zip(*runs):
        assert torch.equal(a.view(torch.int32), c.view(torch.int32))


def per_layer_sites(inet, st):
    """The (batch, row, col) of every layer's input sites, in the order the device path holds them."""
    out, ind = [], st.indices
    pats = device_patterns(inet, st)
    for pat in pats:
        out.append(ind)
        if pat is not None:
            ind = pat[0]
    return out


def test_input_gradients_are_batch_independent(cuda):
    net = seeded_net(device=cuda)
    inet = models.TrainableNet(net)

    def upstream(y, ind):
        return site_wave(models.SparseConvTensor(y, ind, [1, 1], 1))[:, None]

    batch_st, _, _, _ = synthetic.make_batch("poisson2d", 40, [0, 1, 2])
    batch_st = on(batch_st, cuda)
    recs_b, _ = device_walk(inet, batch_st, upstream)
    sites_b = per_layer_sites(inet, batch_st)
    for k in range(3):
        alone, _, _, _ = synthetic.make_batch("poisson2d", 40, [k])
        alone = on(alone, cuda)
        recs_a, _ = device_walk(inet, alone, upstream)
        for i, (rb, ra, sb) in enumerate(zip(recs_b, recs_a, per_layer_sites(inet, alone))):
            if "dX" not in rb:
                continue
            mine = sites_b[i][:, 0] == k
            assert torch.equal(sites_b[i][mine, 1:], sb[:, 1:])
            assert torch.equal(rb["dX"][mine].view(torch.int32), ra["dX"].view(torch.int32)), f"layer {i}"


# ---- 7. training ------------------------------------------------------------------------------------------------------
def test_training_follows_the_module(cuda):
    st, _, _, _ = synthetic.make_batch("poisson2d", 32, list(range(8)), device=cuda)
    x, b = loss_vectors(st)
    x, b = x.float(), b.float()
    mod = seeded_net(device=cuda)
    dev = copy.deepcopy(mod)
    tdev = models.TrainableNet(dev)
    probe = copy.deepcopy(mod)  # step size: the first step moves the parameters by 1e-3 of their norm
    metrics.frobenius_loss(probe(st), x, b).backward()
    gnorm = float(torch.linalg.vector_norm(torch.cat([p.grad.reshape(-1) for p in probe.parameters()])))
    pnorm = float(torch.linalg.vector_norm(torch.cat([p.detach().reshape(-1) for p in probe.parameters()])))
    lr = 1e-3 * pnorm / gnorm
    opt_m = torch.optim.SGD(mod.parameters(), lr=lr)
    opt_d = torch.optim.SGD(dev.parameters(), lr=lr)
    losses = []
    for _ in range(10):
        opt_m.zero_grad()
        opt_d.zero_grad()
        lm = metrics.frobenius_loss(mod(st), x, b)
        ld = metrics.frobenius_loss(tdev(st), x, b)
        lm.backward()
        ld.backward()
        opt_m.step()
        opt_d.step()
        losses.append((float(lm), float(ld)))
    for lm, ld in losses:
        assert abs(ld - lm) <= 1e-4 * abs(lm), losses
    adam = torch.optim.Adam(dev.parameters(), lr=1e-3)
    first = last = None
    for _ in range(20):
        adam.zero_grad()
        loss = metrics.frobenius_loss(tdev(st), x, b)
        loss.backward()
        adam.step()
        first = float(loss) if first is None else first
        last = float(loss)
    with torch.no_grad():
        final = float(metrics.frobenius_loss(tdev(st), x, b))
    assert final < first, (first, last, final)
    print(f"SGD losses (module, device): {losses[0]} .. {losses[-1]}; Adam {first:.6g} -> {final:.6g}")


def test_gradients_accumulate_like_the_module(cuda):
    st = CASES["2d64"](cuda)
    net = seeded_net(device=cuda)
    mod = copy.deepcopy(net)
    tnet = models.TrainableNet(net)
    g = loss_gradient(tnet, st)
    tnet(st).features.backward(g)
    once = grads_of(net)
    tnet(st).features.backward(g)
    for g1, g2 in zip(once, grads_of(net)):
        assert torch.equal(g2, g1 + g1)
    mod(st).features.backward(g)  # the module accumulates the same way: .grad += the new gradient
    mod_once = grads_of(mod)
    mod(st).features.backward(g)
    for g1, g2 in zip(mod_once, grads_of(mod)):
        assert torch.equal(g2, g1 + g1)


@pytest.mark.parametrize("case", ["2d64", "3d32"])
def test_tril_net_training(cuda, case):
    net = seeded_net(models.PreconditionerTrilNet, device=cuda)
    st = shuffled(CASES[case](cuda))
    got = models.TrainableNet(net)(st)
    assert got.indices is st.indices and got.features.grad_fn is not None
    assert torch.equal(got.features.detach().view(torch.int32), models.InferenceNet(net)(st).features.view(torch.int32))
    check_layers(net, st)
    ratios = check_end_to_end(net, st)
    print(f"trilnet {case}: ratios " + ", ".join(f"{k} {v:.2f}" for k, v in ratios.items()))


def test_single_layer_net_trains(cuda):
    torch.manual_seed(3)
    net = models.PreconditionerTrilNet([1, 1]).to(cuda)
    st = CASES["2d64"](cuda)
    check_layers(net, st)
    check_end_to_end(net, st)
