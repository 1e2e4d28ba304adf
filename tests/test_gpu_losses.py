"""The training losses under torch.use_deterministic_algorithms(True): sorted-site products (dp_sorted_spmv_f32,
dp_system_matvec_f32) and the fused loss and its gradient (dp_llt_residual_f32, dp_llt_residual_grad_f32).

Pinned here: every product is bitwise the oracle's sequential loop on sorted sites; results repeat bit for bit, do not
depend on the order of the input's sites, and a system's term and gradients are the same alone and in a batch; values and
gradients are at least as close to fp64 as the atomic path (within a factor of two); and with the flag off nothing of
this runs. Reference values on the PyTorch module path are computed with the flag off: its matmuls need
CUBLAS_WORKSPACE_CONFIG set before CUDA starts.
"""
import contextlib
import json
from pathlib import Path

import numpy as np
import pytest
import torch

import helpers
from deeppreconditioning_b200 import _lib, metrics, model as models, synthetic, utils
from oracle import ckernels

from test_gpu_inference import seeded_net
from test_oracle import _loss_batch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


@contextlib.contextmanager
def flag(enabled):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(enabled, warn_only=False)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


@pytest.fixture
def deterministic():
    with flag(True):
        yield


def bits(t):
    return t.detach().contiguous().view(torch.int32)


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(bits(a), bits(b))


# ---- cases ------------------------------------------------------------------------------------------------------------
def on(st, cuda):
    return helpers.to_device(st, cuda)


def factor_of(st, cls=models.PreconditionerNet):
    with torch.no_grad():
        return models.InferenceNet(seeded_net(cls, device=st.features.device))(st)


def vectors(st, seed=11):
    g = torch.Generator().manual_seed(seed)
    shape = (st.batch_size, st.spatial_shape[0])
    return torch.randn(shape, generator=g).to(st.features.device), torch.randn(shape, generator=g).to(st.features.device)


def case_loss_batch(cuda):
    st, learned, x, b = _loss_batch()
    return on(st, cuda), on(learned, cuda), x.to(cuda), b.to(cuda)


def case_grid(cuda, side, count, cls=models.PreconditionerNet, kind="poisson2d"):
    st = synthetic.make_batch(kind, side, list(range(count)), device=cuda)[0]
    return (st, factor_of(st, cls), *vectors(st))


def case_padded_empty(cuda):
    """Systems 0 and 2 padded to 450 unknowns, system 1 without a site and with x = b = 0."""
    st, _, _, _ = synthetic.make_batch("poisson2d", 20, [3, 4], pad_to=450)
    ind = st.indices.clone()
    ind[ind[:, 0] == 1, 0] = 2
    st = models.SparseConvTensor(st.features.to(cuda), ind.to(cuda), st.spatial_shape, 3)
    x, b = vectors(st)
    x[1], b[1] = 0.0, 0.0
    return st, factor_of(st), x, b


def shuffle(st, seed):
    order = torch.randperm(st.indices.shape[0], generator=torch.Generator().manual_seed(seed)).to(st.indices.device)
    return models.SparseConvTensor(st.features[order], st.indices[order], st.spatial_shape, st.batch_size), order


def case_padded_shuffled(cuda):
    st, ln, x, b = case_padded_empty(cuda)
    return shuffle(st, 1)[0], shuffle(ln, 2)[0], x, b


BUILDERS = {
    "loss_batch": case_loss_batch,
    "2d64x4": lambda cuda: case_grid(cuda, 64, 4),
    "padded_empty": case_padded_empty,
    "padded_shuffled": case_padded_shuffled,
    "3d32_tril": lambda cuda: case_grid(cuda, 32, 1, models.PreconditionerTrilNet, "poisson3d"),
    "2d316x2": lambda cuda: case_grid(cuda, 316, 2),
}
_CACHE = {}


def case(name, cuda):
    if name not in _CACHE:
        with flag(False):
            _CACHE[name] = BUILDERS[name](cuda)
    return _CACHE[name]


# ---- oracle and fp64 --------------------------------------------------------------------------------------------------
def host(st):
    return st.indices.cpu().numpy().astype(np.int64), st.features[:, 0].detach().cpu().numpy()


def oracle_product(st, vec, transpose, keep=None):
    """ckernels.coo_spmv_batch (a sequential loop) on the sites sorted by (b, row, col), or (b, col, row) transposed."""
    ind, f = host(st)
    if keep is not None:
        ind, f = ind[keep(ind)], f[keep(ind)]
    r, c = (ind[:, 2], ind[:, 1]) if transpose else (ind[:, 1], ind[:, 2])
    order = np.lexsort((c, r, ind[:, 0]))
    return ckernels.coo_spmv_batch(ind[order], f[order], np.asarray(vec.detach().cpu().numpy(), np.float32), transpose)


def oracle_system_matvec(st, v):
    diag = oracle_product(st, v, False, keep=lambda ind: ind[:, 1] == ind[:, 2])
    return (oracle_product(st, v, False) + oracle_product(st, v, True)) - diag


def fp64_product(st, vec, transpose):
    """(y64, sum |terms|, row length) per output entry."""
    ind, f = host(st)
    v = vec.detach().cpu().numpy().astype(np.float64)
    r, c = (ind[:, 2], ind[:, 1]) if transpose else (ind[:, 1], ind[:, 2])
    terms = f.astype(np.float64) * v[ind[:, 0], c]
    y, mag, k = np.zeros_like(v), np.zeros_like(v), np.zeros_like(v)
    np.add.at(y, (ind[:, 0], r), terms)
    np.add.at(mag, (ind[:, 0], r), np.abs(terms))
    np.add.at(k, (ind[:, 0], r), 1.0)
    return y, mag, k


def system_matvec64(st, x):
    """A v in fp64 from the stored lower triangle."""
    ind, f = host(st)
    diag = ind[:, 1] == ind[:, 2]
    v = x.detach().cpu().numpy().astype(np.float64)
    y = fp64_product(st, x, False)[0] + fp64_product(st, x, True)[0]
    np.subtract.at(y, (ind[diag, 0], ind[diag, 1]), f[diag].astype(np.float64) * v[ind[diag, 0], ind[diag, 1]])
    return torch.from_numpy(y).to(x.device)


def llt64(ln, x, b, feats64):
    """sum_b || L L^T x_b - b_b || in fp64 with torch ops (autograd in feats64)."""
    ind = ln.indices.long()
    bb, r, c = ind[:, 0], ind[:, 1], ind[:, 2]

    def mv(vec, transpose):
        src, dst = (r, c) if transpose else (c, r)
        return torch.zeros_like(vec).index_put((bb, dst), feats64 * vec[bb, src], accumulate=True)

    return torch.linalg.vector_norm(mv(mv(x, True), False) - b, dim=1)


def frobenius_grad(ln, x, b):
    feats = ln.features.detach().clone().requires_grad_(True)
    loss = metrics.frobenius_loss(ln.replace_feature(feats), x, b)
    (g,) = torch.autograd.grad(loss, feats)
    return loss.detach(), g


def hutchinson_grad(st, ln, v):
    feats = ln.features.detach().clone().requires_grad_(True)
    loss = metrics.hutchinson_trace(st, ln.replace_feature(feats), v)
    (g,) = torch.autograd.grad(loss, feats)
    return loss.detach(), g


def subsystem(st, s):
    keep = st.indices[:, 0] == s
    ind = st.indices[keep].clone()
    ind[:, 0] = 0
    return models.SparseConvTensor(st.features[keep], ind, st.spatial_shape, 1), keep


CASE_NAMES = list(BUILDERS)


# ---- 1. products are the oracle's sequential loop on sorted sites ------------------------------------------------------
@pytest.mark.parametrize("name", CASE_NAMES)
def test_products_are_the_sorted_oracle(cuda, deterministic, name):
    st, ln, x, b = case(name, cuda)
    for transpose in (False, True):
        got = utils.sparse_matvec_mul(ln, x, transpose=transpose)
        assert np.array_equal(got.cpu().numpy().view(np.int32), oracle_product(ln, x, transpose).view(np.int32))
        y64, mag, k = fp64_product(ln, x, transpose)
        err = np.abs(got.cpu().numpy().astype(np.float64) - y64)
        assert np.all(err <= (k + 2) * U * mag), float(np.max(err - (k + 2) * U * mag))
    av = metrics.system_matvec(st, x)
    assert np.array_equal(av.cpu().numpy().view(np.int32), oracle_system_matvec(st, x).view(np.int32))
    # the loss's own products: t = L^T x, r = L t - b
    sites = utils.SortedSites(ln)
    _, _, t, r = utils.llt_residual(sites, utils.site_features(ln, cuda), x[:, None], b[:, None])
    t_want = oracle_product(ln, x, True)
    r_want = oracle_product(ln, torch.from_numpy(t_want), False) - b.cpu().numpy()
    assert np.array_equal(t[:, 0].cpu().numpy().view(np.int32), t_want.view(np.int32))
    assert np.array_equal(r[:, 0].cpu().numpy().view(np.int32), r_want.view(np.int32))


def test_known_answer_under_the_flag(cuda, deterministic):
    indices = torch.tensor([[0, 0, 0], [0, 0, 1], [0, 1, 0], [0, 1, 1], [0, 2, 2],
                            [1, 0, 1], [1, 0, 2], [1, 1, 0], [1, 1, 1], [1, 2, 1]]).int()
    features = torch.tensor([[1, 2, 3, 4, 5, 2, 3, 1, 4, 5]]).T.float()
    batch = models.SparseConvTensor(features.to(cuda), indices.to(cuda), [3, 3], 2)
    vectors_ = torch.tensor([[1, 2, 3], [1, -1, 1]]).float().to(cuda)
    out = utils.sparse_matvec_mul(batch, vectors_, transpose=False)
    assert torch.equal(out.cpu(), torch.tensor([[5, 11, 15], [1, -3, -5]]).float())
    out_t = utils.sparse_matvec_mul(batch, vectors_, transpose=True)
    assert np.array_equal(out_t.cpu().numpy(), oracle_product(batch, vectors_, True))


def test_residual_spans_several_chunks(cuda):
    st, _, _, _ = case("2d316x2", cuda)
    chunk = int(_lib.lib().dp_llt_residual_chunk_rows())
    assert st.spatial_shape[0] >= 4 * chunk, (st.spatial_shape, chunk)


# ---- 2. the order of the input's sites does not matter -----------------------------------------------------------------
def test_shuffled_sites_give_the_same_bits(cuda, deterministic):
    st, ln, x, b = case("padded_empty", cuda)
    st_s, ln_s, _, _ = case("padded_shuffled", cuda)
    _, order = shuffle(ln, 2)
    for transpose in (False, True):
        assert same_bits(utils.sparse_matvec_mul(ln_s, x, transpose), utils.sparse_matvec_mul(ln, x, transpose))
    assert same_bits(metrics.system_matvec(st_s, x), metrics.system_matvec(st, x))
    loss, g = frobenius_grad(ln, x, b)
    loss_s, g_s = frobenius_grad(ln_s, x, b)
    assert same_bits(loss_s, loss) and same_bits(g_s, g[order])
    loss, g = hutchinson_grad(st, ln, x)
    loss_s, g_s = hutchinson_grad(st_s, ln_s, x)
    assert same_bits(loss_s, loss) and same_bits(g_s, g[order])


# ---- 3. two evaluations, the same bits ---------------------------------------------------------------------------------
def evaluate_all(st, ln, x, b, probes):
    out = []
    feats = ln.features.detach().clone().requires_grad_(True)
    vec = x.clone().requires_grad_(True)
    lf = ln.replace_feature(feats)
    for transpose in (False, True):
        y = utils.sparse_matvec_mul(lf, vec, transpose)
        gf, gv = torch.autograd.grad((y * b).sum(), (feats, vec))
        out += [y.detach(), gf, gv]
    out += list(frobenius_grad(ln, x, b)) + list(hutchinson_grad(st, ln, x))
    feats = ln.features.detach().clone().requires_grad_(True)
    gen = torch.Generator(device=x.device).manual_seed(3)
    loss = metrics.inverse_loss(st, ln.replace_feature(feats), probes=probes, generator=gen)
    out += [loss.detach(), torch.autograd.grad(loss, feats)[0]]
    return out


@pytest.mark.parametrize("name", CASE_NAMES)
def test_two_evaluations_are_the_same_bits(cuda, deterministic, name):
    st, ln, x, b = case(name, cuda)
    probes = None if name == "loss_batch" else 4
    first, second = evaluate_all(st, ln, x, b, probes), evaluate_all(st, ln, x, b, probes)
    for i, (a, c) in enumerate(zip(first, second)):
        assert same_bits(a, c), i
        assert torch.isfinite(a).all(), i


# ---- 4. a system alone and in a batch ----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["loss_batch", "2d64x4", "padded_empty", "2d316x2"])
def test_batch_independence(cuda, deterministic, name):
    st, ln, x, b = case(name, cuda)
    feats = ln.features.detach().clone().requires_grad_(True)
    loss, terms = metrics.llt_loss(ln.replace_feature(feats), x[:, None], b[:, None])
    (g,) = torch.autograd.grad(loss, feats)
    _, hut_terms = metrics.llt_loss(ln, x[:, None], metrics.system_matvec(st, x)[:, None], mean=True)
    for s in range(st.batch_size):
        ln_s, keep = subsystem(ln, s)
        st_s, _ = subsystem(st, s)
        f_s = ln_s.features.detach().clone().requires_grad_(True)
        loss_s, terms_s = metrics.llt_loss(ln_s.replace_feature(f_s), x[s:s + 1, None], b[s:s + 1, None])
        assert same_bits(terms_s[0], terms[s]) and same_bits(loss_s, terms[s]), s
        if f_s.numel():
            (g_s,) = torch.autograd.grad(loss_s, f_s)
            assert same_bits(g_s, g[keep]), s
        _, hut_s = metrics.llt_loss(ln_s, x[s:s + 1, None], metrics.system_matvec(st_s, x[s:s + 1])[:, None], mean=True)
        assert same_bits(hut_s[0], hut_terms[s]), s


# ---- 5. accuracy: at least as close to fp64 as the atomic path ---------------------------------------------------------
@pytest.mark.parametrize("name", CASE_NAMES)
def test_as_accurate_as_the_atomic_path(cuda, name):
    st, ln, x, b = case(name, cuda)
    with flag(False):
        atomic = frobenius_grad(ln, x, b) + hutchinson_grad(st, ln, x)
        f64 = ln.features[:, 0].detach().double().requires_grad_(True)
        fro64 = llt64(ln, x.double(), b.double(), f64).sum()
        (gf64,) = torch.autograd.grad(fro64, f64)
        av = system_matvec64(st, x)
        f64h = ln.features[:, 0].detach().double().requires_grad_(True)
        hut64 = llt64(ln, x.double(), av, f64h).mean()
        (gh64,) = torch.autograd.grad(hut64, f64h)
    with flag(True):
        det = frobenius_grad(ln, x, b) + hutchinson_grad(st, ln, x)
    refs = [fro64.detach(), gf64, hut64.detach(), gh64]
    for what, d, a, ref in zip(("frobenius", "d frobenius", "hutchinson", "d hutchinson"), det, atomic, refs):
        d, a = d.double().reshape(-1), a.double().reshape(-1)
        ref = ref.reshape(-1)
        e_det = float(torch.linalg.vector_norm(d - ref))
        e_atomic = float(torch.linalg.vector_norm(a - ref))
        scale = float(torch.linalg.vector_norm(ref))
        assert e_det <= max(2 * e_atomic, (1e-6 if d.numel() == 1 else 1e-5) * scale), (what, e_det, e_atomic, scale)


# ---- 6. the reference's golden values under the flag -------------------------------------------------------------------
def test_golden_values_under_the_flag(cuda):
    golden = json.loads((Path(__file__).parent / "golden" / "metrics_golden.json").read_text())
    st, ln, x, b = case("loss_batch", cuda)
    torch.manual_seed(7)
    vector = torch.randn(st.batch_size, st.spatial_shape[0]).to(cuda)
    with flag(False):
        est_atomic = metrics.inverse_loss(st, ln, probes=256, generator=torch.Generator(device=cuda).manual_seed(1))
    with flag(True):
        assert float(metrics.frobenius_loss(ln, x, b)) == pytest.approx(golden["frobenius_loss"], rel=1e-5)
        assert float(metrics.inverse_loss(st, ln)) == pytest.approx(golden["inverse_loss"], rel=1e-4)
        assert float(metrics.hutchinson_trace(st, ln, vector)) == pytest.approx(golden["hutchinson_trace_seed7"], rel=1e-5)
        est = metrics.inverse_loss(st, ln, probes=256, generator=torch.Generator(device=cuda).manual_seed(1))
    assert float(est) == pytest.approx(float(est_atomic), rel=1e-5)


# ---- 7. zero residual ---------------------------------------------------------------------------------------------------
def test_zero_residual_gives_zero_term_and_gradient(cuda, deterministic):
    st, ln, x, b = case("padded_empty", cuda)
    feats = ln.features.detach().clone().requires_grad_(True)
    loss, terms = metrics.llt_loss(ln.replace_feature(feats), x[:, None], b[:, None])
    (g,) = torch.autograd.grad(loss, feats)
    assert float(terms[1]) == 0.0 and float(terms[0]) > 0 and float(terms[2]) > 0
    assert torch.isfinite(g).all() and torch.isfinite(loss)
    # a zero residual in a system that has sites: L = 0 and b = 0
    zero = ln.replace_feature(torch.zeros_like(ln.features).requires_grad_(True))
    loss0 = metrics.frobenius_loss(zero, x, torch.zeros_like(b))
    (g0,) = torch.autograd.grad(loss0, zero.features)
    assert float(loss0.detach()) == 0.0 and torch.equal(g0, torch.zeros_like(g0))


# ---- 8. refused inputs --------------------------------------------------------------------------------------------------
def test_refused_inputs(cuda, deterministic):
    st, ln, x, b = case("loss_batch", cuda)
    dup = models.SparseConvTensor(torch.cat([ln.features, ln.features[:1]]), torch.cat([ln.indices, ln.indices[:1]]),
                                  ln.spatial_shape, ln.batch_size)
    with pytest.raises(_lib.DpcgError):
        metrics.frobenius_loss(dup, x, b)
    with pytest.raises(_lib.DpcgError):
        utils.sparse_matvec_mul(dup, x, transpose=False)
    with pytest.raises(ValueError):
        metrics.frobenius_loss(ln, x.clone().requires_grad_(True), b)
    with pytest.raises(ValueError):
        metrics.hutchinson_trace(st.replace_feature(st.features.clone().requires_grad_(True)), ln, x)


# ---- 9. with the flag off nothing of this runs ------------------------------------------------------------------------
def spy(monkeypatch, module, names):
    calls = {name: 0 for name in names}
    for name in names:
        fn = getattr(module, name)

        def wrapped(*args, _fn=fn, _name=name, **kwargs):
            calls[_name] += 1
            return _fn(*args, **kwargs)

        monkeypatch.setattr(module, name, wrapped)
    return calls


@pytest.mark.parametrize("enabled", [False, True])
def test_path_follows_the_flag(cuda, monkeypatch, enabled):
    st, ln, x, b = case("loss_batch", cuda)
    new = spy(monkeypatch, utils, ["_sorted_spmv", "system_matvec_sorted", "llt_residual", "llt_residual_grad"])
    old = spy(monkeypatch, utils, ["_coo_spmv"])
    with flag(enabled):
        frobenius_grad(ln, x, b)
        hutchinson_grad(st, ln, x)
        metrics.inverse_loss(st, ln, probes=2)
        utils.sparse_matvec_mul(ln, x, transpose=True)
    if enabled:
        assert all(new.values()) and old["_coo_spmv"] == 0, (new, old)
    else:
        assert not any(new.values()) and old["_coo_spmv"] > 0, (new, old)


# ---- 10. a training run repeats bit for bit ----------------------------------------------------------------------------
def test_training_run_repeats_bit_for_bit(cuda, deterministic):
    st = synthetic.make_batch("poisson2d", 32, list(range(8)), device=cuda)[0]
    x, b = vectors(st, seed=5)
    runs = []
    for _ in range(2):
        net = seeded_net(device=cuda)
        tnet = models.TrainableNet(net)
        adam = torch.optim.Adam(net.parameters(), lr=1e-3)
        losses = []
        for _ in range(20):
            adam.zero_grad()
            loss = metrics.frobenius_loss(tnet(st), x, b)
            loss.backward()
            adam.step()
            losses.append(loss.detach().clone())
        runs.append((torch.stack(losses), [p.detach().clone() for p in net.parameters()]))
    (l1, p1), (l2, p2) = runs
    assert same_bits(l1, l2)
    assert all(same_bits(a, c) for a, c in zip(p1, p2))
    assert float(l1[-1]) < float(l1[0])
