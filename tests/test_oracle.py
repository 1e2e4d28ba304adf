"""CPU tests: pin the oracle against the reference's own vectors and against what the reference executes.

Nothing here touches CUDA. What the reference produced is committed in tests/golden/ (the make_*.py generators there
record how).
"""
import json
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

import helpers
from oracle import ckernels, operators, pcg
from oracle import sparse as osp

GOLDEN = json.loads((Path(__file__).parent / "golden" / "pcg_golden.json").read_text())


def iteration_tolerance(iterations: int) -> int:
    """The reference is itself reproducible only to ~±1-3 iterations on long solves (its own dense-A vs CSR-A runs,
    its explicit-fp32 vs factored M, and MKL's thread-count-dependent reductions differ by that much, see
    tests/golden/pcg_golden.json), so parity is +-1 up to 200 iterations and +-0.5 % beyond."""
    return max(1, int(np.ceil(0.005 * iterations)))


def build_operator(p, name):
    if name == "identity":
        return operators.Identity()
    if name == "jacobi":
        return operators.Jacobi(osp.to_scipy(*p.A).diagonal())
    if name == "multiply":
        return operators.FactoredMultiply(*p.L)
    if name == "explicit":
        return osp.explicit_product(*p.L)
    if name == "ic0_solve":
        return operators.FactoredSolve(*helpers.ic0_factor(p))
    raise KeyError(name)


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=lambda c: f"{c['kind']}{c['side']}-{c['net']}-{c['precond']}-{c['max_iter']}")
def test_oracle_matches_reference_golden(case):
    """oracle.pcg reproduces the iteration counts the unmodified reference produced on the same operands."""
    p = helpers.problem(case["kind"], case["side"], 0, 0.5, case["net"])
    assert p.n == case["n"] and len(p.A[1]) == case["nnz_a"] and len(p.L[1]) == case["nnz_l"]
    assert float(p.b.sum()) == case["b_checksum"] and float(np.sum(p.A[2])) == case["a_checksum"]
    np.testing.assert_allclose(float(np.sum(p.L[2])), case["l_checksum"], rtol=1e-6)  # CNN values: fp32 kernels
    result = pcg.preconditioned_conjugate_gradient(osp.to_torch_csr(*p.A), p.b, build_operator(p, case["precond"]),
                                                   max_iter=case["max_iter"])
    assert result.info == 0
    assert abs(result.iterations - case["iterations"]) <= iteration_tolerance(case["iterations"])
    if case["iterations"] < case["max_iter"]:
        assert result.res < 1e-8 <= result.history[-2]
        a = osp.to_scipy(*p.A)
        true_rel = np.linalg.norm(a @ result.x_hat.numpy() - p.b.numpy()) / np.linalg.norm(p.b.numpy())
        assert true_rel < 2e-4  # sqrt(rtol) with drift margin
    else:
        assert result.iterations == case["max_iter"]


def test_sparse_matvec_mul_known_answer():
    """The reference's only known-answer vector, tests/test_utils.py:11-41."""
    indices = np.array([[0, 0, 0], [0, 0, 1], [0, 1, 0], [0, 1, 1], [0, 2, 2],
                        [1, 0, 1], [1, 0, 2], [1, 1, 0], [1, 1, 1], [1, 2, 1]], np.int32)
    features = np.array([1, 2, 3, 4, 5, 2, 3, 1, 4, 5], np.float32)
    vectors = np.array([[1, 2, 3], [1, -1, 1]], np.float32)
    out = osp.sparse_matvec_mul(indices, features, vectors, transpose=False)
    assert np.array_equal(out, np.array([[5, 11, 15], [1, -3, -5]], np.float32))
    dense = np.zeros((2, 3, 3), np.float32)
    dense[indices[:, 0], indices[:, 1], indices[:, 2]] = features
    out_t = osp.sparse_matvec_mul(indices, features, vectors, transpose=True)
    assert np.array_equal(out_t, np.einsum("bji,bj->bi", dense, vectors))


@pytest.mark.parametrize("kind,side,net", [("poisson2d", 16, "net"), ("poisson3d", 6, "tril")])
def test_assembly_oracle_is_what_the_harness_builds(kind, side, net):
    """test.py:65-68 and test.py:103-105 executed literally (dense) vs the sparse restatement."""
    p = helpers.problem(kind, side, 0, 0.5, net)
    dense = p.systems_tril.dense()[0, 0, : p.n, : p.n]
    dense = dense + torch.tril(dense, -1).T
    want = dense.to(torch.float64).to_sparse_csr()
    assert np.array_equal(want.crow_indices().numpy(), p.A[0]) and np.array_equal(want.col_indices().numpy(), p.A[1])
    assert np.array_equal(want.values().numpy(), p.A[2])
    lower = p.learned.dense()[0, 0, : p.n, : p.n].to(torch.float64).to_sparse_csr()
    assert np.array_equal(lower.crow_indices().numpy(), p.L[0]) and np.array_equal(lower.col_indices().numpy(), p.L[1])
    assert np.array_equal(lower.values().numpy(), p.L[2])
    lt = osp.transpose_csr(*p.L)
    assert (osp.to_scipy(*lt) != osp.to_scipy(*p.L).T).nnz == 0


def test_learned_factor_structure():
    """The structural properties the reference tests on the CNN output, tests/test_model.py:31-42."""
    p = helpers.problem("poisson2d", 16, 0, 0.5, "net")
    lower = p.learned.dense()[0, 0]
    assert lower.shape == torch.Size(p.systems_tril.spatial_shape)
    assert torch.all(lower.diag() != 0)
    assert torch.all(lower.triu(diagonal=1) == 0)
    assert torch.any(lower.tril(diagonal=-1) != 0)
    m = lower.double() @ lower.double().T
    assert torch.all(m == m.T)
    eig = torch.linalg.eigvalsh(m)
    assert torch.all(eig > 0)
    # SURVEY D3: the non-submanifold net dilates the pattern (5x5 box), the 1x1 stand-in keeps tril(A)
    assert len(p.L[1]) > 2 * len(p.T[1])
    q = helpers.problem("poisson2d", 16, 0, 0.5, "tril")
    assert np.array_equal(q.L[0], q.T[0]) and np.array_equal(q.L[1], q.T[1])


@pytest.mark.parametrize("kind,side", [("poisson2d", 24), ("poisson3d", 9)])
def test_c_kernels_against_scipy(kind, side):
    p = helpers.problem(kind, side, 0, 0.5, None)
    a = osp.to_scipy(*p.A)
    x = np.random.default_rng(3).standard_normal(p.n)
    assert np.array_equal(ckernels.spmv_csr(*p.A, x), a @ x)  # bit-exact: same sequential sums
    lval = ckernels.ic0(*p.T)
    l = osp.to_scipy(p.T[0], p.T[1], lval)
    pattern = a.copy()
    pattern.data[:] = 1
    defect = (l @ l.T).multiply(pattern) - a
    assert abs(defect).max() < 1e-13 * abs(a).max()  # IC(0) property: (L L^T)_ij = A_ij on the pattern
    y = ckernels.sptrsv_lower(p.T[0], p.T[1], lval, x)
    y_ref = spla.spsolve_triangular(l, x, lower=True)
    assert np.abs(y - y_ref).max() <= 1e-12 * np.abs(y_ref).max()
    lt = osp.transpose_csr(p.T[0], p.T[1], lval)
    z = ckernels.sptrsv_upper(*lt, y)
    z_ref = spla.spsolve_triangular(sp.csr_matrix(l.T), y_ref, lower=False)
    assert np.abs(z - z_ref).max() <= 1e-12 * np.abs(z_ref).max()


def test_levels_oracle():
    for row in GOLDEN["levels"]:
        p = helpers.problem(row["kind"], row["side"], 0, 0.5, None)
        level, perm, level_ptr = ckernels.levels(p.T[0], p.T[1])
        assert len(level_ptr) - 1 == row["nlevels"]
        side = row["side"]
        assert row["nlevels"] == (2 * side - 1 if row["kind"] == "poisson2d" else 3 * side - 2)  # BASELINE.md §2
        # definition, checked independently
        for i in range(p.n):
            deps = [j for j in p.T[1][p.T[0][i]: p.T[0][i + 1]] if j < i]
            assert level[i] == (1 + max(level[j] for j in deps) if deps else 0)
        assert np.array_equal(np.sort(perm), np.arange(p.n)) and np.all(np.diff(level[perm]) >= 0)
        for l in range(len(level_ptr) - 1):
            seg = perm[level_ptr[l]: level_ptr[l + 1]]
            assert np.all(level[seg] == l) and np.all(np.diff(seg) > 0)  # stable: ascending rows inside a level
        tt = osp.transpose_csr(*p.T)
        level_u, _, lp_u = ckernels.levels(tt[0], tt[1], upper=True)
        assert len(lp_u) == len(level_ptr) and level_u[p.n - 1] == 0


def test_synthetic_systems_are_spd_and_fp32_exact():
    for kind, side in [("poisson2d", 12), ("poisson3d", 6)]:
        p = helpers.problem(kind, side, 3, 0.5, None)
        a = osp.to_scipy(*p.A).toarray()
        assert np.array_equal(a, a.T)
        assert np.linalg.eigvalsh(a).min() > 0
        assert np.array_equal(p.A[2], p.A[2].astype(np.float32).astype(np.float64))  # data_set.py:121 round trip
        assert np.all(np.abs(p.b.numpy()) <= 1) and p.b.dtype == torch.float64
    a5 = helpers.problem("poisson2d", 12, 0, 0.5, None)
    assert len(a5.A[1]) == 5 * 144 - 4 * 12 and len(a5.T[1]) == 3 * 144 - 2 * 12  # SURVEY §8 nnz formulas
    a7 = helpers.problem("poisson3d", 6, 0, 0.5, None)
    assert len(a7.A[1]) == 7 * 216 - 6 * 36 and len(a7.T[1]) == 4 * 216 - 3 * 36


def test_kappa_estimate_from_cg_coefficients_matches_the_dense_spectrum():
    """SURVEY §8f-4: the Lanczos tridiagonal built from a/beta of the reference loop (cg.py:78,82) has the extreme
    eigenvalues of M A; its ratio is what replaces the dense torch.linalg.cond of test.py:111-113 (equal to it for
    M = I, the symmetric-preconditioning condition number otherwise)."""
    from deeppreconditioning_b200 import spectrum

    p = helpers.problem("poisson2d", 16, 0, 0.5, "net")
    A = osp.to_scipy(*p.A).toarray()
    At = osp.to_torch_csr(*p.A)
    L = osp.to_scipy(*p.L).toarray()
    for M, dense, iters in [(operators.Identity(), np.eye(p.n), 400), (operators.Jacobi(A.diagonal()), np.diag(1 / A.diagonal()), 400),
                            (operators.FactoredMultiply(*p.L), L @ L.T, 2000)]:
        r = pcg.preconditioned_conjugate_gradient(At, p.b, M, rtol=1e-20, max_iter=iters)
        assert len(r.alphas) == len(r.betas) == r.iterations and r.betas[0] == 0.0
        lam = np.linalg.eigvals(dense @ A).real
        lo, hi = spectrum.ritz_extremes(r.alphas, r.betas)
        assert lo == pytest.approx(lam.min(), rel=1e-8) and hi == pytest.approx(lam.max(), rel=1e-8)
        assert spectrum.kappa_estimate(r.alphas, r.betas) == pytest.approx(lam.max() / lam.min(), rel=1e-8)
    assert spectrum.kappa_estimate(r.alphas[:1], r.betas[:1]) == 1.0  # one body: a single Ritz value
    assert np.isnan(spectrum.kappa_estimate([], []))
    # at the reference's tolerance the Ritz values are still inside the spectrum: a lower bound
    r8 = pcg.preconditioned_conjugate_gradient(At, p.b, operators.Identity(), max_iter=400)
    k8 = spectrum.kappa_estimate(r8.alphas, r8.betas)
    assert 0.5 * np.linalg.cond(A) < k8 <= np.linalg.cond(A) * (1 + 1e-9)


@pytest.mark.parametrize("kind,side", [("poisson3d", 9), ("poisson2d", 23)])
def test_level_ordering_commutes_with_the_path_on_the_oracle(kind, side):
    """The claims behind precond.LevelOrdering, checked with the CPU restatement only: level order is a topological
    order of tril(A)'s graph, so P tril(A) P^T is the lower triangle of P A P^T and its own levels ascend along the rows
    (level-sorted permutation = identity); IC(0) commutes with the renumbering (bitwise on stencils: no row pair shares two
    neighbours); forward substitution in level order is bitwise the natural one; walking the rows of L^T from the last to
    the first is a valid backward order; and PCG on the renumbered system is the same iteration as cg.py's on the
    natural one (same count, same solution to 1e-8)."""
    p = helpers.problem(kind, side, 0, 0.5, None)
    level, perm, level_ptr = ckernels.levels(p.T[0], p.T[1], False)
    inv = np.empty_like(perm)
    inv[perm] = np.arange(p.n, dtype=perm.dtype)
    A = osp.to_scipy(*p.A)
    T = osp.to_scipy(*p.T)
    A_l = A[perm][:, perm].tocsr()
    T_l = T[perm][:, perm].tocsr()
    for m in (A_l, T_l):
        m.sort_indices()
    assert (sp.triu(T_l, 1)).nnz == 0 and (sp.tril(A_l) != T_l).nnz == 0
    level_l, perm_l, level_ptr_l = ckernels.levels(T_l.indptr, T_l.indices, False)
    assert np.array_equal(perm_l, np.arange(p.n)) and np.array_equal(level_ptr_l, level_ptr)
    assert np.array_equal(level_l, level[perm])
    # IC(0)
    f = ckernels.ic0(*p.T)
    f_l = ckernels.ic0(T_l.indptr, T_l.indices, T_l.data)
    F = sp.csr_matrix((f, p.T[1], p.T[0]), shape=(p.n, p.n))
    want = F[perm][:, perm].tocsr()
    want.sort_indices()
    assert np.array_equal(want.indices, T_l.indices) and np.array_equal(want.data.view(np.int64), f_l.view(np.int64))
    # triangular solves
    b = p.b.numpy()
    y = ckernels.sptrsv_lower(p.T[0], p.T[1], f, b)
    y_l = ckernels.sptrsv_lower(T_l.indptr, T_l.indices, f_l, b[perm])
    assert np.array_equal(y_l, y[perm])
    U_l = sp.csr_matrix((f_l, T_l.indices, T_l.indptr), shape=(p.n, p.n)).T.tocsr()
    U_l.sort_indices()
    z_l = ckernels.sptrsv_upper(U_l.indptr, U_l.indices, U_l.data, y_l)
    Ut = F.T.tocsr()
    Ut.sort_indices()
    z = ckernels.sptrsv_upper(Ut.indptr, Ut.indices, Ut.data, y)
    assert np.array_equal(z_l, z[perm])
    rows = np.repeat(np.arange(p.n), np.diff(U_l.indptr))
    assert np.all(U_l.indices >= rows), "every dependency of row i of L^T is a row j > i: last-to-first is a valid order"
    # the loop itself
    nat = pcg.preconditioned_conjugate_gradient(osp.to_torch_csr(*p.A), p.b, operators.FactoredSolve(p.T[0], p.T[1], f),
                                                max_iter=3000)
    lvl = pcg.preconditioned_conjugate_gradient(osp.to_torch_csr(A_l.indptr, A_l.indices, A_l.data), p.b[torch.from_numpy(perm).long()],
                                                operators.FactoredSolve(T_l.indptr, T_l.indices, f_l), max_iter=3000)
    assert lvl.iterations == nat.iterations
    x_back = torch.empty_like(lvl.x_hat)
    x_back[torch.from_numpy(perm).long()] = lvl.x_hat
    assert torch.linalg.vector_norm(x_back - nat.x_hat) <= 1e-8 * torch.linalg.vector_norm(nat.x_hat)


# ---- threshold incomplete Cholesky (stands in for ilupp.icholt, test.py:86): host routine vs its restatement ------------
def _icholt_host(rowptr, col, val, fill_in, threshold):
    """dp_icholt_host through ctypes: host pointers only, no GPU needed."""
    from deeppreconditioning_b200 import _lib, build

    build.build()
    n = len(rowptr) - 1
    rowptr, col, val = (np.ascontiguousarray(a) for a in (np.asarray(rowptr, np.int32), np.asarray(col, np.int32), np.asarray(val, np.float64)))
    cap = len(col) + n * fill_in + 1
    rp, c, v, nnz = np.empty(n + 1, np.int32), np.empty(cap, np.int32), np.empty(cap, np.float64), np.zeros(1, np.int64)
    status = _lib.lib().dp_icholt_host(n, rowptr.ctypes.data, col.ctypes.data, val.ctypes.data, fill_in, threshold,
                                       rp.ctypes.data, c.ctypes.data, v.ctypes.data, cap, nnz.ctypes.data)
    return status, rp, c[: int(nnz[0])], v[: int(nnz[0])]


@pytest.mark.parametrize("kind,side", [("poisson2d", 16), ("poisson3d", 6), ("poisson2d", 33)])
@pytest.mark.parametrize("fill_in,threshold", [(1, 0.1), (0, 0.0), (3, 0.01), (1000, 0.0)])
def test_icholt_host_is_its_restatement(kind, side, fill_in, threshold):
    """csrc/icholt.cu == oracle/icholt.py bit for bit (same operations, same order), for the reference's default
    arguments (1, 0.1), the no-fill corner, a generous setting and the complete factorisation."""
    from oracle import icholt as oict

    p = helpers.problem(kind, side, 0, 0.5, None)
    status, rp, c, v = _icholt_host(*p.T, fill_in, threshold)
    assert status == 0
    want = oict.icholt(*p.T, fill_in, threshold)
    assert np.array_equal(rp, want[0]) and np.array_equal(c, want[1])
    assert np.array_equal(v.view(np.int64), want[2].view(np.int64))
    L = osp.to_scipy(rp, c, v)
    assert (L.diagonal() > 0).all() and sp.triu(L, 1).nnz == 0
    assert np.all(np.diff(rp) - 1 <= np.diff(p.T[0]) - 1 + fill_in)  # rule 2: at most nnz(A_i) + fill_in off-diagonals
    a = osp.to_scipy(*p.A)
    if fill_in == 1000 and threshold == 0.0:  # nothing dropped: the complete Cholesky factor
        assert abs(L @ L.T - a).max() < 1e-12 * abs(a).max()
    # a usable preconditioner: fewer PCG iterations than Jacobi through the oracle loop
    jac = pcg.preconditioned_conjugate_gradient(osp.to_torch_csr(*p.A), p.b, operators.Jacobi(a.diagonal()), max_iter=3000)
    ict = pcg.preconditioned_conjugate_gradient(osp.to_torch_csr(*p.A), p.b, operators.FactoredSolve(rp, c, v), max_iter=3000)
    assert ict.iterations < jac.iterations and ict.res < 1e-8


def test_icholt_host_rejects_bad_structure():
    p = helpers.problem("poisson2d", 8, 0, 0.5, None)
    rp, c, v = (np.array(a) for a in p.T)
    assert _icholt_host(rp, c, -v, 1, 0.1)[0] == 5            # negative definite: non-positive pivot
    c_bad = c.copy()
    c_bad[rp[3 + 1] - 1] = 2                                  # row 3 without its diagonal in last place
    assert _icholt_host(rp, c_bad, v, 1, 0.1)[0] == 5
    from deeppreconditioning_b200 import _lib
    assert _lib.lib().dp_icholt_host(-1, None, None, None, 0, 0.0, None, None, None, 0, None) == 1


def test_a_norm_error_history_from_cg_coefficients():
    """conjugate_gradient's error column (cg.py:28-30,42-44) from the final error and a_k <r_k, r_k> (the identity the
    CUDA drop-in uses instead of an SpMV per iteration) against the reference's literal evaluation."""
    p = helpers.problem("poisson2d", 32, 0, 0.5, None)
    A = osp.to_torch_csr(*p.A)
    x_true = torch.from_numpy(spla.spsolve(osp.to_scipy(*p.A).tocsc(), p.b.numpy()))
    errors, x = pcg.conjugate_gradient(A, p.b, x_true=x_true, max_iter=3000)
    run = pcg.preconditioned_conjugate_gradient(A, p.b, operators.Identity(), max_iter=3000)
    assert len(run.history) == len(errors)
    bb = float(torch.inner(p.b, p.b))
    e = x - x_true
    tail = np.zeros(len(errors))
    tail[:-1] = np.cumsum([a * r * bb for a, r in zip(run.alphas, run.history[:-1])][::-1])[::-1]
    tail += float(torch.inner(e, A @ e))
    np.testing.assert_allclose(tail, [float(err) for err, _ in errors], rtol=1e-9)


# ---- training losses (SURVEY §8f-3): the dense restatement against the reference module itself --------------------------
def _loss_batch():
    from deeppreconditioning_b200 import model as models, synthetic

    st, sol, rhs, sizes = synthetic.make_batch("poisson2d", 9, [0, 1, 2])
    torch.manual_seed(69)
    with torch.no_grad():
        learned = models.PreconditionerNet(models.DEFAULT_CHANNELS)(st)
    torch.manual_seed(5)
    return st, learned, torch.randn_like(rhs), rhs


def test_metrics_oracle_matches_golden():
    """oracle/metrics.py against the values the unmodified reference metrics.py:13-77 produced on this seeded batch
    (tests/golden/make_metrics_golden.py; the Hutchinson probe is randn(systems.shape[:2]) after manual_seed(7))."""
    from oracle import metrics as om

    golden = json.loads((Path(__file__).parent / "golden" / "metrics_golden.json").read_text())
    st, learned, solution, rhs = _loss_batch()
    lower, tril = learned.dense()[:, 0], st.dense()[:, 0]
    assert float(om.frobenius_loss(lower, solution, rhs)) == pytest.approx(golden["frobenius_loss"], rel=1e-5)
    assert float(om.inverse_loss(tril, lower)) == pytest.approx(golden["inverse_loss"], rel=1e-5)
    torch.manual_seed(7)
    vector = torch.randn(tril.shape[:2])
    assert float(om.hutchinson_trace(tril, lower, vector)) == pytest.approx(golden["hutchinson_trace_seed7"], rel=1e-5)


def test_pack_oracle_round_trip():
    """The packed stream format is lossless where it says so: columns and values rebuild bit for bit; a value beyond fp32
    or a tile wider than 16 bits of columns is reported."""
    p = helpers.problem("poisson2d", 37, 0, 0.5, "net")
    for rowptr, col, val in (p.A, p.L, osp.transpose_csr(*p.L)):
        col16, val32, base, status = osp.pack_csr(rowptr, col, val)
        assert status == 0
        rows = np.repeat(np.arange(len(rowptr) - 1), np.diff(rowptr))
        assert np.array_equal(base[rows // 512, 0] + col16.astype(np.int64), col)
        assert all(col[rowptr[t * 512]:rowptr[min((t + 1) * 512, len(rowptr) - 1)]].max() == b0 + sp - 1 for t, (b0, sp) in enumerate(base))
        assert np.array_equal(val32.astype(np.float64).view(np.int64), np.asarray(val).view(np.int64))
    rowptr, col, val = p.A
    bad = np.array(val, dtype=np.float64)
    bad[5] = 0.1
    assert osp.pack_csr(rowptr, col, bad)[3] == 1
    wide = (np.array([0, 2, 3], np.int32), np.array([0, 70000, 1], np.int32), np.array([1.0, 2.0, 3.0]))
    assert osp.pack_csr(*wide)[3] == 2
