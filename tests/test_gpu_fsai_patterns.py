"""Power patterns of FSAI on the device (dp_csr_pattern_product_*, precond.power_pattern, the "fsai_power" technique).

The symbolic product is integer work, so every pattern is compared bit for bit with the scipy oracle of
test_fsai_patterns_host; FSAI on those patterns is compared bit for bit with oracle_fsai, and PCG with it against the oracle
loop on the bench's 316^2 system.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import helpers
import deeppreconditioning_b200 as dp
from deeppreconditioning_b200 import _lib, model as models, precond, synthetic
from deeppreconditioning_b200.sparse import CsrMatrix
from deeppreconditioning_b200.test import BenchmarkSuite
from oracle import operators, pcg
from oracle import sparse as osp
from test_fsai_host import oracle_factor
from test_fsai_patterns_host import oracle_power_pattern

pytestmark = pytest.mark.gpu


def dev(csr, cuda):
    return CsrMatrix.from_arrays(*csr, device=cuda)


def oracle_product(P, Q, lower):
    """The structural pattern of ``P Q`` (``tril`` of it with ``lower``) by scipy, every value 1.0."""
    Ps, Qs = osp.to_scipy(*P).copy(), osp.to_scipy(*Q).copy()
    Ps.data[:], Qs.data[:] = 1.0, 1.0
    C = Ps @ Qs
    C = sp.tril(C, format="csr") if lower else C.tocsr()
    C.sort_indices()
    return C.indptr.astype(np.int32), C.indices.astype(np.int32), np.ones(C.nnz)


def aat_nnz(L, Lt):
    count = torch.zeros(1, dtype=torch.int64, device=L.device)
    _lib.check(_lib.lib().dp_csr_aat_nnz(L.n, _lib.ptr(L.rowptr), _lib.ptr(L.col), _lib.ptr(Lt.rowptr), _lib.ptr(Lt.col),
                                         _lib.ptr(count), _lib.stream_ptr(L.device)), "dp_csr_aat_nnz")
    return int(count.item())


# ---- patterns ----------------------------------------------------------------------------------------------------------
PATTERN_CASES = [("poisson2d", 64, k) for k in range(1, 6)] + [("poisson2d", 316, 2), ("poisson2d", 316, 3)] + [
    ("poisson3d", 32, k) for k in range(1, 4)]


@pytest.mark.parametrize("kind,side,power", PATTERN_CASES)
def test_power_pattern_is_the_oracle(cuda, kind, side, power):
    p = helpers.problem(kind, side, 0)
    got = precond.power_pattern(dev(p.A, cuda), power)
    want = oracle_power_pattern(p.A, power)
    helpers.assert_csr_equal(got, want)
    longest = int(np.diff(osp.transpose_csr(*want)[0]).max())
    print(f"{kind} {side}: tril(|A|^{power}) {want[1].shape[0] / p.n:.2f} entries per column, longest {longest}")


def test_padded_system(cuda):
    st, _, _, sizes = synthetic.make_batch("poisson2d", 20, [3], pad_to=450)
    assert sizes[0] < 450
    A_host = osp.symmetrise_tril(st.indices.numpy(), st.features.numpy(), 0, 450)
    A = CsrMatrix.from_spconv(helpers.to_device(st, cuda), 450, "symmetrise")
    helpers.assert_csr_equal(A, A_host)
    for power in (2, 3):
        helpers.assert_csr_equal(precond.power_pattern(A, power), oracle_power_pattern(A_host, power))


def test_power_one_is_the_structure_of_tril(cuda):
    p = helpers.problem("poisson2d", 64, 2)
    A = dev(p.A, cuda)
    got, lower = precond.power_pattern(A, 1), A.tril()
    assert torch.equal(got.rowptr, lower.rowptr) and torch.equal(got.col, lower.col)
    assert bool(torch.all(got.val == 1.0))


@pytest.mark.parametrize("lower", [False, True])
def test_product_of_two_patterns(cuda, lower):
    p = helpers.problem("poisson2d", 64, 0, 0.5, "net")
    L, Lt = dev(p.L, cuda), dev(osp.transpose_csr(*p.L), cuda)
    got = precond._pattern_product(L, Lt, lower)
    helpers.assert_csr_equal(got, oracle_product(p.L, osp.transpose_csr(*p.L), lower))
    if not lower:
        assert got.nnz == aat_nnz(L, Lt)  # the density count is the same row union


def long_row_system(n=3000, hub=2200, seed=5):
    """A random SPD pattern (diagonally dominant): rows 0..99 hold only their diagonal, rows 100..n-2 random couplings,
    and row n-1 is coupled to ``hub`` of them, so row n-1 of |A|^2 reaches well over 2000 columns."""
    rng = np.random.default_rng(seed)
    r, c = rng.integers(100, n - 1, size=3 * n), rng.integers(100, n - 1, size=3 * n)
    h = rng.choice(np.arange(100, n - 1), size=hub, replace=False)
    r, c = np.concatenate([r, h]), np.concatenate([c, np.full(hub, n - 1)])
    off = r != c
    M = sp.coo_matrix((np.ones(off.sum()), (r[off], c[off])), shape=(n, n)).tocsr()
    M = ((M + M.T) > 0).astype(np.float64)
    A = sp.diags(np.asarray(M.sum(axis=1)).ravel() + 1.0) - M
    A = A.tocsr()
    A.sort_indices()
    return A.indptr.astype(np.int32), A.indices.astype(np.int32), A.data


def test_long_rows_and_diagonal_rows(cuda):
    A_host = long_row_system()
    n = A_host[0].shape[0] - 1
    assert np.all(np.diff(A_host[0])[:100] == 1)  # rows that hold only a diagonal
    A = dev(A_host, cuda)
    for lower in (False, True):
        want = oracle_product(A_host, A_host, lower)
        helpers.assert_csr_equal(precond._pattern_product(A, A, lower), want)
        longest = int(np.diff(want[0])[n - 1])
        assert longest > 2000, longest  # the general path, far beyond any short-row buffer
    helpers.assert_csr_equal(precond.power_pattern(A, 2), oracle_power_pattern(A_host, 2))


def test_empty_system(cuda):
    empty = CsrMatrix.from_arrays(np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0), device=cuda)
    for power in (1, 2, 3):
        got = precond.power_pattern(empty, power)
        assert got.n == 0 and got.nnz == 0 and got.rowptr.tolist() == [0]


def test_int32_guard(cuda, monkeypatch):
    """46341 rows of P, each with one entry in column 0, times Q whose row 0 is full: 46341^2 = 2,147,488,281 entries
    from kilobytes of input. The total is checked before anything is allocated for the fill."""
    n = 46341
    P = CsrMatrix.from_arrays(np.arange(n + 1, dtype=np.int32), np.zeros(n, np.int32), np.ones(n), device=cuda)
    q_rowptr = np.full(n + 1, n, np.int32)
    q_rowptr[0] = 0
    Q = CsrMatrix.from_arrays(q_rowptr, np.arange(n, dtype=np.int32), np.ones(n), device=cuda)
    calls = []
    monkeypatch.setattr(_lib.lib(), "dp_csr_pattern_product_fill", lambda *args: calls.append(args) or 0)
    with pytest.raises(_lib.DpcgError, match="2147488281"):
        precond._pattern_product(P, Q, False)
    assert not calls


def test_columns_outside_the_matrix(cuda):
    p = helpers.problem("poisson2d", 16, 0)
    A = dev(p.A, cuda)
    for where, value in (("p", p.n), ("q", -1)):
        col = p.A[1].copy()
        col[37] = value
        bad = dev((p.A[0], col, p.A[2]), cuda)
        P, Q = (bad, A) if where == "p" else (A, bad)
        with pytest.raises(_lib.DpcgError, match="outside"):
            precond._pattern_product(P, Q, False)


# ---- FSAI on power patterns ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fp32", [True, False])
@pytest.mark.parametrize("kind,side,power", [("poisson2d", 316, 2), ("poisson2d", 316, 3), ("poisson3d", 32, 2),
                                             ("poisson3d", 32, 3)])
def test_fsai_bitwise_the_oracle(cuda, kind, side, power, fp32):
    p = helpers.problem(kind, side, 0)
    A = dev(p.A, cuda)
    pattern = oracle_power_pattern(p.A, power)
    longest = int(np.diff(osp.transpose_csr(*pattern)[0]).max())
    if kind == "poisson3d" and power == 3:
        assert longest == 32  # the kernel's limit exactly
    M = precond.fsai(A, precond.power_pattern(A, power), fp32=fp32)
    want = oracle_factor(p.A, pattern, fp32)
    helpers.assert_csr_equal(M.L, want)
    helpers.assert_csr_equal(M.Lt, osp.transpose_csr(*want))


def test_fsai_beyond_32_entries_raises(cuda):
    A = dev(helpers.problem("poisson3d", 32, 0).A, cuda)
    with pytest.raises(_lib.DpcgError, match="more than 32 entries"):
        precond.fsai(A, precond.power_pattern(A, 4))  # 65 entries in the longest column


def test_pcg_316_against_the_oracle(cuda):
    p = helpers.problem("poisson2d", 316, 0, 0.5, "net")
    A, b, At = dev(p.A, cuda), p.b.to(cuda), osp.to_torch_csr(*p.A)
    counts = {"tril": dp.pcg_solve(A, b, precond.fsai(A), max_iter=3000).iterations,
              "net": dp.pcg_solve(A, b, precond.fsai(A, dev(p.L, cuda)), max_iter=3000).iterations}
    # The loop sums its dot products in another order than torch, so x is compared at the same iterate. The oracle
    # against itself with every dot product summed in reverse order differs, for k = 2, by 9e-16 at iterate 50, 1e-11 at
    # 150 and 2.2e-8 at 229, its last; for k = 3 by at most 2.3e-15 up to its last iterate, 174. So iterate 50 is held to
    # 1e-8 for both, the last iterate to 1e-6 for k = 2 and to 1e-8 for k = 3.
    for power, last_tol in ((2, 1e-6), (3, 1e-8)):
        M = precond.fsai(A, precond.power_pattern(A, power))
        oracle_m = operators.FactoredMultiply(*oracle_factor(p.A, oracle_power_pattern(p.A, power), True))
        got = dp.pcg_solve(A, b, M, max_iter=3000)
        want = pcg.preconditioned_conjugate_gradient(At, p.b, oracle_m, max_iter=3000)
        assert abs(got.iterations - want.iterations) <= 1, (power, got.iterations, want.iterations)
        counts[power] = got.iterations
        k = min(got.iterations, want.iterations)
        for at, tol in ((50, 1e-8), (k, last_tol)):
            x = got.x_hat if at == got.iterations else dp.pcg_solve(A, b, M, max_iter=at).x_hat
            xo = want.x_hat if at == want.iterations else pcg.preconditioned_conjugate_gradient(At, p.b, oracle_m, max_iter=at).x_hat
            assert torch.linalg.vector_norm(x.cpu() - xo) <= tol * torch.linalg.vector_norm(xo), (power, at)
    print(f"316^2 PCG iterations, FSAI on: tril(A) {counts['tril']}, tril(|A|^2) {counts[2]}, tril(|A|^3) {counts[3]}, "
          f"network pattern {counts['net']}")
    assert counts["tril"] > counts[2] > counts[3]
    assert counts[3] < counts["net"]


def test_packed_stream_and_batches(cuda):
    p = helpers.problem("poisson2d", 316, 0)
    A, b = dev(p.A, cuda), p.b.to(cuda)
    M = precond.fsai(A, precond.power_pattern(A, 3))
    assert M.L.packed() is not None and M.Lt.packed() is not None
    packed = dp.pcg_solve(A, b, M, max_iter=3000)
    plain = dp.pcg_solve(A, b, M, max_iter=3000, pack=False)
    assert packed.iterations == plain.iterations
    assert torch.equal(packed.x_hat.view(torch.int64), plain.x_hat.view(torch.int64))
    q = helpers.problem("poisson2d", 64, 3)
    Aq, bq = dev(q.A, cuda), q.b.to(cuda)
    batch = dp.pcg_solve_batch([(Aq, bq, dp.Jacobi(Aq)), (A, b, M), (Aq, bq, precond.fsai(Aq))], max_iter=3000)
    assert batch[1].iterations == packed.iterations
    assert torch.equal(batch[1].x_hat.view(torch.int64), packed.x_hat.view(torch.int64))


# ---- BenchmarkSuite ----------------------------------------------------------------------------------------------------
def test_benchmark_suite_technique(cuda, tmp_path):
    torch.manual_seed(69)
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS).to(cuda)
    data = synthetic.SyntheticPressureDataSet("poisson2d", 24, number_samples=3, batch_size=1, device=cuda)
    techniques = ("jacobi", "fsai", "fsai_power")
    assert "fsai_power" not in BenchmarkSuite(data, net).techniques  # opt-in only
    suite = BenchmarkSuite(data, net, techniques=techniques, max_iter=5000)
    assert suite.fsai_power == 2
    suite.run()
    suite.dump_csv(tmp_path)
    for name in techniques:
        for store in BenchmarkSuite._STORES:
            assert len(getattr(suite, store)[name]) == 3, (name, store)
        assert all(s == 100 for s in suite.successes[name]) and all(r < 1e-8 for r in suite.residuals[name])
    for k in range(3):
        pk = helpers.problem("poisson2d", 24, k)
        Ls = osp.to_scipy(*oracle_power_pattern(pk.A, 2))
        assert suite.densities["fsai_power"][k] == 100 * (Ls @ Ls.T).nnz / pk.n ** 2
    assert all(a < b for a, b in zip(suite.iterations["fsai_power"], suite.iterations["fsai"]))
    variants = (tmp_path / "variants.csv").read_text()
    assert '\nfsai_power,"FSAI on tril(|A|^2) (GPU), ' in variants
    serial = BenchmarkSuite(data, net, techniques=techniques, max_iter=5000, batch_systems=1)
    serial.run()
    for name in techniques:
        assert serial.iterations[name] == suite.iterations[name] and serial.residuals[name] == suite.residuals[name]
        assert serial.densities[name] == suite.densities[name] and serial.kappas[name] == suite.kappas[name]
    cubed = BenchmarkSuite(data, net, techniques=("fsai_power",), max_iter=5000, fsai_power=3)
    cubed.run()
    cubed.dump_csv(tmp_path / "cubed")
    assert '\nfsai_power,"FSAI on tril(|A|^3) (GPU), ' in (tmp_path / "cubed" / "variants.csv").read_text()
    assert cubed.iterations["fsai_power"] != suite.iterations["fsai_power"]
    assert all(a < b for a, b in zip(cubed.iterations["fsai_power"], suite.iterations["fsai_power"]))
