"""FSAI on the device (dp_fsai_f64, precond.fsai, the "fsai" / "fsai_learned" techniques of BenchmarkSuite).

The kernel and the oracle (tests/fsai_oracle.c: oracle_fsai) run the same arithmetic in the same order with every
operation rounded separately, so the factors are compared bit for bit, in both fp32 modes, on the patterns the comparator
is used with: tril(A) and the factor network's own pattern, in 2-D and 3-D, and a pattern whose columns hold the limit of 32.
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
from test_fsai_host import drop_entry, oracle_factor

pytestmark = pytest.mark.gpu


def band(n, width):
    """Lower pattern with ``width`` entries in every column (fewer in the last ones): L[r, c] for c <= r < c + width."""
    m = sp.diags([np.ones(n - d) for d in range(width)], [-d for d in range(width)], shape=(n, n), format="csr")
    m.sort_indices()
    return m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data


def dev(csr, cuda):
    return CsrMatrix.from_arrays(*csr, device=cuda)


CASES = {
    "2d64_tril": lambda: (helpers.problem("poisson2d", 64, 0), "tril"),
    "2d316_tril": lambda: (helpers.problem("poisson2d", 316, 0), "tril"),
    "2d316_net": lambda: (helpers.problem("poisson2d", 316, 0, 0.5, "net"), "net"),
    "3d32_tril": lambda: (helpers.problem("poisson3d", 32, 0), "tril"),
    "3d32_net": lambda: (helpers.problem("poisson3d", 32, 0, 0.5, "net"), "net"),
    "2d64_band32": lambda: (helpers.problem("poisson2d", 64, 0), "band32"),
}


def pattern_of(p, which):
    return {"tril": lambda: p.T, "net": lambda: p.L, "band32": lambda: band(p.n, 32)}[which]()


@pytest.mark.parametrize("fp32", [True, False])
@pytest.mark.parametrize("case", list(CASES))
def test_bitwise_the_oracle(cuda, case, fp32):
    p, which = CASES[case]()
    pattern = pattern_of(p, which)
    longest = int(np.diff(osp.transpose_csr(*pattern)[0]).max())
    assert longest <= 32 and (which != "band32" or longest == 32)
    M = precond.fsai(dev(p.A, cuda), dev(pattern, cuda), fp32=fp32)
    assert isinstance(M, dp.FactoredMultiply)
    want = oracle_factor(p.A, pattern, fp32)
    helpers.assert_csr_equal(M.L, want)
    helpers.assert_csr_equal(M.Lt, osp.transpose_csr(*want))
    if fp32:
        assert M.L.packed() is not None and M.Lt.packed() is not None  # every value is an fp32 number
    print(f"{case}: nnz(L)/n = {want[1].shape[0] / p.n:.2f}, longest column {longest}")


def test_default_pattern_is_tril(cuda):
    p = helpers.problem("poisson2d", 64, 1)
    M = precond.fsai(dev(p.A, cuda))
    helpers.assert_csr_equal(M.L, oracle_factor(p.A, p.T, True))


def test_errors_name_their_cause(cuda):
    p = helpers.problem("poisson2d", 16, 0)
    A = dev(p.A, cuda)
    with pytest.raises(_lib.DpcgError, match="more than 32 entries"):
        precond.fsai(A, dev(band(p.n, 33), cuda))
    upper = sp.csr_matrix(osp.to_scipy(*p.T) + sp.csr_matrix(([1.0], ([0], [1])), shape=(p.n, p.n)))
    upper.sort_indices()
    with pytest.raises(_lib.DpcgError, match="not lower triangular"):
        precond.fsai(A, dev((upper.indptr, upper.indices, upper.data), cuda))
    with pytest.raises(_lib.DpcgError, match="diagonal in every column"):
        precond.fsai(A, dev(drop_entry(p.T, 7, 7), cuda))
    with pytest.raises(_lib.DpcgError, match="A stores no diagonal"):
        precond.fsai(dev(drop_entry(p.A, 9, 9), cuda), dev(p.T, cuda))
    negative = list(p.A)
    negative[2] = negative[2].copy()
    negative[2][0] = -negative[2][0]  # A_00 < 0 (row 0 stores its diagonal first)
    with pytest.raises(_lib.DpcgError, match="not symmetric positive definite"):
        precond.fsai(dev(negative, cuda), dev(p.T, cuda))
    with pytest.raises(_lib.DpcgError):
        precond.fsai(torch.eye(4, dtype=torch.float64))  # CPU operands
    # the library call itself: a flag per cause
    flag = torch.zeros(1, dtype=torch.int32, device=cuda)
    Lt = dev(p.T, cuda).transpose()
    u_val = torch.empty(Lt.nnz, dtype=torch.float64, device=cuda)
    neg = dev(negative, cuda)
    _lib.check(_lib.lib().dp_fsai_f64(p.n, _lib.ptr(neg.rowptr), _lib.ptr(neg.col), _lib.ptr(neg.val), _lib.ptr(Lt.rowptr),
                                      _lib.ptr(Lt.col), 1, _lib.ptr(u_val), _lib.ptr(flag), _lib.stream_ptr(cuda)))
    assert int(flag.item()) == _lib.DP_ERR_NOT_SPD


def test_empty_system_is_a_no_op(cuda):
    empty = CsrMatrix.from_arrays(np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0), device=cuda)
    M = precond.fsai(empty)
    assert M.L.n == 0 and M.L.nnz == 0 and M.Lt.nnz == 0


def test_pcg_316_against_the_oracle(cuda):
    p = helpers.problem("poisson2d", 316, 0, 0.5, "net")
    A, b, At = dev(p.A, cuda), p.b.to(cuda), osp.to_torch_csr(*p.A)
    jacobi = dp.pcg_solve(A, b, dp.Jacobi(A), max_iter=3000)
    counts = {}
    for which in ("tril", "net"):
        pattern = pattern_of(p, which)
        M = precond.fsai(A, dev(pattern, cuda))
        oracle_m = operators.FactoredMultiply(*oracle_factor(p.A, pattern, True))
        got = dp.pcg_solve(A, b, M, max_iter=3000)
        want = pcg.preconditioned_conjugate_gradient(At, p.b, oracle_m, max_iter=3000)
        assert abs(got.iterations - want.iterations) <= 1, (which, got.iterations, want.iterations)
        counts[which] = got.iterations
        # The loop sums its dot products in another order than torch, so the stop may land one body apart: x is compared
        # at the same iterate. The tril(A) trajectory of this system amplifies any last-bit change: the oracle against
        # itself with reversed dot products differs by 1e-15 at iterate 50, 5.6e-5 at 150 and 5.5e-7 at 334. On the
        # network's pattern the same experiment stays at 1e-15 throughout. So iterate 50 is held to 1e-8 on both, the
        # last iterate to 1e-8 on the network's pattern and to 1e-5 on tril(A).
        k = min(got.iterations, want.iterations)
        for at, tol in ((50, 1e-8), (k, 1e-8 if which == "net" else 1e-5)):
            x = got.x_hat if at == got.iterations else dp.pcg_solve(A, b, M, max_iter=at).x_hat
            xo = want.x_hat if at == want.iterations else pcg.preconditioned_conjugate_gradient(At, p.b, oracle_m, max_iter=at).x_hat
            assert torch.linalg.vector_norm(x.cpu() - xo) <= tol * torch.linalg.vector_norm(xo), (which, at)
    print(f"316^2 PCG iterations: jacobi {jacobi.iterations}, fsai tril(A) {counts['tril']}, fsai net {counts['net']}")
    assert counts["tril"] < min(jacobi.iterations, 624)  # 624: the reference loop's Jacobi count on this system
    assert counts["net"] < counts["tril"]


def test_packed_stream_and_batches(cuda):
    p = helpers.problem("poisson2d", 316, 0, 0.5, "net")
    A, b = dev(p.A, cuda), p.b.to(cuda)
    M = precond.fsai(A, dev(p.L, cuda))
    assert M.L.packed() is not None and M.Lt.packed() is not None
    packed = dp.pcg_solve(A, b, M, max_iter=3000)
    plain = dp.pcg_solve(A, b, M, max_iter=3000, pack=False)
    assert packed.iterations == plain.iterations
    assert torch.equal(packed.x_hat.view(torch.int64), plain.x_hat.view(torch.int64))
    wide = precond.fsai(A, dev(p.L, cuda), fp32=False)
    assert wide.L.packed() is None  # fp64 values: no exact 6-byte copy
    # alone and inside a mixed batch: the same bits
    q = helpers.problem("poisson2d", 64, 3, 0.5, "net")
    Aq, bq = dev(q.A, cuda), q.b.to(cuda)
    Lq, Lqt = dev(q.L, cuda), dev(osp.transpose_csr(*q.L), cuda)
    batch = dp.pcg_solve_batch([(Aq, bq, dp.Jacobi(Aq)), (A, b, M), (Aq, bq, dp.FactoredMultiply(Lq, Lqt)),
                                (Aq, bq, precond.fsai(Aq))], max_iter=3000)
    alone = dp.pcg_solve(Aq, bq, precond.fsai(Aq), max_iter=3000)
    assert batch[1].iterations == packed.iterations
    assert torch.equal(batch[1].x_hat.view(torch.int64), packed.x_hat.view(torch.int64))
    assert batch[3].iterations == alone.iterations
    assert torch.equal(batch[3].x_hat.view(torch.int64), alone.x_hat.view(torch.int64))


def test_benchmark_suite_techniques(cuda, tmp_path):
    torch.manual_seed(69)
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS).to(cuda)
    data = synthetic.SyntheticPressureDataSet("poisson2d", 24, number_samples=3, batch_size=1, device=cuda)
    techniques = ("jacobi", "fsai", "fsai_learned", "learned")
    assert "fsai" not in BenchmarkSuite(data, net).techniques  # opt-in only
    suite = BenchmarkSuite(data, net, techniques=techniques, max_iter=5000)
    suite.run()
    suite.dump_csv(tmp_path)
    for name in techniques:
        for store in BenchmarkSuite._STORES:
            assert len(getattr(suite, store)[name]) == 3, (name, store)
        assert all(0 < i < 5000 for i in suite.iterations[name])
        assert all(s == 100 for s in suite.successes[name]) and all(r < 1e-8 for r in suite.residuals[name])
        assert all(np.isfinite(k) and k >= 1 for k in suite.kappas[name])
    assert suite.densities["fsai_learned"] == suite.densities["learned"]
    assert max(suite.iterations["fsai"]) < min(suite.iterations["jacobi"])
    table = (tmp_path / "table.csv").read_text().splitlines()
    assert table[0] == "technique,kappas,densities,iterations,setups,durations,totals,successes" and len(table) == 5
    assert [line.split(",")[0] for line in table[1:]] == list(techniques)
    assert (tmp_path / "totals.csv").read_text().splitlines()[0] == ",".join(techniques)
    variants = (tmp_path / "variants.csv").read_text()
    assert "\nfsai," in variants and "\nfsai_learned," in variants
    serial = BenchmarkSuite(data, net, techniques=techniques, max_iter=5000, batch_systems=1)
    serial.run()
    for name in techniques:
        assert serial.iterations[name] == suite.iterations[name] and serial.residuals[name] == suite.residuals[name]
        assert serial.densities[name] == suite.densities[name] and serial.kappas[name] == suite.kappas[name]
    # the fsai records are the oracle's factor in the oracle's loop
    for k in range(3):
        pk = helpers.problem("poisson2d", 24, k)
        want = pcg.preconditioned_conjugate_gradient(osp.to_torch_csr(*pk.A), pk.b,
                                                     operators.FactoredMultiply(*oracle_factor(pk.A, pk.T, True)),
                                                     max_iter=5000)
        assert abs(suite.iterations["fsai"][k] - want.iterations) <= 1
