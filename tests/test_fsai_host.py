"""CPU tests of the FSAI comparator (dp_fsai_f64, precond.fsai): argument checks before any CUDA call, and the oracle's
restatement of the kernel's arithmetic against dense solves, the defining property diag(L^T A L) = 1, the exact inverse
on a complete pattern, and a PCG run in which FSAI beats Jacobi. No kernel is launched here."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import fsai_oracle
import helpers
from deeppreconditioning_b200 import _lib, build, precond
from oracle import operators, pcg
from oracle import sparse as osp

OK, INVALID, ALIGNMENT = 0, 1, 2
FAKE = 4096  # a non-null, 16-byte aligned address: never dereferenced by a call that is rejected or has nothing to do


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.lib()


def fsai_call(lib, n=4, a=FAKE, u=FAKE, u_col=FAKE, fp32=1, u_val=FAKE, flag=FAKE):
    return lib.dp_fsai_f64(n, a, a, a, u, u_col, fp32, u_val, flag, None)


def test_argument_validation_without_a_gpu(lib):
    assert lib.dp_fsai_max_row_entries() == 32
    assert fsai_call(lib, n=-1) == INVALID
    assert fsai_call(lib, fp32=2) == INVALID
    assert fsai_call(lib, a=None) == INVALID
    assert fsai_call(lib, u=None) == INVALID
    assert fsai_call(lib, u_col=None) == INVALID
    assert fsai_call(lib, u_val=None) == INVALID
    assert fsai_call(lib, flag=None) == INVALID
    assert fsai_call(lib, u_col=FAKE + 4) == ALIGNMENT
    assert fsai_call(lib, u_val=FAKE + 8) == ALIGNMENT
    assert fsai_call(lib, a=FAKE + 8) == ALIGNMENT
    assert fsai_call(lib, n=0, a=None, u=None, u_col=None, u_val=None, flag=None) == OK  # nothing to do


def test_cpu_operands_raise():
    dense = torch.eye(3, dtype=torch.float64)
    with pytest.raises(_lib.DpcgError):
        precond.fsai(dense)
    with pytest.raises(_lib.DpcgError):
        precond.fsai(dense.to_sparse_csr())


# ---- oracle ---------------------------------------------------------------------------------------------------------
def oracle_factor(A, pattern, fp32=False):
    """The oracle's FSAI factor ``L`` (lower CSR) on the lower pattern ``pattern`` (values ignored)."""
    u_rowptr, u_col, _ = osp.transpose_csr(*pattern)
    u_val = fsai_oracle.fsai(*A, u_rowptr, u_col, fp32)
    return osp.transpose_csr(u_rowptr, u_col, u_val)


def box_pattern(T, n):
    """``tril(A)`` dilated by a 5x5 box in the matrix image (row >= col): a structural stand-in for the factor network's
    pattern (its five 2x2 layers grow every stored site by two rows and columns either way)."""
    rows, cols = osp.to_scipy(*T).nonzero()
    rs, cs = [], []
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            r, c = rows + dy, cols + dx
            ok = (r >= 0) & (r < n) & (c >= 0) & (c < n) & (r >= c)
            rs.append(r[ok]), cs.append(c[ok])
    m = sp.csr_matrix((np.ones(sum(map(len, rs))), (np.concatenate(rs), np.concatenate(cs))), shape=(n, n))
    m.sum_duplicates(), m.sort_indices()
    return m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data


def dense_columns(A, L):
    """Column i of L by a dense solve A[J, J] y = e_0 (numpy) on the same pattern J."""
    Ad, Lc = osp.to_scipy(*A).toarray(), osp.to_scipy(*L).tocsc()
    for i in range(Lc.shape[0]):
        J = Lc.indices[Lc.indptr[i]:Lc.indptr[i + 1]]
        e = np.zeros(len(J))
        e[0] = 1.0
        y = np.linalg.solve(Ad[np.ix_(J, J)], e)
        yield i, J, y / np.sqrt(y[0]), Lc.data[Lc.indptr[i]:Lc.indptr[i + 1]]


@pytest.mark.parametrize("kind,side,pattern", [("poisson2d", 12, "tril"), ("poisson2d", 12, "box"),
                                               ("poisson3d", 5, "tril"), ("poisson3d", 5, "box")])
def test_oracle_matches_dense_solves(kind, side, pattern):
    p = helpers.problem(kind, side, 1)
    pat = p.T if pattern == "tril" else box_pattern(p.T, p.n)
    L = oracle_factor(p.A, pat)
    assert np.array_equal(L[0], pat[0]) and np.array_equal(L[1], pat[1])  # the factor keeps the pattern
    for i, J, want, got in dense_columns(p.A, L):
        assert J[0] == i
        np.testing.assert_allclose(got, want, rtol=1e-13, atol=1e-13 * np.abs(want).max())
    Ls, As = osp.to_scipy(*L), osp.to_scipy(*p.A)
    np.testing.assert_allclose((Ls.T @ As @ Ls).diagonal(), 1.0, rtol=0, atol=1e-13)
    L32 = oracle_factor(p.A, pat, fp32=True)
    assert np.array_equal(L32[2], L[2].astype(np.float32).astype(np.float64))


def test_complete_pattern_gives_the_inverse():
    rng = np.random.default_rng(7)
    n = 32
    B = rng.standard_normal((n, n))
    Ad = B @ B.T + n * np.eye(n)
    As = sp.csr_matrix(Ad)
    A = (As.indptr, As.indices, As.data)
    full = sp.csr_matrix(np.tril(np.ones((n, n))))
    L = oracle_factor(A, (full.indptr, full.indices, full.data))
    Ls = osp.to_scipy(*L).toarray()
    np.testing.assert_allclose(Ls @ Ls.T, np.linalg.inv(Ad), rtol=0, atol=1e-10 * np.abs(np.linalg.inv(Ad)).max())


def drop_entry(csr, row, col):
    """The CSR ``csr`` without its entry ``(row, col)``."""
    m = osp.to_scipy(*csr).tolil()
    m[row, col] = 0
    m = m.tocsr()
    m.eliminate_zeros()
    return m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data


def test_oracle_rejects_what_the_kernel_rejects():
    p = helpers.problem("poisson2d", 6, 0)
    u_rowptr, u_col, _ = osp.transpose_csr(*p.T)
    no_diag = osp.transpose_csr(*drop_entry(p.T, 3, 3))  # column 3 of L without its diagonal
    with pytest.raises(ValueError):
        fsai_oracle.fsai(*p.A, no_diag[0], no_diag[1])
    with pytest.raises(ValueError):  # A without a stored diagonal
        fsai_oracle.fsai(*drop_entry(p.A, 5, 5), u_rowptr, u_col)
    A = list(p.A)
    A[2] = A[2].copy()
    A[2][0] = -A[2][0]  # A_00 < 0 (row 0 stores its diagonal first)
    with pytest.raises(FloatingPointError):
        fsai_oracle.fsai(*A, u_rowptr, u_col)


def test_fsai_pcg_beats_jacobi_at_64():
    p = helpers.problem("poisson2d", 64, 0)
    At = osp.to_torch_csr(*p.A)
    jacobi = pcg.preconditioned_conjugate_gradient(At, p.b, operators.Jacobi(osp.to_scipy(*p.A).diagonal()), max_iter=3000)
    L = oracle_factor(p.A, p.T, fp32=True)
    fsai = pcg.preconditioned_conjugate_gradient(At, p.b, operators.FactoredMultiply(*L), max_iter=3000)
    box = pcg.preconditioned_conjugate_gradient(At, p.b, operators.FactoredMultiply(*oracle_factor(p.A, box_pattern(p.T, p.n), True)),
                                                max_iter=3000)
    print(f"64^2 oracle PCG: jacobi {jacobi.iterations}, fsai tril(A) {fsai.iterations}, fsai box {box.iterations}")
    assert fsai.iterations < jacobi.iterations
    assert box.iterations < fsai.iterations
