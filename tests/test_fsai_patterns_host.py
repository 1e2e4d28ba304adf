"""CPU tests of the power patterns of FSAI (dp_csr_pattern_product_*, precond.power_pattern): argument checks before any
CUDA call, the tests' power-pattern oracle against boolean dense matrix powers, and the iterations FSAI takes on those
patterns in the oracle PCG. No kernel is launched here."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import helpers
from deeppreconditioning_b200 import _lib, build, precond
from oracle import operators, pcg
from oracle import sparse as osp
from test_fsai_host import oracle_factor

OK, INVALID, ALIGNMENT, WORKSPACE = 0, 1, 2, 3
FAKE = 4096  # a non-null, 16-byte aligned address: never dereferenced by a call that is rejected or has nothing to do


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.lib()


def oracle_power_pattern(A, power):
    """The pattern of ``tril(|A|^power)`` (CSR, sorted, every value 1.0): scipy products of the pattern of ``|A|`` with
    ones - all terms positive, so nothing cancels."""
    S = osp.to_scipy(*A).copy()
    S.data[:] = 1.0
    P = S.copy()
    for _ in range(power - 1):
        P = P @ S
    T = sp.tril(P, format="csr")
    T.sort_indices()
    return T.indptr.astype(np.int32), T.indices.astype(np.int32), np.ones(T.nnz)


POINTERS = ("p_rowptr", "p_col", "q_rowptr", "q_col", "c_rowptr")


def count_call(lib, n=4, lower=0, nnz=FAKE, flag=FAKE, ws=FAKE, ws_bytes=None, **ptrs):
    p = {name: ptrs.get(name, FAKE) for name in POINTERS}
    ws_bytes = lib.dp_csr_pattern_product_workspace_bytes(max(n, 0)) if ws_bytes is None else ws_bytes
    return lib.dp_csr_pattern_product_count(n, p["p_rowptr"], p["p_col"], p["q_rowptr"], p["q_col"], lower, p["c_rowptr"],
                                            nnz, flag, ws, ws_bytes, None)


def fill_call(lib, n=4, lower=0, c_col=FAKE, **ptrs):
    p = {name: ptrs.get(name, FAKE) for name in POINTERS}
    return lib.dp_csr_pattern_product_fill(n, p["p_rowptr"], p["p_col"], p["q_rowptr"], p["q_col"], lower, p["c_rowptr"],
                                           c_col, None)


def test_argument_validation_without_a_gpu(lib):
    assert lib.dp_csr_pattern_product_workspace_bytes(0) > 0
    assert lib.dp_csr_pattern_product_workspace_bytes(100000) > 0
    for call in (count_call, fill_call):
        assert call(lib, n=-1) == INVALID
        assert call(lib, lower=2) == INVALID
        assert call(lib, lower=-1) == INVALID
        for name in POINTERS:
            assert call(lib, **{name: None}) == INVALID, (call.__name__, name)
    assert count_call(lib, nnz=None) == INVALID
    assert count_call(lib, flag=None) == INVALID
    assert count_call(lib, ws=None) == INVALID
    assert count_call(lib, ws=FAKE + 8) == ALIGNMENT
    assert count_call(lib, ws_bytes=lib.dp_csr_pattern_product_workspace_bytes(4) - 1) == WORKSPACE
    assert fill_call(lib, c_col=None) == INVALID
    assert fill_call(lib, c_col=FAKE + 4) == ALIGNMENT
    # n = 0 with null pointers: nothing to do, no CUDA call
    nulls = {name: None for name in POINTERS}
    assert count_call(lib, n=0, nnz=None, flag=None, ws=None, ws_bytes=0, **nulls) == OK
    assert fill_call(lib, n=0, c_col=None, **nulls) == OK


def test_power_pattern_rejects_cpu_operands_and_bad_powers():
    dense = torch.eye(3, dtype=torch.float64)
    with pytest.raises(_lib.DpcgError):
        precond.power_pattern(dense)
    with pytest.raises(_lib.DpcgError):
        precond.power_pattern(dense.to_sparse_csr(), 3)
    for power in (0, -1, 2.5):
        with pytest.raises(ValueError):
            precond.power_pattern(dense.to_sparse_csr(), power)


@pytest.mark.parametrize("kind,side", [("poisson2d", 6), ("poisson3d", 3)])
def test_oracle_is_the_boolean_matrix_power(kind, side):
    p = helpers.problem(kind, side, 0)
    S = osp.to_scipy(*p.A).toarray() != 0
    power = np.eye(p.n, dtype=bool)
    for k in range(1, 6):
        power = (power.astype(np.int64) @ S.astype(np.int64)) > 0
        rowptr, col, val = oracle_power_pattern(p.A, k)
        got = osp.to_scipy(rowptr, col, val).toarray()
        assert np.array_equal(got != 0, np.tril(power)), k
        assert np.all(val == 1.0)
        assert all(np.all(np.diff(col[rowptr[i]:rowptr[i + 1]]) > 0) for i in range(p.n))
    k1 = oracle_power_pattern(p.A, 1)
    assert np.array_equal(k1[0], p.T[0]) and np.array_equal(k1[1], p.T[1])  # k = 1 is the structure of tril(A)


def test_fsai_on_power_patterns_in_the_oracle_pcg_at_64():
    p = helpers.problem("poisson2d", 64, 0)
    At = osp.to_torch_csr(*p.A)
    counts = []
    for k in range(1, 5):
        L = oracle_factor(p.A, oracle_power_pattern(p.A, k), True)
        counts.append(pcg.preconditioned_conjugate_gradient(At, p.b, operators.FactoredMultiply(*L), max_iter=3000).iterations)
    print(f"64^2 oracle PCG, FSAI on tril(|A|^k), k = 1..4: {counts}")
    assert counts == [71, 49, 38, 30]
