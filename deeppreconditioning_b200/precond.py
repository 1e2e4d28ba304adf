"""Preconditioner operators ``M`` for ``preconditioned_conjugate_gradient(A, b, M)``.

The reference applies ``M`` by ``@`` (``uibk/deep_preconditioning/cg.py:61,81``) and builds it as an explicit CSR
tensor (``test.py:70-105``). These objects keep the ``@`` contract but stay factored on the device:

===================  =======================================  ==========================================
class                reference constructor                    apply
===================  =======================================  ==========================================
``Identity``         ``_construct_vanilla``   test.py:70-72   ``z = r``
``Jacobi``           ``_construct_jacobi``    test.py:74-79   ``z = r / diag(A)``
``FactoredMultiply`` ``_construct_learned``   test.py:100-105 ``z = L (L^T r)``   (approximate inverse)
``FactoredSolve``    north_star / IC(0)                       ``z = L^-T (L^-1 r)`` (two sync-free SpTRSV)
``fsai(A)``          no reference counterpart (comparator)    ``z = L (L^T r)``   (FSAI: a ``FactoredMultiply``; its
                                                              patterns: ``tril(A)``, ``power_pattern(A, k)``, any)
``CsrOperator``      any explicit CSR ``M``   test.py:88,105  ``z = M r``
===================  =======================================  ==========================================
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .sparse import CsrMatrix, _workspace, as_csr


@dataclass
class TriangularPlan:
    """Level analysis (K3) of a triangular CSR pattern plus the warp-padded execution plan of the solves (K4)."""

    level: torch.Tensor      # int32[n]
    perm: torch.Tensor       # int32[n]   rows stably sorted by level
    level_ptr: torch.Tensor  # int32[nlevels+1]
    nlevels: int
    plan: torch.Tensor       # int32[32*nchunks], -1 = idle lane
    nchunks: int
    max_level_chunks: int
    upper: bool
    ls: "LevelOrdered | None" = None  # level-ordered copy of the factor (narrow levels): level-stream solve
    ts: "LevelOrdered | None" = None  # level-ordered copy of any factor, made on demand: tile-stream batch solve
    _identity: bool | None = None

    @property
    def perm_is_identity(self) -> bool:
        """The matrix is already in the level order of this solve (``precond.LevelOrdering``): the level-stream solve then
        takes its vectors by position (bulk copies instead of a gather through ``perm``). One read-back per plan."""
        if self._identity is None:
            n = self.perm.shape[0]
            self._identity = bool(torch.equal(self.perm, torch.arange(n, dtype=torch.int32, device=self.perm.device)))
        return self._identity


@dataclass
class LevelOrdered:
    """Level-ordered copy of a triangular factor (``dp_sptrsv_permute``), input of the level-stream solve."""

    rowptr: torch.Tensor        # int32[n+1]
    col: torch.Tensor           # int32[nnz], positions in level order
    val: torch.Tensor           # fp64[nnz], entries in the factor's order inside each row
    level_sorted: torch.Tensor  # int32[n]
    nnz: int
    source: tuple               # (data_ptr, version counter) of the values it was copied from (a plan may serve several
                                # factors; an in-place refactorisation bumps the tensor's version and invalidates the copy)
    stats: torch.Tensor | None = None  # device int32[3]: most entries in a tile / in a row, largest dependency distance
    _short: bool | None = None

    @staticmethod
    def key(matrix: CsrMatrix) -> tuple:
        return (matrix.val.data_ptr(), matrix.val._version)

    def matches(self, matrix: CsrMatrix) -> bool:
        return self.source == self.key(matrix)

    @property
    def short_rows(self) -> bool:
        """``DP_TRSV_SHORT_ROWS``: rows short enough for the register path of the tile-stream solve (one read-back per copy)."""
        if self._short is None:
            limits = np.zeros(2, np.int32)
            _lib.lib().dp_sptrsv_ts_limits(limits.ctypes.data)
            self._short = self.stats is not None and int(self.stats[1].item()) <= int(limits[1])
        return self._short


LS_MAX_MEAN_LEVEL_ROWS = 1024  # level-stream solve when n / nlevels is at most this (one CTA must keep up)


def _permute(matrix: CsrMatrix, plan: TriangularPlan, perm: torch.Tensor | None = None):
    """``dp_sptrsv_permute``: the level-ordered copy and its statistics (tile entries, row entries, dependency distance).
    ``perm`` overrides the plan's level order with another valid solve order (``reversed_copy``)."""
    lib, n, dev = _lib.lib(), matrix.n, matrix.device
    perm = plan.perm if perm is None else perm
    i32 = dict(dtype=torch.int32, device=dev)
    rowptr_p, level_sorted = torch.empty(n + 1, **i32), torch.empty(n, **i32)
    col_p = torch.empty(max(matrix.nnz, 1), **i32)
    val_p = torch.empty(max(matrix.nnz, 1), dtype=torch.float64, device=dev)
    stats = torch.zeros(3, **i32)
    ws = _workspace(lib.dp_sptrsv_permute_workspace_bytes(n), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_sptrsv_permute(n, int(plan.upper), _lib.ptr(matrix.rowptr), _lib.ptr(matrix.col), _lib.ptr(matrix.val),
                                         _lib.ptr(perm), _lib.ptr(plan.level), _lib.ptr(rowptr_p), _lib.ptr(col_p),
                                         _lib.ptr(val_p), _lib.ptr(level_sorted), _lib.ptr(stats), _lib.ptr(ws), ws.numel(),
                                         _lib.stream_ptr(dev)), "dp_sptrsv_permute")
    copy = LevelOrdered(rowptr_p, col_p[: matrix.nnz], val_p[: matrix.nnz], level_sorted, matrix.nnz,
                        LevelOrdered.key(matrix), stats)
    return copy, stats


def level_ordered(matrix: CsrMatrix, plan: TriangularPlan) -> LevelOrdered | None:
    """Build the level-ordered copy if the factor qualifies for the level-stream solve, else ``None``."""
    lib, n = _lib.lib(), matrix.n
    if n == 0 or plan.nlevels == 0 or n / plan.nlevels > LS_MAX_MEAN_LEVEL_ROWS:
        return None
    copy, stats = _permute(matrix, plan)
    limits = np.zeros(4, np.int32)
    lib.dp_sptrsv_ls_limits(limits.ctypes.data)
    widest = int(torch.diff(plan.level_ptr).max().item())
    if widest > limits[3] or np.any(stats.cpu().numpy() > limits[:3]):  # once per matrix: tile entries, row entries, dependency distance
        return None
    return copy


def level_ordered_any(matrix: CsrMatrix, plan: TriangularPlan) -> LevelOrdered:
    """The level-ordered copy of ANY triangular factor: input of the tile-stream batch solve (wide levels)."""
    if plan.ls is not None and plan.ls.matches(matrix):
        return plan.ls
    if plan.ts is None or not plan.ts.matches(matrix):
        plan.ts = _permute(matrix, plan)[0]
    return plan.ts


def reversed_copy(upper_matrix: CsrMatrix, plan: TriangularPlan) -> LevelOrdered:
    """Copy of ``U = L^T`` for the tile-stream solve in REVERSED position space (``DP_TRSV_REVERSED``): row ``r`` of the
    copy is row ``n-1-r`` of ``U``. For a system kept in the level order of its forward solve (``LevelOrdering``) that is
    a valid backward order whose dependencies sit one forward level away, so the system's own ``b`` / ``x`` serve both
    solves without a gather."""
    assert plan.upper
    n = upper_matrix.n
    perm = torch.arange(n - 1, -1, -1, dtype=torch.int32, device=upper_matrix.device)
    return _permute(upper_matrix, plan, perm)[0]


def analyse(matrix: CsrMatrix, upper: bool, level_stream: bool = True) -> TriangularPlan:
    """``dp_sptrsv_analyse`` + ``dp_sptrsv_plan_build``. ``upper=False``: lower triangular, diagonal last in each row;
    ``upper=True``: upper triangular (``L^T``), diagonal first. With ``level_stream`` a factor with narrow levels also
    gets its level-ordered copy (``dp_sptrsv_permute``) and is then solved by the level-stream kernel. The copy holds
    the VALUES of ``matrix`` at analysis time: analyse the numeric factor, not just its pattern."""
    lib, n, dev = _lib.lib(), matrix.n, matrix.device
    i32 = dict(dtype=torch.int32, device=dev)
    level, perm = torch.empty(n, **i32), torch.empty(n, **i32)
    level_ptr = torch.empty(n + 1, **i32)
    nlev, flag = torch.zeros(1, **i32), torch.zeros(1, **i32)
    ws = _workspace(lib.dp_sptrsv_analyse_workspace_bytes(n), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_sptrsv_analyse(n, _lib.ptr(matrix.rowptr), _lib.ptr(matrix.col), int(upper), _lib.ptr(level),
                                         _lib.ptr(perm), _lib.ptr(level_ptr), _lib.ptr(nlev), _lib.ptr(flag),
                                         _lib.ptr(ws), ws.numel(), _lib.stream_ptr(dev)), "dp_sptrsv_analyse")
    # plan sizes on the device (chunk prefix over the levels, total, widest level); ONE 12-byte read-back per matrix
    chunk_ptr, summary = torch.empty(n + 1, **i32), torch.empty(3, **i32)
    ws2 = _workspace(lib.dp_sptrsv_plan_sizes_workspace_bytes(n), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_sptrsv_plan_sizes(n, _lib.ptr(nlev), _lib.ptr(level_ptr), _lib.ptr(chunk_ptr), _lib.ptr(summary),
                                            _lib.ptr(ws2), ws2.numel(), _lib.stream_ptr(dev)), "dp_sptrsv_plan_sizes")
    nlevels, nchunks, widest_chunks = (int(v) for v in summary.tolist())
    _lib.raise_on_flag(flag, "dp_sptrsv_analyse (not triangular, or diagonal not first/last in its row)")
    plan = torch.empty(max(nchunks * 32, 1), **i32)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_sptrsv_plan_build(n, nlevels, _lib.ptr(perm), _lib.ptr(level_ptr), _lib.ptr(chunk_ptr),
                                            _lib.ptr(plan), nchunks, _lib.stream_ptr(dev)), "dp_sptrsv_plan_build")
    out = TriangularPlan(level, perm, level_ptr[: nlevels + 1], nlevels, plan, nchunks, widest_chunks, bool(upper))
    if level_stream:
        out.ls = level_ordered(matrix, out)
    return out


def triangular_solve(matrix: CsrMatrix, plan: TriangularPlan, b: torch.Tensor, out: torch.Tensor | None = None,
                     algorithm: str = "auto"):
    """Solve ``T x = b``: level-stream kernel when the plan carries a level-ordered copy (``algorithm`` "auto"/"ls"),
    else the sync-free kernel (``dp_sptrsv_solve_f64``, forced with "syncfree"). Same bits either way."""
    lib, n, dev = _lib.lib(), matrix.n, matrix.device
    assert b.is_cuda and b.dtype == torch.float64 and b.shape == (n,)
    b = b.contiguous()
    x = out if out is not None else torch.empty(n, dtype=torch.float64, device=dev)
    has_ls = plan.ls is not None and plan.ls.matches(matrix)
    if algorithm == "ls" and not has_ls:
        raise _lib.DpcgError("this plan has no level-ordered copy of this matrix (levels too wide or rows too long)")
    if algorithm != "syncfree" and has_ls:
        return _level_stream_batch([(matrix, plan, b)], [x])[0]
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = _workspace(lib.dp_sptrsv_workspace_bytes(), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_sptrsv_solve_f64(n, _lib.ptr(matrix.rowptr), _lib.ptr(matrix.col), _lib.ptr(matrix.val),
                                           int(plan.upper), _lib.ptr(plan.plan), plan.nchunks, plan.max_level_chunks,
                                           _lib.ptr(b), _lib.ptr(x), _lib.ptr(flag), _lib.ptr(ws), ws.numel(),
                                           _lib.stream_ptr(dev)), "dp_sptrsv_solve_f64")
    _lib.raise_on_flag(flag, "dp_sptrsv_solve_f64")
    return x


class PreparedTriangularBatch:
    """Independent solves ``T_s x_s = b_s`` prepared ONCE (descriptors uploaded, workspace allocated) and launched many
    times: ``solve()`` only enqueues kernels. For solves that are repeated with the same factors and vector buffers - new
    right-hand sides are written into the same ``b`` tensors - and for timing the kernels without the per-call host work
    (``dp_sptrsv_ls_prepare`` / ``dp_sptrsv_ls_launch``, ``dp_sptrsv_ts_prepare`` / ``dp_sptrsv_ts_launch``).

    ``algorithm``: "ls" (level-stream, one CTA per system) or "ts" (tile-stream). ``copies``, ``position_space``,
    ``reverse``: as in :func:`triangular_solve_batch`. ``xs`` holds the solutions after ``solve()``."""

    def __init__(self, systems, outs=None, algorithm: str = "ls", copies=None, position_space: bool = False, reverse=None):
        lib = _lib.lib()
        self.algorithm, self.device, self.nsys = algorithm, systems[0][0].device, len(systems)
        dev, nsys = self.device, self.nsys
        self.descs = (_lib.TrsvLsSystem * nsys)()
        self.xs, self._keep = [], []
        max_tiles = nmax = nperm = 0
        short = True
        for i, (matrix, plan, b) in enumerate(systems):
            n = matrix.n
            if copies is not None:
                ls = copies[i]
            else:
                ls = plan.ls if algorithm == "ls" else level_ordered_any(matrix, plan)
            assert b.is_cuda and b.dtype == torch.float64 and b.shape == (n,)
            b = b.contiguous()
            x = outs[i] if outs is not None else torch.empty(n, dtype=torch.float64, device=dev)
            d = self.descs[i]
            d.n, d.nnz, d.upper = n, ls.nnz, int(plan.upper)
            d.rowptr_p, d.col_p, d.val_p = _lib.ptr(ls.rowptr), _lib.ptr(ls.col), _lib.ptr(ls.val)
            d.level_sorted = _lib.ptr(ls.level_sorted)
            if algorithm == "ls":
                by_position = plan.perm_is_identity and b.data_ptr() % 16 == 0 and b.data_ptr() != x.data_ptr()
                d.perm = None if by_position else _lib.ptr(plan.perm)
            else:
                if b.data_ptr() % 16:  # spans of b are moved by 16-byte granular bulk copies
                    b = b.clone()
                d.perm = None if position_space else _lib.ptr(plan.perm)
                d.flags = 2 if ls.short_rows else 0  # DP_TRSV_SHORT_ROWS
                if position_space and reverse is not None and reverse[i]:
                    d.flags |= 1  # DP_TRSV_REVERSED
                short = short and ls.short_rows
                max_tiles, nmax = max(max_tiles, (n + 511) // 512), max(nmax, n)
                nperm += 0 if position_space else 1
            d.b, d.x = _lib.ptr(b), _lib.ptr(x)
            self.xs.append(x), self._keep.append((b, ls, plan))
        self._ts_args = (max_tiles, nmax, int(short), nperm)
        with torch.cuda.device(dev):
            if algorithm == "ls":
                self.flag = None
                self.ws = _workspace(lib.dp_sptrsv_ls_workspace_bytes(nsys), dev)
                _lib.check(lib.dp_sptrsv_ls_prepare(self.descs, nsys, _lib.ptr(self.ws), self.ws.numel(), _lib.stream_ptr(dev)),
                           "dp_sptrsv_ls_prepare")
            else:
                self.flag = torch.zeros(1, dtype=torch.int32, device=dev)
                self.ws = _workspace(lib.dp_sptrsv_ts_workspace_bytes(self.descs, nsys), dev)
                _lib.check(lib.dp_sptrsv_ts_prepare(self.descs, nsys, _lib.ptr(self.ws), self.ws.numel(), _lib.stream_ptr(dev)),
                           "dp_sptrsv_ts_prepare")

    def solve(self):
        """Enqueue the solve on the current stream (asynchronous); returns the list of solution tensors."""
        lib, dev = _lib.lib(), self.device
        with torch.cuda.device(dev):
            if self.algorithm == "ls":
                _lib.check(lib.dp_sptrsv_ls_launch(self.nsys, _lib.ptr(self.ws), self.ws.numel(), _lib.stream_ptr(dev)),
                           "dp_sptrsv_ls_launch")
            else:
                _lib.check(lib.dp_sptrsv_ts_launch(self.nsys, *self._ts_args, _lib.ptr(self.flag), _lib.ptr(self.ws),
                                                   _lib.stream_ptr(dev)), "dp_sptrsv_ts_launch")
        return self.xs

    def check(self) -> None:
        """Raise if the device flagged a time-out or a broken promise (tile-stream; synchronises)."""
        if self.flag is not None:
            _lib.raise_on_flag(self.flag, "dp_sptrsv_ts_launch")


def _level_stream_batch(systems, outs=None, copies=None):
    return PreparedTriangularBatch(systems, outs, "ls", copies).solve()


def _tile_stream_batch(systems, outs=None, copies=None, position_space=False, reverse=None):
    prepared = PreparedTriangularBatch(systems, outs, "ts", copies, position_space, reverse)
    xs = prepared.solve()
    prepared.check()
    return xs


def triangular_solve_batch(systems, outs=None, algorithm: str = "auto", copies=None, position_space: bool = False,
                           reverse=None):
    """Independent solves ``T_s x_s = b_s`` in ONE launch.

    ``systems``: list of ``(matrix, plan, b)``; returns the list of solutions (the data-parallel axis of
    ``BenchmarkSuite.run``, ``test.py:121``). Three kernels, same bits: "ls" (level-stream, one CTA per system: factors
    with narrow levels, chosen by "auto" when every plan carries its copy), "ts" (tile-stream: the tiles of the
    level-ordered copies of all systems dealt to persistent CTAs, for wide levels; the copies are made on demand and
    cached in the plans, or passed as ``copies``), "syncfree" (``dp_sptrsv_solve_batch_f64``, original ordering).
    ``position_space`` ("ts" only): ``b`` and the solutions are in LEVEL ORDER (``b_pos = b[perm]``, ``x = x_pos`` with
    ``x_pos[r] = x[perm[r]]``) - the form a caller uses that keeps all its vectors in that order. ``reverse[i]``: system
    ``i``'s copy is a ``reversed_copy`` and its vectors are in the reverse of the copy's position order.
    """
    lib = _lib.lib()
    dev = systems[0][0].device
    nsys = len(systems)
    if algorithm == "ts":
        return _tile_stream_batch(systems, outs, copies, position_space, reverse)
    assert not position_space, "position-space vectors are a feature of the tile-stream solve"
    if algorithm != "syncfree" and all(plan.ls is not None and plan.ls.matches(m) for m, plan, _ in systems):
        return _level_stream_batch(systems, outs)
    if algorithm == "ls":
        raise _lib.DpcgError("a plan of this batch has no level-ordered copy")
    descs = (_lib.TrsvSystem * nsys)()
    xs, keep = [], []
    for i, (matrix, plan, b) in enumerate(systems):
        n = matrix.n
        assert b.is_cuda and b.dtype == torch.float64 and b.shape == (n,)
        b = b.contiguous()
        x = outs[i] if outs is not None else torch.empty(n, dtype=torch.float64, device=dev)
        d = descs[i]
        d.n, d.upper, d.max_level_chunks, d.nchunks = n, int(plan.upper), plan.max_level_chunks, plan.nchunks
        d.rowptr, d.col, d.val = _lib.ptr(matrix.rowptr), _lib.ptr(matrix.col), _lib.ptr(matrix.val)
        d.plan, d.b, d.x = _lib.ptr(plan.plan), _lib.ptr(b), _lib.ptr(x)
        xs.append(x), keep.append(b)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = _workspace(lib.dp_sptrsv_batch_workspace_bytes(nsys), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_sptrsv_solve_batch_f64(descs, nsys, _lib.ptr(flag), _lib.ptr(ws), ws.numel(),
                                                 _lib.stream_ptr(dev)), "dp_sptrsv_solve_batch_f64")
    _lib.raise_on_flag(flag, "dp_sptrsv_solve_batch_f64")
    return xs


@dataclass
class LevelOrdering:
    """Symmetric renumbering of a system by the level sets of its lower triangle (``x_level[r] = x[perm[r]]``).

    Level order is a topological order of the factor's dependency graph, so ``P tril(A) P^T`` is the lower triangle of
    ``P A P^T``, IC(0) commutes with the renumbering, and CG on the renumbered system is the same iteration up to the
    summation order of its dot products. What it buys: a level of the factor becomes a CONTIGUOUS run of rows (and of
    ``b`` / ``x`` entries), so the triangular solves read the factor and the vectors coalesced instead of one scattered
    sector per row - the form the tile-stream batch solve wants (``position_space=True``), and a better layout for the
    sync-free solves inside the fused PCG kernel as well. Natural ordering is what the reference's data has
    (``data_set.py:85-125``); this is an opt-in for SOLVE-mode preconditioners only.
    """

    perm: torch.Tensor  # int64[n]: position -> original row
    inv: torch.Tensor   # int32[n]: original row -> position
    nlevels: int

    def to_level(self, v: torch.Tensor) -> torch.Tensor:
        return v[self.perm]

    def from_level(self, v: torch.Tensor) -> torch.Tensor:
        out = torch.empty_like(v)
        out[self.perm] = v
        return out

    def renumber(self, tensor):
        """The same COO sites ``(batch, row, col)`` with rows and columns renumbered (a ``SparseConvTensor`` stand-in)."""
        from .model import SparseConvTensor

        idx = tensor.indices.to(self.inv.device)
        new = torch.stack([idx[:, 0], self.inv[idx[:, 1].long()], self.inv[idx[:, 2].long()]], dim=1).to(torch.int32)
        return SparseConvTensor(tensor.features.to(self.inv.device), new.contiguous(), tensor.spatial_shape, tensor.batch_size)


def level_ordering(tril_a: CsrMatrix, plan: TriangularPlan | None = None) -> LevelOrdering:
    """Level analysis (K3) of ``tril(A)`` turned into a symmetric renumbering of the whole system."""
    plan = plan or analyse(tril_a, upper=False, level_stream=False)
    perm = plan.perm.long()
    inv = torch.empty(tril_a.n, dtype=torch.int32, device=tril_a.device)
    inv[perm] = torch.arange(tril_a.n, dtype=torch.int32, device=tril_a.device)
    return LevelOrdering(perm, inv, plan.nlevels)


def incomplete_cholesky0(tril_a: CsrMatrix, plan: TriangularPlan | None = None) -> CsrMatrix:
    """IC(0) factor on the pattern of ``tril(A)`` (``dp_ic0_f64``) — stands in for ``ilupp.ichol0`` (``test.py:84``)."""
    lib, n, dev = _lib.lib(), tril_a.n, tril_a.device
    plan = plan or analyse(tril_a, upper=False)
    l_val = torch.empty(max(tril_a.nnz, 1), dtype=torch.float64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = _workspace(lib.dp_sptrsv_workspace_bytes(), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_ic0_f64(n, _lib.ptr(tril_a.rowptr), _lib.ptr(tril_a.col), _lib.ptr(tril_a.val),
                                  _lib.ptr(l_val), _lib.ptr(plan.plan), plan.nchunks, plan.max_level_chunks,
                                  _lib.ptr(flag), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(dev)), "dp_ic0_f64")
    _lib.raise_on_flag(flag, "dp_ic0_f64 (non-positive pivot)")
    return CsrMatrix(tril_a.rowptr, tril_a.col, l_val[: tril_a.nnz], n)


def incomplete_cholesky_threshold(tril_a: CsrMatrix, fill_in: int = 1, threshold: float = 0.1) -> CsrMatrix:
    """Threshold incomplete Cholesky ICT(p, tau) of ``tril(A)`` (``dp_icholt_host``) - stands in for the reference's default
    comparator ``ilupp.icholt(A, add_fill_in=fill_in, threshold=threshold)`` (``test.py:81-86``). A sequential host
    algorithm (as in the reference): the pattern travels to the host and the factor back; set-up work, not the solve."""
    lib, n, dev = _lib.lib(), tril_a.n, tril_a.device
    rowptr, col, val = (np.ascontiguousarray(a) for a in tril_a.to_host())
    capacity = int(len(col)) + n * max(int(fill_in), 0) + 1
    rowptr_out = np.empty(n + 1, np.int32)
    col_out, val_out = np.empty(capacity, np.int32), np.empty(capacity, np.float64)
    nnz = np.zeros(1, np.int64)
    _lib.check(lib.dp_icholt_host(n, rowptr.ctypes.data, col.ctypes.data, val.ctypes.data, int(fill_in), float(threshold),
                                  rowptr_out.ctypes.data, col_out.ctypes.data, val_out.ctypes.data, capacity,
                                  nnz.ctypes.data), "dp_icholt_host (missing diagonal or non-positive pivot)")
    k = int(nnz[0])
    return CsrMatrix.from_arrays(rowptr_out, col_out[:k].copy(), val_out[:k].copy(), device=dev)


def fsai(A: CsrMatrix, pattern: CsrMatrix | None = None, fp32: bool = True) -> "FactoredMultiply":
    """FSAI (factorized sparse approximate inverse, Kolotilina & Yeremin): ``M = L L^T ~ A^-1`` with ``L`` on a given
    lower-triangular pattern, applied like the learned factor (two SpMVs, ``DP_PRECOND_MULTIPLY``).

    ``A``: the full symmetric matrix. ``pattern``: lower triangular, diagonal stored, values ignored; ``tril(A)`` by
    default. Column ``i`` of ``L`` holds ``y / sqrt(y_0)`` with ``A[J, J] y = e_0`` on the column's pattern ``J`` (at most
    ``dp_fsai_max_row_entries()`` entries), so ``(L^T A L)_ii = 1`` (``dp_fsai_f64``). ``fp32``: every value rounded once
    to fp32, so the factor has an exact packed copy and streams 6 bytes per entry like the learned factor; ``False``
    keeps the fp64 values. Raises :class:`DpcgError` on a pattern the kernel does not accept and when ``A`` is not SPD."""
    if not isinstance(A, CsrMatrix) or not isinstance(pattern, (CsrMatrix, type(None))):
        raise _lib.DpcgError("fsai takes device CsrMatrix operands (there is no CPU path)")
    pattern = A.tril() if pattern is None else pattern
    if pattern.n != A.n or pattern.device != A.device:
        raise ValueError("A and the pattern must have the same size and live on the same device")
    lib, n, dev = _lib.lib(), A.n, A.device
    upper = pattern.transpose()  # the pattern of U = L^T: row i is column i of L, diagonal first
    u_val = torch.empty(max(upper.nnz, 1), dtype=torch.float64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_fsai_f64(n, _lib.ptr(A.rowptr), _lib.ptr(A.col), _lib.ptr(A.val), _lib.ptr(upper.rowptr),
                                   _lib.ptr(upper.col), int(bool(fp32)), _lib.ptr(u_val), _lib.ptr(flag),
                                   _lib.stream_ptr(dev)), "dp_fsai_f64")
    status = int(flag.item())
    if status == _lib.DP_ERR_STRUCTURE:
        raise _lib.DpcgError(f"fsai: the pattern is not lower triangular with its diagonal in every column, a column holds "
                             f"more than {lib.dp_fsai_max_row_entries()} entries, or A stores no diagonal in some row")
    if status == _lib.DP_ERR_NOT_SPD:
        raise _lib.DpcgError("fsai: A is not symmetric positive definite (non-positive pivot in a local Cholesky factor)")
    _lib.raise_on_flag(flag, "dp_fsai_f64")
    Lt = CsrMatrix(upper.rowptr, upper.col, u_val[: upper.nnz], n)
    return FactoredMultiply(Lt.transpose(), Lt)


_INT32_MAX = 2**31 - 1


def _pattern_product(P: CsrMatrix, Q: CsrMatrix, lower: bool) -> CsrMatrix:
    """The structural pattern of ``P Q`` (``tril`` of it with ``lower``), every value 1.0: ``dp_csr_pattern_product_count``,
    one read-back of the total and the device flag, then ``dp_csr_pattern_product_fill``."""
    lib, n, dev = _lib.lib(), P.n, P.device
    if Q.n != n or Q.device != dev:
        raise ValueError("P and Q must have the same size and live on the same device")
    rowptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = _workspace(lib.dp_csr_pattern_product_workspace_bytes(n), dev)
    operands = (_lib.ptr(P.rowptr), _lib.ptr(P.col), _lib.ptr(Q.rowptr), _lib.ptr(Q.col), int(bool(lower)))
    with torch.cuda.device(dev):
        _lib.check(lib.dp_csr_pattern_product_count(n, *operands, _lib.ptr(rowptr), _lib.ptr(total), _lib.ptr(flag),
                                                     _lib.ptr(ws), ws.numel(), _lib.stream_ptr(dev)),
                   "dp_csr_pattern_product_count")
    nnz, status = torch.cat([total, flag.to(torch.int64)]).tolist()
    if status:
        raise _lib.DpcgError(f"pattern product: a column index lies outside [0, {n})")
    if nnz > _INT32_MAX:
        raise _lib.DpcgError(f"pattern product: the result holds {nnz} entries, more than an int32 CSR can index "
                             f"({_INT32_MAX})")
    col = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dp_csr_pattern_product_fill(n, *operands, _lib.ptr(rowptr), _lib.ptr(col), _lib.stream_ptr(dev)),
                   "dp_csr_pattern_product_fill")
    return CsrMatrix(rowptr, col[:nnz], torch.ones(nnz, dtype=torch.float64, device=dev), n)


def power_pattern(A: CsrMatrix, power: int = 2) -> CsrMatrix:
    """The pattern of ``tril(|A|^power)``, every value 1.0: the standard a priori FSAI patterns (Chow, 2000), for
    ``fsai(A, power_pattern(A, k))``. Built on the device by symbolic products (``dp_csr_pattern_product_*``): ``A``,
    then ``power - 2`` full products with ``A``, then one that keeps the lower triangle. ``power = 1`` is the structure
    of ``A.tril()``. Columns grow with ``power``: at most ``k² + k + 1`` entries on a 2-D 5-point system (3, 7, 13, 21, 31
    for k = 1…5) and 4, 13, 32, 65 on a 3-D 7-point one, and ``fsai`` takes columns of at most
    ``dp_fsai_max_row_entries()`` = 32 entries. Raises :class:`DpcgError` for CPU operands and when a product
    would hold more than ``2^31 - 1`` entries, ``ValueError`` for a power that is not an integer of at least 1."""
    if isinstance(power, bool) or not isinstance(power, (int, np.integer)) or power < 1:
        raise ValueError(f"power_pattern: power must be an integer >= 1, got {power!r}")
    if not isinstance(A, CsrMatrix):
        raise _lib.DpcgError("power_pattern takes a device CsrMatrix (there is no CPU path)")
    if power == 1:
        lower = A.tril()
        return CsrMatrix(lower.rowptr, lower.col, torch.ones(lower.nnz, dtype=torch.float64, device=A.device), A.n)
    P = A
    for _ in range(int(power) - 2):
        P = _pattern_product(P, A, lower=False)
    return _pattern_product(P, A, lower=True)


class _Operator:
    precond: int = _lib.PRECOND_IDENTITY

    def _apply(self, r: torch.Tensor) -> torch.Tensor:  # device fp64 in, device fp64 out
        raise NotImplementedError

    def __matmul__(self, r: torch.Tensor) -> torch.Tensor:
        dev = getattr(self, "device", None) or (r.device if r.is_cuda else torch.device("cuda"))
        z = self._apply(r.to(device=dev, dtype=torch.float64))
        return z if r.is_cuda else z.to(r.device)

    def fill(self, system: _lib.PcgSystem) -> None:
        """Write this operator's arrays into a ``dp_pcg_system_t``."""
        system.precond = self.precond

    def stream_matrices(self) -> list:
        """The CSR matrices a PCG iteration streams for this operator (candidates for packed copies)."""
        return []

    def nnz_explicit(self) -> int | None:
        return None


def fill_packed(system: _lib.PcgSystem, tag: str, matrix: CsrMatrix) -> None:
    """Hand the packed stream copy of ``matrix`` (if it has been made and is exact) to the descriptor."""
    pk = matrix._packed or None
    for name in ("col16", "val32", "tile_base"):
        setattr(system, f"{tag}_{name}", _lib.ptr(getattr(pk, name)) if pk is not None else None)


class Identity(_Operator):
    precond = _lib.PRECOND_IDENTITY

    def _apply(self, r):
        return r.clone()


class Jacobi(_Operator):
    precond = _lib.PRECOND_JACOBI

    def __init__(self, matrix) -> None:
        self.dinv = as_csr(matrix).inv_diagonal()
        self.device = self.dinv.device

    def _apply(self, r):
        return self.dinv * r

    def fill(self, system):
        system.precond = self.precond
        system.dinv = _lib.ptr(self.dinv)


class CsrOperator(_Operator):
    precond = _lib.PRECOND_CSR

    def __init__(self, matrix, device=None) -> None:
        self.M = as_csr(matrix, device)
        self.device = self.M.device

    def _apply(self, r):
        return self.M.matvec(r)

    def fill(self, system):
        system.precond = self.precond
        system.m_rowptr, system.m_col, system.m_val = _lib.ptr(self.M.rowptr), _lib.ptr(self.M.col), _lib.ptr(self.M.val)
        system.m_nnz = self.M.nnz
        fill_packed(system, "m", self.M)

    def stream_matrices(self):
        return [self.M]


class FactoredMultiply(_Operator):
    """``M = L L^T`` applied as two SpMVs, never formed (the reference forms it densely in fp32, ``test.py:104``)."""

    precond = _lib.PRECOND_MULTIPLY

    def __init__(self, L: CsrMatrix, Lt: CsrMatrix | None = None) -> None:
        self.L, self.Lt = L, Lt if Lt is not None else L.transpose()
        self.device = L.device

    def _apply(self, r):
        return self.L.matvec(self.Lt.matvec(r))

    def fill(self, system):
        system.precond = self.precond
        system.m_rowptr, system.m_col, system.m_val = _lib.ptr(self.L.rowptr), _lib.ptr(self.L.col), _lib.ptr(self.L.val)
        system.mt_rowptr, system.mt_col, system.mt_val = (_lib.ptr(self.Lt.rowptr), _lib.ptr(self.Lt.col),
                                                          _lib.ptr(self.Lt.val))
        system.m_nnz, system.mt_nnz = self.L.nnz, self.Lt.nnz
        fill_packed(system, "m", self.L)
        fill_packed(system, "mt", self.Lt)

    def stream_matrices(self):
        return [self.L, self.Lt]


class FactoredSolve(FactoredMultiply):
    """``M = (L L^T)^-1`` applied as a forward and a backward sparse triangular solve."""

    precond = _lib.PRECOND_SOLVE

    def __init__(self, L: CsrMatrix, Lt: CsrMatrix | None = None, fwd: TriangularPlan | None = None,
                 bwd: TriangularPlan | None = None, level_stream: bool = True, tile_stream: bool = False) -> None:
        """``tile_stream``: the system is kept in the level order of ``L`` (``LevelOrdering``: checked); both solves of
        a PCG iteration then run as tile-stream batch solves (``DP_SOLVE_TILE_STREAM``; stepped engine, picked by
        ``PcgBatch``) on the iteration's own vectors - the form for batches of 3-D factors."""
        super().__init__(L, Lt)
        self.fwd = fwd or analyse(self.L, upper=False, level_stream=False)
        self.bwd = bwd or analyse(self.Lt, upper=True, level_stream=False)
        self.tile_stream = bool(tile_stream)
        if self.tile_stream:
            n = self.L.n
            if not torch.equal(self.fwd.perm, torch.arange(n, dtype=torch.int32, device=self.L.device)):
                raise _lib.DpcgError("tile_stream=True needs the system in the level order of L (precond.level_ordering)")
            self.fwd_ls = level_ordered_any(self.L, self.fwd)   # identity order: the copy only stores 1 / diagonal
            self.bwd_ls = reversed_copy(self.Lt, self.bwd)
            return
        # level-ordered copies of THIS factor's values (a plan may have been made on another matrix of the same pattern)
        own = lambda plan, m: plan.ls if (plan.ls is not None and plan.ls.matches(m)) else level_ordered(m, plan)
        self.fwd_ls = own(self.fwd, self.L) if level_stream else None
        self.bwd_ls = own(self.bwd, self.Lt) if level_stream else None

    def _apply(self, r):
        if self.tile_stream:
            y = _tile_stream_batch([(self.L, self.fwd, r)], None, [self.fwd_ls], True, [False])[0]
            return _tile_stream_batch([(self.Lt, self.bwd, y)], None, [self.bwd_ls], True, [True])[0]

        def one(m, plan, copy, b):
            if copy is not None:
                return _level_stream_batch([(m, plan, b)], None, [copy])[0]
            return triangular_solve(m, plan, b, algorithm="syncfree")

        return one(self.Lt, self.bwd, self.bwd_ls, one(self.L, self.fwd, self.fwd_ls, r))

    def fill(self, system):
        super().fill(system)
        system.precond = self.precond
        system.fwd_plan, system.bwd_plan = _lib.ptr(self.fwd.plan), _lib.ptr(self.bwd.plan)
        system.fwd_nchunks, system.bwd_nchunks = self.fwd.nchunks, self.bwd.nchunks
        system.fwd_max_level_chunks, system.bwd_max_level_chunks = self.fwd.max_level_chunks, self.bwd.max_level_chunks
        system.solve_algorithm = 0
        if self.tile_stream:  # DP_SOLVE_TILE_STREAM | DP_SOLVE_SHORT_ROWS
            system.solve_algorithm = 1 | (2 if (self.fwd_ls.short_rows and self.bwd_ls.short_rows) else 0)
        for tag, plan, ls in (("fwd", self.fwd, self.fwd_ls), ("bwd", self.bwd, self.bwd_ls)):
            if ls is not None:
                for name, t in (("rowptr", ls.rowptr), ("col", ls.col), ("val", ls.val), ("perm", plan.perm),
                                ("level", ls.level_sorted)):
                    setattr(system, f"{tag}_ls_{name}", _lib.ptr(t))
                if not self.tile_stream and plan.perm_is_identity:
                    setattr(system, f"{tag}_ls_perm", None)  # level-ordered system: vectors by position (bulk copies)


def as_operator(M, device=None) -> _Operator:
    """Coerce the reference's ``M`` argument: ``None`` -> identity, an operator stays, any matrix -> ``CsrOperator``."""
    if M is None:
        return Identity()
    if isinstance(M, _Operator):
        return M
    return CsrOperator(M, device)
