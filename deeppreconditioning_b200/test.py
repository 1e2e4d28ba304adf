"""Drop-in for the hot-path part of ``uibk/deep_preconditioning/test.py``: ``BenchmarkSuite``.

Same class name, constructor fields, private helper names and ``run()`` / ``dump_csv()`` flow as the reference
(``test.py:31-198``); what changes is what the helpers return and where the work runs:

* ``_reconstruct_system``  (test.py:61-68)   -> device :class:`CsrMatrix` via the K1 ``symmetrise`` kernel, not a dense N x N tensor;
* ``_construct_learned``   (test.py:100-105) -> :class:`FactoredMultiply` on the CSR of ``L`` and ``L^T`` (no dense fp32 ``L @ L.T``);
* ``_construct_incomplete_cholesky`` (test.py:81-88) -> same signature and defaults (``icholt(1, 0.1)``; ``ichol0`` when both
  are zero), applied by triangular solves by default (``ic_apply``; SURVEY D2: the reference multiplies by ``L L^T``, which
  approximates ``A`` instead of ``A^-1``, and tags the technique "unstable");
* ``run`` (test.py:119-149) -> the same per-system records, but every technique solves ``batch_systems`` systems per launch
  and the test set is sharded over the ranks of an initialised process group;
* ``preconditioned_conjugate_gradient`` (test.py:138) -> the fused B200 solve.

* ``_compute_kappa`` (test.py:111-113, a dense ``cond(M @ A)``) -> the Lanczos estimate ``lambda_max / lambda_min`` of the
  preconditioned operator from the solve's own CG coefficients (:mod:`.spectrum`, SURVEY §8f-4).

Out of scope (SURVEY §2): dense singular values (``_compute_eigenvalues``, O(n^3)), histogram plots, the ``main()``
pipeline glue (dvc, checkpoint loading).
"""

from __future__ import annotations

import time
from dataclasses import dataclass, field
from pathlib import Path

import numpy as np
import torch

from . import _lib
from .cg import PcgBatch
from .distributed import gather_records, shard_indices
from .precond import (CsrOperator, FactoredMultiply, FactoredSolve, Identity, Jacobi, fsai, incomplete_cholesky0,
                      incomplete_cholesky_threshold, level_ordering, power_pattern)
from .sparse import CsrMatrix

RESULTS_DIRECTORY: Path = Path("./assets/results/")


@dataclass
class BenchmarkSuite:
    """Preconditioner benchmark suite (test.py:31-41).

    Args:
        data_set: The test data set to benchmark on; items are ``(systems_tril, solutions, rhs, original_sizes)``.
        model: The fully convolutional model that maps ``tril(A)`` to ``L``.
        batch_systems: systems solved per kernel launch. The reference walks the test set one system at a time
            (``test.py:121``); the systems are independent, so here every technique solves ``batch_systems`` of them in
            ONE ``dp_pcg_solve_f64`` call (1 = the reference's serial loop). Iteration counts and solutions do not depend on
            it (a system's arithmetic is bitwise the same alone or in any batch).
        shard: with an initialised ``torch.distributed`` process group, rank ``r`` of ``W`` takes systems ``r, r+W, ...``
            and one all-gather at the end of ``run()`` merges the per-system records on every rank (SURVEY §8e).
        ic_apply: how the incomplete-Cholesky comparator is applied: ``"solve"`` (two triangular solves, ``z = L^-T L^-1 r``,
            what an IC preconditioner is) or ``"multiply"`` (the reference's literal ``(L L^T) @ r``, ``test.py:88``, which
            its authors tag "unstable", ``test.py:45``; SURVEY D2).

    Three techniques beyond the reference can be named in ``techniques``: ``"fsai"`` (FSAI on the pattern of ``tril(A)``),
    ``"fsai_power"`` (FSAI on the pattern of ``tril(|A|^fsai_power)``, whose set-up time includes building that pattern)
    and ``"fsai_learned"`` (FSAI on the pattern of the learned factor, whose set-up time includes the model forward that
    supplies the pattern). All are approximate-inverse factors applied like the learned one, two SpMVs per iteration.
    """

    data_set: object
    model: torch.nn.Module
    techniques: tuple[str, ...] = ("vanilla", "jacobi", "incomplete_cholesky", "learned")
    rtol: float = 1e-8       # cg.py:51
    max_iter: int = 1024     # cg.py:51
    level_order_ic: bool = False  # IC(0) comparator on the system renumbered by the factor's level sets (implies IC(0))
    batch_systems: int = 128
    shard: bool = True
    ic_apply: str = "solve"
    ic_fill_in: int = 1        # the arguments run() hands to _construct_incomplete_cholesky: the reference's defaults
    ic_threshold: float = 0.1  # (test.py:81); (0, 0.0) selects IC(0) on the GPU
    fsai_power: int = 2        # "fsai_power": FSAI on tril(|A|^fsai_power)
    kappas: dict = field(default_factory=dict)
    densities: dict = field(default_factory=dict)
    iterations: dict = field(default_factory=dict)
    setups: dict = field(default_factory=dict)
    durations: dict = field(default_factory=dict)
    totals: dict = field(default_factory=dict)
    successes: dict = field(default_factory=dict)
    residuals: dict = field(default_factory=dict)
    variants: dict = field(default_factory=dict)  # technique -> what was actually built (written to variants.csv)

    _STORES = ("kappas", "densities", "iterations", "setups", "durations", "totals", "successes", "residuals")

    def __post_init__(self) -> None:
        for store in self._STORES:
            for name in self.techniques:
                getattr(self, store).setdefault(name, [])

    # ---- operand construction ----------------------------------------------------------------------------------
    def _reconstruct_system(self, system_tril, original_size: int) -> CsrMatrix:
        """Reconstruct the linear system from the sparse lower-triangular tensor (test.py:61-68)."""
        assert system_tril.batch_size == 1, "Set batch size to one for testing"
        matrix = CsrMatrix.from_spconv(system_tril, original_size, mode="symmetrise")
        matrix._lower = CsrMatrix.from_spconv(system_tril, original_size, mode="tril")  # what it was rebuilt from
        return matrix

    def _construct_vanilla(self, matrix: CsrMatrix):
        """The baseline which is no preconditioner (test.py:70-72)."""
        return Identity()

    def _construct_jacobi(self, matrix: CsrMatrix):
        """The Jacobi preconditioner (test.py:74-79)."""
        return Jacobi(matrix)

    def _construct_incomplete_cholesky(self, matrix: CsrMatrix, fill_in: int = 1, threshold: float = 0.1):
        """The incomplete Cholesky preconditioner (test.py:81-88), same defaults as the reference.

        ``fill_in == 0 and threshold == 0.0``: IC(0) on the GPU (``dp_ic0_f64``, stands in for ``ilupp.ichol0``);
        otherwise the threshold factorisation (``dp_icholt_host``, stands in for ``ilupp.icholt(add_fill_in, threshold)``:
        a sequential host algorithm in the reference too). The factor is applied as ``ic_apply`` says."""
        lower = self._tril_of(matrix)
        if fill_in == 0 and threshold == 0.0:
            factor = incomplete_cholesky0(lower)
            self.variants["incomplete_cholesky"] = f"ichol0 (GPU), applied by {self.ic_apply}"
        else:
            factor = incomplete_cholesky_threshold(lower, fill_in, threshold)
            self.variants["incomplete_cholesky"] = f"icholt(add_fill_in={fill_in}, threshold={threshold}) (host), applied by {self.ic_apply}"
        return FactoredSolve(factor) if self.ic_apply == "solve" else FactoredMultiply(factor)

    def _construct_learned(self, system_tril, original_size: int):
        """Our preconditioner (test.py:100-105): model forward, then CSR of ``L`` and ``L^T`` on the device."""
        with torch.no_grad():
            preconditioners_tril = self.model(system_tril)
        lower = CsrMatrix.from_spconv(preconditioners_tril, original_size, mode="tril")
        lower_t = CsrMatrix.from_spconv(preconditioners_tril, original_size, mode="tril_t")
        return FactoredMultiply(lower, lower_t)

    def _construct_fsai(self, matrix: CsrMatrix):
        """FSAI on the pattern of ``tril(A)`` (``precond.fsai``): the classical factor of the learned factor's kind."""
        self.variants["fsai"] = "FSAI on tril(A) (GPU), fp32 values, applied by multiply"
        return fsai(matrix, self._tril_of(matrix))

    def _construct_fsai_power(self, matrix: CsrMatrix):
        """FSAI on the pattern of ``tril(|A|^fsai_power)`` (``precond.power_pattern``, built on the device)."""
        self.variants["fsai_power"] = f"FSAI on tril(|A|^{self.fsai_power}) (GPU), fp32 values, applied by multiply"
        return fsai(matrix, power_pattern(matrix, self.fsai_power))

    def _construct_fsai_learned(self, system_tril, original_size: int):
        """FSAI on the pattern of the ``L`` that ``_construct_learned`` assembles: the classical factor that streams the
        same bytes per iteration as the learned one. Its set-up time covers the model forward that supplies the pattern
        and the assembly of ``A`` from ``system_tril`` besides the FSAI kernel."""
        pattern = self._construct_learned(system_tril, original_size).L
        matrix = CsrMatrix.from_spconv(system_tril, original_size, mode="symmetrise")
        self.variants["fsai_learned"] = "FSAI on the pattern of the learned L (GPU), fp32 values, applied by multiply"
        return fsai(matrix, pattern)

    def _tril_of(self, matrix: CsrMatrix) -> CsrMatrix:
        lower = getattr(matrix, "_lower", None)
        return lower if lower is not None else matrix.tril()

    def _compute_sparsity(self, preconditioner, n: int | None = None) -> float:
        """Density in percent of the explicit ``M`` the reference stores (test.py:107-109): ``100 nnz(M) / n^2``.

        For the factored operators ``nnz(L L^T)`` is counted on the device without forming the product
        (``dp_csr_aat_nnz``); the inverse of an IC factor applied by solves is dense, the reference's number for that
        technique is the density of ``L L^T`` and so is this one."""
        if isinstance(preconditioner, Identity):
            return 100 * n / (n * n)
        if isinstance(preconditioner, Jacobi):
            n = preconditioner.dinv.shape[0]
            return 100 * n / (n * n)
        if isinstance(preconditioner, CsrOperator):
            return 100 * preconditioner.M.nnz / (preconditioner.M.n ** 2)
        lower, lower_t = preconditioner.L, preconditioner.Lt
        count = torch.zeros(1, dtype=torch.int64, device=lower.device)
        with torch.cuda.device(lower.device):
            _lib.check(_lib.lib().dp_csr_aat_nnz(lower.n, _lib.ptr(lower.rowptr), _lib.ptr(lower.col), _lib.ptr(lower_t.rowptr),
                                                 _lib.ptr(lower_t.col), _lib.ptr(count), _lib.stream_ptr(lower.device)),
                       "dp_csr_aat_nnz")
        return 100 * int(count.item()) / (lower.n * lower.n)

    # ---- the benchmark loop ----------------------------------------------------------------------------------------
    def _prepare(self, index: int, device):
        """Lines test.py:122-126 for one item: the system, its right-hand side, the tensor the model consumes."""
        system_tril, _, right_hand_side, original_size = self.data_set[index]
        n = int(original_size[0])
        if not system_tril.indices.is_cuda:
            system_tril = type(system_tril)(system_tril.features.to(device), system_tril.indices.to(device),
                                            system_tril.spatial_shape, system_tril.batch_size)
        matrix = self._reconstruct_system(system_tril, n)
        rhs = right_hand_side[0, :n].squeeze().to(device=device, dtype=torch.float64)  # test.py:124
        return system_tril, matrix, rhs, n

    def run(self) -> None:
        """Run the whole benchmark suite (test.py:119-149): same per-system records, batched launches."""
        import torch.distributed as dist

        device = torch.device("cuda", torch.cuda.current_device())
        total = len(self.data_set)
        sharded = self.shard and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        mine = shard_indices(total, dist.get_rank(), dist.get_world_size()) if sharded else list(range(total))
        step = max(1, int(self.batch_systems))
        rows = {name: [] for name in self.techniques}  # technique -> [index, kappa, density, iterations, setup, duration, success, residual]
        for at in range(0, len(mine), step):
            chunk = mine[at:at + step]
            prepared = [self._prepare(index, device) for index in chunk]
            for name in self.techniques:
                entries, setups, densities = [], [], []
                for system_tril, matrix, rhs, n in prepared:
                    torch.cuda.synchronize()
                    start_time = time.perf_counter()
                    if name in ("learned", "fsai_learned"):
                        preconditioner = getattr(self, f"_construct_{name}")(system_tril, n)
                    elif name == "incomplete_cholesky":
                        preconditioner = self._construct_incomplete_cholesky(matrix, self.ic_fill_in, self.ic_threshold)
                    else:
                        preconditioner = getattr(self, f"_construct_{name}")(matrix)
                    system, b_sys = matrix, rhs
                    if name == "incomplete_cholesky" and self.level_order_ic:
                        # same solve, rows renumbered so that a level of the factor is a contiguous run (precond.LevelOrdering):
                        # the triangular solves read the factor and the vectors coalesced. Counted as set-up time.
                        order = level_ordering(self._tril_of(matrix))
                        renumbered = order.renumber(system_tril)
                        system = CsrMatrix.from_spconv(renumbered, n, mode="symmetrise")
                        system._lower = CsrMatrix.from_spconv(renumbered, n, mode="tril")
                        preconditioner = self._construct_incomplete_cholesky(system, 0, 0.0)
                        b_sys = order.to_level(rhs)
                    torch.cuda.synchronize()
                    setups.append(time.perf_counter() - start_time if name != "vanilla" else 0.0)  # test.py:135
                    densities.append(self._compute_sparsity(preconditioner, n))
                    entries.append((system, b_sys, preconditioner))
                batch = PcgBatch(entries, self.rtol, self.max_iter, history=True)
                torch.cuda.synchronize()
                start_time = time.perf_counter()
                batch.solve()
                torch.cuda.synchronize()
                seconds = time.perf_counter() - start_time
                results = batch.results(seconds)
                # the systems of a launch advance side by side: a system's `duration` (cg.py:69-88) is its share of the
                # launch by iteration count, so that the durations of a technique still add up to the time spent solving
                weight = [max(r.iterations, 1) for r in results]
                for index, result, setup, density, w in zip(chunk, results, setups, densities, weight):
                    duration = seconds * w / sum(weight)
                    # test.py:111-113 takes a dense cond(M @ A); here the solve's own CG coefficients give the Lanczos
                    # estimate lambda_max / lambda_min of the preconditioned operator (spectrum.py)
                    rows[name].append([float(index), result.kappa, density, float(result.iterations), setup, duration,
                                       100.0 * (1 - result.info), result.res])
                del batch, entries
        for name in self.techniques:
            local = torch.tensor(rows[name], dtype=torch.float64).reshape(-1, 8)
            table = gather_records(local, total) if sharded else local
            for row in table.tolist():
                self.kappas[name].append(row[1])
                self.densities[name].append(row[2])
                self.iterations[name].append(int(row[3]))
                self.setups[name].append(row[4])
                self.durations[name].append(row[5])
                self.totals[name].append(row[4] + row[5])
                self.successes[name].append(row[6])
                self.residuals[name].append(row[7])

    def dump_csv(self, directory: Path | None = None) -> None:
        """Dump the durations and iterations to CSV files in the reference's layout (test.py:175-198)."""
        directory = Path(directory) if directory is not None else RESULTS_DIRECTORY
        directory.mkdir(parents=True, exist_ok=True)
        parameters = ["kappas", "densities", "iterations", "setups", "durations", "totals", "successes"]
        with (directory / "table.csv").open(mode="w") as file_io:
            file_io.write("technique," + ",".join(parameters) + "\n")
            for technique in self.techniques:
                line = technique
                for parameter in parameters:
                    line += "," + str(np.mean(getattr(self, parameter)[technique], dtype=float))
                file_io.write(line + "\n")
        with (directory / "totals.csv").open(mode="w") as file_io:
            file_io.write(",".join(self.techniques) + "\n")
            for index in range(len(self.totals[self.techniques[0]])):
                file_io.write(",".join(str(self.totals[t][index]) for t in self.techniques) + "\n")
        if self.variants:  # not in the reference: which comparator variant a column of table.csv holds
            with (directory / "variants.csv").open(mode="w") as file_io:
                file_io.write("technique,variant\n")
                for technique, variant in self.variants.items():
                    file_io.write(f'{technique},"{variant}"\n')
