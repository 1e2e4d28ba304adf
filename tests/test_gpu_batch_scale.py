"""Batched PCG at benchmark scale (run with `-m gpu` on the B200 box): fused batches whose CTAs own many tiles.

The fused engine splits the tiles of the unfinished systems into one contiguous range per CTA and walks each range in
rounds of ROUND_TILES tile-table entries (run_tiles, pcg.cu). The batches here are sized so that the ranges cross system
boundaries, take several rounds, shrink back to one round as systems converge, and so that the active list is compacted
in several chunks. Every system must still give exactly the bits of its own single solve (header of pcg.cu), the same
bits in every engine, and a solution a plain fp64 check on the CPU accepts. A host-side model of the schedule asserts
that each batch really reaches the regime its test is named for, so a retune of the engine cannot quietly disarm a test.
"""
import math
import time
from dataclasses import dataclass

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import deeppreconditioning_b200 as dp
from deeppreconditioning_b200 import _lib as dp_lib
from deeppreconditioning_b200 import model as models, synthetic
from deeppreconditioning_b200.sparse import CsrMatrix
from oracle import operators, pcg
from oracle import sparse as osp
from test_oracle import iteration_tolerance

pytestmark = pytest.mark.gpu

ROUND_TILES = 64        # DPCG_ROUND_TILES in deeppreconditioning_b200/csrc/pcg.cu (kept equal by test_host.py)
TILE_ROWS = 512         # rows of one tile (kTileRows): one CTA, one row per thread
PACKED_CTAS_PER_SM = 2  # the packed engine (544 threads) fits at most two CTAs per SM: the Smem static_assert in pcg.cu
BENCH_SIDE = 316        # the systems of bench.py (config 3)


# ---- host-side model of the fused schedule ----------------------------------------------------------------------------
def tiles_of(n: int) -> int:
    return -(-int(n) // TILE_ROWS)


def cta_ranges(total: int, grid: int):
    """[g0, g1) of every CTA, as run_tiles splits `total` tiles: contiguous, the first `rem` CTAs take one more."""
    quot, rem = divmod(total, grid)
    out = []
    for c in range(grid):
        g0 = c * quot + min(c, rem)
        out.append((g0, g0 + quot + (1 if c < rem else 0)))
    return out


@dataclass
class Schedule:
    """What the fused engine does with a batch: its grid, and the largest tile range of any CTA at every iteration k.

    The active list of iteration k holds the systems with final iteration count >= k: a system is visited by phase A of
    the iteration it finishes in and leaves the list when CTA 0 rebuilds it during that iteration's APPLY1.
    """

    grid: int
    ranges: list

    @classmethod
    def of(cls, tiles, iterations, ctas_per_sm: int) -> "Schedule":
        info = dp_lib.device_info()
        tiles, its = np.asarray(tiles, np.int64), np.asarray(iterations, np.int64)
        grid = min(int(tiles.sum()), info["sm_count"] * ctas_per_sm)  # dp_pcg_solve_f64: min(total_tiles, coop)
        ranges = [-(-int(tiles[its >= k].sum()) // grid) for k in range(int(its.max()) + 1)]
        return cls(grid, ranges)

    def iterations_in(self, lo: int, hi: int) -> int:
        """Iterations whose largest range is in (lo, hi] tiles."""
        return sum(lo < r <= hi for r in self.ranges)

    def report(self, name: str, nsys: int) -> str:
        line = (f"{name}: grid {self.grid} CTAs, {nsys} systems, start {self.ranges[0]} tiles per CTA "
                f"({math.ceil(self.ranges[0] / ROUND_TILES)} table rounds); iterations at > {2 * ROUND_TILES} tiles per CTA: "
                f"{self.iterations_in(2 * ROUND_TILES, 1 << 30)}, at {ROUND_TILES + 1}-{2 * ROUND_TILES}: "
                f"{self.iterations_in(ROUND_TILES, 2 * ROUND_TILES)}, at <= {ROUND_TILES}: {self.iterations_in(0, ROUND_TILES)}")
        print(line)
        return line


def table_rounds(tiles, grid: int):
    """The table rounds (0, 1, ...) of its CTA that each system's tiles fall into at iteration 0."""
    ofs = np.concatenate([[0], np.cumsum(tiles)]).astype(np.int64)
    rnd = np.empty(int(ofs[-1]), np.int64)
    for g0, g1 in cta_ranges(int(ofs[-1]), grid):
        rnd[g0:g1] = np.arange(g1 - g0) // ROUND_TILES
    return [set(rnd[ofs[i]:ofs[i + 1]].tolist()) for i in range(len(tiles))]


# ---- helpers --------------------------------------------------------------------------------------------------------------
def solve(systems, max_iter, **kw):
    """One batch; solutions come back to the host so that several arms can be held side by side."""
    out = dp.pcg_solve_batch(systems, 1e-8, max_iter, history=True, **kw)
    for r in out:
        r.x_hat = r.x_hat.cpu()
    return out


def assert_same_bits(got, want, what):
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.iterations == w.iterations and g.res == w.res, (what, i, g.iterations, w.iterations, g.res, w.res)
        assert g.history == w.history and g.alphas == w.alphas and g.betas == w.betas, (what, i)
        assert torch.equal(g.x_hat.cpu(), w.x_hat.cpu()), (what, i)


def singles(systems, max_iter, **kw):
    """Every system alone (the grid is sized to its own tiles)."""
    return [dp.pcg_solve(A, b, M, x0, max_iter=max_iter, history=True, **kw) for A, b, M, x0 in systems]


def true_residual(A: CsrMatrix, b: torch.Tensor, x: torch.Tensor) -> float:
    """||b - A x|| / ||b|| in fp64 on the CPU, from the device operands copied back."""
    a = osp.to_scipy(*A.to_host())
    bh, xh = b.cpu().numpy(), x.cpu().numpy()
    return float(np.linalg.norm(bh - a @ xh) / np.linalg.norm(bh))


def oracle_operator(name: str, A: CsrMatrix, M):
    """The operator of test_oracle.build_operator, on the device operands copied back."""
    if name == "identity":
        return operators.Identity()
    if name == "jacobi":
        return operators.Jacobi(osp.to_scipy(*A.to_host()).diagonal())
    if name == "multiply":
        return operators.FactoredMultiply(*M.L.to_host())
    raise KeyError(name)


def assert_oracle(A, b, M, x0, name, got, max_iter):
    o = pcg.preconditioned_conjugate_gradient(osp.to_torch_csr(*A.to_host()), b.cpu(), oracle_operator(name, A, M),
                                              x0=None if x0 is None else x0.cpu(), max_iter=max_iter)
    assert abs(got.iterations - o.iterations) <= iteration_tolerance(o.iterations), (name, got.iterations, o.iterations)
    np.testing.assert_allclose(got.history[:11], o.history[:11], rtol=1e-8)


def bench_systems(cuda, indices):
    """(A, b, FactoredMultiply(L, L^T)) of bench.py's systems, built the way its build_chunk does: on the device, the
    random-init PreconditionerNet on the GPU, eight systems per CNN forward."""
    torch.manual_seed(69)  # test.py:205
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS).to(cuda)
    out = []
    for at in range(0, len(indices), 8):
        st, _, rhs, sizes = synthetic.make_batch("poisson2d", BENCH_SIDE, indices[at:at + 8], device=cuda)
        with torch.no_grad():
            learned = net(st)
        for k, n in enumerate(sizes):
            A = CsrMatrix.from_spconv(st, n, "symmetrise", batch=k)
            L = CsrMatrix.from_spconv(learned, n, "tril", batch=k)
            Lt = CsrMatrix.from_spconv(learned, n, "tril_t", batch=k)
            out.append((A, rhs[k, :n].to(torch.float64), dp.FactoredMultiply(L, Lt), None))
        del st, learned
    return out


def poisson_systems(cuda, side, seeds, sigma=0.5, pad_to=None):
    """Variable-coefficient 2-D systems of one size, one make_batch call: [(A, b, n)]."""
    st, _, rhs, sizes = synthetic.make_batch("poisson2d", side, seeds, sigma, device=cuda, pad_to=pad_to)
    n = pad_to or sizes[0]
    out = [(CsrMatrix.from_spconv(st, n, "symmetrise", batch=k), rhs[k, :n].to(torch.float64), n) for k in range(len(seeds))]
    del st
    return out


# ---- 2. a large mixed batch through the benchmarked path (packed copies, fused engine) -------------------------------------
MIXED_MAX_ITER = 640  # the Jacobi systems below converge between ~190 and ~570 iterations; the bench systems saturate


def mixed_batch(cuda):
    """16 bench systems (316^2, CNN factor, multiply mode) among 615 variable-coefficient 2-D systems of sides 96..256
    (distinct seeds, three coefficient contrasts, Jacobi or identity, a nonzero x0 on a few), in a fixed shuffled order."""
    systems, names = [], []
    gen = torch.Generator().manual_seed(7)
    for gi, side in enumerate(range(96, 257, 4)):
        for q, sigma in enumerate((0.3, 0.5, 0.8)):
            js = [j for j in range(15) if j % 3 == q]
            for j, (A, b, n) in zip(js, poisson_systems(cuda, side, [5000 + 15 * gi + j for j in js], sigma)):
                name = "identity" if j % 5 == 4 else "jacobi"
                x0 = torch.randn(n, generator=gen, dtype=torch.float64).to(cuda) if j == 7 and gi % 8 == 0 else None
                systems.append((A, b, dp.Identity() if name == "identity" else dp.Jacobi(A), x0))
                names.append(name)
    order = np.random.default_rng(11).permutation(len(systems)).tolist()
    systems, names = [systems[i] for i in order], [names[i] for i in order]
    for i, s in zip(range(20, 20 + 40 * 16, 40), bench_systems(cuda, list(range(16)))):  # spread over the whole list
        systems.insert(i, s)
        names.insert(i, "multiply")
    return systems, names


def test_large_mixed_batch_crosses_systems_and_table_rounds(cuda):
    """~630 systems, ~43k tiles: each CTA of the packed engine starts with a range of ~147 tiles (three table rounds, no
    early issue) crossing several systems, falls to 65-128 tiles and then to one round as systems converge, while the
    active list (more than 512 systems) is compacted in chunks. Every system is bitwise its own single solve and the same
    in the fused packed, fused fp64-stream and stepped engines; converged ones pass a plain fp64 residual check."""
    t0 = time.perf_counter()
    systems, names = mixed_batch(cuda)
    tiles = [tiles_of(s[0].n) for s in systems]
    nsys, max_iter = len(systems), MIXED_MAX_ITER

    got = solve(systems, max_iter)
    for A, _, M, _ in systems:
        assert A._packed and all(m._packed for m in M.stream_matrices()), "the packed engine did not run"
    its = [r.iterations for r in got]

    # bite guards: the batch went through the regimes this test is about
    sched = Schedule.of(tiles, its, PACKED_CTAS_PER_SM)
    sched.report("large mixed batch (packed)", nsys)
    print(f"  iterations: {len(set(its))} distinct, min {min(its)}, max {max(its)}, "
          f"{sum(i == max_iter for i in its)} saturated at max_iter {max_iter}")
    assert nsys > 512, "the active list must need more than one 512-system chunk"
    assert sched.ranges[0] > 2 * ROUND_TILES, "the start range must take at least three table rounds"
    assert sched.iterations_in(ROUND_TILES, 2 * ROUND_TILES) >= 20
    assert sched.iterations_in(0, ROUND_TILES) >= 20
    assert len(set(its)) >= 100
    assert all(i < max_iter for i, n in zip(its, names) if n == "jacobi"), "every Jacobi system must converge"
    assert all(i == max_iter for i, n in zip(its, names) if n == "multiply")

    # the same batch in the other arms, bit for bit
    assert_same_bits(solve(systems, max_iter, pack=False), got, "fused, fp64 stream")
    assert_same_bits(solve(systems, max_iter, engine="stepped", check_every=1), got, "stepped, every 1")
    assert_same_bits(solve(systems, max_iter, engine="stepped"), got, "stepped")
    # each system alone: one CTA per tile (a 316^2 system is 196 tiles on 196 CTAs) - a wholly different schedule
    assert_same_bits(singles(systems, max_iter), got, "single solves")

    # plain fp64 references on the CPU
    for (A, b, M, x0), r in zip(systems, got):
        if r.iterations < max_iter:
            assert r.res < 1e-8
            assert true_residual(A, b, r.x_hat) < 2e-4
        else:
            assert r.res == r.history[-1] and len(r.history) == max_iter + 1
    rounds = table_rounds(tiles, sched.grid)
    sample = [i for i, n in enumerate(names) if n == "multiply"][:2]
    for want in (1, 2):  # systems streamed in the second and third table round of some CTA
        sample += [i for i in range(nsys) if want in rounds[i] and names[i] != "multiply" and i not in sample][:4]
    sample += [i for i in range(nsys) if systems[i][3] is not None][:2]  # nonzero x0
    sample += [i for i in range(nsys) if names[i] == "identity" and its[i] < max_iter and i not in sample][:2]
    assert len(sample) >= 12
    for i in sample:
        A, b, M, x0 = systems[i]
        assert_oracle(A, b, M, x0, names[i], got[i], max_iter)
    print(f"  wall time {time.perf_counter() - t0:.1f} s")
    del systems, got
    torch.cuda.empty_cache()


# ---- 3. the exact round boundary (fp64 stream, fused engine) ---------------------------------------------------------------
BOUNDARY_MAX_ITER = 1000


@pytest.fixture(scope="module")
def boundary_base(cuda):
    """k Jacobi systems of 316^2 (196 tiles each, distinct seeds) and their single solves, shared by the three batches."""
    info = dp_lib.device_info()
    grid = info["sm_count"] * info["pcg_ctas_per_sm"]  # the unpacked engine's cooperative grid (dp_device_info)
    k = (ROUND_TILES * grid - 2) // tiles_of(BENCH_SIDE ** 2)
    base = []
    for at in range(0, k, 16):
        for A, b, _ in poisson_systems(cuda, BENCH_SIDE, list(range(9000 + at, 9000 + min(k, at + 16)))):
            base.append((A, b, dp.Jacobi(A), None))
    yield grid, base, singles(base, BOUNDARY_MAX_ITER)
    del base
    torch.cuda.empty_cache()


@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_batch_at_the_table_round_boundary(cuda, boundary_base, delta):
    """ROUND_TILES * grid + delta tiles: at -1 and 0 every CTA holds one round of at most ROUND_TILES tiles (and issues the
    next phase's first items early); at +1 CTA 0 gets a one-tile second round. Bitwise the single solves and the stepped
    engine, true residual of every system."""
    grid, base, base_singles = boundary_base
    target = ROUND_TILES * grid + delta
    filler_tiles = target - sum(tiles_of(s[0].n) for s in base)
    assert 1 <= filler_tiles <= 4 * tiles_of(BENCH_SIDE ** 2)
    side = math.isqrt(TILE_ROWS * filler_tiles)
    pad = None if tiles_of(side * side) == filler_tiles else TILE_ROWS * (filler_tiles - 1) + 1  # one row in its last tile
    (A, b, _), = poisson_systems(cuda, side, [9500 + delta], pad_to=pad)
    systems = base + [(A, b, dp.Jacobi(A), None)]
    tiles = [tiles_of(s[0].n) for s in systems]
    assert sum(tiles) == target, (sum(tiles), target)
    assert tiles[-1] == filler_tiles

    got = solve(systems, BOUNDARY_MAX_ITER, pack=False)
    its = [r.iterations for r in got]
    sched = Schedule.of(tiles, its, dp_lib.device_info()["pcg_ctas_per_sm"])
    sched.report(f"round boundary {delta:+d} (fp64 stream)", len(systems))
    ranges = cta_ranges(sum(tiles), sched.grid)
    assert sched.grid == grid
    assert max(g1 - g0 for g0, g1 in ranges) == ROUND_TILES + max(delta, 0) == sched.ranges[0]
    assert (ranges[0][1] - ranges[0][0] == ROUND_TILES + 1) == (delta == 1)
    assert min(its) > 20 and max(its) < BOUNDARY_MAX_ITER  # the boundary holds for many iterations; all converge

    assert_same_bits(got[:-1], base_singles, "single solves")
    assert_same_bits(got[-1:], singles(systems[-1:], BOUNDARY_MAX_ITER), "single solve of the filler")
    assert_same_bits(solve(systems, BOUNDARY_MAX_ITER, engine="stepped"), got, "stepped")
    for (A_, b_, _, _), r in zip(systems, got):
        assert r.res < 1e-8 and true_residual(A_, b_, r.x_hat) < 2e-4
    del systems, got
    torch.cuda.empty_cache()


# ---- 4. many small systems: active-list compaction across chunks ------------------------------------------------------------
SMALL_SIZES = [1, 2, 3, 31, 33, 511, 512, 513]
SMALL_REPEATS = 72  # 8 sizes x 2 kinds x 72 = 1152 systems: three 512-system chunks in rebuild_active


def small_systems(cuda):
    """Random tridiagonal SPD systems (fp32 values; diagonal 2 + a shift spread over 1e-3..3: 5 to ~100 iterations) and
    2-D systems of 5^2 / 22^2 cells padded with unit rows, of every size in SMALL_SIZES, interleaved; Identity and Jacobi
    alternate."""
    rng = np.random.default_rng(2024)
    tri, poisson = [], []
    for n in SMALL_SIZES:
        for _ in range(SMALL_REPEATS):
            if n == 1:
                m = sp.csr_matrix(np.array([[1.0 + rng.random()]]))
            else:
                diag = 2.0 + 10.0 ** rng.uniform(-3, 0.5) + 0.02 * rng.random(n)
                m = sp.diags([-np.ones(n - 1), diag, -np.ones(n - 1)], [-1, 0, 1], format="csr")
            # fp32 values, like the synthetic systems: the matrix has an exact packed copy (the whole batch streams packed)
            m.data = m.data.astype(np.float32).astype(np.float64)
            tri.append((CsrMatrix.from_scipy(m, cuda), torch.from_numpy(rng.standard_normal(n)).to(cuda)))
        side = max(s for s in (1, 5, 22) if s * s <= n)
        seeds = [20000 + 100 * n + j for j in range(SMALL_REPEATS)]
        poisson += [(A, b) for A, b, _ in poisson_systems(cuda, side, seeds, pad_to=None if side * side == n else n)]
    systems, names = [], []
    for i, (A, b) in enumerate(x for pair in zip(tri, poisson) for x in pair):
        name = "jacobi" if (i // 2) % 2 else "identity"
        systems.append((A, b, dp.Jacobi(A) if name == "jacobi" else dp.Identity(), None))
        names.append(name)
    return systems, names


def test_many_small_systems_compact_across_chunks(cuda):
    """1152 systems of 1..513 rows (one or two tiles each, many per CTA) converging at many different iterations, so
    rebuild_active carries its counts across three 512-system chunks again and again. Fused packed, fused fp64 stream and
    stepped agree bit for bit and with the single solves; every system is within one iteration of the oracle with the
    same preconditioner and has a true residual below 2e-4."""
    t0 = time.perf_counter()
    systems, names = small_systems(cuda)
    max_iter = 3000
    got = solve(systems, max_iter)
    assert all(s[0]._packed for s in systems), "the packed engine did not run"
    its = [r.iterations for r in got]
    tiles = [tiles_of(s[0].n) for s in systems]
    Schedule.of(tiles, its, PACKED_CTAS_PER_SM).report("many small systems (packed)", len(systems))
    print(f"  iterations: {len(set(its))} distinct, min {min(its)}, max {max(its)}")
    assert len(systems) > 2 * 512 and sorted({s[0].n for s in systems}) == SMALL_SIZES
    assert len(set(its)) >= 30 and max(its) < max_iter

    assert_same_bits(solve(systems, max_iter, pack=False), got, "fused, fp64 stream")
    assert_same_bits(solve(systems, max_iter, engine="stepped"), got, "stepped")
    assert_same_bits(singles(systems, max_iter), got, "single solves")
    for (A, b, M, _), name, r in zip(systems, names, got):
        o = pcg.preconditioned_conjugate_gradient(osp.to_torch_csr(*A.to_host()), b.cpu(), oracle_operator(name, A, M),
                                                  max_iter=max_iter)
        assert abs(r.iterations - o.iterations) <= 1, (A.n, name, r.iterations, o.iterations)
        assert true_residual(A, b, r.x_hat) < 2e-4, (A.n, name)
    print(f"  wall time {time.perf_counter() - t0:.1f} s")
    del systems, got
    torch.cuda.empty_cache()
