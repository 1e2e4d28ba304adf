"""CPU tests of the host side: the C-ABI library loads and exports what include/dpcg.h declares, descriptor layout,
no-CPU-fallback behaviour, sharding and the result gather (gloo, world_size 2). No kernel is launched here."""
import ctypes
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import helpers
from deeppreconditioning_b200 import _lib, build, distributed
from deeppreconditioning_b200.cg import PcgResult

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.lib()


def test_library_exports_every_declared_symbol(lib):
    header = (ROOT / "include" / "dpcg.h").read_text()
    declared = set(re.findall(r"\b(dp_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations found"
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.dp_version() == 100
    assert lib.dp_status_string(0) == b"ok" and b"aligned" in lib.dp_status_string(2)


def test_descriptor_layout_and_size_queries(lib):
    assert ctypes.sizeof(_lib.PcgSystem) == 10 * 4 + 38 * 8
    assert _lib.PcgSystem.a_col16.offset == 40 + 29 * 8 and _lib.PcgSystem.mt_tile_base.offset == 40 + 37 * 8
    assert lib.dp_csr_pack_tile_rows() == 512
    assert ctypes.sizeof(_lib.PcgParams) == 24
    assert _lib.PcgSystem.a_rowptr.offset == 40 and _lib.PcgSystem.history.offset == 40 + 27 * 8 and _lib.PcgSystem.coef.offset == 40 + 28 * 8
    for n in (1, 31, 32, 33, 511, 512, 513, 99856):
        pad = (n + 31) // 32 * 32
        tiles = (n + 511) // 512
        assert lib.dp_pcg_work_doubles(n) == 8 * pad + 5 * ((tiles + 31) // 32 * 32) + 32
    assert lib.dp_pcg_workspace_bytes(1) >= 512 and lib.dp_pcg_workspace_bytes(1024) > lib.dp_pcg_workspace_bytes(1)
    level_ptr = np.array([0, 1, 33, 97, 100], np.int32)
    assert lib.dp_sptrsv_plan_chunks(4, level_ptr.ctypes.data) == 1 + 1 + 2 + 1
    assert lib.dp_sptrsv_workspace_bytes() >= 8


def test_argument_validation_without_a_gpu(lib):
    """Entry points reject bad arguments before touching CUDA."""
    assert lib.dp_spmv_csr_f64(-1, 0, None, None, None, None, None, None) == 1
    assert lib.dp_spmv_csr_f64(4, 4, 16, 20, 32, 48, 64, None) == 2  # col pointer 20 is not 16-byte aligned
    assert lib.dp_csr_from_coo(None, None, 5, 0, 4, 0, None, None, None, None, None, None, 0, None) == 1
    assert lib.dp_csr_pack(4, 4, 16, 32, 48, 64, 80, None, 96, None) == 1  # no tile_base
    assert lib.dp_csr_pack(4, 4, 16, 32, 48, 66, 80, 96, 112, None) == 2   # col16 pointer 66 is not 16-byte aligned
    assert lib.dp_spmv_csr_packed_f64(4, 4, 16, 32, 48, None, 64, 80, None) == 1
    params = _lib.PcgParams(1e-8, 10, 0, 1, 0)
    assert lib.dp_pcg_solve_f64(None, 1, ctypes.byref(params), None, None, 0, None) == 1


def test_tile_stream_descriptors_limits_and_validation(lib):
    """dp_sptrsv_ts_*: size queries, limits and argument checks that run before any CUDA call."""
    limits = np.zeros(2, np.int32)
    lib.dp_sptrsv_ts_limits(limits.ctypes.data)
    assert limits[0] >= 4 * 512 and limits[1] == 4, "a 512-row tile of a 7-point factor is one pipeline item; rows of <= 4 entries"
    assert ctypes.sizeof(_lib.TrsvLsSystem) == 4 * 4 + 7 * 8 and _lib.TrsvLsSystem.flags.offset == 12
    descs = (_lib.TrsvLsSystem * 2)()
    for d, n, perm in zip(descs, (1000, 513), (None, 64)):
        d.n, d.nnz, d.upper, d.flags = n, 4 * n, 0, 0
        d.rowptr_p, d.col_p, d.val_p, d.perm, d.b, d.x = 16, 32, 48, perm, 64, 80
    base = lib.dp_sptrsv_ts_workspace_bytes(descs, 0)
    # position space: no vectors in the workspace; original numbering: b_pos and x_pos (two padded vectors)
    assert lib.dp_sptrsv_ts_workspace_bytes(descs, 1) - base < 4096
    assert lib.dp_sptrsv_ts_workspace_bytes(descs, 2) - lib.dp_sptrsv_ts_workspace_bytes(descs, 1) >= 2 * 513 * 8
    flag = ctypes.c_void_p(256)
    assert lib.dp_sptrsv_ts_solve_batch_f64(descs, 2, flag, None, 0, None) == 1          # no workspace
    assert lib.dp_sptrsv_ts_solve_batch_f64(descs, 2, flag, ctypes.c_void_p(4096), 64, None) == 3  # workspace too small
    assert lib.dp_sptrsv_ts_solve_batch_f64(None, 2, flag, ctypes.c_void_p(4096), 1 << 30, None) == 1


def test_level_ordering_helpers_on_the_host():
    """precond.LevelOrdering is index plumbing around the K3 analysis: to_level / from_level are inverse gathers and
    renumber() maps the COO sites (batch column untouched) - checked on CPU tensors with a hand-made permutation."""
    from deeppreconditioning_b200 import model as models
    from deeppreconditioning_b200.precond import LevelOrdering

    perm = torch.tensor([2, 0, 3, 1])
    inv = torch.empty(4, dtype=torch.int32)
    inv[perm] = torch.arange(4, dtype=torch.int32)
    order = LevelOrdering(perm, inv, 3)
    v = torch.tensor([10.0, 11.0, 12.0, 13.0], dtype=torch.float64)
    assert order.to_level(v).tolist() == [12.0, 10.0, 13.0, 11.0] and torch.equal(order.from_level(order.to_level(v)), v)
    st = models.SparseConvTensor(torch.ones(3, 1), torch.tensor([[0, 0, 0], [0, 2, 0], [0, 3, 1]], dtype=torch.int32), [4, 4], 1)
    got = order.renumber(st)
    assert got.indices.tolist() == [[0, 1, 1], [0, 0, 1], [0, 2, 3]] and got.indices.dtype == torch.int32
    assert torch.equal(got.features, st.features) and got.spatial_shape == [4, 4] and got.batch_size == 1


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a box WITHOUT a GPU")
def test_no_cpu_fallback():
    """The product path raises instead of computing on the CPU."""
    import deeppreconditioning_b200 as dp

    p = helpers.problem("poisson2d", 8, 0, 0.5, None)
    from oracle import sparse as osp

    with pytest.raises((_lib.DpcgError, RuntimeError, AssertionError)):
        dp.preconditioned_conjugate_gradient(osp.to_torch_csr(*p.A), p.b, None)
    with pytest.raises((_lib.DpcgError, RuntimeError, AssertionError)):
        dp.CsrMatrix.from_spconv(p.systems_tril, p.n, "tril")


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", tmp_path / "libdpcg.so")
    with pytest.raises(_lib.DpcgError, match="no CPU fallback"):
        _lib.lib()


def test_shard_indices_partition():
    for n, world in [(1024, 8), (10, 4), (3, 8), (0, 2)]:
        shards = [distributed.shard_indices(n, r, world) for r in range(world)]
        assert sorted(i for s in shards for i in s) == list(range(n))
        assert max(map(len, shards)) - min(map(len, shards)) <= 1


def test_gather_records_single_process():
    results = [PcgResult(0.0, 10 + i, 0, torch.zeros(1), 1e-9 * (i + 1)) for i in range(3)]
    rec = distributed.make_records([2, 0, 1], results, [1.0, 2.0, 3.0])
    out = distributed.gather_records(rec, 3)
    assert out[:, 0].tolist() == [0.0, 1.0, 2.0] and out[:, 1].tolist() == [11.0, 12.0, 10.0]


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from deeppreconditioning_b200 import distributed
from deeppreconditioning_b200.cg import PcgResult
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
rank, n = dist.get_rank(), 7
mine = distributed.shard_indices(n, rank, 2)
res = [PcgResult(0.0, 100 + i, 0, torch.zeros(1), 1e-9 * i) for i in mine]
out = distributed.gather_records(distributed.make_records(mine, res, [float(i) for i in mine]), n)
assert out.shape == (n, 4), out.shape
assert out[:, 0].tolist() == [float(i) for i in range(n)]
assert out[:, 1].tolist() == [100.0 + i for i in range(n)]
assert out[:, 3].tolist() == [float(i) for i in range(n)]
# the 8-column records of BenchmarkSuite.run (index, kappa, density, iterations, setup, duration, success, residual)
wide = torch.tensor([[float(i), 2.0 * i, 0.5, 10.0 + i, 0.1, 0.2, 100.0, 1e-9] for i in mine], dtype=torch.float64).reshape(-1, 8)
table = distributed.gather_records(wide, n)
assert table.shape == (n, 8) and table[:, 3].tolist() == [10.0 + i for i in range(n)] and table[:, 1].tolist() == [2.0 * i for i in range(n)]
# the bench's step schedule: every system of a step is solved by exactly one rank, a rank's systems are its shard's
import argparse, importlib.util
spec = importlib.util.spec_from_file_location("bench", {root!r} + "/bench.py"); bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
args = argparse.Namespace(systems_total=32, step_systems=8)
for step in range(6):
    both = [bench.step_indices(args, step, r, 2) for r in range(2)]
    assert sorted(both[0] + both[1]) == list(range((step % 4) * 8, (step % 4) * 8 + 8))
    assert all(i % 2 == r for r in range(2) for i in both[r])
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_gather_records_gloo_world_size_2(tmp_path):
    """The N>1 path of SURVEY §8e on CPU: interleaved shards, one all_gather of fixed-size records (ragged: 4 + 3)."""
    port = 29500 + os.getpid() % 2000
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=str(ROOT), port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    for r, proc in enumerate(procs):
        out, _ = proc.communicate(timeout=180)
        assert proc.returncode == 0, out.decode()
        assert f"rank {r} ok" in out.decode()


def test_sludge_pattern_data_set_reads_the_reference_layout(tmp_path):
    """data_set.py:73-130 restated literally on files written in the generator's layout (generate_data.py:109-111):
    80/20 split over sorted folders, lower triangle, padding with trivial equations to the largest system."""
    import scipy.sparse as sp
    from deeppreconditioning_b200 import synthetic
    from deeppreconditioning_b200.data_set import SludgePatternDataSet, write_case

    root = tmp_path / "raw"
    sides = [5, 7, 4, 6, 5, 3, 8, 4, 6, 5]
    for k, side in enumerate(sides):
        rows, cols, vals, rhs = synthetic.poisson2d_tril(side, 0.5, k)
        low = sp.coo_matrix((vals.astype(np.float64), (rows, cols)), shape=(side * side,) * 2)
        full = (low + sp.tril(low, -1).T).tocoo()
        write_case(root / "sludge_patterns" / f"case_{k:04}", full, rhs, np.linspace(0, 1, side * side))
    data = SludgePatternDataSet("test", 1, shuffle=False, root=root, device="cpu")
    train = SludgePatternDataSet("train", 2, shuffle=False, root=root, device="cpu")
    assert len(data) == 2 and len(train) == 4 and data.dof_max == train.dof_max == 64
    for index, folder in enumerate(sorted((root / "sludge_patterns").glob("case_*"))[8:]):
        tril, solutions, right_hand_sides, sizes = data[index]
        # the reference's arithmetic, literally (data_set.py:84-128)
        rows, columns, _, original_size, values = np.load(folder / "matrix.npz").values()
        n, difference = int(original_size[0]), 64 - int(original_size[0])
        (keep,) = np.where(rows >= columns)
        rows, columns, values = rows[keep], columns[keep], values[keep]
        rows = np.append(rows, np.arange(n, 64))
        columns = np.append(columns, np.arange(n, 64))
        values = np.append(values, np.ones((difference,)))
        assert sizes == (n,) and tril.batch_size == 1 and list(tril.spatial_shape) == [64, 64]
        assert tril.features.dtype == torch.float32 and tril.indices.dtype == torch.int32
        assert np.array_equal(tril.features.numpy(), np.expand_dims(values, -1).astype(np.float32))
        assert np.array_equal(tril.indices.numpy(), np.column_stack((np.zeros(len(values)), rows, columns)).astype(np.int32))
        want_rhs = np.pad(np.loadtxt(folder / "right_hand_side.csv"), (0, difference), constant_values=1)
        assert np.array_equal(right_hand_sides.numpy(), want_rhs[None, :].astype(np.float32))
        assert solutions.shape == (1, 64) and float(solutions[0, -1]) == 1.0
    pair = train[1]
    assert pair[3] == (16, 36) and pair[0].batch_size == 2 and set(pair[0].indices[:, 0].tolist()) == {0, 1}
    with pytest.raises(AssertionError):
        SludgePatternDataSet("validation", 1, root=root, device="cpu")


# ---- the CNN side (SURVEY §8f-1): sparse convolution against the dense one, reference checkpoint layout ----------------
@pytest.mark.parametrize("k,padding", [(1, (0, 0)), (2, (1, 0)), (2, (0, 1)), (3, (1, 1))])
def test_sparse_conv_is_the_dense_conv(k, padding):
    """SparseConv2d == torch's dense conv2d on the densified input, at exactly the sites whose window holds an active
    input (spconv's regular, pattern-dilating convolution, model.py:27-40); everything else stays inactive."""
    from deeppreconditioning_b200 import model as models

    torch.manual_seed(3)
    cin, cout, h, w, batch = 5, 7, 19, 23, 2
    dense = torch.randn(batch, h, w, cin) * (torch.rand(batch, h, w, 1) < 0.15)
    x = models.SparseConvTensor.from_dense(dense)
    conv = models.SparseConv2d(cin, cout, k, padding=padding)
    out = conv(x)
    want = torch.nn.functional.conv2d(dense.permute(0, 3, 1, 2), conv.weight.permute(0, 3, 1, 2), conv.bias, padding=padding)
    active = torch.nn.functional.conv2d((dense != 0).any(-1, keepdim=True).permute(0, 3, 1, 2).float(),
                                        torch.ones(1, 1, k, k), padding=padding) > 0
    assert list(want.shape[2:]) == out.spatial_shape
    idx = out.indices.long()
    got_mask = torch.zeros_like(active[:, 0])
    got_mask[idx[:, 0], idx[:, 1], idx[:, 2]] = True
    assert torch.equal(got_mask, active[:, 0]) and out.indices.shape[0] == int(active.sum())  # no duplicates, no extras
    torch.testing.assert_close(out.features, want.permute(0, 2, 3, 1)[idx[:, 0], idx[:, 1], idx[:, 2]], rtol=1e-5, atol=1e-5)


def test_reference_checkpoint_layout_loads():
    """A state dict with the reference's names and spconv 2.x shapes (spconv.SparseSequential of SparseConv2d [out,k,k,in]
    and nn.PReLU, model.py:27-40; 20 678 parameters = the 87 844-byte best.pt of dvc.lock:51-55) loads strictly, and the
    weights land where the forward pass reads them."""
    from deeppreconditioning_b200 import model as models

    channels = models.DEFAULT_CHANNELS
    torch.manual_seed(11)
    state, index = {}, 0
    specs = [(channels[0], channels[1], 1)] + [(a, b, 2) for a, b in zip(channels[1:-2], channels[2:-1])] + [(channels[-2], channels[-1], 1)]
    for n_layer, (cin, cout, k) in enumerate(specs):
        state[f"layers.{index}.weight"] = 0.2 * torch.randn(cout, k, k, cin)
        state[f"layers.{index}.bias"] = 0.2 * torch.randn(cout)
        index += 1
        if n_layer < len(specs) - 1:
            state[f"layers.{index}.weight"] = torch.rand(1)  # nn.PReLU
            index += 1
    assert sum(t.numel() for t in state.values()) == 20678
    net = models.PreconditionerNet(channels)
    assert set(net.state_dict()) == set(state)
    net.load_state_dict(state, strict=True)
    # a 2x2 layer evaluated by hand: out = sum_taps in[y + ky - ph, x + kx - pw] @ W[:, ky, kx, :].T + bias
    layer = net.layers[2]
    x = models.SparseConvTensor(torch.randn(1, 16), torch.tensor([[0, 4, 6]], dtype=torch.int32), [9, 9], 1)
    out = layer(x)
    for site, feat in zip(out.indices.tolist(), out.features):
        ky, kx = 4 - site[1] + layer.padding[0], 6 - site[2] + layer.padding[1]
        torch.testing.assert_close(feat, x.features[0] @ state["layers.2.weight"][:, ky, kx, :].T + state["layers.2.bias"])
    st, _, _, _ = helpers.problem("poisson2d", 16).systems_tril, None, None, None
    with torch.no_grad():
        lower = net(st)
    assert (lower.features[lower.indices[:, 1] < lower.indices[:, 2]] == 0).all()
    assert (lower.features[lower.indices[:, 1] == lower.indices[:, 2]] > 0).all()


def test_bench_line_helpers():
    """bench.py: both arms print the same `config` dictionary (the driver compares them), and the algorithmic byte count
    follows the bytes per stored entry of the stream the engine used (6 from packed copies, 12 from the fp64 CSR)."""
    import argparse
    import sys

    sys.path.insert(0, str(ROOT))
    import bench

    for cfg, gpus in (("c3", 1), ("c3", 8), ("c5", 8)):
        args = argparse.Namespace(config=cfg, gpus=gpus, systems_total=1024, step_systems=128, side=316, net="net",
                                  c5_side=256, c5_per_gpu=8)
        config = bench.workload_config(args)
        assert config == bench.workload_config(args) and "workload" in config and "l2" in config
        assert all(isinstance(v, (str, int)) for v in config.values()), "static values only: no run findings in config"
    assert "1024 x poisson2d 316x316" in bench.workload_config(argparse.Namespace(
        config="c3", gpus=1, systems_total=1024, step_systems=128, side=316, net="net", c5_side=256, c5_per_gpu=8))["workload"]
    n, nnz_a, nnz_l = 99856, 498016, 1494660
    assert bench.iter_bytes(n, nnz_a, nnz_l) == 12 * nnz_a + 24 * nnz_l + 132 * n + 12
    assert bench.iter_bytes(n, nnz_a, nnz_l) - bench.iter_bytes(n, nnz_a, nnz_l, 6) == 6 * (nnz_a + 2 * nnz_l)


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: float64 arrays of the last step's results, solutions sampled at positions that do not
    change from run to run once a step's solutions exceed the budget, and the whole dump under 64 MB."""
    import sys

    sys.path.insert(0, str(ROOT))
    import bench

    gen = torch.Generator().manual_seed(0)
    results = [PcgResult(0.0, 10 + i, 0, torch.randn(20000, dtype=torch.float64, generator=gen), 1e-9 * i) for i in range(3)]
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, [7, 9, 11], results, 4096)  # as if the step had 4096 systems: sampled
    got = {f.name: np.load(f) for f in (tmp_path / "a").iterdir()}
    assert set(got) == {"systems.npy", "iterations.npy", "res.npy", "x_hat.npy", "x_positions.npy"}
    assert all(a.dtype == np.float64 for a in got.values())
    assert all(np.array_equal(a, np.load(tmp_path / "b" / name)) for name, a in got.items())
    pos = got["x_positions.npy"].astype(np.int64)
    assert 0 < len(pos) < 20000 and np.all(np.diff(pos) > 0) and pos[-1] < 20000
    assert np.array_equal(got["x_hat.npy"], np.stack([r.x_hat.numpy()[pos] for r in results]))
    assert got["systems.npy"].tolist() == [7, 9, 11] and got["iterations.npy"].tolist() == [10, 11, 12]
    assert got["res.npy"].tolist() == [r.res for r in results]
    bench.dump_outputs(tmp_path / "c", [0], results[:1], 1)  # fits: every position
    assert np.array_equal(np.load(tmp_path / "c" / "x_hat.npy")[0], results[0].x_hat.numpy())
    x = torch.randn(99856, dtype=torch.float64, generator=gen)  # the default c3 step: 128 systems of 99 856 unknowns
    bench.dump_outputs(tmp_path / "d", list(range(128)), [PcgResult(0.0, 1, 0, x, 0.0)] * 128, 128)
    assert sum(f.stat().st_size for f in (tmp_path / "d").iterdir()) <= 64 << 20


def test_schedule_model_mirrors_the_kernel_constants():
    """The host-side model of the fused schedule in test_gpu_batch_scale.py (whose bite guards assert that its batches
    reach several table rounds) uses the tile-table size and tile height the library is built with."""
    from test_gpu_batch_scale import ROUND_TILES, TILE_ROWS

    csrc = ROOT / "deeppreconditioning_b200" / "csrc"
    defines = re.findall(r"^#define DPCG_ROUND_TILES (\d+)\s*$", (csrc / "pcg.cu").read_text(), re.M)
    assert defines == [str(ROUND_TILES)], defines
    assert not any("DPCG_ROUND_TILES" in flag for flag in build.NVCC_FLAGS), build.NVCC_FLAGS
    common = (csrc / "common.cuh").read_text()
    assert re.search(r"constexpr int kTileRows = kBlock;", common) and re.search(rf"constexpr int kBlock = {TILE_ROWS};", common)
