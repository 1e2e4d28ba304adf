#!/usr/bin/env python
"""Benchmark of the PCG hot path (BASELINE.json metric: PCG solves/sec + ms-to-tol per system; HBM roofline).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config c3|c5] [--dump-outputs DIR]

Workload c3 (default; BASELINE config 3, config.workload): the TEST SET of 1024 independent 316x316 5-point
variable-coefficient pressure systems (N = 99 856 unknowns each, the config-2 shape) with the factor L of a random-init
PreconditionerNet (multiply mode, the reference's `learned` technique), sharded over the N GPUs by interleaved index
(rank r holds systems r, r+N, ...: 1024/N per GPU, resident in HBM). A STEP is one fused-PCG solve (one kernel launch
per GPU) of the next 128 systems of the set (128/N per GPU) to rtol=1e-8 (squared criterion, cg.py:17), max_iter 20000
(the default 1024 saturates, SURVEY §0); eight steps are one pass over the set. The work of a step does not depend on N:
"scaling": "strong". (A whole-set step is 68 s on one GPU; the driver's 25 steps would not fit its time limit.)

Workload c5 (BASELINE config 5): 64 systems 256^3 (7-point, N = 16 777 216) on 8 GPUs = 8 per GPU, IC(0) in solve mode,
systems kept in the level order of the factor, tile-stream triangular solves. A step = one PCG solve of the GPU's 8
systems; "scaling": "weak" (8 per GPU at any N: 64 systems need the HBM of 8 GPUs).

config  : names the workload, identical in both arms; what a run found (iteration statistics, engine, matrix stream format,
          resident bytes, untimed set-up) is in `details`.
value   : solves/s with operands resident in HBM (CUDA events, max over ranks).
e2e     : the same through the reference-facing call with HOST operands (c3: pinned CSR of A and L, b - what
          preconditioned_conjugate_gradient receives from test.py:138; c5: the pinned COO lower triangle and b - what
          the data set yields): H2D copies, L^T assembly / analysis, workspace setup, solve, D2H of x/iterations inside
          the timed region.
roofline: the solve kernels, algorithmic bytes per launch (E nnzA + 2 E nnzL + 132 N + 12 per iteration and system,
          SURVEY §8d; E = bytes the kernel streams per stored entry: 6 from the lossless packed copies the fused engine
          uses when they exist - config 3 -, else 12) / CUDA-event duration, against the measured HBM copy bandwidth
          (MEASURED_PEAKS.json).
cpu_baseline / --impl reference: the CPU restatement of the reference loop (oracle/pcg.py, `as_is`: including the second
          `A @` of cg.py:87), torch CPU CSR operands built on the CPU by oracle/sparse.py (the process never loads
          libdpcg.so), all host threads, on a bounded sample of the same workload. The reference itself is Python and
          cannot travel to the GPU box; tests pin the restatement to it.

--dump-outputs DIR: after the timed steps, what the timed path returned in its last step, as DIR/<name>.npy (float64,
          see dump_outputs). The workload is generated from fixed seeds, so two builds run with the same arguments can be
          compared output for output.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "pcg_solves_per_sec"
UNIT = "solves/s"
RTOL = 1e-8
MAX_ITER = 20000


def parse_args():
    global MAX_ITER
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=["c3", "c5"])
    ap.add_argument("--systems-total", type=int, default=1024, help="c3: size of the test set (sharded over the GPUs)")
    ap.add_argument("--step-systems", type=int, default=128, help="c3: systems of the set solved per step (all GPUs together)")
    ap.add_argument("--c5-side", type=int, default=256)
    ap.add_argument("--c5-per-gpu", type=int, default=8)
    ap.add_argument("--side", type=int, default=316)
    ap.add_argument("--net", default="net", choices=["net", "tril"])
    ap.add_argument("--max-iter", type=int, default=MAX_ITER, help="profiling only: cap the bodies per solve")
    ap.add_argument("--no-extras", action="store_true", help="skip single-system latency and 128^3 kernel numbers")
    ap.add_argument("--dump-outputs", type=Path, metavar="DIR",
                    help="write what the timed path returned in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    MAX_ITER = args.max_iter
    world = max(1, args.gpus)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.systems_total % args.step_systems or args.step_systems % world:
        ap.error("--systems-total must be a multiple of --step-systems, and --step-systems of --gpus")
    return args


def workload_name(args):
    if args.config == "c5":
        world = max(1, args.gpus)
        return (f"{args.c5_per_gpu * world} x poisson3d {args.c5_side}^3 (N={args.c5_side ** 3}), {args.c5_per_gpu} per GPU, "
                f"IC(0) solve mode, level-ordered systems, tile-stream SpTRSV, rtol=1e-8 (squared), max_iter={MAX_ITER}")
    return (f"{args.systems_total} x poisson2d {args.side}x{args.side} (N={args.side ** 2}) test set sharded over the GPUs, "
            f"random-init Preconditioner{'Net' if args.net == 'net' else 'TrilNet'} L, multiply mode, "
            f"rtol=1e-8 (squared), max_iter={MAX_ITER}; step = next {args.step_systems} systems of the set")


def workload_config(args):
    """`config` of the JSON line: the same dictionary in both arms (the driver compares them). What a run found out about
    the workload (iteration counts, engine, resident bytes, set-up time) goes into `details`."""
    world = max(1, args.gpus)
    if args.config == "c5":
        return {"workload": workload_name(args), "systems_total": args.c5_per_gpu * world, "systems_per_gpu": args.c5_per_gpu,
                "l2": "5.2 GB per system-iteration >> 126 MB L2: no flush between timed steps"}
    return {"workload": workload_name(args), "systems_total": args.systems_total, "systems_per_step": args.step_systems,
            "l2": f"a step streams {args.step_systems // world} x 34-55 MB per GPU and iteration >> 126 MB L2: no flush between timed steps"}


def iter_bytes(n, nnz_a, nnz_l, entry_bytes=12):
    """Algorithmic bytes of one PCG iteration (SURVEY §8d): SpMV(A) + SpMV(L^T) + SpMV(L) + 72 N. `entry_bytes`: what the
    kernel streams per stored entry - 12 (fp64 value + int32 column) or 6 from the packed copies (fp32 + uint16)."""
    spmv = lambda nnz: entry_bytes * nnz + 4 * (n + 1) + 16 * n
    return spmv(nnz_a) + 2 * spmv(nnz_l) + 72 * n


def entry_bytes_of(batch):
    """6 when the fused engine streams the packed copies of this batch (every streamed matrix has one), else 12."""
    if os.environ.get("DPCG_NO_PACK", "0")[:1] == "1":
        return 12
    mats = [m for e in batch.entries for m in [e["A"], *e["M"].stream_matrices()]]
    return 6 if all(m._packed for m in mats) else 12


DUMP_X_BYTES = 48 << 20  # solutions and their positions; with the per-system arrays a dump stays under 64 MB


def dump_outputs(directory, systems, results, systems_in_step, rank=0, world=1):
    """--dump-outputs: the PcgResult of every system of the last timed step, as float64 arrays in `directory`:

    systems.npy      index of each system in the workload
    iterations.npy   PCG bodies run per system
    res.npy          final value of the stopping criterion (squared relative residual) per system
    x_hat.npy        solutions [system, position] at the positions of x_positions.npy (c5: in level order, the numbering
                     the solve runs in)
    x_positions.npy  every position when the solutions of a step fit DUMP_X_BYTES, else a sorted sample drawn by a
                     generator with a fixed seed: the same for every run, system and rank (written by rank 0)

    With several ranks, each rank writes its own systems as <name>.rank<r>.npy."""
    directory.mkdir(parents=True, exist_ok=True)
    n = results[0].x_hat.numel()
    assert all(r.x_hat.numel() == n for r in results), "the systems of a step have one size"
    k = min(n, DUMP_X_BYTES // (8 * (systems_in_step + 1)))
    pos = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    index = torch.from_numpy(pos)
    arrays = {"systems": systems, "iterations": [r.iterations for r in results], "res": [r.res for r in results],
              "x_hat": torch.stack([r.x_hat[index.to(r.x_hat.device)].cpu() for r in results]).numpy()}
    if rank == 0:
        arrays["x_positions"] = pos
    suffix = f".rank{rank}" if world > 1 else ""
    for name, value in arrays.items():
        np.save(directory / f"{name}{suffix}.npy", np.asarray(value, dtype=np.float64))


# ---- clocks ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])), smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---- workload -----------------------------------------------------------------------------------------------------------
CNN_BATCH = 8  # systems per CNN forward (the model is batched like data_set.py's loader; assembly picks one batch element)


def step_indices(args, step, rank, world):
    """Global indices of the systems this rank solves in step `step`: the step takes the next `step_systems` systems of
    the set (cyclically); rank r holds the systems with index % world == r (distributed.shard_indices)."""
    nchunks = args.systems_total // args.step_systems
    base = (step % nchunks) * args.step_systems
    return [i for i in range(base, base + args.step_systems) if i % world == rank]


def build_chunk(args, indices, net, device, keep_host):
    """Device operands (A, b, FactoredMultiply(L, L^T)) of the systems `indices`; with keep_host also their pinned HOST
    CSR copies for the e2e leg (what the reference's harness hands to cg.py after `.cpu()`, test.py:68,105)."""
    import deeppreconditioning_b200 as dp
    from deeppreconditioning_b200 import synthetic
    from deeppreconditioning_b200.sparse import CsrMatrix

    systems, host = [], []
    for at in range(0, len(indices), CNN_BATCH):
        group = indices[at:at + CNN_BATCH]
        st, _, rhs, sizes = synthetic.make_batch("poisson2d", args.side, group, device=device)
        with torch.no_grad():
            learned = net(st)
        for k, index in enumerate(group):
            n = sizes[k]
            A = CsrMatrix.from_spconv(st, n, "symmetrise", batch=k)
            L = CsrMatrix.from_spconv(learned, n, "tril", batch=k)
            Lt = CsrMatrix.from_spconv(learned, n, "tril_t", batch=k)
            b = rhs[k, :n].to(torch.float64)
            systems.append((A, b, dp.FactoredMultiply(L, Lt)))
            if keep_host:
                pin = lambda t: t.cpu().pin_memory()
                host.append(dict(index=index, n=n, a=tuple(pin(t) for t in (A.rowptr, A.col, A.val)),
                                 l=tuple(pin(t) for t in (L.rowptr, L.col, L.val)), b=pin(b)))
        del st, learned
    return systems, host


def make_net(args, device):
    from deeppreconditioning_b200 import model as models

    torch.manual_seed(69)  # test.py:205
    cls = models.PreconditionerNet if args.net == "net" else models.PreconditionerTrilNet
    return cls(models.DEFAULT_CHANNELS).to(device)


def dist_setup(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29531")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
        local = 0
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(value, world, device):
    if world == 1:
        return value
    import torch.distributed as dist

    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(value, world, device):
    if world == 1:
        return value
    import torch.distributed as dist

    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def cpu_operands(args, index, net, cnn_device):
    """One system of the c3 set as CPU operands, built WITHOUT libdpcg: the synthetic generator (numpy), the CNN forward
    in PyTorch (on the GPU when there is one, as the reference runs its model, test.py:102,217), and the CSR assembly of
    oracle/sparse.py (the literal test.py:65-68,103-105 arithmetic) on the CPU."""
    from deeppreconditioning_b200 import synthetic
    from oracle import operators
    from oracle import sparse as osp

    st, _, rhs, sizes = synthetic.make_batch("poisson2d", args.side, [index], device=cnn_device)
    n = sizes[0]
    with torch.no_grad():
        learned = net(st)
    ind, feat = st.indices.cpu().numpy(), st.features.cpu().numpy()
    a = osp.symmetrise_tril(ind, feat, 0, n)
    l = osp.tril_coo_to_csr(learned.indices.cpu().numpy(), learned.features.cpu().numpy(), 0, n)
    return osp.to_torch_csr(*a), operators.FactoredMultiply(*l), rhs[0, :n].cpu().to(torch.float64)


def cpu_solve(a, m, b, threads):
    """One system through the CPU restatement of the reference loop, executed as the reference executes it (as_is)."""
    from oracle import pcg

    torch.set_num_threads(threads)
    return pcg.preconditioned_conjugate_gradient(a, b.clone(), m, rtol=RTOL, max_iter=MAX_ITER, as_is=True)


def cpu_solve_sample(host_system, threads):
    """c3 cpu_baseline leg of the GPU arm: the rank's own host CSR operands through the same loop."""
    from oracle import operators
    from oracle import sparse as osp

    a = osp.to_torch_csr(*(t.numpy() for t in host_system["a"]))
    m = operators.FactoredMultiply(*(t.numpy() for t in host_system["l"]))
    return cpu_solve(a, m, host_system["b"], threads)


def peaks():
    path = ROOT / "MEASURED_PEAKS.json"
    if path.exists():
        return float(json.loads(path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---- reference arm ---------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's CPU implementation of the path on the box's host cores (rank 0 only): one system of the set per
    step, distinct systems. Nothing of libdpcg is loaded in this process."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    if args.config == "c5":
        return run_reference_c5(args, threads)
    cnn_device = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    net = make_net(args, cnn_device)
    times, iters = [], []
    for step in range(args.warmup + args.steps):
        index = (step * 41) % args.systems_total  # distinct systems spread over the set
        a, m, b = cpu_operands(args, index, net, cnn_device)
        t0 = time.perf_counter()
        r = cpu_solve(a, m, b, threads)
        dt = time.perf_counter() - t0
        if step >= args.warmup:
            times.append(dt), iters.append(r.iterations)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [index], [r], 1)
    total = float(np.sum(times))
    value = len(times) / total
    sample = (f"1 system of the {args.systems_total}-system set per step ({len(times)} timed, distinct systems), cg.py:70-88 "
              f"as is (second A@ of cg.py:87 included), torch CPU CSR operands built by oracle/sparse.py; "
              f"mean {np.mean(iters):.0f} iterations")
    assert not any("libdpcg" in line for line in open("/proc/self/maps")), "the reference arm must not load libdpcg.so"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def c5_iterations_hint():
    path = ROOT / "profiles" / "c5_iterations.json"
    return json.loads(path.read_text()) if path.exists() else {}


def run_reference_c5(args, threads):
    """c5 on the CPU: one 256^3 IC(0)-PCG solve is minutes of host time (two sequential triangular solves of 67 M entries
    per iteration), so a step is a bounded sample: the first `sample_iters` bodies of one system. solves/s is quoted
    for the iteration count the GPU arm needs on that system (profiles/c5_iterations.json)."""
    from deeppreconditioning_b200 import synthetic
    from oracle import ckernels, operators, pcg
    from oracle import sparse as osp

    ckernels.build()
    sample_iters = 3
    st, _, rhs, sizes = synthetic.make_batch("poisson3d", args.c5_side, [0])
    n = sizes[0]
    ind, feat = st.indices.numpy(), st.features.numpy()
    a = osp.to_torch_csr(*osp.symmetrise_tril(ind, feat, 0, n))
    t = osp.tril_coo_to_csr(ind, feat, 0, n)
    m = operators.FactoredSolve(t[0], t[1], ckernels.ic0(*t))
    b = rhs[0, :n].to(torch.float64)
    torch.set_num_threads(threads)
    times = []
    for step in range(args.warmup + args.steps):
        r = pcg.preconditioned_conjugate_gradient(a, b.clone(), m, rtol=RTOL, max_iter=sample_iters, as_is=True)
        if step >= args.warmup:
            times.append(r.seconds)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [0], [r], 1)
    per_iter = float(np.mean(times)) / sample_iters
    need = int(c5_iterations_hint().get(str(args.c5_side), 0)) or None
    value = 1.0 / (per_iter * need) if need else None
    sample = (f"{sample_iters} PCG bodies of one {args.c5_side}^3 system per step ({1e3 * per_iter:.0f} ms per iteration, oracle IC(0) "
              f"+ sequential C triangular solves); solves/s extrapolated to the {need} iterations the GPU arm needs")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "ms_per_iteration": 1e3 * per_iter},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---- our arm ------------------------------------------------------------------------------------------------------------
def extras(device, host0):
    """Single-system latency (BASELINE config 2) and HBM-bound kernel numbers on 128^3 (config 4)."""
    import deeppreconditioning_b200 as dp
    from deeppreconditioning_b200 import precond, synthetic
    from deeppreconditioning_b200.sparse import CsrMatrix

    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        best = float("inf")
        for _ in range(reps):
            a, b = ev(), ev()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b))
        return best

    # config 2: one 316^2 system, CNN L (multiply) vs IC(0) (solve) vs Jacobi
    A = CsrMatrix.from_arrays(*host0["a"], device=device)
    L = CsrMatrix.from_arrays(*host0["l"], device=device)
    b = host0["b"].to(device)
    n = A.n
    single = {}
    st, _, _, _ = synthetic.make_batch("poisson2d", int(round(n ** 0.5)), [host0["index"]], device=device)
    T = CsrMatrix.from_spconv(st, n, "tril")
    t0 = time.perf_counter()
    fwd = precond.analyse(T, False, level_stream=False)
    factor = precond.incomplete_cholesky0(T, fwd)
    ic = dp.FactoredSolve(factor, None, fwd)
    torch.cuda.synchronize()
    ic_setup_ms = 1e3 * (time.perf_counter() - t0)
    ic_sync_free = dp.FactoredSolve(factor, None, fwd, level_stream=False)
    for name, M in [("cnn_multiply", dp.FactoredMultiply(L)), ("ic0_solve", ic), ("ic0_solve_sync_free", ic_sync_free),
                    ("jacobi", dp.Jacobi(A)), ("identity", dp.Identity())]:
        batch = dp.PcgBatch([(A, b, M)], RTOL, MAX_ITER)

        def go():
            batch.reset()
            batch.solve()

        ms = timed(go)
        r = batch.results()[0]
        nnz_l = L.nnz if name == "cnn_multiply" else (T.nnz if name.startswith("ic0_solve") else 0)
        single[name] = {"ms_to_tol": ms, "iterations": r.iterations, "us_per_iteration": 1e3 * ms / max(r.iterations, 1),
                        "res": r.res, "bytes_per_matrix_entry": entry_bytes_of(batch),
                        "algorithmic_gbs": iter_bytes(n, A.nnz, nnz_l, entry_bytes_of(batch)) * r.iterations / ms / 1e6}
    single["ic0_solve"]["setup_ms_analysis_plus_factorisation"] = ic_setup_ms
    single["ic0_solve"]["levels"] = fwd.nlevels
    single["ic0_solve"]["triangular_solves"] = "level-stream (one CTA, dependencies polled in a shared-memory window)"
    single["ic0_solve_sync_free"]["triangular_solves"] = "sync-free (dependencies polled through L2)"
    out["single_system_316x316"] = single

    # the two triangular-solve kernels on the IC(0) factor of that system, alone and as a batch of independent solves
    fplan = precond.analyse(factor, False)
    r0, y0 = b.clone(), torch.empty_like(b)
    trsv_bytes2 = 12 * factor.nnz + 4 * (n + 1) + 16 * n
    trsv2 = {"levels": fplan.nlevels}
    # (the batch entry points are timed through PreparedTriangularBatch: descriptors uploaded once, solve() = kernel launches
    # only. Timed through the one-shot call a 128-system batch showed 0.63 ms where the kernel takes 0.27: the host staged
    # 128 descriptors between the two events)
    one_ls = precond.PreparedTriangularBatch([(factor, fplan, r0)], [y0], "ls")
    for key, fn in (("level_stream", one_ls.solve), ("sync_free", lambda: precond.triangular_solve(factor, fplan, r0, y0, algorithm="syncfree"))):
        ms = timed(fn, reps=5)
        trsv2[key] = {"ms": ms, "us_per_level": 1e3 * ms / fplan.nlevels, "algorithmic_gbs": trsv_bytes2 / ms / 1e6}
    import copy

    def clone_system():  # distinct memory per system: a shared factor would make every CTA hit the same L2 lines
        f = CsrMatrix(factor.rowptr.clone(), factor.col.clone(), factor.val.clone(), factor.n)
        p = copy.copy(fplan)
        p.perm = fplan.perm.clone()
        p.ls = copy.copy(fplan.ls)
        for field in ("rowptr", "col", "val", "level_sorted"):
            setattr(p.ls, field, getattr(fplan.ls, field).clone())
        p.ls.source = type(p.ls).key(f)
        return (f, p, r0.clone())

    nb2 = 128
    batch2 = [clone_system() for _ in range(nb2)]
    outs2 = [torch.empty_like(b) for _ in range(nb2)]
    ms = timed(precond.PreparedTriangularBatch(batch2, outs2, "ls").solve, reps=3)
    trsv2["level_stream_batch128"] = {"ms": ms, "algorithmic_gbs": nb2 * trsv_bytes2 / ms / 1e6,
                                      "frac_of_hbm_peak": nb2 * trsv_bytes2 / ms / 1e6 / peaks()[0],
                                      "note": "128 copies of the factor in distinct memory, one CTA per system, vectors in the "
                                              "original numbering (b gathered / x scattered through the level permutation)"}
    del batch2, outs2
    # the same factor of the system kept in LEVEL ORDER (precond.LevelOrdering: perm = identity, vectors coalesced)
    order = precond.level_ordering(T)
    st_lo = order.renumber(st)
    T_lo = CsrMatrix.from_spconv(st_lo, n, "tril")
    A_lo = CsrMatrix.from_spconv(st_lo, n, "symmetrise")
    b_lo = order.to_level(b)
    factor_lo = precond.incomplete_cholesky0(T_lo)
    fplan_lo = precond.analyse(factor_lo, False)
    y_lo = torch.empty_like(b_lo)
    ms = timed(precond.PreparedTriangularBatch([(factor_lo, fplan_lo, b_lo)], [y_lo], "ls").solve, reps=5)
    trsv2["level_stream_level_order"] = {"ms": ms, "us_per_level": 1e3 * ms / fplan_lo.nlevels, "algorithmic_gbs": trsv_bytes2 / ms / 1e6}

    def clone_lo():
        f = CsrMatrix(factor_lo.rowptr.clone(), factor_lo.col.clone(), factor_lo.val.clone(), factor_lo.n)
        p = copy.copy(fplan_lo)
        p.perm = fplan_lo.perm.clone()
        p.ls = copy.copy(fplan_lo.ls)
        for field in ("rowptr", "col", "val", "level_sorted"):
            setattr(p.ls, field, getattr(fplan_lo.ls, field).clone())
        p.ls.source = type(p.ls).key(f)
        return (f, p, b_lo.clone())

    batch_lo = [clone_lo() for _ in range(nb2)]
    outs_lo = [torch.empty_like(b_lo) for _ in range(nb2)]
    ms = timed(precond.PreparedTriangularBatch(batch_lo, outs_lo, "ls").solve, reps=3)
    trsv2["level_stream_batch128_level_order"] = {"ms": ms, "algorithmic_gbs": nb2 * trsv_bytes2 / ms / 1e6,
                                                  "frac_of_hbm_peak": nb2 * trsv_bytes2 / ms / 1e6 / peaks()[0],
                                                  "note": "same, systems renumbered by the factor's level sets: vectors coalesced"}
    del batch_lo, outs_lo
    out["sptrsv_316x316_ic0"] = trsv2
    # IC(0)-PCG on the level-ordered system (config 2's comparator in its fastest form)
    batch = dp.PcgBatch([(A_lo, b_lo, dp.FactoredSolve(factor_lo, None, fplan_lo))], RTOL, MAX_ITER)

    def go_lo():
        batch.reset()
        batch.solve()

    ms = timed(go_lo)
    r = batch.results()[0]
    single["ic0_solve_level_order"] = {"ms_to_tol": ms, "iterations": r.iterations, "us_per_iteration": 1e3 * ms / max(r.iterations, 1),
                                       "res": r.res, "algorithmic_gbs": iter_bytes(n, A.nnz, T.nnz) * r.iterations / ms / 1e6,
                                       "triangular_solves": "level-stream on the system renumbered by the factor's level sets"}
    del batch

    # the drop-in itself: BenchmarkSuite.run() (test.py:119-149) on 64 systems of the set, `learned` technique, one launch
    try:
        from deeppreconditioning_b200.test import BenchmarkSuite

        nsuite = 64
        data = synthetic.SyntheticPressureDataSet("poisson2d", int(round(n ** 0.5)), number_samples=nsuite, batch_size=1, device=device)
        suite = BenchmarkSuite(data, make_net(argparse.Namespace(net="net"), device), techniques=("learned",), rtol=RTOL,
                               max_iter=MAX_ITER, batch_systems=nsuite)
        t0 = time.perf_counter()
        suite.run()
        wall = time.perf_counter() - t0
        solve_s = float(sum(suite.durations["learned"]))
        out["benchmark_suite_learned_64"] = {
            "solves_per_s_solve_only": nsuite / solve_s, "solve_s": solve_s, "setup_s_mean_per_system": float(np.mean(suite.setups["learned"])),
            "wall_s_run": wall, "iterations_mean": float(np.mean(suite.iterations["learned"])),
            "note": "durations = the launch's time shared out by iteration count (cg.py:69-88 per system in the reference); set-up = CNN "
                    "forward in PyTorch + assembly of L and L^T per system (test.py:130-135); history and CG coefficients recorded"}
        del suite, data
        torch.cuda.empty_cache()
    except Exception as exc:  # an extra must never take the bench line down
        out["benchmark_suite_learned_64"] = {"skipped": repr(exc)[:200]}

    # config 4: 128^3, HBM-bound SpMV and SpTRSV
    st, _, rhs, sizes = synthetic.make_batch("poisson3d", 128, [0], device=device)
    n3 = sizes[0]
    A3, T3 = CsrMatrix.from_spconv(st, n3, "symmetrise"), CsrMatrix.from_spconv(st, n3, "tril")
    x = rhs[0, :n3].to(torch.float64)
    y = torch.empty_like(x)
    peak, _ = peaks()
    ms = timed(lambda: A3.matvec(x, y), reps=10)
    spmv_bytes = 12 * A3.nnz + 4 * (n3 + 1) + 16 * n3
    out["spmv_128^3"] = {"ms": ms, "algorithmic_gbs": spmv_bytes / ms / 1e6, "frac_of_hbm_peak": spmv_bytes / ms / 1e6 / peak}
    if A3.packed() is not None:  # the same product from the lossless 6-byte copy (same bits): half the matrix bytes
        ms = timed(lambda: A3.matvec(x, y, packed=True), reps=10)
        pbytes = 6 * A3.nnz + 4 * (n3 + 1) + 16 * n3
        out["spmv_128^3_packed"] = {"ms": ms, "algorithmic_gbs": pbytes / ms / 1e6, "frac_of_hbm_peak": pbytes / ms / 1e6 / peak,
                                    "speedup_vs_fp64_stream": out["spmv_128^3"]["ms"] / ms}
    fwd3 = precond.analyse(T3, False)
    ms = timed(lambda: precond.triangular_solve(T3, fwd3, x, y), reps=5)
    trsv_bytes = 12 * T3.nnz + 4 * (n3 + 1) + 16 * n3
    out["sptrsv_128^3"] = {"ms": ms, "levels": fwd3.nlevels, "algorithmic_gbs": trsv_bytes / ms / 1e6,
                           "frac_of_hbm_peak": trsv_bytes / ms / 1e6 / peak, "us_per_level": 1e3 * ms / fwd3.nlevels,
                           "bound": "levels x (store -> L2 -> poll) latency, not HBM: see profiles/README.md"}
    # config 5 operator size: SpMV on one 256^3 system (1.9 GB per product, far beyond the 126 MB L2)
    del y
    try:
        st5, _, rhs5, sizes5 = synthetic.make_batch("poisson3d", 256, [0], device=device)
        n5 = sizes5[0]
        A5 = CsrMatrix.from_spconv(st5, n5, "symmetrise")
        del st5
        x5 = rhs5[0, :n5].to(torch.float64)
        y5 = torch.empty_like(x5)
        ms = timed(lambda: A5.matvec(x5, y5), reps=5)
        bytes5 = 12 * A5.nnz + 4 * (n5 + 1) + 16 * n5
        out["spmv_256^3"] = {"ms": ms, "n": n5, "nnz": A5.nnz, "algorithmic_gbs": bytes5 / ms / 1e6,
                             "frac_of_hbm_peak": bytes5 / ms / 1e6 / peak}
        del A5, x5, y5, rhs5
        torch.cuda.empty_cache()
    except Exception as exc:  # an extra must never take the bench line down (host memory on small boxes)
        out["spmv_256^3"] = {"skipped": repr(exc)[:200]}

    # config 4 proper: single-system PCG on 128^3 (654 MB per iteration with a tril-pattern factor: HBM bound)
    from deeppreconditioning_b200 import model as models

    torch.manual_seed(69)
    with torch.no_grad():
        learned3 = models.PreconditionerTrilNet(models.DEFAULT_CHANNELS).to(device)(st)
    L3 = CsrMatrix.from_spconv(learned3, n3, "tril")
    del learned3
    b3 = rhs[0, :n3].to(torch.float64)
    ic3 = dp.FactoredSolve(precond.incomplete_cholesky0(T3, fwd3), None, fwd3)
    pcg3 = {}
    for name, M, nnz_l in [("jacobi", dp.Jacobi(A3), 0), ("cnn_tril_multiply", dp.FactoredMultiply(L3), L3.nnz),
                           ("ic0_solve", ic3, T3.nnz)]:
        batch3 = dp.PcgBatch([(A3, b3, M)], RTOL, MAX_ITER)

        def go3():
            batch3.reset()
            batch3.solve()

        ms = timed(go3, reps=2)
        r = batch3.results()[0]
        eb = entry_bytes_of(batch3)
        gbs = iter_bytes(n3, A3.nnz, nnz_l, eb) * r.iterations / ms / 1e6
        pcg3[name] = {"ms_to_tol": ms, "iterations": r.iterations, "us_per_iteration": 1e3 * ms / max(r.iterations, 1),
                      "res": r.res, "bytes_per_matrix_entry": eb, "algorithmic_gbs": gbs, "frac_of_hbm_peak": gbs / peak}
        del batch3
    pcg3["ic0_solve"]["triangular_solves"] = "sync-free (levels of up to 12 k rows: not level-stream material)"
    out["pcg_single_system_128^3"] = pcg3
    del L3, ic3
    # several independent solves in flight (the batch axis of configs 3/5): bytes grow, the critical path does not
    nb = 16
    import copy as _copy

    def clone3():  # distinct memory per system (a shared factor would be served from L2)
        m = CsrMatrix(T3.rowptr.clone(), T3.col.clone(), T3.val.clone(), T3.n)
        p = _copy.copy(fwd3)
        p.plan = fwd3.plan.clone()
        return (m, p, x.clone())

    batch3d = [clone3() for _ in range(nb)]
    outs = [torch.empty_like(x) for _ in range(nb)]
    ms = timed(lambda: precond.triangular_solve_batch(batch3d, outs, algorithm="syncfree"), reps=3)
    out["sptrsv_batch16_128^3"] = {"ms": ms, "systems": nb, "algorithmic_gbs": nb * trsv_bytes / ms / 1e6,
                                   "frac_of_hbm_peak": nb * trsv_bytes / ms / 1e6 / peak,
                                   "note": "16 copies of the factor in distinct memory, warps dealt to the systems"}
    del batch3d, outs
    # the same batch through the tile-stream solve (trsv_ts.cuh): level-ordered copies, TMA tile pipeline
    base3 = precond.level_ordered_any(T3, fwd3)

    def ts_batch(T, plan, base, rhs_vec, nb, position_space):
        systems, copies, outs = [], [], []
        for _ in range(nb):  # distinct memory per system
            c = _copy.copy(base)
            c.rowptr, c.col, c.val = base.rowptr.clone(), base.col.clone(), base.val.clone()
            p = _copy.copy(plan)
            p.perm = plan.perm.clone()
            rhs_s = rhs_vec[plan.perm.long()] if position_space else rhs_vec.clone()
            systems.append((T, p, rhs_s)), copies.append(c), outs.append(torch.empty_like(rhs_vec))
        prepared = precond.PreparedTriangularBatch(systems, outs, "ts", copies, position_space)
        ms = timed(prepared.solve, reps=3)
        prepared.check()
        return ms

    ts = {}
    for key, pos in [("original_numbering", False), ("level_order_vectors", True)]:
        ms = ts_batch(T3, fwd3, base3, x, nb, pos)
        ts[key] = {"ms": ms, "algorithmic_gbs": nb * trsv_bytes / ms / 1e6, "frac_of_hbm_peak": nb * trsv_bytes / ms / 1e6 / peak}
    out["sptrsv_batch16_128^3"]["tile_stream"] = ts
    del base3
    torch.cuda.empty_cache()
    # config 5, one GPU's share: 8 independent 256^3 factors (1.14 GB each), vectors in level order
    try:
        st5, _, rhs5, sizes5 = synthetic.make_batch("poisson3d", 256, [0], device=device)
        n5 = sizes5[0]
        T5 = CsrMatrix.from_spconv(st5, n5, "tril")
        del st5
        x5 = rhs5[0, :n5].to(torch.float64)
        del rhs5
        fwd5 = precond.analyse(T5, False, level_stream=False)
        base5 = precond.level_ordered_any(T5, fwd5)
        bytes5 = 12 * T5.nnz + 4 * (n5 + 1) + 16 * n5
        widths = torch.diff(fwd5.level_ptr)
        entry = {"n": n5, "nnz": T5.nnz, "levels": fwd5.nlevels, "widest_level_rows": int(widths.max())}
        for nb5 in (1, 8):
            ms = ts_batch(T5, fwd5, base5, x5, nb5, True)
            entry[f"{nb5}_systems"] = {"ms": ms, "algorithmic_gbs": nb5 * bytes5 / ms / 1e6,
                                       "frac_of_hbm_peak": nb5 * bytes5 / ms / 1e6 / peak}
        entry["note"] = ("tile-stream solve, vectors in level order, 8 distinct copies of the factor; the time includes arming "
                         "the solution vectors (8 B per row on top of the algorithmic bytes)")
        out["sptrsv_tile_stream_256^3"] = entry
        del T5, x5, fwd5, base5
        torch.cuda.empty_cache()
    except Exception as exc:  # an extra must never take the bench line down
        out["sptrsv_tile_stream_256^3"] = {"skipped": repr(exc)[:200]}
    # IC(0)-PCG on a batch of 8 x 128^3 (solve mode): natural order, level order, level order + tile-stream solves
    try:
        pcg8 = {}
        for key, level, tile_stream in [("natural_order", False, False), ("level_order", True, False),
                                        ("level_order_tile_stream", True, True)]:
            systems8 = []
            for i in range(8):
                st8, _, rhs8, sizes8 = synthetic.make_batch("poisson3d", 128, [i], device=device)
                n8 = sizes8[0]
                b8 = rhs8[0, :n8].to(torch.float64)
                T8 = CsrMatrix.from_spconv(st8, n8, "tril")
                if level:
                    order = precond.level_ordering(T8)
                    st8 = order.renumber(st8)
                    T8 = CsrMatrix.from_spconv(st8, n8, "tril")
                    b8 = order.to_level(b8)
                A8 = CsrMatrix.from_spconv(st8, n8, "symmetrise")
                plan8 = precond.analyse(T8, False, level_stream=False)
                F8 = precond.incomplete_cholesky0(T8, plan8)
                systems8.append((A8, b8, dp.FactoredSolve(F8, None, plan8, level_stream=False, tile_stream=tile_stream)))
            batch8 = dp.PcgBatch(systems8, RTOL, MAX_ITER)

            def go8():
                batch8.reset()
                batch8.solve()

            ms = timed(go8, reps=2)
            res8 = batch8.results()
            its = [r.iterations for r in res8]
            gbs = iter_bytes(n8, A8.nnz, T8.nnz) * sum(its) / ms / 1e6
            pcg8[key] = {"ms_to_tol": ms, "iterations": its, "us_per_iteration": 1e3 * ms / max(its),
                         "algorithmic_gbs": gbs, "frac_of_hbm_peak": gbs / peak}
            del batch8
            batch1 = dp.PcgBatch(systems8[:1], RTOL, MAX_ITER)  # config 4 in this form: one 128^3 system

            def go1():
                batch1.reset()
                batch1.solve()

            ms1 = timed(go1, reps=2)
            it1 = batch1.results()[0].iterations
            pcg8[key]["single_system"] = {"ms_to_tol": ms1, "iterations": it1, "us_per_iteration": 1e3 * ms1 / max(it1, 1)}
            del batch1, systems8
            torch.cuda.empty_cache()
        out["pcg_ic0_batch8_128^3"] = pcg8
    except Exception as exc:
        out["pcg_ic0_batch8_128^3"] = {"skipped": repr(exc)[:200]}
    return out


def run_ours(args):
    from deeppreconditioning_b200 import _lib
    from deeppreconditioning_b200 import build as dp_build

    rank, world, local = dist_setup(args)
    if not os.environ.get("DPCG_LIB") and dp_build.stale():
        # sources newer than the library in the tree: this process builds its own copy, outside the tree (which may be
        # read-only)
        tmp = Path(tempfile.mkdtemp(prefix="dpcg-"))
        atexit.register(shutil.rmtree, tmp, True)
        _lib.LIB_PATH = dp_build.build(force=True, out=tmp / "libdpcg.so")
    barrier(world)
    device = torch.device("cuda", local)
    if args.config == "c5":
        line = run_c5(args, rank, world, device)
    else:
        line = run_c3(args, rank, world, device)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


def run_c3(args, rank, world, device):
    """BASELINE config 3: the 1024-system test set, sharded; a step = one fused solve of the next 128 systems."""
    import deeppreconditioning_b200 as dp
    from deeppreconditioning_b200.distributed import gather_records, make_records
    from deeppreconditioning_b200.sparse import CsrMatrix

    local = device.index
    nsteps = args.warmup + args.steps
    nchunks = min(args.systems_total // args.step_systems, nsteps)  # chunks of the set the run touches
    net = make_net(args, device)
    t_setup = time.perf_counter()
    chunk_idx, batches, host = [], [], None
    for c in range(nchunks):
        mine = step_indices(args, c, rank, world)
        systems, h = build_chunk(args, mine, net, device, keep_host=(c == 0))
        if c == 0:
            host = h
        chunk_idx.append(mine)
        batches.append(dp.PcgBatch(systems, RTOL, MAX_ITER, engine="fused", device=device))
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup
    resident_gb = torch.cuda.memory_allocated(device) / 1e9

    # ---- resident-operand measurement -----------------------------------------------------------------------------
    for step in range(args.warmup):
        batch = batches[step % nchunks]
        batch.reset()
        batch.solve()
    barrier(world)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = []  # (chunk, start event, stop event) of every timed launch
    barrier(world)
    start.record()
    for step in range(args.warmup, nsteps):
        c = step % nchunks
        batches[c].reset()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        batches[c].solve()  # ONE kernel launch: pcg_fused_kernel
        k1.record()
        launches.append((c, k0, k1))
    stop.record()
    barrier(world)
    elapsed_ms = max_over_ranks(start.elapsed_time(stop), world, device)
    clocks = sampler.stop() if rank == 0 else None
    value = args.step_systems * args.steps / (elapsed_ms / 1e3)

    # results of every chunk that was solved (warm-up or timed): iteration statistics of the set
    solved = sorted({s % nchunks for s in range(nsteps)})
    results = {c: batches[c].results() for c in solved}
    if args.dump_outputs:
        last = (nsteps - 1) % nchunks
        dump_outputs(args.dump_outputs, chunk_idx[last], results[last], args.step_systems, rank, world)
    kernel_ms = [k0.elapsed_time(k1) for _, k0, k1 in launches]
    entry_bytes = {c: entry_bytes_of(batches[c]) for c in solved}
    chunk_bytes = {c: sum(iter_bytes(e["A"].n, e["A"].nnz, e["M"].L.nnz, entry_bytes[c]) * r.iterations
                          for e, r in zip(batches[c].entries, results[c])) for c in solved}
    packed_run = all(v == 6 for v in entry_bytes.values())
    bytes_per_sysit = float(np.mean([iter_bytes(e["A"].n, e["A"].nnz, e["M"].L.nnz, entry_bytes[c])
                                     for c in solved for e in batches[c].entries]))
    local_bytes = float(sum(chunk_bytes[c] for c, _, _ in launches))
    local_gbs = local_bytes / (sum(kernel_ms) / 1e3) / 1e9
    peak, peak_source = peaks()
    mean_gbs = sum_over_ranks(local_gbs, world, device) / world

    # per-system records: the only collective of the path (SURVEY §8e)
    idx = [i for c in solved for i in chunk_idx[c]]
    res = [r for c in solved for r in results[c]]
    ms_of = {c: [m for (cc, _, _), m in zip(launches, kernel_ms) if cc == c] for c in solved}
    ms = [float(np.mean(ms_of[c])) if ms_of[c] else 0.0 for c in solved for _ in chunk_idx[c]]
    # (the gather wants one record per index 0..n-1: chunks are contiguous index ranges starting at 0)
    records = gather_records(make_records(idx, res, ms), len(solved) * args.step_systems)
    iterations = records[:, 1].numpy()

    # ---- e2e: host operands through the public call ------------------------------------------------------------------
    h2d = sum(sum(t.numel() * t.element_size() for t in h["a"] + h["l"]) + h["b"].numel() * 8 for h in host)
    d2h = sum(h["n"] * 8 + 12 for h in host)

    def e2e_step():
        systems = []
        for h in host:
            A = CsrMatrix.from_arrays(*h["a"], device=device)
            L = CsrMatrix.from_arrays(*h["l"], device=device)
            systems.append((A, h["b"], dp.FactoredMultiply(L)))  # b stays a (pinned) host tensor: x_hat returns to host
        return dp.pcg_solve_batch(systems, RTOL, MAX_ITER, device=device)

    e2e_steps = max(1, min(args.steps, 3))
    e2e_step()
    barrier(world)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out = e2e_step()
    barrier(world)
    e2e_s = max_over_ranks(time.perf_counter() - t0, world, device)
    assert [r.iterations for r in out] == [r.iterations for r in results[0]], "e2e and resident runs disagree"
    e2e_value = args.step_systems * e2e_steps / e2e_s
    h2d_all, d2h_all = int(sum_over_ranks(h2d, world, device)), int(sum_over_ranks(d2h, world, device))

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only) -----------------------------------------------------------
    cpu = extra = None
    if rank == 0 and world == 1:
        threads = os.cpu_count() or 1
        nsample = min(3, len(host))  # bounded sample: ~10-15 s of CPU work
        t0 = time.perf_counter()
        cpu_runs = [cpu_solve_sample(host[i], threads) for i in range(nsample)]
        dt = time.perf_counter() - t0
        cpu_iters = [r.iterations for r in cpu_runs]
        cpu = {"value": nsample / dt, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"systems {[h['index'] for h in host[:nsample]]} of the set, one after the other, cg.py:70-88 as is "
                         f"(second A@ of cg.py:87 included): {cpu_iters} iterations in {dt:.2f} s "
                         f"(GPU, same operands: {[r.iterations for r in results[0][:nsample]]} iterations)",
               "ms_per_iteration": 1e3 * dt / max(sum(cpu_iters), 1)}
        if not args.no_extras:
            del batches[1:]
            torch.cuda.empty_cache()
            extra = extras(device, host[0])
    if rank != 0:
        return None
    # DRAM traffic of the fused kernel: ncu (--set full) measured dram__bytes_read+write on a short launch of the same
    # kernel and workload shape; profiles/traffic.json keeps it per system-iteration, scaled here to the mean launch.
    traffic, traffic_source = None, None
    tpath = ROOT / "profiles" / "traffic.json"
    if tpath.exists():
        tj = json.loads(tpath.read_text())
        per_iter = tj.get("pcg_fused_kernel_packed_dram_bytes_per_system_iteration" if packed_run
                          else "pcg_fused_kernel_dram_bytes_per_system_iteration")
        if per_iter:
            its = [sum(r.iterations for r in results[c]) for c, _, _ in launches]
            traffic = float(per_iter) * float(np.mean(its))
            traffic_source = tj.get("source_packed" if packed_run else "source", "profiles/traffic.json (ncu --set full capture of a short launch, scaled by iterations)")
    per_gpu = args.step_systems // world
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "details": {"systems_per_gpu_per_step": per_gpu, "systems_resident_per_gpu": nchunks * per_gpu,
                   "resident_gb_per_gpu": resident_gb,
                   "iterations_mean": float(iterations.mean()), "iterations_min": int(iterations.min()),
                   "iterations_max": int(iterations.max()), "systems_measured": int(len(iterations)),
                   "engine": "fused persistent cooperative kernel", "setup_s_untimed": setup_s,
                   "matrix_stream": ("packed copies (dp_csr_pack, lossless: fp32 value + uint16 tile-relative column = 6 B per "
                                     "entry, widened on load, same fp64 arithmetic and bits)" if packed_run
                                     else "fp64 value + int32 column = 12 B per entry"),
                   "bytes_per_system_iteration": bytes_per_sysit},
        "ms_to_tol_per_system": elapsed_ms / args.steps / per_gpu,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h_all, "steps": e2e_steps},
        "gpu_launches": args.steps * world,
        "roofline": {"bound": "hbm", "kernel": "pcg_fused_kernel", "achieved": mean_gbs, "peak": peak, "unit": "GB/s",
                     "frac": mean_gbs / peak, "traffic": traffic, "traffic_source": traffic_source, "peak_source": peak_source,
                     "bytes_per_launch": local_bytes / len(launches), "ms_per_launch": float(np.mean(kernel_ms))},
        "cpu_baseline": cpu,
    }
    if extra:
        line["extras"] = extra
    return line


def run_c5(args, rank, world, device):
    """BASELINE config 5: 8 systems 256^3 per GPU (64 on 8 GPUs), IC(0) solve mode on level-ordered systems with
    tile-stream triangular solves. A step = one PCG solve of the GPU's batch."""
    import deeppreconditioning_b200 as dp
    from deeppreconditioning_b200 import model as models
    from deeppreconditioning_b200 import precond, synthetic
    from deeppreconditioning_b200.sparse import CsrMatrix

    local = device.index
    side, per_gpu = args.c5_side, args.c5_per_gpu
    mine = [rank * per_gpu + i for i in range(per_gpu)]

    def prepare(st, rhs, n):
        """From the data set's item (COO lower triangle + rhs, on the device) to a batch entry: level ordering (K3),
        assembly of A and tril(A) in that order (K1), IC(0), L^T, level-ordered copies of both factors."""
        T = CsrMatrix.from_spconv(st, n, "tril")
        order = precond.level_ordering(T)
        del T
        st = order.renumber(st)
        T = CsrMatrix.from_spconv(st, n, "tril")
        A = CsrMatrix.from_spconv(st, n, "symmetrise")
        plan = precond.analyse(T, False, level_stream=False)
        F = precond.incomplete_cholesky0(T, plan)
        b = order.to_level(rhs[0, :n].to(device=device, dtype=torch.float64))
        return (A, b, dp.FactoredSolve(F, None, plan, level_stream=False, tile_stream=True)), order

    t_setup = time.perf_counter()
    systems, host = [], None
    for index in mine:
        st, _, rhs, sizes = synthetic.make_batch("poisson3d", side, [index])
        n = sizes[0]
        if host is None:  # the e2e leg runs on pinned host buffers of the rank's first system
            host = (st.features.pin_memory(), st.indices.pin_memory(), rhs.pin_memory(), n)
        dev_st = models.SparseConvTensor(st.features.to(device), st.indices.to(device), st.spatial_shape, 1)
        entry, _ = prepare(dev_st, rhs, n)
        systems.append(entry)
        del st, dev_st
    batch = dp.PcgBatch(systems, RTOL, MAX_ITER, device=device)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup
    resident_gb = torch.cuda.memory_allocated(device) / 1e9
    nnz_a, nnz_l = systems[0][0].nnz, systems[0][2].L.nnz

    for _ in range(args.warmup):
        batch.reset()
        batch.solve()
    barrier(world)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    start.record()
    for _ in range(args.steps):
        batch.reset()
        batch.solve()
    stop.record()
    barrier(world)
    elapsed_ms = max_over_ranks(start.elapsed_time(stop), world, device)
    local_ms = start.elapsed_time(stop)
    clocks = sampler.stop() if rank == 0 else None
    results = batch.results()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, mine, results, per_gpu * world, rank, world)
    its = [r.iterations for r in results]
    value = per_gpu * world * args.steps / (elapsed_ms / 1e3)
    local_bytes = float(sum(iter_bytes(n, nnz_a, nnz_l) * i for i in its))
    local_gbs = local_bytes * args.steps / (local_ms / 1e3) / 1e9
    peak, peak_source = peaks()
    mean_gbs = sum_over_ranks(local_gbs, world, device) / world
    all_its = sum_over_ranks(float(sum(its)), world, device)

    # e2e: one system from HOST COO (what the data set yields) through set-up and solve, solution back to the host
    feats, inds, rhs_h, n = host
    del batch, systems
    torch.cuda.empty_cache()

    def e2e_step():
        dev_st = models.SparseConvTensor(feats.to(device, non_blocking=True), inds.to(device, non_blocking=True), [n, n], 1)
        entry, order = prepare(dev_st, rhs_h.to(device, non_blocking=True), n)
        out = dp.pcg_solve_batch([entry], RTOL, MAX_ITER, device=device)[0]
        return order.from_level(out.x_hat).cpu(), out.iterations

    e2e_step()
    barrier(world)
    t0 = time.perf_counter()
    _, e2e_its = e2e_step()
    barrier(world)
    e2e_s = max_over_ranks(time.perf_counter() - t0, world, device)
    e2e_value = world / e2e_s
    h2d = feats.numel() * 4 + inds.numel() * 4 + n * 4
    if rank != 0:
        return None
    return {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "details": {"resident_gb_per_gpu": resident_gb,
                   "iterations": its, "iterations_mean_all_ranks": all_its / (per_gpu * world),
                   "engine": "stepped (tile-stream SpTRSV launches between the fused phases)", "setup_s_untimed": setup_s},
        "ms_to_tol_per_system": elapsed_ms / args.steps / per_gpu,
        "us_per_iteration": 1e3 * elapsed_ms / args.steps / max(its),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": (n * 8 + 12) * world,
                "steps": 1, "note": f"one system per GPU from the pinned host COO lower triangle: level analysis, assembly, IC(0), "
                                    f"solve ({e2e_its} iterations), x back in the original numbering"},
        "gpu_launches": int(args.steps * world * (5 * max(its) + 8)),
        "roofline": {"bound": "hbm", "kernel": "sptrsv_ts_batch_kernel + pcg_phase_kernel (whole iteration)", "achieved": mean_gbs,
                     "peak": peak, "unit": "GB/s", "frac": mean_gbs / peak, "traffic": None, "peak_source": peak_source,
                     "bytes_per_launch": local_bytes, "ms_per_launch": local_ms / args.steps,
                     "note": "launch = one whole solve of the batch (the stepped engine's kernels together)"},
        "cpu_baseline": None,
    }


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
