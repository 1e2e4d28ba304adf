"""FSAI against the learned factor on the bench's 316^2 systems: set-up cost and PCG iterations / solve time.

    python tools/fsai_bench.py [--reps N] [--systems 128] [--quick] [--out DIR]

Set-up, for 1 and 8 systems (bench.py's CNN_BATCH), every timing warmed first and taken with CUDA events over --reps
repetitions (mean and min per call):
  fsai_kernel_*       dp_fsai_f64 alone on the pattern of U = L^T made beforehand, per pattern (tril(A), learned L);
  fsai_*              precond.fsai(A, pattern): the transpose of the pattern, the kernel, the transpose of U, and the
                      packed copies of L and L^T (dp_csr_pack) that the fused PCG engine streams;
  learned             InferenceNet forward on the batch and the L / L^T assembly (CsrMatrix.from_spconv) of every system;
  power_pattern_k     precond.power_pattern(A, k) alone: the pattern of tril(|A|^k) by symbolic products, k = 2, 3, 4;
  fsai_power_k        power_pattern(A, k) and precond.fsai on it, with the packed copies of L and L^T.
FSAI has no batched entry point: 8 systems are 8 calls in a row (one system has ~10^5 independent rows).
Solve: one PcgBatch of --systems systems of the bench set (systems 0.., seeds of synthetic.poisson2d_tril), rtol 1e-8 on
the squared criterion, max_iter 20000, fused engine on the packed copies, per technique learned / fsai_learned / fsai /
fsai_power_2..4 / jacobi: iterations (mean, min, max) and the time of one solve (CUDA events, after one warm-up solve).
Prints one JSON line with the GPU's name and power limit read in the same run (and writes it to DIR/fsai_bench.json).
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import deeppreconditioning_b200 as dp  # noqa: E402
from deeppreconditioning_b200 import _lib, model as models, precond, synthetic  # noqa: E402
from deeppreconditioning_b200.sparse import CsrMatrix, pack_many  # noqa: E402
from inference_bench import gpu_info, timed  # noqa: E402

CNN_BATCH = 8
RTOL, MAX_ITER = 1e-8, 20000
POWERS = (2, 3, 4)


def make_systems(indices, side, inet, device):
    """(A, b, learned FactoredMultiply) of the bench set's systems `indices`, built as bench.py builds them."""
    out = []
    for at in range(0, len(indices), CNN_BATCH):
        group = indices[at:at + CNN_BATCH]
        st, _, rhs, sizes = synthetic.make_batch("poisson2d", side, group, device=device)
        with torch.no_grad():
            learned = inet(st)
        for k in range(len(group)):
            n = sizes[k]
            A = CsrMatrix.from_spconv(st, n, "symmetrise", batch=k)
            L = CsrMatrix.from_spconv(learned, n, "tril", batch=k)
            Lt = CsrMatrix.from_spconv(learned, n, "tril_t", batch=k)
            out.append((A, rhs[k, :n].to(torch.float64), dp.FactoredMultiply(L, Lt)))
        del st, learned
    return out


def setup_case(systems, inet, side, reps) -> dict:
    nsys = len(systems)
    device = systems[0][0].device
    lib = _lib.lib()
    patterns = {"tril": [A.tril() for A, _, _ in systems], "learned": [M.L for _, _, M in systems]}
    res = {"systems": nsys}
    for name, pats in patterns.items():
        uppers = [p.transpose() for p in pats]
        vals = [torch.empty(max(u.nnz, 1), dtype=torch.float64, device=device) for u in uppers]
        flag = torch.zeros(1, dtype=torch.int32, device=device)

        def kernel_only():
            for (A, _, _), u, v in zip(systems, uppers, vals):
                _lib.check(lib.dp_fsai_f64(A.n, _lib.ptr(A.rowptr), _lib.ptr(A.col), _lib.ptr(A.val), _lib.ptr(u.rowptr),
                                           _lib.ptr(u.col), 1, _lib.ptr(v), _lib.ptr(flag), _lib.stream_ptr(device)),
                           "dp_fsai_f64")

        def full():
            for p in pats:
                p._t = None  # CsrMatrix caches its transpose: time the pattern's transpose too
            ops = [precond.fsai(A, p) for (A, _, _), p in zip(systems, pats)]
            pack_many([m for op in ops for m in (op.L, op.Lt)])
            return ops

        res[f"fsai_kernel_{name}"] = timed(kernel_only, reps)
        _lib.raise_on_flag(flag, "dp_fsai_f64")
        res[f"fsai_{name}"] = timed(full, reps)
        res[f"nnz_per_row_{name}"] = sum(u.nnz for u in uppers) / sum(u.n for u in uppers)
        res[f"longest_column_{name}"] = max(int(torch.diff(u.rowptr).max()) for u in uppers)
    for k in POWERS:
        res[f"power_pattern_{k}"] = timed(lambda: [precond.power_pattern(A, k) for A, _, _ in systems], reps)

        def full_power():
            ops = [precond.fsai(A, precond.power_pattern(A, k)) for A, _, _ in systems]
            pack_many([m for op in ops for m in (op.L, op.Lt)])
            return ops

        res[f"fsai_power_{k}"] = timed(full_power, reps)
        uppers = [precond.power_pattern(A, k).transpose() for A, _, _ in systems]
        res[f"nnz_per_row_power_{k}"] = sum(u.nnz for u in uppers) / sum(u.n for u in uppers)
        res[f"longest_column_power_{k}"] = max(int(torch.diff(u.rowptr).max()) for u in uppers)
    st, _, _, sizes = synthetic.make_batch("poisson2d", side, list(range(nsys)), device=device)

    def learned():
        with torch.no_grad():
            out = inet(st)
        return [(CsrMatrix.from_spconv(out, sizes[k], "tril", batch=k), CsrMatrix.from_spconv(out, sizes[k], "tril_t", batch=k))
                for k in range(nsys)]

    res["learned"] = timed(learned, reps)
    return res


def solve_case(systems) -> dict:
    ops = {"learned": lambda A, M: M,
           "fsai_learned": lambda A, M: precond.fsai(A, M.L),
           "fsai": lambda A, M: precond.fsai(A),
           **{f"fsai_power_{k}": (lambda k: lambda A, M: precond.fsai(A, precond.power_pattern(A, k)))(k) for k in POWERS},
           "jacobi": lambda A, M: dp.Jacobi(A)}
    res = {}
    for name, make in ops.items():
        batch = dp.PcgBatch([(A, b, make(A, M)) for A, b, M in systems], RTOL, MAX_ITER)
        batch.solve()
        torch.cuda.synchronize()
        batch.reset()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        batch.solve()
        stop.record()
        stop.synchronize()
        results = batch.results()
        iters = np.array([r.iterations for r in results])
        res[name] = {"iterations_mean": float(iters.mean()), "iterations_min": int(iters.min()),
                     "iterations_max": int(iters.max()), "converged": int(sum(r.res < RTOL for r in results)),
                     "solve_ms": start.elapsed_time(stop),
                     "packed": all(m.packed() is not None for e in batch.entries for m in [e["A"], *e["M"].stream_matrices()])}
        del batch
        torch.cuda.empty_cache()
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--systems", type=int, default=128, help="systems of the PCG batch")
    ap.add_argument("--quick", action="store_true", help="64^2 systems (a rehearsal)")
    ap.add_argument("--out", help="directory for fsai_bench.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fsai_bench needs a CUDA device")
    device = torch.device("cuda", 0)
    side = 64 if args.quick else 316
    torch.manual_seed(69)  # bench.py make_net / test.py:205
    inet = models.InferenceNet(models.PreconditionerNet(models.DEFAULT_CHANNELS).to(device))
    systems = make_systems(list(range(args.systems)), side, inet, device)
    result = {"gpu": gpu_info(), "torch": torch.__version__, "side": side, "reps": args.reps,
              "setup": {f"batch{nb}": setup_case(systems[:nb], inet, side, args.reps) for nb in (1, CNN_BATCH)},
              "solve": {"systems": args.systems, **solve_case(systems)}}
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).mkdir(parents=True, exist_ok=True)
        (Path(args.out) / "fsai_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
