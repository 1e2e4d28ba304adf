"""The factor network's forward: PyTorch module vs InferenceNet (dp_spconv_* kernels), alone and with the L / L^T assembly.

    python tools/inference_bench.py --out DIR [--reps N] [--quick]

Cases: PreconditionerNet on batches of 1 and 8 systems of 316^2 (bench.py's CNN_BATCH), PreconditionerTrilNet on one
128^3 system. Every shape is warmed first, then timed with CUDA events over --reps repetitions (mean and min per call).
Rates: GFLOP/s from the exact (site, tap) pair counts of every layer (2 pairs cin cout), feature bytes/s from the
features each layer reads per pair and writes per output site. Then BenchmarkSuite on 64 systems of 316^2, learned
technique only, with each model: the mean of `setups` (the same measurement as bench.py's benchmark_suite_learned_64).
Prints the JSON and writes it to DIR/inference_bench.json together with the GPU's name and power limit.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from deeppreconditioning_b200 import model as models, spconv, synthetic  # noqa: E402
from deeppreconditioning_b200.sparse import CsrMatrix  # noqa: E402


def gpu_info() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as exc:  # the numbers stay labelled with the device name
        info["power_limit_and_max_sm_clock"] = f"unavailable: {exc!r}"[:120]
    return info


def timed(fn, reps: int) -> dict:
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        fn()
        stop.record()
        stop.synchronize()
        times.append(start.elapsed_time(stop))
    return {"ms_mean": float(np.mean(times)), "ms_min": float(np.min(times)), "reps": reps}


def work_counts(inet, st) -> dict:
    """Exact (site, tap) pairs, FLOP and feature bytes of the forward on `st`."""
    batch, (h, w) = st.batch_size, st.spatial_shape
    nsites = int(st.indices.shape[0])
    rowptr = col = perm = None
    if any(c.k == 2 for c, _ in inet.steps):
        rowptr, col, perm = spconv.sort_sites(st.indices, batch, h, w)
    flop = byts = 0
    layers = []
    for conv, _ in inet.steps:
        cout, _, _, cin = conv.weight.shape
        if conv.k == 2:
            rowptr, col, rules, _ = spconv.conv_rules(rowptr, col, batch, h, w, conv.padding, perm)
            perm = None
            pairs, nout = int((rules >= 0).sum()), int(rules.shape[0])
            h, w = h + 2 * conv.padding[0] - 1, w + 2 * conv.padding[1] - 1
        else:
            pairs = nout = nsites
        nsites = nout
        layers.append({"k": conv.k, "cin": cin, "cout": cout, "sites_out": nout, "pairs": pairs})
        flop += 2 * pairs * cin * cout
        byts += 4 * (pairs * cin + nout * cout)
    return {"layers": layers, "gflop": flop / 1e9, "feature_gb": byts / 1e9}


def assembly(out, sizes):
    for k, n in enumerate(sizes):
        CsrMatrix.from_spconv(out, n, "tril", batch=k)
        CsrMatrix.from_spconv(out, n, "tril_t", batch=k)


def case(name, net, st, sizes, reps) -> dict:
    inet = models.InferenceNet(net)
    counts = work_counts(inet, st)

    def torch_fwd():
        with torch.no_grad():
            return net(st)

    def torch_setup():
        assembly(torch_fwd(), sizes)

    def dev_setup():
        assembly(inet(st), sizes)

    res = {"systems": len(sizes), "sites_in": int(st.indices.shape[0]), **counts}
    res["pytorch_forward"] = timed(torch_fwd, reps)
    res["inference_net"] = timed(lambda: inet(st), reps)
    res["pytorch_forward_plus_assembly"] = timed(torch_setup, reps)
    res["inference_net_plus_assembly"] = timed(dev_setup, reps)
    for key in ("pytorch_forward", "inference_net"):
        ms = res[key]["ms_min"]
        res[key]["gflops"] = counts["gflop"] / ms * 1e3
        res[key]["feature_gbs"] = counts["feature_gb"] / ms * 1e3
    res["speedup_forward"] = res["pytorch_forward"]["ms_min"] / res["inference_net"]["ms_min"]
    res["speedup_setup"] = res["pytorch_forward_plus_assembly"]["ms_min"] / res["inference_net_plus_assembly"]["ms_min"]
    res["assembly_share_of_pytorch_setup"] = 1 - res["pytorch_forward"]["ms_min"] / res["pytorch_forward_plus_assembly"]["ms_min"]
    want, got = torch_fwd(), inet(st)
    assert torch.equal(want.indices, got.indices)
    d = (got.features.double() - want.features.double())
    ref = want.features.double()
    res["normwise_rel_diff"] = float(torch.linalg.vector_norm(d) / torch.linalg.vector_norm(ref))
    res["max_abs_diff_over_max_abs"] = float(d.abs().max() / ref.abs().max())
    print(name, json.dumps({k: v for k, v in res.items() if k != "layers"}), flush=True)
    return res


def suite_setups(net, device, nsys) -> dict:
    from deeppreconditioning_b200.test import BenchmarkSuite

    data = synthetic.SyntheticPressureDataSet("poisson2d", 316, number_samples=nsys, batch_size=1, device=device)
    out = {}
    for label, model in (("pytorch", net), ("inference_net", models.InferenceNet(net))):
        suite = BenchmarkSuite(data, model, techniques=("learned",), rtol=1e-8, max_iter=20000, batch_systems=nsys)
        suite.run()
        out[label] = {"setup_s_mean_per_system": float(np.mean(suite.setups["learned"])),
                      "solve_s": float(sum(suite.durations["learned"])),
                      "iterations_mean": float(np.mean(suite.iterations["learned"])),
                      "densities_mean": float(np.mean(suite.densities["learned"]))}
        print("suite", label, json.dumps(out[label]), flush=True)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for inference_bench.json")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--quick", action="store_true", help="64^2 / 16^3 systems and 4 suite systems (a rehearsal)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("inference_bench needs a CUDA device")
    device = torch.device("cuda", 0)
    side2, side3, nsuite = (64, 16, 4) if args.quick else (316, 128, 64)
    result = {"gpu": gpu_info(), "torch": torch.__version__, "reps": args.reps, "cases": {}}
    torch.manual_seed(69)  # bench.py make_net / test.py:205
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS).to(device)
    for nb in (1, 8):
        st, _, _, sizes = synthetic.make_batch("poisson2d", side2, list(range(nb)), device=device)
        result["cases"][f"net_{side2}sq_batch{nb}"] = case(f"net {side2}^2 x{nb}", net, st, sizes, args.reps)
        del st
        torch.cuda.empty_cache()
    torch.manual_seed(69)
    tril = models.PreconditionerTrilNet(models.DEFAULT_CHANNELS).to(device)
    st, _, _, sizes = synthetic.make_batch("poisson3d", side3, [0], device=device)
    result["cases"][f"trilnet_{side3}cube"] = case(f"trilnet {side3}^3", tril, st, sizes, args.reps)
    del st
    torch.cuda.empty_cache()
    result["benchmark_suite_learned"] = {"systems": nsuite, **suite_setups(net, device, nsuite)}
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "inference_bench.json").write_text(json.dumps(result, indent=1))
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
