"""The training loss with torch.use_deterministic_algorithms off (dp_coo_spmv_batch_f32, fp32 atomics) and on (sorted
sites: dp_spconv_sort_sites twice, dp_llt_residual_f32 and its gradient).

    python tools/loss_bench.py --out DIR [--reps N] [--quick]

Cases: metrics.frobenius_loss on PreconditionerNet's L for 1 and 8 systems of 316^2 (bench.py's CNN_BATCH), forward
alone (under no_grad) and forward plus backward into L's features; and one TrainableNet step (forward, frobenius_loss,
backward into the parameters' .grad, as tools/training_bench.py times it) on the same batches. Every timing is warmed
first, then taken with CUDA events over --reps calls (mean and min per call). The deterministic timings include what the
flag costs elsewhere: torch fills torch.empty outputs with NaN while torch.utils.deterministic.fill_uninitialized_memory
is set, and the JSON records that setting. Writes DIR/loss_bench.json with the GPU's name and power limit.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from deeppreconditioning_b200 import metrics, model as models, synthetic  # noqa: E402
from inference_bench import gpu_info, timed  # noqa: E402

PATHS = {"atomic": False, "deterministic": True}


@contextlib.contextmanager
def deterministic(enabled: bool):
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(enabled)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def case(name, net, st, reps) -> dict:
    g = torch.Generator().manual_seed(11)
    n = st.spatial_shape[0]
    x = torch.randn(st.batch_size, n, generator=g).to(st.features.device)
    b = torch.randn(st.batch_size, n, generator=g).to(st.features.device)
    tnet = models.TrainableNet(net)
    with torch.no_grad():
        lower = tnet(st)
    feats = lower.features.detach().clone().requires_grad_(True)
    params = list(net.parameters())

    def loss_forward():
        with torch.no_grad():
            return metrics.frobenius_loss(lower, x, b)

    def loss_backward():
        feats.grad = None
        loss = metrics.frobenius_loss(lower.replace_feature(feats), x, b)
        loss.backward()
        return loss

    def step():
        for p in params:
            p.grad = None
        loss = metrics.frobenius_loss(tnet(st), x, b)
        loss.backward()
        return loss

    res = {"systems": st.batch_size, "n": n, "factor_sites": int(lower.indices.shape[0])}
    for path, flag in PATHS.items():
        with deterministic(flag):
            res[f"{path}_loss_forward"] = timed(loss_forward, reps)
            res[f"{path}_loss_forward_backward"] = timed(loss_backward, reps)
            res[f"{path}_trainable_net_step"] = timed(step, reps)
            res[f"{path}_loss_value"] = float(loss_forward())
    res["loss_rel_diff"] = abs(res["deterministic_loss_value"] - res["atomic_loss_value"]) / abs(res["atomic_loss_value"])
    for what in ("loss_forward", "loss_forward_backward", "trainable_net_step"):
        res[f"{what}_deterministic_over_atomic"] = res[f"deterministic_{what}"]["ms_min"] / res[f"atomic_{what}"]["ms_min"]
    print(name, json.dumps(res), flush=True)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for loss_bench.json")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="64^2 systems (a rehearsal)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("loss_bench needs a CUDA device")
    device = torch.device("cuda", 0)
    side = 64 if args.quick else 316
    result = {"gpu": gpu_info(), "torch": torch.__version__, "reps": args.reps,
              "fill_uninitialized_memory": bool(torch.utils.deterministic.fill_uninitialized_memory), "cases": {}}
    torch.manual_seed(69)  # bench.py make_net / test.py:205
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS).to(device)
    for nb in (1, 8):
        st, _, _, _ = synthetic.make_batch("poisson2d", side, list(range(nb)), device=device)
        result["cases"][f"net_{side}sq_batch{nb}"] = case(f"net {side}^2 x{nb}", net, st, args.reps)
        del st
        torch.cuda.empty_cache()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "loss_bench.json").write_text(json.dumps(result, indent=1))
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
