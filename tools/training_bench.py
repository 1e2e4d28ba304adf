"""One training step of the factor network: PyTorch module vs TrainableNet (dp_spconv_* forward and backward kernels).

    python tools/training_bench.py --out DIR [--reps N] [--quick]

A step is the forward, metrics.frobenius_loss and the backward into the parameters' .grad (no optimizer step).
Cases: PreconditionerNet on batches of 1 and 8 systems of 316^2 (bench.py's CNN_BATCH), PreconditionerTrilNet on one
128^3 system. Every case is warmed first, then timed with CUDA events over --reps steps (mean and min per step), and
torch.cuda.max_memory_allocated is read over one step of each path (reset before it). Prints one JSON line per case and
writes the whole result to DIR/training_bench.json together with the GPU's name and power limit.
"""
from __future__ import annotations

import argparse
import copy
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from deeppreconditioning_b200 import metrics, model as models, synthetic  # noqa: E402
from inference_bench import gpu_info, timed  # noqa: E402


def peak_bytes(fn) -> int:
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return int(torch.cuda.max_memory_allocated())


def case(name, net, st, reps) -> dict:
    g = torch.Generator().manual_seed(11)
    n = st.spatial_shape[0]
    x = torch.randn(st.batch_size, n, generator=g).to(st.features.device)
    b = torch.randn(st.batch_size, n, generator=g).to(st.features.device)
    mod, dev = net, copy.deepcopy(net)
    tdev = models.TrainableNet(dev)

    def step(model, params):
        def run():
            for p in params:
                p.grad = None
            loss = metrics.frobenius_loss(model(st), x, b)
            loss.backward()
            return loss
        return run

    mod_step, dev_step = step(mod, list(mod.parameters())), step(tdev, list(dev.parameters()))
    res = {"systems": st.batch_size, "sites_in": int(st.indices.shape[0])}
    res["module_step"] = timed(mod_step, reps)
    res["trainable_net_step"] = timed(dev_step, reps)
    res["module_peak_bytes"] = peak_bytes(mod_step)
    res["trainable_net_peak_bytes"] = peak_bytes(dev_step)
    res["speedup_step"] = res["module_step"]["ms_min"] / res["trainable_net_step"]["ms_min"]
    lm, ld = float(mod_step()), float(dev_step())
    res["loss_module"], res["loss_trainable_net"] = lm, ld
    num = sum(float(torch.linalg.vector_norm(pd.grad.double() - pm.grad.double()) ** 2)
              for pm, pd in zip(mod.parameters(), dev.parameters()))
    den = sum(float(torch.linalg.vector_norm(pm.grad.double()) ** 2) for pm in mod.parameters())
    res["grad_normwise_rel_diff"] = (num / den) ** 0.5
    print(name, json.dumps(res), flush=True)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for training_bench.json")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--quick", action="store_true", help="64^2 / 16^3 systems (a rehearsal)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("training_bench needs a CUDA device")
    device = torch.device("cuda", 0)
    side2, side3 = (64, 16) if args.quick else (316, 128)
    result = {"gpu": gpu_info(), "torch": torch.__version__, "reps": args.reps, "cases": {}}
    torch.manual_seed(69)  # bench.py make_net / test.py:205
    net = models.PreconditionerNet(models.DEFAULT_CHANNELS).to(device)
    for nb in (1, 8):
        st, _, _, _ = synthetic.make_batch("poisson2d", side2, list(range(nb)), device=device)
        result["cases"][f"net_{side2}sq_batch{nb}"] = case(f"net {side2}^2 x{nb}", net, st, args.reps)
        del st
        torch.cuda.empty_cache()
    torch.manual_seed(69)
    tril = models.PreconditionerTrilNet(models.DEFAULT_CHANNELS).to(device)
    st, _, _, _ = synthetic.make_batch("poisson3d", side3, [0], device=device)
    result["cases"][f"trilnet_{side3}cube"] = case(f"trilnet {side3}^3", tril, st, args.reps)
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "training_bench.json").write_text(json.dumps(result, indent=1))
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
