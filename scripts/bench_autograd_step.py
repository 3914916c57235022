"""One training step through autograd vs ``training_step``, at 64 pairs on one GPU, in fp32 and tf32.

    python scripts/bench_autograd_step.py [--pairs 64] [--steps 10] [--warmup 3] [--rounds 5] [--out FILE]

autograd: ``predict5(training=True)`` with ``model.differentiable = True``, the reference's loss (model5_b.py:912-1155,
loss_mode 1) assembled from the drop-in operators (se3.exp, se3.transform, chamfer_loss, comp, earth_mover_distance,
F.cross_entropy, boundary_topk + index_points), ``loss.backward()`` and ``torch.optim.Adam``.
training_step: ``Trainer.training_step`` (the same forward and backward kernels, its own loss kernels and fused Adam).

Synthetic batch and weights as scripts/bench_train.py.  Each path runs on its own model.  Per round every path times
``--steps`` steps (host clock around work that ends in a device synchronise); the paths alternate within a round, so
drift on the shared machine hits both.  One JSON line per precision: median and spread (max - min) over rounds of
the ms per step, the overhead of autograd in percent of training_step, the GPU's name and power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import types

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from scripts.bench_train import make_training_batch  # noqa: E402


def reference_loss(model, batch):
    from puzzlenet_b200 import losses, se3
    from puzzlenet_b200 import pointnet_util as pu
    from puzzlenet_b200.emd import earth_mover_distance
    fpc, mrpc, igt, rpc, fpcb, rpcb, fpc_idx, rpc_idx = batch
    out, _, de_fpcb, de_mrpcb = model.predict5(batch, fpc.shape[0], training=True)
    mat = se3.exp(out)
    de_mrpc = se3.transform(mat, mrpc.permute(0, 2, 1)).permute(0, 2, 1)
    d1, d2 = model.chamfer_loss(rpc, de_mrpc)
    loss = d1.mean() + d2.mean() + model.comp(mat, igt) + earth_mover_distance(de_mrpc, rpc, transpose=False).mean()
    loss = loss + F.cross_entropy(de_fpcb, fpc_idx.long()) + F.cross_entropy(de_mrpcb, rpc_idx.long())
    bnd_f = pu.index_points(fpc, losses.boundary_topk(de_fpcb))
    bnd_m = pu.index_points(mrpc, losses.boundary_topk(de_mrpcb))
    c1, c2 = model.chamfer_loss(bnd_f, fpcb)
    c3, c4 = model.chamfer_loss(se3.transform(mat, bnd_m.permute(0, 2, 1)).permute(0, 2, 1), rpcb)
    return loss + c3.mean() + c4.mean() + c1.mean() + c2.mean()


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--lr", type=float, default=1e-5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_autograd_step.py needs a GPU"
    dev = torch.device("cuda", 0)
    from puzzlenet_b200.model5_b import TouchedRegraster
    from puzzlenet_b200.training import Trainer
    from puzzlenet_b200.weights import synthetic_state_dict
    batch = make_training_batch(a.pairs, 64, dev)
    info = gpu_info()
    lines = []
    for prec in ("fp32", "tf32"):
        models = {}
        for path in ("autograd", "training_step"):
            m = TouchedRegraster(types.SimpleNamespace(dataset="vase", loss_mode=1, loss_sum=False, lr=a.lr))
            m.load_state_dict(synthetic_state_dict(0))
            m.to(dev)
            m._trainer_state = Trainer(m, m.C, precision=prec)
            models[path] = m
        ma, mt = models["autograd"], models["training_step"]
        ma.differentiable = True
        opt = torch.optim.Adam(ma.parameters(), lr=a.lr)

        def autograd_step():
            opt.zero_grad()
            reference_loss(ma, batch).backward()
            opt.step()

        def trainer_step():
            mt.trainer_state().training_step(batch)

        steps = dict(autograd=autograd_step, training_step=trainer_step)
        for fn in steps.values():
            for _ in range(a.warmup):
                fn()
        times = {k: [] for k in steps}
        for _ in range(a.rounds):
            for k, fn in steps.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(a.steps):
                    fn()
                torch.cuda.synchronize()
                times[k].append((time.perf_counter() - t0) * 1e3 / a.steps)
        med = {k: statistics.median(v) for k, v in times.items()}
        line = {"metric": "ms per training step, autograd vs training_step", "precision": prec, "pairs": a.pairs,
                "steps": a.steps, "rounds": a.rounds,
                "autograd_ms": round(med["autograd"], 3),
                "autograd_spread_ms": round(max(times["autograd"]) - min(times["autograd"]), 3),
                "training_step_ms": round(med["training_step"], 3),
                "training_step_spread_ms": round(max(times["training_step"]) - min(times["training_step"]), 3),
                "overhead_pct": round(100.0 * (med["autograd"] / med["training_step"] - 1.0), 2),
                "gpu": info}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
