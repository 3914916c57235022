"""BASELINE config 5: multi-piece greedy assembly -- all-pairs matching of 32 DublinCity-like 11000-point pieces
(496 candidate pairs) sharded over the GPUs of one box.

    python scripts/bench_assembly.py [--pieces 32] [--points 11000] [--iters 10] [--scorer predict5|embedding]
    python scripts/bench_assembly.py --alternate [--rescore]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        scripts/bench_assembly.py

Pieces are synthetic (SURVEY.md §8d C5: the union of 3-6 random planar rectangles per piece, seed 5+piece); weights
are synthetic_state_dict(0).  One JSON line from rank 0: time per full assembly (FPS down-sampling of the pieces,
pair scoring, the all_gather of [n_pairs, 8] rows, host-side greedy merge).  Pair scoring is ``--scorer predict5``
(ModelScorer: one predict5 + pz_pair_score per 64 pairs) or ``--scorer embedding`` (EmbeddingScorer: every piece
encoded once, then the pair heads per pair; a fresh scorer per assembly, so its encoding is timed too).

``--alternate`` times single assemblies of both scorers in turn (the order swapped every iteration) in one process and
reports, per scorer, the median and the spread of the per-assembly times, their ratio, the largest difference between
the two scorers' rows when predict5 is given each pair's per-piece FPS starts, and the GPU's name and power limit."""
import argparse
import json
import os
import sys
import time
import types

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def dublin_like_piece(seed: int, n: int) -> np.ndarray:
    rng = np.random.default_rng(5 + seed)
    k = int(rng.integers(3, 7))
    per = np.full(k, n // k)
    per[: n - per.sum()] += 1
    parts = []
    for c in per:
        origin = rng.uniform(-0.4, 0.4, 3)
        u = rng.normal(size=3); u /= np.linalg.norm(u)
        v = rng.normal(size=3); v -= u * (u @ v); v /= np.linalg.norm(v)
        ext = rng.uniform(0.2, 0.6, 2)
        ab = rng.uniform(0, 1, (c, 2)) * ext
        parts.append(origin + ab[:, :1] * u + ab[:, 1:] * v + rng.normal(0, 0.002, (c, 3)))
    pts = np.concatenate(parts).astype(np.float32)
    pts -= pts.mean(0)
    return pts / np.abs(pts).max() * 0.5


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pieces", type=int, default=32)
    ap.add_argument("--points", type=int, default=11000)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--rescore", action="store_true")
    ap.add_argument("--scorer", choices=("predict5", "embedding"), default="predict5")
    ap.add_argument("--alternate", action="store_true", help="time both scorers alternately (ignores --scorer)")
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from puzzlenet_b200 import assembly
    from puzzlenet_b200.model5_b import TouchedRegraster
    from puzzlenet_b200.weights import synthetic_state_dict
    model = TouchedRegraster(types.SimpleNamespace(dataset="vase"))
    model.load_state_dict(synthetic_state_dict(0))
    model.to(dev).eval()
    model.precision = a.precision
    pieces = [dublin_like_piece(i, a.points) for i in range(a.pieces)]
    starts = [int(np.random.default_rng(100 + i).integers(0, a.points)) for i in range(a.pieces)]
    n_pairs = a.pieces * (a.pieces - 1) // 2

    def make_scorer(kind):
        return assembly.ModelScorer(model) if kind == "predict5" else assembly.EmbeddingScorer(model)

    def once(kind=a.scorer):
        scorer = make_scorer(kind)
        torch.manual_seed(1234)
        clouds = assembly.downsample_pieces(pieces, 1024, starts=starts, device=dev)
        if a.rescore:
            return assembly.assemble(clouds, scorer, batch=64, rescore=True)
        pairs, rows = assembly.score_all_pairs(clouds, scorer, batch=64)
        return assembly.greedy_assemble(a.pieces, pairs, rows)[::2]

    if a.alternate:
        alternate(a, once, model, pieces, starts, dev, world, rank, n_pairs)
        if world > 1:
            dist.destroy_process_group()
        return
    for _ in range(a.warmup):
        once()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(a.iters):
        poses, merges = once()
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    if rank == 0:
        ms = dt.item() / a.iters * 1e3
        print(json.dumps({"metric": "assemblies/sec (config 5)", "pieces": a.pieces, "points_per_piece": a.points,
                          "pairs": n_pairs, "n_gpus": world, "ms_per_assembly": ms,
                          "pairs_per_s": n_pairs / ms * 1e3, "merges": len(merges), "precision": a.precision,
                          "rescore": a.rescore, "scorer": a.scorer, "timing": "host wall clock around whole assemblies (includes "
                          "H2D of the raw pieces, the NCCL all_gathers and the host-side greedy merge), max over ranks"}))
    if world > 1:
        dist.destroy_process_group()


def gpu_info():
    """(name, power limit in W or None) of the current GPU; read-only nvidia-smi query."""
    import subprocess
    idx = torch.cuda.current_device()
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        limit = float(out)
    except (OSError, ValueError, subprocess.SubprocessError):
        limit = None
    return torch.cuda.get_device_name(idx), limit


def rows_max_diff(model, pieces, starts, dev):
    """max |rows(EmbeddingScorer) - rows(predict5 with each pair's per-piece FPS starts)| over all pairs."""
    from puzzlenet_b200 import assembly, losses
    from puzzlenet_b200.weights import make_batch
    torch.manual_seed(1234)
    clouds = assembly.downsample_pieces(pieces, 1024, starts=starts, device=dev)
    emb_scorer = assembly.EmbeddingScorer(model)
    pairs, rows = assembly.score_all_pairs(clouds, emb_scorer, batch=64)
    st = emb_scorer.emb.starts
    diff = 0.0
    for lo in range(0, pairs.shape[0], 64):
        sel = pairs[lo:lo + 64]
        I, J = sel[:, 0], sel[:, 1]
        s4 = torch.stack([st[0, I], st[1, I], st[2, J], st[3, J]]).contiguous()
        fpc, mrpc = clouds[I.to(dev)], clouds[J.to(dev)]
        out6, _, de_f, de_m = model.predict5(make_batch(fpc, mrpc), sel.shape[0], starts=s4)
        s = losses.pair_score(out6, de_f, de_m, fpc, mrpc)
        ref = torch.cat([out6, s[:, 10:11], torch.ones(sel.shape[0], 1, device=dev)], dim=1)
        diff = max(diff, (rows[lo:lo + 64] - ref).abs().max().item())
    return diff


def alternate(a, once, model, pieces, starts, dev, world, rank, n_pairs):
    kinds = ("predict5", "embedding")

    def timed(kind):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        once(kind)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return dt.item() * 1e3

    for _ in range(a.warmup):
        for k in kinds:
            timed(k)
    ms = {k: [] for k in kinds}
    for it in range(a.iters):
        for k in (kinds if it % 2 == 0 else kinds[::-1]):
            ms[k].append(timed(k))
    diff = rows_max_diff(model, pieces, starts, dev)
    name, limit = gpu_info()
    if rank == 0:
        res = {}
        for k in kinds:
            v = np.asarray(ms[k])
            res[k] = {"ms_per_assembly_median": float(np.median(v)), "ms_min": float(v.min()), "ms_max": float(v.max()),
                      "spread_pct": float((v.max() - v.min()) / np.median(v) * 100), "ms_all": [round(x, 3) for x in v]}
        print(json.dumps({"metric": "assembly ms, predict5 vs embedding scorer (config 5)", "pieces": a.pieces,
                          "points_per_piece": a.points, "pairs": n_pairs, "n_gpus": world, "precision": a.precision,
                          "rescore": a.rescore, "iters": a.iters, "warmup": a.warmup, "scorer": "alternate", **res,
                          "speedup_median": res["predict5"]["ms_per_assembly_median"]
                          / res["embedding"]["ms_per_assembly_median"],
                          "rows_max_abs_diff_matched_starts": diff, "gpu": name, "power_limit_w": limit,
                          "timing": "host wall clock around each single assembly, device-synchronised, max over "
                                    "ranks; scorers alternate, order swapped every iteration"}))


if __name__ == "__main__":
    main()
