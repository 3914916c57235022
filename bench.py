#!/usr/bin/env python
"""bench.py -- pairs/sec of the PuzzleNet pair-matching forward (predict5) at B=64 pairs x 1024 points.

One step = one pass of the hot path (`TouchedRegraster.predict5`, need=False, eval) over one batch of 64
synthetic piece pairs per GPU (BASELINE.json configs[1]).  Prints ONE JSON line (rank 0).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--precision split|bf16|fp32] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...     # the reference algorithm's CPU path (oracle port), same metric and config

The headline precision is `split` (fp16 hi/lo operand planes, three tcgen05 MMAs per product, fp32 accumulation): the
tensor-core path that meets EVERY tolerance north_star states (features / logits 1e-4, rotation 0.01 deg, translation
1e-4).  The plain-bf16 path (2e-2 on features; it does not meet the pose bound) and the fp32 FFMA path are timed in the
same run and reported beside it (`bf16_path`, `fp32_path`), each with the parity figures of its own outputs.

value : device-resident inputs (128 rotating batches = 201 MB, larger than the 126 MB L2), K steps bracketed by one pair
        of CUDA events; batches alternate over --pipes CUDA streams, each replaying one captured CUDA graph per forward
        (the same schedule as the e2e leg, minus the host copies); max over ranks; the K-step region is repeated
        --repeats times and the MEDIAN is reported (spread alongside).
single_stream : the same K steps launched eagerly on ONE stream with per-step events and an L2 flush between steps
        (the latency view: what a plain `predict5` call costs; the kernels of the split path chain by programmatic
        dependent launch here).  The per-stage events that feed the rooflines come from separate passes with the stage
        recorder on.
e2e   : same metric through the public API from pinned HOST buffers: H2D of both clouds + FPS starts and D2H of the
        twist + both boundary-logit tensors inside the timed region.
parity: the outputs the LAST e2e step copied to the host, checked against the CPU oracle on 8 pairs of that batch (pairs
        are independent in eval mode), plus the same check of the other precisions' outputs on the same batch.
--dump-outputs DIR : what predict5 returned in the last step of the value leg (twist `out` [64,6], boundary logits
        `de_fpcb` / `de_mrpcb` [64,2,1024]) as DIR/<name>.npy.  Inputs and weights are seeded, so two builds run with the
        same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B_PAIRS = 64          # pairs per GPU per step (train.py default batch, BASELINE configs[1])
N_POINTS = 1024
METRIC = "pairs/sec PuzzleNet fwd B=64 N=1024"
UNIT = "pairs/s"
PARITY_PAIRS = list(range(0, B_PAIRS, 8))     # the 8 pairs of a batch the oracle re-computes

# dense MACs of one pair forward as the reference executes it (SURVEY.md §8d: 7.347 GFLOP/pair)
FLOP_PER_PAIR_REFERENCE = 7.347e9
DTYPES = {"fp32": "f32", "bf16": "bf16",
          "split": "f16x3 (fp16 hi/lo operand planes, 3 tcgen05 MMAs per product, fp32 accumulate)"}


def workload_config():
    """The `config` object: identical in both arms (--impl ours / reference)."""
    return {"workload": "predict5 fwd (need=False, eval), B=64 pairs x 1024 pts per step (BASELINE configs[1])",
            "pairs_per_step": B_PAIRS, "points": N_POINTS,
            "weights": "synthetic_state_dict(0) (no checkpoint is shipped with the reference)",
            "inputs": "synthetic_pairs: uniform-cube clouds, seeded",
            "l2": "GPU arm: inputs larger than L2 (128 rotating device-resident batches = 201 MB); its single_stream leg "
                  "writes a 256 MiB flush between steps, outside the per-step events.  CPU arm: not applicable"}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        # "under load": the upper half of the samples (idle samples before/after the region drag the median)
        sm.sort()
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU legs (oracle port of the reference's torch-CPU algorithm): cpu_baseline and --impl reference
# --------------------------------------------------------------------------------------------------
def _time_cpu_predict5(pairs: int, reps: int, threads: int, warmup: int = 1):
    """[seconds per call] of oracle.puzzle_oracle.predict5 on `pairs` pairs with `threads` intra-op threads."""
    import torch
    from oracle import puzzle_oracle as po
    from puzzlenet_b200.weights import synthetic_pairs, synthetic_state_dict
    torch.set_num_threads(threads)
    sd = synthetic_state_dict(0)
    fpc, mrpc = synthetic_pairs(pairs, seed=64)
    times = []
    with torch.no_grad():
        for i in range(warmup + reps):
            torch.manual_seed(1234 + i)
            t0 = time.perf_counter()
            po.predict5(sd, fpc, mrpc)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    return times


def _time_cpu_c3(clouds: int, threads: int):
    """BASELINE config 3 on the CPU (SURVEY §8d): sample_and_group(1024, 0, 32, xyz [B,11000,3], feats [B,11000,64],
    knn=True) + Linear(67,128)+ReLU+Linear(128,128)+ReLU+max, seconds per cloud (one repetition, bounded)."""
    import torch
    from oracle import puzzle_oracle as po
    from puzzlenet_b200.weights import synthetic_state_dict
    torch.set_num_threads(threads)
    sd = synthetic_state_dict(0)
    xyz = torch.rand(clouds, 11000, 3, generator=torch.Generator().manual_seed(3)) - 0.5
    feat = torch.randn(clouds, 11000, 64, generator=torch.Generator().manual_seed(4))
    with torch.no_grad():
        torch.manual_seed(5)
        t0 = time.perf_counter()
        _, grouped = po.sample_and_group(1024, 0, 32, xyz, feat, knn=True)
        h = torch.relu(po._lin(sd, "Encoder.mlp4", torch.relu(po._lin(sd, "Encoder.mlp3", grouped)))).max(dim=-2).values
        dt = time.perf_counter() - t0
    assert h.shape == (clouds, 1024, 128)
    return dt / clouds


def cpu_baseline_protocol():
    """BASELINE.md §3: the reference's torch-CPU path (oracle port) on this box's host cores, all cores AND one thread
    (the reference forces OMP_NUM_THREADS=1, test.py:4-5), C2 (bounded sample of the B=64 batch), C1 (B=4) and C3 (per
    cloud), >= 3 repetitions each with min and median."""
    import torch
    cores = os.cpu_count() or 1
    out = {"cpu_model": _cpu_model(), "cores": cores, "kind": "port",
           "what": "oracle.puzzle_oracle.predict5 = the reference's torch-CPU op sequence (pinned against the unmodified "
                   "reference's stored outputs by tests/test_oracle_golden.py), fp32, eval mode"}

    def summarise(times, pairs):
        return {"pairs_per_call": pairs, "reps": len(times), "s_min": min(times), "s_median": statistics.median(times),
                "pairs_per_s_median": pairs / statistics.median(times), "pairs_per_s_best": pairs / min(times)}

    out["c2_all_cores"] = summarise(_time_cpu_predict5(16, 3, cores), 16)
    out["c2_1_thread"] = summarise(_time_cpu_predict5(4, 3, 1), 4)
    out["c1_b4_all_cores"] = summarise(_time_cpu_predict5(4, 3, cores), 4)
    out["c1_b4_1_thread"] = summarise(_time_cpu_predict5(4, 3, 1, warmup=0), 4)
    try:
        out["c3_per_cloud_s_all_cores"] = _time_cpu_c3(2, cores)
    except Exception as e:  # noqa: BLE001 -- host RAM on an unknown box
        out["c3_per_cloud_s_all_cores"] = f"failed: {e!r}"[:120]
    torch.set_num_threads(cores)
    out["value"] = out["c2_all_cores"]["pairs_per_s_median"]
    out["unit"] = UNIT
    out["sample"] = ("C2: 3 reps x 16 pairs (all cores) / 3 reps x 4 pairs (1 thread) of the B=64 workload; C1: 3 reps x B=4; "
                     "C3: 1 rep x 2 clouds; 1 warm-up call each")
    return out


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path (the oracle port; the reference itself is not an
    installable package, DESIGN.md §2) with all host threads, on the GPU arm's config: B=64 pairs per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0                                    # the other ranks exit without work
    import torch
    cores = os.cpu_count() or 1
    pairs = B_PAIRS
    probe = _time_cpu_predict5(8, 1, cores, warmup=1)[0] / 8           # seconds per pair, warm
    budget_s = 200.0
    while pairs > 8 and probe * pairs * (args.steps + args.warmup) > budget_s:
        pairs //= 2                                  # bounded sample: keep the whole run within a few minutes
    times = _time_cpu_predict5(pairs, args.steps, cores, warmup=args.warmup)
    sec = statistics.mean(times)
    value = pairs / sec
    cfg = workload_config()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "cpu_model": _cpu_model(),
                         "sample": f"{args.steps} steps x {pairs} pairs per step"
                                   + ("" if pairs == B_PAIRS else f" (bounded sample of the {B_PAIRS}-pair step)")
                                   + ", oracle.puzzle_oracle.predict5 (torch CPU fp32, all host threads)",
                         "s_per_step_min_median": [min(times), statistics.median(times)]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_line(line)
    return 0


# --------------------------------------------------------------------------------------------------
# the other BASELINE configs (3, 4, 5), short runs at every N: every rank takes part, rank 0 reports
# --------------------------------------------------------------------------------------------------
def _max_over_ranks(x, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item()


def _timed(fn, iters, warm=2, groups=3):
    """ms per call: the best of `groups` event-bracketed loops of `iters` calls (a one-off allocator / driver stall inside
    one loop -- seen once as a 40x outlier on a freshly released CUDA-graph pool -- does not end up in the record)."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    best, out = None, None
    for _ in range(groups):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        best = ms if best is None else min(best, ms)
    return best, out


def _bench_c3(dev, world, hbm_peak, iters=5):
    """BASELINE config 3: FPS 11000->1024, kNN k=32, gather + MLP 67->128->128 + max-pool, B=64 clouds PER GPU (weak
    scaling; ms = max over ranks).  Fractions of the HBM peak are on the algorithmic bytes of SURVEY §8(d)."""
    import torch
    from puzzlenet_b200 import pointnet_util as pu
    from puzzlenet_b200.weights import synthetic_state_dict
    B, N, S, K, D, C2 = 64, 11000, 1024, 32, 64, 128
    rank = int(os.environ.get("RANK", "0"))
    xyz = (torch.rand(B, N, 3, generator=torch.Generator().manual_seed(3 + rank)) - 0.5).to(dev)
    feat = torch.randn(B, N, D, generator=torch.Generator().manual_seed(4 + rank)).to(dev)
    sd = synthetic_state_dict(0)
    w1, b1 = sd["Encoder.mlp3.weight"].to(dev), sd["Encoder.mlp3.bias"].to(dev)
    w2, b2 = sd["Encoder.mlp4.weight"].to(dev), sd["Encoder.mlp4.bias"].to(dev)
    torch.manual_seed(5)
    with torch.no_grad():
        t_fps, fps_idx = _timed(lambda: pu.farthest_point_sample(xyz, S), iters)
        new_xyz = pu.index_points(xyz, fps_idx)
        t_knn, idx = _timed(lambda: pu.knn_point(K, xyz, new_xyz), iters)
        stages = {"fps": (t_fps, B * (12 * N + 8 * S)), "knn": (t_knn, B * (12 * N + 12 * S + 8 * S * K))}
        group_bytes = B * (12 * N + 4 * N * D + 8 * S + 8 * S * K + 12 * S + 4 * S * C2)
        for name, prec in (("split", 2), ("bf16", 1), ("fp32", 0)):
            t, _ = _timed(lambda: pu.group_mlp_maxpool(xyz, feat, new_xyz, idx, w1, b1, w2, b2, precision=prec), iters)
            stages[f"group_mlp_maxpool_{name}"] = (t, group_bytes)
        t_sg, _ = _timed(lambda: pu.sample_and_group(S, 0, K, xyz, feat, False, True), max(2, iters // 2))
        stages["sample_and_group_materialising"] = (t_sg, B * (12 * N + 4 * N * D + 12 * S + 4 * S * K * (3 + D)))
        # the group stage alone (index_points + centre + concat, pointnet_util.py:123-130): the HBM-bound part of the path
        from puzzlenet_b200 import _lib

        def group_only(xyz_, feat_, nx_, idx_, n_, s_):
            b_ = xyz_.shape[0]
            out = torch.empty(b_, s_, K, 3 + D, device=dev)
            fn = lambda: _lib.call("pz_group_concat", xyz_.data_ptr(), feat_.data_ptr(), nx_.data_ptr(), idx_.data_ptr(), b_, n_,  # noqa: E731
                                   D, s_, K, out.data_ptr(), None, _lib.stream_ptr())
            return _timed(fn, iters)[0], b_ * (12 * n_ + 4 * n_ * D + 8 * s_ * K + 12 * s_ + 4 * s_ * K * (3 + D))
        stages["group_gather_concat_only"] = group_only(xyz, feat, new_xyz, idx, N, S)
        # ... and at the C2 shape (128 clouds x 1024 points -> 512 groups), the shape of the model's first stage
        x2 = xyz[:, :1024].repeat(2, 1, 1).contiguous()
        f2 = feat[:, :1024].repeat(2, 1, 1).contiguous()
        nx2 = x2[:, :512].contiguous()
        idx2 = pu.knn_point(K, x2, nx2)
        stages["group_gather_concat_only_c2_shape"] = group_only(x2, f2, nx2, idx2, 1024, 512)
    res = {"workload": f"C3: FPS {N}->{S}, kNN k={K}, gather+MLP 67->128->128+max-pool, B={B} clouds per GPU", "n_gpus": world,
           "clouds_total": B * world, "note": "FPS / kNN are latency / issue bound (SURVEY 8d): their HBM fraction is "
           "reported on the compulsory bytes as the contract asks; the materialising sample_and_group API is the HBM-bound one"}
    for k, (ms, byts) in stages.items():
        ms = _max_over_ranks(ms, dev, world)
        gbs = byts / (ms / 1e3) / 1e9
        res[k] = {"ms": round(ms, 4), "algorithmic_MB_per_gpu": round(byts / 1e6, 2), "GBps_per_gpu": round(gbs, 1),
                  "frac_hbm_peak": round(gbs / hbm_peak, 5)}
    return res


def _bench_training(dev, world, pairs=B_PAIRS, steps=4, warmup=2):
    """BASELINE config 4: training step (pose + boundary losses + EMD), `pairs` per GPU, data-parallel with the bucketed
    NCCL all-reduce of the flat gradient buffer; pairs/s = all ranks' pairs / max-over-ranks step time."""
    import types
    import torch
    from puzzlenet_b200.model5_b import TouchedRegraster
    from puzzlenet_b200.training import Trainer
    from puzzlenet_b200.weights import synthetic_state_dict
    from scripts.bench_train import make_training_batch
    rank = int(os.environ.get("RANK", "0"))
    out = {"workload": f"training_step (loss_mode 1: chamfer + pose + EMD + boundary CE/chamfer), {pairs} pairs per GPU, "
                       f"global batch {pairs * world}", "unit": UNIT, "n_gpus": world}
    batch = make_training_batch(pairs, 64 + rank, dev)
    for prec in ("tf32", "fp32"):
        model = TouchedRegraster(types.SimpleNamespace(dataset="vase", loss_mode=1, loss_sum=False, lr=1e-5))
        model.load_state_dict(synthetic_state_dict(0))
        model.to(dev)
        tr = Trainer(model, precision=prec)
        first = last = None
        for _ in range(warmup):
            loss = tr.training_step(batch)["loss"]
            first = loss if first is None else first
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            last = tr.training_step(batch)["loss"]
        e1.record()
        torch.cuda.synchronize()
        ms = _max_over_ranks(e0.elapsed_time(e1) / steps, dev, world)
        # exposed communication: one more step with the phases separated by events (all-reduce after backward, no overlap)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        tr.overlap_allreduce = False
        ev[0].record()
        tr.forward_backward(batch)
        ev[1].record()
        w = tr.all_reduce_grads()
        ev[2].record()
        tr.optimizer_step(w)
        torch.cuda.synchronize()
        out[prec] = {"value": pairs * world / ms * 1e3, "ms_per_step": ms, "loss_first_last": [first, last],
                     "allreduce_ms_unoverlapped": _max_over_ranks(ev[1].elapsed_time(ev[2]), dev, world),
                     "forward_backward_ms": _max_over_ranks(ev[0].elapsed_time(ev[1]), dev, world),
                     "grad_elems_allreduced": tr.flat.n if world > 1 else 0}
        del tr, model
        torch.cuda.empty_cache()
    return out


def _bench_assembly(model, dev, world, pieces=32, points=11000, iters=5):
    """BASELINE config 5: 32 pieces x 11000 points, 496 candidate pairs sharded over the ranks (strong scaling)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from puzzlenet_b200 import assembly
    from scripts.bench_assembly import dublin_like_piece
    raw = [dublin_like_piece(i, points) for i in range(pieces)]
    starts = [int(np.random.default_rng(100 + i).integers(0, points)) for i in range(pieces)]
    scorer = assembly.ModelScorer(model, pipes=4)     # batches of 64 pairs alternate over 4 streams, one graph replay each
    model.cuda_graphs = True

    def once():
        torch.manual_seed(1234)
        clouds = assembly.downsample_pieces(raw, 1024, starts=starts, device=dev)
        pairs, rows = assembly.score_all_pairs(clouds, scorer, batch=64)
        return assembly.greedy_assemble(pieces, pairs, rows)

    for _ in range(3):
        once()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(iters):
        _, _, merges = once()
    torch.cuda.synchronize()
    ms = _max_over_ranks((time.perf_counter() - t0) / iters * 1e3, dev, world)
    model.cuda_graphs = False
    n_pairs = pieces * (pieces - 1) // 2
    return {"workload": f"{pieces} pieces x {points} pts: FPS 11000->1024 (pieces sharded), {n_pairs} pairs scored (pairs "
                        "sharded), greedy merge", "n_gpus": world, "scaling": "strong", "precision": model.precision,
            "ms_per_assembly": ms, "pairs_per_s": n_pairs / ms * 1e3, "merges": len(merges),
            "timing": "host wall clock incl. H2D of the raw pieces, the all_gathers and the host-side merge; max over ranks"}


def _bench_emd(dev):
    """EMD (A13) at b=64, n=m=1024: ours vs the reference's own kernels compiled for sm_100a with their original launch
    shapes (oracle/_ref/libemd_ref.so -- the kernel-to-beat BASELINE.md §3 names), same GPU, same inputs."""
    import ctypes
    import torch
    from puzzlenet_b200 import emd_cuda
    b, n, m = 64, 1024, 1024
    g = torch.Generator().manual_seed(0)
    x1 = (torch.randn(b, n, 3, generator=g) * 0.5).to(dev)
    x2 = (torch.randn(b, m, 3, generator=g) * 0.5).to(dev)
    gc = torch.ones(b, device=dev)
    match = emd_cuda.approxmatch_forward(x1, x2)
    res = {"b": b, "n": n, "m": m,
           "ours_ms": {"approxmatch": _timed(lambda: emd_cuda.approxmatch_forward(x1, x2), 5)[0],
                       "matchcost": _timed(lambda: emd_cuda.matchcost_forward(x1, x2, match), 5)[0],
                       "matchcost_backward": _timed(lambda: emd_cuda.matchcost_backward(gc, x1, x2, match), 5)[0]}}
    # exp2 floor: 30 * n * m exponentials per item on the MUFU pipe (16 per SM and clock)
    res["approxmatch_mufu_floor_ms"] = 30.0 * b * n * m / (148 * 16 * 1.965e9) * 1e3
    so = os.path.join(ROOT, "oracle", "_ref", "libemd_ref.so")
    if os.path.isfile(so):
        ref = ctypes.CDLL(so)
        vp = ctypes.c_void_p
        rmatch = torch.empty(b, m, n, device=dev)
        temp = torch.empty(32 * (n + m) * 2, device=dev)
        cost = torch.empty(b, device=dev)
        g1, g2 = torch.empty(b, n, 3, device=dev), torch.empty(b, m, 3, device=dev)
        st = vp(torch.cuda.current_stream().cuda_stream)
        res["reference_kernels_ms"] = {
            "approxmatch": _timed(lambda: ref.emd_ref_approxmatch(b, n, m, vp(x1.data_ptr()), vp(x2.data_ptr()), vp(rmatch.data_ptr()), vp(temp.data_ptr()), st), 3)[0],
            "matchcost": _timed(lambda: ref.emd_ref_matchcost(b, n, m, vp(x1.data_ptr()), vp(x2.data_ptr()), vp(rmatch.data_ptr()), vp(cost.data_ptr()), st), 3)[0],
            "matchcost_backward": _timed(lambda: ref.emd_ref_matchcost_grad(b, n, m, vp(gc.data_ptr()), vp(x1.data_ptr()), vp(x2.data_ptr()), vp(rmatch.data_ptr()), vp(g1.data_ptr()), vp(g2.data_ptr()), st), 3)[0],
        }
        res["speedup_vs_reference_kernels"] = {k: round(res["reference_kernels_ms"][k] / res["ours_ms"][k], 2) for k in res["ours_ms"]}
        res["max_abs_match_diff"] = (match - rmatch).abs().max().item()
    else:
        res["reference_kernels_ms"] = "oracle/_ref/libemd_ref.so not built"
    return res


def _torch_gpu_baseline(dev, steps=3):
    """The real "today on a GPU" number (BASELINE.md §3): the reference's torch op sequence -- the oracle port, with only
    the placement of arange / randint / constants following the input's device -- on the SAME B200, B=64, stock
    ATen / cuBLAS kernels; once as written (five torch.cuda.empty_cache() per sample_and_group) and once without them."""
    import torch
    from oracle import puzzle_oracle as po
    from puzzlenet_b200.weights import synthetic_pairs, synthetic_state_dict
    sd = {k: v.to(dev) for k, v in synthetic_state_dict(0).items()}
    fpc, mrpc = (t.to(dev) for t in synthetic_pairs(B_PAIRS, seed=64))
    out = {"what": "oracle.puzzle_oracle.predict5 on CUDA tensors (stock PyTorch kernels), B=64, eval, fp32 (TF32 off)",
           "unit": UNIT}
    torch.backends.cuda.matmul.allow_tf32 = False
    for key, flag in (("as_written_with_empty_cache", True), ("without_empty_cache", False)):
        po.REFERENCE_EMPTY_CACHE = flag
        try:
            with torch.no_grad():
                torch.manual_seed(1)
                po.predict5(sd, fpc, mrpc)            # warm-up (cuBLAS handles, allocator)
                torch.cuda.synchronize()
                times = []
                for i in range(steps):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.manual_seed(2 + i)
                    e0.record()
                    po.predict5(sd, fpc, mrpc)
                    e1.record()
                    torch.cuda.synchronize()
                    times.append(e0.elapsed_time(e1))
            out[key] = {"ms_per_step_min": min(times), "ms_per_step_median": statistics.median(times),
                        "value": B_PAIRS / statistics.median(times) * 1e3}
        finally:
            po.REFERENCE_EMPTY_CACHE = False
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import types
    import torch
    import torch.distributed as dist
    from puzzlenet_b200 import _lib
    from puzzlenet_b200.model5_b import TouchedRegraster
    from puzzlenet_b200.weights import make_batch, synthetic_pairs, synthetic_state_dict

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (puzzlenet_b200 has no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    sd = synthetic_state_dict(0)
    model = TouchedRegraster(types.SimpleNamespace(dataset="vase"))
    model.load_state_dict(sd, strict=True)
    model.to(dev).eval()
    model.precision = args.precision
    B = B_PAIRS
    nsets = 4                                         # distinct synthetic batches, rotated
    host, host_plain = [], []
    for i in range(nsets):
        fpc, mrpc = synthetic_pairs(B, seed=64 + 1000 * rank + i)
        g = torch.Generator().manual_seed(5 + i)
        starts = torch.stack([torch.randint(0, n, (B,), generator=g) for n in (1024, 512, 1024, 512)])
        host_plain.append((fpc, mrpc, starts))
        host.append((fpc.pin_memory(), mrpc.pin_memory(), starts.pin_memory()))
    resident = [(f.to(dev), m.to(dev), s.to(dev)) for f, m, s in host]
    batches = [make_batch(f, m) for f, m, _ in resident]
    # pipelined leg: enough distinct resident batches that one rotation exceeds L2 (128 x 1.57 MB = 201 MB > 126 MB)
    n_rot = 128
    rot = []
    for i in range(n_rot):
        fpc, mrpc = synthetic_pairs(B, seed=10_000 + 1000 * rank + i)
        g = torch.Generator().manual_seed(500 + i)
        starts = torch.stack([torch.randint(0, n, (B,), generator=g) for n in (1024, 512, 1024, 512)])
        rot.append((make_batch(fpc.to(dev), mrpc.to(dev)), starts.to(dev)))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident(i):
        return model.predict5(batches[i % nsets], 0, starts=resident[i % nsets][2])

    for i in range(args.warmup):
        step_resident(i)
    barrier()

    # ---- single-stream leg: device-resident inputs, eager launches, per-step events, L2 flush between steps
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = lib.pz_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()
        ev[i][0].record()
        step_resident(i)
        ev[i][1].record()
    barrier()
    wall = time.perf_counter() - t_wall0
    launches = lib.pz_launch_count() - launches0
    total_ms = sum(a.elapsed_time(b) for a, b in ev)

    # ---- the same steps with the stage recorder on (an event after every stage: the kernels are then launched without
    # programmatic dependent launch, so this pass is slower than the leg above and only its per-stage split is used)
    lib.pz_profile_enable(1)
    for i in range(min(args.steps, 20)):
        flush.zero_()
        step_resident(i)
    torch.cuda.synchronize()
    calls, stages = _lib.profile_collect()
    lib.pz_profile_enable(0)

    # ---- per-kernel durations for the rooflines: the same steps once more with the internal side stream switched off,
    # so that every stage's CUDA-event time is its own (above, the geometry chain overlaps the feature chain)
    lib.pz_profile_enable(2)
    for i in range(min(args.steps, 20)):
        flush.zero_()
        step_resident(i)
    torch.cuda.synchronize()
    calls_serial, stages_serial = _lib.profile_collect()
    lib.pz_profile_enable(0)

    # ---- pipelined schedule: several CUDA streams (--pipes) alternate so that the copies and the latency-bound stages
    # (FPS chain, pose MLP) of one batch overlap the tensor-core stages of the others
    pipes = [torch.cuda.Stream(device=dev) for _ in range(args.pipes)]
    out_hosts = [(torch.empty(B, 6).pin_memory(), torch.empty(B, 2, 1024).pin_memory(), torch.empty(B, 2, 1024).pin_memory())
                 for _ in range(args.pipes)]
    h2d = sum(t.numel() * t.element_size() for t in host[0])
    d2h = sum(t.numel() * t.element_size() for t in out_hosts[0])

    last_resident = {}        # what predict5 returned in the last step of the latest run_resident (--dump-outputs)

    def run_resident(n):
        for i in range(n):
            with torch.cuda.stream(pipes[i % len(pipes)]):
                bt, st_ = rot[i % n_rot]
                r = model.predict5(bt, 0, starts=st_)
        last_resident.update(out=r[0], de_fpcb=r[2], de_mrpcb=r[3])

    def step_e2e(i):
        f, m, s = host[i % nsets]
        fd, md = f.to(dev, non_blocking=True), m.to(dev, non_blocking=True)
        out, _, de_f, de_m = model.predict5(make_batch(fd, md), 0, starts=s)
        out_host = out_hosts[i % len(out_hosts)]
        out_host[0].copy_(out, non_blocking=True)
        out_host[1].copy_(de_f, non_blocking=True)
        out_host[2].copy_(de_m, non_blocking=True)

    def run_e2e(n):
        for i in range(n):
            with torch.cuda.stream(pipes[i % len(pipes)]):
                step_e2e(i)

    def timed_region(fn, n):
        """one K-step region inside one event pair on the main stream, which forks to / joins the pipes"""
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        main_stream = torch.cuda.current_stream()
        a.record()
        for p_ in pipes:
            p_.wait_stream(main_stream)
        fn(n)
        for p_ in pipes:
            main_stream.wait_stream(p_)
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def pipelined(precision, reps):
        """(value region times [ms], e2e region times [ms]) of `precision`, CUDA graphs unless --no-graphs"""
        model.precision = precision
        model.cuda_graphs = not args.no_graphs
        try:
            run_resident(max(2 * len(pipes), args.warmup))
            v = [timed_region(run_resident, args.steps) for _ in range(reps)]
            run_e2e(max(len(pipes), args.warmup))
            e = [timed_region(run_e2e, args.steps) for _ in range(reps)]
        finally:
            model.cuda_graphs = False
            model.precision = args.precision
        return v, e

    value_regions, e2e_regions = pipelined(args.precision, args.repeats)
    # the headline's last timed step (last value region, step K-1, batch rot[(K-1) % n_rot]): its outputs for --dump-outputs
    dump = {k: v.float().cpu().numpy() for k, v in last_resident.items()} if args.dump_outputs else None
    # the outputs of the LAST e2e step are in its pinned host slot: keep them for the parity check below
    last = args.steps - 1
    e2e_last = tuple(t.clone() for t in out_hosts[last % len(out_hosts)])
    e2e_last_inputs = host_plain[last % nsets]
    clocks = sampler.stop() if sampler else None

    # ---- the other precisions of BASELINE configs[1] ("fp32 and bf16"), same run
    others = {}
    if not args.single_precision:
        for prec in ("split", "bf16"):
            if prec != args.precision:
                v, e = pipelined(prec, max(1, min(3, args.repeats)))
                others[prec] = (statistics.median(v), statistics.median(e), args.steps, "pipelined over CUDA streams, graph replays")
        if args.precision != "fp32":       # the FFMA path: single stream, few steps (11 ms per step)
            model.precision = "fp32"
            k2 = min(args.steps, 10)
            for i in range(3):
                step_resident(i)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(k2):
                step_resident(i)
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            others["fp32"] = (t.item(), None, k2, "single stream, eager launches")
            model.precision = args.precision

    # ---- parity of what was timed (rank 0): outputs of the last e2e step vs the CPU oracle, 8 pairs of that batch; and
    # the other precisions' outputs on the same batch
    parity_all = None
    if rank == 0 and not args.no_parity:
        from oracle import parity as pz_parity
        fpc_h, mrpc_h, starts_h = e2e_last_inputs
        idx = torch.as_tensor(PARITY_PAIRS)
        ref = pz_parity.oracle_subset(sd, fpc_h, mrpc_h, starts_h, idx)
        parity_all = {}
        p = pz_parity.predict5_parity(sd, fpc_h, mrpc_h, starts_h, *e2e_last, PARITY_PAIRS, ref=ref)
        p.update(source="outputs of the last timed e2e step (pinned host buffers)", precision=args.precision,
                 within_claimed_bounds=pz_parity.within(p, args.precision),
                 bounds=dict(zip(("rel", "rel_elem", "rot_deg", "trans"), pz_parity.BOUNDS[args.precision])),
                 claims_pose_tolerance=pz_parity.POSE_CLAIMED[args.precision])
        parity_all[args.precision] = p
        for prec in ("split", "bf16", "fp32"):
            if prec == args.precision:
                continue
            model.precision = prec
            out, _, de_f, de_m = model.predict5(make_batch(fpc_h.to(dev), mrpc_h.to(dev)), 0, starts=starts_h)
            torch.cuda.synchronize()
            q = pz_parity.predict5_parity(sd, fpc_h, mrpc_h, starts_h, out, de_f, de_m, PARITY_PAIRS, ref=ref)
            q.update(source="eager predict5 on the same batch", precision=prec,
                     within_claimed_bounds=pz_parity.within(q, prec),
                     bounds=dict(zip(("rel", "rel_elem", "rot_deg", "trans"), pz_parity.BOUNDS[prec])),
                     claims_pose_tolerance=pz_parity.POSE_CLAIMED[prec])
            parity_all[prec] = q
        model.precision = args.precision

    # ---- reduce over ranks: max time, total pairs
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = t.item()
    pairs_total = B * args.steps * world
    value_ms, e2e_ms = statistics.median(value_regions), statistics.median(e2e_regions)
    value = pairs_total / (value_ms / 1e3)
    single_value = pairs_total / (total_ms / 1e3)
    e2e_value = pairs_total / (e2e_ms / 1e3)
    launches_eager_per_step = launches / max(args.steps, 1)

    # ---- the other BASELINE configs at this N (every rank takes part)
    peaks = _peaks()
    other_configs = None
    if not args.no_extras:
        other_configs = {}
        model._graphs.clear()            # hand the captured graphs' workspaces back before the extras allocate theirs
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        for key, fn in (("config3_sample_and_group_microbench", lambda: _bench_c3(dev, world, peaks["hbm"])),
                        ("config4_training_step", lambda: _bench_training(dev, world)),
                        ("config5_assembly", lambda: _bench_assembly(model, dev, world))):
            try:
                other_configs[key] = fn()
            except Exception as e:   # noqa: BLE001 -- extras must never take the headline line down
                other_configs[key] = {"error": repr(e)[:300]}
                if world > 1:        # keep the ranks in step after a failure on one of them
                    torch.cuda.synchronize()
        if rank == 0 and world == 1:
            try:
                other_configs["emd_microbench"] = _bench_emd(dev)
            except Exception as e:   # noqa: BLE001
                other_configs["emd_microbench"] = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant stage (live per-stage CUDA events from the timed steps)
    def per_step_of(stage_list, ncalls):
        agg = {}
        for name, ms in stage_list:
            if not name.startswith("_"):
                agg[name] = agg.get(name, 0.0) + ms
        return {k: v / max(ncalls, 1) for k, v in agg.items()}

    per_step_overlapped = per_step_of(stages, calls)
    per_step = per_step_of(stages_serial, calls_serial)
    clouds = 2 * B
    mma_factor = 3 if args.precision == "split" else 1
    fused = args.precision == "bf16"
    split_fused = args.precision == "split" and not os.environ.get("PZ_ATTN_NO_FUSE")
    chained = split_fused and not os.environ.get("PZ_ATTN_NO_CHAIN")
    # algorithmic work of each stage per step (DESIGN.md §4): FLOPs of the reference's product for the dense stages (tensor
    # bound; the split path EXECUTES three MMAs per product -- `executed` below), compulsory bytes for the geometry stages
    # (SURVEY.md §8d; they are latency / issue bound, the HBM fraction is reported truthfully).  (work, bound, launches)
    work = {
        "sg1_gather_layer2_maxpool": (2.0 * clouds * 512 * 32 * 128 * 128, "tensor", 1),
        "sg2_gather_layer2_maxpool": (2.0 * clouds * 256 * 32 * 256 * 256, "tensor", 1),
        "tail_linear_maxpool": (2.0 * clouds * 256 * 1280 * 1024, "tensor", 1),
        "tail_linear": (2.0 * clouds * 256 * 1280 * 1024, "tensor", 1),
        "attn_layer_fused": (4 * 2.0 * clouds * 256 * 256 * (384 + 64 + 256 + 256), "tensor", 1),
        # split path (default build): the out-projection and the NEXT layer's q|k|v projections run inside the attention kernel
        # (attention_split.cu); only layer 0's projections are launches of their own
        "attn_qkv_proj": ((1 if chained else 4) * 2.0 * clouds * 256 * 256 * 384, "tensor",
                          (2 if chained else 8) if not fused and args.precision != "fp32" else 12),
        "attn_out_proj": (4 * 2.0 * clouds * 256 * 256 * 256, "tensor", 4),
        "attn_softmax_av": (2.0 * clouds * 256 * 256 * (4 * (64 + 256) + (4 * 256 if split_fused else 0) + (3 * 384 if chained else 0)),
                            "tensor", 4),
        "fps1": (clouds * (12 * 1024 + 8 * 512), "hbm", 1),
        "fps2": (clouds * (12 * 512 + 8 * 256), "hbm", 1),
        "knn1": (clouds * (12 * 1024 + 12 * 512 + 8 * 512 * 32), "hbm", 1),
        "knn2": (clouds * (12 * 512 + 12 * 256 + 8 * 256 * 32), "hbm", 1),
    }
    tensor_note = {"fp32": "fp32 path: the GEMMs run on the FFMA pipe; shown against the tensor-pipe peak",
                   "bf16": "tcgen05 bf16 x bf16 -> fp32",
                   "split": "tcgen05 fp16 hi/lo planes: `achieved` counts the reference's product once (algorithmic FLOPs); the "
                            "kernel executes 3 MMAs per product, see `executed`"}[args.precision]

    def roof(name):
        w, bound, nl = work[name]
        sec = per_step[name] / 1e3
        if bound == "tensor":
            ach, peak, unit, src = w / sec / 1e12, peaks["tf_sust"], "TFLOP/s", f"{peaks['src']} bf16 sustained"
        else:
            ach, peak, unit, src = w / sec / 1e9, peaks["hbm"], "GB/s", f"{peaks['src']} copy"
        r = {"bound": bound, "kernel": name, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
             "traffic": None, "peak_source": src, "ms_per_launch": per_step[name] / nl, "launches_per_step": nl}
        if bound == "tensor":
            r["note"] = tensor_note
            if mma_factor != 1:
                r["executed"] = {"achieved": ach * mma_factor, "unit": unit, "frac": ach * mma_factor / peak,
                                 "what": "MMA FLOPs issued to the tensor pipe (3 per algorithmic FLOP)"}
            if name.startswith("sg") and args.precision != "fp32":
                # the gathered operand: rows x channels of layer-1 output fetched through L2 (fp32 in the split path,
                # bf16 in the bf16 path); each source row is gathered ~16 times, so this traffic never reaches HBM
                rows_k = {"sg1_gather_layer2_maxpool": (clouds * 512 * 32, 128), "sg2_gather_layer2_maxpool": (clouds * 256 * 32, 256)}[name]
                gb = rows_k[0] * rows_k[1] * (4 if args.precision == "split" else 2) / 1e9
                r["l2_gather"] = {"GB_per_launch": round(gb, 3), "GBps": round(gb / sec, 1),
                                  "what": "gathered P rows (L2 -> SM); scripts/l2_probe.cu measures 14-20 TB/s for random 128-byte "
                                          "row pieces when enough loads are in flight: the producers, not L2, bound this stage"}
        elif name.startswith("knn"):
            r["note"] = ("fp32 ALU + selection bound, not HBM bound (SURVEY 8d); the HBM fraction is reported on the compulsory "
                         "bytes as the contract asks")
        elif name.startswith("fps"):
            r["note"] = "serial arg-max chain (S dependent iterations per cloud): latency bound, cannot approach HBM peak"
        return r

    rooflines = {k: roof(k) for k in work if per_step.get(k, 0) > 0}
    ncu_traffic = _ncu_traffic(args.precision)
    for k, r in rooflines.items():
        if k in ncu_traffic:
            r["traffic"] = ncu_traffic[k]["bytes"]
            r["traffic_source"] = ncu_traffic[k]["source"]
    # dominant kernel = the stage with the largest live time among those with a defined roofline
    roofline = rooflines[max(rooflines, key=lambda k: per_step[k])] if rooflines else None

    cpu_baseline = torch_gpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_protocol()
    if world == 1 and not args.no_torch_gpu_baseline:
        try:
            torch_gpu = _torch_gpu_baseline(dev)
        except Exception as e:   # noqa: BLE001
            torch_gpu = {"error": repr(e)[:300]}

    def path_line(prec):
        if prec not in others:
            return None
        v_ms, e_ms, k, how = others[prec]
        d = {"value": B * k * world / (v_ms / 1e3), "unit": UNIT, "ms_per_step": v_ms / k, "steps": k, "how": how,
             "dtype": DTYPES[prec]}
        if e_ms is not None:
            d["e2e"] = {"value": B * k * world / (e_ms / 1e3), "unit": UNIT, "ms_per_step": e_ms / k}
        if parity_all and prec in parity_all:
            d["parity"] = parity_all[prec]
        return d

    cfg = workload_config()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": value_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPES[args.precision], "precision": args.precision, "data": "synthetic", "config": cfg,
        "schedule": {"parallelism": f"dp{world} (pairs sharded, no forward collective)",
                     "streams": f"batches alternate over {args.pipes} CUDA streams"
                                + ("" if args.no_graphs else ", one captured CUDA graph replay per forward"),
                     "repeats": args.repeats,
                     "value_ms_per_step_all_repeats": [round(x / args.steps, 5) for x in value_regions],
                     "e2e_ms_per_step_all_repeats": [round(x / args.steps, 5) for x in e2e_regions],
                     "reported": "median over the repeats of the K-step region"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / args.steps,
                "how": f"public API predict5 from pinned host buffers; batches alternate over {args.pipes} CUDA streams"
                       + ("" if args.no_graphs else ", each replaying one captured CUDA graph per forward")},
        "parity": parity_all[args.precision] if parity_all else None,
        "single_stream": {"value": single_value, "unit": UNIT, "ms_per_step": total_ms / args.steps,
                          "how": "eager launches on one stream (programmatic dependent launch between the split path's "
                                 "kernels), per-step CUDA events, L2 flushed between steps"},
        "gpu_launches": int(round(launches_eager_per_step * args.steps)),
        "gpu_launches_note": f"{launches_eager_per_step:.0f} kernels per forward (counted on the eager single-stream leg; "
                             "the value / e2e legs replay the same kernels from a captured CUDA graph)",
        "roofline": roofline,
        "roofline_all": {k: {"bound": v["bound"], "achieved": round(v["achieved"], 3), "unit": v["unit"],
                             "frac": round(v["frac"], 5),
                             **({"executed_frac": round(v["executed"]["frac"], 5)} if "executed" in v else {})}
                         for k, v in rooflines.items()},
        "cpu_baseline": cpu_baseline,
        "torch_gpu_baseline": torch_gpu,
        "stages_ms_per_step": {k: round(v, 4) for k, v in sorted(per_step.items(), key=lambda kv: -kv[1])},
        "stages_note": "stages_ms_per_step: CUDA events, stages back to back on one stream (used for the rooflines); "
                       "stages_ms_per_step_timed_region: the same events with the schedule of a plain call (bf16 / fp32 "
                       "paths: the geometry chain on a second stream, overlapping the feature chain; split path: one chain)",
        "stages_ms_per_step_timed_region": {k: round(v, 4) for k, v in sorted(per_step_overlapped.items(), key=lambda kv: -kv[1])},
        "split_path": path_line("split"), "bf16_path": path_line("bf16"), "fp32_path": path_line("fp32"),
        "other_configs": other_configs,
        "gflop_per_pair_reference_count": FLOP_PER_PAIR_REFERENCE / 1e9,
        "wall_s_single_stream_region": wall,
    }
    line = {k: v for k, v in line.items() if not (k.endswith("_path") and v is None)}
    if dump is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    emit_line(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def _ncu_traffic(precision):
    """DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed `ncu --set full` captures
    of this same forward (profiles/): {stage: {bytes, source}}; empty where no capture of the current kernels exists."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.isfile(path):
        return {}
    try:
        return json.load(open(path)).get(precision, {})
    except Exception:
        return {}


_REAL_STDOUT = None


def emit_line(line) -> None:
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.buffer.write(data)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("PZ_PRECISION", "split"), choices=["fp32", "bf16", "split"])
    ap.add_argument("--repeats", type=int, default=5, help="repetitions of the K-step timed region (median reported)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--single-precision", action="store_true", help="skip the runs of the other precisions")
    ap.add_argument("--pipes", type=int, default=4, help="CUDA streams the value / e2e legs alternate batches over")
    ap.add_argument("--no-graphs", action="store_true", help="value / e2e legs: eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-extras", action="store_true", help="skip the short config 3 / 4 / 5 / EMD runs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline path returned (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    args.repeats = max(args.repeats, 1)
    # stdout carries exactly ONE JSON line: libraries that write to file descriptor 1 themselves (NCCL prints its version
    # banner there when NCCL_DEBUG is set) are pointed at stderr for the whole run; emit_line writes to the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
