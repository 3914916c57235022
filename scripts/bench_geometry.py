"""The encoder's geometry (FPS 1024 -> 512, kNN 32, FPS 512 -> 256, kNN 32, centre projections Q1 / Q2) as one launch
per cloud vs the six launches it replaces, at 64 and 256 pairs (128 and 512 clouds).

    python scripts/bench_geometry.py [--pairs 64 256] [--workers 16] [--launches 50] [--rounds 9] [--out FILE]

Variants:
  fused_W<n>  geometry_c2_kernel with n kNN worker warps (the library builds --workers' first value)
  fps_only    geometry_c2_kernel without workers: the two FPS chains alone, i.e. the fused kernel's latency floor
  separate    fps_kernel, knn_kernel, centre_proj_f32_kernel, fps_kernel, knn_kernel, centre_proj_f32_kernel
scripts/bench_geometry.cu (geometry.cu plus the entry points) is compiled with nvcc into a temporary directory.  Every
variant's indices and Q rows are first checked bit for bit against `separate`.  Per round every variant runs --launches
back-to-back forwards' geometry bracketed by one pair of CUDA events; variants alternate within a round.  The clouds
(6 MB at 512 clouds) stay in L2 between launches, as they do in the forward.  One JSON line per batch: median and spread
(max - min) over rounds of the ms per launch set, the GPU's name and power limit."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build(tmp):
    so = os.path.join(tmp, "bench_geometry.so")
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    subprocess.check_call([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", os.path.join(ROOT, "scripts", "bench_geometry.cu"), "-o", so, "-lcudart"])
    return ctypes.CDLL(so)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name()


class Problem:
    """Seeded clouds, FPS starts and layer-1 weights of both grouped MLPs (two weight sets) for `pairs` pairs."""

    def __init__(self, pairs, dev):
        g = torch.Generator().manual_seed(1000 + pairs)
        self.B, self.C = pairs, 2 * pairs
        C = self.C
        self.xyz = (torch.rand(C, 1024, 3, generator=g) - 0.5).to(dev)
        self.s1 = torch.randint(0, 1024, (C,), generator=g).to(dev)
        self.s2 = torch.randint(0, 512, (C,), generator=g).to(dev)
        self.w1 = [torch.randn(128, 67, generator=g).to(dev) for _ in range(2)]
        self.w2 = [torch.randn(256, 131, generator=g).to(dev) for _ in range(2)]

    def outputs(self):
        C, dev = self.C, self.xyz.device
        i64, f32, i32 = dict(device=dev, dtype=torch.int64), dict(device=dev, dtype=torch.float32), dict(device=dev, dtype=torch.int32)
        return dict(fps1=torch.full((C, 512), -1, **i64), knn1=torch.full((C, 512, 32), -1, **i64),
                    fps2=torch.full((C, 256), -1, **i64), knn2=torch.full((C, 256, 32), -1, **i64),
                    nx1=torch.zeros(C, 512, 3, **f32), nx2=torch.zeros(C, 256, 3, **f32),
                    knn1r=torch.full((C, 512, 32), -1, **i32), knn2r=torch.full((C, 256, 32), -1, **i32),
                    Q1=torch.zeros(C * 512, 128, **f32), Q2=torch.zeros(C * 256, 256, **f32))

    def args(self, o):
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        return [p(self.xyz), p(self.s1), p(self.s2), self.C, self.B, p(o["fps1"]), p(o["knn1"]), p(o["fps2"]), p(o["knn2"]),
                p(o["nx1"]), p(o["nx2"]), p(o["knn1r"]), p(o["knn2r"]), p(o["Q1"]), p(o["Q2"]), p(self.w1[0]), p(self.w1[1]),
                67, p(self.w2[0]), p(self.w2[1]), 131, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, nargs="+", default=[64, 256])
    ap.add_argument("--workers", type=int, nargs="+", default=[16, 12, 8], choices=[8, 12, 16])
    ap.add_argument("--launches", type=int, default=50, help="forwards' geometry per timed window")
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_geometry.py needs a GPU"
    torch.cuda.set_device(0)
    info = gpu_info()
    with tempfile.TemporaryDirectory() as tmp:
        lib = build(tmp)
        lib.geo_last_error.restype = ctypes.c_char_p

        def check(rc):
            if rc != 0:
                raise RuntimeError(f"geometry launch failed ({rc}): {lib.geo_last_error().decode()}")

        lines = []
        for pairs in a.pairs:
            prob = Problem(pairs, torch.device("cuda", 0))
            variants = {f"fused_W{w}": (lambda o, w=w: lib.geo_fused(w, *prob.args(o))) for w in a.workers}
            variants["fps_only"] = lambda o: lib.geo_fused(0, *prob.args(o))
            variants["separate"] = lambda o: lib.geo_separate(*prob.args(o))
            outs = {k: prob.outputs() for k in variants}
            for k, fn in variants.items():
                check(fn(outs[k]))
            torch.cuda.synchronize()
            ref = outs["separate"]
            for k, o in outs.items():
                names = ("fps1", "fps2", "nx1", "nx2") if k == "fps_only" else tuple(ref)
                bad = [n for n in names if not torch.equal(o[n], ref[n])]
                if bad:
                    raise AssertionError(f"{pairs} pairs: {k} differs from the separate launches in {bad}")
            times = {k: [] for k in variants}
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            for k, fn in variants.items():   # warm-up
                for _ in range(3):
                    check(fn(outs[k]))
            for _ in range(a.rounds):
                for k, fn in variants.items():
                    ev[0].record()
                    for _ in range(a.launches):
                        fn(outs[k])
                    ev[1].record()
                    ev[1].synchronize()
                    times[k].append(ev[0].elapsed_time(ev[1]) / a.launches)
            line = {"metric": "ms per forward's encoder geometry (both stages)", "pairs": pairs, "clouds": prob.C,
                    "launches": a.launches, "rounds": a.rounds, "gpu": info}
            for k, v in times.items():
                line[k] = {"median_ms": round(statistics.median(v), 4), "spread_ms": round(max(v) - min(v), 4)}
            print(json.dumps(line), flush=True)
            lines.append(line)
    if a.out:
        with open(a.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    sys.exit(main())
