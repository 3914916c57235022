"""Microbenchmark of pz_gemm_tf32 / pz_sgemm on the GEMM shapes of one training step (64 pairs per GPU).
    python scripts/bench_gemm_tf32.py"""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from puzzlenet_b200 import _lib

DEV = "cuda:0"


def timed(fn, iters=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    st = torch.cuda.current_stream().cuda_stream
    rows = []
    R1, R2, T = 64 * 512 * 32, 64 * 256 * 32, 64 * 256
    shapes = [("fwd  mlp4  [1.05M,128]x[128,128]", 0, 0, R1, 128, 128, 1),
              ("dgrad mlp4", 0, 1, R1, 128, 128, 1),
              ("wgrad mlp4 (K = 1.05M rows)", 1, 1, 128, 128, R1, 296),
              ("fwd  mlp6  [0.52M,256]x[256,256]", 0, 0, R2, 256, 256, 1),
              ("dgrad mlp6", 0, 1, R2, 256, 256, 1),
              ("wgrad mlp6 (K = 0.52M rows)", 1, 1, 256, 256, R2, 296),
              ("fwd  tail  [16384,1280]x[1024,1280]", 0, 0, T, 1024, 1280, 1),
              ("fwd  v/out [16384,256]x[256,256]", 0, 0, T, 256, 256, 1)]
    for name, a_mn, b_mn, M, N, K, sk in shapes:
        A = torch.randn((K, M) if a_mn else (M, K), device=DEV)
        B = torch.randn((K, N) if b_mn else (N, K), device=DEV)
        C = torch.zeros(M, N, device=DEV)
        f = lambda: _lib.call("pz_gemm_tf32", a_mn, b_mn, M, N, K, A.data_ptr(), A.shape[1], B.data_ptr(), B.shape[1],
                              C.data_ptr(), N, sk, None, 0, None, 0, 0, st)
        ms = timed(f)
        gb = 4 * (A.numel() + B.numel() + C.numel()) / 1e9
        g = lambda: _lib.call("pz_sgemm", a_mn, b_mn, M, N, K, 1.0, A.data_ptr(), A.shape[1], B.data_ptr(), B.shape[1], 0.0,
                              C.data_ptr(), N, 1, 0, 0, 0, 1 if sk == 1 else 64, None, 0, None, 0, None, 0, st)
        ms32 = timed(g, 3)
        rows.append({"gemm": name, "tf32_ms": round(ms, 4), "tf32_tflops": round(2.0 * M * N * K / ms / 1e9, 1),
                     "compulsory_GBps": round(gb / ms * 1e3, 1), "sgemm_fp32_ms": round(ms32, 4)})
        del A, B, C
    print(json.dumps({"rows": rows}, indent=1))


if __name__ == "__main__":
    main()
