"""ctypes binding of ``libpuzzlenet_sm100.so`` (C ABI: ``include/puzzlenet_b200.h``).

There is deliberately no fallback: if the shared library is missing or a call
returns non-zero, a ``RuntimeError`` is raised -- the CUDA path is the only
product path (no eager / CPU substitute).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpuzzlenet_sm100.so")

PZ_PREC_FP32 = 0
PZ_PREC_BF16 = 1
PZ_PREC_SPLIT = 2
ABI_VERSION = 7
PZ_SCORE_COLS = 12
PZ_FLAG_NEED = 1
PZ_FLAG_REUSE_PACKS = 2

c_f32p = C.c_void_p   # device pointers travel as integers
c_i64p = C.c_void_p
c_stream = C.c_void_p


class PzEncoderWeights(C.Structure):
    _fields_ = ([(f"{n}_{s}", C.c_void_p) for n in ("mlp1", "mlp2", "mlp3", "mlp4", "mlp5", "mlp6") for s in ("w", "b")]
                + [(f"bn{i}_{s}", C.c_void_p) for i in (1, 2) for s in ("w", "b", "mean", "var")]
                + [(f"{n}_{s}", C.c_void_p * 4) for n in ("q", "k", "v", "o") for s in ("w", "b")]
                + [("out_w", C.c_void_p), ("out_b", C.c_void_p)])


class PzEncoderOutputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("f_global", "x2", "attention", "out", "x_feature", "fps1", "knn1",
                                          "f1f", "fps2", "knn2", "f2f", "att_cat")]


class PzHeadWeights(C.Structure):
    _fields_ = ([("tf_w", C.c_void_p * 5), ("tf_b", C.c_void_p * 5)]
                + [(f"{n}_{s}", C.c_void_p * 3) for n in ("pre_fpc", "pre_rpc", "seg_fpc", "seg_rpc") for s in ("w", "b")])


class PzPieceEmbeddings(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("f_global", "local", "tilemax", "de_mrpcb")]


# name -> (restype, argtypes); mirrors include/puzzlenet_b200.h one to one
SIGNATURES = {
    "pz_abi_version": (C.c_int, []),
    "pz_last_error": (C.c_char_p, []),
    "pz_device_arch": (C.c_int, []),
    "pz_launch_count": (C.c_longlong, []),
    "pz_profile_enable": (C.c_int, [C.c_int]),
    "pz_profile_attention_timeline": (C.c_int, [C.c_void_p, C.c_longlong]),
    "pz_profile_collect": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.c_int]),
    "pz_fps": (C.c_int, [c_f32p, C.c_int, C.c_int, c_i64p, C.c_int, c_i64p, c_f32p, c_stream]),
    "pz_sqdist": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_stream]),
    "pz_knn": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_i64p, c_f32p, c_stream]),
    "pz_ball_query": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, c_i64p, c_stream]),
    "pz_gather": (C.c_int, [C.c_void_p, c_i64p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, c_stream]),
    "pz_group_concat": (C.c_int, [c_f32p, c_f32p, c_f32p, c_i64p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  c_f32p, c_f32p, c_stream]),
    "pz_plane_split": (C.c_int, [c_f32p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, c_f32p, c_f32p, C.c_void_p,
                                 C.c_int, c_stream]),
    "pz_group_mlp_workspace_bytes": (C.c_size_t, [C.c_int] * 7),
    "pz_group_mlp_maxpool": (C.c_int, [c_f32p, c_f32p, c_f32p, c_i64p, c_f32p, c_f32p, c_f32p, c_f32p]
                             + [C.c_int] * 8 + [c_f32p, C.c_void_p, C.c_size_t, c_stream]),
    "pz_linear": (C.c_int, [c_f32p, C.c_int, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, C.c_int, c_f32p,
                            C.c_int, C.c_int, c_stream]),
    "pz_linear_bf16": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p,
                                 C.c_int, c_f32p, C.c_int, c_stream]),
    "pz_offset_attention_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "pz_offset_attention": (C.c_int, [c_f32p] * 9 + [C.c_int] * 4 + [c_f32p, c_f32p, C.c_void_p, C.c_size_t, c_stream]),
    "pz_scaled_dot_attention": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p,
                                          c_stream]),
    "pz_encoder_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "pz_encoder_forward": (C.c_int, [C.POINTER(PzEncoderWeights), C.c_int, C.c_int, c_f32p, c_i64p, c_i64p, C.c_int,
                                     C.POINTER(PzEncoderOutputs), C.c_void_p, C.c_size_t, c_stream]),
    "pz_predict5_workspace_bytes": (C.c_size_t, [C.c_int]),
    "pz_predict5": (C.c_int, [C.POINTER(PzEncoderWeights), C.POINTER(PzHeadWeights), c_f32p, c_f32p, C.c_int, c_i64p,
                              C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p,
                              C.c_size_t, c_stream]),
    "pz_encode_pieces_workspace_bytes": (C.c_size_t, [C.c_int]),
    "pz_encode_pieces": (C.c_int, [C.POINTER(PzEncoderWeights), C.POINTER(PzHeadWeights), c_f32p, C.c_int, c_i64p,
                                   C.c_int, C.c_int, C.POINTER(PzPieceEmbeddings), C.c_void_p, C.c_size_t, c_stream]),
    "pz_predict_pairs_workspace_bytes": (C.c_size_t, [C.c_int]),
    "pz_predict_pairs": (C.c_int, [C.POINTER(PzHeadWeights), C.POINTER(PzPieceEmbeddings), C.c_int, c_i64p, C.c_int,
                                   C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_size_t, c_stream]),
    "pz_se3_exp": (C.c_int, [c_f32p, C.c_int, c_f32p, c_stream]),
    "pz_se3_exp_backward": (C.c_int, [c_f32p, c_f32p, C.c_int, c_f32p, c_stream]),
    "pz_chamfer": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, C.c_void_p, C.c_void_p, c_stream]),
    "pz_chamfer_grad": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, c_f32p, c_f32p,
                                  c_f32p, c_f32p, c_stream]),
    "pz_comp": (C.c_int, [c_f32p, c_f32p, C.c_int, c_f32p, c_stream]),
    "pz_comp_backward": (C.c_int, [c_f32p, c_f32p, C.c_int, c_f32p, c_f32p, c_stream]),
    "pz_se3_transform": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, c_f32p, c_stream]),
    "pz_boundary_topk": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, c_i64p, c_f32p, c_stream]),
    "pz_topk": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_i64p, c_f32p, c_stream]),
    "pz_pair_score": (C.c_int, [c_f32p] * 10 + [C.c_int, c_f32p, c_i64p, c_i64p, c_f32p, c_f32p, c_stream]),
    "pz_sgemm": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, c_f32p, C.c_longlong, c_f32p,
                           C.c_longlong, C.c_float, c_f32p, C.c_longlong, C.c_int, C.c_longlong, C.c_longlong,
                           C.c_longlong, C.c_int, c_f32p, C.c_int, c_f32p, C.c_longlong, c_f32p, C.c_longlong, c_stream]),
    "pz_gemm_tf32": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, C.c_longlong, c_f32p, C.c_longlong,
                               c_f32p, C.c_longlong, C.c_int, c_f32p, C.c_int, c_f32p, C.c_longlong, C.c_int, c_stream]),
    "pz_gemm_tf32_batched": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, C.c_longlong, c_f32p,
                                       C.c_longlong, c_f32p, C.c_longlong, C.c_int, C.c_longlong, C.c_longlong,
                                       C.c_longlong, C.c_int, c_f32p, C.c_int, c_f32p, C.c_longlong, C.c_int, c_stream]),
    "pz_gather_sub_relu": (C.c_int, [c_f32p, c_f32p, c_i64p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p,
                                     c_stream]),
    "pz_group_scatter_grad": (C.c_int, [c_f32p, c_i64p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p,
                                        c_stream]),
    "pz_softmax_forward": (C.c_int, [c_f32p, C.c_longlong, C.c_int, C.c_float, c_f32p, c_stream]),
    "pz_colsum": (C.c_int, [c_f32p, C.c_longlong, C.c_longlong, C.c_int, C.c_float, c_f32p, c_stream]),
    "pz_axpby": (C.c_int, [C.c_longlong, C.c_int, C.c_float, c_f32p, C.c_longlong, C.c_float, c_f32p, C.c_longlong,
                           c_f32p, C.c_longlong, c_stream]),
    "pz_bn_point_train_forward": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, c_f32p,
                                            C.c_float, C.c_float, C.c_int, c_f32p, c_f32p, c_f32p, c_stream]),
    "pz_bn_point_train_backward": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_f32p,
                                             C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, c_stream]),
    "pz_maxpool_forward": (C.c_int, [c_f32p, C.c_longlong, C.c_int, C.c_int, c_f32p, C.c_void_p, c_stream]),
    "pz_maxpool_backward": (C.c_int, [c_f32p, c_f32p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, c_f32p,
                                      c_stream]),
    "pz_scatter_add_rows": (C.c_int, [c_f32p, C.c_longlong, C.c_int, C.c_int, c_i64p, C.c_longlong, C.c_longlong,
                                      C.c_int, c_f32p, C.c_longlong, c_stream]),
    "pz_softmax_backward": (C.c_int, [c_f32p, c_f32p, C.c_longlong, C.c_int, C.c_float, c_f32p, c_stream]),
    "pz_cross_entropy": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_float, c_f32p, c_f32p, c_stream]),
    "pz_bias_act": (C.c_int, [C.c_longlong, C.c_int, c_f32p, C.c_longlong, c_f32p, C.c_int, c_stream]),
    "pz_relu_gate": (C.c_int, [C.c_longlong, C.c_int, c_f32p, C.c_longlong, c_f32p, C.c_longlong, c_f32p, C.c_longlong,
                               c_stream]),
    "pz_broadcast_rows": (C.c_int, [c_f32p, C.c_longlong, C.c_int, C.c_int, c_f32p, C.c_longlong, c_stream]),
    "pz_group_sum": (C.c_int, [c_f32p, C.c_longlong, C.c_longlong, C.c_int, C.c_int, c_f32p, c_stream]),
    "pz_pose_grad": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int, c_f32p, C.c_float, C.c_int, C.c_float, c_f32p,
                               c_stream]),
    "pz_adam_step": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, C.c_longlong, C.c_float, C.c_float, C.c_float,
                               C.c_float, C.c_int, C.c_float, c_stream]),
    "pz_emd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "pz_emd_approxmatch": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, C.c_void_p, C.c_size_t,
                                     c_stream]),
    "pz_emd_matchcost": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_stream]),
    "pz_emd_matchcost_grad": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p,
                                        c_stream]),
}

_lock = threading.Lock()
_lib = None
launch_count = 0   # number of C-ABI compute calls issued by this process (bench.py reports it)


def load():
    """Load the shared library once; raise loudly if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C puzzlenet_b200/csrc`. puzzlenet_b200 has no CPU or eager fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)       # AttributeError here == ABI mismatch, which must be loud
            fn.restype = res
            fn.argtypes = args
        if lib.pz_abi_version() != ABI_VERSION:
            raise RuntimeError(f"libpuzzlenet_sm100.so ABI {lib.pz_abi_version()} != binding {ABI_VERSION}")
        _lib = lib
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().pz_last_error().decode("utf-8", "replace")
        if status < 0 and status in (-1,):
            raise ValueError(f"{what}: {msg}")
        raise RuntimeError(f"{what} failed with status {status}: {msg}")


def call(name: str, *args) -> None:
    """Invoke an int-returning entry point and raise on failure."""
    global launch_count
    launch_count += 1
    check(getattr(load(), name)(*args), name)


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("puzzlenet_b200 only runs on CUDA tensors (no CPU fallback); got a "
                               f"{t.device} tensor")


def profile_collect(max_stages: int = 48):
    """-> (calls, [(stage name, summed ms)]) for the calls recorded since pz_profile_enable(1)."""
    ms = (C.c_double * max_stages)()
    names = (C.c_char_p * max_stages)()
    calls = C.c_int(0)
    n = load().pz_profile_collect(ms, names, C.byref(calls), max_stages)
    if n < 0:
        check(n, "pz_profile_collect")
    return calls.value, [(names[i].decode(), ms[i]) for i in range(n)]
