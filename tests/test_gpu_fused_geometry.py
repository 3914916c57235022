"""GPU: the encoder's geometry runs as one launch per cloud (geometry_c2_kernel).  Its FPS and kNN indices must equal,
bit for bit, those of pz_fps + pz_knn composed by hand, in every precision, at the batch sizes of 1, 2, 64 and 256 pairs,
for start indices at both ends of the range and random ones, and on clouds that force distance ties: one repeated point,
every point duplicated (the kNN's incremental path for more than 64 candidates under its bound) and a lattice."""
import ctypes

import pytest
import torch

from puzzlenet_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _clouds(kind, C, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "random":
        return torch.rand(C, 1024, 3, generator=g) - 0.5
    if kind == "one_point":
        return (torch.rand(C, 1, 3, generator=g) - 0.5).expand(C, 1024, 3).contiguous()
    if kind == "duplicates":   # 128 distinct points, each 8 times, interleaved
        base = torch.rand(C, 128, 3, generator=g) - 0.5
        return base.repeat(1, 8, 1).contiguous()
    if kind == "lattice":      # 8 x 8 x 16 integer grid, shuffled per cloud, some clouds scaled
        ax = [torch.arange(8.0), torch.arange(8.0), torch.arange(16.0)]
        grid = torch.stack(torch.meshgrid(*ax, indexing="ij"), -1).reshape(1024, 3)
        perm = torch.stack([torch.randperm(1024, generator=g) for _ in range(C)])
        scale = torch.where(torch.arange(C) % 2 == 0, 1.0, 0.125).view(C, 1, 1)
        return grid[perm] * scale
    raise ValueError(kind)


def _starts(mode, C, n, seed):
    if mode == "zero":
        return torch.zeros(C, dtype=torch.int64)
    if mode == "last":
        return torch.full((C,), n - 1, dtype=torch.int64)
    return torch.randint(0, n, (C,), generator=torch.Generator().manual_seed(seed))


def _reference(xyz, s1, s2):
    """pz_fps + pz_knn for both stages, launch by launch."""
    C = xyz.shape[0]
    st = _lib.stream_ptr()
    fps1 = torch.empty(C, 512, dtype=torch.int64, device=DEV)
    x1 = torch.empty(C, 512, 3, device=DEV)
    knn1 = torch.empty(C, 512, 32, dtype=torch.int64, device=DEV)
    fps2 = torch.empty(C, 256, dtype=torch.int64, device=DEV)
    x2 = torch.empty(C, 256, 3, device=DEV)
    knn2 = torch.empty(C, 256, 32, dtype=torch.int64, device=DEV)
    _lib.call("pz_fps", xyz.data_ptr(), C, 1024, s1.data_ptr(), 512, fps1.data_ptr(), x1.data_ptr(), st)
    _lib.call("pz_knn", x1.data_ptr(), xyz.data_ptr(), C, 512, 1024, 32, knn1.data_ptr(), None, st)
    _lib.call("pz_fps", x1.data_ptr(), C, 512, s2.data_ptr(), 256, fps2.data_ptr(), x2.data_ptr(), st)
    _lib.call("pz_knn", x2.data_ptr(), x1.data_ptr(), C, 256, 512, 32, knn2.data_ptr(), None, st)
    return dict(fps1=fps1, knn1=knn1, fps2=fps2, knn2=knn2, x2=x2)


def _encoder(model, precision, xyz, s1, s2):
    """pz_encoder_forward with both encoders (E = 2, as pz_predict5 runs them): the geometry's index outputs and x2."""
    from puzzlenet_b200.model5_b import PRECISIONS, _encoder_struct
    C = xyz.shape[0]
    B = C // 2
    res = dict(fps1=torch.full((C, 512), -1, dtype=torch.int64, device=DEV),
               knn1=torch.full((C, 512, 32), -1, dtype=torch.int64, device=DEV),
               fps2=torch.full((C, 256), -1, dtype=torch.int64, device=DEV),
               knn2=torch.full((C, 256, 32), -1, dtype=torch.int64, device=DEV),
               x2=torch.full((C, 256, 3), float("nan"), device=DEV),
               f_global=torch.empty(C, 1024, device=DEV))
    outs = _lib.PzEncoderOutputs()
    for k, v in res.items():
        setattr(outs, k, v.data_ptr())
    w = (_lib.PzEncoderWeights * 2)(_encoder_struct(model.Encoder), _encoder_struct(model.Encoder2))
    lib = _lib.load()
    ws_bytes = lib.pz_encoder_workspace_bytes(2, B)
    ws = torch.empty(ws_bytes, device=DEV, dtype=torch.uint8)
    _lib.call("pz_encoder_forward", w, 2, B, xyz.data_ptr(), s1.data_ptr(), s2.data_ptr(), PRECISIONS[precision],
              ctypes.byref(outs), ws.data_ptr(), ws_bytes, _lib.stream_ptr())
    return res


def _check(model, precision, kind, pairs, start_mode, seed):
    C = 2 * pairs
    xyz = _clouds(kind, C, seed).to(DEV)
    s1 = _starts(start_mode, C, 1024, seed + 1).to(DEV)
    s2 = _starts(start_mode, C, 512, seed + 2).to(DEV)
    ref = _reference(xyz, s1, s2)
    got = _encoder(model, precision, xyz, s1, s2)
    torch.cuda.synchronize()
    for k in ("fps1", "knn1", "fps2", "knn2", "x2"):
        assert torch.equal(got[k], ref[k]), f"{precision} {kind} pairs={pairs} starts={start_mode}: {k} differs"


@pytest.mark.parametrize("precision", ["split", "bf16", "fp32"])
@pytest.mark.parametrize("pairs", [1, 2, 64, 256])
def test_encoder_geometry_matches_separate_kernels(cuda_model, precision, pairs):
    for i, start_mode in enumerate(("zero", "last", "random")):
        _check(cuda_model, precision, "random", pairs, start_mode, seed=100 * pairs + i)


@pytest.mark.parametrize("kind", ["one_point", "duplicates", "lattice"])
@pytest.mark.parametrize("start_mode", ["zero", "last", "random"])
def test_encoder_geometry_ties(cuda_model, kind, start_mode):
    _check(cuda_model, "split", kind, 4, start_mode, seed=7)
