"""A forward does not depend on what a forward in another precision left in its workspace.

Each precision carves its own scratch layout out of the same workspace, so the buffers of one precision overlap those of
the others.  For every ordered pair (a, b) of distinct precisions, a forward in precision b on a workspace that a
forward in precision a has just used must give bit-for-bit what precision b gives on a freshly zeroed workspace:
predict5 with need=True and matched FPS starts (weight packs rebuilt, never reused), and the encoder alone with every
intermediate output requested."""
import ctypes
import itertools

import pytest
import torch

from puzzlenet_b200 import _lib
from puzzlenet_b200.model5_b import PRECISIONS, _encoder_struct, _Workspace
from puzzlenet_b200.weights import synthetic_pairs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ORDERED_PAIRS = list(itertools.permutations(PRECISIONS, 2))


def _starts(B, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randint(0, n, (B,), generator=g) for n in (1024, 512, 1024, 512)]).to(DEV)


def _predict5(model, precision, fpc, mrpc, starts, ws):
    model.precision = precision
    try:
        return model._launch(fpc, mrpc, starts, True, ws, None, reuse_packs=False)
    finally:
        model.precision = "fp32"


@pytest.mark.parametrize("B", [3, 64])
@pytest.mark.parametrize("first, second", ORDERED_PAIRS)
def test_predict5_independent_of_previous_precision(cuda_model, B, first, second):
    fpc, mrpc = (t.to(DEV) for t in synthetic_pairs(B, seed=5))
    starts = _starts(B, 9)
    nbytes = _lib.load().pz_predict5_workspace_bytes(B)
    fresh = _predict5(cuda_model, second, fpc, mrpc, starts, _Workspace(torch.zeros(nbytes, device=DEV, dtype=torch.uint8)))
    ws = _Workspace(torch.zeros(nbytes, device=DEV, dtype=torch.uint8))
    _predict5(cuda_model, first, fpc, mrpc, starts, ws)
    reused = _predict5(cuda_model, second, fpc, mrpc, starts, ws)
    torch.cuda.synchronize()
    names = ("out6", "de_fpcb", "de_mrpcb", "x2_fpc", "attention_fpc", "x2_mrpc", "attention_mrpc")
    for name, a, b in zip(names, fresh, reused):
        assert torch.equal(a, b), f"{first} -> {second} B={B}: {name} differs from a forward on a fresh workspace"


def _encoder(model, precision, xyz, start1, start2, ws):
    B = xyz.shape[0]
    f32 = dict(device=DEV, dtype=torch.float32)
    i64 = dict(device=DEV, dtype=torch.int64)
    res = dict(f_global=torch.zeros(B, 1024, **f32), x2=torch.zeros(B, 256, 3, **f32),
               attention=torch.zeros(B, 256, 256, **f32), out=torch.zeros(B, 256, 1024, **f32),
               x_feature=torch.zeros(B, 1024, 64, **f32), fps1=torch.zeros(B, 512, **i64),
               knn1=torch.zeros(B, 512, 32, **i64), f1f=torch.zeros(B, 512, 128, **f32), fps2=torch.zeros(B, 256, **i64),
               knn2=torch.zeros(B, 256, 32, **i64), f2f=torch.zeros(B, 256, 256, **f32),
               att_cat=torch.zeros(B, 256, 1280, **f32))
    outs = _lib.PzEncoderOutputs()
    for k, v in res.items():
        setattr(outs, k, v.data_ptr())
    w = _encoder_struct(model.Encoder)
    _lib.call("pz_encoder_forward", ctypes.byref(w), 1, B, xyz.data_ptr(), start1.data_ptr(), start2.data_ptr(),
              PRECISIONS[precision], ctypes.byref(outs), ws.data_ptr(), ws.numel(), _lib.stream_ptr())
    return res


@pytest.mark.parametrize("B", [3, 64])
@pytest.mark.parametrize("first, second", ORDERED_PAIRS)
def test_encoder_independent_of_previous_precision(cuda_model, B, first, second):
    xyz = synthetic_pairs(B, seed=6)[0].to(DEV)
    starts = _starts(B, 10)
    nbytes = _lib.load().pz_encoder_workspace_bytes(1, B)
    fresh = _encoder(cuda_model, second, xyz, starts[0], starts[1], torch.zeros(nbytes, device=DEV, dtype=torch.uint8))
    ws = torch.zeros(nbytes, device=DEV, dtype=torch.uint8)
    _encoder(cuda_model, first, xyz, starts[0], starts[1], ws)
    reused = _encoder(cuda_model, second, xyz, starts[0], starts[1], ws)
    torch.cuda.synchronize()
    for name, a in fresh.items():
        assert torch.equal(a, reused[name]), f"{first} -> {second} B={B}: {name} differs from a forward on a fresh workspace"
