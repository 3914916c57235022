"""CPU: pair scoring from per-piece encodings -- argument errors of pz_encode_pieces / pz_predict_pairs (decided before
any CUDA call), the Python layer's index and staleness checks, and the FPS-start draws of encode_pieces."""
import ctypes
import types

import pytest
import torch

from puzzlenet_b200 import _lib
from puzzlenet_b200 import model5_b
from puzzlenet_b200.model5_b import PieceEmbeddings, TouchedRegraster


def test_argument_errors_without_gpu():
    lib = _lib.load()
    one = ctypes.c_void_p(16)
    emb = _lib.PzPieceEmbeddings(16, 16, 16, 16)
    null_emb = _lib.PzPieceEmbeddings(16, 16, None, 16)
    enc = (_lib.PzEncoderWeights * 2)()
    heads = _lib.PzHeadWeights()
    # pz_encode_pieces: null pointers (also inside the embeddings), P < 1
    assert lib.pz_encode_pieces(None, None, None, 4, None, 0, 0, None, None, 0, None) == -1
    assert b"null" in lib.pz_last_error()
    assert lib.pz_encode_pieces(enc, ctypes.byref(heads), one, 4, one, 0, 0, ctypes.byref(null_emb), one, 1 << 30,
                                None) == -1
    assert lib.pz_encode_pieces(enc, ctypes.byref(heads), one, 0, one, 0, 0, ctypes.byref(emb), one, 1 << 30, None) == -1
    assert b"P must be" in lib.pz_last_error()
    # pz_predict_pairs: n == 0 is a no-op, then null pointers, P < 1
    assert lib.pz_predict_pairs(None, None, 4, None, 0, 0, 0, None, None, None, None, 0, None) == 0
    assert lib.pz_predict_pairs(None, None, 4, None, 3, 0, 0, None, None, None, None, 0, None) == -1
    assert lib.pz_predict_pairs(ctypes.byref(heads), ctypes.byref(null_emb), 4, one, 3, 0, 0, one, one, one, one,
                                1 << 30, None) == -1
    assert lib.pz_predict_pairs(ctypes.byref(heads), ctypes.byref(emb), 0, one, 3, 0, 0, one, one, one, one, 1 << 30,
                                None) == -1
    assert lib.pz_predict_pairs(ctypes.byref(heads), ctypes.byref(emb), 4, one, -1, 0, 0, one, one, one, one, 1 << 30,
                                None) == -1
    # every embedding buffer (and the copied de_mrpcb output) is accessed with 16-byte vectors
    odd = ctypes.c_void_p(20)
    for bad in (_lib.PzPieceEmbeddings(16, 20, 16, 16), _lib.PzPieceEmbeddings(16, 16, 20, 16)):
        assert lib.pz_encode_pieces(enc, ctypes.byref(heads), one, 4, one, 0, 0, ctypes.byref(bad), one, 1 << 30,
                                    None) == -1
        assert b"aligned" in lib.pz_last_error()
    full = _lib.PzHeadWeights()                                            # non-null heads: the checks get that far
    for name, _ in full._fields_:
        arr = getattr(full, name)
        for k in range(len(arr)):
            arr[k] = 16
    assert lib.pz_predict_pairs(ctypes.byref(full), ctypes.byref(emb), 4, one, 3, 0, 0, one, one, odd, one, 1 << 30,
                                None) == -1
    assert b"aligned" in lib.pz_last_error()
    # size limits: P per encode call (grid height of the fp32 tile-max pass), n per pair call (int point counts)
    assert lib.pz_encode_pieces(enc, ctypes.byref(heads), one, 4096, one, 0, 0, ctypes.byref(emb), one, 1 << 30,
                                None) == -2
    assert lib.pz_predict_pairs(ctypes.byref(heads), ctypes.byref(emb), 4, one, (1 << 20) + 1, 0, 0, one, one, one, one,
                                1 << 30, None) == -2


def test_workspace_sizes_grow():
    lib = _lib.load()
    assert lib.pz_encode_pieces_workspace_bytes(0) == 0 and lib.pz_predict_pairs_workspace_bytes(0) == 0
    enc = [lib.pz_encode_pieces_workspace_bytes(p) for p in (1, 5, 32, 64)]
    pairs = [lib.pz_predict_pairs_workspace_bytes(n) for n in (1, 45, 496, 4096)]
    assert 0 < enc[0] < enc[1] < enc[2] < enc[3]
    assert 0 < pairs[0] < pairs[1] < pairs[2] < pairs[3]
    # encoding P pieces needs predict5's scratch for B = P (both encoders over [clouds; clouds]) and a little more
    assert enc[2] > lib.pz_predict5_workspace_bytes(32)


@pytest.fixture(scope="module")
def cpu_model(state_dict):
    m = TouchedRegraster(types.SimpleNamespace(dataset="vase"))
    m.load_state_dict(state_dict, strict=True)
    return m.eval()


def _cpu_embeddings(model, P):
    return PieceEmbeddings(P, "cpu", torch.zeros(4, P, dtype=torch.int64), model.precision, model._weights_key())


def test_predict_pairs_rejects_bad_indices(cpu_model):
    emb = _cpu_embeddings(cpu_model, 5)
    for bad in ([[0, 5]], [[-1, 2]], [[1, 2], [7, 0]]):
        with pytest.raises(IndexError):
            cpu_model.predict_pairs(emb, torch.tensor(bad))
    with pytest.raises(ValueError):
        cpu_model.predict_pairs(emb, torch.tensor([0, 1]))                # not [n,2]
    with pytest.raises(IndexError):
        emb.reencode(cpu_model, [5], torch.zeros(1, 1024, 3))
    out6, _, de_f, de_m = cpu_model.predict_pairs(emb, torch.zeros(0, 2, dtype=torch.int64))   # n == 0: no launch
    assert out6.shape == (0, 6) and de_f.shape == (0, 2, 1024) and de_m.shape == (0, 2, 1024)


def test_predict_pairs_rejects_stale_embeddings(cpu_model):
    emb = _cpu_embeddings(cpu_model, 3)
    pairs = torch.tensor([[0, 1]])
    cpu_model.precision = "split"
    try:
        with pytest.raises(ValueError, match="stale"):
            cpu_model.predict_pairs(emb, pairs)
    finally:
        cpu_model.precision = "fp32"
    with torch.no_grad():
        cpu_model.MLPFpcb[0].bias.add_(0.0)                                # an in-place write bumps the version
    with pytest.raises(ValueError, match="stale"):
        cpu_model.predict_pairs(emb, pairs)
    with pytest.raises(ValueError, match="stale"):
        emb.reencode(cpu_model, [0], torch.zeros(1, 1024, 3))


def test_weights_written_behind_torch_make_embeddings_stale(cpu_model):
    """the Trainer's Adam step and parameter broadcasts write through raw pointers (no _version bump); they report it
    through _invalidate_inference_state, after which older embeddings are rejected"""
    from puzzlenet_b200.training import Trainer
    emb = _cpu_embeddings(cpu_model, 3)
    assert emb.is_current(cpu_model)
    Trainer._invalidate_inference_state(types.SimpleNamespace(model=cpu_model))
    assert not emb.is_current(cpu_model)
    with pytest.raises(ValueError, match="stale"):
        cpu_model.predict_pairs(emb, torch.tensor([[0, 1]]))
    assert _cpu_embeddings(cpu_model, 3).is_current(cpu_model)


def test_encode_pieces_draws_like_predict5(cpu_model, monkeypatch):
    """encode_pieces(c) takes exactly predict5(make_batch(c, c), P)'s four FPS-start draws from the CPU generator:
    same values, same order, and the generator ends in the same state."""
    from puzzlenet_b200.weights import make_batch
    P = 7
    clouds = torch.rand(P, 1024, 3)
    seen = {}
    monkeypatch.setattr(_lib, "require_cuda", lambda *t: None)            # no device is touched below
    monkeypatch.setattr(PieceEmbeddings, "_encode", lambda self, model, c, starts, rows: None)

    def fake_launch(self, fpc, mrpc, starts, need, ws, outs, reuse_packs=None, shared=False):
        seen["starts"] = starts.clone()
        z = torch.zeros(fpc.shape[0], 6)
        return z, z, z, None, None, None, None

    monkeypatch.setattr(TouchedRegraster, "_launch", fake_launch)
    torch.manual_seed(77)
    cpu_model.predict5(make_batch(clouds, clouds), P)
    after_predict5 = torch.rand(4)
    torch.manual_seed(77)
    emb = cpu_model.encode_pieces(clouds)
    after_encode = torch.rand(4)
    assert torch.equal(emb.starts, seen["starts"])
    assert torch.equal(after_encode, after_predict5)
    assert emb.starts[[0, 2]].max() < 1024 and emb.starts[[1, 3]].max() < 512
    assert emb.f_global.shape == (2, P, 1024) and emb.local.shape == (2, P, 1024, 64)
    assert emb.tilemax.shape == (2, P, 8, 64) and emb.de_mrpcb.shape == (P, 2, 1024)
    assert model5_b.ENCODE_CHUNK == 64
