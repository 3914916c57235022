"""GPU: the forward at the batch limits the C ABI promises (include/puzzlenet_b200.h) -- ``pz_encode_pieces`` with
``PZ_MAX_PIECES`` pieces, ``pz_predict_pairs`` with ``PZ_MAX_PAIRS`` pairs and ``pz_predict5`` on either side of
B = 256, where the fp32 stage-1 gather GEMM first has more than 65535 row tiles (the limit of a grid's y dimension,
which once held them) -- each issued as ONE C call.

Every cloud and every pair is computed independently of the others, so sampled rows of a large call must equal, bit for
bit, the same rows computed by a small call (the sizes the rest of the suite ties to predict5 and the CPU oracle); two
rows per case are also checked against the CPU oracle directly.  The sampled rows include the first and last ones and,
at the encode limit, the pieces on either side of the first 2^31-element offset into the [clouds*256, 1280] attention
concat (Encoder2 clouds 6553 / 6554 = pieces 2458 / 2459).

The calls need up to ~70 GB of device memory: each case checks what is free first, and the module keeps a model of its
own so that its workspaces are released after every case."""
import gc
import types

import pytest
import torch

from oracle import parity
from puzzlenet_b200 import _lib, model5_b
from puzzlenet_b200.weights import make_batch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PRECISIONS = ["fp32", "bf16", "split"]
MAX_PIECES = 4095           # PZ_MAX_PIECES
MAX_PAIRS = 1 << 20         # PZ_MAX_PAIRS
GB = float(1 << 30)
F32 = 4


@pytest.fixture(scope="module")
def big_model(state_dict):
    from puzzlenet_b200.model5_b import TouchedRegraster
    m = TouchedRegraster(types.SimpleNamespace(dataset="vase"))
    m.load_state_dict(state_dict, strict=True)
    m.to(DEV).eval()
    yield m
    m._ws.clear()
    del m
    gc.collect()
    torch.cuda.empty_cache()


@pytest.fixture
def model(big_model):
    yield big_model
    big_model.precision = "fp32"
    big_model._ws.clear()         # the workspaces of one case are up to 49 GB: release them before the next
    gc.collect()
    torch.cuda.empty_cache()


def _require_free(nbytes, what):
    free, total = torch.cuda.mem_get_info()
    if free < nbytes * 1.05:
        pytest.skip(f"{what} needs {nbytes / GB:.1f} GB of device memory; {free / GB:.1f} GB of {total / GB:.1f} GB "
                    f"are free")


def _clouds(P, seed):
    return torch.rand(P, 1024, 3, generator=torch.Generator().manual_seed(seed)).to(DEV) - 0.5


def _starts(P, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randint(0, hi, (P,), generator=g) for hi in (1024, 512, 1024, 512)])


def _sample(fixed, n, count, seed):
    """the fixed rows inside [0, n) plus up to ``count`` other seeded random rows, sorted"""
    rows = {r for r in fixed if 0 <= r < n}
    want = len(rows) + count
    for r in torch.randperm(n, generator=torch.Generator().manual_seed(seed)).tolist():
        if len(rows) >= want:
            break
        rows.add(r)
    return sorted(rows)


def _calls(fn):
    """(result, number of C-ABI compute calls fn issued)"""
    n0 = _lib.launch_count
    r = fn()
    return r, _lib.launch_count - n0


def _assert_rows_equal(got, ref, what):
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    if not torch.equal(got, ref):
        bad = (got != ref).reshape(got.shape[0], -1).any(1).nonzero().flatten().tolist()
        raise AssertionError(f"{what}: sampled rows {bad} differ, max |diff| {(got - ref).abs().max().item():.3e}")


def _assert_oracle(state_dict, clouds, starts, pairs, got, precision):
    """got = (out6, de_fpcb, de_mrpcb) of ``pairs [k,2]`` (fpc piece, mrpc piece) against the CPU oracle's predict5"""
    I, J = pairs[:, 0], pairs[:, 1]
    c = clouds.cpu()
    st = torch.stack([starts[0, I], starts[1, I], starts[2, J], starts[3, J]])
    p = parity.predict5_parity(state_dict, c[I], c[J], st, *got)
    assert parity.within(p, precision), p


# ------------------------------------------------------------------------------------------- a. encode at the limit
@pytest.mark.parametrize("precision", PRECISIONS)
def test_encode_pieces_at_max_pieces(model, state_dict, precision, monkeypatch):
    lib = _lib.load()
    P = MAX_PIECES
    emb_bytes = 2 * P * (1024 + 1024 * 64 + 8 * 64) * F32 + P * 2 * 1024 * F32
    _require_free(lib.pz_encode_pieces_workspace_bytes(P) + emb_bytes + P * 1024 * 3 * F32, f"pz_encode_pieces(P={P})")
    monkeypatch.setattr(model5_b, "ENCODE_CHUNK", P)
    model.precision = precision
    clouds, starts = _clouds(P, 101), _starts(P, 102)
    big, calls = _calls(lambda: model.encode_pieces(clouds, starts=starts))
    assert calls == 1
    torch.cuda.synchronize()

    rows = _sample([0, 1, 2047, 2458, 2459, P - 2, P - 1], P, 8, 103)
    small = model.encode_pieces(clouds[rows], starts=starts[:, rows])
    idx = torch.tensor(rows, device=DEV)
    for name in ("f_global", "local", "tilemax"):
        for role in (0, 1):
            _assert_rows_equal(getattr(big, name)[role, idx], getattr(small, name)[role], f"{name}[{role}]")
    _assert_rows_equal(big.de_mrpcb[idx], small.de_mrpcb, "de_mrpcb")

    # both roles of two pieces past the 2^31-element offset, pinned to the oracle through their diagonal pairs
    diag = torch.tensor([[2459, 2459], [P - 1, P - 1]])
    out6, _, de_f, de_m = model.predict_pairs(big, diag)
    _assert_oracle(state_dict, clouds, starts, diag, (out6, de_f, de_m), precision)


# ------------------------------------------------------------------------------------------- b. pairs at the limit
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("n", [1, 4097, MAX_PAIRS])
def test_predict_pairs_up_to_max_pairs(model, state_dict, precision, n, monkeypatch):
    lib = _lib.load()
    P = 64
    _require_free(lib.pz_predict_pairs_workspace_bytes(n) + n * (6 + 2 * 2 * 1024) * F32 + n * 2 * 8
                  + lib.pz_encode_pieces_workspace_bytes(P), f"pz_predict_pairs(n={n})")
    monkeypatch.setattr(model5_b, "PAIR_CHUNK", MAX_PAIRS)
    model.precision = precision
    clouds, starts = _clouds(P, 201), _starts(P, 202)
    emb = model.encode_pieces(clouds, starts=starts)
    pairs = torch.randint(0, P, (n, 2), generator=torch.Generator().manual_seed(203 + n))
    (out6, _, de_f, de_m), calls = _calls(lambda: model.predict_pairs(emb, pairs))
    assert calls == 1
    torch.cuda.synchronize()

    rows = _sample([0, n // 2, n - 2, n - 1], n, 64, 204)
    ref = model.predict_pairs(emb, pairs[rows])
    idx = torch.tensor(rows, device=DEV)
    for got, r, name in ((out6, ref[0], "out6"), (de_f, ref[2], "de_fpcb"), (de_m, ref[3], "de_mrpcb")):
        _assert_rows_equal(got[idx], r, name)

    check = sorted({n // 2, n - 1})
    ci = torch.tensor(check, device=DEV)
    _assert_oracle(state_dict, clouds, starts, pairs[check], (out6[ci], de_f[ci], de_m[ci]), precision)


# ------------------------------------------------------------------------ c. predict5 at the fp32 gather-grid edge
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("B", [255, 256])
def test_predict5_either_side_of_b256(model, state_dict, precision, B):
    lib = _lib.load()
    _require_free(lib.pz_predict5_workspace_bytes(B) + B * (6 + 4 * 1024 + 2 * 1024 * 3) * F32, f"pz_predict5(B={B})")
    model.precision = precision
    g = torch.Generator().manual_seed(300 + B)
    fpc, mrpc = torch.rand(B, 1024, 3, generator=g) - 0.5, torch.rand(B, 1024, 3, generator=g) - 0.5
    starts = _starts(B, 301 + B)
    (out6, _, de_f, de_m), calls = _calls(lambda: model.predict5(make_batch(fpc.to(DEV), mrpc.to(DEV)), B,
                                                                  starts=starts))
    assert calls == 1

    rows = _sample([0, 1, B - 2, B - 1], B, 12, 302)
    ref = model.predict5(make_batch(fpc[rows].to(DEV), mrpc[rows].to(DEV)), len(rows),
                         starts=starts[:, rows].contiguous())
    idx = torch.tensor(rows, device=DEV)
    for got, r, name in ((out6, ref[0], "out6"), (de_f, ref[2], "de_fpcb"), (de_m, ref[3], "de_mrpcb")):
        _assert_rows_equal(got[idx], r, name)

    p = parity.predict5_parity(state_dict, fpc, mrpc, starts, out6, de_f, de_m, pairs=[rows[4], B - 1])
    assert parity.within(p, precision), p
