"""CPU: sizes outside what the C ABI supports are rejected with PZ_ERR_UNSUPPORTED before any CUDA call, and the
largest supported sizes get past those checks (they stop at the empty workspace, PZ_ERR_WORKSPACE, also before any
CUDA call).  Dummy non-null pointers stand in for the device buffers: no check that passes may dereference them, so
this runs without a GPU."""
import ctypes

import pytest

from puzzlenet_b200 import _lib

PZ_ERR_UNSUPPORTED = -2
PZ_ERR_WORKSPACE = -3
INT_MAX = 2**31 - 1
MAX_CLOUDS = 65535                 # PZ_MAX_CLOUDS
DUMMY = ctypes.c_void_p(16)        # non-null and 16-byte aligned; never dereferenced
PRECISIONS = (_lib.PZ_PREC_FP32, _lib.PZ_PREC_BF16, _lib.PZ_PREC_SPLIT)


def _dummy_struct(cls):
    """a host weight struct whose every pointer is DUMMY (the null-pointer checks read these, nothing else does)"""
    s = cls()
    for name, typ in cls._fields_:
        if hasattr(typ, "_length_"):
            arr = getattr(s, name)
            for i in range(typ._length_):
                arr[i] = DUMMY.value
        else:
            setattr(s, name, DUMMY.value)
    return s


def _group_mlp(lib, B, N, S, precision, D=64, C1=128, C2=128):
    return lib.pz_group_mlp_maxpool(*([DUMMY] * 8), B, N, D, S, 32, C1, C2, precision, DUMMY, DUMMY, 0, None)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_group_mlp_maxpool_rejects_int32_overflow(precision):
    lib = _lib.load()
    # B*S*K = 4096 * 16384 * 32 = 2^31 grouped rows: one past INT_MAX
    assert _group_mlp(lib, 4096, 1024, 16384, precision) == PZ_ERR_UNSUPPORTED
    assert b"B*S*K = 2147483648" in lib.pz_last_error()
    # B*N = 65536 * 32768 = 2^31 source points (B*S*K = 8 M is fine)
    assert _group_mlp(lib, 65536, 32768, 4, precision) == PZ_ERR_UNSUPPORTED
    assert b"B*N = 2147483648" in lib.pz_last_error()
    # B*S*K = 2^31 - 256 (a multiple of 256, as the tensor-core paths need) is inside the range
    assert _group_mlp(lib, 1, 1024, (2**31 - 256) // 32, precision) == PZ_ERR_WORKSPACE
    assert _group_mlp(lib, 1, INT_MAX - 127, 8, precision) == PZ_ERR_WORKSPACE   # B*N = INT_MAX - 127


def test_predict5_batch_limit():
    lib = _lib.load()
    enc = (_lib.PzEncoderWeights * 2)(_dummy_struct(_lib.PzEncoderWeights), _dummy_struct(_lib.PzEncoderWeights))
    heads = _dummy_struct(_lib.PzHeadWeights)

    def predict5(B, precision):
        return lib.pz_predict5(enc, ctypes.byref(heads), DUMMY, DUMMY, B, DUMMY, precision, 0, DUMMY, DUMMY, DUMMY,
                               None, None, None, None, DUMMY, 0, None)

    for precision in PRECISIONS:
        assert predict5(MAX_CLOUDS // 2 + 1, precision) == PZ_ERR_UNSUPPORTED
        assert b"B = 32768 > 32767" in lib.pz_last_error()
        assert predict5(INT_MAX, precision) == PZ_ERR_UNSUPPORTED
        assert predict5(MAX_CLOUDS // 2, precision) == PZ_ERR_WORKSPACE


def test_encoder_forward_cloud_limit():
    lib = _lib.load()
    enc = (_lib.PzEncoderWeights * 2)(_dummy_struct(_lib.PzEncoderWeights), _dummy_struct(_lib.PzEncoderWeights))
    outs = _lib.PzEncoderOutputs()

    def forward(E, B, precision):
        return lib.pz_encoder_forward(enc, E, B, DUMMY, DUMMY, DUMMY, precision, ctypes.byref(outs), DUMMY, 0, None)

    for precision in PRECISIONS:
        assert forward(1, MAX_CLOUDS + 1, precision) == PZ_ERR_UNSUPPORTED
        assert b"65536 clouds > 65535" in lib.pz_last_error()
        assert forward(2, MAX_CLOUDS // 2 + 1, precision) == PZ_ERR_UNSUPPORTED
        assert forward(2, INT_MAX, precision) == PZ_ERR_UNSUPPORTED      # E*B is not formed in 32 bits
        assert forward(1, MAX_CLOUDS, precision) == PZ_ERR_WORKSPACE
        assert forward(2, MAX_CLOUDS // 2, precision) == PZ_ERR_WORKSPACE
