"""CPU: the opt-in autograd of the train-mode forward is off by default, and the two backward entry points of the
pose operators reject bad arguments before any CUDA call."""
import ctypes
import types

import pytest

from puzzlenet_b200 import _lib


def test_differentiable_is_opt_in():
    from puzzlenet_b200.model5_b import TouchedRegraster
    model = TouchedRegraster(types.SimpleNamespace(dataset="vase"))
    assert model.differentiable is False
    with pytest.raises(NotImplementedError):           # predict6 has no train-mode forward without the opt-in
        model.predict6([None] * 8, 0, training=True, pretrain=True)


def test_pose_backward_argument_errors():
    lib = _lib.load()
    one = ctypes.c_void_p(16)
    assert lib.pz_se3_exp_backward(None, one, 2, one, None) == -1
    assert b"null" in lib.pz_last_error()
    assert lib.pz_se3_exp_backward(one, one, 2, None, None) == -1
    assert lib.pz_se3_exp_backward(one, one, 0, one, None) == -1
    assert lib.pz_se3_exp_backward(one, one, -3, one, None) == -1
    assert lib.pz_comp_backward(one, one, 2, None, one, None) == -1
    assert lib.pz_comp_backward(None, one, 2, one, one, None) == -1
    assert lib.pz_comp_backward(one, one, 0, one, one, None) == -1
    assert b"B must be" in lib.pz_last_error()
