"""Pose exponential map used to turn predict5's twist into R, t (reference: se_math/se3.py:57-80
``exp``, :110-120 ``transform``)."""
from __future__ import annotations

import torch

from . import _lib


def _exp_raw(x_: torch.Tensor) -> torch.Tensor:
    g = torch.empty(x_.shape[0], 4, 4, device=x_.device, dtype=torch.float32)
    with torch.cuda.device(x_.device):
        _lib.call("pz_se3_exp", x_.data_ptr(), x_.shape[0], g.data_ptr(), _lib.stream_ptr())
    return g


class _ExpFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_):
        ctx.save_for_backward(x_)
        return _exp_raw(x_)

    @staticmethod
    def backward(ctx, dg):
        x_, = ctx.saved_tensors
        dx = torch.zeros_like(x_)
        if x_.shape[0]:
            dg = dg.contiguous().float()
            with torch.cuda.device(x_.device):
                _lib.call("pz_se3_exp_backward", x_.data_ptr(), dg.data_ptr(), x_.shape[0], dx.data_ptr(),
                          _lib.stream_ptr())
        return dx


def exp(x: torch.Tensor) -> torch.Tensor:
    """twist [*, 6] (omega first, v last) -> [*, 4, 4] on the GPU (one tiny kernel); differentiable when ``x``
    requires grad (``pz_se3_exp_backward``)."""
    _lib.require_cuda(x)
    x_ = x.reshape(-1, 6).contiguous().float()
    g = _ExpFunction.apply(x_) if x_.requires_grad else _exp_raw(x_)
    return g.view(*x.shape[:-1], 4, 4)


def transform(g: torch.Tensor, a: torch.Tensor) -> torch.Tensor:
    """se3.py:110-120 -- g [*,4,4], a [*,3(,N)]; plain torch (a 3x3 matmul, not worth a kernel)."""
    g_ = g.view(-1, 4, 4)
    R = g_[:, 0:3, 0:3].contiguous().view(*(g.size()[0:-2]), 3, 3)
    p = g_[:, 0:3, 3].contiguous().view(*(g.size()[0:-2]), 3)
    if len(g.size()) == len(a.size()):
        return R.matmul(a) + p.unsqueeze(-1)
    return R.matmul(a.unsqueeze(-1)).squeeze(-1) + p
