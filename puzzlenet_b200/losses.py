"""Loss-side and post-forward operators of the reference model, on the CUDA library.

* :func:`chamfer_loss`     -- ``TouchedRegraster.chamfer_loss`` model5_b.py:1495-1505 (differentiable)
* :func:`comp`             -- ``TouchedRegraster.comp`` model5_b.py:1512-1519 (differentiable)
* :func:`boundary_topk`    -- ``torch.topk(torch.softmax(l, 1)[:, 1, :], 128, 1)[1]`` model5_b.py:1323-1330
* :func:`transform_points` -- ``se3.transform`` (se_math/se3.py:110-120) for ``[B,n,3]`` points
* :func:`pair_score`       -- the whole post-forward part of ``test_step`` (model5_b.py:1314-1358) in one launch

CUDA only, no fallback (``_lib`` raises when the shared library is missing).
"""
from __future__ import annotations

import torch

from . import _lib

SCORE_COLS = _lib.PZ_SCORE_COLS
#: column names of :func:`pair_score`'s result
SCORE_NAMES = ("r_isotropic_deg", "t_isotropic", "t_mse", "t_mae", "fpc_inter", "fpc_union", "mrpc_inter",
               "mrpc_union", "cd_fpc", "cd_rpc", "cd_pair", "reserved")


def _f32(t: torch.Tensor) -> torch.Tensor:
    _lib.require_cuda(t)
    return t.contiguous().float()


def _chamfer_raw(x, y, want_arg):
    B, n, _ = x.shape
    m = y.shape[1]
    d_x = torch.empty(B, m, device=x.device, dtype=torch.float32)
    d_y = torch.empty(B, n, device=x.device, dtype=torch.float32)
    a_x = torch.empty(B, m, device=x.device, dtype=torch.int32) if want_arg else None
    a_y = torch.empty(B, n, device=x.device, dtype=torch.int32) if want_arg else None
    with torch.cuda.device(x.device):
        _lib.call("pz_chamfer", x.data_ptr(), y.data_ptr(), B, n, m, d_x.data_ptr(), d_y.data_ptr(),
                  a_x.data_ptr() if want_arg else None, a_y.data_ptr() if want_arg else None, _lib.stream_ptr())
    return d_x, d_y, a_x, a_y


class _ChamferFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y):
        d_x, d_y, a_x, a_y = _chamfer_raw(x, y, True)
        ctx.save_for_backward(x, y, a_x, a_y)
        return d_x, d_y

    @staticmethod
    def backward(ctx, g_x, g_y):
        x, y, a_x, a_y = ctx.saved_tensors
        B, n, _ = x.shape
        m = y.shape[1]
        gx, gy = torch.empty_like(x), torch.empty_like(y)
        g_x, g_y = g_x.contiguous().float(), g_y.contiguous().float()
        with torch.cuda.device(x.device):
            _lib.call("pz_chamfer_grad", x.data_ptr(), y.data_ptr(), B, n, m, a_x.data_ptr(), a_y.data_ptr(),
                      g_x.data_ptr(), g_y.data_ptr(), gx.data_ptr(), gy.data_ptr(), _lib.stream_ptr())
        return gx, gy


def chamfer_loss(a: torch.Tensor, b: torch.Tensor):
    """model5_b.py:1495-1505.  a [B,n,3], b [B,m,3] -> ``(torch.min(P,1)[0] [B,m], torch.min(P,2)[0] [B,n])`` with
    ``P[i,j] = |a_i|^2 + |b_j|^2 - 2 a_i.b_j`` (the reference only works for n == m because of its ``expand_as``;
    any n, m is accepted here).  The [B,n,m] matrix is never materialised."""
    x, y = _f32(a), _f32(b)
    if x.dim() != 3 or y.dim() != 3 or x.shape[2] != 3 or y.shape[2] != 3 or x.shape[0] != y.shape[0]:
        raise ValueError(f"chamfer_loss expects [B,n,3] and [B,m,3]; got {tuple(a.shape)} and {tuple(b.shape)}")
    if x.requires_grad or y.requires_grad:
        return _ChamferFunction.apply(x, y)
    d_x, d_y, _, _ = _chamfer_raw(x, y, False)
    return d_x, d_y


def _comp_raw(g_, h_):
    loss = torch.empty(1, device=g_.device, dtype=torch.float32)
    with torch.cuda.device(g_.device):
        _lib.call("pz_comp", g_.data_ptr(), h_.data_ptr(), g_.shape[0], loss.data_ptr(), _lib.stream_ptr())
    return loss[0]


class _CompFunction(torch.autograd.Function):
    """gradient w.r.t. g only: igt is the ground truth (the reference's loss never differentiates it)"""

    @staticmethod
    def forward(ctx, g_, h_):
        ctx.save_for_backward(g_, h_)
        return _comp_raw(g_, h_)

    @staticmethod
    def backward(ctx, dloss):
        g_, h_ = ctx.saved_tensors
        dg = torch.empty_like(g_)
        dloss = dloss.contiguous().float()
        with torch.cuda.device(g_.device):
            _lib.call("pz_comp_backward", g_.data_ptr(), h_.data_ptr(), g_.shape[0], dloss.data_ptr(), dg.data_ptr(),
                      _lib.stream_ptr())
        return dg, None


def comp(g: torch.Tensor, igt: torch.Tensor) -> torch.Tensor:
    """model5_b.py:1512-1519: ``mse(g.matmul(igt), I) * 16`` -> 0-d tensor; differentiable w.r.t. ``g`` when it
    requires grad (``pz_comp_backward``)."""
    g_, h_ = _f32(g).view(-1, 4, 4), _f32(igt).view(-1, 4, 4)
    assert g_.shape == h_.shape
    if g_.requires_grad:
        return _CompFunction.apply(g_, h_)
    return _comp_raw(g_, h_)


def boundary_topk(logits: torch.Tensor, k: int = 128, return_prob: bool = False):
    """logits [B,2,N] -> int64 [B,k] indices of the k largest class-1 softmax probabilities, descending."""
    l_ = _f32(logits)
    if l_.dim() != 3 or l_.shape[1] != 2:
        raise ValueError(f"boundary_topk expects [B,2,N]; got {tuple(logits.shape)}")
    B, _, N = l_.shape
    idx = torch.empty(B, k, device=l_.device, dtype=torch.int64)
    prob = torch.empty(B, k, device=l_.device, dtype=torch.float32) if return_prob else None
    with torch.cuda.device(l_.device):
        _lib.call("pz_boundary_topk", l_.data_ptr(), B, N, k, idx.data_ptr(),
                  prob.data_ptr() if return_prob else None, _lib.stream_ptr())
    return (idx, prob) if return_prob else idx


def transform_points(g: torch.Tensor, pts: torch.Tensor) -> torch.Tensor:
    """se3.transform for points stored [B,n,3]: ``(R p + t)``; equals
    ``se3.transform(g, pts.permute(0,2,1)).permute(0,2,1)`` of the reference call sites (model5_b.py:948-949)."""
    g_, p_ = _f32(g).view(-1, 4, 4), _f32(pts)
    out = torch.empty_like(p_)
    with torch.cuda.device(p_.device):
        _lib.call("pz_se3_transform", g_.data_ptr(), p_.data_ptr(), p_.shape[0], p_.shape[1], out.data_ptr(),
                  _lib.stream_ptr())
    return out


def pair_score(out6, de_fpcb, de_mrpcb, fpc, src, fpcb=None, rpcb=None, fpc_idx=None, rpc_idx=None, igt=None,
               return_boundaries: bool = False):
    """One launch for everything ``test_step`` does after ``predict5`` (model5_b.py:1314-1358).

    Returns ``scores [B, SCORE_COLS]`` (columns: :data:`SCORE_NAMES`) and, with ``return_boundaries``,
    ``(scores, idx_f, idx_m, bnd_f, bnd_m)``.  ``src`` is the cloud the second boundary is gathered from before it is
    aligned with ``se3.exp(out6)``: ``rpc`` in ``test_step``, ``mrpc`` when scoring candidate pairs for assembly."""
    out6, de_fpcb, de_mrpcb, fpc, src = (_f32(t) for t in (out6, de_fpcb, de_mrpcb, fpc, src))
    B = out6.shape[0]
    if fpc.shape != (B, 1024, 3) or src.shape != (B, 1024, 3) or de_fpcb.shape != (B, 2, 1024) \
            or de_mrpcb.shape != (B, 2, 1024):
        raise ValueError("pair_score expects out6 [B,6], logits [B,2,1024] and clouds [B,1024,3]")
    opt = [None if t is None else _f32(t) for t in (fpcb, rpcb, fpc_idx, rpc_idx, igt)]
    for t, numel in zip(opt, (B * 384, B * 384, B * 1024, B * 1024, B * 16)):    # fpc_idx may come as [B,1024,1]
        if t is not None and t.numel() != numel:
            raise ValueError(f"pair_score: optional input of shape {tuple(t.shape)} has the wrong size")
    dev = out6.device
    scores = torch.empty(B, SCORE_COLS, device=dev, dtype=torch.float32)
    idx_f = idx_m = bnd_f = bnd_m = None
    if return_boundaries:
        idx_f = torch.empty(B, 128, device=dev, dtype=torch.int64)
        idx_m = torch.empty(B, 128, device=dev, dtype=torch.int64)
        bnd_f = torch.empty(B, 128, 3, device=dev, dtype=torch.float32)
        bnd_m = torch.empty(B, 128, 3, device=dev, dtype=torch.float32)
    p = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    with torch.cuda.device(dev):
        _lib.call("pz_pair_score", out6.data_ptr(), de_fpcb.data_ptr(), de_mrpcb.data_ptr(), fpc.data_ptr(),
                  src.data_ptr(), *(p(t) for t in opt), B, scores.data_ptr(), p(idx_f), p(idx_m), p(bnd_f), p(bnd_m),
                  _lib.stream_ptr())
    if return_boundaries:
        return scores, idx_f, idx_m, bnd_f, bnd_m
    return scores


def topk(values: torch.Tensor, k: int, largest: bool = True):
    """``torch.topk(values, k, 1)`` for [B, N <= 1024] rows -> (vals [B,k], idx [B,k]); ties: lowest index first."""
    v = _f32(values)
    B, N = v.shape
    idx = torch.empty(B, k, device=v.device, dtype=torch.int64)
    vals = torch.empty(B, k, device=v.device, dtype=torch.float32)
    with torch.cuda.device(v.device):
        _lib.call("pz_topk", v.data_ptr(), B, N, k, 1 if largest else 0, idx.data_ptr(), vals.data_ptr(),
                  _lib.stream_ptr())
    return vals, idx
