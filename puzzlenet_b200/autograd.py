"""Autograd through the train-mode forward (``TouchedRegraster.differentiable = True``).

One ``torch.autograd.Function`` wraps the Trainer's train-mode forward (``Trainer._forward``) and its hand-written
backward below the outputs (``Trainer._backward``), so that any loss built on predict5 / predict6 with torch ops or
the drop-in operators trains the network on the same kernels as ``training_step``.

Inputs of the node: the two clouds and every live parameter (``_Flat.live``; the unused decoders and ``dt`` get no
gradient, as in the reference).  FPS / kNN indices are constants.  State:

* the graph owns its activations: the forward runs on a buffer store of its own (``Trainer._scope``), so later
  forwards, ``training_step`` or ``predict5_train`` on the same Trainer cannot overwrite them; they are released with
  the graph;
* each backward writes into a freshly zeroed flat gradient buffer and returns views of it, never the Trainer's own
  ``flat.grads``.
"""
from __future__ import annotations

import torch

from . import _lib
from .training import NPTS, S2


class _TrainForward(torch.autograd.Function):
    @staticmethod
    def forward(ctx, trainer, pretrain, need, starts, fpc, mrpc, *params):
        ctx.set_materialize_grads(False)
        B = fpc.shape[0]
        store = {}
        with torch.cuda.device(trainer.dev), trainer._scope(store=store):
            fw = trainer._forward(fpc, mrpc, starts, pretrain=pretrain)
            out6, de_f, de_m, x2f, af, x2m, am = trainer._outputs(fw, B, need)
        trainer._invalidate_inference_state()         # the BatchNorm running statistics were updated in place
        ctx.trainer, ctx.fw, ctx.B, ctx.pretrain, ctx.need = trainer, fw, B, pretrain, need
        # saved for autograd's checks: a second backward without retain_graph, or a parameter modified in place
        # between forward and backward, raises as it does for torch's own ops
        ctx.save_for_backward(*params)
        outs = (out6,) if pretrain else (out6, de_f, de_m)
        if need:
            outs += (x2f, af, x2m, am)
            if not (fpc.requires_grad or mrpc.requires_grad):
                ctx.mark_non_differentiable(x2f, x2m)    # x2 depends on the clouds only
        return outs

    @staticmethod
    def backward(ctx, *grads):
        ctx.saved_tensors                  # raises after the graph was freed by an earlier backward
        tr, fw, B = ctx.trainer, ctx.fw, ctx.B
        grads = list(grads)
        dout6 = grads.pop(0)
        dde = (None, None) if ctx.pretrain else (grads.pop(0), grads.pop(0))
        dx2f, daf, dx2m, dam = grads if ctx.need else (None,) * 4
        dev = tr.dev
        R0 = B * NPTS
        dout6 = torch.zeros(B, 6, device=dev) if dout6 is None else dout6.contiguous().float()
        dlf = dlm = None
        if not ctx.pretrain:               # [B,2,1024] -> the point-major [B*1024,2] the seg-head backward reads
            dlf, dlm = (torch.zeros(R0, 2, device=dev) if d is None else d.float().permute(0, 2, 1).reshape(R0, 2)
                        for d in dde)
        dattn = tuple(None if d is None else d.contiguous().float() for d in (daf, dam))
        dx2 = tuple(None if d is None else d.contiguous().float().view(B * S2, 3) for d in (dx2f, dx2m))
        want = ctx.needs_input_grad[4:6]
        dxyz = tuple(torch.zeros(B, NPTS, 3, device=dev) if w else None for w in want)
        flat_grads = torch.zeros(tr.flat.n, device=dev)
        grad_of = tr.flat.views(flat_grads)
        with torch.cuda.device(dev), tr._scope(grad_of=grad_of):
            tr._backward(fw, B, dout6, dlf, dlm, dattn=dattn, dx2=dx2, dxyz=dxyz)
        # predict6 reaches neither Encoder2 nor the boundary heads: no gradient for them, as under torch autograd
        dparams = [grad_of[id(p)] if need and not (ctx.pretrain and not n.startswith(("Encoder.", "tfMLP."))) else None
                   for p, n, need in zip(tr.flat.live, tr.flat.names, ctx.needs_input_grad[6:])]
        return (None, None, None, None, dxyz[0], dxyz[1], *dparams)


def train_forward(trainer, fpc, mrpc, starts, need, pretrain=False):
    """The train-mode forward with an autograd graph -> ``(out6, de_fpcb, de_mrpcb, x2_fpc, attention_fpc, x2_mrpc,
    attention_mrpc)``; ``de_*`` are None for predict6 (``pretrain``: both clouds through ``Encoder``), the last four
    None without ``need``.  ``starts`` int64 [4,B] or None (drawn as predict5 draws them)."""
    _lib.require_cuda(fpc, mrpc)
    fpc, mrpc = fpc.contiguous().float(), mrpc.contiguous().float()
    if fpc.dim() != 3 or fpc.shape[1:] != (NPTS, 3) or mrpc.shape != fpc.shape:
        raise ValueError(f"expected two [B,1024,3] clouds; got {tuple(fpc.shape)} and {tuple(mrpc.shape)}")
    outs = _TrainForward.apply(trainer, pretrain, need, starts, fpc, mrpc, *trainer.flat.live)
    outs = list(outs)
    out6 = outs.pop(0)
    de_f, de_m = (None, None) if pretrain else (outs.pop(0), outs.pop(0))
    x2f, af, x2m, am = outs if need else (None,) * 4
    return out6, de_f, de_m, x2f, af, x2m, am
