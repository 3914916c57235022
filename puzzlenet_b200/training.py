"""Training step of the reference model on the CUDA library (SURVEY.md §8 row A15, BASELINE config 4).

``TouchedRegraster.training_step`` (model5_b.py:912-1155, the non-pretrain branch) gets its backward pass from
torch autograd; here the graph is sequenced explicitly over hand-written kernels (``csrc/train.cu``, ``losses.cu``,
``emd.cu``, ``geometry.cu``): a train-mode forward that keeps the activations it needs (batch-statistics BatchNorm
over the point index, model5_b.py:424-425), the loss terms, the backward pass into ONE flat gradient buffer, one
NCCL all-reduce of that buffer under ``torch.distributed`` (7.27 M live parameters, SURVEY.md Appendix C) and one
fused Adam launch (model5_b.py:1453-1457).  fp32 throughout, like the reference (no AMP).

``Trainer(model, config).training_step(batch)`` returns the same dictionary of logged terms as the reference logs.
torch is used for memory, streams and the collective only -- no autograd, no torch math on the step.
"""
from __future__ import annotations

import contextlib
import math
from typing import Dict, Optional

import torch
import torch.distributed as dist

from . import _lib, losses

NPTS, S1, S2, KNN = 1024, 512, 256, 32


def _p(t):
    return None if t is None else t.data_ptr()


def _st():
    return _lib.stream_ptr()


# ------------------------------------------------------------------------------------------------ kernel wrappers
def gemm(A, B, C, M, N, K, ta=False, tb=False, lda=None, ldb=None, ldc=None, alpha=1.0, beta=0.0, batch=1,
         sa=0, sb=0, sc=0, splitk=1, bias=None, relu=False, mask=None, ldmask=0, residual=None, ldres=0):
    _lib.call("pz_sgemm", int(ta), int(tb), M, N, K, alpha, _p(A), lda, _p(B), ldb, beta, _p(C), ldc, batch, sa, sb, sc,
              splitk, _p(bias), int(relu), _p(mask), ldmask, _p(residual), ldres, _st())


def _splitk(rows: int, out_tiles: int) -> int:
    """split the reduction (row) dimension of a weight-gradient GEMM so that about 4 waves of 148 CTAs run"""
    want = max(1, (4 * 148) // max(out_tiles, 1))
    return max(1, min(want, rows // 256 if rows >= 512 else 1))


def _al16(*ts):
    return all(t is None or t.data_ptr() % 16 == 0 for t in ts)


def _gemm_tf32(a_mn, b_mn, M, N, K, A, lda, B, ldb, C, ldc, splitk=1, bias=None, relu=False, mask=None, ldmask=0,
               accumulate=False):
    _lib.call("pz_gemm_tf32", int(a_mn), int(b_mn), M, N, K, _p(A), lda, _p(B), ldb, _p(C), ldc, splitk, _p(bias),
              int(relu), _p(mask), ldmask, int(accumulate), _st())


def bgemm_tf32(a_mn, b_mn, M, N, K, A, lda, B, ldb, C, ldc, batch, sa, sb, sc):
    """per-cloud products of the attention layers on the tensor cores (TF32)"""
    _lib.call("pz_gemm_tf32_batched", int(a_mn), int(b_mn), M, N, K, _p(A), lda, _p(B), ldb, _p(C), ldc, batch, sa, sb, sc,
              1, None, 0, None, 0, 0, _st())


def linear_fwd(x, ldx, M, lin, out, ldo, relu=False, W=None, K=None, tf32=False):
    """out[M, N] = act(x[M, K] W^T + b).  ``W``/``K`` override the weight with a zero-padded copy (row stride K);
    ``tf32`` routes shapes the tensor-core kernel supports to ``pz_gemm_tf32``."""
    N, K0 = lin.weight.shape
    W = lin.weight if W is None else W
    K = K0 if K is None else K
    if tf32 and M % 128 == 0 and N % 64 == 0 and K % 32 == 0 and ldx % 4 == 0 and ldo % 4 == 0 \
            and _al16(x, W, out, lin.bias):
        _gemm_tf32(0, 0, M, N, K, x, ldx, W, K, out, ldo, bias=lin.bias, relu=relu)
    elif M <= 128 and K >= 512 and ldo == N:
        # skinny layer (the pose MLP: M = batch size): one 128-row tile per 128 columns would leave the GPU idle for a
        # 2048-deep reduction -> split K over the grid into a zeroed output, then bias + ReLU in place
        out.zero_()
        gemm(x, W, out, M, N, K, tb=True, lda=ldx, ldb=K, ldc=ldo, splitk=max(2, min(K // 64, 296 // max(1, (N + 127) // 128))))
        _lib.call("pz_bias_act", M, N, _p(out), ldo, _p(lin.bias), int(relu), _st())
    else:
        gemm(x, W, out, M, N, K, tb=True, lda=ldx, ldb=K, ldc=ldo, bias=lin.bias, relu=relu)


def linear_bwd(dy, lddy, x, ldx, M, lin, gw, gb, dx=None, lddx=0, mask=None, ldmask=0, beta=0.0, W=None, K=None,
               tf32=False, bias_grad=True):
    """dW += dy^T x, db += colsum(dy); dx = (beta*dx +) dy W, gated by (mask > 0) when given.  ``W``/``K``: as in
    linear_fwd (``gw`` then has row stride K as well)."""
    N, K0 = lin.weight.shape
    W = lin.weight if W is None else W
    K = K0 if K is None else K
    if tf32 and N % 128 == 0 and K % 64 == 0 and M % 32 == 0 and M >= 4096 and lddy % 4 == 0 and ldx % 4 == 0 \
            and _al16(dy, x, gw):
        tiles = (N // 128) * (K // (256 if K % 256 == 0 else 128 if K % 128 == 0 else 64))
        kblocks = M // 32
        sk = max(2, min(max(kblocks // 8, 1), -(-2 * 148 // tiles)))
        _gemm_tf32(1, 1, N, K, M, dy, lddy, x, ldx, gw, K, splitk=sk)
    else:
        tiles = ((N + 127) // 128) * ((K + 127) // 128)
        sk = _splitk(M, tiles)
        if sk > 1:          # partial sums are atomically added into the (pre-zeroed) flat gradient buffer
            gemm(dy, x, gw, N, K, M, ta=True, lda=lddy, ldb=ldx, ldc=K, splitk=sk)
        else:
            gemm(dy, x, gw, N, K, M, ta=True, lda=lddy, ldb=ldx, ldc=K, beta=1.0)
    if bias_grad:
        _lib.call("pz_colsum", _p(dy), lddy, M, N, 1.0, _p(gb), _st())
    if dx is not None:
        if tf32 and M % 128 == 0 and K % 64 == 0 and N % 32 == 0 and lddy % 4 == 0 and lddx % 4 == 0 \
                and beta in (0.0, 1.0) and _al16(dy, W, dx, mask) and (mask is None or ldmask % 4 == 0):
            _gemm_tf32(0, 1, M, K, N, dy, lddy, W, K, dx, lddx, mask=mask, ldmask=ldmask, accumulate=beta == 1.0)
        elif M <= 128 and N >= 256 and beta == 0.0 and lddx == K:
            dx.zero_()                       # skinny data gradient: split the reduction over the output channels
            gemm(dy, W, dx, M, K, N, lda=lddy, ldb=K, ldc=lddx, splitk=max(2, min(N // 64, 296 // max(1, (K + 127) // 128))))
            if mask is not None:
                _lib.call("pz_relu_gate", M, K, _p(dx), lddx, _p(mask), ldmask, _p(dx), lddx, _st())
        else:
            gemm(dy, W, dx, M, K, N, lda=lddy, ldb=K, ldc=lddx, beta=beta, mask=mask, ldmask=ldmask)


def axpby(rows, cols, a, x, ldx, b, y, ldy, out, ldo):
    _lib.call("pz_axpby", rows, cols, a, _p(x), ldx, b, _p(y), ldy, _p(out), ldo, _st())


def total(t: torch.Tensor, out: torch.Tensor, slot: int):
    """out[slot] = sum of all elements of t (bias-gradient kernel on a one-column view)"""
    _lib.call("pz_colsum", _p(t), 1, t.numel(), 1, 0.0, out.data_ptr() + 4 * slot, _st())


class _Flat:
    """All live parameters as views of one flat fp32 buffer (+ a same-shaped gradient buffer): one all-reduce and
    one Adam launch per step (views start on 256-byte boundaries; the padding stays zero).  The parameters without gradient in the reference (the two unused decoders and ``dt``,
    SURVEY.md Appendix C) stay outside."""

    def __init__(self, model):
        live = [(n, p) for n, p in model.named_parameters()
                if not n.startswith(("fpc_decoder", "rpc_decoder")) and n != "dt"]
        self.names = [n for n, _ in live]
        pad = lambda n: (n + 63) // 64 * 64          # 256-byte aligned views (the TF32 GEMMs need 16-byte rows)  # noqa: E731
        n_total = sum(pad(p.numel()) for _, p in live)
        dev = live[0][1].device
        self.params = torch.zeros(n_total, device=dev, dtype=torch.float32)
        self.grads = torch.zeros(n_total, device=dev, dtype=torch.float32)
        self.exp_avg = torch.zeros(n_total, device=dev, dtype=torch.float32)
        self.exp_avg_sq = torch.zeros(n_total, device=dev, dtype=torch.float32)
        self.live = [p for _, p in live]
        self.offsets = []
        self.segments: Dict[str, list] = {}          # gradient buckets: "Encoder", "Encoder2", "heads" -> [lo, hi)
        off = 0
        with torch.no_grad():
            for name, p in live:
                n = p.numel()
                seg = name.split(".")[0] if name.startswith(("Encoder.", "Encoder2.")) else "heads"
                lo_hi = self.segments.setdefault(seg, [off, off])
                assert lo_hi[1] == off, "parameters of one bucket must be contiguous in named_parameters() order"
                lo_hi[1] = off + pad(n)
                self.params[off:off + n].copy_(p.reshape(-1))
                p.data = self.params[off:off + n].view_as(p)
                self.offsets.append(off)
                off += pad(n)
        self.n = n_total
        self.grad_of: Dict[int, torch.Tensor] = self.views(self.grads)

    def views(self, grads: torch.Tensor) -> Dict[int, torch.Tensor]:
        """id(parameter) -> its gradient as a view of the flat buffer ``grads`` (laid out like ``self.grads``)"""
        return {id(p): grads[off:off + p.numel()].view_as(p) for p, off in zip(self.live, self.offsets)}

    def g(self, p):
        return self.grad_of[id(p)]


class _EncoderCtx:
    pass


class _LinView:
    """the (weight, bias) pair linear_fwd / linear_bwd read, for a weight that is a copy of a column block"""

    def __init__(self, weight, bias):
        self.weight, self.bias = weight, bias


def all_reduce_bucket(flat: torch.Tensor, lo: int, hi: int, async_op: bool = True):
    """Sum ``flat[lo:hi]`` over the ranks of the default process group (NCCL on GPUs, gloo in the CPU tests).
    Returns the work handle (``None`` outside a process group)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1 or hi <= lo:
        return None
    return dist.all_reduce(flat[lo:hi], op=dist.ReduceOp.SUM, async_op=async_op)


class Trainer:
    """``Trainer(model, config)``: ``config`` carries the reference's options (train.py:40-55): ``lr``, ``loss_mode``,
    ``loss_sum``, ``use_emd3``, ``use_emd2``, ``use_cd2`` (the last two add terms that are functions of FPS-selected
    input points only, model5_b.py:937-942: they shift the loss value but carry no weight gradient)."""

    def __init__(self, model, config=None, lr: Optional[float] = None, precision: str = "fp32"):
        """``precision``: "fp32" (FFMA pipe, matches the reference's CPU arithmetic to ~1e-6) or "tf32" (every large
        Linear of forward and backward on the tcgen05 tensor cores in TF32 -- the arithmetic stock PyTorch 1.10
        uses for nn.Linear on Ampere-or-newer GPUs; gradients agree with fp32 to ~1e-2 relative)."""
        if precision not in ("fp32", "tf32"):
            raise ValueError("precision must be 'fp32' or 'tf32'")
        self.precision = precision
        self.tf32 = precision == "tf32"
        self.model = model
        c = config if config is not None else model.C
        self.loss_mode = int(getattr(c, "loss_mode", 0))
        self.loss_sum = bool(getattr(c, "loss_sum", False))
        self.use_emd3 = bool(getattr(c, "use_emd3", False))
        self.use_emd2 = bool(getattr(c, "use_emd2", False))
        self.use_cd2 = bool(getattr(c, "use_cd2", False))
        self.lr0 = float(lr if lr is not None else getattr(c, "lr", 0.9e-3))
        self.flat = _Flat(model)
        self.step_count = 0
        self.overlap_allreduce = True        # bucketed all-reduce started from inside backward (no-op for world size 1)
        self._pending, self._reduced = [], set()
        self.dev = self.flat.params.device
        self._buf: Dict[str, torch.Tensor] = {}
        self._grad_of = self.flat.grad_of          # where the backward writes parameter gradients (see _scope)
        self.sync_replicas()

    def sync_replicas(self, src: int = 0):
        """What DistributedDataParallel does at construction (the reference trains under Lightning DDP): rank ``src``'s
        parameters, BatchNorm buffers and optimizer state become every rank's, so replicas that were built with
        unseeded initialisation -- or of which only one loaded a checkpoint -- cannot silently diverge.  Called by the
        constructor and by :meth:`load_state_dict`; a no-op outside a process group."""
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return
        f = self.flat
        meta = torch.tensor([float(self.step_count), self.lr0], device=self.dev, dtype=torch.float64)
        dist.broadcast(meta, src)
        self.step_count, self.lr0 = int(meta[0].item()), float(meta[1].item())
        for t in (f.params, f.exp_avg, f.exp_avg_sq):
            dist.broadcast(t, src)
        for buf in self.model.buffers():          # BN running statistics and num_batches_tracked
            dist.broadcast(buf, src)
        for p in self.model.parameters():         # parameters outside the flat buffer (unused decoders, dt)
            if id(p) not in f.grad_of:
                dist.broadcast(p.data, src)
        self._invalidate_inference_state()

    def _invalidate_inference_state(self):
        """Parameters were written behind torch's back (no _version bump): drop what the inference path derived from
        them -- the weight packs inside its workspaces and the captured CUDA graphs -- and mark piece embeddings
        encoded before now as stale."""
        for ws in getattr(self.model, "_ws", {}).values():
            ws.pack_key = None
        getattr(self.model, "_graphs", {}).clear()
        self.model._weights_generation = getattr(self.model, "_weights_generation", 0) + 1

    # -------------------------------------------------------------------------------------------- scratch
    def buf(self, name, *shape, dtype=torch.float32):
        t = self._buf.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            t = torch.empty(*shape, device=self.dev, dtype=dtype)
            self._buf[name] = t
        return t

    @contextlib.contextmanager
    def _scope(self, store: Optional[Dict[str, torch.Tensor]] = None, grad_of: Optional[Dict[int, torch.Tensor]] = None):
        """Run the forward / backward methods on another buffer namespace (``store``: a graph's own activations, which
        later calls on this Trainer must not overwrite) and / or into other parameter-gradient views (``grad_of``, as
        returned by ``_Flat.views``)."""
        saved = self._buf, self._grad_of
        self._buf = saved[0] if store is None else store
        self._grad_of = saved[1] if grad_of is None else grad_of
        try:
            yield
        finally:
            self._buf, self._grad_of = saved

    def _g(self, p):
        return self._grad_of[id(p)]

    # -------------------------------------------------------------------------------------------- grouped layer 1
    def _group_layer1_forward(self, tag, lin, xyz, feat, D, centres, idx, B, N, S, out):
        """relu(lin([xyz_j - c_s ; feat_j])) for every (group, neighbour) WITHOUT the [B,S,K,3+D] tensor:
        W [xyz_j - c_s ; f_j] + b = P_j - Q_s  with  P = feat W_f^T + xyz W_x^T + b  per source point and
        Q = centres W_x^T per group (two small GEMMs), then one gather kernel writes relu(P_j - Q_s).
        Returns what the backward needs."""
        C1 = lin.weight.shape[0]
        wx, wf = self.buf(tag + ".wx", C1, 3), self.buf(tag + ".wf", C1, D)
        axpby(C1, 3, 1.0, lin.weight, 3 + D, 0.0, None, 0, wx, 3)                     # W[:, 0:3]
        axpby(C1, D, 1.0, lin.weight[:, 3:], 3 + D, 0.0, None, 0, wf, D)              # W[:, 3:]
        lin_f = _LinView(wf, lin.bias)
        P, Q = self.buf(tag + ".P", B * N, C1), self.buf(tag + ".Q", B * S, C1)
        linear_fwd(feat, D, B * N, lin_f, P, C1, tf32=self.tf32)
        gemm(xyz, wx, P, B * N, C1, 3, tb=True, lda=3, ldb=3, ldc=C1, beta=1.0)
        gemm(centres, wx, Q, B * S, C1, 3, tb=True, lda=3, ldb=3, ldc=C1)
        _lib.call("pz_gather_sub_relu", _p(P), _p(Q), _p(idx), B * S, KNN, S, N, C1, _p(out), _st())
        return dict(lin=lin, lin_f=lin_f, wx=wx, xyz=xyz, feat=feat, D=D, centres=centres, idx=idx, N=N, S=S, C1=C1)

    def _group_layer1_backward(self, tag, st, B, d_pre, dfeat, dxyz=None, dcentres=None):
        """d_pre [B*S*K, C1] = gradient w.r.t. the layer's pre-activation (ReLU-gated).  Adds the weight / bias
        gradients of ``lin`` and accumulates d loss / d feat into ``dfeat`` [B*N, D]; with ``dxyz`` [B*N, 3] and
        ``dcentres`` [B*S, 3] also d loss / d xyz_j and d loss / d c_s (accumulated into)."""
        G, lin, C1, D, N, S = self._g, st["lin"], st["C1"], st["D"], st["N"], st["S"]
        dP, dQ = self.buf(tag + ".dP", B * N, C1), self.buf(tag + ".dQ", B * S, C1)
        dP.zero_()
        _lib.call("pz_group_scatter_grad", _p(d_pre), _p(st["idx"]), B * S, KNN, S, N, C1, _p(dP), _p(dQ), _st())
        gwf, gwx = self.buf(tag + ".gwf", C1, D), self.buf(tag + ".gwx", C1, 3)
        gwf.zero_()
        gwx.zero_()
        # P = feat W_f^T + b + xyz W_x^T :  dW_f, db, dfeat from dP;  dW_x = dP^T xyz + dQ^T centres
        linear_bwd(dP, C1, st["feat"], D, B * N, st["lin_f"], gwf, G(lin.bias), dfeat, D, beta=1.0, tf32=self.tf32)
        gemm(dP, st["xyz"], gwx, C1, 3, B * N, ta=True, lda=C1, ldb=3, ldc=3, splitk=_splitk(B * N, 1))
        gemm(dQ, st["centres"], gwx, C1, 3, B * S, ta=True, lda=C1, ldb=3, ldc=3, splitk=max(2, _splitk(B * S, 1)))
        gw = G(lin.weight)                                                            # [C1, 3 + D]: add both column blocks
        axpby(C1, 3, 1.0, gwx, 3, 1.0, gw, 3 + D, gw, 3 + D)
        axpby(C1, D, 1.0, gwf, D, 1.0, gw[:, 3:], 3 + D, gw[:, 3:], 3 + D)
        if dxyz is not None:                                                          # dxyz += dP W_x ; dc += dQ W_x
            gemm(dP, st["wx"], dxyz, B * N, 3, C1, lda=C1, ldb=3, ldc=3, beta=1.0)
            gemm(dQ, st["wx"], dcentres, B * S, 3, C1, lda=C1, ldb=3, ldc=3, beta=1.0)

    # -------------------------------------------------------------------------------------------- encoder
    def _encoder_forward(self, tag, enc, xyz, start1, start2):
        """PCTransformer_nonsort.forward in train mode (model5_b.py:443-478), keeping what backward needs."""
        B = xyz.shape[0]
        c = _EncoderCtx()
        c.B, c.enc, c.xyz, c.tag = B, enc, xyz, tag
        R0 = B * NPTS
        b = lambda n, *s, **k: self.buf(f"{tag}.{n}", *s, **k)  # noqa: E731
        # stem: relu(bn(linear)) x2, BatchNorm1d(1024) over the point index with batch statistics
        c.h1, c.y1, c.h2, c.xf = b("h1", R0, 64), b("y1", R0, 64), b("h2", R0, 64), b("xf", R0, 64)
        c.bn = [b("bn1m", NPTS), b("bn1s", NPTS), b("bn2m", NPTS), b("bn2s", NPTS)]
        linear_fwd(xyz, 3, R0, enc.mlp1, c.h1, 64, tf32=self.tf32)
        _lib.call("pz_bn_point_train_forward", _p(c.h1), B, NPTS, 64, _p(enc.bn1.weight), _p(enc.bn1.bias),
                  _p(enc.bn1.running_mean), _p(enc.bn1.running_var), 0.1, 1e-5, 1, _p(c.y1), _p(c.bn[0]), _p(c.bn[1]), _st())
        linear_fwd(c.y1, 64, R0, enc.mlp2, c.h2, 64, tf32=self.tf32)
        _lib.call("pz_bn_point_train_forward", _p(c.h2), B, NPTS, 64, _p(enc.bn2.weight), _p(enc.bn2.bias),
                  _p(enc.bn2.running_mean), _p(enc.bn2.running_var), 0.1, 1e-5, 1, _p(c.xf), _p(c.bn[2]), _p(c.bn[3]), _st())
        # sample_and_group(512, 0, 32, xyz, x_feature, knn) + mlp3/mlp4 + max over the 32 neighbours
        c.fps1, c.x1 = b("fps1", B, S1, dtype=torch.int64), b("x1", B, S1, 3)
        c.knn1 = b("knn1", B, S1, KNN, dtype=torch.int64)
        _lib.call("pz_fps", _p(xyz), B, NPTS, _p(start1), S1, _p(c.fps1), _p(c.x1), _st())
        _lib.call("pz_knn", _p(c.x1), _p(xyz), B, S1, NPTS, KNN, _p(c.knn1), None, _st())
        R1 = B * S1 * KNN
        c.a1, c.a2 = b("a1", R1, 128), b("a2", R1, 128)
        c.sg1 = self._group_layer1_forward(tag + ".sg1", enc.mlp3, xyz, c.xf, 64, c.x1, c.knn1, B, NPTS, S1, c.a1)
        linear_fwd(c.a1, 128, R1, enc.mlp4, c.a2, 128, relu=True, tf32=self.tf32)
        c.f1f, c.arg1 = b("f1f", B * S1, 128), b("arg1", B * S1, 128, dtype=torch.int32)
        _lib.call("pz_maxpool_forward", _p(c.a2), B * S1, KNN, 128, _p(c.f1f), _p(c.arg1), _st())
        # stage 2 on the 512 centroids
        c.fps2, c.x2 = b("fps2", B, S2, dtype=torch.int64), b("x2", B, S2, 3)
        c.knn2 = b("knn2", B, S2, KNN, dtype=torch.int64)
        _lib.call("pz_fps", _p(c.x1), B, S1, _p(start2), S2, _p(c.fps2), _p(c.x2), _st())
        _lib.call("pz_knn", _p(c.x2), _p(c.x1), B, S2, S1, KNN, _p(c.knn2), None, _st())
        R2 = B * S2 * KNN
        c.b1, c.b2 = b("b1", R2, 256), b("b2", R2, 256)
        c.sg2 = self._group_layer1_forward(tag + ".sg2", enc.mlp5, c.x1, c.f1f, 128, c.x2, c.knn2, B, S1, S2, c.b1)
        linear_fwd(c.b1, 256, R2, enc.mlp6, c.b2, 256, relu=True, tf32=self.tf32)
        T = B * S2
        c.cat = b("cat", T, 1280)                   # [att1 | att2 | att3 | att4 | f2f]  (model5_b.py:467, :472)
        c.f2f, c.arg2 = c.cat[:, 1024:], b("arg2", T, 256, dtype=torch.int32)
        c.f2f_c = b("f2f_c", T, 256)
        _lib.call("pz_maxpool_forward", _p(c.b2), T, KNN, 256, _p(c.f2f_c), _p(c.arg2), _st())
        axpby(T, 256, 1.0, c.f2f_c, 256, 0.0, None, 0, c.f2f, 1280)
        # four offset-attention layers (model5_b.py:92-101)
        c.q, c.k, c.v, c.A, c.r, c.ro = [], [], [], [], [], []
        for l in range(4):
            att = getattr(enc, f"atten{l + 1}")
            x = c.cat[:, 1024:] if l == 0 else c.cat[:, (l - 1) * 256:]
            q, k, v = b(f"q{l}", T, 64), b(f"k{l}", T, 64), b(f"v{l}", T, 256)
            A, r, ro, vals = b(f"A{l}", B, S2, S2), b(f"r{l}", T, 256), b(f"ro{l}", T, 256), b("vals", T, 256)
            linear_fwd(x, 1280, T, att.mlpq, q, 64, tf32=self.tf32)
            linear_fwd(x, 1280, T, att.mlpk, k, 64, tf32=self.tf32)
            linear_fwd(x, 1280, T, att.mlpv, v, 256, tf32=self.tf32)
            if self.tf32:       # S = q k^T, softmax, vals = A v: two batched TF32 GEMMs around one softmax kernel
                bgemm_tf32(0, 0, S2, S2, 64, q, 64, k, 64, A, S2, B, S2 * 64, S2 * 64, S2 * S2)
                _lib.call("pz_softmax_forward", _p(A), B * S2, S2, 1.0 / math.sqrt(64.0), _p(A), _st())
                bgemm_tf32(0, 1, S2, 256, S2, A, S2, v, 256, vals, 256, B, S2 * S2, S2 * 256, S2 * 256)
            else:
                _lib.call("pz_scaled_dot_attention", _p(q), _p(k), _p(v), B, S2, 64, 256, _p(vals), _p(A), _st())
            axpby(T, 256, 1.0, x, 1280, -1.0, vals, 256, r, 256)                              # r = x - A v
            linear_fwd(r, 256, T, att.out, ro, 256, relu=True, tf32=self.tf32)                                # relu(W_o r + b_o)
            axpby(T, 256, 1.0, x, 1280, 1.0, ro, 256, c.cat[:, l * 256:], 1280)               # x + relu(...)
            for lst, t in zip((c.q, c.k, c.v, c.A, c.r, c.ro), (q, k, v, A, r, ro)):
                lst.append(t)
        c.out = b("out", T, 1024)
        linear_fwd(c.cat, 1280, T, enc.out, c.out, 1024, tf32=self.tf32)
        c.fg, c.argo = b("fg", B, 1024), b("argo", B, 1024, dtype=torch.int32)
        _lib.call("pz_maxpool_forward", _p(c.out), B, S2, 1024, _p(c.fg), _p(c.argo), _st())
        return c

    def _encoder_backward(self, c, dfg, dxf, accumulate=False, dattn=None, dxyz=None, dx2=None):
        """dfg [B,1024] = d loss / d f_global; dxf [B*1024,64] = d loss / d x_feature from the boundary heads
        (accumulated into, then consumed).  Writes every parameter gradient of the encoder.  Optional gradients of
        the other outputs: ``dattn`` [B,256,256] of the mean attention map, ``dx2`` [B*256,3] of the stage-2 centres.
        ``dxyz`` [B*1024,3] (zeroed by the caller) receives d loss / d xyz through the stem, both grouping stages and
        the centres (FPS and kNN indices are constants)."""
        enc, B, tag, G = c.enc, c.B, c.tag, self._g
        b = lambda n, *s, **k: self.buf(f"{tag}.{n}", *s, **k)  # noqa: E731
        T, R1, R2, R0 = B * S2, B * S1 * KNN, B * S2 * KNN, B * NPTS
        dout = b("dout", T, 1024)
        _lib.call("pz_maxpool_backward", _p(dfg), _p(c.fg), _p(c.argo), B, S2, 1024, 0, _p(dout), _st())
        dcat = b("dcat", T, 1280)
        linear_bwd(dout, 1024, c.cat, 1280, T, enc.out, G(enc.out.weight), G(enc.out.bias), dcat, 1280, tf32=self.tf32)
        dcur, dz, dr = b("dcur", T, 256), b("dz", T, 256), b("dr", T, 256)
        dq, dk, dv = b("dq", T, 64), b("dk", T, 64), b("dv", T, 256)
        dA, dS = b("dA", B, S2, S2), b("dS", B, S2, S2)
        axpby(T, 256, 1.0, dcat[:, 768:], 1280, 0.0, None, 0, dcur, 256)
        LL = S2 * S2
        for l in (3, 2, 1, 0):
            att = getattr(enc, f"atten{l + 1}")
            x = c.cat[:, 1024:] if l == 0 else c.cat[:, (l - 1) * 256:]
            q, k, v, A, r, ro = c.q[l], c.k[l], c.v[l], c.A[l], c.r[l], c.ro[l]
            # out_l = x + relu(W_o r + b_o)
            _lib.call("pz_relu_gate", T, 256, _p(dcur), 256, _p(ro), 256, _p(dz), 256, _st())
            linear_bwd(dz, 256, r, 256, T, att.out, G(att.out.weight), G(att.out.bias), dr, 256, tf32=self.tf32)
            # r = x - A v :  dx = dcur + dr ; dvals = -dr
            axpby(T, 256, 1.0, dcur, 256, 1.0, dr, 256, dcur, 256)
            # vals = A v (per cloud):  dv = A^T dvals ; dA = dvals v^T
            if self.tf32:
                dvals = b("dvals", T, 256)
                axpby(T, 256, -1.0, dr, 256, 0.0, None, 0, dvals, 256)
                bgemm_tf32(1, 1, S2, 256, S2, A, S2, dvals, 256, dv, 256, B, LL, S2 * 256, S2 * 256)
                bgemm_tf32(0, 0, S2, S2, 256, dvals, 256, v, 256, dA, S2, B, S2 * 256, S2 * 256, LL)
            else:
                gemm(A, dr, dv, S2, 256, S2, ta=True, lda=S2, ldb=256, ldc=256, alpha=-1.0, batch=B, sa=LL, sb=S2 * 256,
                     sc=S2 * 256)
                gemm(dr, v, dA, S2, S2, 256, tb=True, lda=256, ldb=256, ldc=S2, alpha=-1.0, batch=B, sa=S2 * 256,
                     sb=S2 * 256, sc=LL)
            if dattn is not None:                    # attention = mean of the four maps (model5_b.py:468-469)
                axpby(B * S2, S2, 0.25, dattn, S2, 1.0, dA, S2, dA, S2)
            _lib.call("pz_softmax_backward", _p(A), _p(dA), B * S2, S2, 1.0 / math.sqrt(64.0), _p(dS), _st())
            # S = q k^T :  dq = dS k ; dk = dS^T q
            if self.tf32:
                bgemm_tf32(0, 1, S2, 64, S2, dS, S2, k, 64, dq, 64, B, LL, S2 * 64, S2 * 64)
                bgemm_tf32(1, 1, S2, 64, S2, dS, S2, q, 64, dk, 64, B, LL, S2 * 64, S2 * 64)
            else:
                gemm(dS, k, dq, S2, 64, S2, lda=S2, ldb=64, ldc=64, batch=B, sa=LL, sb=S2 * 64, sc=S2 * 64)
                gemm(dS, q, dk, S2, 64, S2, ta=True, lda=S2, ldb=64, ldc=64, batch=B, sa=LL, sb=S2 * 64, sc=S2 * 64)
            linear_bwd(dq, 64, x, 1280, T, att.mlpq, G(att.mlpq.weight), G(att.mlpq.bias), dcur, 256, beta=1.0, tf32=self.tf32)
            linear_bwd(dk, 64, x, 1280, T, att.mlpk, G(att.mlpk.weight), G(att.mlpk.bias), dcur, 256, beta=1.0, tf32=self.tf32)
            linear_bwd(dv, 256, x, 1280, T, att.mlpv, G(att.mlpv.weight), G(att.mlpv.bias), dcur, 256, beta=1.0, tf32=self.tf32)
            # dcur is now d loss / d x of this layer; x is also a column slice of cat
            src = dcat[:, 1024:] if l == 0 else dcat[:, (l - 1) * 256:]
            axpby(T, 256, 1.0, dcur, 256, 1.0, src, 1280, dcur, 256)
        # dcur = d loss / d f2f ;  sg2: max over neighbours <- relu(mlp6(relu(mlp5(g2))))
        db2, db1 = b("db2", R2, 256), b("db1", R2, 256)
        _lib.call("pz_maxpool_backward", _p(dcur), _p(c.f2f_c), _p(c.arg2), T, KNN, 256, 1, _p(db2), _st())
        # bias gradient of the pooled layer from the [groups, C] gradient (32x fewer rows than the scattered db2):
        # sum_rows db2 = sum_groups (f2f > 0 ? dcur : 0)
        gated = b("gated2", T, 256)
        _lib.call("pz_relu_gate", T, 256, _p(dcur), 256, _p(c.f2f_c), 256, _p(gated), 256, _st())
        _lib.call("pz_colsum", _p(gated), 256, T, 256, 1.0, _p(G(enc.mlp6.bias)), _st())
        linear_bwd(db2, 256, c.b1, 256, R2, enc.mlp6, G(enc.mlp6.weight), G(enc.mlp6.bias), db1, 256, mask=c.b1, ldmask=256,
                   tf32=self.tf32, bias_grad=False)
        df1f = b("df1f", B * S1, 128)
        df1f.zero_()
        dx1 = dxc2 = None
        if dxyz is not None:
            dx1, dxc2 = b("dx1", B * S1, 3), b("dxc2", B * S2, 3)
            dx1.zero_()
            if dx2 is None:
                dxc2.zero_()
            else:
                axpby(B * S2, 3, 1.0, dx2, 3, 0.0, None, 0, dxc2, 3)
        self._group_layer1_backward(tag + ".sg2", c.sg2, B, db1, df1f, dx1, dxc2)
        if dxyz is not None:                         # x2 = x1[fps2]
            _lib.call("pz_scatter_add_rows", _p(dxc2), 3, 0, 3, _p(c.fps2), B * S2, S2, S1, _p(dx1), 3, _st())
        # sg1
        da2, da1 = b("da2", R1, 128), b("da1", R1, 128)
        _lib.call("pz_maxpool_backward", _p(df1f), _p(c.f1f), _p(c.arg1), B * S1, KNN, 128, 1, _p(da2), _st())
        gated1 = b("gated1", B * S1, 128)
        _lib.call("pz_relu_gate", B * S1, 128, _p(df1f), 128, _p(c.f1f), 128, _p(gated1), 128, _st())
        _lib.call("pz_colsum", _p(gated1), 128, B * S1, 128, 1.0, _p(G(enc.mlp4.bias)), _st())
        linear_bwd(da2, 128, c.a1, 128, R1, enc.mlp4, G(enc.mlp4.weight), G(enc.mlp4.bias), da1, 128, mask=c.a1, ldmask=128,
                   tf32=self.tf32, bias_grad=False)
        self._group_layer1_backward(tag + ".sg1", c.sg1, B, da1, dxf, dxyz, dx1)
        if dxyz is not None:                         # x1 = xyz[fps1]
            _lib.call("pz_scatter_add_rows", _p(dx1), 3, 0, 3, _p(c.fps1), B * S1, S1, NPTS, _p(dxyz), 3, _st())
        # stem
        dh2, dy1, dh1 = b("dh2", R0, 64), b("dy1", R0, 64), b("dh1", R0, 64)
        _lib.call("pz_bn_point_train_backward", _p(c.h2), _p(c.xf), _p(dxf), B, NPTS, 64, _p(enc.bn2.weight), _p(c.bn[2]),
                  _p(c.bn[3]), 1, int(accumulate), _p(dh2), _p(G(enc.bn2.weight)), _p(G(enc.bn2.bias)), _st())
        linear_bwd(dh2, 64, c.y1, 64, R0, enc.mlp2, G(enc.mlp2.weight), G(enc.mlp2.bias), dy1, 64, tf32=self.tf32)
        _lib.call("pz_bn_point_train_backward", _p(c.h1), _p(c.y1), _p(dy1), B, NPTS, 64, _p(enc.bn1.weight), _p(c.bn[0]),
                  _p(c.bn[1]), 1, int(accumulate), _p(dh1), _p(G(enc.bn1.weight)), _p(G(enc.bn1.bias)), _st())
        linear_bwd(dh1, 64, c.xyz, 3, R0, enc.mlp1, G(enc.mlp1.weight), G(enc.mlp1.bias), dxyz, 3, beta=1.0,
                   tf32=self.tf32)

    # -------------------------------------------------------------------------------------------- MLP stacks
    def _mlp_forward(self, tag, seq, x, ldx, M):
        """nn.Sequential(Linear, ReLU, ..., Linear): returns the list of layer outputs (post-ReLU but the last)."""
        lins = [m for m in seq if isinstance(m, torch.nn.Linear)]
        acts = []
        cur, ld = x, ldx
        for i, lin in enumerate(lins):
            y = self.buf(f"{tag}.y{i}", M, lin.weight.shape[0])
            linear_fwd(cur, ld, M, lin, y, lin.weight.shape[0], relu=i + 1 < len(lins), tf32=self.tf32)
            acts.append(y)
            cur, ld = y, lin.weight.shape[0]
        return lins, acts

    def _mlp_backward(self, tag, lins, acts, x, ldx, M, dy, dx, lddx):
        """dy = gradient of the last (linear) output; returns nothing, fills dx [M, in] (may be None)."""
        G = self._g
        for i in range(len(lins) - 1, -1, -1):
            lin = lins[i]
            xin, ldin = (acts[i - 1], lins[i - 1].weight.shape[0]) if i > 0 else (x, ldx)
            if i > 0:
                dprev = self.buf(f"{tag}.d{i - 1}", M, ldin)
                linear_bwd(dy, lin.weight.shape[0], xin, ldin, M, lin, G(lin.weight), G(lin.bias), dprev, ldin,
                           mask=acts[i - 1], ldmask=ldin, tf32=self.tf32)
                dy = dprev
            else:
                linear_bwd(dy, lin.weight.shape[0], xin, ldin, M, lin, G(lin.weight), G(lin.bias), dx, lddx, tf32=self.tf32)

    # -------------------------------------------------------------------------------------------- the step
    def _forward(self, fpc, mrpc, starts, pretrain=False):
        """train-mode predict5 (model5_b.py:672-759 with training=True): both encoders, the pose head and the two
        boundary heads; returns every buffer the backward pass reads.  Must run inside ``torch.cuda.device``."""
        m = self.model
        B = fpc.shape[0]
        if starts is None:
            starts = torch.stack([torch.randint(0, 1024, (B,), dtype=torch.long),
                                  torch.randint(0, 512, (B,), dtype=torch.long),
                                  torch.randint(0, 1024, (B,), dtype=torch.long),
                                  torch.randint(0, 512, (B,), dtype=torch.long)])
        starts = starts.to(self.dev, torch.int64).contiguous()
        ef = self._encoder_forward("E1", m.Encoder, fpc, starts[0], starts[1])
        em = self._encoder_forward("E2", m.Encoder if pretrain else m.Encoder2, mrpc, starts[2], starts[3])
        R0 = B * NPTS
        # ---- pose head: tfMLP(cat(f_global_fpc, f_global_mrpc))  (model5_b.py:723-725)
        f = self.buf("f", B, 2048)
        axpby(B, 1024, 1.0, ef.fg, 1024, 0.0, None, 0, f, 2048)
        axpby(B, 1024, 1.0, em.fg, 1024, 0.0, None, 0, f[:, 1024:], 2048)
        tf_l, tf_a = self._mlp_forward("tf", m.tfMLP, f, 2048, B)
        if pretrain:           # predict6 (model5_b.py:647-658): shared encoder, pose head only
            return dict(ef=ef, em=em, f=f, tf_l=tf_l, tf_a=tf_a, out6=tf_a[-1])
        # ---- boundary heads (model5_b.py:729-754; both "global" vectors come from the mrpc branch, D6)
        lf_l, lf_a = self._mlp_forward("lf", m.MLPLocalPreFpc, ef.xf, 64, R0)
        lm_l, lm_a = self._mlp_forward("lm", m.MLPLocalPreRpc, em.xf, 64, R0)
        gmax, garg = self.buf("gmax", B, 64), self.buf("garg", B, 64, dtype=torch.int32)
        _lib.call("pz_maxpool_forward", _p(lm_a[-1]), B, NPTS, 64, _p(gmax), _p(garg), _st())
        seg_f, seg_m = self.buf("seg_f", R0, 128), self.buf("seg_m", R0, 128)
        for seg, loc in ((seg_f, lf_a[-1]), (seg_m, lm_a[-1])):
            _lib.call("pz_broadcast_rows", _p(gmax), B, NPTS, 64, _p(seg), 128, _st())
            axpby(R0, 64, 1.0, loc, 64, 0.0, None, 0, seg[:, 64:], 128)
        sf_l, sf_a = self._mlp_forward("sf", m.MLPFpcb, seg_f, 128, R0)
        sm_l, sm_a = self._mlp_forward("sm", m.MLPRpcb, seg_m, 128, R0)
        return dict(ef=ef, em=em, f=f, tf_l=tf_l, tf_a=tf_a, out6=tf_a[-1], lf_l=lf_l, lf_a=lf_a, lm_l=lm_l, lm_a=lm_a,
                    gmax=gmax, garg=garg, seg_f=seg_f, seg_m=seg_m, sf_l=sf_l, sf_a=sf_a, sm_l=sm_l, sm_a=sm_a,
                    logit_f=sf_a[-1], logit_m=sm_a[-1])            # logits are [B*1024, 2] (point-major)

    def predict5_train(self, fpc, mrpc, starts=None):
        """``predict5(batch, _, need=True, training=True)`` (model5_b.py:672-759): the train-mode forward (batch
        statistics in, and running statistics updated by, the four BatchNorm layers) without the backward pass ->
        ``(out, [0], x2_fpc, attention_fpc, x2_mrpc, attention_mrpc, de_fpcb, de_mrpcb)``."""
        fpc, mrpc = fpc.contiguous().float(), mrpc.contiguous().float()
        _lib.require_cuda(fpc, mrpc)
        with torch.cuda.device(self.dev):
            fw = self._forward(fpc, mrpc, starts)
            out6, de_f, de_m, x2f, af, x2m, am = self._outputs(fw, fpc.shape[0], need=True)
        self._invalidate_inference_state()            # the BatchNorm running statistics were updated in place
        return out6, [0], x2f, af, x2m, am, de_f, de_m

    def _outputs(self, fw, B, need):
        """The train-mode forward's outputs as fresh tensors: ``(out6, de_fpcb, de_mrpcb, x2_fpc, attention_fpc,
        x2_mrpc, attention_mrpc)``; ``de_*`` are None after predict6's forward, the last four None without ``need``."""
        res = [None] * 4
        if need:
            res = []
            for e in (fw["ef"], fw["em"]):
                att = torch.empty(B, S2, S2, device=self.dev)
                n = B * S2
                axpby(n, S2, 0.25, e.A[0], S2, 0.25, e.A[1], S2, att, S2)          # mean of the 4 maps (:468-469)
                axpby(n, S2, 0.25, e.A[2], S2, 1.0, att, S2, att, S2)
                axpby(n, S2, 0.25, e.A[3], S2, 1.0, att, S2, att, S2)
                res += [e.x2.clone(), att]
        de_f = de_m = None
        if "logit_f" in fw:
            de_f = fw["logit_f"].view(B, NPTS, 2).permute(0, 2, 1).contiguous()
            de_m = fw["logit_m"].view(B, NPTS, 2).permute(0, 2, 1).contiguous()
        return (fw["out6"].clone(), de_f, de_m, *res)

    def _pose_losses(self, out6, mrpc, rpc, igt, B):
        """The pose part of training_step (model5_b.py:947-1029): mat = se3.exp(out), de_mrpc = mat . mrpc,
        chamfer(rpc, de_mrpc), comp(mat, igt), EMD(de_mrpc, rpc) -> loss sums in ``vals[0..3]`` and d loss / d out6
        for the configured ``loss_mode``."""
        vals = self.buf("loss_terms", 16)
        vals.zero_()
        mat = self.buf("mat", B, 4, 4)
        _lib.call("pz_se3_exp", _p(out6), B, _p(mat), _st())
        de_mrpc = losses.transform_points(mat, mrpc)
        red = 1.0 if self.loss_sum else 1.0 / (B * NPTS)
        d1, d2, a1, a2 = losses._chamfer_raw(rpc, de_mrpc, True)           # d1 per de_mrpc point, d2 per rpc point
        total(d1, vals, 0)
        total(d2, vals, 1)
        _lib.call("pz_comp", _p(mat), _p(igt), B, vals.data_ptr() + 4 * 2, _st())
        from . import emd_cuda
        match = emd_cuda.approxmatch_forward(de_mrpc, rpc)
        cost = emd_cuda.matchcost_forward(de_mrpc, rpc, match)
        total(cost, vals, 3)
        w_re = {0: 1, 1: 1, 2: 0, 3: 0, 4: 1, 5: 0, 6: 1}[self.loss_mode]
        w_g = {0: 1, 1: 1, 2: 0, 3: 1, 4: 0, 5: 1, 6: 0}[self.loss_mode]
        w_emd = {0: 0, 1: 1, 2: 1, 3: 1, 4: 1, 5: 0, 6: 0}[self.loss_mode]
        emd_red = 1.0 if self.loss_sum else 1.0 / B
        dde = self.buf("dde", B, NPTS, 3)
        gw1 = torch.full((B, NPTS), red * w_re, device=self.dev)
        gx, gy = self.buf("ch_gx", B, NPTS, 3), self.buf("ch_gy", B, NPTS, 3)
        _lib.call("pz_chamfer_grad", _p(rpc), _p(de_mrpc), B, NPTS, NPTS, _p(a1), _p(a2), _p(gw1), _p(gw1), _p(gx),
                  _p(gy), _st())
        gc = torch.full((B,), emd_red * w_emd, device=self.dev)
        g1, _ = emd_cuda.matchcost_backward(gc, de_mrpc, rpc, match)
        axpby(B * NPTS, 3, 1.0, gy, 3, 1.0, g1, 3, dde, 3)
        dout6 = self.buf("dout6", B, 6)
        _lib.call("pz_pose_grad", _p(out6), _p(mrpc), _p(dde), NPTS, _p(igt), float(w_g), B, 0.0, _p(dout6), _st())
        return vals, mat, de_mrpc, dout6, (w_re, w_g, w_emd)

    def _attention_peak_terms(self, ef, em, B, vals):
        """model5_b.py:937-942, :1001-1012: ``x2att = x2[:, topk(attention.mean(1), 32)[1][:, 0]]`` -- for every
        cloud the FPS point that receives the most attention, gathered for ALL batch items (the reference's indexing
        yields [B,B,3]) -- then chamfer (``loss_cd2``) and EMD (``emd2``) between the two [B,B,3] sets -> vals[12..14].
        Values only: nothing here depends on the weights differentiably."""
        from . import emd_cuda, pointnet_util as pu
        peaks = []
        for e in (ef, em):
            att = self.buf(e.tag + ".attmean", B, S2, S2)
            n = B * S2
            axpby(n, S2, 0.25, e.A[0], S2, 0.25, e.A[1], S2, att, S2)            # mean of the 4 maps (:468-469)
            axpby(n, S2, 0.25, e.A[2], S2, 1.0, att, S2, att, S2)
            axpby(n, S2, 0.25, e.A[3], S2, 1.0, att, S2, att, S2)
            colmean = self.buf(e.tag + ".attcol", B, S2)
            _lib.call("pz_group_sum", _p(att), S2, B, S2, S2, _p(colmean), _st())   # sum over the query index (dim 1)
            _, top = losses.topk(colmean, 32, largest=True)
            idx = top[:, 0].contiguous().view(1, B).expand(B, B).contiguous()       # the same B indices for every cloud
            peaks.append(pu.index_points(e.x2, idx))                                # [B, B, 3]
        c1, c2, _, _ = losses._chamfer_raw(peaks[0], peaks[1], False)
        total(c1, vals, 12)
        total(c2, vals, 13)
        match = emd_cuda.approxmatch_forward(peaks[0], peaks[1])
        total(emd_cuda.matchcost_forward(peaks[0], peaks[1], match), vals, 14)

    def _peak_term_values(self, v, B):
        red = 1.0 if self.loss_sum else 1.0 / (B * B)
        return dict(loss_cd2=(v[12] + v[13]) * red, emd2=v[14])               # emd2 is summed in both modes (:1033-1036)

    def forward_backward_pretrain(self, batch, starts=None) -> Dict[str, float]:
        """The pretraining branch of training_step (model5_b.py:928-931, :1048-1050: ``current_epoch <
        pretrain_epochs``): predict6 -- BOTH clouds through ``Encoder`` -- and the pose losses only.  ``Encoder``
        back-propagates twice, its gradients add; ``Encoder2`` and the boundary heads get none."""
        fpc, mrpc, igt, rpc = [t.contiguous().float() for t in batch[:4]]
        _lib.require_cuda(fpc, mrpc, igt, rpc)
        B = fpc.shape[0]
        self.flat.grads.zero_()
        with torch.cuda.device(self.dev):
            fw = self._forward(fpc, mrpc, starts, pretrain=True)
            out6 = fw["out6"]
            vals, mat, de_mrpc, dout6, (w_re, w_g, w_emd) = self._pose_losses(out6, mrpc, rpc, igt, B)
            self._backward(fw, B, dout6)
            if self.use_emd2 or self.use_cd2:
                self._attention_peak_terms(fw["ef"], fw["em"], B, vals)
            v = vals.cpu().tolist()
        self.last = dict(out=out6, de_mrpc=de_mrpc, mat=mat)
        n_re = 1.0 if self.loss_sum else B * NPTS
        terms = dict(loss_re=(v[0] + v[1]) / n_re, loss_g=v[2], loss_emd=v[3] * (1.0 if self.loss_sum else 1.0 / B))
        terms["loss"] = w_re * terms["loss_re"] + w_g * terms["loss_g"] + w_emd * terms["loss_emd"]
        if self.use_emd2 or self.use_cd2:
            terms.update(self._peak_term_values(v, B))
            terms["loss"] += (terms["emd2"] if self.use_emd2 else 0.0) + (terms["loss_cd2"] if self.use_cd2 else 0.0)
        return terms

    def forward_backward(self, batch, starts=None) -> Dict[str, float]:
        """Train-mode predict5 + losses + backward into ``self.flat.grads`` (zeroed first).  ``starts`` [4,B] as in
        ``predict5``.  Returns the logged terms as python floats (one device->host copy)."""
        fpc, mrpc, igt, rpc, fpcb, rpcb, fpc_idx, rpc_idx = [t.contiguous().float() for t in batch[:8]]
        _lib.require_cuda(fpc, mrpc, igt, rpc, fpcb, rpcb, fpc_idx, rpc_idx)
        B = fpc.shape[0]
        self.flat.grads.zero_()
        with torch.cuda.device(self.dev):
            fw = self._forward(fpc, mrpc, starts)
            ef, em, out6, logit_f, logit_m = fw["ef"], fw["em"], fw["out6"], fw["logit_f"], fw["logit_m"]
            R0 = B * NPTS
            # ---- losses
            vals, mat, de_mrpc, dout6, (w_re, w_g, w_emd) = self._pose_losses(out6, mrpc, rpc, igt, B)
            from . import emd_cuda
            # cross entropy of both boundary heads
            dlf, dlm = self.buf("dlf", R0, 2), self.buf("dlm", R0, 2)
            _lib.call("pz_cross_entropy", _p(logit_f), _p(fpc_idx), B, NPTS, 1, 1.0, vals.data_ptr() + 4 * 4, _p(dlf), _st())
            _lib.call("pz_cross_entropy", _p(logit_m), _p(rpc_idx), B, NPTS, 1, 1.0, vals.data_ptr() + 4 * 5, _p(dlm), _st())
            # predicted boundaries: top-128 by class-1 probability, gathered from the inputs (no weight gradient
            # through the selection); the mrpc boundary is aligned by the predicted pose -> gradient into out6
            de_f = logit_f.view(B, NPTS, 2).permute(0, 2, 1).contiguous()
            de_m = logit_m.view(B, NPTS, 2).permute(0, 2, 1).contiguous()
            idx_f, idx_m = losses.boundary_topk(de_f), losses.boundary_topk(de_m)
            from . import pointnet_util as pu
            bnd_f, bnd_m = pu.index_points(fpc, idx_f), pu.index_points(mrpc, idx_m)
            c1, c2, _, _ = losses._chamfer_raw(bnd_f, fpcb, False)
            total(c1, vals, 6)
            total(c2, vals, 7)
            inv_bnd = losses.transform_points(mat, bnd_m)
            c1, c2, b1a, b2a = losses._chamfer_raw(inv_bnd, rpcb, True)
            total(c1, vals, 8)
            total(c2, vals, 9)
            gwb = torch.full((B, 128), 1.0 / (B * 128), device=self.dev)
            gbx, gby = self.buf("chb_gx", B, 128, 3), self.buf("chb_gy", B, 128, 3)
            _lib.call("pz_chamfer_grad", _p(inv_bnd), _p(rpcb), B, 128, 128, _p(b1a), _p(b2a), _p(gwb), _p(gwb), _p(gbx),
                      _p(gby), _st())
            match_f = emd_cuda.approxmatch_forward(bnd_f, fpcb)
            total(emd_cuda.matchcost_forward(bnd_f, fpcb, match_f), vals, 10)
            match_m = emd_cuda.approxmatch_forward(inv_bnd, rpcb)
            total(emd_cuda.matchcost_forward(inv_bnd, rpcb, match_m), vals, 11)
            if self.use_emd3:
                gcb = torch.full((B,), 1.0 / B, device=self.dev)
                g1b, _ = emd_cuda.matchcost_backward(gcb, inv_bnd, rpcb, match_m)
                axpby(B * 128, 3, 1.0, gbx, 3, 1.0, g1b, 3, gbx, 3)
            _lib.call("pz_pose_grad", _p(out6), _p(bnd_m), _p(gbx), 128, None, 0.0, B, 1.0, _p(dout6), _st())
            self._backward(fw, B, dout6, dlf, dlm, overlap_allreduce=True)
            if self.use_emd2 or self.use_cd2:
                self._attention_peak_terms(ef, em, B, vals)
            v = vals.cpu().tolist()
        self.last = dict(out=out6, de_fpcb=de_f, de_mrpcb=de_m, de_mrpc=de_mrpc, mat=mat, idx_f=idx_f, idx_m=idx_m)
        n_re = 1.0 if self.loss_sum else B * NPTS
        terms = dict(loss_re=(v[0] + v[1]) / n_re, loss_g=v[2], loss_emd=v[3] * (1.0 if self.loss_sum else 1.0 / B),
                     ce_f=v[4], ce_m=v[5], loss_fpcb=(v[6] + v[7]) / (B * 128), loss_mrpcb=(v[8] + v[9]) / (B * 128),
                     emd_fpcb=v[10] / B, emd_mrpcb=v[11] / B)
        loss = w_re * terms["loss_re"] + w_g * terms["loss_g"] + w_emd * terms["loss_emd"]
        loss += terms["ce_f"] + terms["ce_m"] + terms["loss_mrpcb"] + terms["loss_fpcb"]
        if self.use_emd3:
            loss += terms["emd_fpcb"] + terms["emd_mrpcb"]
        if self.use_emd2 or self.use_cd2:
            terms.update(self._peak_term_values(v, B))
            loss += (terms["emd2"] if self.use_emd2 else 0.0) + (terms["loss_cd2"] if self.use_cd2 else 0.0)
        terms["loss"] = loss
        return terms

    def _backward(self, fw, B, dout6, dlf=None, dlm=None, dattn=(None, None), dx2=(None, None), dxyz=(None, None),
                  overlap_allreduce=False):
        """Backward of the train-mode forward ``fw`` (``_forward``) from gradients of its outputs, added into the
        parameter gradients (zeroed by the caller): ``dout6`` [B,6] of the pose; ``dlf`` / ``dlm`` [B*1024,2] of the
        point-major logits of the two boundary heads (predict5 only; both or neither); per cloud (fpc, mrpc) optional
        ``dattn`` [B,256,256] of the mean attention map and ``dx2`` [B*256,3] of the stage-2 centres; ``dxyz``
        [B*1024,3] per cloud (zeroed by the caller) receive d loss / d cloud.  With ``fw`` from predict6 both clouds
        went through ``Encoder`` and its gradients from the two passes add.  ``overlap_allreduce``: start each
        gradient bucket's all-reduce as soon as it is final."""
        R0 = B * NPTS
        pretrain = "logit_f" not in fw
        # ---- pose head
        df = self.buf("df", B, 2048)
        self._mlp_backward("tf", fw["tf_l"], fw["tf_a"], fw["f"], 2048, B, dout6, df, 2048)
        dfg_f, dfg_m = self.buf("dfg_f", B, 1024), self.buf("dfg_m", B, 1024)
        axpby(B, 1024, 1.0, df, 2048, 0.0, None, 0, dfg_f, 1024)
        axpby(B, 1024, 1.0, df[:, 1024:], 2048, 0.0, None, 0, dfg_m, 1024)
        if pretrain:                # no boundary heads: nothing reaches x_feature from above
            dxf_f = dxf_m = self.buf("dxf_f", R0, 64)
            dxf_f.zero_()
        else:
            # ---- boundary heads
            dseg_f, dseg_m = self.buf("dseg_f", R0, 128), self.buf("dseg_m", R0, 128)
            self._mlp_backward("sf", fw["sf_l"], fw["sf_a"], fw["seg_f"], 128, R0, dlf, dseg_f, 128)
            self._mlp_backward("sm", fw["sm_l"], fw["sm_a"], fw["seg_m"], 128, R0, dlm, dseg_m, 128)
            dg_f, dg_m = self.buf("dg_f", B, 64), self.buf("dg_m", B, 64)
            _lib.call("pz_group_sum", _p(dseg_f), 128, B, NPTS, 64, _p(dg_f), _st())
            _lib.call("pz_group_sum", _p(dseg_m), 128, B, NPTS, 64, _p(dg_m), _st())
            axpby(B, 64, 1.0, dg_f, 64, 1.0, dg_m, 64, dg_f, 64)
            dloc_m, dloc_f = self.buf("dloc_m", R0, 64), self.buf("dloc_f", R0, 64)
            _lib.call("pz_maxpool_backward", _p(dg_f), _p(fw["gmax"]), _p(fw["garg"]), B, NPTS, 64, 0, _p(dloc_m), _st())
            axpby(R0, 64, 1.0, dloc_m, 64, 1.0, dseg_m[:, 64:], 128, dloc_m, 64)
            axpby(R0, 64, 1.0, dseg_f[:, 64:], 128, 0.0, None, 0, dloc_f, 64)
            dxf_f, dxf_m = self.buf("dxf_f", R0, 64), self.buf("dxf_m", R0, 64)
            self._mlp_backward("lf", fw["lf_l"], fw["lf_a"], fw["ef"].xf, 64, R0, dloc_f, dxf_f, 64)
            self._mlp_backward("lm", fw["lm_l"], fw["lm_a"], fw["em"].xf, 64, R0, dloc_m, dxf_m, 64)
            if overlap_allreduce:
                self._bucket_ready("heads")
        # ---- encoders
        self._encoder_backward(fw["ef"], dfg_f, dxf_f, dattn=dattn[0], dxyz=dxyz[0], dx2=dx2[0])
        if overlap_allreduce and not pretrain:
            self._bucket_ready("Encoder")
        if pretrain:
            dxf_m.zero_()
        self._encoder_backward(fw["em"], dfg_m, dxf_m, accumulate=pretrain, dattn=dattn[1], dxyz=dxyz[1], dx2=dx2[1])
        if overlap_allreduce and not pretrain:
            self._bucket_ready("Encoder2")

    def _bucket_ready(self, name):
        """Called by the backward pass as soon as a gradient bucket is final: start its all-reduce so that it
        overlaps the rest of backward (heads -> Encoder -> Encoder2; SURVEY.md §8e)."""
        if self.overlap_allreduce:
            lo, hi = self.flat.segments[name]
            w = all_reduce_bucket(self.flat.grads, lo, hi)
            if w is not None:
                self._pending.append(w)
                self._reduced.add(name)

    def all_reduce_grads(self):
        """Finish the gradient all-reduce: wait for the buckets started during backward and reduce the ones that
        were not (all of them when ``overlap_allreduce`` is off).  Returns the world size."""
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return 1
        rest = [n for n in self.flat.segments if n not in self._reduced]
        if len(rest) == len(self.flat.segments):
            dist.all_reduce(self.flat.grads, op=dist.ReduceOp.SUM)          # one collective for the whole buffer
        else:
            for n in rest:
                lo, hi = self.flat.segments[n]
                self._pending.append(all_reduce_bucket(self.flat.grads, lo, hi))
        for w in self._pending:
            if w is not None:
                w.wait()
        self._pending, self._reduced = [], set()
        return dist.get_world_size()

    def optimizer_step(self, world: int = 1):
        """Adam(lr) with StepLR(step_size=50, gamma=0.999) stepped per iteration (model5_b.py:1453-1457)."""
        self.step_count += 1
        lr = self.lr0 * (0.999 ** ((self.step_count - 1) // 50))
        f = self.flat
        with torch.cuda.device(self.dev):
            _lib.call("pz_adam_step", _p(f.params), _p(f.grads), _p(f.exp_avg), _p(f.exp_avg_sq), f.n, lr, 0.9, 0.999, 1e-8,
                      self.step_count, 1.0 / world, _st())
        self._invalidate_inference_state()
        return lr

    # -------------------------------------------------------------------------------------------- checkpoint / resume
    def state_dict(self):
        """Optimizer state for checkpoint / resume (the model's own ``state_dict()`` holds the parameters -- they are
        views of the flat buffer, so nothing else is needed): Adam moments, step count, base learning rate."""
        return {"step": self.step_count, "lr0": self.lr0, "precision": self.precision, "n": self.flat.n,
                "exp_avg": self.flat.exp_avg.detach().clone(), "exp_avg_sq": self.flat.exp_avg_sq.detach().clone()}

    def load_state_dict(self, sd):
        if int(sd["n"]) != self.flat.n:
            raise ValueError(f"optimizer state holds {sd['n']} elements, this model's flat buffer {self.flat.n}")
        self.step_count = int(sd["step"])
        self.lr0 = float(sd["lr0"])
        self.flat.exp_avg.copy_(sd["exp_avg"])
        self.flat.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.sync_replicas()

    def training_step(self, batch, starts=None, pretrain: bool = False) -> Dict[str, float]:
        terms = self.forward_backward_pretrain(batch, starts) if pretrain else self.forward_backward(batch, starts)
        world = self.all_reduce_grads()
        terms["lr"] = self.optimizer_step(world)
        return terms
