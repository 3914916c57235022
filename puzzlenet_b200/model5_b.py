"""Drop-in for the live part of the reference's ``model5_b`` (the "PuzzleNet forward").

Mirrors, with identical names, constructor arguments, ``state_dict`` keys and return
conventions:

* ``scaled_dot_production(q, k, v, mask=None)``            model5_b.py:67-75
* ``layerAttention(config, embed_dim)``                    model5_b.py:83-101
* ``PCTransformer_nonsort(config, num_points=1024)``       model5_b.py:411-478
* ``BiDecoderNoneCross(config)`` (parameters only)         model5_b.py:325-352
* ``TouchedRegraster(config)`` with ``predict5`` / ``predict6`` / ``forward`` / ``test_step`` /
  ``chamfer_loss`` / ``comp`` / ``compute_metrics``        model5_b.py:519-759, :612-668, :1292-1358, :1426-1519

Parameters live in ordinary ``nn.Linear`` / ``nn.BatchNorm1d`` modules so that a reference
checkpoint's ``state_dict`` loads unchanged, but ``forward`` never calls them: compute goes
through ``libpuzzlenet_sm100.so`` (hand-written sm_100a kernels, C ABI in
``include/puzzlenet_b200.h``).  CUDA only; no eager fallback.

Deviations from the reference, all documented in DESIGN.md:
* ``TouchedRegraster.forward`` delegates to ``predict5`` (the reference's ``forward`` calls the
  broken ``predict4``, SURVEY.md D2).
* ``training_step`` runs forward, losses, the hand-written backward, the gradient all-reduce and Adam itself
  (``puzzlenet_b200/training.py``; Lightning: manual optimization).  By default ``predict5(training=True)`` is the
  train-mode forward without an autograd graph and ``predict6(training=True)`` raises; with the opt-in
  ``differentiable = True`` both record a graph whose backward runs the same hand-written kernels
  (``puzzlenet_b200/autograd.py``), so a custom loss trains with ``loss.backward()`` and any ``torch.optim``
  optimizer.
* The class derives from ``nn.Module`` when ``pytorch_lightning`` is not installed.
"""
from __future__ import annotations

import ctypes
import math

import torch
import torch.nn as nn

from . import _lib
from . import losses, metrics
from . import se3 as se3  # noqa: F401  (model5_b.py:13 exposes se3 the same way)
from . import pointnet_util as pu

try:  # pragma: no cover - depends on the environment
    import pytorch_lightning as pl
    _Base = pl.LightningModule
except Exception:  # pytorch_lightning is not part of this image
    _Base = nn.Module

PRECISIONS = {"fp32": _lib.PZ_PREC_FP32, "bf16": _lib.PZ_PREC_BF16, "split": _lib.PZ_PREC_SPLIT}
PACKED_PRECISIONS = ("bf16", "split")     # precisions whose converted weight packs live in the caller's workspace


class _Workspace:
    """A predict5 workspace and the key of the weight packs it currently holds (None: no valid pack)."""
    __slots__ = ("buf", "pack_key")

    def __init__(self, buf: torch.Tensor):
        self.buf = buf
        self.pack_key = None


def _ptr(t):
    return None if t is None else t.data_ptr()


def _param(t: torch.Tensor) -> torch.Tensor:
    _lib.require_cuda(t)
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise TypeError("puzzlenet_b200 expects contiguous float32 parameters")
    return t


def scaled_dot_production(q, k, v, mask=None):
    """model5_b.py:67-75 -> (values, attention)."""
    if mask is not None:
        raise NotImplementedError("mask is unused on the live path (model5_b.py:97 calls it with mask=None)")
    _lib.require_cuda(q, k, v)
    q, k, v = q.contiguous().float(), k.contiguous().float(), v.contiguous().float()
    lead = q.shape[:-2]
    L, Dk, Dv = q.shape[-2], q.shape[-1], v.shape[-1]
    B = int(math.prod(lead)) if lead else 1
    values = torch.empty(*lead, L, Dv, device=q.device, dtype=torch.float32)
    attention = torch.empty(*lead, L, L, device=q.device, dtype=torch.float32)
    with torch.cuda.device(q.device):
        _lib.call("pz_scaled_dot_attention", q.data_ptr(), k.data_ptr(), v.data_ptr(), B, L, Dk, Dv,
                  values.data_ptr(), attention.data_ptr(), _lib.stream_ptr())
    return values, attention


class layerAttention(nn.Module):
    """model5_b.py:83-101 -- offset attention: ``x + relu(out(x - softmax(qk^T/sqrt(d)) v))``."""

    def __init__(self, config, embed_dim) -> None:
        super().__init__()
        self.C = config
        self.mlpq = nn.Linear(embed_dim, embed_dim // 4)
        self.mlpk = nn.Linear(embed_dim, embed_dim // 4)
        self.mlpv = nn.Linear(embed_dim, embed_dim)
        self.out = nn.Linear(embed_dim, embed_dim)
        self.precision = "fp32"

    def forward(self, xyz):
        _lib.require_cuda(xyz)
        x = xyz.contiguous().float()
        B, L, Cc = x.shape
        lib = _lib.load()
        ws_bytes = lib.pz_offset_attention_workspace_bytes(B, L, Cc)
        ws = torch.empty(max(ws_bytes, 1), device=x.device, dtype=torch.uint8)
        out = torch.empty_like(x)
        attn = torch.empty(B, L, L, device=x.device, dtype=torch.float32)
        p = [_param(t).data_ptr() for t in (self.mlpq.weight, self.mlpq.bias, self.mlpk.weight, self.mlpk.bias,
                                            self.mlpv.weight, self.mlpv.bias, self.out.weight, self.out.bias)]
        with torch.cuda.device(x.device):
            _lib.call("pz_offset_attention", x.data_ptr(), *p, B, L, Cc, PRECISIONS[self.precision], out.data_ptr(),
                      attn.data_ptr(), ws.data_ptr(), ws_bytes, _lib.stream_ptr())
        return out, attn


def _encoder_struct(enc: "PCTransformer_nonsort") -> _lib.PzEncoderWeights:
    w = _lib.PzEncoderWeights()
    for name in ("mlp1", "mlp2", "mlp3", "mlp4", "mlp5", "mlp6"):
        lin = getattr(enc, name)
        setattr(w, f"{name}_w", _param(lin.weight).data_ptr())
        setattr(w, f"{name}_b", _param(lin.bias).data_ptr())
    for i in (1, 2):
        bn = getattr(enc, f"bn{i}")
        setattr(w, f"bn{i}_w", _param(bn.weight).data_ptr())
        setattr(w, f"bn{i}_b", _param(bn.bias).data_ptr())
        setattr(w, f"bn{i}_mean", _param(bn.running_mean).data_ptr())
        setattr(w, f"bn{i}_var", _param(bn.running_var).data_ptr())
    for l in range(4):
        att = getattr(enc, f"atten{l + 1}")
        for short, lin in (("q", att.mlpq), ("k", att.mlpk), ("v", att.mlpv), ("o", att.out)):
            getattr(w, f"{short}_w")[l] = _param(lin.weight).data_ptr()
            getattr(w, f"{short}_b")[l] = _param(lin.bias).data_ptr()
    w.out_w = _param(enc.out.weight).data_ptr()
    w.out_b = _param(enc.out.bias).data_ptr()
    return w


class PCTransformer_nonsort(nn.Module):
    """model5_b.py:411-478.  ``forward(xyz [B,1024,3])`` ->
    ``(f_global [B,1024], x2 [B,256,3], attention [B,256,256], out [B,256,1024], x_feature [B,1024,64])``."""

    def __init__(self, config, num_points=1024) -> None:
        super().__init__()
        self.C = config
        feature_size = 64
        gs2_feature_size = 128
        self.mlp1 = nn.Linear(3, 64)
        self.mlp2 = nn.Linear(64, feature_size)
        self.mlp3 = nn.Linear(feature_size + 3, 128)
        self.mlp4 = nn.Linear(128, gs2_feature_size)
        self.mlp5 = nn.Linear(gs2_feature_size + 3, gs2_feature_size * 2)
        self.mlp6 = nn.Linear(gs2_feature_size * 2, gs2_feature_size * 2)
        self.bn1 = nn.BatchNorm1d(num_points)
        self.bn2 = nn.BatchNorm1d(num_points)
        self.sg1 = pu.sample_and_group          # model5_b.py:427-429 stores the function objects
        self.fps = pu.farthest_point_sample
        self.sg2 = pu.sample_and_group
        self.atten1 = layerAttention(self.C, gs2_feature_size * 2)
        self.atten2 = layerAttention(self.C, gs2_feature_size * 2)
        self.atten3 = layerAttention(self.C, gs2_feature_size * 2)
        self.atten4 = layerAttention(self.C, gs2_feature_size * 2)
        self.out = nn.Linear(gs2_feature_size * 2 * 5, 1024)
        self.num_points = num_points
        self.precision = "fp32"

    def forward(self, xyz, return_intermediates: bool = False):
        if self.training:
            raise NotImplementedError("a standalone PCTransformer_nonsort only runs in eval mode; the train-mode "
                                      "forward/backward lives in TouchedRegraster.training_step "
                                      "(puzzlenet_b200/training.py)")
        _lib.require_cuda(xyz)
        x = xyz.contiguous().float()
        if x.dim() != 3 or x.shape[1] != 1024 or x.shape[2] != 3:
            raise ValueError(f"PCTransformer_nonsort expects [B,1024,3] (BatchNorm1d(1024) pins N); got {tuple(x.shape)}")
        B = x.shape[0]
        dev = x.device
        # the reference draws the two FPS starts inside sample_and_group, stage 1 then stage 2
        start1 = torch.randint(0, 1024, (B,), dtype=torch.long).to(dev)
        start2 = torch.randint(0, 512, (B,), dtype=torch.long).to(dev)
        f32 = dict(device=dev, dtype=torch.float32)
        res = dict(f_global=torch.empty(B, 1024, **f32), x2=torch.empty(B, 256, 3, **f32),
                   attention=torch.empty(B, 256, 256, **f32), out=torch.empty(B, 256, 1024, **f32),
                   x_feature=torch.empty(B, 1024, 64, **f32))
        if return_intermediates:
            i64 = dict(device=dev, dtype=torch.int64)
            res.update(fps1=torch.empty(B, 512, **i64), knn1=torch.empty(B, 512, 32, **i64),
                       f1f=torch.empty(B, 512, 128, **f32), fps2=torch.empty(B, 256, **i64),
                       knn2=torch.empty(B, 256, 32, **i64), f2f=torch.empty(B, 256, 256, **f32),
                       att_cat=torch.empty(B, 256, 1280, **f32))
        outs = _lib.PzEncoderOutputs()
        for k, v in res.items():
            setattr(outs, k, v.data_ptr())
        w = _encoder_struct(self)
        lib = _lib.load()
        ws_bytes = lib.pz_encoder_workspace_bytes(1, B)
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
        with torch.cuda.device(dev):
            _lib.call("pz_encoder_forward", ctypes.byref(w), 1, B, x.data_ptr(), start1.data_ptr(), start2.data_ptr(),
                      PRECISIONS[self.precision], ctypes.byref(outs), ws.data_ptr(), ws_bytes, _lib.stream_ptr())
        if return_intermediates:
            return res
        return res["f_global"], res["x2"], res["attention"], res["out"], res["x_feature"]


class BiDecoderNoneCross(nn.Module):
    """model5_b.py:325-352 -- instantiated by TouchedRegraster (:537-538) but never called on the live
    path; kept so checkpoints load (``fpc_decoder.*`` / ``rpc_decoder.*`` keys)."""

    def __init__(self, config, num_points=1024) -> None:
        super().__init__()
        self.C = config
        self.mlp1 = nn.Linear(512, 512)
        self.mlp2 = nn.Linear(512, 256)
        self.mlp3 = nn.Linear(256, 2)

    def forward(self, f_local, f_global):
        raise NotImplementedError("BiDecoderNoneCross is unused by predict5 (model5_b.py:732-736 are commented out)")


def _seq(*sizes):
    layers = []
    for i in range(len(sizes) - 1):
        layers.append(nn.Linear(sizes[i], sizes[i + 1]))
        if i + 2 < len(sizes):
            layers.append(nn.ReLU())
    return nn.Sequential(*layers)


def _draw_starts(B: int) -> torch.Tensor:
    """predict5's four FPS-start draws on the CPU generator, in the reference's order -> int64 [4,B]."""
    return torch.stack([torch.randint(0, 1024, (B,), dtype=torch.long),
                        torch.randint(0, 512, (B,), dtype=torch.long),
                        torch.randint(0, 1024, (B,), dtype=torch.long),
                        torch.randint(0, 512, (B,), dtype=torch.long)])


def _pieces_arg(clouds) -> torch.Tensor:
    _lib.require_cuda(clouds)
    clouds = clouds.contiguous().float()
    if clouds.dim() != 3 or clouds.shape[0] < 1 or clouds.shape[1:] != (1024, 3):
        raise ValueError(f"expected pieces [P,1024,3] with P >= 1; got {tuple(clouds.shape)}")
    return clouds


ENCODE_CHUNK = 64     # pieces per pz_encode_pieces call: bounds the workspace (that of predict5 with B = 64)
PAIR_CHUNK = 4096     # pairs per pz_predict_pairs call: bounds its workspace (~70 MB)


class PieceEmbeddings:
    """Per-piece state of :meth:`TouchedRegraster.encode_pieces` (layout: ``PzPieceEmbeddings`` in
    include/puzzlenet_b200.h): ``f_global [2,P,1024]``, ``local [2,P,1024,64]``, ``tilemax [2,P,8,64]`` (role 0 = the
    piece as fpc, role 1 = as mrpc), ``de_mrpcb [P,2,1024]``, plus the FPS ``starts [4,P]`` (CPU) they were encoded
    with, the precision, the device and the model's weights key (``TouchedRegraster._weights_key``) at encode time."""

    def __init__(self, P: int, device, starts, precision: str, param_key):
        starts = torch.as_tensor(starts)
        if starts.shape != (4, P):
            raise ValueError(f"starts must be [4,{P}]; got {tuple(starts.shape)}")
        f32 = dict(device=device, dtype=torch.float32)
        self.f_global = torch.empty(2, P, 1024, **f32)
        self.local = torch.empty(2, P, 1024, 64, **f32)
        self.tilemax = torch.empty(2, P, 8, 64, **f32)
        self.de_mrpcb = torch.empty(P, 2, 1024, **f32)
        self.starts = starts.to("cpu", torch.int64).clone()
        self.precision = precision
        self.device = torch.device(device)
        self.param_key = param_key

    @property
    def P(self) -> int:
        return self.de_mrpcb.shape[0]

    def struct(self) -> _lib.PzPieceEmbeddings:
        return _lib.PzPieceEmbeddings(self.f_global.data_ptr(), self.local.data_ptr(), self.tilemax.data_ptr(),
                                      self.de_mrpcb.data_ptr())

    def is_current(self, model) -> bool:
        """False once the model's parameters or precision changed after these embeddings were encoded."""
        return model.precision == self.precision and model._weights_key() == self.param_key

    def _check_current(self, model):
        if not self.is_current(model):
            raise ValueError("these piece embeddings are stale: the model's parameters or precision changed since "
                             "they were encoded (encode the pieces again)")

    def reencode(self, model, rows, clouds, starts=None) -> None:
        """Encode ``clouds [k,1024,3]`` again as pieces ``rows`` (k indices in ``[0,P)``), in place; ``starts [4,k]``
        default to predict5's draws for ``B = k``.  The model must be the one the embeddings were built with."""
        self._check_current(model)
        rows = [int(r) for r in rows]
        if any(r < 0 or r >= self.P for r in rows):
            raise IndexError(f"reencode: piece index outside [0, {self.P})")
        clouds = _pieces_arg(clouds)
        if clouds.shape[0] != len(rows):
            raise ValueError("reencode: one cloud per row")
        starts = _draw_starts(len(rows)) if starts is None else torch.as_tensor(starts).to(torch.int64)
        self.starts[:, rows] = starts
        self._encode(model, clouds, starts.to(self.device, non_blocking=True), rows)

    def _encode(self, model, clouds, starts, rows):
        """pz_encode_pieces over ``clouds`` (device starts [4,k]) into pieces ``rows``, ENCODE_CHUNK pieces a call;
        a call that covers every piece in order writes straight into the tensors, others go through a chunk buffer."""
        for m in (model.Encoder, model.Encoder2, model.tfMLP, model.fpc_decoder, model.rpc_decoder):
            m.eval()
        enc = (_lib.PzEncoderWeights * 2)(_encoder_struct(model.Encoder), _encoder_struct(model.Encoder2))
        heads = model._head_struct()
        for lo in range(0, len(rows), ENCODE_CHUNK):
            sel = rows[lo:lo + ENCODE_CHUNK]
            k = len(sel)
            direct = sel == list(range(self.P))
            dst = self if direct else PieceEmbeddings(k, self.device, self.starts[:, sel], self.precision, self.param_key)
            ws = model._workspace(k, self.device, "pz_encode_pieces")
            flags = _lib.PZ_FLAG_REUSE_PACKS if model._packs_reusable(ws) else 0
            with torch.cuda.device(self.device):
                _lib.call("pz_encode_pieces", enc, ctypes.byref(heads), clouds[lo:lo + k].data_ptr(), k,
                          starts[:, lo:lo + k].contiguous().data_ptr(), PRECISIONS[self.precision], flags,
                          ctypes.byref(dst.struct()), ws.buf.data_ptr(), ws.buf.numel(), _lib.stream_ptr())
            if not direct:
                idx = torch.tensor(sel, device=self.device)
                self.f_global[:, idx] = dst.f_global
                self.local[:, idx] = dst.local
                self.tilemax[:, idx] = dst.tilemax
                self.de_mrpcb[idx] = dst.de_mrpcb


class TouchedRegraster(_Base):
    """model5_b.py:519-759.  ``predict5(batch, batch_indic, need=False, training=False)`` is the forward
    that train/test execute; ``batch`` is the 8-tuple ``(fpc, mrpc, igt, rpc, fpcb, mrpcb, fpc_idx, rpc_idx)``
    of which only ``[0]`` and ``[1]`` (both [B,1024,3]) are computed on."""

    def __init__(self, config):
        super().__init__()
        if hasattr(self, "save_hyperparameters"):
            try:
                self.save_hyperparameters()
            except Exception:  # pragma: no cover
                pass
        self.C = config
        self.Encoder = PCTransformer_nonsort(config)
        self.Encoder2 = PCTransformer_nonsort(config)
        self.fpc_decoder = BiDecoderNoneCross(config)
        self.rpc_decoder = BiDecoderNoneCross(config)
        self.dt = nn.Parameter(torch.full((1, 6), 1.0e-2), requires_grad=True)   # model5_b.py:541-543
        self.tfMLP = _seq(2048, 1024, 512, 512, 256, 6)
        self.MLPLocalPreRpc = _seq(64, 64, 64, 64)
        self.MLPLocalPreFpc = _seq(64, 64, 64, 64)
        self.MLPRpcb = _seq(128, 64, 32, 2)
        self.MLPFpcb = _seq(128, 64, 32, 2)
        self.precision = "fp32"
        self._ws = {}
        self._graphs = {}
        self._capture_stream = None
        self._trainer_state = None
        self._weights_generation = 0  # bumped whenever the weights change behind torch's back (see _weights_key)
        self.cuda_graphs = False      # opt-in: replay one captured CUDA graph per forward (see _graph_replay)
        self.differentiable = False   # opt-in: training=True forwards record an autograd graph (puzzlenet_b200/autograd.py)
        self.graph_static_outputs = False   # True: return the graph's own output buffers (overwritten by the next replay)
        self.max_graphs = 16          # captured graphs kept (one per batch size, need, precision, device, stream); LRU

    # ---- weights as C structs (rebuilt per call: ~100 data_ptr() reads, no device work)
    def _head_struct(self) -> _lib.PzHeadWeights:
        h = _lib.PzHeadWeights()
        for j, li in enumerate((0, 2, 4, 6, 8)):
            h.tf_w[j] = _param(self.tfMLP[li].weight).data_ptr()
            h.tf_b[j] = _param(self.tfMLP[li].bias).data_ptr()
        for field, mod in (("pre_fpc", self.MLPLocalPreFpc), ("pre_rpc", self.MLPLocalPreRpc),
                           ("seg_fpc", self.MLPFpcb), ("seg_rpc", self.MLPRpcb)):
            for j, li in enumerate((0, 2, 4)):
                getattr(h, f"{field}_w")[j] = _param(mod[li].weight).data_ptr()
                getattr(h, f"{field}_b")[j] = _param(mod[li].bias).data_ptr()
        return h

    def _workspace(self, B: int, device, kind: str = "pz_predict5") -> "_Workspace":
        """One workspace per (entry point, batch size, device, CUDA stream): calls issued on different streams may
        overlap on the GPU (a pipelined caller alternates streams), so they must not share scratch.  At most four are
        kept per entry point.  The validity of the bf16 / split weight packs stored inside a workspace is a property
        of the workspace OBJECT (``_Workspace.pack_key``), never of its address: an evicted workspace takes its key
        with it, so a block the caching allocator hands to a workspace of another batch size (other pack offset) can
        never be taken for a packed one."""
        key = (kind, B, str(device), torch.cuda.current_stream(device).cuda_stream)
        ws = self._ws.get(key)
        if ws is None:
            nbytes = getattr(_lib.load(), kind + "_workspace_bytes")(B)
            ws = _Workspace(torch.empty(nbytes, device=device, dtype=torch.uint8))
            same = [k for k in self._ws if k[0] == kind]
            if len(same) >= 4:
                self._ws.pop(same[0])
            self._ws[key] = ws
        return ws

    def _param_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def _weights_key(self):
        """Identifies the weights state that piece embeddings were computed from: ``_param_key`` misses writes that
        bypass torch (the Trainer's Adam step, parameter broadcasts, train-mode BatchNorm statistics), so those bump
        ``_weights_generation`` (``Trainer._invalidate_inference_state``)."""
        return self._param_key(), self._weights_generation

    def _packs_reusable(self, ws: "_Workspace", shared: bool = False) -> bool:
        """Whether the weight packs inside ``ws`` are still valid, and record that they will be after this call: they
        are reusable while no parameter was touched (in-place writes bump _version, reallocation changes data_ptr) and
        the workspace object / precision are the same."""
        if self.precision not in PACKED_PRECISIONS:
            ws.pack_key = None
            return False
        key = (self._param_key(), shared, self.precision)
        reuse = ws.pack_key == key
        ws.pack_key = key
        return reuse

    def _launch(self, fpc, mrpc, starts, need, ws, outs, reuse_packs=None, shared=False):
        """Allocate (unless given) the outputs and the workspace and enqueue pz_predict5 on the current stream.
        ``shared``: both clouds go through ``self.Encoder`` (predict6, model5_b.py:647-653)."""
        B, dev = fpc.shape[0], fpc.device
        f32 = dict(device=dev, dtype=torch.float32)
        if outs is None:
            out6, de_fpcb, de_mrpcb = torch.empty(B, 6, **f32), torch.empty(B, 2, 1024, **f32), torch.empty(B, 2, 1024, **f32)
            x2f = x2m = af = am = None
            if need:
                x2f, x2m = torch.empty(B, 256, 3, **f32), torch.empty(B, 256, 3, **f32)
                af, am = torch.empty(B, 256, 256, **f32), torch.empty(B, 256, 256, **f32)
            outs = (out6, de_fpcb, de_mrpcb, x2f, af, x2m, am)
        out6, de_fpcb, de_mrpcb, x2f, af, x2m, am = outs
        enc = (_lib.PzEncoderWeights * 2)(_encoder_struct(self.Encoder),
                                          _encoder_struct(self.Encoder if shared else self.Encoder2))
        heads = self._head_struct()
        if ws is None:
            ws = self._workspace(B, dev)
        flags = _lib.PZ_FLAG_NEED if need else 0
        if reuse_packs is None:
            reuse_packs = self._packs_reusable(ws, shared)
        elif self.precision not in PACKED_PRECISIONS:
            ws.pack_key = None
        if reuse_packs:
            flags |= _lib.PZ_FLAG_REUSE_PACKS
        with torch.cuda.device(dev):
            _lib.call("pz_predict5", enc, ctypes.byref(heads), fpc.data_ptr(), mrpc.data_ptr(), B, starts.data_ptr(),
                      PRECISIONS[self.precision], flags, out6.data_ptr(), de_fpcb.data_ptr(),
                      de_mrpcb.data_ptr(), _ptr(x2f), _ptr(af), _ptr(x2m), _ptr(am), ws.buf.data_ptr(), ws.buf.numel(),
                      _lib.stream_ptr())
        return outs

    def _graph_replay(self, fpc, mrpc, starts, need, shared=False):
        """CUDA-graph mode (``model.cuda_graphs = True``): the 22 launches of one forward (both streams of the
        internal fork/join included) are captured once per (batch size, need, precision, stream) and replayed.
        Inputs are copied into static buffers; the results are copied out of the graph's static output buffers into
        fresh tensors (``graph_static_outputs = True`` returns the static buffers themselves: they are overwritten by
        the next call on the same stream).  A change of any parameter re-captures; at most ``max_graphs`` graphs are
        kept, least recently used first out."""
        B, dev = fpc.shape[0], fpc.device
        stream = torch.cuda.current_stream(dev)
        key = (B, bool(need), self.precision, str(dev), stream.cuda_stream, shared)
        g = self._graphs.get(key)
        pkey = self._param_key()
        if g is None or g["pkey"] != pkey:
            f32 = dict(device=dev, dtype=torch.float32)
            st = dict(fpc=torch.empty(B, 1024, 3, **f32), mrpc=torch.empty(B, 1024, 3, **f32),
                      starts=torch.empty(4, B, device=dev, dtype=torch.int64),
                      ws=_Workspace(torch.empty(_lib.load().pz_predict5_workspace_bytes(B), device=dev,
                                                dtype=torch.uint8)))
            st["fpc"].copy_(fpc); st["mrpc"].copy_(mrpc); st["starts"].copy_(starts)
            outs = self._launch(st["fpc"], st["mrpc"], st["starts"], need, st["ws"], None, reuse_packs=False,
                                shared=shared)                                           # builds the packs
            stream.synchronize()
            graph = torch.cuda.CUDAGraph()
            cap = stream
            if stream.cuda_stream == 0:          # capture is not allowed on the legacy default stream
                if self._capture_stream is None:
                    self._capture_stream = torch.cuda.Stream(device=dev)
                cap = self._capture_stream
            with torch.cuda.graph(graph, stream=cap):
                self._launch(st["fpc"], st["mrpc"], st["starts"], need, st["ws"], outs,
                             reuse_packs=self.precision in PACKED_PRECISIONS, shared=shared)
            g = dict(pkey=pkey, st=st, outs=outs, graph=graph)
            self._graphs.pop(key, None)
            while len(self._graphs) >= self.max_graphs:          # evict the least recently used entry, not the whole cache
                self._graphs.pop(next(iter(self._graphs)))
            self._graphs[key] = g
        else:
            self._graphs[key] = self._graphs.pop(key)             # mark as most recently used
        st = g["st"]
        st["fpc"].copy_(fpc, non_blocking=True)
        st["mrpc"].copy_(mrpc, non_blocking=True)
        st["starts"].copy_(starts, non_blocking=True)
        g["graph"].replay()
        if self.graph_static_outputs:
            return g["outs"]
        # fresh tensors, like the reference (and like eager mode): the graph's own output buffers are overwritten by the
        # next replay on this stream, so a caller that keeps two results alive must not see them alias
        return tuple(None if t is None else t.clone() for t in g["outs"])

    def forward(self, batch, bat):
        # The reference's forward() calls predict4, which needs modules that are commented out of
        # __init__ (SURVEY.md D2) and raises AttributeError; predict5 is what train/test run.
        return self.predict5(batch, bat)

    def predict5(self, batch, batch_indic, need=False, training=False, starts=None):
        """model5_b.py:672-759.  ``starts`` (optional, not in the reference): int64 [4,B] FPS start
        indices in the reference's draw order; when omitted the four ``torch.randint`` draws are taken
        from the CPU generator exactly as the reference does (SURVEY.md Appendix A).  ``training=True`` runs the
        train-mode forward in the Trainer's precision; with ``differentiable`` set and grad mode on, its outputs
        (``x2_*`` / ``attention_*`` too) are connected to autograd: the parameters and, when they require grad, the
        clouds receive gradients."""
        if training:
            # train-mode forward (model5_b.py:684-690: batch-statistics BatchNorm, running stats updated)
            _lib.require_cuda(batch[0], batch[1])
            self._train_mode()
            if self.differentiable and torch.is_grad_enabled():
                from .autograd import train_forward
                out6, de_f, de_m, x2f, af, x2m, am = train_forward(self.trainer_state(), batch[0], batch[1], starts,
                                                                   need)
                r = (out6, [0], x2f, af, x2m, am, de_f, de_m)
            else:
                r = self.trainer_state().predict5_train(batch[0], batch[1], starts)
            return r if need else (r[0], r[0], r[6], r[7])
        return self._predict(batch, need, starts, shared=False)

    def _train_mode(self):
        for mod in (self.Encoder, self.Encoder2, self.tfMLP, self.fpc_decoder, self.rpc_decoder):
            mod.train()

    def predict6(self, batch, batch_indic, need=False, training=False, pretrain=False, starts=None):
        """model5_b.py:612-668 -- the pretraining forward: BOTH clouds go through ``self.Encoder`` and only the pose
        is predicted.  ``pretrain=False`` reaches ``self.Decoder`` / ``self.mrpcbDecoder`` in the reference, which
        its constructor does not create (AttributeError there); it raises here as well.  ``training=True`` needs
        ``differentiable`` (the train-mode forward with an autograd graph, as in predict5; ``Encoder`` is applied
        twice and its gradients from the two passes add)."""
        if training and not self.differentiable:
            raise NotImplementedError("puzzlenet_b200.predict6(training=True) needs model.differentiable = True; "
                                      "otherwise the pretraining branch trains through training_step(pretrain=True)")
        if not pretrain:
            raise AttributeError("'TouchedRegraster' object has no attribute 'Decoder' (model5_b.py:661: predict6 "
                                 "only works with pretrain=True)")
        if training:
            _lib.require_cuda(batch[0], batch[1])
            self._train_mode()
            from .autograd import train_forward
            out6, _, _, x2f, af, x2m, am = train_forward(self.trainer_state(), batch[0], batch[1], starts, need,
                                                         pretrain=True)
            return (out6, [0], x2f, af, x2m, am) if need else out6
        r = self._predict(batch, need, starts, shared=True)
        if not need:
            return r[0]
        return r[0], [0], r[2], r[3], r[4], r[5]

    # ---- pair scoring from per-piece encodings (not in the reference): predict5 split at its pair boundary
    def encode_pieces(self, clouds, starts=None) -> "PieceEmbeddings":
        """Everything ``predict5`` computes per cloud, once per piece: both encoders, ``MLPLocalPre{Fpc,Rpc}`` and the
        mrpc boundary head (``pz_encode_pieces``).  ``clouds [P,1024,3]`` on the GPU; ``starts`` int64 [4,P] FPS starts
        in predict5's order (Encoder s1, Encoder s2, Encoder2 s1, Encoder2 s2) -- when omitted they are drawn exactly
        as ``predict5`` with ``B = P`` draws them, so ``encode_pieces(c)`` consumes the same random numbers as
        ``predict5(make_batch(c, c), P)``.  Eval mode only; pieces are encoded in chunks of at most
        ``ENCODE_CHUNK``."""
        clouds = _pieces_arg(clouds)
        P, dev = clouds.shape[0], clouds.device
        starts = _draw_starts(P) if starts is None else starts
        emb = PieceEmbeddings(P, dev, starts, self.precision, self._weights_key())
        emb._encode(self, clouds, emb.starts.to(dev, non_blocking=True), list(range(P)))
        return emb

    def predict_pairs(self, emb: "PieceEmbeddings", pairs):
        """``(out6, out6, de_fpcb, de_mrpcb)`` -- what ``predict5(need=False)`` returns for the pairs
        ``(clouds[i], clouds[j])`` of ``pairs [n,2]`` (i = fpc piece, j = mrpc piece) with the pieces' FPS starts, from
        the embeddings of :meth:`encode_pieces` (``pz_predict_pairs``: the pose MLP and the fpc boundary head only).
        Raises ``IndexError`` for an index outside ``[0,P)`` and ``ValueError`` when the parameters or the precision
        changed since ``emb`` was built."""
        emb._check_current(self)
        pairs = torch.as_tensor(pairs)
        if pairs.dim() != 2 or pairs.shape[1] != 2 or pairs.dtype.is_floating_point:
            raise ValueError(f"predict_pairs expects integer pairs [n,2]; got {pairs.dtype} {tuple(pairs.shape)}")
        n = pairs.shape[0]
        if n:
            lo, hi = (int(v) for v in torch.aminmax(pairs))       # one host synchronisation for device pairs
            if lo < 0 or hi >= emb.P:
                raise IndexError(f"predict_pairs: piece index {lo if lo < 0 else hi} outside [0, {emb.P})")
        pairs = pairs.to(device=emb.device, dtype=torch.int64, non_blocking=True).contiguous()
        f32 = dict(device=emb.device, dtype=torch.float32)
        out6, de_fpcb, de_mrpcb = torch.empty(n, 6, **f32), torch.empty(n, 2, 1024, **f32), torch.empty(n, 2, 1024, **f32)
        for lo in range(0, n, PAIR_CHUNK):
            hi = min(n, lo + PAIR_CHUNK)
            self._launch_pairs(emb, pairs[lo:hi], out6[lo:hi], de_fpcb[lo:hi], de_mrpcb[lo:hi])
        return out6, out6, de_fpcb, de_mrpcb

    def _launch_pairs(self, emb, pairs, out6, de_fpcb, de_mrpcb):
        """Enqueue pz_predict_pairs on the current stream (no checks: ``pairs`` int64 [n,2] on emb's device, in range);
        CUDA-graph capturable once the workspace's weight images are built."""
        n = pairs.shape[0]
        ws = self._workspace(max(64, 1 << (n - 1).bit_length()), emb.device, "pz_predict_pairs")
        flags = _lib.PZ_FLAG_REUSE_PACKS if self._packs_reusable(ws) else 0
        heads = self._head_struct()
        with torch.cuda.device(emb.device):
            _lib.call("pz_predict_pairs", ctypes.byref(heads), ctypes.byref(emb.struct()), emb.P, pairs.data_ptr(), n,
                      PRECISIONS[self.precision], flags, out6.data_ptr(), de_fpcb.data_ptr(), de_mrpcb.data_ptr(),
                      ws.buf.data_ptr(), ws.buf.numel(), _lib.stream_ptr())

    def _predict(self, batch, need, starts, shared):
        for m in (self.Encoder, self.Encoder2, self.tfMLP, self.fpc_decoder, self.rpc_decoder):
            m.eval()                                              # model5_b.py:677-683
        fpc, mrpc = batch[0], batch[1]
        _unused = (batch[2], batch[3], batch[4], batch[5], batch[6], batch[7])    # model5_b.py:693-699 index them
        if fpc.dim() == 2:
            fpc, mrpc = fpc.unsqueeze(0), mrpc.unsqueeze(0)
        _lib.require_cuda(fpc, mrpc)
        fpc, mrpc = fpc.contiguous().float(), mrpc.contiguous().float()
        if fpc.shape[1:] != (1024, 3) or mrpc.shape != fpc.shape:
            raise ValueError(f"predict5 expects two [B,1024,3] clouds; got {tuple(fpc.shape)} and {tuple(mrpc.shape)}")
        B, dev = fpc.shape[0], fpc.device
        if starts is None:
            starts = _draw_starts(B)
        starts = starts.to(device=dev, dtype=torch.int64, non_blocking=True).contiguous()
        if self.cuda_graphs:
            out6, de_fpcb, de_mrpcb, x2f, af, x2m, am = self._graph_replay(fpc, mrpc, starts, need, shared)
        else:
            out6, de_fpcb, de_mrpcb, x2f, af, x2m, am = self._launch(fpc, mrpc, starts, need, None, None,
                                                                     shared=shared)
        if not need:
            return out6, out6, de_fpcb, de_mrpcb
        return out6, [0], x2f, af, x2m, am, de_fpcb, de_mrpcb

    # ---- training (model5_b.py:912-1155, :1453-1457)
    automatic_optimization = False     # Lightning: training_step below runs backward + optimizer itself

    def trainer_state(self):
        """The :class:`puzzlenet_b200.training.Trainer` bound to this model (created on first use: it re-homes the
        live parameters into one flat buffer; options are read from ``self.C``)."""
        if getattr(self, "_trainer_state", None) is None:
            from .training import Trainer
            self._trainer_state = Trainer(self, self.C)
        return self._trainer_state

    def training_step(self, batch, batch_indic, starts=None, pretrain=None):
        """model5_b.py:912-1155 (non-pretrain branch) + the optimizer step of :1453-1457.  The reference returns a
        loss for autograd; there is no autograd graph here -- forward, losses, the hand-written backward, the
        gradient all-reduce and Adam all happen inside this call (Lightning: manual optimization).  Returns
        ``{'loss': 0-d tensor, 'terms': dict of the logged scalars}``."""
        if pretrain is None:      # model5_b.py:928: pretrain = self.current_epoch < self.C.pretrain_epochs
            epoch = getattr(self, "current_epoch", None)
            pretrain = epoch is not None and epoch < getattr(self.C, "pretrain_epochs", 0)
        terms = self.trainer_state().training_step(batch, starts, pretrain=bool(pretrain))
        if hasattr(self, "log"):
            try:
                for k, v in terms.items():
                    self.log("train/" + k, v)
            except Exception:      # outside a Lightning loop self.log raises
                pass
        return {"loss": torch.tensor(terms["loss"]), "terms": terms}

    def configure_optimizers(self):
        """model5_b.py:1453-1457: Adam(lr) + StepLR(50, 0.999) are fused into ``pz_adam_step`` inside
        :meth:`training_step`; nothing is handed to Lightning."""
        return None

    # ---- loss-side helpers and the evaluation step (same names as the reference methods)
    def chamfer_loss(self, a, b):
        """model5_b.py:1495-1505."""
        return losses.chamfer_loss(a, b)

    def comp(self, g, igt):
        """model5_b.py:1512-1519."""
        return losses.comp(g, igt)

    def compute_metrics(self, R, t, igt):
        """model5_b.py:1426-1440 (host-side numpy/scipy, as in the reference's metrics.py)."""
        return metrics.compute_metrics(R, t, igt)

    def test_step(self, batch, batch_idx):
        """model5_b.py:1292-1358 -> ``[1,10]``: mean r_mse, r_mae, t_mse, t_mae, r_isotropic, t_isotropic, then the
        batch IoU of both boundary predictions and the two boundary chamfer distances.  The forward is one
        ``pz_predict5``; everything after it is ONE ``pz_pair_score`` launch plus the host-side Euler-angle
        errors (scipy, exactly as the reference computes them)."""
        batch = ([b.unsqueeze(0) if b.dim() == 2 else b for b in batch[:-2]]             # model5_b.py:1281-1292
                 + [b.unsqueeze(0) if b.dim() == 1 else b for b in batch[-2:]])
        fpc, mrpc, igt, rpc, fpcb, rpcb, fpc_idx, rpc_idx = batch[:8]
        out, _, de_fpcb, de_mrpcb = self.predict5(batch, fpc.shape[0], training=False, need=False)
        s = losses.pair_score(out, de_fpcb, de_mrpcb, fpc, rpc, fpcb, rpcb, fpc_idx, rpc_idx, igt).double()
        mat = se3.exp(out)
        r_mse, r_mae = metrics.anisotropic_R_error(mat[:, :3, :3], igt[:, :3, :3].permute(0, 2, 1))
        m = s.mean(0)
        tot = s.sum(0)
        scores = [float(r_mse.mean()), float(r_mae.mean()), m[2], m[3], m[0], m[1], tot[4] / tot[5], tot[6] / tot[7],
                  m[8], m[9]]
        return torch.stack([torch.as_tensor(v, dtype=torch.float64, device=out.device) for v in scores]).unsqueeze(0)
