"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the PuzzleNet hot path.

A plain torch-CPU (fp32, ATen) restatement of the reference algorithm for the
encoder + pair-matching forward.  It is the checker the CUDA path is compared
with; it is *never* on the product path.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import it.

Pinning: the reference has no golden vectors for this part of the path
(SURVEY.md §8c) -- it is pinned by executing the unmodified reference torch
code in the build container (``oracle/make_golden.py`` -> ``tests/golden/``)
and comparing with those stored outputs (``tests/test_oracle_golden.py``).

Everything is functional: weights come in as a ``state_dict``-style mapping
with the reference's key names (SURVEY.md Appendix C), so the same dictionary
drives the reference model, this oracle and the CUDA implementation.

Each function cites the reference lines it restates (paths are relative to
the reference root).
"""
from __future__ import annotations

import math
from typing import Dict, Mapping, Optional

import torch

Tensor = torch.Tensor

# bench.py's "stock PyTorch on the same GPU" baseline runs these same functions on CUDA tensors (only the placement of
# arange / randint / constants follows the input's device; on CPU tensors nothing changes).  The reference additionally
# calls torch.cuda.empty_cache() five times per sample_and_group; the baseline can switch that on to time the reference
# as written.
REFERENCE_EMPTY_CACHE = False

# --------------------------------------------------------------------------
# point-cloud operators (pointnet_util.py)
# --------------------------------------------------------------------------


def sq_norm3(diff: Tensor) -> Tensor:
    """((dx*dx)+(dy*dy))+(dz*dz), every op rounded to fp32, no FMA.

    This is the arithmetic contract for every distance on the path: ATen's CPU
    ``sum(dim=-1)`` over 3 elements associates left to right (SURVEY.md §8c),
    which is what pointnet_util.py:36 and :70 evaluate.
    """
    sq = diff * diff
    return (sq[..., 0] + sq[..., 1]) + sq[..., 2]


def square_distance(src: Tensor, dst: Tensor) -> Tensor:
    """pointnet_util.py:22-36 -- direct (src-dst)^2 form -> [B, S, N]."""
    return sq_norm3(src.unsqueeze(2) - dst.unsqueeze(1))


def index_points(points: Tensor, idx: Tensor) -> Tensor:
    """pointnet_util.py:39-50 -- batched row gather; idx [B,S] or [B,S,K]."""
    b = points.shape[0]
    flat = idx.reshape(b, -1)
    rows = torch.arange(b, device=points.device).unsqueeze(1)
    return points[rows, flat].reshape(*idx.shape, points.shape[-1])


def draw_fps_start(batch: int, n: int) -> Tensor:
    """pointnet_util.py:65 -- ONE draw from the CPU default generator per call."""
    return torch.randint(0, n, (batch,), dtype=torch.long)


def farthest_point_sample(xyz: Tensor, npoint: int, start: Optional[Tensor] = None) -> Tensor:
    """pointnet_util.py:53-73.

    distance starts at 1e10; each step records the current farthest index,
    lowers ``distance`` with the squared distance to it and picks the argmax
    (first maximum wins, as ``torch.max`` does on CPU).
    """
    b, n, _ = xyz.shape
    dev = xyz.device                      # "cpu" for the oracle proper; a CUDA device only in bench.py's torch-on-GPU baseline
    far = (draw_fps_start(b, n) if start is None else start.clone().long()).to(dev)
    picked = torch.empty(b, npoint, dtype=torch.long, device=dev)
    mind = torch.full((b, n), 1e10, dtype=xyz.dtype, device=dev)
    rows = torch.arange(b, device=dev)
    for s in range(npoint):
        picked[:, s] = far
        c = xyz[rows, far].unsqueeze(1)
        mind = torch.minimum(mind, sq_norm3(xyz - c))
        far = torch.max(mind, dim=-1).indices
    return picked


def knn_select(dists: Tensor, k: int):
    """pointnet_util.py:119 -- ``argsort()[:, :, :k]``.

    The reference's sort is unstable, so the order among equal distances is
    undefined there; the oracle fixes it to (distance, index) ascending with a
    stable sort.  Returns (idx [B,S,k], d2 [B,S,k]).
    """
    vals, idx = torch.sort(dists, dim=-1, stable=True)
    return idx[..., :k], vals[..., :k]


def query_ball_point(radius: float, nsample: int, xyz: Tensor, new_xyz: Tensor) -> Tensor:
    """pointnet_util.py:76-96 -- first ``nsample`` in-radius indices, padded with the first."""
    b, n, _ = xyz.shape
    s = new_xyz.shape[1]
    d2 = square_distance(new_xyz, xyz)
    cand = torch.arange(n, device=xyz.device).view(1, 1, n).expand(b, s, n).clone()
    cand[d2 > radius ** 2] = n
    cand = torch.sort(cand, dim=-1).values[:, :, :nsample]
    first = cand[:, :, :1].expand(-1, -1, nsample)
    return torch.where(cand == n, first, cand)


def sample_and_group(npoint: int, radius: float, nsample: int, xyz: Tensor, points: Optional[Tensor],
                     returnfps: bool = False, knn: bool = False, start: Optional[Tensor] = None,
                     return_idx: bool = False):
    """pointnet_util.py:99-136 -- FPS, centre gather, kNN / ball query, group, centre, concat."""
    b, n, c = xyz.shape
    fps_idx = farthest_point_sample(xyz, npoint, start)
    if REFERENCE_EMPTY_CACHE and xyz.is_cuda:     # pointnet_util.py:114,116,122,124,126 (no-ops on the CPU)
        for _ in range(5):
            torch.cuda.empty_cache()
    new_xyz = index_points(xyz, fps_idx)
    if knn:
        idx, _ = knn_select(square_distance(new_xyz, xyz), nsample)
    else:
        idx = query_ball_point(radius, nsample, xyz, new_xyz)
    grouped_xyz = index_points(xyz, idx)
    rel = grouped_xyz - new_xyz.view(b, npoint, 1, c)
    new_points = rel if points is None else torch.cat([rel, index_points(points, idx)], dim=-1)
    if return_idx:
        return new_xyz, new_points, grouped_xyz, fps_idx, idx
    if returnfps:
        return new_xyz, new_points, grouped_xyz, fps_idx
    return new_xyz, new_points


# --------------------------------------------------------------------------
# network blocks (model5_b.py)
# --------------------------------------------------------------------------


def _lin(sd: Mapping[str, Tensor], name: str, x: Tensor) -> Tensor:
    return torch.nn.functional.linear(x, sd[name + ".weight"], sd[name + ".bias"])


def _bn_point_index_eval(sd: Mapping[str, Tensor], name: str, x: Tensor, eps: float = 1e-5,
                         train: bool = False, bn_state: Optional[dict] = None) -> Tensor:
    """nn.BatchNorm1d(1024) on [B, 1024, 64]: dim 1 (the point index) is the channel
    (model5_b.py:424-425, :447-448; SURVEY.md D7).  Eval mode -> running statistics; ``train`` -> batch statistics
    over (B, 64) per point, with the momentum-0.1 running-stat update written into ``bn_state`` when given."""
    if not train:
        return torch.nn.functional.batch_norm(
            x, sd[name + ".running_mean"], sd[name + ".running_var"],
            sd[name + ".weight"], sd[name + ".bias"], training=False, momentum=0.1, eps=eps)
    rm = sd[name + ".running_mean"].detach().clone()
    rv = sd[name + ".running_var"].detach().clone()
    y = torch.nn.functional.batch_norm(x, rm, rv, sd[name + ".weight"], sd[name + ".bias"], training=True,
                                       momentum=0.1, eps=eps)
    if bn_state is not None:
        bn_state[name + ".running_mean"], bn_state[name + ".running_var"] = rm, rv
    return y


def scaled_dot_production(q: Tensor, k: Tensor, v: Tensor):
    """model5_b.py:67-75 (mask=None branch)."""
    logits = torch.matmul(q, k.transpose(-2, -1)) / math.sqrt(q.shape[-1])
    attn = torch.softmax(logits, dim=-1)
    return torch.matmul(attn, v), attn


def layer_attention(sd: Mapping[str, Tensor], prefix: str, x: Tensor):
    """model5_b.py:92-101 -- offset attention: x + relu(W_o (x - A v))."""
    vals, attn = scaled_dot_production(_lin(sd, prefix + ".mlpq", x), _lin(sd, prefix + ".mlpk", x),
                                       _lin(sd, prefix + ".mlpv", x))
    return x + torch.relu(_lin(sd, prefix + ".out", x - vals)), attn


def encoder_forward(sd: Mapping[str, Tensor], prefix: str, xyz: Tensor,
                    starts: Optional[tuple] = None, train_bn: bool = False,
                    bn_state: Optional[dict] = None) -> Dict[str, Tensor]:
    """PCTransformer_nonsort.forward, model5_b.py:443-478, eval mode.

    ``starts`` = (start1 [B], start2 [B]) FPS start indices; None -> drawn from the
    CPU generator in the reference's order (stage 1 then stage 2).
    Returns every intermediate of SURVEY.md Appendix A.
    """
    p = prefix
    s1, s2 = (None, None) if starts is None else starts
    x_feature = torch.relu(_bn_point_index_eval(sd, p + ".bn1", _lin(sd, p + ".mlp1", xyz), train=train_bn,
                                                bn_state=bn_state))
    x_feature = torch.relu(_bn_point_index_eval(sd, p + ".bn2", _lin(sd, p + ".mlp2", x_feature), train=train_bn,
                                                bn_state=bn_state))
    x1, f1, _, fps1, knn1 = sample_and_group(512, 0, 32, xyz, x_feature, knn=True, start=s1, return_idx=True)
    f1f = torch.relu(_lin(sd, p + ".mlp4", torch.relu(_lin(sd, p + ".mlp3", f1)))).max(dim=-2).values
    x2, f2, _, fps2, knn2 = sample_and_group(256, 0, 32, x1, f1f, knn=True, start=s2, return_idx=True)
    f2f = torch.relu(_lin(sd, p + ".mlp6", torch.relu(_lin(sd, p + ".mlp5", f2)))).max(dim=-2).values
    cur, atts, maps = f2f, [], []
    for i in (1, 2, 3, 4):
        cur, a = layer_attention(sd, f"{p}.atten{i}", cur)
        atts.append(cur)
        maps.append(a)
    attention = (maps[0] + maps[1] + maps[2] + maps[3]) / 4
    out = _lin(sd, p + ".out", torch.cat(atts + [f2f], dim=-1))
    f_global = out.max(dim=1).values
    return dict(f_global=f_global, x2=x2, attention=attention, out=out, x_feature=x_feature,
                x1=x1, fps1=fps1, knn1=knn1, f1f=f1f, fps2=fps2, knn2=knn2, f2f=f2f,
                att=atts, maps=maps)


def _seq(sd: Mapping[str, Tensor], name: str, x: Tensor, layers) -> Tensor:
    for j, li in enumerate(layers):
        x = _lin(sd, f"{name}.{li}", x)
        if j + 1 < len(layers):
            x = torch.relu(x)
    return x


def predict5(sd: Mapping[str, Tensor], fpc: Tensor, mrpc: Tensor, need: bool = False,
             starts: Optional[tuple] = None, train_bn: bool = False,
             bn_state: Optional[dict] = None) -> Dict[str, Tensor]:
    """TouchedRegraster.predict5, model5_b.py:672-759, eval mode.

    ``starts`` = ((fpc stage1, fpc stage2), (mrpc stage1, mrpc stage2)); None draws the
    four starts from the CPU generator in the reference's order (SURVEY.md App. A).
    Replicates D6: BOTH "global" vectors are max-pools of the *mrpc* local features
    (model5_b.py:741-744).
    """
    if fpc.dim() == 2:
        fpc, mrpc = fpc.unsqueeze(0), mrpc.unsqueeze(0)
    st1, st2 = (None, None) if starts is None else starts
    e1 = encoder_forward(sd, "Encoder", fpc, st1, train_bn, bn_state)
    e2 = encoder_forward(sd, "Encoder2", mrpc, st2, train_bn, bn_state)
    out6 = _seq(sd, "tfMLP", torch.cat([e1["f_global"], e2["f_global"]], dim=-1), (0, 2, 4, 6, 8))
    loc_f = _seq(sd, "MLPLocalPreFpc", e1["x_feature"], (0, 2, 4))
    loc_m = _seq(sd, "MLPLocalPreRpc", e2["x_feature"], (0, 2, 4))
    g = loc_m.max(dim=1, keepdim=True).values.expand(-1, loc_m.shape[1], -1)      # D6
    de_fpcb = _seq(sd, "MLPFpcb", torch.cat([g, loc_f], dim=-1), (0, 2, 4)).permute(0, 2, 1)
    de_mrpcb = _seq(sd, "MLPRpcb", torch.cat([g, loc_m], dim=-1), (0, 2, 4)).permute(0, 2, 1)
    return dict(out=out6, de_fpcb=de_fpcb, de_mrpcb=de_mrpcb, enc_fpc=e1, enc_mrpc=e2,
                loc_fpc=loc_f, loc_mrpc=loc_m)


# --------------------------------------------------------------------------
# pose (se_math/se3.py, so3.py, sinc.py) and the pose-parity metrics (metrics.py)
# --------------------------------------------------------------------------


def _sinc123(t: Tensor):
    """sinc.py:6-18, :96-108, :126-138 -- Taylor branch for |t| < 0.01."""
    small = t.abs() < 0.01
    t2 = t * t
    ts = torch.where(small, torch.ones_like(t), t)          # keep the large branch finite
    s1 = torch.where(small, 1 - t2 / 6 * (1 - t2 / 20 * (1 - t2 / 42)), torch.sin(ts) / ts)
    s2 = torch.where(small, 1 / 2 * (1 - t2 / 12 * (1 - t2 / 30 * (1 - t2 / 56))), (1 - torch.cos(ts)) / (ts * ts))
    s3 = torch.where(small, 1 / 6 * (1 - t2 / 20 * (1 - t2 / 42 * (1 - t2 / 72))), (ts - torch.sin(ts)) / ts ** 3)
    return s1, s2, s3


def se3_exp(x: Tensor) -> Tensor:
    """se3.py:57-80 -- twist [.., 6] (omega first, v last) -> [.., 4, 4]."""
    x_ = x.reshape(-1, 6)
    w, v = x_[:, :3], x_[:, 3:]
    t = w.norm(p=2, dim=1).view(-1, 1, 1)
    zero = torch.zeros_like(w[:, 0])
    W = torch.stack([torch.stack([zero, -w[:, 2], w[:, 1]], 1),
                     torch.stack([w[:, 2], zero, -w[:, 0]], 1),
                     torch.stack([-w[:, 1], w[:, 0], zero], 1)], 1)     # so3.py:16-26
    S = W.bmm(W)
    eye = torch.eye(3, dtype=x.dtype)
    s1, s2, s3 = _sinc123(t)
    R = eye + s1 * W + s2 * S
    V = eye + s2 * W + s3 * S
    p = V.bmm(v.reshape(-1, 3, 1))
    g = torch.zeros(x_.shape[0], 4, 4, dtype=x.dtype)
    g[:, :3, :3], g[:, :3, 3:], g[:, 3, 3] = R, p, 1
    return g.view(*x.shape[:-1], 4, 4)


def se3_transform(g: Tensor, a: Tensor) -> Tensor:
    """se3.py:110-120 -- apply g [B,4,4] to a [B,3,N]."""
    return g[..., :3, :3].matmul(a) + g[..., :3, 3].unsqueeze(-1)


def rotation_error_deg(r1: Tensor, r2: Tensor) -> Tensor:
    """metrics.py:54-70 isotropic_R_error, evaluated in float64: in fp32 the formula acos((tr-1)/2) cannot resolve
    angles below ~0.03 deg (1 ulp of tr near 3 is 2.4e-7 -> acos(1 - 1.2e-7) = 0.028 deg), which is coarser than
    the 0.01 deg bound this function is used to check."""
    r1, r2 = r1.double(), r2.double()
    rr = r2.transpose(1, 2).matmul(r1)
    tr = rr[:, 0, 0] + rr[:, 1, 1] + rr[:, 2, 2]
    return torch.acos(torch.clamp((tr - 1) / 2, -1, 1)) / math.pi * 180


def translation_error(t1: Tensor, t2: Tensor) -> Tensor:
    """|t1 - t2| -- the quantity north_star bounds by 1e-4."""
    return (t1 - t2).norm(dim=-1)


# --------------------------------------------------------------------------
# loss-side operators and the test_step epilogue (model5_b.py:1292-1358, :1495-1519)
# --------------------------------------------------------------------------


def chamfer_loss(a: Tensor, b: Tensor):
    """model5_b.py:1495-1505 (dataset.py:1135-1145 is identical): the EXPANDED form through three bmm's,
    P = rx^T + ry - 2 zz; returns (min over dim 1 [B,m], min over dim 2 [B,n]).  n must equal m (expand_as)."""
    xx = torch.bmm(a, a.transpose(2, 1))
    yy = torch.bmm(b, b.transpose(2, 1))
    zz = torch.bmm(a, b.transpose(2, 1))
    d = torch.arange(0, a.shape[1])
    rx = xx[:, d, d].unsqueeze(1).expand_as(xx)
    ry = yy[:, d, d].unsqueeze(1).expand_as(yy)
    P = rx.transpose(2, 1) + ry - 2 * zz
    return torch.min(P, 1)[0], torch.min(P, 2)[0]


def comp(g: Tensor, igt: Tensor) -> Tensor:
    """model5_b.py:1512-1519."""
    A = g.matmul(igt)
    eye = torch.eye(4).to(A).view(1, 4, 4).repeat(A.size(0), 1, 1)
    return torch.nn.functional.mse_loss(A, eye, reduction="mean") * 16


def boundary_prob(logits: Tensor) -> Tensor:
    """model5_b.py:1323-1328: class-1 softmax probability, logits [B,2,N] -> [B,N]."""
    return torch.softmax(logits, dim=1)[:, 1, :]


def boundary_topk(logits: Tensor, k: int = 128) -> Tensor:
    """model5_b.py:1327/:1329 -- torch.topk(prob, k, 1)[1]; ties are resolved to the LOWEST index here
    (torch.topk leaves them unspecified), which is the order the CUDA kernel documents."""
    p = boundary_prob(logits)
    order = torch.sort(-p, dim=1, stable=True).indices
    return order[:, :k]


def inv_R_t(R: Tensor, t: Tensor):
    """metrics.py:7-10."""
    inv_R = R.permute(0, 2, 1).contiguous()
    return inv_R, torch.squeeze(-inv_R @ t[..., None], -1)


def test_step_scores(out6: Tensor, de_fpcb: Tensor, de_mrpcb: Tensor, fpc: Tensor, src: Tensor,
                     fpcb: Tensor, rpcb: Tensor, fpc_idx: Tensor, rpc_idx: Tensor, igt: Tensor) -> Dict[str, Tensor]:
    """Everything test_step does after predict5 (model5_b.py:1314-1358 with metrics.py:54-84), per pair.
    ``src`` is the cloud the second boundary is gathered from (``rpc`` in test_step)."""
    mat = se3_exp(out6)
    R, t = mat[:, :3, :3], mat[:, :3, 3]
    inv_R, inv_t = inv_R_t(igt[:, :3, :3], igt[:, :3, 3])
    rr = torch.matmul(inv_R.permute(0, 2, 1).contiguous(), R)
    tr = rr[:, 0, 0] + rr[:, 1, 1] + rr[:, 2, 2]
    r_iso = torch.acos(torch.clamp((tr - 1) / 2, -1, 1)) / math.pi * 180
    R2, t2 = inv_R_t(inv_R, inv_t)
    t_iso = torch.norm(torch.squeeze(R2 @ t[..., None], -1) + t2, dim=-1)
    t_mse = ((t - inv_t) ** 2).mean(1)
    t_mae = (t - inv_t).abs().mean(1)
    idx_f, idx_m = boundary_topk(de_fpcb), boundary_topk(de_mrpcb)
    B = fpc.shape[0]
    pred_f = torch.zeros(B, 1024).scatter(1, idx_f, 1)
    pred_m = torch.zeros(B, 1024).scatter(1, idx_m, 1)
    gf, gm = fpc_idx.reshape(B, 1024), rpc_idx.reshape(B, 1024)
    inter_f = torch.logical_and(pred_f, gf).sum(1).float()
    union_f = torch.logical_or(pred_f, gf).sum(1).float()
    inter_m = torch.logical_and(pred_m, gm).sum(1).float()
    union_m = torch.logical_or(pred_m, gm).sum(1).float()
    bnd_f = torch.gather(fpc, 1, idx_f.unsqueeze(-1).repeat(1, 1, 3))
    bnd_m = torch.gather(src, 1, idx_m.unsqueeze(-1).repeat(1, 1, 3))
    bnd_m = se3_transform(mat, bnd_m.permute(0, 2, 1)).permute(0, 2, 1)
    c1, c2 = chamfer_loss(fpcb, bnd_f)
    cd_fpc = c1.mean(1) + c2.mean(1)
    c1, c2 = chamfer_loss(rpcb, bnd_m)
    cd_rpc = c1.mean(1) + c2.mean(1)
    c1, c2 = chamfer_loss(bnd_f, bnd_m)
    cd_pair = c1.mean(1) + c2.mean(1)
    return dict(r_iso=r_iso, t_iso=t_iso, t_mse=t_mse, t_mae=t_mae, inter_f=inter_f, union_f=union_f,
                inter_m=inter_m, union_m=union_m, cd_fpc=cd_fpc, cd_rpc=cd_rpc, cd_pair=cd_pair,
                idx_f=idx_f, idx_m=idx_m, bnd_f=bnd_f, bnd_m=bnd_m, mat=mat)


# --------------------------------------------------------------------------
# dataset-side preprocessing (dataset.py) -- numpy, as in the reference
# --------------------------------------------------------------------------


def dataset_fps(points, npoints: int, start: Optional[int] = None):
    """CADDataset.fps, dataset.py:1147-1163 (same code at :286, :437, :510, :582, :835, :1042): numpy FPS on ONE
    cloud, float64 running distance, fp32 candidate distance, strict '<' update, first arg-max; returns the
    selected POINTS (not indices).  ``start`` None draws np.random.randint(0, N) like the reference."""
    import numpy as np
    if points.shape[0] < npoints:
        return None
    N = points.shape[0]
    xyz = points[:, :3]
    centroids = np.zeros((npoints,))
    distance = np.ones((N,)) * 1e10
    farthest = np.random.randint(0, N) if start is None else int(start)
    for i in range(npoints):
        centroids[i] = farthest
        centroid = xyz[farthest, :]
        dist = np.sum((xyz - centroid) ** 2, -1)
        mask = dist < distance
        distance[mask] = dist[mask]
        farthest = np.argmax(distance, -1)
    return points[centroids.astype(np.int32)]


def plane_split(points, z=None):
    """dataset.py:761-775 -- random-plane cut (normal ~ U[0,1)^3, offset ~ U[0,1/3)) -> (up, down)."""
    import numpy as np
    normal = np.random.rand(3, 1)
    if z is None:
        z = np.random.rand(1) / 3
    dis = np.dot(points, normal) + z
    return points[(dis >= 0)[:, 0]], points[(dis < 0)[:, 0]]


def get_boundary(fpc: Tensor, de_mrpc: Tensor):
    """CADDataset.get_boundary, dataset.py:1357-1367: the 128 points of each half closest to the other half.
    -> (fpc boundary [128,3], mrpc boundary [128,3], fpc_idx [1024] 0/1, rpc_idx [1024] 0/1)."""
    cd1, cd2 = chamfer_loss(fpc.unsqueeze(0), de_mrpc.unsqueeze(0))
    top1 = torch.topk(-cd1, 128)
    cdxyz1 = de_mrpc[top1[1][0]]
    top2 = torch.topk(-cd2, 128)
    cdxyz2 = fpc[top2[1][0]]
    fpc_idx = torch.zeros(1024)
    fpc_idx[top2[1][0]] = 1
    rpc_idx = torch.zeros(1024)
    rpc_idx[top1[1][0]] = 1
    return cdxyz2, cdxyz1, fpc_idx, rpc_idx


def predict6(sd: Mapping[str, Tensor], fpc: Tensor, mrpc: Tensor, starts: Optional[tuple] = None) -> Dict[str, Tensor]:
    """TouchedRegraster.predict6(pretrain=True), model5_b.py:612-658: both clouds through ``Encoder``, pose only."""
    st1, st2 = (None, None) if starts is None else starts
    e1 = encoder_forward(sd, "Encoder", fpc, st1)
    e2 = encoder_forward(sd, "Encoder", mrpc, st2)
    out6 = _seq(sd, "tfMLP", torch.cat([e1["f_global"], e2["f_global"]], dim=-1), (0, 2, 4, 6, 8))
    return dict(out=out6, enc_fpc=e1, enc_mrpc=e2)
