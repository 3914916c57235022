"""Deterministic inputs shared by oracle/make_golden.py and the tests (kept in sync by import)."""
import torch

FPS_SEED = 1234


def golden_inputs():
    g = torch.Generator().manual_seed(7)
    xyz = torch.rand(2, 300, 3, generator=g) - 0.5
    feat = torch.randn(2, 300, 8, generator=g)
    xyz[1, 17] = xyz[1, 3]
    big = torch.rand(1, 11000, 3, generator=torch.Generator().manual_seed(3)) - 0.5
    twist = torch.randn(8, 6, generator=g) * 0.7
    twist[0, :3] *= 1e-3
    twist[1, :3] = 0
    return xyz, feat, big, twist


def epilogue_inputs(batch, se3_exp):
    """Ground-truth side of a test batch (rpc, boundaries, boundary masks, igt) for the test_step goldens;
    ``se3_exp`` is whichever exp map the caller pins (reference / oracle / CUDA -- igt is an input)."""
    g = torch.Generator().manual_seed(5)
    rpc = torch.rand(batch, 1024, 3, generator=g) - 0.5
    fpcb = torch.rand(batch, 128, 3, generator=g) - 0.5
    rpcb = torch.rand(batch, 128, 3, generator=g) - 0.5
    fpc_idx = (torch.rand(batch, 1024, generator=g) < 0.125).float()
    rpc_idx = (torch.rand(batch, 1024, generator=g) < 0.125).float()
    twist = torch.randn(batch, 6, generator=g) * 0.3
    twist2 = torch.randn(batch, 6, generator=g) * 0.3
    return dict(rpc=rpc, fpcb=fpcb, rpcb=rpcb, fpc_idx=fpc_idx, rpc_idx=rpc_idx, twist=twist, twist2=twist2,
                igt=se3_exp(twist))


def dataset_inputs():
    """One 'raw' piece for the dataset-side goldens: 6000 points of a unit-ish blob (numpy fp32)."""
    g = torch.Generator().manual_seed(9)
    return (torch.randn(6000, 3, generator=g) * 0.3).numpy()


def training_inputs(batch, se3_exp):
    """A training batch with a consistent geometry: rpc is a cloud, mrpc = igt . rpc (so the pose losses have a
    meaningful target), fpc an independent cloud, boundaries / masks random (they are inputs only)."""
    g = torch.Generator().manual_seed(77)
    fpc = torch.rand(batch, 1024, 3, generator=g) - 0.5
    rpc = torch.rand(batch, 1024, 3, generator=g) - 0.5
    twist = torch.randn(batch, 6, generator=g) * 0.3
    igt = se3_exp(twist)
    mrpc = (igt[:, :3, :3] @ rpc.permute(0, 2, 1) + igt[:, :3, 3:]).permute(0, 2, 1).contiguous()
    fpcb = torch.rand(batch, 128, 3, generator=g) - 0.5
    rpcb = torch.rand(batch, 128, 3, generator=g) - 0.5
    fpc_idx = (torch.rand(batch, 1024, generator=g) < 0.125).float()
    rpc_idx = (torch.rand(batch, 1024, generator=g) < 0.125).float()
    return [fpc, mrpc, igt, rpc, fpcb, rpcb, fpc_idx, rpc_idx]


EMD_CASES = [(4, 1024, 1024), (3, 128, 128), (2, 96, 200)]      # (b, n, m) of the EMD kernel goldens
EMD_MATCH_SAMPLE = 49152                                       # match entries stored per case (all of them if fewer)


def emd_inputs(b, n, m):
    """Clouds xyz1 (b,n,3), xyz2 (b,m,3) of one EMD kernel golden case, and the flat indices into match (b,m,n) whose
    values are stored: every entry of a small match, a fixed random sample of a large one (the full (4,1024,1024)
    match is 16 MB)."""
    g = torch.Generator().manual_seed(n)
    x1 = torch.randn(b, n, 3, generator=g) * 0.5
    x2 = torch.randn(b, m, 3, generator=g) * 0.5
    total = b * m * n
    if total <= EMD_MATCH_SAMPLE:
        idx = torch.arange(total)
    else:
        idx = torch.randperm(total, generator=torch.Generator().manual_seed(total))[:EMD_MATCH_SAMPLE].sort().values
    return x1, x2, idx


def pointnet_block_inputs():
    g = torch.Generator().manual_seed(17)
    return torch.rand(2, 200, 3, generator=g) - 0.5, torch.randn(2, 200, 8, generator=g)


def seed_block(module, seed):
    """deterministic parameters + non-trivial BatchNorm running statistics for a PointNet++ block (either the
    reference's class or the mirror: the state_dict keys are the same)"""
    g = torch.Generator().manual_seed(1000 + seed)
    with torch.no_grad():
        for name, p in sorted(module.state_dict().items()):
            if "num_batches_tracked" in name:
                continue
            if name.endswith("running_var"):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
            elif name.endswith("running_mean") or name.endswith("bias"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
            elif name.endswith("weight") and p.dim() == 1:
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
            else:
                p.copy_(torch.randn(p.shape, generator=g) * 0.3)
    return module
