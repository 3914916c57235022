"""GPU parity: approximate EMD vs the C oracle (known-answer pinned) and vs stored B200 outputs that stand for the
reference's own kernels (tests/golden/emd_kernels.npz; oracle/make_golden_emd.py says where they come from)."""
import os

import numpy as np
import pytest
import torch

from oracle import emd_oracle as eo
from tests.golden_inputs import EMD_CASES, emd_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "emd_kernels.npz")


@pytest.fixture(scope="module")
def emd_gold():
    return dict(np.load(GOLDEN))


def test_known_answer():
    """PyTorchEMD/test_emd_loss.py:8-33: cost 0.71 per item and the closed-form gradients."""
    from puzzlenet_b200.emd import earth_mover_distance
    p1 = torch.tensor([[[1.7, -0.1, 0.1], [0.1, 1.2, 0.3]]]).repeat(3, 1, 1).to(DEV).requires_grad_()
    p2 = torch.tensor([[[0.3, 1.8, 0.2], [1.2, -0.2, 0.3]]]).repeat(3, 1, 1).to(DEV).requires_grad_()
    d = earth_mover_distance(p1, p2, transpose=False)
    np.testing.assert_allclose(d.detach().cpu().numpy(), [0.71] * 3, rtol=1e-5)
    (d[0] / 2 + d[1] * 2 + d[2] / 3).backward()
    q1 = p1.detach().clone().requires_grad_()
    q2 = p2.detach().clone().requires_grad_()
    gt = sum(w * (((q1[i, 0] - q2[i, 1]) ** 2).sum() + ((q1[i, 1] - q2[i, 0]) ** 2).sum())
             for i, w in enumerate((0.5, 2.0, 1 / 3)))
    gt.backward()
    np.testing.assert_allclose(p1.grad.cpu().numpy(), q1.grad.cpu().numpy(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(p2.grad.cpu().numpy(), q2.grad.cpu().numpy(), rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("b,n,m", [(3, 64, 64), (2, 128, 128), (2, 100, 40), (2, 48, 96), (2, 1024, 1024), (1, 1500, 700)])
def test_vs_c_oracle(b, n, m):
    from puzzlenet_b200 import emd_cuda
    rng = np.random.default_rng(n + m)
    x1 = rng.standard_normal((b, n, 3)).astype(np.float32) * 0.5
    x2 = rng.standard_normal((b, m, 3)).astype(np.float32) * 0.5
    t1, t2 = torch.from_numpy(x1).to(DEV), torch.from_numpy(x2).to(DEV)
    match = emd_cuda.approxmatch_forward(t1, t2)
    assert match.shape == (b, m, n)
    cost = emd_cuda.matchcost_forward(t1, t2, match)
    ref_match = eo.approxmatch(x1, x2)
    ref_cost = eo.matchcost(x1, x2, ref_match)
    # __expf (GPU) vs expf (C oracle): 1e-4 relative on the cost, 1e-3 on match/gradients (SURVEY.md §8c)
    np.testing.assert_allclose(cost.cpu().numpy(), ref_cost, rtol=1e-4)
    assert np.abs(match.cpu().numpy() - ref_match).max() < 1e-3
    gc = torch.linspace(0.5, 1.5, b, device=DEV)
    g1, g2 = emd_cuda.matchcost_backward(gc, t1, t2, match)
    r1, r2 = eo.matchcost_grad(gc.cpu().numpy(), x1, x2, match.cpu().numpy())
    np.testing.assert_allclose(g1.cpu().numpy(), r1, rtol=1e-3, atol=1e-4)
    np.testing.assert_allclose(g2.cpu().numpy(), r2, rtol=1e-3, atol=1e-4)


def test_transpose_default_and_2d_inputs():
    from puzzlenet_b200.emd import earth_mover_distance
    a = torch.randn(2, 64, 3, device=DEV)
    b = torch.randn(2, 64, 3, device=DEV)
    c1 = earth_mover_distance(a.transpose(1, 2), b.transpose(1, 2))          # default transpose=True: (b,3,n)
    c2 = earth_mover_distance(a, b, transpose=False)
    assert torch.equal(c1, c2)
    assert earth_mover_distance(a[0], b[0], transpose=False).shape == (1,)
    with pytest.raises(AssertionError):
        earth_mover_distance(a.cpu(), b.cpu(), transpose=False)              # emd.py:10


@pytest.mark.parametrize("b,n,m", EMD_CASES)
def test_vs_reference_kernels_on_gpu(b, n, m, emd_gold):
    """Same GPU, same __expf, the reference kernels' test inputs: ours vs the stored outputs (the reference's kernels, or
    ours at a commit that matched them within these tolerances: the file's `source`).  Where the whole match is stored
    the gradients are taken on it, as they were when stored."""
    from puzzlenet_b200 import emd_cuda
    key = f"{b}_{n}_{m}"
    x1, x2, idx = emd_inputs(b, n, m)
    x1, x2, idx = x1.to(DEV), x2.to(DEV), idx.to(DEV)
    match = emd_cuda.approxmatch_forward(x1, x2)
    cost = emd_cuda.matchcost_forward(x1, x2, match)
    np.testing.assert_allclose(cost.cpu().numpy(), emd_gold[f"{key}/cost"], rtol=1e-4)
    rmatch = emd_gold[f"{key}/match"]
    assert np.abs(match.flatten()[idx].cpu().numpy() - rmatch).max() < 1e-4
    if rmatch.size == match.numel():
        match = torch.from_numpy(rmatch).to(DEV).view(b, m, n)
    g1, g2 = emd_cuda.matchcost_backward(torch.ones(b, device=DEV), x1, x2, match)
    np.testing.assert_allclose(g1.cpu().numpy(), emd_gold[f"{key}/grad1"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(g2.cpu().numpy(), emd_gold[f"{key}/grad2"], rtol=1e-4, atol=1e-5)
