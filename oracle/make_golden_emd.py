"""TEST INFRASTRUCTURE ONLY -- freeze EMD kernel outputs on a B200 for tests/test_gpu_emd.py::test_vs_reference_kernels_on_gpu.

For every case of tests.golden_inputs.EMD_CASES: cost (b), the sampled entries of match (b,m,n), and the gradients
(b,n,3) / (b,m,3) of matchcost for grad_cost = 1 on that match.  Where oracle/_ref/libemd_ref.so (the reference's own
kernels, `make -C oracle ref`) is present they come from it.  Otherwise they come from puzzlenet_b200.emd_cuda at a commit
whose kernels passed the same-GPU comparison with that library on exactly these inputs (cost rtol 1e-4, match 1e-4
absolute, gradients rtol 1e-4 / atol 1e-5).  The file records which (`source`).

    python oracle/make_golden_emd.py [OUT]     (on a B200) -> tests/golden/emd_kernels.npz
"""
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests.golden_inputs import EMD_CASES, emd_inputs  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "emd_kernels.npz")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libemd_ref.so")


def _reference(x1, x2):
    """The reference kernels with their own launch shapes (oracle/emd_ref_launcher.cu)."""
    ref = ctypes.CDLL(REF_SO)
    b, n, m = x1.shape[0], x1.shape[1], x2.shape[1]
    dev, vp = x1.device, ctypes.c_void_p
    match, temp = torch.empty(b, m, n, device=dev), torch.empty(32 * (n + m) * 2, device=dev)
    cost, gc = torch.empty(b, device=dev), torch.ones(b, device=dev)
    g1, g2 = torch.empty(b, n, 3, device=dev), torch.empty(b, m, 3, device=dev)
    st = vp(torch.cuda.current_stream().cuda_stream)
    p = lambda t: vp(t.data_ptr())  # noqa: E731
    assert ref.emd_ref_approxmatch(b, n, m, p(x1), p(x2), p(match), p(temp), st) == 0
    assert ref.emd_ref_matchcost(b, n, m, p(x1), p(x2), p(match), p(cost), st) == 0
    assert ref.emd_ref_matchcost_grad(b, n, m, p(gc), p(x1), p(x2), p(match), p(g1), p(g2), st) == 0
    return match, cost, g1, g2


def _ours(x1, x2):
    from puzzlenet_b200 import emd_cuda
    match = emd_cuda.approxmatch_forward(x1, x2)
    cost = emd_cuda.matchcost_forward(x1, x2, match)
    g1, g2 = emd_cuda.matchcost_backward(torch.ones(x1.shape[0], device=x1.device), x1, x2, match)
    return match, cost, g1, g2


def main(path=GOLDEN):
    source = "reference kernels (oracle/_ref/libemd_ref.so)" if os.path.isfile(REF_SO) else "puzzlenet_b200.emd_cuda"
    run = _reference if os.path.isfile(REF_SO) else _ours
    out = {"source": np.array(source)}
    for b, n, m in EMD_CASES:
        x1, x2, idx = emd_inputs(b, n, m)
        match, cost, g1, g2 = run(x1.cuda(), x2.cuda())
        torch.cuda.synchronize()
        key = f"{b}_{n}_{m}"
        out[f"{key}/cost"] = cost.cpu().numpy()
        out[f"{key}/match"] = match.flatten()[idx.cuda()].cpu().numpy()
        out[f"{key}/grad1"] = g1.cpu().numpy()
        out[f"{key}/grad2"] = g2.cpu().numpy()
    np.savez_compressed(path, **out)
    print("wrote", path, f"{os.path.getsize(path) / 1024:.0f} KiB from", source)


if __name__ == "__main__":
    main(*sys.argv[1:])
