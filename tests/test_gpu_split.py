"""The split path (PZ_PREC_SPLIT: fp16 hi/lo operand planes, three tcgen05 MMAs per product, fp32 accumulation) block by
block against the CPU oracle, at the fp32 tolerance of north_star (1e-4 relative; measured ~1e-6).  The kernels:
split_rowgemm_pair_kernel / split_gather_kernel / split_gather_pair_kernel (gemm_split.cu: CTA pairs, TMA),
attention_split_kernel (attention_split.cu), head_*_split_kernel (heads_split.cu), stem_tc_kernel<true> (encoder.cu); the
one-CTA kernels (split_rowgemm_kernel, the 128-row split_gather_kernel) through the group-MLP shapes that reach them.
End to end at B=64: tests/test_gpu_b64_parity.py."""
import numpy as np
import pytest
import torch

from oracle import parity
from oracle import puzzle_oracle as po
from puzzlenet_b200.weights import make_batch, synthetic_pairs
from tests.golden_inputs import FPS_SEED

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-4


@pytest.mark.parametrize("B", [1, 3, 150])
def test_layer_attention_split(state_dict, B):
    """q|k and v projections, q k^T, softmax, P v, offset, out-projection + residual: values AND the attention map."""
    from puzzlenet_b200.model5_b import layerAttention
    g = torch.Generator().manual_seed(5)
    layer = layerAttention(None, 256)
    pre = "Encoder2.atten2."
    layer.load_state_dict({k[len(pre):]: v for k, v in state_dict.items() if k.startswith(pre)})
    layer.precision = "split"
    x = torch.randn(B, 256, 256, generator=g) * 0.5
    out, a = layer.to(DEV)(x.to(DEV))
    torch.cuda.synchronize()
    ro, ra = po.layer_attention(state_dict, pre[:-1], x)
    errs = dict(out=parity.rel(out, ro), out_elem=parity.rel_elem(out, ro), attn=parity.rel(a, ra))
    print(f"split attention layer B={B}:", errs)
    assert max(errs.values()) < TOL, errs
    np.testing.assert_allclose(a.sum(-1).cpu().numpy(), 1.0, atol=1e-5)


_STAGE1, _STAGE2 = ("Encoder.mlp3", "Encoder.mlp4"), ("Encoder2.mlp5", "Encoder2.mlp6")


@pytest.mark.parametrize("layers, B, N, S, seed", [
    pytest.param(_STAGE1, 2, 1024, 128, 3, id="1"),
    pytest.param(_STAGE2, 2, 512, 64, 4, id="2"),
    # B*N = 384 rows tile by 128 but not by 256: the one-CTA row GEMMs split_rowgemm_kernel<128,3> (C1 = 128) and
    # split_rowgemm_kernel<256,2> (C1 = 256)
    pytest.param(_STAGE1, 3, 128, 32, 5, id="1-rows128"),
    pytest.param(_STAGE2, 3, 128, 32, 6, id="2-rows128"),
    # C1 = 256 with C2 = 128 (no encoder layer has it, so seeded random weights): the 128-row split_gather_kernel
    pytest.param(None, 2, 512, 64, 7, id="c1_256-c2_128"),
])
def test_group_mlp_maxpool_split(state_dict, layers, B, N, S, seed):
    """Layer 1 over source points (row GEMM, fp32 P), fp32 Q, gathered relu(P - Q) formed in registers, three-MMA layer 2,
    max over the 32 neighbours: both stage shapes of the encoder (67->128->128 on 1024 points, 131->256->256 on 512) and
    the shapes that reach the one-CTA kernels."""
    from puzzlenet_b200 import pointnet_util as pu
    g = torch.Generator().manual_seed(seed)
    sd = state_dict
    if layers is None:
        sd = {"a.weight": torch.randn(256, 3 + 64, generator=g) / 67 ** 0.5, "a.bias": torch.randn(256, generator=g) / 67 ** 0.5,
              "b.weight": torch.randn(128, 256, generator=g) / 16, "b.bias": torch.randn(128, generator=g) / 16}
        layers = ("a", "b")
    la, lb = layers
    D = sd[la + ".weight"].shape[1] - 3
    xyz = torch.rand(B, N, 3, generator=g) - 0.5
    feat = torch.randn(B, N, D, generator=g)
    torch.manual_seed(8)
    nx, npts, _, _, idx = po.sample_and_group(S, 0, 32, xyz, feat, knn=True, return_idx=True)
    ref = torch.relu(po._lin(sd, lb, torch.relu(po._lin(sd, la, npts)))).max(-2).values
    got = pu.group_mlp_maxpool(xyz.to(DEV), feat.to(DEV), nx.to(DEV), idx.to(DEV),
                               sd[la + ".weight"].to(DEV), sd[la + ".bias"].to(DEV),
                               sd[lb + ".weight"].to(DEV), sd[lb + ".bias"].to(DEV), precision=2)
    errs = dict(rel=parity.rel(got, ref), elem=parity.rel_elem(got, ref))
    print(f"split group MLP {la} B={B} N={N}:", errs)
    assert got.shape == ref.shape and max(errs.values()) < TOL, errs


def test_encoder_split_intermediates(cuda_model, state_dict):
    fpc, _ = synthetic_pairs(2, seed=64)
    cuda_model.Encoder.precision = "split"
    try:
        torch.manual_seed(FPS_SEED)
        got = cuda_model.Encoder(fpc.to(DEV), return_intermediates=True)
        torch.cuda.synchronize()
    finally:
        cuda_model.Encoder.precision = "fp32"
    torch.manual_seed(FPS_SEED)
    ref = po.encoder_forward(state_dict, "Encoder", fpc)
    for name in ("fps1", "knn1", "fps2", "knn2"):
        assert torch.equal(got[name].cpu(), ref[name]), name
    errs = {n: parity.rel(got[n], ref[n]) for n in ("x_feature", "f1f", "f2f", "attention", "out", "f_global")}
    errs["att_cat"] = parity.rel(got["att_cat"], torch.cat(ref["att"] + [ref["f2f"]], -1))
    print("split encoder rel errors:", errs)
    assert max(errs.values()) < TOL, errs


@pytest.mark.parametrize("B", [1, 5])
def test_predict5_split_vs_oracle(cuda_model, state_dict, B):
    fpc, mrpc = synthetic_pairs(B, seed=100 + B)
    cuda_model.precision = "split"
    try:
        torch.manual_seed(B)
        out, _, de_f, de_m = cuda_model.predict5(make_batch(fpc.to(DEV), mrpc.to(DEV)), 0)
        torch.cuda.synchronize()
        again = cuda_model.predict5(make_batch(fpc.to(DEV), mrpc.to(DEV)), 0,
                                    starts=None if False else None)   # second call re-uses the weight planes
    finally:
        cuda_model.precision = "fp32"
    torch.manual_seed(B)
    ref = po.predict5(state_dict, fpc, mrpc)
    errs = dict(out=parity.rel(out, ref["out"]), de_f=parity.rel(de_f, ref["de_fpcb"]), de_m=parity.rel(de_m, ref["de_mrpcb"]),
                de_f_elem=parity.rel_elem(de_f, ref["de_fpcb"]))
    rot, trans = parity.pose_errors(out, ref["out"])
    print(f"split predict5 B={B}:", errs, "rotation [deg]", rot, "translation", trans)
    assert max(errs.values()) < TOL, errs
    assert rot < 0.01 and trans < 1e-4
    assert again[0].shape == out.shape


def test_split_chain_is_race_free_at_b64(cuda_model):
    """The split forward is ONE chain of launches linked by programmatic dependent launch, and consecutive attention
    launches hand over per cloud (counters in the tail's scratch): 40 eager forwards back to back on one workspace, alternating
    two inputs, must reproduce the first result of each input bit for bit."""
    a = synthetic_pairs(64, seed=900)
    b = synthetic_pairs(64, seed=901)
    ba, bb = (make_batch(x[0].to(DEV), x[1].to(DEV)) for x in (a, b))
    starts = torch.stack([torch.randint(0, n, (64,), generator=torch.Generator().manual_seed(i))
                          for i, n in enumerate((1024, 512, 1024, 512))]).to(DEV)
    cuda_model.precision = "split"
    try:
        first = {}
        for i in range(40):
            key, batch = ("a", ba) if i % 2 == 0 else ("b", bb)
            out, _, de_f, de_m = cuda_model.predict5(batch, 0, starts=starts)
            got = (out.clone(), de_f.clone(), de_m.clone())
            if key not in first:
                first[key] = got
            else:
                for x, y in zip(got, first[key]):
                    assert torch.equal(x, y), (i, key)
        torch.cuda.synchronize()
    finally:
        cuda_model.precision = "fp32"
    assert not torch.equal(first["a"][0], first["b"][0])
