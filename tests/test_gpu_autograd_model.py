"""GPU: autograd through the train-mode forward (``TouchedRegraster.differentiable = True``) and through the pose
operators ``se3.exp`` / ``comp``.  Gradients of arbitrary losses against torch-CPU autograd over the oracle; the
reference's own training loss, assembled from the drop-in operators, against ``Trainer.forward_backward``; graph
ownership, optimizers and TF32."""
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import puzzle_oracle as po
from oracle import train_oracle as to
from puzzlenet_b200.weights import make_batch, synthetic_state_dict
from tests.golden_inputs import FPS_SEED, training_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SKIP = ("fpc_decoder", "rpc_decoder")


def _fresh_model(differentiable=True):
    from puzzlenet_b200.model5_b import TouchedRegraster
    model = TouchedRegraster(types.SimpleNamespace(dataset="vase", loss_mode=1, loss_sum=False, lr=0.9e-3))
    model.load_state_dict(synthetic_state_dict(0), strict=True)
    model = model.to(DEV)
    model.differentiable = differentiable
    return model


def _starts(B, seed=FPS_SEED):
    torch.manual_seed(seed)
    return torch.stack([torch.randint(0, 1024, (B,)), torch.randint(0, 512, (B,)),
                        torch.randint(0, 1024, (B,)), torch.randint(0, 512, (B,))])


def _grad_sd():
    return {k: (v.clone().requires_grad_() if v.is_floating_point() and "running" not in k else v.clone())
            for k, v in synthetic_state_dict(0).items()}


def _rel(a, b):
    return ((a.detach().cpu().double() - b.detach().cpu().double()).norm()
            / b.detach().cpu().double().norm().clamp_min(1e-30)).item()


def _weights(B, seed=3):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(*s, generator=g) for s in ((B, 6), (B, 2, 1024), (B, 2, 1024), (B, 256, 256), (B, 256, 3))]


def _custom_loss(out6, de_f, de_m, att_f, x2_m, w, use):
    terms = [(w[0] * out6).sum(), (w[1] * de_f).sum(), (w[2] * de_m).sum(), (w[3] * att_f).sum(), (w[4] * x2_m).sum()]
    return sum(t for t, u in zip(terms, use) if u)


def _check_param_grads(model, ref_of, tol):
    """every live parameter's .grad vs ``ref_of(name)`` (None: the reference leaves it without gradient)"""
    worst = {}
    for name, p in model.named_parameters():
        if name.startswith(SKIP) or name == "dt":
            assert p.grad is None, name
            continue
        ref = ref_of(name)
        if ref is None:
            assert p.grad is None or p.grad.abs().max().item() == 0.0, name
            continue
        assert p.grad is not None, name
        if name.endswith("mlpk.bias"):            # mathematically zero (constant per softmax row)
            continue
        worst[name] = _rel(p.grad, ref)
    bad = {k: v for k, v in worst.items() if not v < tol}
    assert not bad, bad
    return worst


@pytest.mark.parametrize("use", [(1, 1, 1, 1, 1), (0, 0, 1, 0, 0)], ids=["all_outputs", "de_mrpcb_only"])
def test_arbitrary_upstream_gradients_match_oracle_autograd(use):
    """L = sum w1 out6 + w2 de_fpcb + w3 de_mrpcb + w4 attention_fpc + w5 x2_mrpc (need=True, B=2, fp32): every
    parameter gradient and both cloud gradients within relative L2 1e-3 of CPU autograd over the oracle; with only
    de_mrpcb used, the other outputs' gradients are None and contribute nothing"""
    B = 2
    batch = training_inputs(B, po.se3_exp)
    st = _starts(B)
    w = _weights(B)
    model = _fresh_model()
    fpc = batch[0].to(DEV).requires_grad_()
    mrpc = batch[1].to(DEV).requires_grad_()
    r = model.predict5([fpc, mrpc] + [t.to(DEV) for t in batch[2:]], B, need=True, training=True, starts=st)
    assert len(r) == 8 and r[1] == [0]
    L = _custom_loss(r[0], r[6], r[7], r[3], r[4], [t.to(DEV) for t in w], use)
    L.backward()
    sd = _grad_sd()
    cf, cm = batch[0].clone().requires_grad_(), batch[1].clone().requires_grad_()
    o = po.predict5(sd, cf, cm, need=True, starts=((st[0], st[1]), (st[2], st[3])), train_bn=True)
    Lr = _custom_loss(o["out"], o["de_fpcb"], o["de_mrpcb"], o["enc_fpc"]["attention"], o["enc_mrpc"]["x2"], w, use)
    Lr.backward()
    np.testing.assert_allclose(L.item(), Lr.item(), rtol=1e-4)
    worst = _check_param_grads(model, lambda n: sd[n].grad, 1e-3)
    assert len(worst) > (100 if all(use) else 10)
    for got, ref, name in ((fpc.grad, cf.grad, "fpc"), (mrpc.grad, cm.grad, "mrpc")):
        if ref is None:
            assert got is None or got.abs().max().item() == 0.0, name
        else:
            assert _rel(got, ref) < 1e-3, (name, _rel(got, ref))
    print("worst parameter gradient error:", max(worst.values()))


def _reference_loss(model, batch, B, st, pretrain=False):
    """training_step's loss (model5_b.py:912-1155, loss_mode 1) assembled from the drop-in operators"""
    from puzzlenet_b200 import losses, se3
    from puzzlenet_b200 import pointnet_util as pu
    from puzzlenet_b200.emd import earth_mover_distance
    fpc, mrpc, igt, rpc, fpcb, rpcb, fpc_idx, rpc_idx = batch
    if pretrain:
        out = model.predict6(batch, B, training=True, pretrain=True, starts=st)
    else:
        out, _, _, _, _, _, de_fpcb, de_mrpcb = model.predict5(batch, B, need=True, training=True, starts=st)
    mat = se3.exp(out)
    de_mrpc = se3.transform(mat, mrpc.permute(0, 2, 1)).permute(0, 2, 1)
    d1, d2 = model.chamfer_loss(rpc, de_mrpc)
    loss = d1.mean() + d2.mean() + model.comp(mat, igt) + earth_mover_distance(de_mrpc, rpc, transpose=False).mean()
    if pretrain:
        return loss
    loss = loss + F.cross_entropy(de_fpcb, fpc_idx.long()) + F.cross_entropy(de_mrpcb, rpc_idx.long())
    bnd_f = pu.index_points(fpc, losses.boundary_topk(de_fpcb))
    bnd_m = pu.index_points(mrpc, losses.boundary_topk(de_mrpcb))
    c1, c2 = model.chamfer_loss(bnd_f, fpcb)
    inv_bnd_m = se3.transform(mat, bnd_m.permute(0, 2, 1)).permute(0, 2, 1)
    c3, c4 = model.chamfer_loss(inv_bnd_m, rpcb)
    return loss + c3.mean() + c4.mean() + c1.mean() + c2.mean()


@pytest.mark.parametrize("pretrain", [False, True], ids=["predict5", "predict6_pretrain"])
def test_reference_loss_end_to_end_matches_trainer_and_oracle(pretrain):
    """the reference's loss through the differentiable forward + loss.backward() vs Trainer.forward_backward on the
    same batch and starts (loss rtol 1e-5, gradients relative L2 1e-4, BatchNorm running statistics bit-identical)
    and vs the CPU training oracle (loss 2e-4; gradients 1e-3, 1e-2 for the pretraining branch, whose tolerance
    test_pretraining_branch_matches_oracle_and_reference explains)"""
    from puzzlenet_b200.training import Trainer
    B = 2
    batch = [t.to(DEV) for t in training_inputs(B, po.se3_exp)]
    st = _starts(B)
    model = _fresh_model()
    loss = _reference_loss(model, batch, B, st, pretrain)
    loss.backward()
    twin = _fresh_model(differentiable=False)
    tr = Trainer(twin)
    terms = tr.forward_backward_pretrain(batch, starts=st) if pretrain else tr.forward_backward(batch, starts=st)
    torch.cuda.synchronize()
    np.testing.assert_allclose(loss.item(), terms["loss"], rtol=1e-5)
    used = (lambda n: n.startswith(("Encoder.", "tfMLP."))) if pretrain else (lambda n: True)  # noqa: E731
    twin_p = dict(twin.named_parameters())
    worst = _check_param_grads(model, lambda n: tr.flat.g(twin_p[n]) if used(n) else None, 1e-4)
    print("worst gradient error vs Trainer:", max(worst.values()))
    for name, buf in model.named_buffers():
        assert torch.equal(buf, twin.get_buffer(name)), name
    sd = _grad_sd()
    torch.manual_seed(FPS_SEED)
    ref = to.training_loss(sd, [t.cpu() for t in batch], pretrain=pretrain)
    ref["loss"].backward()
    np.testing.assert_allclose(loss.item(), ref["loss"].item(), rtol=2e-4)
    _check_param_grads(model, lambda n: sd[n].grad, 1e-2 if pretrain else 1e-3)


def test_pose_operator_backward():
    """se3.exp backward vs float64 CPU autograd of the oracle's se3_exp over twists with |omega| < 0.01 (Taylor
    branch) and |omega| > 1 (max abs error <= 1e-5); comp backward vs torch autograd of the oracle's comp (rtol
    1e-5); without grad nothing is recorded"""
    from puzzlenet_b200 import losses, se3
    g = torch.Generator().manual_seed(11)
    n = 64
    w = torch.randn(n, 3, generator=g)
    w = w / w.norm(dim=1, keepdim=True)
    mag = torch.cat([torch.rand(n // 2, generator=g) * 0.009 + 1e-4, torch.rand(n // 2, generator=g) * 2 + 1.0])
    x = torch.cat([w * mag[:, None], torch.randn(n, 3, generator=g)], 1)
    dg = torch.randn(n, 4, 4, generator=g)
    xd = x.to(DEV).requires_grad_()
    gd = se3.exp(xd)
    (gd * dg.to(DEV)).sum().backward()
    xr = x.double().requires_grad_()
    (po.se3_exp(xr) * dg.double()).sum().backward()
    err = (xd.grad.cpu().double() - xr.grad).abs().max().item()
    assert err <= 1e-5, err
    assert se3.exp(x.to(DEV)).grad_fn is None
    # comp
    gm = torch.randn(n, 4, 4, generator=g)
    igt = po.se3_exp(torch.randn(n, 6, generator=g) * 0.3)
    gmd = gm.to(DEV).requires_grad_()
    (3.0 * losses.comp(gmd, igt.to(DEV))).backward()
    gmr = gm.double().requires_grad_()
    (3.0 * po.comp(gmr, igt.double())).backward()
    np.testing.assert_allclose(gmd.grad.cpu().numpy(), gmr.grad.numpy(), rtol=1e-5, atol=1e-6 * gmr.grad.abs().max().item())
    assert losses.comp(gm.to(DEV), igt.to(DEV)).grad_fn is None


def test_default_records_no_graph():
    model = _fresh_model(differentiable=False)
    batch = [t.to(DEV) for t in training_inputs(2, po.se3_exp)]
    batch[0].requires_grad_()
    r = model.predict5(batch, 2, need=True, training=True, starts=_starts(2))
    assert not any(t.requires_grad for t in (r[0], r[2], r[3], r[4], r[5], r[6], r[7]))
    with pytest.raises(NotImplementedError):
        model.predict6(batch, 2, training=True, pretrain=True)


def _grads(model):
    return {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}


def _disagree(got, ref):
    """tensors whose gradients differ by more than fp32 summation-order noise: relative L2 1e-5, and 1e-3 for the q / k
    projections, whose gradient cancels nearly equal terms in the softmax Jacobian of the near-one-hot attention
    rows (see test_tf32_training_step_close_to_fp32) and so amplifies the order of the backward's fp32 atomics
    (measured up to 1.1e-4 between two identical backward passes on a B200).  Overwritten saved activations would
    show up as O(1) differences."""
    bad = {}
    for n in ref:
        tol = 1e-3 if ".mlpq." in n or ".mlpk." in n else 1e-5
        if not n.endswith("mlpk.bias") and not _rel(got[n], ref[n]) < tol:
            bad[n] = _rel(got[n], ref[n])
    return bad


def _zero(model):
    for p in model.parameters():
        p.grad = None


def test_graph_ownership_and_fresh_gradient_buffers():
    from puzzlenet_b200.training import Trainer
    B = 2
    full = [t.to(DEV) for t in training_inputs(2 * B, po.se3_exp)]
    ba, bb = [t[:B] for t in full], [t[B:] for t in full]
    sa, sb = _starts(B, 1), _starts(B, 2)
    w = [t.to(DEV) for t in _weights(B)]
    model = _fresh_model()
    model._trainer_state = Trainer(model, lr=0.0)       # training_step below must leave the weights as they are

    def loss_of(batch, st):
        r = model.predict5(batch, B, need=True, training=True, starts=st)
        return _custom_loss(r[0], r[6], r[7], r[3], r[4], w, (1, 1, 1, 1, 0))

    # separate runs: the gradients accumulate into .grad
    loss_of(ba, sa).backward()
    loss_of(bb, sb).backward()
    sep = _grads(model)
    _zero(model)
    # two graphs alive at once, one backward through both
    (loss_of(ba, sa) + loss_of(bb, sb)).backward()
    both = _grads(model)
    bad = _disagree(both, sep)
    assert not bad, bad
    # training_step and predict5_train between a forward and its backward do not touch its saved state
    _zero(model)
    loss_of(ba, sa).backward()
    ref = _grads(model)
    _zero(model)
    L = loss_of(ba, sa)
    model.training_step(bb, 0, starts=sb)
    model.trainer_state().predict5_train(bb[0], bb[1], sb)
    L.backward()
    got = _grads(model)
    bad = _disagree(got, ref)
    assert not bad, bad
    with pytest.raises(RuntimeError):
        L.backward()                                    # the graph was freed by the first backward
    # successive backward calls never share gradient storage, with each other or with the Trainer's buffer
    first = {n: p.grad for n, p in model.named_parameters() if p.grad is not None}
    _zero(model)
    loss_of(ba, sa).backward()
    flat = model.trainer_state().flat.grads.untyped_storage().data_ptr()
    for n, p in model.named_parameters():
        if p.grad is not None:
            s = p.grad.untyped_storage().data_ptr()
            assert s != first[n].untyped_storage().data_ptr() and s != flat, n
    # activations are released with the graph: memory returns to its level before the forward
    del first, got, ref, L
    _zero(model)
    torch.cuda.synchronize()
    m0 = torch.cuda.memory_allocated()
    L = loss_of(ba, sa)
    assert torch.cuda.memory_allocated() > m0 + (10 << 20)
    del L
    assert torch.cuda.memory_allocated() == m0
    L = loss_of(ba, sa)
    L.backward()
    del L
    _zero(model)
    assert torch.cuda.memory_allocated() == m0


def test_torch_optim_adam_lowers_loss_and_eval_sees_the_update():
    """three torch.optim.Adam steps over model.parameters() with a custom loss on a fixed batch lower the loss; eval
    predict5 (split precision) afterwards agrees with the oracle on the updated state dict at the split tolerances"""
    B = 2
    batch = [t.to(DEV) for t in training_inputs(B, po.se3_exp)]
    st = _starts(B)
    model = _fresh_model()
    opt = torch.optim.Adam(model.parameters(), lr=1e-5)

    def step():
        opt.zero_grad()
        r = model.predict5(batch, B, training=True, starts=st)
        loss = r[0].pow(2).mean() + F.cross_entropy(r[2], batch[6].long()) + F.cross_entropy(r[3], batch[7].long())
        loss.backward()
        opt.step()
        return loss.item()

    seen = [step() for _ in range(4)]
    assert all(np.isfinite(seen)) and seen[3] < seen[2] < seen[1] < seen[0], seen
    model.eval()
    model.precision = "split"
    out, _, de_f, de_m = model.predict5(make_batch(batch[0], batch[1]), B, starts=st)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    assert not torch.equal(sd["tfMLP.0.weight"], synthetic_state_dict(0)["tfMLP.0.weight"])
    ref = po.predict5(sd, batch[0].cpu(), batch[1].cpu(), starts=((st[0], st[1]), (st[2], st[3])))
    for got, key in ((out, "out"), (de_f, "de_fpcb"), (de_m, "de_mrpcb")):
        err = (got.cpu() - ref[key]).abs().max() / ref[key].abs().max()
        assert err < 1e-4, (key, err.item())


def test_tf32_trainer_gradients_close_to_fp32():
    """with a TF32 Trainer installed the arbitrary-gradient loss's parameter gradients agree with fp32 within the
    tolerances of test_tf32_training_step_close_to_fp32 (relative L2 1e-1, cosine 0.99; 0.9 for q / k)"""
    from puzzlenet_b200.training import Trainer
    B = 2
    batch = [t.to(DEV) for t in training_inputs(B, po.se3_exp)]
    st = _starts(B)
    w = [t.to(DEV) for t in _weights(B)]
    res = {}
    for prec in ("fp32", "tf32"):
        model = _fresh_model()
        model._trainer_state = Trainer(model, model.C, precision=prec)
        r = model.predict5(batch, B, need=True, training=True, starts=st)
        _custom_loss(r[0], r[6], r[7], r[3], r[4], w, (1, 1, 1, 1, 1)).backward()
        res[prec] = _grads(model)
    worst = {}
    for n, g32 in res["fp32"].items():
        if n.endswith("mlpk.bias") or g32.numel() < 4096:
            continue
        gtf = res["tf32"][n]
        cos = torch.dot(gtf.flatten(), g32.flatten()) / (gtf.norm() * g32.norm()).clamp_min(1e-30)
        qk = ".mlpq." in n or ".mlpk." in n
        assert cos.item() > (0.9 if qk else 0.99), (n, cos.item())
        if not qk:
            worst[n] = _rel(gtf, g32)
    bad = {k: v for k, v in worst.items() if not v < 1e-1}
    assert not bad, bad
    assert max(worst.values()) > 1e-6          # the tensor-core path really ran
