"""GPU: pair scoring from per-piece encodings (TouchedRegraster.encode_pieces / predict_pairs, EmbeddingScorer) gives
what predict5 gives for the same pairs with the same FPS starts -- bit for bit, in every precision."""
import numpy as np
import pytest
import torch

from oracle import parity

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PRECISIONS = ["fp32", "bf16", "split"]


@pytest.fixture
def model(cuda_model):
    yield cuda_model
    cuda_model.precision = "fp32"


def _clouds(P, seed):
    return torch.rand(P, 1024, 3, generator=torch.Generator().manual_seed(seed)).to(DEV) - 0.5


def _predict5_pairs(model, clouds, starts, pairs):
    """predict5 on the batch (clouds[I], clouds[J]) with the pieces' own starts (I = fpc pieces, J = mrpc pieces)."""
    from puzzlenet_b200.weights import make_batch
    I, J = pairs[:, 0], pairs[:, 1]
    st = torch.stack([starts[0, I], starts[1, I], starts[2, J], starts[3, J]]).contiguous()
    return model.predict5(make_batch(clouds[I.to(DEV)], clouds[J.to(DEV)]), pairs.shape[0], starts=st)


def _assert_equal_and_within(got, ref, precision):
    p = parity.predict5_parity(None, got[0], None, None, got[0], got[2], got[3],
                               ref=dict(out=ref[0].cpu(), de_fpcb=ref[2].cpu(), de_mrpcb=ref[3].cpu()))
    assert parity.within(p, precision), p
    for k in (0, 2, 3):
        assert torch.equal(got[k], ref[k]), (k, (got[k] - ref[k]).abs().max().item())


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("P", [1, 5, 64])
def test_diagonal_pairs_equal_predict5_bitwise(model, precision, P):
    from puzzlenet_b200.weights import make_batch
    model.precision = precision
    c = _clouds(P, 10 + P)
    torch.manual_seed(7)
    emb = model.encode_pieces(c)
    got = model.predict_pairs(emb, torch.arange(P).repeat(2, 1).T)
    torch.manual_seed(7)
    ref = model.predict5(make_batch(c, c), P)
    for k in (0, 2, 3):
        assert torch.equal(got[k], ref[k]), (k, (got[k] - ref[k]).abs().max().item())


def _arbitrary_pairs():
    """45 pairs over 7 pieces: i == j, repeats, both orders, a count that is no multiple of 4, 16 or 64."""
    fixed = torch.tensor([[0, 0], [6, 6], [1, 2], [2, 1], [1, 2], [6, 0], [0, 6], [3, 3], [3, 3]])
    rnd = torch.randint(0, 7, (36, 2), generator=torch.Generator().manual_seed(5))
    return torch.cat([fixed, rnd])


@pytest.mark.parametrize("precision", PRECISIONS)
def test_arbitrary_pairs_equal_predict5(model, precision):
    model.precision = precision
    c = _clouds(7, 21)
    pairs = _arbitrary_pairs()
    assert pairs.shape == (45, 2)
    torch.manual_seed(3)
    emb = model.encode_pieces(c)
    got = model.predict_pairs(emb, pairs)
    ref = _predict5_pairs(model, c, emb.starts, pairs)
    _assert_equal_and_within(got, ref, precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_reencode_and_chunked_encoding(model, precision):
    """re-encoding a subset in place, and P > 64 (two pz_encode_pieces calls), give the same pairs as predict5."""
    model.precision = precision
    P = 70
    c = _clouds(P, 31)
    torch.manual_seed(4)
    emb = model.encode_pieces(c)
    c2 = c.clone()
    c2[[3, 66]] = _clouds(2, 32)
    emb.reencode(model, [3, 66], c2[[3, 66]])
    pairs = torch.tensor([[3, 66], [66, 3], [3, 3], [0, 69], [69, 64], [65, 1], [66, 66]])
    _assert_equal_and_within(model.predict_pairs(emb, pairs), _predict5_pairs(model, c2, emb.starts, pairs), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_predict_pairs_graph_capture(model, precision):
    model.precision = precision
    c = _clouds(7, 41)
    pairs = _arbitrary_pairs()
    torch.manual_seed(5)
    emb = model.encode_pieces(c)
    eager = model.predict_pairs(emb, pairs)
    pairs_dev = pairs.to(DEV)
    outs = [torch.full_like(eager[k], float("nan")) for k in (0, 2, 3)]
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        model._launch_pairs(emb, pairs_dev, *outs)
    graph.replay()
    torch.cuda.synchronize()
    for got, ref in zip(outs, (eager[0], eager[2], eager[3])):
        assert torch.equal(got, ref)


class _Predict5Scorer:
    """the same rows through predict5, with the FPS starts of each pair's pieces"""

    def __init__(self, model, starts):
        self.model, self.starts = model, starts

    def score_indexed(self, clouds, pairs):
        from puzzlenet_b200 import assembly, losses
        out6, _, de_f, de_m = _predict5_pairs(self.model, clouds, self.starts, pairs)
        idx = pairs.to(clouds.device)
        s = losses.pair_score(out6, de_f, de_m, clouds[idx[:, 0]], clouds[idx[:, 1]])
        rows = torch.empty(pairs.shape[0], assembly.ROW_COLS, device=clouds.device)
        rows[:, :6], rows[:, 6], rows[:, 7] = out6, s[:, 10], 1.0
        return rows


@pytest.mark.parametrize("precision", PRECISIONS)
def test_embedding_scorer_matches_predict5_scorer(model, precision):
    from puzzlenet_b200 import assembly
    model.precision = precision
    c = _clouds(8, 51)
    torch.manual_seed(6)
    scorer = assembly.EmbeddingScorer(model)
    pairs, rows = assembly.score_all_pairs(c, scorer)
    assert scorer.encoded == 8
    _, ref_rows = assembly.score_all_pairs(c, _Predict5Scorer(model, scorer.emb.starts))
    assert torch.isfinite(rows).all() and torch.all(rows[:, 7] == 1)
    rel = parity.rel(rows, ref_rows.cpu())
    assert rel < parity.BOUNDS[precision][0], rel
    assert torch.equal(rows, ref_rows)
    poses, _, merges = assembly.greedy_assemble(8, pairs, rows)
    ref_poses, _, ref_merges = assembly.greedy_assemble(8, pairs, ref_rows)
    assert [m[:2] for m in merges] == [m[:2] for m in ref_merges]
    np.testing.assert_allclose(poses, ref_poses, atol=1e-5)
    # unchanged clouds: nothing is encoded again
    assembly.score_all_pairs(c, scorer)
    assert scorer.encoded == 8


@pytest.mark.parametrize("precision", PRECISIONS)
def test_assemble_rescore_reencodes_one_piece_per_merge(model, precision):
    from puzzlenet_b200 import assembly
    model.precision = precision
    clouds = _clouds(6, 4)
    scorer = assembly.EmbeddingScorer(model)
    deltas = []
    score_indexed = scorer.score_indexed

    def counting(cl, pairs):
        before = scorer.encoded
        r = score_indexed(cl, pairs)
        deltas.append(scorer.encoded - before)
        return r

    scorer.score_indexed = counting
    torch.manual_seed(0)
    poses, merges = assembly.assemble(clouds, scorer, batch=64, rescore=True)
    assert poses.shape == (6, 4, 4) and len(merges) == 5
    for k in range(6):                                       # every pose is a rigid motion
        R = poses[k][:3, :3]
        np.testing.assert_allclose(R @ R.T, np.eye(3), atol=1e-5)
        np.testing.assert_allclose(poses[k][3], [0, 0, 0, 1], atol=1e-12)
    np.testing.assert_allclose(poses[0], np.eye(4), atol=1e-12)   # pairs are i < j: piece 0 ends up as the root
    # the first pass encodes all 6 pieces; each merge that leaves pieces to re-score re-encodes the merged one only
    assert deltas == [6, 1, 1, 1, 1], deltas


def test_trainer_step_makes_embeddings_stale(state_dict):
    """an Adam step writes the parameters through raw pointers: embeddings from before it are rejected, and a scorer
    re-encodes every piece and then agrees with predict5 under the new weights"""
    import types
    from puzzlenet_b200 import assembly
    from puzzlenet_b200.model5_b import TouchedRegraster
    from puzzlenet_b200.training import Trainer
    model = TouchedRegraster(types.SimpleNamespace(dataset="vase", loss_mode=1, loss_sum=False, lr=0.9e-3))
    model.load_state_dict(state_dict, strict=True)
    model.to(DEV)
    tr = Trainer(model, lr=1e-3)
    c = _clouds(4, 61)
    pairs = torch.tensor([[0, 1], [2, 3], [3, 0]])
    scorer = assembly.EmbeddingScorer(model)
    torch.manual_seed(8)
    before = scorer.score_indexed(c, pairs)
    emb = scorer.emb
    tr.flat.grads.copy_(torch.randn(tr.flat.n, generator=torch.Generator().manual_seed(0)) * 0.1)
    tr.optimizer_step()
    with pytest.raises(ValueError, match="stale"):
        model.predict_pairs(emb, pairs)
    after = scorer.score_indexed(c, pairs)
    assert scorer.encoded == 8 and scorer.emb is not emb
    assert not torch.equal(after, before)
    assert torch.equal(after, _Predict5Scorer(model, scorer.emb.starts).score_indexed(c, pairs))
