"""Multi-piece assembly on top of the pair network (SURVEY.md §3.5 / §8 row F3, BASELINE config 5).

The reference ships no code for this step (SURVEY D10), only the description: run the pair network on every
candidate pair of pieces, score a pair by the distance between the two predicted boundaries after the predicted
alignment -- the quantity ``test_step`` computes as ``cd_fpc`` / ``cd_rpc`` (model5_b.py:1351-1358) -- and merge
greedily.  This module supplies

* :func:`downsample_pieces` -- FPS 11000 -> 1024 of every piece, pieces sharded over ranks, one ``all_gather``;
* :func:`score_pairs` / :func:`score_all_pairs` -- batched ``predict5`` + one ``pz_pair_score`` launch per batch
  (:class:`ModelScorer`), or per-piece encodings + pair heads (:class:`EmbeddingScorer`), candidate pairs sharded over
  ranks, ONE ``all_gather`` of ``[n_pairs, 8]`` rows (twist 6, score, 1.0);
* :func:`greedy_assemble` -- host-side greedy merge (Kruskal over the score table) composing the pair poses into one
  pose per piece;
* :func:`assemble` -- the optional re-scoring loop: after each merge the merged piece is re-sampled to 1024 points
  and re-scored against the remaining pieces.

No data-path collective inside the forward; NCCL (or gloo in the CPU tests) only moves the final rows.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import sharding

ROW_COLS = 8      # twist (omega, v) [6], pair score, valid flag


class ModelScorer:
    """``scorer(fpc [b,1024,3], mrpc [b,1024,3]) -> rows [b, ROW_COLS]`` through the CUDA library:
    one ``pz_predict5`` and one ``pz_pair_score`` (assembly mode: ``src = mrpc``, no ground truth)."""

    def __init__(self, model, pipes: int = 1):
        """``pipes`` > 1: :func:`score_pairs` spreads its batches round-robin over that many CUDA streams (batches are
        independent), so the latency-bound stages of one batch overlap the tensor-core stages of the others -- the
        schedule ``bench.py`` times.  Combine with ``model.cuda_graphs = True`` for one graph replay per batch."""
        self.model = model
        self.pipes = max(1, int(pipes))
        self._streams = {}

    def streams(self, device):
        key = str(device)
        if key not in self._streams:
            self._streams[key] = [torch.cuda.Stream(device=device) for _ in range(self.pipes)]
        return self._streams[key]

    def __call__(self, fpc: torch.Tensor, mrpc: torch.Tensor) -> torch.Tensor:
        from . import losses
        from .weights import make_batch
        out6, _, de_f, de_m = self.model.predict5(make_batch(fpc, mrpc), fpc.shape[0])
        s = losses.pair_score(out6, de_f, de_m, fpc, mrpc)
        rows = torch.empty(fpc.shape[0], ROW_COLS, device=fpc.device, dtype=torch.float32)
        rows[:, :6] = out6
        rows[:, 6] = s[:, 10]
        rows[:, 7] = 1.0
        return rows


class EmbeddingScorer:
    """``scorer.score_indexed(clouds [P,1024,3], pairs [n,2]) -> rows [n, ROW_COLS]``: the rows :class:`ModelScorer`
    gives, computed from per-piece encodings -- every piece goes through both encoders once
    (``TouchedRegraster.encode_pieces``), each pair through the pose MLP and the fpc boundary head only
    (``predict_pairs``), then one ``pz_pair_score`` launch.

    The scorer keeps the embeddings of the clouds it last saw and a device copy of those clouds.  On each call it
    compares the copy with ``clouds`` (one host synchronisation) and re-encodes only the pieces whose rows changed, so
    ``assemble(rescore=True)`` re-encodes one piece per merge; a change of the model's parameters or precision
    re-encodes every piece.  FPS starts are drawn from the CPU generator as ``encode_pieces`` / ``reencode`` draw them.
    Under ``torch.distributed`` the pairs stay sharded by :func:`score_all_pairs` and every rank encodes all P pieces
    itself (replicated work, cheap at P = 32); the ranks' CPU generators must then be seeded alike, as they are for
    ``ModelScorer``.  Pairs are scored ``chunk`` at a time (one ``predict_pairs`` and one ``pz_pair_score`` per chunk),
    which bounds the memory of a call."""

    def __init__(self, model, chunk: int = 4096):
        self.model = model
        self.chunk = max(1, int(chunk))
        self.emb = None
        self._clouds = None
        self.encoded = 0          # pieces encoded so far

    def _refresh(self, clouds: torch.Tensor) -> None:
        emb, m = self.emb, self.model
        if (emb is None or self._clouds.shape != clouds.shape or self._clouds.device != clouds.device
                or not emb.is_current(m)):
            self.emb = m.encode_pieces(clouds)
            self._clouds = clouds.clone()
            self.encoded += clouds.shape[0]
            return
        changed = torch.nonzero((self._clouds != clouds).flatten(1).any(1)).flatten().tolist()
        if changed:
            emb.reencode(m, changed, clouds[changed])
            self._clouds[changed] = clouds[changed]
            self.encoded += len(changed)

    def score_indexed(self, clouds: torch.Tensor, pairs: torch.Tensor) -> torch.Tensor:
        from . import losses
        rows = torch.empty(pairs.shape[0], ROW_COLS, device=clouds.device, dtype=torch.float32)
        if pairs.shape[0] == 0:
            return rows
        clouds = clouds.contiguous().float()
        self._refresh(clouds)
        for lo in range(0, pairs.shape[0], self.chunk):
            sel = pairs[lo:lo + self.chunk]
            out6, _, de_f, de_m = self.model.predict_pairs(self.emb, sel)
            idx = sel.to(clouds.device)
            s = losses.pair_score(out6, de_f, de_m, clouds[idx[:, 0]], clouds[idx[:, 1]])
            r = rows[lo:lo + sel.shape[0]]
            r[:, :6] = out6
            r[:, 6] = s[:, 10]
            r[:, 7] = 1.0
        return rows


def downsample_pieces(pieces: Sequence, npoints: int = 1024, starts: Optional[Sequence[int]] = None,
                      device=None) -> torch.Tensor:
    """[P, npoints, 3]: every raw piece ([N_i, 3], N_i <= 16384) farthest-point-sampled on the GPU
    (``dataset.fps_batch`` = ``CADDataset.fps``, dataset.py:1147-1163).  Under ``torch.distributed`` rank r samples
    its contiguous share of the pieces and the results are all-gathered (393 KB for 32 pieces)."""
    from . import dataset
    P = len(pieces)
    if starts is None:
        starts = [np.random.randint(0, int(p.shape[0])) for p in pieces]     # drawn on every rank alike

    def fn(lo, hi):
        if hi == lo:
            dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
            return torch.empty(0, npoints, 3, device=dev)
        return dataset.fps_batch(pieces[lo:hi], npoints, starts=list(starts[lo:hi]), device=device)

    return sharding.run_sharded(P, fn)


def score_pairs(clouds: torch.Tensor, pairs: torch.Tensor, scorer: Callable, batch: int = 64) -> torch.Tensor:
    """rows [len(pairs), ROW_COLS] for the given (i, j) index pairs: piece i is the fixed cloud (``fpc``), piece j
    the one the predicted pose moves (``mrpc``).  Local, no communication.  A scorer with ``score_indexed`` (such as
    :class:`EmbeddingScorer`) gets the whole list at once."""
    if hasattr(scorer, "score_indexed"):
        return scorer.score_indexed(clouds, pairs)
    n = pairs.shape[0]
    rows = torch.empty(n, ROW_COLS, device=clouds.device, dtype=torch.float32)
    pairs = pairs.to(clouds.device)
    pipes = int(getattr(scorer, "pipes", 1))
    if pipes > 1 and n > batch and clouds.is_cuda:
        cur = torch.cuda.current_stream(clouds.device)
        streams = scorer.streams(clouds.device)
        for st in streams:
            st.wait_stream(cur)
        for bi, lo in enumerate(range(0, n, batch)):
            with torch.cuda.stream(streams[bi % pipes]):
                sel = pairs[lo:lo + batch]
                rows[lo:lo + sel.shape[0]] = scorer(clouds[sel[:, 0]].contiguous(), clouds[sel[:, 1]].contiguous())
        for st in streams:
            cur.wait_stream(st)
        return rows
    for lo in range(0, n, batch):
        sel = pairs[lo:lo + batch]
        rows[lo:lo + sel.shape[0]] = scorer(clouds[sel[:, 0]].contiguous(), clouds[sel[:, 1]].contiguous())
    return rows


def score_all_pairs(clouds: torch.Tensor, scorer: Callable, batch: int = 64,
                    pairs: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """All P(P-1)/2 unordered pairs (or the given list), sharded over the ranks of the default process group;
    every rank returns the full ``(pairs [n,2], rows [n, ROW_COLS])`` after one all_gather."""
    if pairs is None:
        pairs = sharding.all_pairs(clouds.shape[0])
    rows = sharding.run_sharded(pairs.shape[0], lambda lo, hi: score_pairs(clouds, pairs[lo:hi], scorer, batch))
    return pairs, rows


# ----------------------------------------------------------------------------- host-side greedy merge

def _se3_exp_np(x: np.ndarray) -> np.ndarray:
    """se_math/se3.py:57-80 in float64 (host-side pose composition only).  Scalar arithmetic on Python floats: the
    31 calls of one assembly were the largest part of the host-side merge when written with 3x3 numpy temporaries."""
    import math
    w0, w1, w2, v0, v1, v2 = (float(t) for t in x[:6])
    t = math.sqrt(w0 * w0 + w1 * w1 + w2 * w2)
    if abs(t) < 0.01:
        t2 = t * t
        s1 = 1 - t2 / 6 * (1 - t2 / 20 * (1 - t2 / 42))
        s2 = 0.5 * (1 - t2 / 12 * (1 - t2 / 30 * (1 - t2 / 56)))
        s3 = 1 / 6 * (1 - t2 / 20 * (1 - t2 / 42 * (1 - t2 / 72)))
    else:
        s1, s2, s3 = math.sin(t) / t, (1 - math.cos(t)) / t ** 2, (t - math.sin(t)) / t ** 3
    # W = [[0,-w2,w1],[w2,0,-w0],[-w1,w0,0]];  S = W W = w w^T - |w|^2 I
    W = ((0.0, -w2, w1), (w2, 0.0, -w0), (-w1, w0, 0.0))
    ww = (w0, w1, w2)
    n2 = t * t
    v = (v0, v1, v2)
    g = np.eye(4)
    for r in range(3):
        pr = 0.0
        for c in range(3):
            S_rc = ww[r] * ww[c] - (n2 if r == c else 0.0)
            g[r, c] = (1.0 if r == c else 0.0) + s1 * W[r][c] + s2 * S_rc
            pr += ((1.0 if r == c else 0.0) + s2 * W[r][c] + s3 * S_rc) * v[c]
        g[r, 3] = pr
    return g


def greedy_assemble(n_pieces: int, pairs, rows, max_score: Optional[float] = None):
    """Greedy merge over a fixed score table: visit candidate pairs by ascending score and accept a pair when its
    pieces are still in different components (Kruskal).  A pair (i, j) with twist x says ``exp(x)`` maps piece j
    into piece i's frame, so accepting it re-expresses j's whole component in i's component frame.

    Returns ``(poses [P,4,4] float64, component [P] int, merges)``: ``poses[k]`` maps piece k into the frame of its
    component's root piece; ``merges`` = ``[(i, j, score), ...]`` in acceptance order.  Pairs scoring above
    ``max_score`` are never accepted (several components may remain)."""
    pairs = np.asarray(pairs.cpu() if isinstance(pairs, torch.Tensor) else pairs, dtype=np.int64).reshape(-1, 2)
    rows = np.asarray(rows.cpu() if isinstance(rows, torch.Tensor) else rows, dtype=np.float64).reshape(-1, ROW_COLS)
    if pairs.shape[0] != rows.shape[0]:
        raise ValueError("greedy_assemble: pairs and rows disagree in length")
    poses = np.tile(np.eye(4), (n_pieces, 1, 1))
    merges: List[Tuple[int, int, float]] = []
    order = np.lexsort((np.arange(rows.shape[0]), rows[:, 6]))        # ascending score, ties by pair order
    # the edge loop runs on plain Python lists (a numpy scalar access per edge costs more than the whole merge logic);
    # `members[c]` lists the pieces of component c, `comp[k]` is piece k's component
    score = rows[:, 6].tolist()
    valid = ((rows[:, 7] != 0) & np.isfinite(rows[:, 6])).tolist()
    pi, pj = pairs[:, 0].tolist(), pairs[:, 1].tolist()
    comp = list(range(n_pieces))
    members = {k: [k] for k in range(n_pieces)}
    for e in order.tolist():
        if not valid[e]:
            continue
        if max_score is not None and score[e] > max_score:
            break
        i, j = pi[e], pj[e]
        ci, cj = comp[i], comp[j]
        if ci == cj:
            continue
        # new pose of every piece k in j's component:  T_i . g_ij . T_j^-1 . T_k   (T_j is rigid: inverse = [R^T, -R^T t])
        tj = poses[j]
        tj_inv = np.eye(4)
        tj_inv[:3, :3] = tj[:3, :3].T
        tj_inv[:3, 3] = -tj[:3, :3].T @ tj[:3, 3]
        move = poses[i] @ _se3_exp_np(rows[e, :6]) @ tj_inv
        moved = members.pop(cj)
        poses[moved] = move @ poses[moved]
        for k in moved:
            comp[k] = ci
        members[ci] += moved
        merges.append((i, j, score[e]))
        if len(merges) == n_pieces - 1:
            break
    return poses, np.asarray(comp), merges


def assemble(clouds: torch.Tensor, scorer: Callable, batch: int = 64, rescore: bool = True,
             max_score: Optional[float] = None):
    """Greedy assembly of P pieces ([P,1024,3] on the GPU).

    ``rescore=False``: one sharded all-pairs pass + :func:`greedy_assemble`.
    ``rescore=True``: after each merge the two pieces are replaced by their union in the fixed piece's frame,
    re-sampled to 1024 points (``dataset.fps``-style FPS from point 0), and only the pairs that involve the merged
    piece are re-scored (the next P-2 pairs, sharded like the first pass).

    Returns ``(poses [P,4,4] float64 numpy, merges)`` with ``poses[k]`` mapping original piece k into the frame of
    the surviving root piece."""
    P = clouds.shape[0]
    pairs, rows = score_all_pairs(clouds, scorer, batch)
    if not rescore:
        poses, _, merges = greedy_assemble(P, pairs, rows, max_score)
        return poses, merges
    from . import dataset
    clouds = clouds.clone()
    alive = list(range(P))
    poses = np.tile(np.eye(4), (P, 1, 1))
    members = {k: [k] for k in range(P)}
    table = {(int(a), int(b)): r for (a, b), r in zip(pairs.tolist(), rows.cpu().numpy().astype(np.float64))}
    merges = []
    while len(alive) > 1:
        cand = [(r[6], a, b) for (a, b), r in table.items() if np.isfinite(r[6])]
        if not cand:
            break
        score, i, j = min(cand)
        if max_score is not None and score > max_score:
            break
        g = _se3_exp_np(table[(i, j)][:6])
        for k in members[j]:
            poses[k] = g @ poses[k]          # i < j: piece i keeps its frame, j's members move into it
        # clouds[] always holds a piece in its own root frame, so the union is  cloud_i U g . cloud_j
        gj = torch.from_numpy(g).to(clouds.device, torch.float32)
        moved = clouds[j] @ gj[:3, :3].T + gj[:3, 3]
        union = torch.cat([clouds[i], moved], dim=0)
        clouds[i] = dataset.fps(union, 1024, start=0)
        members[i] += members.pop(j)
        alive.remove(j)
        merges.append((i, j, float(score)))
        table = {k: v for k, v in table.items() if i not in k and j not in k}
        others = [k for k in alive if k != i]
        if others:
            new_pairs = torch.tensor([(min(i, k), max(i, k)) for k in others], dtype=torch.int64)
            _, new_rows = score_all_pairs(clouds, scorer, batch, pairs=new_pairs)
            for (a, b), r in zip(new_pairs.tolist(), new_rows.cpu().numpy().astype(np.float64)):
                table[(a, b)] = r
    return poses, merges
