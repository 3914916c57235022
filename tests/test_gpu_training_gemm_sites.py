"""Every matrix product of the training step, replayed at the configuration the step issues it with and checked
against a float64 reference.

A proxy in place of ``training._lib`` records each ``pz_sgemm`` / ``pz_gemm_tf32`` / ``pz_gemm_tf32_batched`` call of
``Trainer.forward_backward`` and ``forward_backward_pretrain`` (fp32 and TF32, 8 and 64 pairs): sizes, leading
dimensions, batch strides, split-K, alpha / beta and the epilogue flags, which optional operands were given, and each
pointer's address mod 16.  Each distinct configuration is then replayed on buffers laid out exactly as the call
addresses them:

* every input element inside the allocation but outside the logical operand (the gap between a row's width and its
  stride, between batches, and before an operand that starts at a 4- / 8- / 12-byte offset) is NaN, so a read outside
  the operand shows up as NaN in the result;
* every output element outside the M x N windows holds a finite sentinel that must survive the call;
* a window the call does not read starts as NaN, so an element the kernel never writes is caught as well.

Two passes per configuration:

* exact: small-integer operands (K * max|a| * max|b| <= 2^22) are exact in TF32 and fp32 and so are all partial
  sums, whatever the accumulation order, split-K partition or atomic order -- the result must EQUAL the float64
  reference, which checks addressing, tiling, k coverage and the epilogue order;
* precision: |C - ref| <= 2^-10 (|A||B|) + n 2^-24 S for TF32 and <= n 2^-24 S for pz_sgemm, with S the magnitude sum
  of every term and n = ceil(K / splitk) + splitk + 2 the longest fp32 rounding chain.  The operands are normal
  magnitudes whose 16 bits below the bf16 mantissa read 0x4CCC, with signs chosen so that every product a_ik b_kj is
  >= 0: rounding them to TF32 (nearest or toward zero) shrinks every product by 0.4 - 0.8 x 2^-10 of itself, to bf16
  by 2.4 - 4.8 x 2^-10, and those losses add up instead of cancelling.  With random signs and random low bits they
  would cancel like a random walk, and a product that silently ran at lower precision would still fit the
  worst-case bounds once K reaches a few thousand.

The CPU tests run the same builder and checks on torch emulations of hand-written configurations, with and without
injected faults, to show that each check catches what it is meant to catch.
"""
import dataclasses
import math
import time
import types

import pytest
import torch

ENTRIES = ("pz_sgemm", "pz_gemm_tf32", "pz_gemm_tf32_batched")
SENTINEL = -7777.25
OPERANDS = ("A", "B", "C", "bias", "mask", "residual")
# a product of two operands that lost the 13 bits below the TF32 mantissa loses at least this fraction of itself
# (precision fill: both operands shrink by 0.4 TF32 ulp, 0.2 - 0.4 x 2^-10 of their value)
TF32_LOSS_FLOOR = 0.4 * 2.0 ** -10


@dataclasses.dataclass(frozen=True)
class Site:
    """One GEMM call as the step makes it.  ``ta``: pz_sgemm transA / pz_gemm_tf32 a_mn_major (A stored K x M,
    A[k*lda + m]).  ``tb``: pz_sgemm transB (B stored N x K) / pz_gemm_tf32 b_mn_major (B stored K x N).
    ``align``: byte address mod 16 of A, B, C, bias, mask, residual (0 where absent)."""
    entry: str
    ta: int
    tb: int
    M: int
    N: int
    K: int
    lda: int
    ldb: int
    ldc: int
    batch: int = 1
    sa: int = 0
    sb: int = 0
    sc: int = 0
    splitk: int = 1
    alpha: float = 1.0
    beta: float = 0.0
    accumulate: int = 0
    relu: int = 0
    bias: bool = False
    mask: bool = False
    residual: bool = False
    ldmask: int = 0
    ldres: int = 0
    align: tuple = (0, 0, 0, 0, 0, 0)

    @property
    def tf32(self):
        return self.entry != "pz_sgemm"

    @property
    def beta_eff(self):
        return 1.0 if self.accumulate else self.beta

    @property
    def reads_c(self):
        return self.splitk > 1 or self.beta_eff != 0.0

    @property
    def chain(self):
        """longest chain of fp32 roundings one output element goes through"""
        return -(-self.K // self.splitk) + self.splitk + 2


def site_of_call(name, args):
    """the Site of one recorded ``_lib.call(name, *args)``"""
    mod16 = lambda p: 0 if p is None else int(p) % 16  # noqa: E731
    if name == "pz_sgemm":
        (ta, tb, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, batch, sa, sb, sc, splitk, bias, relu, mask, ldmask,
         res, ldres, _) = args
        acc = 0
    else:
        if name == "pz_gemm_tf32":
            ta, tb, M, N, K, A, lda, B, ldb, C, ldc, splitk, bias, relu, mask, ldmask, acc, _ = args
            batch, sa, sb, sc = 1, 0, 0, 0
        else:
            (ta, tb, M, N, K, A, lda, B, ldb, C, ldc, batch, sa, sb, sc, splitk, bias, relu, mask, ldmask, acc,
             _) = args
        alpha, beta, res, ldres = 1.0, 0.0, None, 0
    return Site(name, int(ta), int(tb), int(M), int(N), int(K), int(lda), int(ldb), int(ldc), int(batch), int(sa),
                int(sb), int(sc), int(splitk), float(alpha), float(beta), int(acc), int(relu), bias is not None,
                mask is not None, res is not None, int(ldmask), int(ldres),
                tuple(mod16(p) for p in (A, B, C, bias, mask, res)))


# ------------------------------------------------------------------------------------------------ buffers
def layouts(s):
    """name -> (logical shape [batch, rows, cols], element strides, element offset) of every operand the call
    addresses: A as [batch, M, K], B as [batch, K, N], C / mask / residual as [batch, M, N], bias as [1, 1, N]"""
    sa, sb, sc = (s.sa, s.sb, s.sc) if s.batch > 1 else (0, 0, 0)
    b_nk = s.tb if not s.tf32 else 1 - s.tb              # B(k, n) at B[n*ldb + k]
    assert all(a % 4 == 0 for a in s.align), s
    off = dict(zip(OPERANDS, (a // 4 for a in s.align)))
    lay = {"A": ((s.batch, s.M, s.K), (sa, 1, s.lda) if s.ta else (sa, s.lda, 1), off["A"]),
           "B": ((s.batch, s.K, s.N), (sb, 1, s.ldb) if b_nk else (sb, s.ldb, 1), off["B"]),
           "C": ((s.batch, s.M, s.N), (sc, s.ldc, 1), off["C"])}
    if s.bias:
        lay["bias"] = ((1, 1, s.N), (0, 0, 1), off["bias"])
    if s.mask:
        lay["mask"] = ((s.batch, s.M, s.N), (sc, s.ldmask, 1), off["mask"])
    if s.residual:
        lay["residual"] = ((s.batch, s.M, s.N), (sc, s.ldres, 1), off["residual"])
    return lay


def extent(shape, strides, offset):
    return offset + sum((n - 1) * st for n, st in zip(shape, strides)) + 1


def int_range(K):
    """largest r <= 16 with K r^2 <= 2^22: every partial sum of a product of values in [-r, r] is an integer < 2^22"""
    return max(1, min(16, math.isqrt(2 ** 22 // max(K, 1))))


def _crafted(shape, g, device):
    """normal magnitudes whose low 16 bits read 0x4CCC: rounding to 10 mantissa bits drops 0.4 ulp, to 7 bits 0.3 ulp
    (both toward zero, under round-to-nearest as under truncation)"""
    x = torch.randn(shape, generator=g, device=device).abs().clamp_min(2.0 ** -60)
    return ((x.view(torch.int32) & ~0xFFFF) | 0x4CCC).view(torch.float32)


def operand_values(s, mode, g, device):
    """logical values of every input operand and of the initial C window"""
    lay = layouts(s)
    v = {}
    if mode == "exact":
        r = int_range(s.K)
        ints = lambda shape, hi: torch.randint(-hi, hi + 1, shape, generator=g, device=device).float()  # noqa: E731
        v["A"], v["B"] = ints(lay["A"][0], r), ints(lay["B"][0], r)
        for n in ("bias", "residual"):
            if n in lay:
                v[n] = ints(lay[n][0], 16)
        c0 = ints(lay["C"][0], 16)
    else:
        sign = torch.randint(0, 2, (s.batch, s.K), generator=g, device=device).float() * 2 - 1
        v["A"] = _crafted(lay["A"][0], g, device) * sign[:, None, :]
        v["B"] = _crafted(lay["B"][0], g, device) * sign[:, :, None]
        for n in ("bias", "residual"):
            if n in lay:
                v[n] = torch.randn(lay[n][0], generator=g, device=device)
        c0 = torch.randn(lay["C"][0], generator=g, device=device)
    if "mask" in lay:
        v["mask"] = torch.randint(-1, 2, lay["mask"][0], generator=g, device=device).float()
    if s.splitk > 1:
        c0.zero_()              # split-K adds partial sums into a pre-zeroed window, as training.py zeroes it
    elif not s.reads_c:
        c0.fill_(float("nan"))  # never read: an element the kernel does not write stays NaN
    v["C"] = c0
    return v


def build_buffers(s, vals):
    """flat allocation of exactly the extent each operand addresses, NaN (inputs) or SENTINEL (output) outside the
    logical operand -> (flat buffers, logical views into them)"""
    flat, views = {}, {}
    for n, (shape, strides, off) in layouts(s).items():
        fill = SENTINEL if n == "C" else float("nan")
        flat[n] = torch.full((extent(shape, strides, off),), fill, device=vals[n].device)
        views[n] = flat[n].as_strided(shape, strides, off)
        views[n].copy_(vals[n])
    return flat, views


def reference(s, vals):
    """float64 result and the magnitude sums the precision bounds scale with: (|alpha| |A||B|, S)"""
    A, B = vals["A"].double(), vals["B"].double()
    mag = abs(s.alpha) * torch.matmul(A.abs(), B.abs())
    out = s.alpha * torch.matmul(A, B)
    total = mag.clone()
    c0 = vals["C"].double()
    if s.splitk > 1:
        return out + c0, mag, total + c0.abs()
    if s.bias:
        out += vals["bias"].double()
        total += vals["bias"].double().abs()
    if s.beta_eff != 0.0:
        out += s.beta_eff * c0
        total += abs(s.beta_eff) * c0.abs()
    if s.relu:
        out.clamp_(min=0.0)
    if s.mask:
        out = torch.where(vals["mask"] > 0, out, torch.zeros((), dtype=out.dtype, device=out.device))
    if s.residual:
        out += vals["residual"].double()
        total += vals["residual"].double().abs()
    return out, mag, total


def check(s, flat, views, ref, mag, total, mode):
    """-> {check name: failure message or None} for "sentinel", "nan" and the pass (``mode``), and "ratio": the
    largest |C - ref| / bound of the precision pass"""
    shape, strides, off = layouts(s)["C"]
    win = torch.zeros(flat["C"].numel(), dtype=torch.bool, device=flat["C"].device)
    win.as_strided(shape, strides, off).fill_(True)
    res = {}
    changed = torch.nonzero(~win & (flat["C"] != SENTINEL)).flatten()
    res["sentinel"] = (f"{changed.numel()} element(s) outside the M x N window changed, first at flat index "
                       f"{changed[0].item()}") if changed.numel() else None
    C = views["C"]
    bad = torch.nonzero(~torch.isfinite(C))
    res["nan"] = f"{bad.shape[0]} non-finite output(s), first at {tuple(bad[0].tolist())}" if bad.shape[0] else None
    if mode == "exact":
        wrong = torch.nonzero(~(C.double() == ref))
        res["exact"] = None
        if wrong.shape[0]:
            i = tuple(wrong[0].tolist())
            res["exact"] = (f"{wrong.shape[0]} output(s) differ from the exact result, first at {i}: "
                            f"{C[i].item()} != {ref[i].item()}")
    else:
        bound = s.chain * 2.0 ** -24 * total + (2.0 ** -10 * mag if s.tf32 else 0.0)
        ratio = ((C.double() - ref).abs() / bound).nan_to_num(nan=math.inf).max().item()
        res["ratio"] = ratio
        res["precision"] = None if ratio <= 1.0 else f"error reaches {ratio:.3g} x the bound"
    return res


def replay(s, run, mode, device, seed=0):
    """build the buffers of ``s``, run ``run(s, views, flat)`` on them and check the result"""
    g = torch.Generator(device=device).manual_seed(seed)
    vals = operand_values(s, mode, g, device)
    ref, mag, total = reference(s, vals)
    flat, views = build_buffers(s, vals)
    run(s, views, flat)
    if str(device).startswith("cuda"):
        torch.cuda.synchronize()
    return check(s, flat, views, ref, mag, total, mode)


def launch(s, views, flat):
    """the call itself, through the C ABI"""
    from puzzlenet_b200 import _lib
    p = lambda n: views[n].data_ptr() if n in views else None  # noqa: E731
    st = torch.cuda.current_stream().cuda_stream
    if s.entry == "pz_sgemm":
        _lib.call(s.entry, s.ta, s.tb, s.M, s.N, s.K, s.alpha, p("A"), s.lda, p("B"), s.ldb, s.beta, p("C"), s.ldc,
                  s.batch, s.sa, s.sb, s.sc, s.splitk, p("bias"), s.relu, p("mask"), s.ldmask, p("residual"), s.ldres,
                  st)
    elif s.entry == "pz_gemm_tf32":
        _lib.call(s.entry, s.ta, s.tb, s.M, s.N, s.K, p("A"), s.lda, p("B"), s.ldb, p("C"), s.ldc, s.splitk,
                  p("bias"), s.relu, p("mask"), s.ldmask, s.accumulate, st)
    else:
        _lib.call(s.entry, s.ta, s.tb, s.M, s.N, s.K, p("A"), s.lda, p("B"), s.ldb, p("C"), s.ldc, s.batch, s.sa,
                  s.sb, s.sc, s.splitk, p("bias"), s.relu, p("mask"), s.ldmask, s.accumulate, st)


# ------------------------------------------------------------------------------------------------ coverage
def _tf32_mode(s, a_mn, b_mn):
    return s.tf32 and (s.ta, s.tb) == (a_mn, b_mn)


# kernel configurations the training step must keep exercising; a family that disappears from training.py is removed
# from this list on purpose
FAMILIES = {
    "tf32 forward, K-major operands, lda != K":
        lambda s: s.entry == "pz_gemm_tf32" and _tf32_mode(s, 0, 0) and s.lda != s.K,
    "tf32 dgrad with a ReLU mask": lambda s: _tf32_mode(s, 0, 1) and s.batch == 1 and s.mask,
    "tf32 dgrad with accumulate": lambda s: _tf32_mode(s, 0, 1) and s.batch == 1 and s.accumulate,
    "tf32 wgrad with split-K": lambda s: _tf32_mode(s, 1, 1) and s.splitk > 1,
    "tf32 weights-resident shape":
        lambda s: s.entry == "pz_gemm_tf32" and s.splitk == 1 and s.N == 128 and s.M // 128 >= 4 * 148 and s.K <= 256,
    "tf32 64-wide tiles (N % 128 != 0)": lambda s: s.tf32 and s.N % 128 != 0,
    "batched tf32 (0, 0): S = q k^T, dA = dvals v^T": lambda s: s.batch > 1 and _tf32_mode(s, 0, 0),
    "batched tf32 (0, 1): vals = A v, dq = dS k": lambda s: s.batch > 1 and _tf32_mode(s, 0, 1),
    "batched tf32 (1, 1): dv = A^T dvals, dk = dS^T q": lambda s: s.batch > 1 and _tf32_mode(s, 1, 1),
    "sgemm transA with split-K": lambda s: not s.tf32 and s.ta and s.splitk > 1,
    "sgemm batched with alpha = -1": lambda s: not s.tf32 and s.batch > 1 and s.alpha == -1.0,
    "sgemm beta = 1 (accumulating data gradient)": lambda s: not s.tf32 and not s.ta and s.beta == 1.0 and s.K >= 64,
    "sgemm ReLU-mask epilogue": lambda s: not s.tf32 and s.mask,
    "skinny split-K (M <= 128)": lambda s: not s.tf32 and not s.ta and s.M <= 128 and s.splitk > 1,
}


class _Recorder:
    """stands in for ``training._lib``: records the GEMM calls, forwards every call unchanged"""

    def __init__(self, lib):
        self._lib = lib
        self.sites = {}

    def call(self, name, *args):
        if name in ENTRIES:
            self.sites.setdefault(site_of_call(name, args), None)
        return self._lib.call(name, *args)

    def __getattr__(self, name):
        return getattr(self._lib, name)


@pytest.fixture(scope="module")
def captured():
    """(precision, pairs) -> the distinct GEMM configurations of one forward_backward + one
    forward_backward_pretrain, in first-call order"""
    from oracle import puzzle_oracle as po
    from puzzlenet_b200 import _lib, training
    from puzzlenet_b200.model5_b import TouchedRegraster
    from puzzlenet_b200.weights import synthetic_state_dict
    from tests.golden_inputs import FPS_SEED, training_inputs
    out = {}
    sd = synthetic_state_dict(0)
    for prec in ("fp32", "tf32"):
        for B in (8, 64):
            model = TouchedRegraster(types.SimpleNamespace(dataset="vase", loss_mode=1, loss_sum=False, lr=0.9e-3))
            model.load_state_dict(sd, strict=True)
            model.to("cuda:0")
            torch.manual_seed(FPS_SEED)
            starts = torch.stack([torch.randint(0, 1024, (B,)), torch.randint(0, 512, (B,)),
                                  torch.randint(0, 1024, (B,)), torch.randint(0, 512, (B,))])
            batch = [t.to("cuda:0") for t in training_inputs(B, po.se3_exp)]
            rec = _Recorder(_lib)
            with pytest.MonkeyPatch.context() as mp:
                mp.setattr(training, "_lib", rec)
                tr = training.Trainer(model, precision=prec)
                tr.forward_backward(batch, starts=starts)
                tr.forward_backward_pretrain(batch, starts=starts)
                torch.cuda.synchronize()
            out[(prec, B)] = list(rec.sites)
            del tr, model
            torch.cuda.empty_cache()
    for (prec, B), sites in out.items():
        print(f"captured {prec} B={B}: {len(sites)} distinct GEMM configurations")
    return out


def _union(captured):
    return list(dict.fromkeys(s for sites in captured.values() for s in sites))


@pytest.mark.gpu
def test_captured_sites_cover_every_gemm_family(captured):
    sites = _union(captured)
    assert all(len(v) > 0 for v in captured.values())
    missing = [name for name, fam in FAMILIES.items() if not any(fam(s) for s in sites)]
    assert not missing, f"the training step no longer issues: {missing}"
    # the TF32 step runs its large layers on the tensor cores at both batch sizes
    for B in (8, 64):
        assert sum(s.tf32 for s in captured[("tf32", B)]) >= 10
        assert not any(s.tf32 for s in captured[("fp32", B)])


@pytest.mark.gpu
def test_sgemm_bound_is_below_what_tf32_operands_would_lose(captured):
    """the fp32 precision bound n 2^-24 stays below the least relative loss of a product whose operands lost the
    TF32-dropped bits, so a pz_sgemm call that ran at TF32 precision fails the precision pass"""
    worst = max((s for s in _union(captured) if not s.tf32), key=lambda s: s.chain)
    ratio = worst.chain * 2.0 ** -24 / TF32_LOSS_FLOOR
    print(f"largest sgemm bound / TF32 loss floor: {ratio:.3f} ({worst})")
    assert ratio < 1.0, worst


def _replay_all(captured, mode):
    sites = _union(captured)
    fails, worst = [], {}
    t0 = time.perf_counter()
    for i, s in enumerate(sites):
        r = replay(s, launch, mode, "cuda:0", seed=i)
        msgs = [f"{k}: {r[k]}" for k in ("sentinel", "nan", mode) if r[k]]
        if msgs:
            fails.append((s, msgs))
        if mode == "precision":
            names = [n for n, fam in FAMILIES.items() if fam(s)] or ["(other) " + ("tf32" if s.tf32 else "sgemm")]
            for n in names:
                worst[n] = max(worst.get(n, 0.0), r["ratio"])
    print(f"{mode} pass: {len(sites)} configurations replayed in {time.perf_counter() - t0:.1f} s")
    for n, v in worst.items():
        print(f"  precision {n}: largest error / bound = {v:.3f}")
    assert not fails, "\n".join(f"{s}\n    " + "\n    ".join(m) for s, m in fails)


@pytest.mark.gpu
def test_every_gemm_site_exact_with_integer_operands(captured):
    _replay_all(captured, "exact")


@pytest.mark.gpu
def test_every_gemm_site_within_rounding_bound(captured):
    _replay_all(captured, "precision")


# ------------------------------------------------------------------------------------------------ the checker on CPU
def _tf32_round(x):
    """round-to-nearest-even to a 10-bit mantissa"""
    i = x.contiguous().view(torch.int32)
    return ((i + 0x0FFF + ((i >> 13) & 1)) & ~0x1FFF).view(torch.float32)


def emulate(fault=None):
    """a torch-CPU stand-in for the kernels, optionally with one injected fault: fp32 products (operands rounded to
    TF32 first for the tensor-core entry points), split-K partials added in order, then the epilogue in the
    documented order (+ bias, + beta C, ReLU, mask, + residual)"""

    def run(s, views, flat):
        A, B = views["A"].clone(), views["B"].clone()
        rnd = _tf32_round if s.tf32 or fault == "tf32_operands" else (lambda x: x)
        if fault == "bf16_operands":
            rnd = lambda x: x.bfloat16().float()  # noqa: E731
        A, B = rnd(A), rnd(B)
        if fault == "drop_kblock":
            A[:, :, 32:64] = 0
        if fault == "lda_gap_read":          # row 0 read one element past its K columns
            A[0, 0, 0] += flat["A"][layouts(s)["A"][2] + s.K]
        kc = -(-s.K // s.splitk)
        acc = torch.zeros(s.batch, s.M, s.N)
        for k0 in range(0, s.K, kc):
            acc += s.alpha * torch.matmul(A[:, :, k0:k0 + kc], B[:, k0:k0 + kc, :])
        if fault == "shift_tile":            # the first 128 x 64 tile reads its columns one to the right
            acc[:, :128, :64] = acc[:, :128, 1:65].clone()
        C = views["C"]
        if s.splitk > 1:
            C += acc
            return
        keep = views["mask"] > 0 if s.mask else None
        if fault == "mask_before_relu":      # gate the raw product, ahead of everything that precedes the ReLU
            acc = torch.where(keep, acc, torch.zeros(()))
        if s.bias:
            acc += views["bias"]
        if s.beta_eff != 0.0:
            acc += s.beta_eff * C
        if s.relu:
            acc.clamp_(min=0.0)
        if s.mask and fault != "mask_before_relu":
            acc = torch.where(keep, acc, torch.zeros(()))
        if s.residual:
            acc += views["residual"]
        C.copy_(acc)
        if fault == "ldc_gap_write":         # one store past the N columns of row 1
            flat["C"][layouts(s)["C"][2] + s.ldc + s.N] = 1.0

    return run


HAND_SITES = {
    # K-major forward, strided A / B / C, 64-wide column remainder, bias + ReLU
    "tf32_fwd": Site("pz_gemm_tf32", 0, 0, 256, 192, 96, lda=100, ldb=104, ldc=200, bias=True, relu=1),
    # data gradient: B MN-major, mask with its own stride, accumulate into C
    "tf32_dgrad": Site("pz_gemm_tf32", 0, 1, 256, 128, 64, lda=68, ldb=132, ldc=136, mask=True, ldmask=140,
                       accumulate=1),
    # weight gradient: both MN-major, split-K
    "tf32_wgrad": Site("pz_gemm_tf32", 1, 1, 128, 64, 1024, lda=132, ldb=68, ldc=64, splitk=3),
    # batched with gaps between the batches
    "tf32_batched": Site("pz_gemm_tf32_batched", 0, 1, 128, 64, 64, lda=64, ldb=68, ldc=72, batch=3,
                         sa=128 * 64 + 32, sb=64 * 68 + 16, sc=128 * 72 + 8),
    "sgemm_ta_splitk": Site("pz_sgemm", 1, 0, 70, 40, 300, lda=72, ldb=44, ldc=41, splitk=5, alpha=0.5,
                            align=(4, 8, 12, 0, 0, 0)),
    "sgemm_batched_neg": Site("pz_sgemm", 1, 1, 60, 50, 70, lda=61, ldb=73, ldc=53, batch=2, sa=70 * 61 + 5,
                              sb=50 * 73 + 3, sc=60 * 53 + 7, alpha=-1.0, align=(12, 4, 8, 0, 0, 0)),
    "sgemm_epilogue": Site("pz_sgemm", 0, 1, 90, 70, 40, lda=41, ldb=43, ldc=72, beta=1.0, relu=1, bias=True,
                           mask=True, ldmask=75, residual=True, ldres=71, align=(0, 4, 8, 12, 4, 8)),
    # long reductions, where random-walk cancellation would hide lost bits from plain normal operands
    "sgemm_long_k": Site("pz_sgemm", 1, 0, 32, 32, 131072, lda=32, ldb=32, ldc=32, splitk=148),
    "tf32_long_k": Site("pz_gemm_tf32", 1, 1, 128, 64, 32768, lda=128, ldb=64, ldc=64, splitk=8),
}


@pytest.mark.parametrize("mode", ["exact", "precision"])
@pytest.mark.parametrize("name", list(HAND_SITES))
def test_checker_accepts_a_correct_emulation(name, mode):
    r = replay(HAND_SITES[name], emulate(), mode, "cpu")
    assert r["sentinel"] is None and r["nan"] is None and r[mode] is None, r


@pytest.mark.parametrize("fault,name,caught_by", [
    ("drop_kblock", "tf32_fwd", "exact"),
    ("drop_kblock", "sgemm_ta_splitk", "exact"),
    ("shift_tile", "tf32_fwd", "exact"),
    ("ldc_gap_write", "sgemm_epilogue", "sentinel"),
    ("ldc_gap_write", "tf32_batched", "sentinel"),
    ("lda_gap_read", "tf32_fwd", "nan"),
    ("lda_gap_read", "sgemm_epilogue", "nan"),
    ("mask_before_relu", "sgemm_epilogue", "exact"),
    ("mask_before_relu", "tf32_dgrad", "exact"),
    ("bf16_operands", "tf32_fwd", "precision"),
    ("bf16_operands", "tf32_long_k", "precision"),
    ("tf32_operands", "sgemm_epilogue", "precision"),
    ("tf32_operands", "sgemm_long_k", "precision"),
])
def test_checker_catches_injected_fault(fault, name, caught_by):
    mode = "precision" if caught_by == "precision" else "exact"
    r = replay(HAND_SITES[name], emulate(fault), mode, "cpu")
    assert r[caught_by] is not None, r


def test_site_of_call_reads_every_entry_point():
    """the recorder's argument unpacking matches the wrappers in training.py"""
    from puzzlenet_b200 import training

    class Fake:
        def __init__(self):
            self.calls = []

        def call(self, name, *args):
            self.calls.append(site_of_call(name, args))

        def stream_ptr(self):
            return 0

    class T:
        def __init__(self, ptr):
            self.ptr = ptr

        def data_ptr(self):
            return self.ptr

    fake = Fake()
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(training, "_lib", fake)
        training.gemm(T(4), T(8), T(12), 5, 6, 7, ta=True, lda=9, ldb=10, ldc=11, alpha=-1.0, beta=0.5, batch=2, sa=1,
                      sb=2, sc=3, bias=T(16), relu=True, mask=T(36), ldmask=13, residual=T(40), ldres=14)
        training._gemm_tf32(1, 0, 128, 64, 32, T(0), 36, T(16), 40, T(32), 44, splitk=3)
        training._gemm_tf32(0, 1, 128, 64, 32, T(0), 36, T(16), 40, T(32), 44, mask=T(48), ldmask=48,
                            accumulate=True)
        training.bgemm_tf32(0, 1, 256, 64, 256, T(0), 256, T(16), 64, T(32), 64, 4, 65536, 16384, 16384)
    assert fake.calls == [
        Site("pz_sgemm", 1, 0, 5, 6, 7, 9, 10, 11, 2, 1, 2, 3, 1, -1.0, 0.5, 0, 1, True, True, True, 13, 14,
             (4, 8, 12, 0, 4, 8)),
        Site("pz_gemm_tf32", 1, 0, 128, 64, 32, 36, 40, 44, splitk=3),
        Site("pz_gemm_tf32", 0, 1, 128, 64, 32, 36, 40, 44, mask=True, ldmask=48, accumulate=1),
        Site("pz_gemm_tf32_batched", 0, 1, 256, 64, 256, 256, 64, 64, batch=4, sa=65536, sb=16384, sc=16384),
    ]
