"""The tcgen05 contraction (csrc/gemm_tcgen05.cu) on every launch plan its dispatcher can choose, against exact and float64
references, plus the split-K entry and the fp32 verification kernel (csrc/gemm_simt.cu).

A launch plan (dmm_gemm_plan) is a tile cell -- BN in {64, 128, 256}, one CTA or a CTA pair, and the tail-wave split in
{1, 2, 4} -- with an epilogue kind (TMA, register single-pass, register split-bf16) and a shared-memory ring depth.  CASES
names the plan each case must get at 148 SMs; tests/test_gemm_plan_cpu.py checks, without a GPU, that the cases cover every
(cell, kind) pair and every TMA ring depth a sweep of shapes reaches, and that the plans written here are the query's.

Conventions (those of test_joint_kernels_gpu.py):
- Every caller-provided buffer is larger than its documented region (extra rows, a leading dimension beyond the width) and
  is filled with a sentinel first: NaN for the outputs and for the padding of every input, so a read of padding shows up
  as a NaN in the result.  After the call nothing outside [M, round_up(N, 4 fp32 / 8 bf16)] may have changed (the header
  lets the 16-byte store units overwrite the padding up to that boundary).
- Exact work is compared bit for bit.  The exact-arithmetic run uses small-integer bf16 operands (hi and independently
  chosen lo parts), integer bias / post bias / residual and power-of-two alpha and beta: every product and partial sum is
  an integer below 2^24, so the fp32 result does not depend on the summation order or on how the tensor pipe aligns its
  sums, and a dropped or repeated k block or pass, a wrong pass pairing, or a misplaced tile, tail slice, row, column,
  bias or residual element changes at least one integer.
- Everything else is compared against float64 computed on the device, within a bound derived in numeric_bound().
"""
import math
from typing import NamedTuple

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NUM_SMS = 148
U = 2.0 ** -24
TMA, REG, X3 = "tma", "reg", "x3"
KIND_CODE = {TMA: 0, REG: 1, X3: 2}                 # enum dmm_gemm_epilogue_kind


class Case(NamedTuple):
    M: int
    N: int
    K: int
    kind: str
    res: str      # "", "f32", "bf16"; "=out": the residual aliases the output of its type (in place)
    outs: str     # f: out_f32, h: out_hi, l: out_lo
    lo: str       # a: a_lo, b: b_lo, r: res_lo
    cmax: bool
    post: bool    # post stage (post_bias) on the bf16 output
    pre: bool     # res_pre_act
    plan: tuple   # expected (bn, ctas, split, stages, nbuf)

    @property
    def id(self):
        bn, ctas, split, stages, _ = self.plan
        return f"{self.kind}-bn{bn}x{ctas}-split{split}-st{stages}-M{self.M}-N{self.N}-K{self.K}"

    @property
    def flags(self):
        from diffmm_b200 import _lib as L
        f = 0
        f |= L.GEMM_A_LO if "a" in self.lo else 0
        f |= L.GEMM_B_LO if "b" in self.lo else 0
        f |= L.GEMM_RESIDUAL if self.res.startswith("f32") else 0
        f |= L.GEMM_RES_HI if self.res.startswith("bf16") else 0
        f |= L.GEMM_RES_LO if "r" in self.lo else 0
        f |= L.GEMM_OUT_F32 if "f" in self.outs else 0
        f |= L.GEMM_OUT_HI if "h" in self.outs else 0
        f |= L.GEMM_OUT_LO if "l" in self.outs else 0
        return f


# Nine tile cells x three epilogue kinds, plus the TMA ring depths 7 / 6 / 3 of further cases.  Edges on the way: M in {1,
# 127, 128, 129, 255, 256, 257} (257 on a pair tile: the second pair's peer CTA lies entirely past M), N ragged at 32, at
# sub_bn and at BN, tail slices that start at or beyond N (N = 12673, 25100, 500000, 21300, 18945), K in {1, 15, 16, 17, 63,
# 64, 65, 1024, 4100}, and in-place residuals in every epilogue.  Production shapes: (640, 7050, 1024) is baby's output
# layer with cmax, (4700, 1024, 1024) the hidden-space step (in-place fp32 state, bf16 output, 2 ring stages), (1, 18945)
# scoring against a catalog, (2000, 7050) the bf16x3 rebuild's in-place call.
CASES = [
    # (64, 1, 1)
    Case(257, 200, 65, TMA, "f32=out", "fh", "", True, True, False, (64, 1, 1, 5, 2)),
    Case(1, 33, 1, TMA, "", "h", "", False, True, False, (64, 1, 1, 7, 1)),
    Case(127, 64, 17, TMA, "f32", "f", "", True, False, True, (64, 1, 1, 6, 2)),
    Case(128, 96, 16, REG, "bf16=out", "h", "", True, True, False, (64, 1, 1, 8, 1)),
    Case(255, 100, 15, X3, "f32=out", "fhl", "ab", True, True, False, (64, 1, 1, 8, 1)),
    # (128, 1, 1)
    Case(129, 4737, 63, TMA, "f32", "f", "", True, False, False, (128, 1, 1, 4, 2)),
    Case(1, 9473, 1024, TMA, "", "fh", "", True, False, False, (128, 1, 1, 5, 1)),
    Case(1, 9473, 64, REG, "bf16", "fh", "", True, True, False, (128, 1, 1, 6, 1)),
    Case(256, 4737, 63, X3, "", "fhl", "", True, False, False, (128, 1, 1, 6, 1)),
    # (128, 1, 2): the second 64-column slice of the last column block starts at N
    Case(257, 12673, 17, TMA, "", "h", "", False, True, False, (128, 1, 2, 5, 1)),
    Case(257, 12673, 64, REG, "bf16=out", "h", "", True, False, False, (128, 1, 2, 6, 1)),
    Case(257, 12673, 65, X3, "bf16", "f", "ar", True, False, True, (128, 1, 2, 6, 1)),
    # (256, 1, 1)
    Case(4700, 1024, 1024, TMA, "f32=out", "fh", "", False, True, False, (256, 1, 1, 2, 2)),
    Case(1, 18945, 64, TMA, "", "f", "", True, False, False, (256, 1, 1, 3, 1)),
    Case(257, 9473, 15, REG, "bf16", "f", "", True, False, False, (256, 1, 1, 4, 1)),
    Case(640, 7050, 1024, X3, "", "fhl", "ab", True, False, False, (256, 1, 1, 4, 1)),
    # (256, 1, 2)
    Case(513, 25100, 16, TMA, "f32", "f", "", True, False, False, (256, 1, 2, 3, 2)),
    Case(513, 25100, 17, REG, "bf16=out", "h", "", False, True, False, (256, 1, 2, 4, 1)),
    Case(513, 25100, 1, X3, "", "fhl", "b", True, False, False, (256, 1, 2, 4, 1)),
    # (256, 1, 4): N % 256 = 32, three of the four 64-column slices of the last block start beyond N
    Case(127, 500000, 16, TMA, "", "f", "", True, False, False, (256, 1, 4, 3, 1)),
    Case(1, 500000, 64, REG, "bf16=out", "fh", "", True, False, False, (256, 1, 4, 4, 1)),
    Case(1, 500000, 63, X3, "f32=out", "fhl", "ab", True, False, False, (256, 1, 4, 4, 1)),
    # (256, 2, 1)
    Case(257, 6273, 64, TMA, "f32=out", "fh", "", True, True, False, (256, 2, 1, 4, 2)),
    Case(129, 9473, 65, REG, "bf16", "fh", "", True, False, False, (256, 2, 1, 6, 1)),
    Case(257, 6273, 4100, X3, "bf16=out", "hl", "abr", False, True, False, (256, 2, 1, 6, 1)),
    # (256, 2, 2)
    Case(385, 21300, 15, TMA, "", "f", "", True, False, False, (256, 2, 2, 5, 1)),
    Case(385, 21300, 16, REG, "bf16", "h", "", False, True, False, (256, 2, 2, 6, 1)),
    Case(385, 21300, 64, X3, "f32=out", "f", "ab", True, False, False, (256, 2, 2, 6, 1)),
    # (256, 2, 4)
    Case(385, 18945, 17, TMA, "f32", "h", "", False, True, False, (256, 2, 4, 4, 2)),
    Case(385, 18945, 63, REG, "bf16=out", "h", "", True, False, False, (256, 2, 4, 6, 1)),
    Case(2000, 7050, 1024, X3, "f32=out", "f", "ab", True, False, False, (256, 2, 4, 6, 1)),
]

# split-K entry: (M, N, K, expected ksplit); the plan sweep of test_gemm_plan_cpu.py must reach no other factor
SPLITK_CASES = [(1, 100, 4096, 1), (1, 129, 1024, 2), (1, 129, 1536, 3), (1024, 1024, 7050, 4), (1, 129, 2560, 5),
                (1, 129, 3072, 6), (1, 129, 3584, 7), (257, 130, 4096, 8)]


def plan_of(M, N, K, flags):
    import ctypes as C
    from diffmm_b200 import _lib as L
    pl = L.GemmLaunchPlan()
    rc = L.load().dmm_gemm_plan(NUM_SMS, M, N, K, flags, C.byref(pl))
    return rc, pl


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


@pytest.fixture(scope="module", autouse=True)
def b200(ops):
    from diffmm_b200 import _lib
    t = torch.zeros(1, device=DEV)
    n = _lib.load().dmm_num_sms(ops._ctx(t))
    assert n == NUM_SMS, f"the case table is written for {NUM_SMS} SMs, the device has {n}"


def pad(n, m):
    return (n + m - 1) // m * m


def i32(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(i32(a), i32(b))


def buf32(rows, cols):
    """fp32 sentinel buffer of 3 extra rows and a leading dimension 12 beyond round_up(cols, 4) (a multiple of 4)."""
    return torch.full((rows + 3, pad(cols, 4) + 12), float("nan"), device=DEV)


def buf16(rows, cols):
    """bf16 sentinel buffer: 3 extra rows, leading dimension 16 beyond round_up(cols, 8)."""
    return torch.full((rows + 3, pad(cols, 8) + 16), float("nan"), dtype=torch.bfloat16, device=DEV)


def assert_outside_untouched(buf, before, rows, cols):
    """Nothing of buf outside [rows, :round_up(cols, 16 bytes)] differs from `before`."""
    w = pad(cols, 4 if buf.dtype == torch.float32 else 8)
    a, b = i32(buf).clone(), i32(before)
    a[:rows, :w] = b[:rows, :w]
    assert torch.equal(a, b), "the kernel wrote outside the region the header allows"


def place(buf, vals):
    buf[:vals.shape[0], :vals.shape[1]] = vals
    return buf[:vals.shape[0], :vals.shape[1]]


def vec32(vals):
    b = torch.full((pad(vals.numel(), 4) + 12,), float("nan"), device=DEV)
    b[:vals.numel()] = vals
    return b[:vals.numel()]


def chunk_max(v):
    """cmax of fp32 [M, N]: NaN-propagating maxima of the 32-column chunks."""
    M, N = v.shape
    w = torch.full((M, pad(N, 32)), float("-inf"), device=DEV)
    w[:, :N] = v
    w = w.view(M, -1, 32)
    m = w.amax(dim=2)
    return torch.where(torch.isnan(w).any(dim=2), torch.full_like(m, float("nan")), m)


def split_ref(v):
    hi = v.to(torch.bfloat16)
    return hi, (v - hi.float()).to(torch.bfloat16)


def operands(c, gen, exact):
    """bf16 hi (and lo) views of A [M, K] and B [N, K] in buffers with lda = ldb = round_up(K, 8) + 8 and NaN padding."""
    def one(rows):
        if exact:
            hi = torch.randint(-4, 5, (rows, c.K), generator=gen, device=DEV).float()
            lo = torch.randint(-4, 5, (rows, c.K), generator=gen, device=DEV).float()
        else:
            x = torch.randn((rows, c.K), generator=gen, device=DEV)
            if rows == c.N:
                x = x / math.sqrt(c.K)
            hi = x.to(torch.bfloat16).float()
            lo = x - hi
        return (place(buf16(rows, c.K + 8), hi.to(torch.bfloat16)), place(buf16(rows, c.K + 8), lo.to(torch.bfloat16)))
    return one(c.M), one(c.N)


class Run(NamedTuple):
    out_f32: torch.Tensor
    out_hi: torch.Tensor
    out_lo: torch.Tensor
    cmax: torch.Tensor
    bufs: list          # (buffer, value before the call, rows, cols) of every output buffer


def make_inputs(c, exact, seed):
    gen = torch.Generator(device=DEV)
    gen.manual_seed(seed)
    (a_hi, a_lo), (b_hi, b_lo) = operands(c, gen, exact)
    if exact:
        bias = torch.randint(-8, 9, (c.N,), generator=gen, device=DEV).float()
        pbias = torch.randint(-8, 9, (c.N,), generator=gen, device=DEV).float()
        res = torch.randint(-16, 17, (c.M, c.N), generator=gen, device=DEV).float()
        res_lo = torch.randint(-16, 17, (c.M, c.N), generator=gen, device=DEV).float()
        alpha, beta = [(2.0, 0.5), (0.5, -2.0), (1.0, 1.0), (-1.0, 0.25)][seed % 4]
    else:
        bias = torch.randn((c.N,), generator=gen, device=DEV) * 0.1
        pbias = torch.randn((c.N,), generator=gen, device=DEV) * 0.3
        r = torch.randn((c.M, c.N), generator=gen, device=DEV)
        res, res_lo = (r, None) if c.res.startswith("f32") else split_ref(r)
        res, res_lo = (res.float(), None if res_lo is None else res_lo.float())
        alpha, beta = 0.75, 0.5
    return dict(a_hi=a_hi, a_lo=a_lo, b_hi=b_hi, b_lo=b_lo, bias=bias, pbias=pbias, res=res, res_lo=res_lo, alpha=alpha,
                beta=beta)


def run_case(ops, c, inp, act, post_act):
    """One dmm_gemm_bf16_tn call of case c on sentinel buffers; in-place residuals are written into the output buffers."""
    M, N = c.M, c.N
    out_f32 = buf32(M, N)[:M, :N] if "f" in c.outs else None
    out_hi = buf16(M, N)[:M, :N] if "h" in c.outs else None
    out_lo = buf16(M, N)[:M, :N] if "l" in c.outs else None
    residual = res_hi = res_lo = None
    if c.res.startswith("f32"):
        residual = out_f32 if c.res.endswith("=out") else place(buf32(M, N), inp["res"])
        residual.copy_(inp["res"])
    elif c.res.startswith("bf16"):
        hi = inp["res"].to(torch.bfloat16)
        lo = (inp["res_lo"] if inp["res_lo"] is not None else inp["res"] * 0).to(torch.bfloat16)
        res_hi = out_hi if c.res.endswith("=out") else buf16(M, N)[:M, :N]
        res_hi.copy_(hi)
        if "r" in c.lo:
            res_lo = out_lo if c.res.endswith("=out") else buf16(M, N)[:M, :N]
            res_lo.copy_(lo)
    cmax = buf32(M, (N + 31) // 32)[:M, :(N + 31) // 32] if c.cmax else None
    before = [(t._base, t._base.clone(), t.shape[0], t.shape[1]) for t in (out_f32, out_hi, out_lo, cmax) if t is not None]
    ops.gemm_bf16_tn(inp["a_hi"], inp["a_lo"] if "a" in c.lo else None, inp["b_hi"], inp["b_lo"] if "b" in c.lo else None,
                     M, N, c.K, bias=vec32(inp["bias"]), act=act, alpha=inp["alpha"], beta=inp["beta"], residual=residual,
                     out_f32=out_f32, out_hi=out_hi, out_lo=out_lo, res_hi=res_hi, res_lo=res_lo, res_pre_act=c.pre,
                     post_bias=vec32(inp["pbias"]) if c.post else None, post_act=post_act, cmax=cmax)
    torch.cuda.synchronize()
    return Run(out_f32, out_hi, out_lo, cmax, before)


def reference_terms(c, inp):
    """float64 [M, N]: the contraction sum_pass A_pass . B_pass^T (no lo.lo term) and its magnitude product."""
    ah, bh = inp["a_hi"].double(), inp["b_hi"].double()
    al, bl = inp["a_lo"].double(), inp["b_lo"].double()
    acc, mag = ah @ bh.T, ah.abs() @ bh.abs().T
    if "a" in c.lo:
        acc, mag = acc + al @ bh.T, mag + al.abs() @ bh.abs().T
    if "b" in c.lo:
        acc, mag = acc + ah @ bl.T, mag + ah.abs() @ bl.abs().T
    return acc, mag


def residual_of(c, inp):
    if c.res.startswith("f32"):
        return inp["res"].double()
    if c.res.startswith("bf16"):
        r = inp["res"].to(torch.bfloat16).double()
        if "r" in c.lo:
            r = r + inp["res_lo"].to(torch.bfloat16).double()
        return r
    return None


def epilogue_ref(c, inp, acc, act):
    """The epilogue's value v (float64), in the kernel's order of operations."""
    R = residual_of(c, inp)
    t = acc + inp["bias"].double()
    if R is not None and c.pre:
        t = t + inp["beta"] * R
    if act:
        t = torch.tanh(t)
    if R is not None and not c.pre:
        return inp["alpha"] * t + inp["beta"] * R
    return inp["alpha"] * t


def check_outputs_in_place(run):
    for buf, before, rows, cols in run.bufs:
        assert_outside_untouched(buf, before, rows, cols)


@pytest.mark.parametrize("c", CASES, ids=[c.id for c in CASES])
def test_plan_of_each_case(c):
    rc, pl = plan_of(c.M, c.N, c.K, c.flags)
    assert rc == 0
    assert (pl.bn, pl.ctas, pl.split, pl.stages, pl.nbuf, pl.epilogue, pl.ksplit) == c.plan + (KIND_CODE[c.kind], 1)


@pytest.mark.parametrize("c", CASES, ids=[c.id for c in CASES])
def test_exact_arithmetic(ops, c):
    inp = make_inputs(c, True, seed=CASES.index(c))
    run = run_case(ops, c, inp, act=0, post_act=0)
    acc, _ = reference_terms(c, inp)
    v64 = epilogue_ref(c, inp, acc, act=0)
    assert v64.abs().max() < 2 ** 23
    v = v64.float()
    assert torch.equal(v.double(), v64)                     # the reference itself is exact in fp32
    if run.out_f32 is not None:
        assert same_bits(run.out_f32, v)
    if run.cmax is not None:
        assert same_bits(run.cmax, chunk_max(v))
    if run.out_hi is not None:
        w = v + vec32(inp["pbias"]) if c.post else v          # the post stage without activation: exact too
        hi, lo = split_ref(w)
        assert same_bits(run.out_hi, hi)
        if run.out_lo is not None:
            assert same_bits(run.out_lo, lo)
    check_outputs_in_place(run)
    # a second call on the same inputs gives the same bits
    again = run_case(ops, c, inp, act=0, post_act=0)
    for x, y in zip(run[:4], again[:4]):
        assert x is None or same_bits(x, y)


# Numerical bound.  NVIDIA does not document how the tensor pipe accumulates inside one tcgen05.mma, so this is the model
# assumed: the products of bf16 (or bf16 hi / lo) values are exact, and each MMA instruction (UMMA_K = 16 products of one
# pass) adds them to the fp32 accumulator with an error of at most 2^-22 (two units of 2^-24, room for truncating instead
# of rounding alignment) times the magnitudes involved, which never exceed the magnitude product S = sum_pass |A| |B|^T.
# Over n = passes * ceil(K / 16) instructions: |acc - exact| <= n 2^-22 S.  The epilogue then adds one fp32 rounding per
# operation (u |value|), fast_tanh its own error E_FAST, tanh.approx.f32 (the single-pass post stage) the absolute error
# bound the PTX ISA states for it, 2^-10.987, and bf16 rounding 2^-8 of the value (hi alone) or 2^-16 (hi + lo).
# fast_tanh = 1 - 2 / (exp(2x) + 1) with __expf and __fdividef: exp's relative error (ex2.approx, ~2^-22, plus the rounding
# of 2x log2(e), < 2^-24 |2x log2 e|) is damped by the factor 2 exp(2x) / (exp(2x) + 1)^2 <= 1/2 and by 1/cosh^2 for large x,
# the division adds ~2 ulp of a value <= 2 and the subtraction one of 1: below 2^-20 in all; E_FAST = 2^-20.  The sum is
# first-order and doubled (SLACK) for the second-order terms.
E_FAST = 2.0 ** -20
E_APPROX = 2.0 ** -10.987
SLACK = 2.0


def numeric_bound(c, inp, acc, mag):
    """(v, e_v): the float64 epilogue value and the bound of |out_f32 - v|; and the same for the bf16 output."""
    R = residual_of(c, inp)
    n_pass = 1 + ("a" in c.lo) + ("b" in c.lo)
    e = n_pass * math.ceil(c.K / 16) * 2.0 ** -22 * mag
    t = acc + inp["bias"].double()
    e = e + U * t.abs()
    if R is not None and c.pre:
        t = t + inp["beta"] * R
        e = e + U * t.abs()
    t = torch.tanh(t)
    e = e + E_FAST
    if R is not None and not c.pre:
        v = inp["alpha"] * t + inp["beta"] * R
        e = abs(inp["alpha"]) * e + U * v.abs()
    else:
        v = inp["alpha"] * t
        e = abs(inp["alpha"]) * e
    w = v + (inp["pbias"].double() if c.post else 0.0)
    ew = e + U * w.abs()
    y = torch.tanh(w)
    ey = ew + (E_FAST if c.kind == X3 else E_APPROX)
    ey = ey + (2.0 ** -16 if "l" in c.outs else 2.0 ** -8) * (y.abs() + ey)
    return v, SLACK * e, y, SLACK * ey


def assert_within(got, want, bound, what):
    err = (got.double() - want).abs()
    ratio = (err / bound).max().item()
    assert not torch.isnan(err).any() and ratio <= 1.0, f"{what}: error / bound = {ratio:.3g}"


@pytest.mark.parametrize("c", CASES, ids=[c.id for c in CASES])
def test_numerical(ops, c):
    """Random normal operands, act = 1 and post_act = 1, against float64 of the same bf16 operand values."""
    inp = make_inputs(c, False, seed=1000 + CASES.index(c))
    run = run_case(ops, c, inp, act=1, post_act=1 if "h" in c.outs else 0)
    acc, mag = reference_terms(c, inp)
    v, ev, y, ey = numeric_bound(c, inp, acc, mag)
    if run.out_f32 is not None:
        assert_within(run.out_f32, v, ev, "out_f32")
        if run.cmax is not None:
            assert same_bits(run.cmax, chunk_max(run.out_f32))
    if run.out_hi is not None:
        got = run.out_hi.double() + (run.out_lo.double() if run.out_lo is not None else 0.0)
        assert_within(got, y, ey, "out_hi + out_lo" if run.out_lo is not None else "out_hi")
    check_outputs_in_place(run)


NAN_CASES = [c for c in CASES if c.cmax and "f" in c.outs]


@pytest.mark.parametrize("c", NAN_CASES, ids=[c.id for c in NAN_CASES])
def test_non_finite_row_stays_in_its_row(ops, c):
    """A NaN in one row of A and an inf in another change only those rows' outputs; the NaN row's cmax entries are all
    NaN, every other cmax entry is the maximum of the row's written chunk."""
    inp = make_inputs(c, True, seed=2000 + CASES.index(c))
    clean = run_case(ops, c, inp, act=0, post_act=0)
    rows = sorted({0, c.M - 1})
    inp["a_hi"][rows[0], c.K // 2] = float("nan")
    if len(rows) > 1:
        inp["a_hi"][rows[1], 0] = float("inf")
    bad = run_case(ops, c, inp, act=0, post_act=0)
    keep = torch.ones(c.M, dtype=torch.bool, device=DEV)
    keep[rows] = False
    for x, y in zip(clean[:4], bad[:4]):
        if x is not None:
            assert same_bits(x[keep], y[keep])
    assert torch.isnan(bad.out_f32[rows[0]]).all()
    assert torch.isnan(bad.cmax[rows[0]]).all()
    assert not torch.isfinite(bad.out_f32[rows]).any()
    # NaN where the written chunk holds one (whatever its payload), the chunk's maximum bit for bit elsewhere
    want = chunk_max(bad.out_f32)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(bad.cmax), nan) and same_bits(bad.cmax[~nan], want[~nan])
    check_outputs_in_place(bad)


def test_comparison_rejects_perturbed_outputs(ops):
    """The bit comparison of the exact runs catches one flipped last bit, two swapped columns and one shifted row."""
    c = CASES[0]
    inp = make_inputs(c, True, seed=3000)
    out = run_case(ops, c, inp, act=0, post_act=0).out_f32
    assert same_bits(out, out.clone())
    flip = out.clone()
    i32(flip)[5, 7] ^= 1
    assert not same_bits(out, flip)
    swap = out.clone()
    swap[:, [3, 4]] = swap[:, [4, 3]]
    assert not torch.equal(out[:, 3], out[:, 4]) and not same_bits(out, swap)
    shift = out.clone()
    shift[9] = torch.roll(shift[9], 1)
    assert not same_bits(out, shift)


@pytest.mark.parametrize("c", CASES, ids=[c.id for c in CASES])
def test_simt_kernel_matches_bit_for_bit(ops, c):
    """dmm_gemm_f32_tn on fp32 copies of the integer operands gives the tcgen05 result's bits."""
    inp = make_inputs(c, True, seed=CASES.index(c))
    tc = run_case(ops, c, inp, act=0, post_act=0)
    # [a_hi | a_lo] . [b_hi + b_lo | b_hi]^T over 2K columns: the three passes of the split-bf16 product, no lo.lo term
    a, b = inp["a_hi"].float(), inp["b_hi"].float() + (inp["b_lo"].float() if "b" in c.lo else 0.0)
    if "a" in c.lo:
        a, b = torch.cat([a, inp["a_lo"].float()], dim=1), torch.cat([b, inp["b_hi"].float()], dim=1)
    K = a.shape[1]
    a = place(buf32(c.M, K + 8), a)
    b = place(buf32(c.N, K + 8), b)
    R = residual_of(c, inp)
    M, N = c.M, c.N
    out = place(buf32(M, N), torch.zeros((M, N), device=DEV)) if "f" in c.outs else None
    hi = buf16(M, N)[:M, :N] if "h" in c.outs else None
    lo = buf16(M, N)[:M, :N] if "l" in c.outs else None
    ops.gemm_f32_tn(a, b, M, N, K, bias=vec32(inp["bias"]), alpha=inp["alpha"], beta=inp["beta"],
                    residual=None if R is None else place(buf32(M, N), R.float()), out_f32=out, out_hi=hi, out_lo=lo,
                    res_pre_act=c.pre, post_bias=vec32(inp["pbias"]) if c.post else None)
    torch.cuda.synchronize()
    for x, y in ((out, tc.out_f32), (hi, tc.out_hi), (lo, tc.out_lo)):
        if x is not None:
            assert same_bits(x, y)


def test_simt_kernel_rejects_cmax(ops):
    from diffmm_b200 import _lib
    import ctypes as C
    a = torch.zeros((64, 64), device=DEV)
    out = torch.full((64, 64), float("nan"), device=DEV)
    cmax = torch.full((64, 4), float("nan"), device=DEV)
    ep = ops._epilogue(None, 0, 1.0, 0.0, None, out, None, None, cmax=cmax)
    with pytest.raises(_lib.DiffMMError, match="cmax"):
        _lib.call("dmm_gemm_f32_tn", ops._ctx(a), ops._p(a), 64, ops._p(a), 64, 64, 64, 64, C.byref(ep), ops._stream())
    torch.cuda.synchronize()
    assert torch.isnan(out).all() and torch.isnan(cmax).all()


@pytest.mark.parametrize("M,N,K,ks", SPLITK_CASES, ids=[f"ksplit{k}-M{m}-N{n}-K{kk}" for m, n, kk, k in SPLITK_CASES])
def test_splitk_exact(ops, M, N, K, ks):
    """dmm_gemm_bf16_tn_splitk at every split factor: integer operands make the fixed-order sum of the slabs exact, so
    out_f32 and its bf16 copies (hi = bf16_rn(c), lo = bf16_rn(c - hi)) are compared bit for bit."""
    from diffmm_b200 import _lib as L
    rc, pl = plan_of(M, N, K, L.GEMM_SPLITK | L.GEMM_OUT_F32 | L.GEMM_OUT_HI | L.GEMM_OUT_LO)
    assert rc == 0 and pl.ksplit == ks
    c = Case(M, N, K, TMA, "", "f", "", False, False, False, None)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(ks)
    (a, _), (b, _) = operands(c, gen, True)
    want = (a.double() @ b.double().T).float()
    out = place(buf32(M, N), torch.zeros((M, N), device=DEV))
    hi, lo = buf16(M, N)[:M, :N], buf16(M, N)[:M, :N]
    before = [(t._base, t._base.clone()) for t in (out, hi, lo)]
    ops.gemm_bf16_tn_splitk(a, b, M, N, K, out_f32=out, out_hi=hi, out_lo=lo)
    torch.cuda.synchronize()
    assert same_bits(out, want)
    whi, wlo = split_ref(want)
    assert same_bits(hi, whi) and same_bits(lo, wlo)
    for buf, b0 in before:
        assert_outside_untouched(buf, b0, M, N)
    hi2 = buf16(M, N)[:M, :N]
    ops.gemm_bf16_tn_splitk(a, b, M, N, K, out_hi=hi2)
    torch.cuda.synchronize()
    assert same_bits(hi2, whi)


def test_every_argument_check_rejects_and_writes_nothing(ops):
    """One violation of each DMM_CHECK_ARG of run_gemm (all but the cuTensorMapEncodeTiled lookup, which a context always
    has, and the split-K one, which only the split-K entry can reach): the call fails and the outputs are untouched."""
    import ctypes as C
    from diffmm_b200 import _lib
    from diffmm_b200._lib import DiffMMError
    M, N, K = 128, 200, 64
    a = buf16(M, K)
    b = buf16(N, K)
    a[:] = 1
    b[:] = 1
    out = buf32(M, N)
    hi, lo = buf16(M, N), buf16(M, N)
    cm = buf32(M, 8)
    res = buf32(M, N)
    rh = buf16(M, N)
    bias = vec32(torch.zeros(N + 8, device=DEV))
    snapshot = [(t, t.clone()) for t in (out, hi, lo, cm)]
    A, B = a[:M, :K], b[:N, :K]
    o, h, l = out[:M, :N], hi[:M, :N], lo[:M, :N]
    z16 = lambda ld: torch.zeros((M, ld), dtype=torch.bfloat16, device=DEV)   # noqa: E731  (leading dimension ld)
    z32 = lambda ld: torch.zeros((M, ld), device=DEV)                         # noqa: E731
    plain = (A, None, B, None, M, N, K)
    calls = [
        ((A, None, B, None, M, 0, K), dict(out_f32=o)),                                  # empty problem
        ((A, None, B, None, 1 << 31, N, K), dict(out_f32=o)),                            # dimension too large
        ((z16(56), None, B, None, M, N, K), dict(out_f32=o)),                            # lda < K
        ((z16(68), None, B, None, M, N, K), dict(out_f32=o)),                            # lda % 8
        ((a[:M, 1:K + 1], None, B, None, M, N, K), dict(out_f32=o)),                     # misaligned operand
        (plain, dict(out_f32=out[:M, 1:N + 1])),                                         # misaligned epilogue buffer
        (plain, dict(out_f32=o, residual=z32(196))),                                     # ld_res < N
        (plain, dict(out_f32=o, residual=res[:M, :N], res_hi=rh[:M, :N])),              # residual and res_hi
        (plain, dict(out_f32=o, res_hi=z16(204))),                                       # ld_res16 % 8
        (plain, dict(out_f32=o, res_lo=rh[:M, :N])),                                     # res_lo without res_hi
        (plain, dict(out_f32=o, res_hi=rh[:M, 1:N + 1])),                                # misaligned res_hi
        (plain, dict(out_f32=z32(202))),                                                 # ld_out % 4
        (plain, dict(out_hi=z16(204))),                                                  # ld_out16 % 8
        (plain, dict(out_f32=o, out_lo=l)),                                              # out_lo without out_hi
        (plain, dict(out_f32=o, act=2)),                                                 # unknown activation
        (plain, dict(out_hi=h, post_act=2)),                                             # unknown post activation
        (plain, dict(out_f32=o, post_act=1)),                                            # post stage without out_hi
        (plain, dict(out_hi=h, post_bias=bias[1:N + 1])),                                # misaligned post_bias
        (plain, dict(out_f32=o, cmax=z32(6))),                                           # ld_cmax < ceil(N / 32)
    ]
    for args, kw in calls:
        with pytest.raises(DiffMMError):
            ops.gemm_bf16_tn(*args, **kw)
    ep = ops._epilogue(None, 0, 1.0, 0.0, None, o, None, None)
    with pytest.raises(DiffMMError):                                                     # null operand
        _lib.call("dmm_gemm_bf16_tn", ops._ctx(A), None, None, K, ops._p(B), None, K, M, N, K, C.byref(ep), ops._stream())
    torch.cuda.synchronize()
    for t, t0 in snapshot:
        assert same_bits(t, t0), "a rejected call wrote an output"
