"""The staging kernels at the head of the reverse chain (csrc/pack.cu), one entry point at a time, against float64 or
bit-exact restatements of what each one computes: time_bias, time_embedding, gemv_f32, bias_act_pack, csr_axpy_bf16,
csr_qsample_values, q_sample, csr_gather_act (per-slice and row-split kernels), rows_long_first, csr_rows_to_dense.

Conventions (those of test_train_kernels_gpu.py):
- split(v) is hi = bf16_rn(v), lo = bf16_rn(v - hi): dmm_split_bf16, the operand format of the contractions.
- Every output buffer is larger than the documented region (extra rows, leading dimensions beyond the width) and is
  filled with a sentinel first; after the call everything outside the region must still hold the sentinel.
- Exact integer and fp32 work is compared bit for bit; everything else against float64 within a bound derived, in a
  comment next to it, from the order of the kernel's operations.  u = 2^-24 is the unit roundoff of fp32 and
  gamma(n) = n u / (1 - n u) bounds the relative error of n roundings in a chain (Higham, ch. 3)."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
SENT16 = 0x7F3A          # a NaN pattern of bf16: never a value any of these kernels writes
SENT32 = float("nan")    # bits 0x7FC00000
NAN32_BITS = np.int32(0x7FC00000)
F32 = np.float32


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


def gamma(n):
    n = np.asarray(n, dtype=np.float64)
    return n * U / (1.0 - n * U)


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def f64(t):
    return t.detach().double().cpu().numpy()


def bits(t):
    """int16 / int32 bit view of a bf16 / fp32 tensor on the host (NaN-safe equality)."""
    return t.detach().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).cpu().numpy()


def bf16_rn(v):
    """Round-to-nearest-even bf16 bits (uint16) of a finite fp32 array."""
    b = np.ascontiguousarray(v, dtype=F32).view(np.uint32).astype(np.uint64)
    return ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint16)


def bf16_val(b):
    return (np.asarray(b).astype(np.uint16).astype(np.uint32) << 16).view(F32)


def split_np(v):
    """(hi, lo) bf16 bits of the fp32 array v: dmm_split_bf16 (v - hi is exact in fp32)."""
    v = np.asarray(v, dtype=F32)
    hi = bf16_rn(v)
    return hi, bf16_rn(v - bf16_val(hi))


def u16(t):
    return bits(t).view(np.uint16)


def is_nan16(b):
    return (b & 0x7FFF) > 0x7F80


def rn_bf16_64(v):
    """Round-to-nearest-even of float64 values to the bf16 grid (8 significant bits), as float64."""
    v = np.asarray(v, dtype=np.float64)
    _, ex = np.frexp(v)
    step = np.ldexp(1.0, np.maximum(ex - 8, -133))
    return np.round(v / step) * step              # np.round: half to even; v / step is exact (power of two)


def assert_split_within(hi, lo, center, err):
    """(hi, lo) is split(y) of some fp32 y with |y - center| <= err (lo None: hi = bf16_rn(y)).  Rounding to nearest is
    monotone, so hi lies between the roundings of the interval's ends and lo between those of the ends minus hi."""
    a, b = center - err, center + err
    hv = bf16_val(hi).astype(np.float64)
    ok = (rn_bf16_64(a) <= hv) & (hv <= rn_bf16_64(b))
    if lo is not None:
        lv = bf16_val(lo).astype(np.float64)
        ok &= (rn_bf16_64(a - hv) <= lv) & (lv <= rn_bf16_64(b - hv))
    assert ok.all(), f"{(~ok).sum()} outputs are not the split of a value within the bound, first at {np.argwhere(~ok)[0]}"


def tanh_err(x):
    """Bound on |tanh_k(x) - tanh(x)| for the kernels' tanh_k(x) = 1 - __fdividef(2, __expf(2x) + 1) (the same formula as
    the contraction epilogue's fast_tanh), x fp32.  With t = e^{2x} and q = 2 / (t + 1) = 1 - tanh(x):
    - __expf(2x) carries at most 2 + 1.173 |2x| ulp (CUDA guide), a relative error eps <= (2 + 2.35 |x|) 2^-23 of t,
      which moves tanh by (dq/dt) t eps = 2t / (t + 1)^2 eps = eps / (2 cosh^2 x);
    - t + 1 is rounded (relative u): q moves by q u;
    - __fdividef is within 2 ulp of q;
    - 1 - q is exact by Sterbenz for q in [1/2, 2]; otherwise it rounds: half an ulp of the result.
    The maximum over x is about 8 u = 4.75e-7 (near x = -0.56), inside the 5e-7 that test_round2_gpu.py holds the
    epilogue's tanh to."""
    x = np.asarray(x, dtype=np.float64)
    th = np.tanh(x)
    q = 1.0 - th
    ulp = lambda v: np.ldexp(1.0, np.frexp(np.abs(v))[1] - 24)      # fp32 ulp of the binade of v  # noqa: E731
    e = (2.0 + 2.35 * np.abs(x)) * 2.0 ** -23 / (2.0 * np.cosh(np.minimum(np.abs(x), 300.0)) ** 2)
    e += q * U + 2.0 * ulp(np.minimum(q, np.nextafter(2.0, 0.0)))   # q < 2 for finite x, even where float64 says 2
    e += np.where((q >= 0.5) & (q <= 2.0), 0.0, 0.5 * ulp(th))
    return e


def test_tanh_bound_meets_the_epilogue_bound():
    x = np.linspace(-30, 30, 600001)
    assert tanh_err(x).max() < 5e-7


def bf16_buf(rows, ld):
    b = torch.empty((rows, ld), dtype=torch.bfloat16, device=DEV)
    b.view(torch.int16).fill_(SENT16)
    return b


def f32_buf(*shape):
    return torch.full(shape, SENT32, dtype=torch.float32, device=DEV)


def assert_sentinel(buf, region_rows, region_cols, col0=0):
    """Everything of buf outside [:region_rows, col0:col0 + region_cols] still holds the sentinel."""
    b = bits(buf)
    s = NAN32_BITS if buf.dtype == torch.float32 else np.int16(SENT16)
    mask = np.ones(b.shape, dtype=bool)
    mask[:region_rows, col0:col0 + region_cols] = False
    assert (b[mask] == s).all(), "a kernel wrote outside its documented region"


def strided(a, extra=5, offset=0):
    """fp32 device copy of the host array a [R, C] as a view with leading dimension C + extra, starting `offset` elements
    into its buffer (offset 1: rows not 16-byte aligned)."""
    R, C = a.shape
    ld = C + extra
    buf = torch.full((R * ld + offset,), 1e30, dtype=torch.float32, device=DEV)
    v = buf[offset:].view(R, ld)
    v[:, :C] = T(np.asarray(a, dtype=F32))
    return v[:, :C]


def make_csr(rng, lens, n_cols, bad_every=0):
    """CSR rows with the given lengths, distinct in-range item ids; with bad_every > 0 every bad_every-th non-empty row
    also holds ids the kernels must skip (n_cols, n_cols + 3, -1, -5) at random positions."""
    ptr, idx = [0], []
    for r, n in enumerate(lens):
        row = list(rng.choice(n_cols, min(int(n), n_cols), replace=False))
        if bad_every and n and r % bad_every == 0:
            for bad in (n_cols, n_cols + 3, -1, -5):
                row.insert(int(rng.integers(0, len(row) + 1)), bad)
        idx += row
        ptr.append(len(idx))
    return np.array(ptr, dtype=np.int64), np.array(idx, dtype=np.int32)


# ---------------------------------------------------------------------------------------------- time embedding
def temb_ref(t, d, emb_w, emb_b):
    """Model.py:196-202 from the fp32 angle f32(t) * f32(f_j) that the reference (and oracle.time_embedding) forms, the
    sinusoid and the d x d Linear in float64.  Returns (e, bound on e, temb, bound on temb) for the kernels, which form
    the same angle in fp32 and then accumulate
        e_j = cosf / sinf(ang_j)  (0 for the padding column of an odd d),
        temb_o = emb_b[o] + sum_j fmaf(e_j, emb_w[o, j])        (d roundings in a chain).
    The kernels' f_j = expf(fl(fl(-logf(1e4) j) / half)) may differ from numpy's f32 frequency: logf is within 1 ulp,
    the two roundings of the argument a_j can then each differ by an ulp (|a_j| 3.5 2^-23 in all), expf is within 2 ulp
    and the reference's frequency within half an ulp, so |df_j| <= f_j (3.5 |a_j| + 2.5) 2^-23; the angle moves by
    t |df_j| plus one ulp of its own rounding, and cosf / sinf add 2 ulp (<= 2^-23 absolute)."""
    t = np.asarray(t, dtype=np.int64)
    half = d // 2
    a = (-F32(math.log(10000)) * np.arange(half, dtype=F32) / F32(half)).astype(F32)
    fj = np.exp(a.astype(np.float64)).astype(F32)
    ang = (t.astype(F32)[:, None] * fj[None, :]).astype(F32)
    e = np.concatenate([np.cos(ang.astype(np.float64)), np.sin(ang.astype(np.float64))], 1)
    de = t[:, None] * fj[None, :].astype(np.float64) * (3.5 * np.abs(a) + 2.5) * 2.0 ** -23
    de = de + np.spacing(np.abs(ang)).astype(np.float64) + 2.0 ** -23
    be = np.concatenate([de, de], 1)
    if d % 2:
        e = np.concatenate([e, np.zeros((len(t), 1))], 1)
        be = np.concatenate([be, np.zeros((len(t), 1))], 1)
    w = emb_w.astype(np.float64)
    aw = np.abs(w)
    temb = e @ w.T + emb_b.astype(np.float64)
    btemb = gamma(d) * (np.abs(emb_b) + (np.abs(e) + be) @ aw.T) + be @ aw.T
    return e, be, temb, btemb


TB_D = [2, 9, 10, 64]
TB_N = [1, 255, 256, 257, 1030]


@pytest.mark.parametrize("n_out", TB_N)
@pytest.mark.parametrize("d", TB_D)
def test_time_bias(ops, d, n_out):
    """bias_eff[i, h] = b[h] + sum_j fmaf(W[h, col0 + j], temb_j(t0 + i)) for n_t steps reaching t = 999, several CTAs per
    step, col0 != 0 and ld_w > col0 + d; bias None on every other shape.  Also against b + W[:, col0:col0+d] temb(t)
    with temb from dmm_time_embedding: two implementations of the same sinusoid."""
    rng = np.random.default_rng(100 * d + n_out)
    n_t = 6
    t0 = 1000 - n_t if n_out != 256 else 0
    col0 = 37
    emb_w = (rng.standard_normal((d, d)) / np.sqrt(d)).astype(F32)
    emb_b = (rng.standard_normal(d) * 0.1).astype(F32)
    W = (rng.standard_normal((n_out, col0 + d + 3)) * 0.2).astype(F32)
    b = None if TB_N.index(n_out) % 2 else (rng.standard_normal(n_out) * 0.3).astype(F32)
    weight = strided(W, extra=11)
    out = torch.full((n_t * n_out + 40,), SENT32, dtype=torch.float32, device=DEV)
    ops.time_bias(T(emb_w), T(emb_b), weight, col0, None if b is None else T(b), t0, n_t, out=out[:n_t * n_out])
    torch.cuda.synchronize()
    assert (bits(out)[n_t * n_out:] == NAN32_BITS).all(), "time_bias wrote past its n_t x n_out outputs"
    got = f64(out[:n_t * n_out]).reshape(n_t, n_out)
    steps = np.arange(t0, t0 + n_t)
    _, _, temb, btemb = temb_ref(steps, d, emb_w, emb_b)
    Wt = W[:, col0:col0 + d].astype(np.float64)
    b64 = np.zeros(n_out) if b is None else b.astype(np.float64)
    want = b64[None] + temb @ Wt.T
    # fp32 chain of d fmaf's from b[h] over the kernel's temb (which is within btemb of temb)
    bound = gamma(d) * (np.abs(b64)[None] + (np.abs(temb) + btemb) @ np.abs(Wt).T) + btemb @ np.abs(Wt).T
    assert np.all(np.abs(got - want) <= bound), f"time_bias off by {np.abs(got - want).max()} (bound {bound.min()})"

    te = f32_buf(n_t, d)
    ops.time_embedding(T(emb_w), T(emb_b), n_t, t=T(steps), temb_f32=te)
    other = b64[None] + f64(te) @ Wt.T
    # both within their bounds of the same float64 value: the time_bias bound plus |W| times the temb bound
    assert np.all(np.abs(got - other) <= bound + btemb @ np.abs(Wt).T)


@pytest.mark.parametrize("per_row", [True, False], ids=["t", "t_all"])
@pytest.mark.parametrize("d", TB_D)
def test_time_embedding(ops, d, per_row):
    """temb against float64 (odd d: zero padding column), and a_hi / a_lo at col0 > 0 of a wider row the bit-exact split
    of the temb_f32 the same call wrote; the other columns and the row past n_rows are untouched."""
    rng = np.random.default_rng(d + 7 * per_row)
    n_rows, col0 = 300, 13
    t = rng.integers(0, 1000, n_rows)
    t[:3] = [0, 999, 1]
    if not per_row:
        t[:] = 999
    emb_w = (rng.standard_normal((d, d)) / np.sqrt(d)).astype(F32)
    emb_b = (rng.standard_normal(d) * 0.1).astype(F32)
    ld_a = col0 + d + 11
    a_hi, a_lo = bf16_buf(n_rows + 1, ld_a), bf16_buf(n_rows + 1, ld_a)
    te = f32_buf(n_rows + 1, d)
    kw = dict(t=T(t)) if per_row else dict(t_all=999)
    ops.time_embedding(T(emb_w), T(emb_b), n_rows, a_hi=a_hi[:n_rows], a_lo=a_lo[:n_rows], col0=col0,
                       temb_f32=te[:n_rows], **kw)
    torch.cuda.synchronize()
    assert_sentinel(a_hi, n_rows, d, col0)
    assert_sentinel(a_lo, n_rows, d, col0)
    assert_sentinel(te, n_rows, d)
    _, _, temb, btemb = temb_ref(t, d, emb_w, emb_b)
    got = f64(te[:n_rows])
    assert np.all(np.abs(got - temb) <= btemb)
    hi, lo = split_np(te[:n_rows].cpu().numpy())
    assert np.array_equal(u16(a_hi[:n_rows, col0:col0 + d]), hi)
    assert np.array_equal(u16(a_lo[:n_rows, col0:col0 + d]), lo)


# ---------------------------------------------------------------------------------------------- gemv_f32
@pytest.mark.parametrize("n_rows", [1, 1024, 1025])
@pytest.mark.parametrize("K", [1, 3, 4, 5, 7050, 7060, 500003])
def test_gemv_f32(ops, K, n_rows):
    """y = W[:, :K] x on its three paths: float4 loads (ld_w % 4 == 0, x aligned) with the scalar tail of K % 4 columns,
    rows not 16-byte aligned (ld_w % 4 != 0), and x a view starting at element 1."""
    g = torch.Generator(device=DEV).manual_seed(K + n_rows)
    xs = torch.randn(K + 1, device=DEV, generator=g)
    for path in ("aligned", "ld_odd", "x_offset"):
        ld = (K + 3) // 4 * 4 + 4 if path != "ld_odd" else K + (1 if (K + 1) % 4 else 2)
        buf = torch.full((n_rows, ld), 1e30, device=DEV)
        buf[:, :K] = torch.randn((n_rows, K), device=DEV, generator=g)
        w = buf[:, :K]
        x = xs[1:] if path == "x_offset" else xs[:K].clone()
        out = torch.full((n_rows + 1,), SENT32, device=DEV)
        ops.gemv_f32(w, K, x, out[:n_rows])
        torch.cuda.synchronize()
        assert bits(out)[n_rows] == NAN32_BITS
        want = w.double() @ x.double()
        # each of the 128 threads runs one fmaf chain: vector path 4 ceil(K / 512) terms plus at most one of the K % 4
        # tail, scalar path ceil(K / 128); then 5 shuffle levels and (r0 + r1) + (r2 + r3): 7 more roundings
        n = max(4 * -(-K // 512) + 1, -(-K // 128)) + 7
        bound = float(gamma(n)) * (w.double().abs() @ x.double().abs())
        err = (out[:n_rows].double() - want).abs()
        assert bool((err <= bound).all()), f"{path}: off by {float(err.max())}"
        del buf, w


# ---------------------------------------------------------------------------------------------- bias_act_pack
ZSPECIAL = [0.0, 1e-6, -1e-6, 20.0, -20.0, float("nan"), 1e-7, -0.3, 0.55]


def _z_with_specials(rng, n_rows, n_cols):
    z = (rng.standard_normal((n_rows, n_cols)) * 1.5).astype(F32)
    pos = rng.choice(n_rows * n_cols, min(len(ZSPECIAL) * 3, n_rows * n_cols), replace=False)
    z.flat[pos] = np.resize(np.array(ZSPECIAL, dtype=F32), len(pos))
    z[0, :min(n_cols, len(ZSPECIAL))] = ZSPECIAL[:n_cols]
    z[:, -1] = np.resize(np.array(ZSPECIAL, dtype=F32), n_rows)      # the tail group's last column sees every value
    return z


def check_act_split(hi, lo, x, act):
    """hi (and lo, if given) of act(x) for the fp32 pre-activations x: act 0 the exact split; act 1 the split of an fp32
    value within tanh_err of tanh(x).  NaN in, NaN out."""
    nan = np.isnan(x)
    assert is_nan16(hi[nan]).all() and (lo is None or is_nan16(lo[nan]).all())
    xf = np.where(nan, 0, x).astype(F32)
    if act == 0:
        h, l = split_np(xf)
        assert np.array_equal(hi[~nan], h[~nan])
        if lo is not None:
            assert np.array_equal(lo[~nan], l[~nan])
    else:
        assert_split_within(hi[~nan], None if lo is None else lo[~nan], np.tanh(xf[~nan].astype(np.float64)),
                            tanh_err(xf[~nan]))


@pytest.mark.parametrize("act", [0, 1])
@pytest.mark.parametrize("n_cols", [1, 3, 4, 5, 1023, 1030])
def test_bias_act_pack(ops, n_cols, act):
    """h = act(z + b) for z with 0, +-1e-6, +-20 and NaN, hi only and hi + lo, with and without bias; the ragged last
    group of n_cols % 4 columns takes the scalar path."""
    rng = np.random.default_rng(n_cols * 2 + act)
    n_rows = 37
    z = _z_with_specials(rng, n_rows, n_cols)
    ld = (n_cols + 3) // 4 * 4 + 4
    zbuf = torch.full((n_rows + 1, ld), 1e30, device=DEV)
    zbuf[:n_rows, :n_cols] = T(z)
    for with_bias in (True, False):
        b = (rng.standard_normal(n_cols) * 0.7).astype(F32)
        for with_lo in (False, True):
            h_hi, h_lo = bf16_buf(n_rows + 1, ld), bf16_buf(n_rows + 1, ld)
            ops.bias_act_pack(zbuf[:n_rows, :n_cols], T(b) if with_bias else None, act, h_hi[:n_rows],
                              h_lo[:n_rows] if with_lo else None)
            torch.cuda.synchronize()
            assert_sentinel(h_hi, n_rows, n_cols)
            assert_sentinel(h_lo, n_rows if with_lo else 0, n_cols)
            x = (z + b[None]).astype(F32) if with_bias else z          # the kernel's fp32 sum (one rounding)
            check_act_split(u16(h_hi[:n_rows, :n_cols]), u16(h_lo[:n_rows, :n_cols]) if with_lo else None, x, act)


# ---------------------------------------------------------------------------------------------- csr_axpy_bf16
@pytest.mark.parametrize("beta", [0.0, -0.3, 1.7])
@pytest.mark.parametrize("sel", ["row0", "row_ids"])
@pytest.mark.parametrize("with_lo", [False, True], ids=["hi", "hi_lo"])
def test_csr_axpy_bf16(ops, with_lo, sel, beta):
    """x[r, c] += beta at the CSR entries of each selected row: v = f32(hi) (+ f32(lo)) + beta, then the RNE split.
    Empty rows, ids >= n_cols and negative ids (skipped), a repeated and a permuted user; every other position of the
    buffer (other columns, padding, unselected rows) keeps its bits."""
    rng = np.random.default_rng(int(round(beta * 10)) + 40 + 3 * with_lo + (sel == "row_ids"))
    n_users, n_cols = 60, 1030
    lens = rng.integers(0, 40, n_users)
    lens[[2, 9, 10]] = 0
    lens[5] = 300
    indptr, indices = make_csr(rng, lens, n_cols, bad_every=3)
    if sel == "row0":
        row0, n_rows, users = 4, 41, np.arange(4, 45)
    else:
        users = np.array([7, 7, 2, 5, 31, 0, 59, 13, 9, 44, 3, 7, 58, 21], dtype=np.int64)
        row0, n_rows = 0, len(users)
    ld = n_cols + 5
    x = (rng.standard_normal((n_rows + 2, ld)) * 2).astype(F32)
    hi0, lo0 = split_np(x)
    x_hi = T(hi0.view(np.int16)).view(torch.bfloat16)
    x_lo = T(lo0.view(np.int16)).view(torch.bfloat16)
    ops.csr_axpy_bf16(T(indptr), T(indices), n_rows, n_cols, beta, x_hi[:n_rows, :n_cols],
                      x_lo[:n_rows, :n_cols] if with_lo else None,
                      row_ids=T(users) if sel == "row_ids" else None, row0=row0)
    torch.cuda.synchronize()
    want_hi, want_lo = hi0.copy(), lo0.copy()
    for r, u in enumerate(users):
        c = indices[indptr[u]:indptr[u + 1]]
        c = c[(c >= 0) & (c < n_cols)]
        v = bf16_val(hi0[r, c])
        if with_lo:
            v = (v + bf16_val(lo0[r, c])).astype(F32)
        v = (v + F32(beta)).astype(F32)
        h, l = split_np(v)
        want_hi[r, c] = h
        if with_lo:
            want_lo[r, c] = l
    assert np.array_equal(u16(x_hi), want_hi)
    assert np.array_equal(u16(x_lo), want_lo)


# ---------------------------------------------------------------------------------------------- q_sample values
def norm_rel(n_cols):
    """Relative error bound of the kernels' 1 / max(||n||, 1e-12): the squared norm is a sum of positive terms, each
    thread's fmaf chain (float4 path: 4 ceil(n / 1024) terms plus at most one of the tail; scalar path: ceil(n / 256))
    then 5 shuffle levels and the sequential sum of the 8 warp sums (7 additions): gamma(N) relative; sqrtf and the
    division are correctly rounded (no fast math): sqrt(1 + gamma(N)) (1 + u)^2 - 1."""
    N = max(4 * -(-n_cols // 1024) + 1, -(-n_cols // 256)) + 12
    return np.sqrt(1 + gamma(N)) * (1 + U) ** 2 - 1


@pytest.mark.parametrize("sel", ["row0", "row_ids"])
@pytest.mark.parametrize("n_cols", [1, 3, 4, 7050, 70001])
def test_csr_qsample_values(ops, n_cols, sel):
    """vals[e] = a + b n[c] / max(||n||, 1e-12) on caller-given noise rows: an all-zero noise row (values exactly a), an
    empty row, skipped ids (values exactly a), rows of an odd ld_noise (row_ids: mixed float4 and scalar norm paths).
    Entries of rows that are not selected keep the sentinel.  Then against q_sample(mode=1) on the densified rows."""
    rng = np.random.default_rng(n_cols + (sel == "row_ids"))
    n_users = 50
    lens = rng.integers(1, 30, n_users)
    lens[[4, 17]] = 0
    lens[6] = min(n_cols, 600)
    indptr, indices = make_csr(rng, lens, n_cols, bad_every=5)
    if sel == "row0":
        row0, users = 3, np.arange(3, 3 + 30)
        extra = 4                                    # ld_noise % 4 == 0: every row on the float4 path
    else:
        # distinct users: vals is indexed like indices, so two selected rows of one user would write the same entries
        users = np.array([6, 17, 0, 33, 12, 49, 20, 1, 2, 45, 5], dtype=np.int64)
        row0, extra = 0, 3                           # ld_noise % 4 != 0: rows alternate between both paths
    n_rows = len(users)
    noise = rng.standard_normal((n_rows, n_cols)).astype(F32)
    noise[2] = 0.0
    ld = (n_cols + 3) // 4 * 4 + extra
    nz = strided(noise, extra=ld - n_cols)
    a, b = 0.8123, 0.3377
    vals = torch.full((len(indices),), SENT32, device=DEV)
    ops.csr_qsample_values(T(indptr), T(indices), n_rows, n_cols, nz, a, b, vals,
                           row_ids=T(users) if sel == "row_ids" else None, row0=row0)
    torch.cuda.synchronize()
    got = f64(vals)
    gbits = bits(vals)
    written = np.zeros(len(indices), dtype=bool)
    rho = norm_rel(n_cols)
    af, bf = float(F32(a)), float(F32(b))
    qs_rows, qs_vals, qs_bound = [], [], []
    for r, u in enumerate(users):
        e0, e1 = indptr[u], indptr[u + 1]
        written[e0:e1] = True
        c = indices[e0:e1]
        ok = (c >= 0) & (c < n_cols)
        nrm = max(np.sqrt((noise[r].astype(np.float64) ** 2).sum()), 1e-12)
        y = bf * np.where(ok, noise[r, np.where(ok, c, 0)], 0.0) / nrm
        want = af + y
        # b n inv carries rho and the two products' roundings; the final addition rounds once more
        rel = (1 + rho) * (1 + gamma(2)) - 1
        bound = np.abs(y) * rel * (1 + U) + U * np.abs(want)
        assert np.all(np.abs(got[e0:e1] - want) <= bound), f"row {r}: off by {np.abs(got[e0:e1] - want).max()}"
        if r == 2 or not ok.all():
            assert np.all(got[e0:e1][(~ok) | (r == 2)] == af), "zero noise and skipped ids must give exactly coef_a"
        qs_rows.append((r, c[ok], e0 + np.nonzero(ok)[0]))
        qs_bound.append(bound[ok])
    assert (gbits[~written] == NAN32_BITS).all(), "entries of rows that were not selected were written"

    # q_sample(mode=1) on the same rows densified: the same quantity, but its norm is reduced in another order (scalar
    # loads, one fmaf chain per thread over columns tid, tid + 256, ...), so the two agree within the sum of their
    # bounds, not bit for bit
    x0 = np.zeros((n_rows, n_cols), dtype=F32)
    for r, c, _ in qs_rows:
        x0[r, c] = 1.0
    xt = f32_buf(n_rows, n_cols)
    ca, cb = T(np.full(n_rows, a, dtype=F32)), T(np.full(n_rows, b, dtype=F32))
    ops.q_sample(T(x0), nz, ca, cb, 1, x_t=xt)
    xq = f64(xt)
    for (r, c, e), bd in zip(qs_rows, qs_bound):
        assert np.all(np.abs(xq[r, c] - got[e]) <= 2 * bd)


# ---------------------------------------------------------------------------------------------- q_sample
@pytest.mark.parametrize("n_cols", [1, 7, 1003, 7050])
@pytest.mark.parametrize("mode", [0, 1])
def test_q_sample(ops, mode, n_cols):
    """x_t = a_r x0 + b_r noise (mode 0) or a_r x0 + b_r sign(x0) noise / max(||noise_r||, 1e-12) (mode 1) with x0 of
    both signs and zeros, one all-zero noise row and distinct per-row coefficients; a_hi / a_lo are the bit-exact split
    of the x_t the same call wrote."""
    rng = np.random.default_rng(n_cols * 2 + mode)
    n_rows = 45
    x0 = rng.standard_normal((n_rows, n_cols)).astype(F32) * (rng.random((n_rows, n_cols)) < 0.5)
    x0[1] = 0.0
    noise = rng.standard_normal((n_rows, n_cols)).astype(F32)
    noise[3] = 0.0
    ca = rng.random(n_rows).astype(F32)
    cb = rng.random(n_rows).astype(F32)
    ld = n_cols + 6
    xt = f32_buf(n_rows + 1, ld)
    a_hi, a_lo = bf16_buf(n_rows + 1, ld), bf16_buf(n_rows + 1, ld)
    ops.q_sample(strided(x0, 3), strided(noise, 1, offset=1), T(ca), T(cb), mode, x_t=xt[:n_rows, :n_cols],
                 a_hi=a_hi[:n_rows, :n_cols], a_lo=a_lo[:n_rows, :n_cols])
    torch.cuda.synchronize()
    for buf in (xt, a_hi, a_lo):
        assert_sentinel(buf, n_rows, n_cols)
    x64, n64 = x0.astype(np.float64), noise.astype(np.float64)
    a64, b64 = ca.astype(np.float64)[:, None], cb.astype(np.float64)[:, None]
    if mode == 0:
        nn, rel = n64, 0.0
    else:
        nrm = np.maximum(np.sqrt((n64 ** 2).sum(1, keepdims=True)), 1e-12)
        nn, rel = np.sign(x64) * n64 / nrm, (1 + norm_rel(n_cols)) * (1 + U) - 1     # and the rounding of n inv
    want = a64 * x64 + b64 * nn
    # a x + b n': products and sum rounded (or contracted into one fmaf): gamma(2) over |a x| + |b n'|, n' within rel
    bound = gamma(2) * (np.abs(a64 * x64) + np.abs(b64 * nn)) + np.abs(b64 * nn) * rel * (1 + gamma(2))
    got = f64(xt[:n_rows, :n_cols])
    assert np.all(np.abs(got - want) <= bound), f"x_t off by {np.abs(got - want).max()}"
    hi, lo = split_np(xt[:n_rows, :n_cols].cpu().numpy())
    assert np.array_equal(u16(a_hi[:n_rows, :n_cols]), hi) and np.array_equal(u16(a_lo[:n_rows, :n_cols]), lo)


# ---------------------------------------------------------------------------------------------- csr_gather_act
GA_N = [1, 7, 9, 255, 257, 1030]
GA_CASES = ["binary_hi", "weighted_hi", "binary_split", "weighted_split"]


@pytest.mark.parametrize("kernel", ["per_slice", "row_split"])
@pytest.mark.parametrize("case", GA_CASES)
@pytest.mark.parametrize("n_out", GA_N)
def test_csr_gather_act_kernels(ops, n_out, case, kernel):
    """z = sum over a row's entries of vals * (hi + lo) of W^T, h = act(z + bias) split, on the per-slice kernel (order
    None or a plain permutation) and the row-split kernel (a rows_long_first order, n_out <= 1024): weighted rows,
    split weights, row_ids with a repeated and a permuted user, empty rows (z = 0, h = act(bias)), skipped ids; the table
    rows past n_cols hold huge values, so a gathered out-of-range id would show."""
    if kernel == "row_split" and n_out > 1024:
        pytest.skip("the row-split kernel takes at most 1024 output columns")
    ci = GA_CASES.index(case)
    weighted, with_lo = "weighted" in case, "split" in case
    rng = np.random.default_rng(n_out * 10 + ci)
    n_cols, n_users, thr = 600, 70, 8
    lens = rng.integers(0, 7, n_users)
    lens[[3, 40]] = 0
    lens[[5, 6, 50]] = [40, 9, 130]            # longer than the threshold: the long-row role of the row-split kernel
    lens[7] = thr                              # exactly at it: a short row
    indptr, indices = make_csr(rng, lens, n_cols, bad_every=4)
    ld_w = (n_out + 7) // 8 * 8 + 8
    W = (rng.standard_normal((n_cols + 9, ld_w)) * 0.3).astype(F32)
    W[n_cols:] = 1e4
    w_hi, w_lo = split_np(W)
    t_hi = T(w_hi.view(np.int16)).view(torch.bfloat16)
    t_lo = T(w_lo.view(np.int16)).view(torch.bfloat16) if with_lo else None
    vals = (rng.standard_normal(len(indices)) * 0.8).astype(F32) if weighted else None
    if weighted:
        vals[::5] = 1.0
    bias_buf = (rng.standard_normal(n_out + 1) * 0.5).astype(F32)
    bias_t = T(bias_buf)[ci % 2:ci % 2 + n_out]        # every other case: a bias that is not 16-byte aligned
    if ci % 2:
        users = np.array([5, 3, 5, 50, 0, 12, 7, 69, 6, 33, 40, 21, 2, 1, 64, 9], dtype=np.int64)
        row0, row_ids = 0, T(users)
    else:
        row0 = 2
        users = np.arange(row0, row0 + 60)
        row_ids = None
    n_rows = len(users)
    if kernel == "row_split":
        sel_ptr = np.concatenate([[0], np.cumsum(np.diff(indptr)[users])]).astype(np.int64)
        order = ops.rows_long_first(T(sel_ptr), 0, n_rows, thr)
    else:
        order = None if ci % 2 else T(rng.permutation(n_rows).astype(np.int32))

    # float64 reference of z and its bound: the kernels accumulate in fp32 in stored order, one rounding per term (hi,
    # then lo, of each entry; skipped ids and padded slots add exact zeros): gamma(m) over the absolute terms
    hv, lv = bf16_val(w_hi).astype(np.float64), bf16_val(w_lo).astype(np.float64)
    z64 = np.zeros((n_rows, n_out))
    zb = np.zeros((n_rows, n_out))
    for r, u in enumerate(users):
        e0, e1 = indptr[u], indptr[u + 1]
        c = indices[e0:e1]
        ok = (c >= 0) & (c < n_cols)
        v = vals[e0:e1][ok].astype(np.float64) if weighted else np.ones(ok.sum())
        parts = hv[c[ok], :n_out] + (lv[c[ok], :n_out] if with_lo else 0)
        absp = np.abs(hv[c[ok], :n_out]) + (np.abs(lv[c[ok], :n_out]) if with_lo else 0)
        z64[r] = v @ parts
        zb[r] = gamma((2 if with_lo else 1) * ok.sum()) * (np.abs(v) @ absp)

    ld_h = (n_out + 7) // 8 * 8 + 8
    ld_z = (n_out + 3) // 4 * 4 + 4
    h_prev = None
    for act in (0, 1):
        h_hi, h_lo = bf16_buf(n_rows + 2, ld_h), bf16_buf(n_rows + 2, ld_h)
        z = f32_buf(n_rows + 2, ld_z)
        ops.csr_gather_act(T(indptr), T(indices), n_rows, n_cols, t_hi, t_lo, bias_t, act, n_out, h_hi[:n_rows],
                           h_lo[:n_rows] if with_lo else None, row_ids=row_ids, row0=row0, z_f32=z[:n_rows],
                           order=order, vals=None if vals is None else T(vals))
        torch.cuda.synchronize()
        assert_sentinel(h_hi, n_rows, n_out)
        assert_sentinel(h_lo, n_rows if with_lo else 0, n_out)
        assert_sentinel(z, n_rows, n_out)
        zg = z[:n_rows, :n_out].cpu().numpy()
        err = np.abs(zg.astype(np.float64) - z64)
        assert np.all(err <= zb), f"z off by {err.max()} at {np.unravel_index(np.argmax(err - zb), err.shape)}"
        x = (zg + bias_buf[ci % 2:ci % 2 + n_out][None]).astype(F32)      # the kernels' fp32 z + bias
        check_act_split(u16(h_hi[:n_rows, :n_out]), u16(h_lo[:n_rows, :n_out]) if with_lo else None, x, act)
        if act == 1:
            h_prev = (h_hi.clone(), h_lo.clone())
    # without z_f32 the activations are the same bits
    h_hi, h_lo = bf16_buf(n_rows + 2, ld_h), bf16_buf(n_rows + 2, ld_h)
    ops.csr_gather_act(T(indptr), T(indices), n_rows, n_cols, t_hi, t_lo, bias_t, 1, n_out, h_hi[:n_rows],
                       h_lo[:n_rows] if with_lo else None, row_ids=row_ids, row0=row0, order=order,
                       vals=None if vals is None else T(vals))
    assert np.array_equal(bits(h_hi), bits(h_prev[0])) and np.array_equal(bits(h_lo), bits(h_prev[1]))


# ---------------------------------------------------------------------------------------------- rows_long_first
@pytest.mark.parametrize("threshold", [0, 5, 32])
@pytest.mark.parametrize("n_rows", [1, 31, 32, 33, 257, 100000])
def test_rows_long_first(ops, n_rows, threshold):
    """A permutation of the block's rows whose first counters[0] entries are exactly the rows of MORE than `threshold`
    entries: rows of exactly `threshold` entries are short; warps of 32 rows that are all long and all short."""
    rng = np.random.default_rng(n_rows + threshold)
    row0 = 17
    n_all = row0 + n_rows + 5
    lens = rng.choice([0, threshold, threshold + 1, 2 * threshold + 3], n_all)
    if n_rows >= 96:
        lens[row0:row0 + 32] = threshold + 1 + rng.integers(0, 3, 32)       # a warp of long rows
        lens[row0 + 32:row0 + 64] = rng.integers(0, threshold + 1, 32)      # a warp of short rows
    lens[row0 + n_rows - 1] = threshold
    if n_rows > 1:
        lens[row0 + n_rows - 2] = threshold + 1
    indptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    order = ops.rows_long_first(T(indptr), row0, n_rows, threshold)
    torch.cuda.synchronize()
    o = order.cpu().numpy()
    n_long = int(order._dmm_counters[0].item())
    assert np.array_equal(np.sort(o), np.arange(n_rows)), "not a permutation of the rows"
    long_rows = np.nonzero(lens[row0:row0 + n_rows] > threshold)[0]
    assert n_long == len(long_rows)
    assert np.array_equal(np.sort(o[:n_long]), long_rows)


# ---------------------------------------------------------------------------------------------- csr_rows_to_dense
@pytest.mark.parametrize("sel", ["row0", "row_ids"])
@pytest.mark.parametrize("n_cols", [1, 5, 7, 300, 1031])
def test_csr_rows_to_dense(ops, n_cols, sel):
    """Dense 0/1 rows in fp32 and bf16 with odd leading dimensions and a buffer that starts one element in, so that rows
    are not 16-byte aligned and zero_row's scalar head and tail run; ids out of range are skipped; padding columns and
    the rows past n_rows keep the sentinel."""
    rng = np.random.default_rng(n_cols + 5 * (sel == "row_ids"))
    n_users = 40
    lens = rng.integers(0, min(n_cols, 12) + 1, n_users)
    lens[3] = 0
    lens[8] = n_cols
    indptr, indices = make_csr(rng, lens, n_cols, bad_every=3)
    if sel == "row0":
        row0, users, row_ids = 6, np.arange(6, 6 + 27), None
    else:
        users = np.array([8, 3, 8, 0, 39, 21, 2, 11], dtype=np.int64)
        row0, row_ids = 0, T(users)
    n_rows = len(users)
    ld_x, ld_a = n_cols + 3, n_cols + (1 if n_cols % 2 == 0 else 2)     # odd ld_a: bf16 rows at 2-byte offsets
    xflat = torch.full(((n_rows + 1) * ld_x + 1,), SENT32, device=DEV)
    aflat = torch.empty(((n_rows + 1) * ld_a + 1,), dtype=torch.bfloat16, device=DEV)
    aflat.view(torch.int16).fill_(SENT16)
    xbuf = xflat[1:].view(n_rows + 1, ld_x)
    abuf = aflat[1:].view(n_rows + 1, ld_a)
    ops.csr_rows_to_dense(T(indptr), T(indices), n_rows, n_cols, row_ids=row_ids, row0=row0,
                          x_f32=xbuf[:n_rows, :n_cols], a_bf16=abuf[:n_rows, :n_cols])
    torch.cuda.synchronize()
    assert bits(xflat)[0] == NAN32_BITS and bits(aflat)[0] == SENT16
    assert_sentinel(xbuf, n_rows, n_cols)
    assert_sentinel(abuf, n_rows, n_cols)
    want = np.zeros((n_rows, n_cols), dtype=F32)
    for r, u in enumerate(users):
        c = indices[indptr[u]:indptr[u + 1]]
        want[r, c[(c >= 0) & (c < n_cols)]] = 1.0
    assert np.array_equal(bits(xbuf[:n_rows, :n_cols]), want.view(np.int32))
    assert np.array_equal(u16(abuf[:n_rows, :n_cols]), bf16_rn(want))
