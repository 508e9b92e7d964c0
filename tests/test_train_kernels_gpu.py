"""The kernels of the fused Denoise training step (csrc/train.cu), one entry point at a time, against plain float64 (or
bit-exact fp32) restatements of what each one computes; then the whole step (train_step.DenoiseLossFn) at the shapes
the other whole-step tests never use: batches below 64 rows, odd and extreme time-embedding widths, empty x0 rows and
a saturated model.

Conventions:
- split(v) is hi = bf16_rn(v), lo = bf16_rn(v - hi): dmm_split_bf16, the operand format of the contractions.
- Every output buffer is larger than the documented region (extra rows, leading dimensions beyond the width) and is
  filled with a sentinel first; after the call everything outside the region must still hold the sentinel.
- Sizes are ragged: B in {1, 5, 63, 300, 1025} rows, widths in {1, 7, 1003, 6710}, so that width mod 4 and mod 8 and
  the tails of the 32 x 32 tiles all vary."""
import ast
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BS = [1, 5, 63, 300, 1025]
IS = [1, 7, 1003, 6710]
U24 = 2.0 ** -24
SENT16 = 0x7F3A          # a NaN pattern of bf16: never a value any of these kernels writes
SENT32 = float("nan")    # bits 0x7FC00000
NAN32_BITS = np.int32(0x7FC00000)


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def f64(t):
    return t.detach().double().cpu().numpy()


def bits(t):
    """int16 / int32 bit view of a bf16 / fp32 tensor on the host (NaN-safe equality)."""
    return t.detach().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).cpu().numpy()


def split(v):
    """(hi, lo) bf16 of an fp32 tensor: the reference of dmm_split_bf16."""
    hi = v.bfloat16()
    return hi, (v - hi.float()).bfloat16()


def bf16_buf(rows, ld):
    b = torch.empty((rows, ld), dtype=torch.bfloat16, device=DEV)
    b.view(torch.int16).fill_(SENT16)
    return b


def f32_buf(*shape):
    return torch.full(shape, SENT32, dtype=torch.float32, device=DEV)


def assert_sentinel(buf, region_rows, region_cols):
    """Everything of buf outside [:region_rows, :region_cols] still holds the sentinel."""
    b = bits(buf)
    s = NAN32_BITS if buf.dtype == torch.float32 else np.int16(SENT16)
    mask = np.ones(b.shape, dtype=bool)
    mask[:region_rows, :region_cols] = False
    assert (b[mask] == s).all(), "a kernel wrote outside its documented region"


def strided(a, extra=5):
    """fp32 device copy of the host array a [R, C] as a view with leading dimension C + extra."""
    R, C = a.shape
    buf = torch.full((R, C + extra), 1e30, dtype=torch.float32, device=DEV)
    buf[:, :C] = T(a.astype(np.float32))
    return buf[:, :C]


# ---------------------------------------------------------------------------------------------- train_prep
def temb64(t, d, emb_w, emb_b):
    """Model.py:196-202 in float64: [cos(t f), sin(t f)] (zero column appended for odd d), then the d x d Linear."""
    half = d // 2
    freqs = np.exp(-math.log(10000.0) * np.arange(half, dtype=np.float64) / half)
    ang = t.astype(np.float64)[:, None] * freqs[None]
    e = np.concatenate([np.cos(ang), np.sin(ang)], 1)
    if d % 2:
        e = np.concatenate([e, np.zeros((len(t), 1))], 1)
    return e, e @ emb_w.astype(np.float64).T + emb_b.astype(np.float64)


def _run_train_prep(ops, B, I, d, t, seed):
    rng = np.random.default_rng(seed)
    x0 = rng.standard_normal((B, I)).astype(np.float32) * (rng.random((B, I)) < 0.3)
    noise = rng.standard_normal((B, I)).astype(np.float32)
    tab_a = rng.random(1000).astype(np.float32)
    tab_b = rng.random(1000).astype(np.float32)
    emb_w = (rng.standard_normal((d, d)) / np.sqrt(d)).astype(np.float32)
    emb_b = (rng.standard_normal(d) * 0.1).astype(np.float32)
    ld_a = ops.pad_to(I + d, 64) + 64
    ld_x = ops.pad_to(I, 2) + 10
    a_hi, a_lo, x0_hi = bf16_buf(B + 1, ld_a), bf16_buf(B + 1, ld_a), bf16_buf(B + 1, ld_x)
    te_raw = f32_buf(B + 1, d)
    ops.train_prep(strided(x0), strided(noise, 3), T(t), T(tab_a), T(tab_b), T(emb_w), T(emb_b), a_hi[:B], a_lo[:B],
                   x0_hi[:B], te_raw[:B])
    torch.cuda.synchronize()
    for buf, cols in ((a_hi, I + d), (a_lo, I + d), (x0_hi, I), (te_raw, d)):
        assert_sentinel(buf, B, cols)
    return x0, noise, tab_a, tab_b, emb_w, emb_b, a_hi[:B], a_lo[:B], x0_hi[:B], te_raw[:B]


def _check_temb(t, d, emb_w, emb_b, a_hi, a_lo, te_raw, I):
    e64, want = temb64(t, d, emb_w, emb_b)
    # a frequency the kernel and numpy round 1 ulp apart moves the angle by about t 2^-24; expf / cosf / sinf add a few
    # ulp of their own
    tol_e = (4e-7 + 8.0 * t * U24)[:, None]
    got_e = f64(te_raw)
    assert np.all(np.abs(got_e - e64) <= tol_e)
    if d % 2:
        assert np.all(got_e[:, d - 1] == 0.0), "the padding column of an odd time embedding must be exactly 0"
    got = f64(a_hi[:, I:I + d]) + f64(a_lo[:, I:I + d])
    aw = np.abs(emb_w.astype(np.float64))
    tol = tol_e @ np.ones((1, d)) * aw.sum(1)[None] + 2.0 ** -16 * (np.abs(e64) @ aw.T + np.abs(emb_b))
    assert np.all(np.abs(got - want) <= tol)


@pytest.mark.parametrize("I", IS)
@pytest.mark.parametrize("B", BS)
def test_train_prep(ops, B, I):
    d = [2, 9, 10, 64][(BS.index(B) + IS.index(I)) % 4]
    rng = np.random.default_rng(B * 7 + I)
    t = rng.integers(0, 1000, B)
    x0, noise, tab_a, tab_b, emb_w, emb_b, a_hi, a_lo, x0_hi, te_raw = _run_train_prep(ops, B, I, d, t, B + I)
    # x_t = fl(fl(a_t x0) + fl(b_t noise)): explicit __fmul_rn / __fadd_rn, so numpy float32 reproduces it bit for bit
    xt = tab_a[t][:, None] * x0 + tab_b[t][:, None] * noise
    hi, lo = split(torch.from_numpy(xt))
    assert np.array_equal(bits(a_hi[:, :I]), bits(hi)) and np.array_equal(bits(a_lo[:, :I]), bits(lo))
    assert np.array_equal(bits(x0_hi[:, :I]), bits(torch.from_numpy(x0).bfloat16()))
    _check_temb(t, d, emb_w, emb_b, a_hi, a_lo, te_raw, I)


@pytest.mark.parametrize("d", [2, 9, 10, 64])
def test_train_prep_time_embedding_every_step(ops, d):
    """Every t of a 1000-step schedule, for the narrowest, an odd, the shipped and the widest embedding; I = 7 leaves an
    unpaired last column next to the 32-bit pair stores and puts the embedding at an odd column."""
    B, I = 1000, 7
    t = np.arange(B)[::-1].copy()
    _, _, _, _, emb_w, emb_b, a_hi, a_lo, _, te_raw = _run_train_prep(ops, B, I, d, t, d)
    _check_temb(t, d, emb_w, emb_b, a_hi, a_lo, te_raw, I)


# ---------------------------------------------------------------------------------------------- gate
@pytest.mark.parametrize("B", BS)
def test_gate_fwd_and_bwd_pre(ops, B):
    rng = np.random.default_rng(B)
    p = (rng.standard_normal((B, 64)) * 0.7).astype(np.float32)
    gw = (rng.standard_normal((64, 64)) / 8).astype(np.float32)
    gb = (rng.standard_normal(64) * 0.1).astype(np.float32)
    sig = f32_buf(B + 1, 64)
    g_hi, g_lo = bf16_buf(B + 1, 72), bf16_buf(B + 1, 72)
    ops.gate_fwd(strided(p, 8), T(gw), T(gb), sig[:B], g_hi[:B], g_lo[:B])
    torch.cuda.synchronize()
    for buf in (sig, g_hi, g_lo):
        assert_sentinel(buf, B, 64)
    pre = p.astype(np.float64) @ gw.astype(np.float64).T + gb
    s64 = 1.0 / (1.0 + np.exp(-pre))
    s = sig[:B].cpu().numpy()
    # fp32 fma chain over 64 products, then expf and a division: s' <= 1/4 damps the sum's error
    tol_s = 0.25 * 66 * U24 * (np.abs(p.astype(np.float64)) @ np.abs(gw.astype(np.float64)).T + np.abs(gb)) + 4 * U24
    assert np.all(np.abs(s - s64) <= tol_s)
    g = torch.from_numpy(p * s)                   # G = fl(P sig): one rounding
    hi, lo = split(g)
    assert np.array_equal(bits(g_hi[:B, :64]), bits(hi)) and np.array_equal(bits(g_lo[:B, :64]), bits(lo))
    assert np.all(np.abs(g.double().numpy() - p * s64) <= np.abs(p) * tol_s + 2 * U24 * np.abs(p * s64))
    # single-pass mode: no lo output
    g_hi2 = bf16_buf(B + 1, 64)
    ops.gate_fwd(strided(p, 8), T(gw), T(gb), sig[:B], g_hi2[:B], None)
    assert np.array_equal(bits(g_hi2[:B]), bits(hi))
    assert_sentinel(g_hi2, B, 64)
    # d pre = ((dG P) s) (1 - s), in that order, in fp32
    dg = rng.standard_normal((B, 64)).astype(np.float32)
    dpre = f32_buf(B + 1, 64)
    ops.gate_bwd_pre(strided(dg, 3), strided(p, 8), sig[:B], dpre[:B])
    torch.cuda.synchronize()
    assert_sentinel(dpre, B, 64)
    want = dg * p * s * (np.float32(1.0) - s)
    assert np.array_equal(bits(dpre[:B]), want.view(np.int32))


# ---------------------------------------------------------------------------------------------- loss tail
def _schedule50():
    from diffmm_b200.Conf import Config
    from diffmm_b200.Model import GaussianDiffusion
    cfg = Config()
    cfg.hyper.steps = 50
    cfg.hyper.noise_scale = 0.5
    gd = GaussianDiffusion(cfg).to(DEV)
    return gd._train_tables(DEV)[2]


def _dcos_du(u, v, eps=1e-8):
    """float64 derivative of cos(u, v) = u.v / (max(|u|, eps) max(|v|, eps)) w.r.t. u, row-wise: the clamped norm is a
    constant, so its branch has no second term."""
    a, b = np.linalg.norm(u, axis=1), np.linalg.norm(v, axis=1)
    ac, bc = np.maximum(a, eps), np.maximum(b, eps)
    cos = (u * v).sum(1) / (ac * bc)
    sec = np.where((a > eps)[:, None], cos[:, None] * u / (ac * np.where(a > 0, a, 1.0))[:, None], 0.0)
    return v / (ac * bc)[:, None] - sec, (v / (ac * bc)[:, None], np.abs(cos[:, None] * u) / (ac * np.maximum(a, eps))[:, None])


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("I", IS)
@pytest.mark.parametrize("B", [5, 63, 300])
def test_diff_loss_fwd_bwd(ops, B, I, offset):
    """offset 1 shifts every row of diff off its 16-byte alignment (the scalar branch of the squared sum).  Rows 0-3
    reach the clamps: ui = 0 (x0 = 0), um = 0, both, and 0 < |um| < eps."""
    rng = np.random.default_rng(B * 11 + I + offset)
    w_tab = _schedule50()
    t = rng.integers(0, 50, B)
    t[: min(B, 5) // 2] = 0
    diffbuf = torch.full((B, ops.pad_to(I, 4) + 4), 1e30, device=DEV)     # 16-byte aligned rows
    diff_np = rng.standard_normal((B, I)).astype(np.float32) * 0.3
    diffbuf[:, offset:offset + I] = T(diff_np)
    diff = diffbuf[:, offset:offset + I]
    x0f = rng.standard_normal((B, 64)).astype(np.float32)
    umd = rng.standard_normal((B, 64)).astype(np.float32)
    ui = rng.standard_normal((B, 64)).astype(np.float32)
    ui[0] = 0.0                                  # an empty x0 row
    umd[1] = -x0f[1]                             # um = 0 exactly
    umd[2], ui[2] = -x0f[2], 0.0
    x0f[3], umd[3] = 0.0, rng.standard_normal(64) * 1e-10     # 0 < |um| < eps
    xfe = torch.full((B, 128), 1e30, device=DEV)
    xfe[:, :64], xfe[:, 64:] = T(x0f), T(ui)
    sw = 0.1
    loss = torch.full((B + 1,), float("nan"), dtype=torch.float64, device=DEV)
    mse, um, stats = f32_buf(B + 1), f32_buf(B + 1, 64), f32_buf(B + 1, 3)
    ops.diff_loss_fwd(diff, strided(umd, 64), xfe[:, :64], xfe[:, 64:], T(t), w_tab, sw, loss[:B], mse[:B], um[:B], stats[:B])
    torch.cuda.synchronize()
    assert torch.isnan(loss[B]) and bits(mse)[B] == NAN32_BITS
    assert_sentinel(um, B, 64)
    assert_sentinel(stats, B, 3)
    u = umd + x0f
    assert np.array_equal(bits(um[:B]), u.view(np.int32))
    u64, v64, d64 = u.astype(np.float64), ui.astype(np.float64), diff_np.astype(np.float64)
    mse64 = (d64 ** 2).sum(1) / I
    assert np.all(np.abs(mse[:B].cpu().numpy() - mse64) <= (I / 128 + 10) * 2 * U24 * mse64)
    st = stats[:B].cpu().numpy()
    dot, a, b = (u64 * v64).sum(1), np.linalg.norm(u64, axis=1), np.linalg.norm(v64, axis=1)
    assert np.all(np.abs(st[:, 0] - dot) <= 70 * U24 * (np.abs(u64 * v64)).sum(1))
    assert np.all(np.abs(st[:, 1] - a) <= 40 * U24 * a) and np.all(np.abs(st[:, 2] - b) <= 40 * U24 * b)
    ac, bc = np.maximum(a, 1e-8), np.maximum(b, 1e-8)
    cos = dot / (ac * bc)
    wt = f64(w_tab)[t]
    want = wt * mse64 + sw * (1.0 - cos)
    tol = wt * (I / 128 + 12) * 2 * U24 * mse64 + sw * 200 * U24 * (np.abs(u64 * v64).sum(1) / (ac * bc) + 1)
    assert np.all(np.abs(f64(loss[:B]) - want) <= tol)

    # backward
    g = rng.standard_normal(B) * 0.01
    g[min(B, 5) - 1] = 0.0                       # c = 0: dumc must be 0, not a division by zero
    cm = f32_buf(B + 1)
    d_hi, d_lo = bf16_buf(B + 1, 72), bf16_buf(B + 1, 72)
    ops.diff_loss_bwd(T(g), um[:B], xfe[:, 64:], stats[:B], T(t), w_tab, sw, I, cm[:B], d_hi[:B], d_lo[:B], None)
    torch.cuda.synchronize()
    assert_sentinel(d_hi, B, 64)
    assert_sentinel(d_lo, B, 64)
    c = cm.cpu().numpy()
    assert bits(cm)[B] == NAN32_BITS
    assert np.array_equal(c[:B].view(np.int32), (g * wt * 2.0 / I).astype(np.float32).view(np.int32))
    got = c[:B, None].astype(np.float64) * (f64(d_hi[:B, :64]) + f64(d_lo[:B, :64]))
    assert np.isfinite(got).all()
    gs = (g.astype(np.float32) * np.float32(sw)).astype(np.float64)[:, None]
    dcos, (t1, t2) = _dcos_du(u64, v64)
    want = -gs * dcos
    # fp32 norms, cosine and quotient dum / cm, then the 2^-17 of the split pair: relative to the larger term (|cos| <= 1
    # bounds the error of the cosine by the same scale)
    scale = np.abs(gs) * (np.abs(t1).max(1, keepdims=True) + t2.max(1, keepdims=True))
    assert np.all(np.abs(got - want) <= 3e-5 * scale + 1e-30)
    # torch's F.cosine_similarity gradient agrees except for 0 < |um| <= eps (row 3): it clamps the norm in place outside
    # autograd, so its backward keeps the -cos um / (eps |um|) term of the unclamped norm; the kernel differentiates
    # the clamped function, whose clamped norm is a constant
    uu = torch.from_numpy(u64).requires_grad_(True)
    torch.nn.functional.cosine_similarity(uu, torch.from_numpy(v64), dim=-1, eps=1e-8).sum().backward()
    tg = (-gs * uu.grad.numpy())
    keep = np.ones(B, dtype=bool)
    keep[3] = False
    assert np.all(np.abs(got - tg)[keep] <= 3e-5 * scale[keep] + 1e-30)
    # single-pass mode: no lo output; hi is the same
    d_hi2 = bf16_buf(B + 1, 64)
    ops.diff_loss_bwd(T(g), um[:B], xfe[:, 64:], stats[:B], T(t), w_tab, sw, I, cm[:B], d_hi2[:B], None, None)
    assert np.array_equal(bits(d_hi2[:B]), bits(d_hi[:B, :64]))


# ---------------------------------------------------------------------------------------------- hidden layer backward
@pytest.mark.parametrize("scaled", [True, False])
@pytest.mark.parametrize("H", [1, 7, 1003])
@pytest.mark.parametrize("B", BS)
def test_hidden_bwd(ops, B, H, scaled):
    """As the step calls it: h in fp32, with the row scale cm (top activation) and without (cm = NULL)."""
    rng = np.random.default_rng(B * 13 + H + scaled)
    z = rng.standard_normal((B, H)) * np.where(rng.random((B, H)) < 0.5, 6.0, 0.5)
    h = np.tanh(z).astype(np.float32)
    h.flat[:: 7] = np.float32(0.99995)            # |h| > 0.999: 1 - h^2 is as small as the bf16 rounding of h
    assert (np.abs(h) > 0.999).mean() >= 1 / 7
    dh = rng.standard_normal((B, H)).astype(np.float32)
    cm = (rng.standard_normal(B) * 1e-3).astype(np.float32) if scaled else None
    ld16, Bp = ops.pad_to(H, 64) + 8, ops.pad_to(B, 64)
    dz = f32_buf(B + 1, H + 5)
    dz_hi, dz_lo = bf16_buf(B + 1, ld16), bf16_buf(B + 1, ld16)
    dzt_hi, dzt_lo, hct_hi, hct_lo = (bf16_buf(H + 1, Bp) for _ in range(4))
    ops.hidden_bwd(strided(dh, 3), strided(h, 1), None, None, T(cm) if scaled else None, H, dz[:B, :H], dz_hi[:B],
                   dz_lo[:B], dzt_hi[:H], dzt_lo[:H], hct_hi[:H], hct_lo[:H])
    torch.cuda.synchronize()
    assert_sentinel(dz, B, H)
    assert_sentinel(dz_hi, B, H)
    assert_sentinel(dz_lo, B, H)
    for buf in (dzt_hi, dzt_lo, hct_hi, hct_lo):
        assert_sentinel(buf, H, Bp)
    s = cm.astype(np.float64)[:, None] if scaled else 1.0
    sdh = np.abs(s * dh.astype(np.float64))
    want = s * dh * (1.0 - h.astype(np.float64) ** 2)
    got = dz[:B, :H].cpu()
    # a few fp32 ulp of |s dh|: 1 - h h may or may not be fused into an FMA
    assert np.all(np.abs(got.double().numpy() - want) <= 4 * U24 * sdh + 1e-45)
    hi, lo = split(got)
    assert np.array_equal(bits(dz_hi[:B, :H]), bits(hi)) and np.array_equal(bits(dz_lo[:B, :H]), bits(lo))
    # the transposes: exact, with zeros in the batch columns [B, Bp)
    assert np.array_equal(bits(dzt_hi[:H, :B]), bits(hi).T) and np.array_equal(bits(dzt_lo[:H, :B]), bits(lo).T)
    hc = torch.from_numpy(cm[:, None] * h if scaled else h)
    chi, clo = split(hc)
    assert np.array_equal(bits(hct_hi[:H, :B]), bits(chi).T) and np.array_equal(bits(hct_lo[:H, :B]), bits(clo).T)
    for buf in (dzt_hi, dzt_lo, hct_hi, hct_lo):
        assert (bits(buf[:H, B:]) == 0).all()


# ---------------------------------------------------------------------------------------------- transpose_bf16
@pytest.mark.parametrize("with_lo", [True, False])
@pytest.mark.parametrize("C", [1, 7, 45, 1003])
@pytest.mark.parametrize("R", BS)
def test_transpose_bf16(ops, R, C, with_lo):
    rng = np.random.default_rng(R + C)
    src = torch.from_numpy(rng.standard_normal((R, C + 9)).astype(np.float32)).to(DEV)
    s_hi, s_lo = split(src)
    ld_dst = ops.pad_to(R, 64)
    d_hi, d_lo = bf16_buf(C + 1, ld_dst), bf16_buf(C + 1, ld_dst)
    ops.transpose_bf16(s_hi[:, :C], s_lo[:, :C] if with_lo else None, R, C, d_hi[:C], d_lo[:C] if with_lo else None)
    torch.cuda.synchronize()
    assert_sentinel(d_hi, C, ld_dst)
    assert np.array_equal(bits(d_hi[:C, :R]), bits(s_hi[:, :C]).T)
    assert (bits(d_hi[:C, R:]) == 0).all()
    if with_lo:
        assert_sentinel(d_lo, C, ld_dst)
        assert np.array_equal(bits(d_lo[:C, :R]), bits(s_lo[:, :C]).T)
        assert (bits(d_lo[:C, R:]) == 0).all()
    else:
        assert (bits(d_lo) == np.int16(SENT16)).all()


# ---------------------------------------------------------------------------------------------- colsum
@pytest.mark.parametrize("scaled", [True, False])
@pytest.mark.parametrize("R", [0, 1, 2, 3, 4, 5, 63, 300, 1025, 1026])
def test_colsum(ops, R, scaled):
    rng = np.random.default_rng(R * 2 + scaled)
    C = 1003
    x = rng.standard_normal((R, C)).astype(np.float32)
    sc = rng.standard_normal(R).astype(np.float32) if scaled else None
    xs = strided(x, 7) if R else torch.zeros((0, C + 7), device=DEV)[:, :C]      # an empty batch: no storage at all
    out = ops.colsum(xs, T(sc) if scaled else None)
    terms = (sc.astype(np.float64)[:, None] if scaled else 1.0) * x.astype(np.float64)
    tol = max(R, 1) * 2 * U24 * np.abs(terms).sum(0)
    got = out.cpu().numpy()
    assert np.all(np.abs(got - terms.sum(0)) <= tol)
    if R == 0:
        assert (bits(out) == 0).all()
    # rows added in a fixed order: two calls agree bit for bit
    assert np.array_equal(bits(ops.colsum(xs, T(sc) if scaled else None)), bits(out))


# ---------------------------------------------------------------------------------------------- atb_small
@pytest.mark.parametrize("R", [0, 1, 7, 9, 1025])
@pytest.mark.parametrize("m,n", [(1, 1), (10, 10), (64, 64), (10, 64), (64, 1)])
def test_atb_small(ops, R, m, n):
    """x is a column slice of a wider matrix (the step passes dtemb = dxa[:, I:I + d]); below 8 rows some of the 8 row
    slices are empty."""
    rng = np.random.default_rng(R + 100 * m + n)
    I = 1003
    wide = rng.standard_normal((R, I + m)).astype(np.float32)
    y = rng.standard_normal((R, n)).astype(np.float32)
    xw = torch.from_numpy(np.ascontiguousarray(wide)).to(DEV) if R else torch.zeros((0, I + m), device=DEV)
    x = xw[:, I:I + m]
    yd = strided(y, 2) if R else torch.zeros((0, n + 2), device=DEV)[:, :n]
    out = ops.atb_small(x, yd)
    x64, y64 = wide[:, I:].astype(np.float64), y.astype(np.float64)
    want = x64.T @ y64
    tol = (R + 16) * U24 * (np.abs(x64).T @ np.abs(y64))
    assert np.all(np.abs(out.cpu().numpy() - want) <= tol)
    assert np.array_equal(bits(ops.atb_small(x, yd)), bits(out))


# ---------------------------------------------------------------------------------------------- the whole step
def _model(denoise_dim, I, d, precision, seed):
    from diffmm_b200.Conf import Config
    from diffmm_b200.Model import Denoise, GaussianDiffusion
    cfg = Config()
    cfg.base.denoise_dim, cfg.base.precision, cfg.base.d_emb_size = denoise_dim, precision, d
    cfg.data.item_num = I
    cfg.hyper.steps, cfg.hyper.noise_scale = 50, 0.5
    torch.manual_seed(seed)
    gd = GaussianDiffusion(cfg).to(DEV)
    out_dims = ast.literal_eval(denoise_dim) + [I]
    den = Denoise(out_dims[::-1], out_dims, cfg).to(DEV)
    return cfg, gd, den


def _saturate(cfg, gd, den, inputs, med=4.0):
    """Scales every tanh layer, bottom up, until the median |pre-activation| on `inputs` is `med`: then most |h| > 0.99
    (|z| > 2.65), where tanh' = 1 - h^2 needs h beyond bf16, without driving whole layers to |h| = 1."""
    layers = list(den.in_layers) + list(den.out_layers)[:-1]
    for k, layer in enumerate(layers):
        z = _training_losses64(cfg, gd, den, *inputs)[3][k]
        with torch.no_grad():
            s = med / float(z.abs().median())
            layer.weight.mul_(s)
            layer.bias.mul_(s)


def _training_losses64(cfg, gd, den, x0, i_embs, feat, t, noise):
    """Model.py:385-428 with Denoise.forward (Model.py:183-220) in float64 autograd, odd time embeddings zero-padded;
    returns the per-row loss, the float64 leaf parameters, the hidden activations and their pre-activations."""
    P = {n: p.detach().double().requires_grad_(True) for n, p in den.named_parameters()}
    L = len(den.in_layers)
    x0d, f = x0.double(), feat.double()
    x_t = gd.sqrt_alphas_cumprod[t].float().double()[:, None] * x0d + \
        gd.sqrt_one_minus_alphas_cumprod[t].float().double()[:, None] * noise.double()
    d = den.time_emb_dim
    half = d // 2
    freqs = torch.exp(-math.log(10000.0) * torch.arange(half, device=DEV, dtype=torch.float64) / half)
    temp = t[:, None].double() * freqs[None]
    e = torch.cat([torch.cos(temp), torch.sin(temp)] + ([torch.zeros_like(temp[:, :1])] if d % 2 else []), -1)
    temb = e @ P["emb_layer.weight"].t() + P["emb_layer.bias"]
    proj = x_t @ f
    gate = torch.sigmoid(proj @ P["gate_layer.weight"].t() + P["gate_layer.bias"])
    h = torch.cat([x_t + (proj * gate) @ f.t(), temb], -1)
    acts, zs = [], []
    for k in range(L):
        zs.append(h @ P[f"in_layers.{k}.weight"].t() + P[f"in_layers.{k}.bias"])
        h = torch.tanh(zs[-1])
        acts.append(h)
    for k in range(L):
        h = h @ P[f"out_layers.{k}.weight"].t() + P[f"out_layers.{k}.bias"]
        if k != L - 1:
            zs.append(h)
            h = torch.tanh(h)
            acts.append(h)
    mse = ((h - x0d) ** 2).mean(-1)
    ac = gd.alphas_cumprod
    snr = lambda tt: ac[tt] / (1 - ac[tt] + 1e-8)  # noqa: E731
    w = torch.where(t == 0, 1.0, snr(torch.clamp(t - 1, min=0)) - snr(t))
    um, ui = h @ f, x0d @ i_embs.double()
    sim = 1 - torch.nn.functional.cosine_similarity(um, ui, dim=-1)
    reg = (i_embs.double() ** 2).sum() * cfg.train.reg
    return w * mse + sim * cfg.hyper.sim_weight + reg * cfg.train.reg, P, acts, zs


def _rel(got, want):
    return float((got.double() - want.double()).abs().max() / (want.double().abs().max() + 1e-30))


STEP_CASES = [(B, d, dims, prec) for prec in ("bf16x3", "bf16") for dims in ("[136]", "[96, 160]")
              for B in (1, 5, 63) for d in (2, 9, 64)]


# The saturated model runs in bf16x3 only: single-pass bf16 computes tanh with tanh.approx.f32 (absolute error ~5e-4
# near |h| = 1), so there tanh' of a saturated unit is mostly rounding noise, on the fused and the per-op path alike.
@pytest.mark.parametrize("B,d,denoise_dim,precision,saturate",
                         [c + (False,) for c in STEP_CASES] + [(63, 9, "[96, 160]", "bf16x3", True),
                                                               (5, 10, "[136]", "bf16x3", True)])
def test_fused_step_small_batches_and_time_embeddings(B, d, denoise_dim, precision, saturate, monkeypatch):
    """GaussianDiffusion.training_losses on the fused step (B < 64: every weight-gradient contraction has K = B < 64)
    against float64 autograd: the loss row by row, every gradient, and dW1's item and time-embedding columns scored
    apart (their scales differ).  A 50-step schedule with t = 0 present; every fourth x0 row is empty."""
    from diffmm_b200 import train_step
    I = 1003
    cfg, gd, den = _model(denoise_dim, I, d, precision, seed=B + d)
    rng = np.random.default_rng(B * 3 + d)
    x0n = (rng.random((B, I)) < 0.01).astype(np.float32)
    x0n[1::4] = 0.0
    x0 = T(x0n)
    feat = T(rng.standard_normal((I, 64)).astype(np.float32) * 0.1)
    i_embs = T(rng.standard_normal((I, 64)).astype(np.float32) * 0.1)
    tn = rng.integers(0, 50, B)
    tn[0] = 0
    t = T(tn)
    noise = T(rng.standard_normal((B, I)).astype(np.float32))
    if saturate:
        _saturate(cfg, gd, den, (x0, i_embs, feat, t, noise))
    calls = []
    orig = train_step.denoise_loss
    monkeypatch.setattr(train_step, "denoise_loss", lambda *a, **k: (calls.append(1), orig(*a, **k))[1])
    monkeypatch.setenv("DIFFMM_FUSED_TRAIN", "1")
    den.zero_grad(set_to_none=True)
    losses = gd.training_losses(den, x0, i_embs, feat, timesteps=t, noise=noise)
    assert len(calls) == 1, "the fused step was not selected"
    losses.mean().backward()
    grads = {n: p.grad.detach().clone() for n, p in den.named_parameters()}
    assert all(torch.isfinite(g).all() for g in grads.values())
    want, P, acts, _ = _training_losses64(cfg, gd, den, x0, i_embs, feat, t, noise)
    if saturate:
        assert all(float((h.abs() > 0.99).double().mean()) > 0.5 for h in acts)
    want.mean().backward()
    got_l, want_l = losses.detach().double(), want.detach()
    if precision == "bf16x3":
        assert float(((got_l - want_l).abs() / want_l.abs()).max()) <= 2e-4
        tol_g = 1e-3
    else:
        assert _rel(got_l, want_l) <= 1e-1
        tol_g = 1e-1
    for k, p in P.items():
        g, w = grads[k], p.grad
        if k == "in_layers.0.weight":
            parts = {"item columns": (g[:, :I], w[:, :I]), "time-embedding columns": (g[:, I:], w[:, I:])}
        else:
            parts = {"": (g, w)}
        for part, (gg, ww) in parts.items():
            assert _rel(gg, ww) <= tol_g, (k, part, _rel(gg, ww))
