"""The two kernels behind recommend.score_pairs / recommend.rank_candidates, through ops (the C ABI), at ragged sizes,
with leading dimensions wider than the data, aligned (float4) and unaligned (scalar) rows, and every output
sentinel-filled first (nothing outside [rows, n] / [P] may change):
  * exactness: on embeddings a + b 2^-9 (every product and partial sum exact in fp32) both kernels equal the float64
    evaluation of the documented bf16x3 / bf16 formulas bit for bit, and rank_candidates over every item equals
    score_topn (many exact ties: the item-ascending tie order against the library's top-k);
  * random normal embeddings: scores within a derived bound of float64, rankings equal to a numpy lexsort of the kernel's
    own score_pairs scores, and rank_candidates' scores equal to score_pairs' bit for bit;
  * edge cases: duplicates, -1 / out-of-range padding, empty rows, fewer distinct candidates than n, and scores of
    +-0, +-inf and NaN from embeddings that hold them."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SENT = np.float32(7.25)
ISENT = -7


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _order_key(x):
    """The top-k kernels' order-preserving key: -0.0 ties with +0.0, NaN by its bits."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).copy()
    u[u == 0x80000000] = 0
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def _split(x):
    """hi = bf16_rn(x), lo = bf16_rn(x - hi) (fp32 difference), as float64."""
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    hi = t.bfloat16().float()
    lo = (t - hi).bfloat16().float()
    return hi.double().numpy(), lo.double().numpy()


def _mats(u, it, x3):
    """float64 [U, I] for every (user row, item row) pair: the documented formula, sum over d of hi_u hi_i
    (+ hi_u lo_i + lo_u hi_i), and the sum of the |terms|.  Exact on the exact inputs (multiples of 2^-9 far inside
    float64's 53 bits); within float64 rounding otherwise."""
    uh, ul = _split(u)
    ih, il = _split(it)
    if not x3:
        return uh @ ih.T, np.abs(uh) @ np.abs(ih).T
    return (uh @ ih.T + uh @ il.T + ul @ ih.T,
            np.abs(uh) @ np.abs(ih).T + np.abs(uh) @ np.abs(il).T + np.abs(ul) @ np.abs(ih).T)


def _embed(rows, D, ld, seed, kind, aligned=True):
    """fp32 [rows, D] inside a sentinel-filled buffer of leading dimension ld; aligned=False starts the view one float in
    (rows no longer 16-byte aligned: the scalar-load path)."""
    rng = np.random.default_rng(seed)
    if kind == "exact":
        a = rng.integers(-3, 4, (rows, D))
        b = np.where(a == 0, 0, rng.integers(-1, 2, (rows, D)))       # x = 0 stays 0: every term a multiple of 2^-9
        x = (a + b * 2.0 ** -9).astype(np.float32)
    else:
        x = rng.standard_normal((rows, D)).astype(np.float32)
    off = 0 if aligned else 1
    buf = np.full((max(rows, 1), ld + off), SENT, dtype=np.float32)
    buf[:rows, off:off + D] = x
    dev = T(buf)
    return x, dev[:rows, off:off + D]


def _exact_bits(abs_sum):
    """Significant bits the exact-case sums can need: every term is a multiple of 2^-9 and every partial sum is bounded
    by the sum of |terms|."""
    return int(np.ceil(np.log2(max(float(abs_sum.max()), 1.0) * 2.0 ** 9)))


def _f32(x):
    """float64 -> fp32 with a zero as +0.0 (the kernels' zero)."""
    return (np.asarray(x) + 0.0).astype(np.float32)


# ------------------------------------------------------------------------------------------------ score_pairs
@pytest.mark.parametrize("x3", [True, False])
@pytest.mark.parametrize("D", [1, 7, 64, 200])
@pytest.mark.parametrize("P", [0, 1, 33, 1_000_000])
@pytest.mark.parametrize("aligned", [True, False])
def test_score_pairs_exact(ops, P, D, x3, aligned):
    U, I = 37, 1001
    u, ud = _embed(U, D, D + 5 if not aligned else ((D + 3) // 4) * 4 + 4, seed=D + 1, kind="exact", aligned=aligned)
    it, idev = _embed(I, D, D + 9 if not aligned else ((D + 3) // 4) * 4 + 8, seed=D + 2, kind="exact", aligned=aligned)
    rng = np.random.default_rng(P + D)
    pu = rng.integers(0, U, P).astype(np.int64)
    pi = rng.integers(0, I, P).astype(np.int32)
    out = torch.full((P + 3,), float(SENT), device=DEV)
    ops.score_pairs(ud, idev, T(pu), T(pi), x3, out[:P])
    got = out.cpu().numpy()
    assert np.all(got[P:] == SENT)
    if P == 0:
        return
    f, a = _mats(u, it, x3)
    bits = _exact_bits(a)
    assert bits <= (20 if D <= 64 else 22), bits             # exact in fp32 (24 significant bits)
    want = _f32(f[pu, pi])
    assert np.array_equal(got[:P].view(np.int32), want.view(np.int32))


@pytest.mark.parametrize("D", [1, 7, 64, 200])
def test_score_pairs_random_within_derived_bound(ops, D):
    """Against float64:
      * the documented formula: n fp32 additions of exact products (n = 3D or D), lane sums then a 3-level butterfly:
        |err| <= (n + 8) 2^-24 sum|terms|;
      * the exact product u . i (bf16x3): x = hi + lo + e with |e| <= 2^-16 |x| (two roundings to 8 significant bits),
        so u_d i_d - (terms) = lo_u lo_i + e_u (hi_i + lo_i) + e_i (hi_u + lo_u) + e_u e_i, at most 3 2^-16 (1 + 2^-6)
        |u_d i_d|, and sum|terms| <= (1 + 2^-5) sum|u_d i_d|: |err| <= (3 2^-16 (1 + 2^-6) + (3D + 8) 2^-24 (1 + 2^-5))
        sum|u_d i_d|;
      * the exact product (bf16): |u_d i_d - hi_u hi_i| <= 2^-7 (1 + 2^-7) |u_d i_d| and |hi_u hi_i| <= (1 + 2^-6)
        |u_d i_d|: |err| <= (2^-7 (1 + 2^-7) + (D + 8) 2^-24 (1 + 2^-6)) sum|u_d i_d|."""
    U, I, P = 300, 5000, 200_000
    u, ud = _embed(U, D, D + 3, seed=10 + D, kind="normal")
    it, idev = _embed(I, D, D + 1, seed=20 + D, kind="normal")
    rng = np.random.default_rng(D)
    pu = rng.integers(0, U, P).astype(np.int64)
    pi = rng.integers(0, I, P).astype(np.int32)
    u64, i64 = u.astype(np.float64), it.astype(np.float64)
    exact = (u64 @ i64.T)[pu, pi]
    mag = (np.abs(u64) @ np.abs(i64).T)[pu, pi]
    for x3 in (True, False):
        out = torch.empty(P, device=DEV)
        ops.score_pairs(ud, idev, T(pu), T(pi), x3, out)
        got = out.cpu().numpy().astype(np.float64)
        f, a = _mats(u, it, x3)
        n = 3 * D if x3 else D
        assert np.all(np.abs(got - f[pu, pi]) <= (n + 8) * 2.0 ** -24 * (1 + 2.0 ** -20) * a[pu, pi])
        if x3:
            bound = (3 * 2.0 ** -16 * (1 + 2.0 ** -6) + (3 * D + 8) * 2.0 ** -24 * (1 + 2.0 ** -5)) * mag
        else:
            bound = (2.0 ** -7 * (1 + 2.0 ** -7) + (D + 8) * 2.0 ** -24 * (1 + 2.0 ** -6)) * mag
        assert np.all(np.abs(got - exact) <= bound)


def test_score_pairs_aligned_and_unaligned_rows_agree(ops):
    """The float4 and the scalar load paths add in the same order: the same bits."""
    for D in (1, 7, 64, 200):
        U, I, P = 50, 700, 20_000
        _, ua = _embed(U, D, ((D + 3) // 4) * 4, seed=D, kind="normal", aligned=True)
        _, ia = _embed(I, D, ((D + 3) // 4) * 4 + 4, seed=D + 7, kind="normal", aligned=True)
        ub, ib = ua.clone(), torch.empty((I, D + 3), device=DEV)[:, 1:D + 1]
        ib.copy_(ia)
        rng = np.random.default_rng(D)
        pu, pi = T(rng.integers(0, U, P).astype(np.int64)), T(rng.integers(0, I, P).astype(np.int32))
        for x3 in (True, False):
            a, b = torch.empty(P, device=DEV), torch.empty(P, device=DEV)
            ops.score_pairs(ua, ia, pu, pi, x3, a)
            ops.score_pairs(ub, ib, pu, pi, x3, b)
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (D, x3)


def test_score_pairs_out_of_range_is_nan(ops):
    D = 64
    u, ud = _embed(5, D, D, seed=0, kind="normal")
    it, idev = _embed(9, D, D, seed=1, kind="normal")
    pu = np.array([0, -1, 5, 4, 2, 1 << 40], dtype=np.int64)
    pi = np.array([0, 3, 3, 9, -1, 8], dtype=np.int32)
    out = torch.full((6,), float(SENT), device=DEV)
    ops.score_pairs(ud, idev, T(pu), T(pi), True, out)
    got = out.cpu().numpy()
    assert not np.isnan(got[0]) and np.all(np.isnan(got[1:]))


def test_score_pairs_zero_pairs_and_rejects(ops):
    from diffmm_b200 import _lib
    e = torch.zeros((0, 64), device=DEV)
    lib = _lib.load()
    ctx = _lib.ctx(0)
    # zero pairs: a no-op with NULL device pointers
    assert lib.dmm_score_pairs(ctx, None, 64, 0, None, 64, 0, 64, None, None, 0, 1, None, None) == 0
    z = torch.zeros(0, dtype=torch.int64, device=DEV)
    ops.score_pairs(e, e, z, z.int(), True, torch.zeros(0, device=DEV))
    for D, ld, x3 in ((0, 64, 1), (1025, 2048, 1), (64, 63, 1), (64, 64, 2)):
        assert lib.dmm_score_pairs(ctx, None, ld, 1, None, ld, 1, D, None, None, 1, x3, None, None) != 0


# ------------------------------------------------------------------------------------------------ rank_candidates
def _reference_ranking(scores_of, cand, n, n_items):
    """Per row: the distinct valid candidates ranked by (order key desc, item asc), first n, padded with (-1, -inf).
    scores_of(row, items) -> fp32 scores."""
    B = cand.shape[0]
    items = np.full((B, n), -1, dtype=np.int32)
    scores = np.full((B, n), -np.inf, dtype=np.float32)
    for r in range(B):
        c = np.unique(cand[r][(cand[r] >= 0) & (cand[r] < n_items)])
        if c.size == 0:
            continue
        s = scores_of(r, c)
        order = np.lexsort((c, -_order_key(s).astype(np.int64)))[:n]
        items[r, :order.size] = c[order]
        scores[r, :order.size] = s[order]
    return items, scores


def _run_rank(ops, ud, idev, cand, n, x3):
    """rank_candidates into sentinel-filled buffers (wider than [B, n]); returns (items, scores) [B, n] after checking
    that nothing outside was written."""
    B = cand.shape[0]
    ib = torch.full((B + 2, n + 3), ISENT, dtype=torch.int32, device=DEV)
    sb = torch.full((B + 2, n + 5), float(SENT), device=DEV)
    cbuf = np.full((B, cand.shape[1] + 3), 12345678, dtype=np.int32)    # a wider ld_c; the pad columns are out of range
    cbuf[:, :cand.shape[1]] = cand
    ops.rank_candidates(ud, idev, T(cbuf)[:, :cand.shape[1]], n, x3, ib[:B, :n], sb[:B, :n])
    gi, gs = ib.cpu().numpy(), sb.cpu().numpy()
    assert np.all(gi[B:] == ISENT) and np.all(gi[:, n:] == ISENT)
    assert np.all(gs[B:] == SENT) and np.all(gs[:, n:] == SENT)
    return gi[:B, :n], gs[:B, :n]


def _pair_scores(ops, ud, idev, rows, items, x3):
    out = torch.empty(len(rows), device=DEV)
    ops.score_pairs(ud, idev, T(np.asarray(rows, dtype=np.int64)), T(np.asarray(items, dtype=np.int32)), x3, out)
    return out.cpu().numpy()


def _candidates(B, C, I, seed, pad=True):
    """Random candidate rows with duplicates, -1 padding, out-of-range ids, an all-empty row and short rows."""
    rng = np.random.default_rng(seed)
    cand = rng.integers(0, I, (B, C)).astype(np.int32)
    if pad and C > 1:
        for r in range(B):
            kind = r % 6
            if kind == 1:
                cand[r, rng.random(C) < 0.3] = -1                       # -1 padding
            elif kind == 2:
                cand[r, :] = cand[r, 0]                                 # one item C times
            elif kind == 3:
                cand[r, :] = -1                                         # entirely empty
            elif kind == 4:
                cand[r, C // 2:] = rng.choice([-1, I, I + 77, -5], C - C // 2)   # padding and out-of-range ids
            elif kind == 5:
                cand[r] = rng.integers(0, min(I, 3), C)                 # fewer distinct candidates than n
    return cand


@pytest.mark.parametrize("C", [1, 2, 31, 101, 1000, 4096])
@pytest.mark.parametrize("nk", ["1", "10", "C"])
@pytest.mark.parametrize("D", [7, 64])
def test_rank_candidates_random(ops, C, nk, D):
    n = {"1": 1, "10": 10, "C": min(C, 1024)}[nk]
    if n > C:
        pytest.skip("n > C")
    B, U, I = 37, 41, 5003
    _, ud = _embed(U, D, D + 3, seed=C + D, kind="normal", aligned=False)
    _, idev = _embed(I, D, ((D + 3) // 4) * 4 + 4, seed=C + D + 1, kind="normal")
    urows = ud[:B]
    cand = _candidates(B, C, I, seed=C * 3 + n)
    uc, ic = urows.contiguous(), idev.contiguous()      # the reference scores through the other load path
    for x3 in (True, False):
        gi, gs = _run_rank(ops, urows, idev, cand, n, x3)
        wi, ws = _reference_ranking(lambda r, c: _pair_scores(ops, uc, ic, np.full(c.size, r), c, x3), cand, n, I)
        assert np.array_equal(gi, wi), x3
        assert np.array_equal(gs.view(np.int32), ws.view(np.int32)), x3
    if C > 1:
        assert np.all(gi[3] == -1) and np.all(np.isneginf(gs[3]))       # the empty row


@pytest.mark.parametrize("D", [1, 7, 64, 200])
@pytest.mark.parametrize("x3", [True, False])
def test_rank_candidates_exact_formula(ops, D, x3):
    """Exact inputs: the emitted scores are the float64 formula, bit for bit."""
    B, I, C, n = 29, 800, 300, 64
    u, ud = _embed(B, D, D + 2, seed=D, kind="exact", aligned=False)
    it, idev = _embed(I, D, D + 6, seed=D + 3, kind="exact", aligned=False)
    f, a = _mats(u, it, x3)
    assert _exact_bits(a) <= 22
    cand = _candidates(B, C, I, seed=D)
    gi, gs = _run_rank(ops, ud, idev, cand, n, x3)
    wi, ws = _reference_ranking(lambda r, c: _f32(f[r, c]), cand, n, I)
    assert np.array_equal(gi, wi)
    assert np.array_equal(gs.view(np.int32), ws.view(np.int32))


@pytest.mark.parametrize("I,n,D", [(1000, 10, 64), (1000, 1000, 64), (4096, 100, 7), (257, 257, 200), (33, 5, 1)])
@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_rank_candidates_every_item_equals_score_topn(I, n, D, precision):
    """Every item a candidate (in a different order per row): the same items and score bits as score_topn, whose
    contraction is exact on these inputs too.  Scores of small integers (+ 2^-9) tie everywhere, so this pins the tie
    order (item ascending) against the library's top-k."""
    from diffmm_b200 import recommend
    B = 40
    u, ud = _embed(B, D, D, seed=I + D, kind="exact")
    it, idev = _embed(I, D, D, seed=I + D + 1, kind="exact")
    rng = np.random.default_rng(I)
    cand = np.stack([rng.permutation(I) for _ in range(B)]).astype(np.int32)
    gi, gs = recommend.rank_candidates(ud, idev, cand, n, precision=precision)
    wi, ws = recommend.score_topn(ud.contiguous(), idev.contiguous(), n, precision=precision)
    assert torch.equal(gi, wi)
    assert torch.equal(gs.view(torch.int32), ws.view(torch.int32))
    s = gs.cpu().numpy()
    assert (s[:, 1:] == s[:, :-1]).sum() > 0 or n == 1 or I < 64      # ties were there to break


def test_rank_candidates_special_scores(ops):
    """Scores of +-0, +-inf and NaN from embeddings that hold them (zero rows, -0.0 entries, 1e30 entries, NaN entries):
    ranked in the library's total order, every real candidate listed with its score (-inf included)."""
    D, I = 8, 12
    it = np.zeros((I, D), dtype=np.float32)
    it[0] = 1e30                     # x user 1e30 -> +inf
    it[1] = -1e30                    # -> -inf
    it[2, 0] = np.nan                # -> NaN
    it[3, :4], it[3, 4:] = 1e30, -1e30   # inf - inf -> NaN
    it[4] = -0.0                     # -> +0 (the sum starts at +0.0)
    it[5] = 0.0
    it[6] = 1.0
    it[7] = -1.0
    it[8] = -1e-30                   # underflowing products: a zero score, returned as +0.0
    it[9] = 2.0
    it[10] = -2.0
    it[11] = 1e-3
    us = np.stack([np.full(D, 1e30, np.float32), np.full(D, -0.0, np.float32), np.full(D, 1e-30, np.float32),
                   np.ones(D, np.float32)])
    B = us.shape[0]
    ud, idev = T(us), T(it)
    cand = np.stack([np.r_[np.arange(I), [1, 1, -1, 3]] for _ in range(B)]).astype(np.int32)
    for x3 in (True, False):
        s = _pair_scores(ops, ud, idev, np.repeat(np.arange(B), I), np.tile(np.arange(I), B), x3).reshape(B, I)
        assert np.isposinf(s[0, 0]) and np.isneginf(s[0, 1]) and np.isnan(s[0, 2]) and np.isnan(s[0, 3])
        assert np.all(s[1].view(np.uint32)[~np.isnan(s[1])] == 0) and np.all(s[2].view(np.uint32)[[4, 5, 8]] == 0)
        gi, gs = _run_rank(ops, ud, idev, cand, I, x3)
        wi, ws = _reference_ranking(lambda r, c: s[r, c], cand, I, I)
        assert np.array_equal(gi, wi)
        assert np.array_equal(gs.view(np.int32), ws.view(np.int32))
        assert 1 in gi[0].tolist() and np.isneginf(gs[0, gi[0].tolist().index(1)])   # -inf candidate listed


def test_rank_candidates_many_rows(ops):
    B, I, D, C, n = 20_000, 7050, 64, 101, 10
    _, ud = _embed(B, D, D, seed=1, kind="normal")
    _, idev = _embed(I, D, D, seed=2, kind="normal")
    rng = np.random.default_rng(3)
    cand = rng.integers(-1, I, (B, C)).astype(np.int32)
    gi, gs = _run_rank(ops, ud, idev, cand, n, True)
    ok = cand >= 0
    s = np.full((B, C), np.nan, dtype=np.float32)
    s[ok] = _pair_scores(ops, ud, idev, np.nonzero(ok)[0], cand[ok], True)
    for r in range(0, B, 97):
        c, first = np.unique(cand[r][ok[r]], return_index=True)
        sr = s[r][ok[r]][first]
        o = np.lexsort((c, -_order_key(sr).astype(np.int64)))[:n]
        assert np.array_equal(gi[r], c[o]) and np.array_equal(gs[r].view(np.int32), sr[o].view(np.int32)), r
    assert np.all(np.diff(_order_key(gs).astype(np.int64), axis=1) <= 0)


def test_rank_candidates_zero_rows_and_rejects(ops):
    from diffmm_b200 import _lib
    lib = _lib.load()
    ctx = _lib.ctx(0)
    assert lib.dmm_rank_candidates(ctx, None, 64, None, 64, 10, 64, None, 5, 0, 5, 5, 1, None, 5, None, 5, None) == 0
    bad = [(0, 1), (4097, 10), (5, 0), (5, 6), (2000, 1025)]            # (C, N)
    for C, N in bad:
        rc = lib.dmm_rank_candidates(ctx, None, 64, None, 64, 10, 64, None, max(C, 1), 0, C, N, 1, None, max(N, 1), None,
                                     max(N, 1), None)
        assert rc != 0, (C, N)
    assert lib.dmm_rank_candidates(ctx, None, 64, None, 64, 10, 1025, None, 5, 0, 5, 5, 1, None, 5, None, 5, None) != 0
