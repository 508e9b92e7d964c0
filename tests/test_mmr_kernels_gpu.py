"""dmm_mmr_rerank through ops.mmr_rerank (the C ABI), at ragged sizes, with leading dimensions wider than the data and
every output sentinel-filled first (nothing outside [rows, N] may change):
  (a) items and relevance bit-identical to a numpy float32 restatement of the arithmetic include/diffmm_b200.h documents
      (sim in four interleaved partial sums, m by fmax, obj = fl(fl(lam rel) - fl(mu m)), ties by relevance then item);
  (b) lam = 1 is the relevance ranking (relevance descending, item ascending) bit for bit;
  (c) on random inputs, every pick along the kernel's own path is a float64 arg-max of obj within a bound derived from
      that order of operations;
  (d) constructed cases with a known answer: orthonormal one-hot vectors, and clusters of identical vectors whose
      first picks lam = 0.5 must spread over the clusters.
Rows hold empty slots (-1), out-of-range ids, duplicates with differing relevance, and rows with no valid candidate."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SENT = np.float32(7.25)
ISENT = -7
U = 2.0 ** -24


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
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32).astype(np.int64)


def _distinct(vec_rows, cand, rel):
    """The row's distinct valid candidates in the kernel's candidate order (relevance desc, item asc): (items, rel)."""
    seen, items, rels = set(), [], []
    for c, it in enumerate(cand):
        if 0 <= it < vec_rows and int(it) not in seen:
            seen.add(int(it))
            items.append(int(it))
            rels.append(rel[c])
    items = np.array(items, dtype=np.int64)
    rels = np.array(rels, dtype=np.float32)
    o = np.lexsort((items, -_order_key(rels)))
    return items[o], rels[o]


def _sim32(V):
    """sim(j, k) for every pair of rows of V (float32 [n, D]) in the documented order: s_q = +0.0 (q = 0..3), for d
    ascending s_{d mod 4} = fl(s_{d mod 4} + fl(v_j[d] v_k[d])), sim = fl(fl(s_0 + s_1) + fl(s_2 + s_3))."""
    n, D = V.shape
    s = np.zeros((4, n, n), dtype=np.float32)
    for d in range(D):
        s[d % 4] = s[d % 4] + V[:, d][:, None] * V[:, d][None, :]
    return (s[0] + s[1]) + (s[2] + s[3])


def mmr_ref(vec, cand, rel, N, lam):
    """numpy float32 restatement of dmm_mmr_rerank for one row: (items int64 [N], relevance fp32 [N])."""
    items, rels = _distinct(vec.shape[0], cand, rel)
    nv = items.size
    out_i = np.full(N, -1, dtype=np.int64)
    out_r = np.full(N, -np.inf, dtype=np.float32)
    if nv == 0:
        return out_i, out_r
    lam = np.float32(lam)
    mu = np.float32(1) - lam
    S = _sim32(vec[items].astype(np.float32))
    lr = lam * rels
    m = np.full(nv, -np.inf, dtype=np.float32)
    picked = np.zeros(nv, dtype=bool)
    for s in range(min(N, nv)):
        obj = lr if s == 0 else lr - mu * m
        key = np.where(picked, -1, _order_key(obj))
        p = int(np.argmax(key))                      # first maximum: the smallest j, i.e. larger relevance, then item
        out_i[s], out_r[s] = items[p], rels[p]
        picked[p] = True
        m = np.fmax(m, S[:, p])
    return out_i, out_r


def _run(ops, vec, cand, rel, N, lam, ld_extra=(0, 0, 0, 0, 0)):
    """ops.mmr_rerank with every operand inside a wider buffer and sentinel-filled outputs; returns (items, rel) [B, N]
    after checking that nothing outside [B, N] changed."""
    B, C = cand.shape
    I, D = vec.shape
    ev, ec, er, ei, eo = ld_extra
    vb = np.full((I, D + ev), SENT, dtype=np.float32)
    vb[:, :D] = vec
    cb = np.full((B, C + ec), 12345, dtype=np.int32)
    cb[:, :C] = cand
    rb = np.full((B, C + er), SENT, dtype=np.float32)
    rb[:, :C] = rel
    ib = torch.full((B + 1, N + ei), ISENT, dtype=torch.int32, device=DEV)
    ob = torch.full((B + 1, N + eo), float(SENT), dtype=torch.float32, device=DEV)
    ops.mmr_rerank(T(vb)[:, :D], T(cb)[:, :C], T(rb)[:, :C], N, lam, ib[:B, :N], ob[:B, :N])
    ib, ob = ib.cpu().numpy(), ob.cpu().numpy()
    assert np.all(ib[B] == ISENT) and np.all(ib[:, N:] == ISENT)
    assert np.all(ob[B] == SENT) and np.all(ob[:, N:] == SENT)
    return ib[:B, :N].astype(np.int64), ob[:B, :N]


def _rows(rng, B, C, I, kind="normal"):
    """Candidate rows with empty slots, out-of-range ids and duplicates (differing relevance); row 1 has no valid
    candidate.  Relevance: normal, or small integers (many exact ties)."""
    cand = rng.integers(0, I, (B, C)).astype(np.int32)
    mask = rng.random((B, C))
    cand[mask < 0.08] = -1
    cand[(mask >= 0.08) & (mask < 0.12)] = I + 3                 # out of range
    if C > 2:
        dup = rng.random((B, C)) < 0.1
        cand[:, 1:][dup[:, 1:]] = cand[:, :-1][dup[:, 1:]]       # repeats of the slot before
    if B > 1:
        cand[1] = np.where(rng.random(C) < 0.5, -1, I + 7)
    if kind == "int":
        rel = rng.integers(-3, 4, (B, C)).astype(np.float32)
    else:
        rel = rng.standard_normal((B, C)).astype(np.float32)
    rel[cand < 0] = np.nan                                        # never read at an empty slot
    return cand, rel


def _unit(rng, I, D):
    v = rng.standard_normal((I, D)).astype(np.float32)
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


SHAPES = [(1, 1), (2, 3), (31, 64), (32, 128), (33, 256), (255, 64), (255, 128), (512, 64), (1024, 1), (1024, 3),
          (1024, 32), (128, 256), (33, 1), (2, 256)]


@pytest.mark.parametrize("C,D", SHAPES)
@pytest.mark.parametrize("lam", [0.0, 0.3, 0.5, 1.0])
def test_mmr_bit_exact_restatement(ops, C, D, lam):
    rng = np.random.default_rng(C * 1000 + D + int(lam * 10))
    B, I = 6, max(2 * C, 8)
    vec = _unit(rng, I, D)
    cand, rel = _rows(rng, B, C, I, kind="int" if C % 2 else "normal")
    for N in sorted({1, C}):
        gi, gr = _run(ops, vec, cand, rel, N, lam, ld_extra=(3, 5, 1, 2, 7))
        for b in range(B):
            wi, wr = mmr_ref(vec, cand[b], rel[b], N, lam)
            assert np.array_equal(gi[b], wi), (b, N)
            assert np.array_equal(gr[b].view(np.int32), wr.view(np.int32)), (b, N)
        assert np.all(gi[1] == -1) and np.all(np.isneginf(gr[1]))


@pytest.mark.parametrize("C,D", [(33, 64), (512, 64), (1024, 8)])
def test_mmr_lam1_is_relevance_ranking(ops, C, D):
    rng = np.random.default_rng(C + D)
    B, I = 8, 3 * C
    vec = rng.standard_normal((I, D)).astype(np.float32)                  # not unit: sims of any size
    cand, rel = _rows(rng, B, C, I, kind="int")
    gi, gr = _run(ops, vec, cand, rel, C, 1.0)
    for b in range(B):
        items, rels = _distinct(I, cand[b], rel[b])
        wi = np.full(C, -1, dtype=np.int64)
        wr = np.full(C, -np.inf, dtype=np.float32)
        wi[:items.size], wr[:items.size] = items, rels
        assert np.array_equal(gi[b], wi), b
        assert np.array_equal(gr[b].view(np.int32), wr.view(np.int32)), b


@pytest.mark.parametrize("C,D,lam", [(100, 64, 0.5), (200, 64, 0.3), (512, 64, 0.7), (64, 256, 0.5), (1024, 16, 0.5)])
def test_mmr_picks_are_float64_argmax(ops, C, D, lam):
    """Along the kernel's picks, each pick's float64 obj is within 2 x the bound of the float64 maximum.  Bound of
    |obj32 - obj64| for candidate j: sim: (ceil(D/4) + 2) sequential fp32 additions of products each rounded once, so
    |sim32 - sim64| <= (ceil(D/4) + 3) u' sum_d |v_j v_k|; m: the max of perturbed values moves by at most the largest
    perturbation; mu = fl(1 - lam), the two products and the difference: one rounding each (u' = 1.01 u)."""
    rng = np.random.default_rng(C + D)
    B, I = 4, 4 * C
    vec = _unit(rng, I, D)
    cand, rel = _rows(rng, B, C, I)
    rel = (rel * 0.1).astype(np.float32)                                   # relevance on the scale of the penalty
    gi, _ = _run(ops, vec, cand, rel, min(C, 64), lam)
    lam32 = float(np.float32(lam))
    mu = 1.0 - lam32
    up = 1.01 * U
    for b in range(B):
        items, rels = _distinct(I, cand[b], rel[b])
        V = vec[items].astype(np.float64)
        S = V @ V.T
        Sabs = np.abs(V) @ np.abs(V).T
        serr = ((D + 3) // 4 + 3) * up * Sabs
        lr = lam32 * rels.astype(np.float64)
        m = np.full(items.size, -np.inf)
        merr = np.zeros(items.size)
        alive = np.ones(items.size, dtype=bool)
        pos = {int(it): j for j, it in enumerate(items)}
        for s, it in enumerate(gi[b]):
            if it < 0:
                assert s == min(items.size, min(C, 64)) and np.all(gi[b][s:] == -1)
                break
            obj = lr if s == 0 else lr - mu * m
            pen = 0.0 if s == 0 else mu * np.abs(m)
            err = up * (np.abs(lr) + 2 * pen + np.abs(obj)) + (0.0 if s == 0 else mu * merr + up * pen)
            p = pos[int(it)]
            assert alive[p], (b, s)
            best = np.max(np.where(alive, obj - err, -np.inf))
            assert obj[p] + err[p] >= best, (b, s, obj[p], best)
            alive[p] = False
            m = np.maximum(m, S[:, p])
            merr = np.maximum(merr, serr[:, p])


def test_mmr_orthonormal_is_relevance_order(ops):
    """One-hot rows: sim = 0 between distinct items, so every lam in (0, 1] keeps the relevance order, and lam = 0 starts
    with the most relevant item and then keeps it too (all obj tie at 0: relevance breaks the tie)."""
    C = 16
    vec = np.eye(C, dtype=np.float32)
    rel = np.array([[3, 9, 1, 7, 5, 2, 8, 4, 6, 0, 11, 10, 15, 13, 12, 14]], dtype=np.float32)
    cand = np.arange(C, dtype=np.int32)[None, :]
    want = np.argsort(-rel[0], kind="stable")
    for lam in (0.0, 0.25, 0.5, 1.0):
        gi, gr = _run(ops, vec, cand, rel, C, lam)
        assert np.array_equal(gi[0], want), lam
        assert np.array_equal(gr[0], rel[0][want])


def test_mmr_clusters_textbook_sequence(ops):
    """Three clusters of identical vectors (A: items 0..2 on e0, B: 3..5 on e1, C: 6..8 on e2) with dyadic relevance,
    A's above B's above C's.  At lam = 0.5 a second pick from a cluster costs 0.5, more than any relevance gap, so the
    first three picks alternate clusters (A, B, C); then every candidate has m = 1 and relevance decides.  lam = 1 is
    the relevance order; lam = 0 starts with the most relevant item and alternates the same way."""
    vec = np.zeros((9, 3), dtype=np.float32)
    for k in range(3):
        vec[3 * k:3 * k + 3, k] = 1
    rel = np.array([1.0, 0.96875, 0.9375, 0.90625, 0.875, 0.84375, 0.8125, 0.78125, 0.75], dtype=np.float32)
    cand = np.array([[8, 2, 5, 0, 3, 7, 1, 4, 6]], dtype=np.int32)             # slot order is irrelevant
    rel_c = rel[cand]
    mmr = [0, 3, 6, 1, 2, 4, 5, 7, 8]
    for lam, want in ((0.5, mmr), (0.0, mmr), (1.0, list(range(9)))):
        gi, gr = _run(ops, vec, cand, rel_c, 9, lam)
        assert gi[0].tolist() == want, lam
        assert np.array_equal(gr[0], rel[want]), lam
    gi, _ = _run(ops, vec, cand, rel_c, 3, 0.5)                                  # N < C: the first three picks
    assert gi[0].tolist() == [0, 3, 6]
    # duplicates: the first occurrence's relevance counts (item 0 listed again later with a larger relevance)
    cand2 = np.array([[0, 3, 0, 1]], dtype=np.int32)
    rel2 = np.array([[0.5, 0.75, 2.0, 0.625]], dtype=np.float32)
    gi, gr = _run(ops, vec, cand2, rel2, 4, 1.0)
    assert gi[0].tolist() == [3, 1, 0, -1] and gr[0].tolist() == [0.75, 0.625, 0.5, -np.inf]


def test_mmr_ties_go_to_smaller_item(ops):
    """Equal relevance and equal vectors: every obj ties, so the order is item ascending whatever the slot order."""
    I, C = 40, 32
    vec = np.ones((I, 4), dtype=np.float32) * 0.5
    rng = np.random.default_rng(5)
    cand = rng.permutation(I)[:C].astype(np.int32)[None, :]
    rel = np.full((1, C), 0.25, dtype=np.float32)
    for lam in (0.0, 0.5, 1.0):
        gi, _ = _run(ops, vec, cand, rel, C, lam)
        assert gi[0].tolist() == sorted(cand[0].tolist()), lam


def test_mmr_many_rows(ops):
    """More rows than one wave of CTAs, C = 200, D = 64, N = 20 (a diversified top-20 from a pool of 200)."""
    rng = np.random.default_rng(9)
    B, C, D, I, N = 3000, 200, 64, 5000, 20
    vec = _unit(rng, I, D)
    cand, rel = _rows(rng, B, C, I)
    gi, gr = _run(ops, vec, cand, rel, N, 0.5)
    for b in list(range(0, B, 97)) + [B - 1]:
        wi, wr = mmr_ref(vec, cand[b], rel[b], N, 0.5)
        assert np.array_equal(gi[b], wi) and np.array_equal(gr[b].view(np.int32), wr.view(np.int32)), b


@pytest.mark.parametrize("bad", [2 ** 32 + 5, -2 ** 32 + 3, 2 ** 31])
def test_mmr_rerank_rejects_ids_outside_int32_before_the_cast(bad):
    """recommend.mmr_rerank checks int64 ids as given: 2^32 + 5 must not pass as item 5 after the int32 cast, whether the
    ids are CUDA or host data and wherever the relevance lives."""
    from diffmm_b200 import recommend
    I = 50
    v = torch.from_numpy(_unit(np.random.default_rng(0), I, 8)).to(DEV)
    cand = np.array([[0, 1, 2], [3, -1, 4]], dtype=np.int64)
    rel = np.array([[0.5, 0.25, 0.0], [1.0, 0.0, 0.5]], dtype=np.float32)
    want_i, want_r = recommend.mmr_rerank(v, cand, rel, 3, 0.5)
    bad_cand = cand.copy()
    bad_cand[1, 2] = bad
    for c, r in ((T(bad_cand), T(rel)), (T(bad_cand), rel), (bad_cand, T(rel)), (bad_cand, rel)):
        with pytest.raises(ValueError, match="candidates"):
            recommend.mmr_rerank(v, c, r, 3, 0.5)
    got_i, got_r = recommend.mmr_rerank(v, T(cand), rel, 3, 0.5)        # in-range int64 CUDA ids: the host result
    assert torch.equal(got_i, want_i) and torch.equal(got_r.view(torch.int32), want_r.view(torch.int32))


def test_mmr_zero_rows_and_rejects(ops):
    from diffmm_b200 import _lib
    lib = _lib.load()
    ctx = _lib.ctx(0)
    assert lib.dmm_mmr_rerank(ctx, None, 64, 10, 64, None, 5, None, 5, 0, 5, 5, 0.5, None, 5, None, 5, None) == 0
    for C, D, N, lam in ((0, 8, 1, 0.5), (1025, 8, 1, 0.5), (8, 0, 1, 0.5), (8, 257, 1, 0.5), (513, 64, 1, 0.5),
                         (8, 8, 0, 0.5), (8, 8, 9, 0.5), (8, 8, 1, -0.01), (8, 8, 1, 1.01), (8, 8, 1, float("nan"))):
        rc = lib.dmm_mmr_rerank(ctx, None, max(D, 1), 10, D, None, max(C, 1), None, max(C, 1), 0, C, N, lam, None,
                                max(N, 1), None, max(N, 1), None)
        assert rc != 0, (C, D, N, lam)
    v = torch.zeros((10, 8), device=DEV)
    c = torch.zeros((2, 4), dtype=torch.int32, device=DEV)
    r = torch.zeros((2, 4), device=DEV)
    i = torch.zeros((2, 2), dtype=torch.int32, device=DEV)
    o = torch.zeros((2, 2), device=DEV)
    for args in ((v.double(), c, r, 2, 0.5, i, o), (v, c.long(), r, 2, 0.5, i, o), (v, c, r[:, :3], 2, 0.5, i, o),
                 (v, c, r, 3, 0.5, i, o), (v, c, r, 2, 1.5, i, o), (v, c.t(), r, 2, 0.5, i, o),
                 (v, c, r, 2, 0.5, i.long(), o), (v, c, r, 2, 0.5, i, o[:1])):
        with pytest.raises(ValueError):
            ops.mmr_rerank(*args)
