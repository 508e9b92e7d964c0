"""The three kernels behind diffmm_b200.recommend, each on its own at ragged sizes, with leading dimensions wider than the
data and every output sentinel-filled first (nothing outside the documented region may change):
  * dmm_eval_mask_scores_cmax: the scores of dmm_eval_mask_scores bit for bit, every chunk maximum it touched recomputed
    exactly (NaN-propagating), every other one untouched, and the pruned top-k on the refreshed maxima equal to the
    whole-row top-k;
  * dmm_topn_rank: rank order (score desc, column asc in the top-k kernels' total order) against numpy's lexsort, -inf
    slots as item -1, every prefix equal to the top-k set of its length;
  * dmm_eval_metrics_cutoffs: the reference's literal per-user calcRes (Main.py:422-448) on every prefix, bit for bit."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SENT = np.float32(7.25)


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _ptr(lists):
    p = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=p[1:])
    return p


def _order_key(x):
    """The top-k kernels' order-preserving key (csrc/topk.cu order_key): -0.0 ties with +0.0, NaN by its bits."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).copy()
    u[u == 0x80000000] = 0
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def _rank(row):
    """Column order of one row: key descending, then column ascending."""
    return np.lexsort((np.arange(row.shape[0]), -_order_key(row).astype(np.int64)))


def _chunk_max(rows, n_cols):
    """max over the 32-column chunks of the columns < n_cols, NaN if any of them is NaN."""
    n_chunks = (n_cols + 31) // 32
    pad = np.full((rows.shape[0], n_chunks * 32), -np.inf, dtype=np.float32)
    pad[:, :n_cols] = rows[:, :n_cols]
    with np.errstate(invalid="ignore"):
        return pad.reshape(rows.shape[0], n_chunks, 32).max(axis=2)


def _same_bits(a, b):
    """Bitwise equality where neither is NaN, NaN at the same places (max.NaN writes the canonical NaN)."""
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int32), b[~nb].view(np.int32))


# ------------------------------------------------------------------------------------------------ mask + chunk maxima
def _mask_case(rows_n, I, seed):
    """Scores, the exclusion CSR and the evaluated rows (unsorted, repeated).  Planted: a row whose best chunk is entirely
    excluded (with several high scores in its other chunks, so a stale maximum would select the wrong chunk), a row
    masked down to a single item, NaN in an excluded and in a kept chunk, and users without exclusions."""
    rng = np.random.default_rng(seed)
    U = max(rows_n // 2, 1) + 3
    rows = rng.integers(0, U, rows_n).astype(np.int64)
    rows[: min(rows_n, U)] = rng.permutation(U)[: min(rows_n, U)]
    scores = rng.standard_normal((rows_n, I)).astype(np.float32)
    train = []
    for u in range(U):
        n_tr = int(rng.integers(0, min(40, I) + 1)) if u % 6 else 0
        train.append(np.sort(rng.choice(I, n_tr, replace=False)).astype(np.int32))
    n_chunks = (I + 31) // 32
    for r in range(rows_n):
        u = rows[r]
        kind = r % 5
        if kind == 1 and n_chunks >= 2:                 # best chunk entirely excluded
            c = int(rng.integers(0, n_chunks))
            cols = np.arange(32 * c, min(32 * c + 32, I))
            scores[r, cols] = 100.0 + rng.random(len(cols)).astype(np.float32)
            others = np.setdiff1d(np.arange(I), cols)[: 3 * 32]
            scores[r, others] += 10.0                   # several high scores in the chunks after it
            train[u] = np.union1d(train[u], cols).astype(np.int32)
        elif kind == 2 and I > 1:                       # masked down to a single item
            keep = int(rng.integers(0, I))
            train[u] = np.setdiff1d(np.arange(I), [keep]).astype(np.int32)
        elif kind == 3:                                 # NaN in a chunk the mask touches and in one it does not
            if len(train[u]):
                scores[r, (int(train[u][0]) // 32) * 32 + 0 if I > 1 else 0] = np.nan
            scores[r, int(rng.integers(0, I))] = np.nan
    return U, train, rows, scores


@pytest.mark.parametrize("I", [1, 31, 32, 33, 7050, 8193, 100003])
@pytest.mark.parametrize("rows_n", [1, 5, 63, 1025])
def test_mask_refreshes_chunk_maxima(ops, rows_n, I):
    if rows_n * I > 30_000_000:
        rows_n = 300                                    # 1025 x 100003: keep the host reference in memory bounds
    U, train, rows, scores = _mask_case(rows_n, I, seed=rows_n * 7 + I)
    fill = np.float32(-np.inf) if I % 2 else np.float32(-1e8)
    n_chunks = (I + 31) // 32
    ld, ldc = I + 5, ((n_chunks + 3) // 4) * 4 + 4
    sbuf = np.full((rows_n, ld), SENT, dtype=np.float32)
    sbuf[:, :I] = scores
    ptr, idx, rid = T(_ptr(train)), T(np.concatenate(train) if sum(map(len, train)) else np.zeros(0, np.int32)), T(rows)
    if idx.numel() == 0:
        idx = torch.zeros(1, dtype=torch.int32, device=DEV)

    # reference scores: dmm_eval_mask_scores
    plain = T(sbuf)
    ops.eval_mask_scores(ptr, idx, rid, plain[:, :I], I, float(fill))
    masked = plain.cpu().numpy()
    want_cmax = _chunk_max(masked, I)
    touched = np.zeros((rows_n, n_chunks), dtype=bool)
    for r, u in enumerate(rows):
        touched[r, train[u] // 32] = True

    # (a) exact initial maxima (what the contraction writes): everything exact afterwards
    cbuf = np.full((rows_n, ldc), SENT, dtype=np.float32)
    cbuf[:, :n_chunks] = _chunk_max(sbuf, I)
    s_dev, c_dev = T(sbuf), T(cbuf)
    ops.eval_mask_scores_cmax(ptr, idx, rid, s_dev[:, :I], I, c_dev, float(fill))
    got_s, got_c = s_dev.cpu().numpy(), c_dev.cpu().numpy()
    assert np.array_equal(got_s.view(np.int32), masked.view(np.int32))
    assert _same_bits(got_c[:, :n_chunks], want_cmax)
    assert np.array_equal(got_c[:, n_chunks:], cbuf[:, n_chunks:])

    # (b) sentinel maxima: exactly the touched chunks are rewritten
    c2 = T(np.full((rows_n, ldc), SENT, dtype=np.float32))
    s2 = T(sbuf)
    ops.eval_mask_scores_cmax(ptr, idx, rid, s2[:, :I], I, c2, float(fill))
    g2 = c2.cpu().numpy()
    assert _same_bits(g2[:, :n_chunks][touched], want_cmax[touched])
    assert np.all(g2[:, :n_chunks][~touched] == SENT) and np.all(g2[:, n_chunks:] == SENT)

    # (c) the pruned top-k on the refreshed maxima selects what the whole-row top-k selects
    for k in sorted({min(k, I) for k in (1, 2, 5, 20)}):
        kptr = torch.arange(rows_n + 1, dtype=torch.int64, device=DEV) * k
        whole = torch.empty(rows_n * k, dtype=torch.int32, device=DEV)
        pruned = torch.full((rows_n * k,), -7, dtype=torch.int32, device=DEV)
        ops.topk_edges(s_dev[:, :I], I, kptr, 0, None, whole)
        ops.topk_edges_pruned(s_dev[:, :I], I, c_dev, kptr, 0, None, pruned)
        assert torch.equal(whole, pruned), k


def test_mask_cmax_zero_rows_and_bad_ld(ops):
    from diffmm_b200._lib import DiffMMError
    s = torch.zeros((0, 64), device=DEV)
    c = torch.zeros((0, 4), device=DEV)
    ptr = torch.zeros(2, dtype=torch.int64, device=DEV)
    idx = torch.zeros(1, dtype=torch.int32, device=DEV)
    ops.eval_mask_scores_cmax(ptr, idx, torch.zeros(0, dtype=torch.int64, device=DEV), s, 64, c)
    s = torch.zeros((1, 100), device=DEV)
    with pytest.raises(DiffMMError):
        ops.eval_mask_scores_cmax(ptr, idx, torch.zeros(1, dtype=torch.int64, device=DEV), s, 100, torch.zeros((1, 3), device=DEV))


# ------------------------------------------------------------------------------------------------ ranking
def _rank_scores(rows_n, I, N, seed):
    """Quantised scores (exact ties everywhere, straddling every prefix length), explicit -0.0 / +0.0, +NaN and -NaN,
    and rows padded with -inf so that fewer than N finite scores remain."""
    rng = np.random.default_rng(seed)
    s = (np.round(rng.standard_normal((rows_n, I)) * 3) / 4).astype(np.float32)
    for r in range(rows_n):
        kind = r % 4
        if kind == 1:
            z = rng.choice(I, min(I, 6), replace=False)
            s[r, z[::2]] = np.float32(0.0)
            s[r, z[1::2]] = np.float32(-0.0)
            s[r] = np.where(s[r] > 0, -s[r], s[r])          # the zeros are the row's best scores
        elif kind == 2:
            s[r, rng.choice(I, min(I, 3), replace=False)] = np.nan
            s[r, int(rng.integers(0, I))] = -np.float32(np.nan)
        elif kind == 3:
            keep = max(N // 2, 1) - 1
            s[r, rng.permutation(I)[keep:]] = -np.inf        # keep - 1 finite scores (none when N <= 2)
    return s


@pytest.mark.parametrize("N", [1, 7, 32, 33, 64, 65, 257, 1000, 1024])
@pytest.mark.parametrize("rows_n", [1, 5, 63])
def test_topn_rank(ops, rows_n, N):
    I = N + 37 if N < 1000 else 1503
    s = _rank_scores(rows_n, I, N, seed=N * 11 + rows_n)
    ld = I + 3
    sbuf = np.full((rows_n, ld), SENT, dtype=np.float32)
    sbuf[:, :I] = s
    s_dev = T(sbuf)
    kptr = torch.arange(rows_n + 1, dtype=torch.int64, device=DEV) * N
    sel = torch.empty(rows_n * N, dtype=torch.int32, device=DEV)
    ops.topk_edges(s_dev[:, :I], I, kptr, 0, None, sel)
    ib = torch.full((rows_n, N + 2), -7, dtype=torch.int32, device=DEV)
    sb = torch.full((rows_n, N + 3), float(SENT), dtype=torch.float32, device=DEV)
    ops.topn_rank(s_dev[:, :I], sel.view(rows_n, N), N, ib[:, :N], sb[:, :N])
    items, scores = ib.cpu().numpy(), sb.cpu().numpy()
    assert np.all(items[:, N:] == -7) and np.all(scores[:, N:] == SENT)
    assert np.array_equal(s_dev.cpu().numpy().view(np.int32), sbuf.view(np.int32))     # input untouched
    n_pad = 0
    for r in range(rows_n):
        order = _rank(s[r])[:N]
        want_scores = s[r, order]
        want_items = np.where(np.isneginf(want_scores), -1, order)
        n_pad += int((want_items == -1).sum())
        assert np.array_equal(items[r, :N], want_items), r
        assert np.array_equal(scores[r, :N].view(np.int32), want_scores.view(np.int32)), r
    assert n_pad > 0 or rows_n < 4 or N <= 2
    # every prefix is the top-k set of its length
    for k in sorted({1, max(N // 2, 1), max(N - 1, 1), N}):
        kp = torch.arange(rows_n + 1, dtype=torch.int64, device=DEV) * k
        tk = torch.empty(rows_n * k, dtype=torch.int32, device=DEV)
        ops.topk_edges(s_dev[:, :I], I, kp, 0, None, tk)
        tk = tk.view(rows_n, k).cpu().numpy()
        for r in range(rows_n):
            cols = np.sort(_rank(s[r])[:k])             # the ranked columns before the -1 mapping
            assert np.array_equal(tk[r], cols), (k, r)
            pref = items[r, :k]
            assert np.array_equal(np.sort(pref[pref >= 0]), np.sort(cols[~np.isneginf(s[r, cols])])), (k, r)


def test_topn_rank_many_rows(ops):
    rows_n, N, I = 1025, 100, 8193
    s = _rank_scores(rows_n, I, N, seed=5)
    s_dev = T(s)
    kptr = torch.arange(rows_n + 1, dtype=torch.int64, device=DEV) * N
    sel = torch.empty(rows_n * N, dtype=torch.int32, device=DEV)
    ops.topk_edges(s_dev, I, kptr, 0, None, sel)
    items = torch.empty((rows_n, N), dtype=torch.int32, device=DEV)
    scores = torch.empty((rows_n, N), dtype=torch.float32, device=DEV)
    ops.topn_rank(s_dev, sel.view(rows_n, N), N, items, scores)
    items = items.cpu().numpy()
    for r in range(rows_n):
        order = _rank(s[r])[:N]
        assert np.array_equal(items[r], np.where(np.isneginf(s[r, order]), -1, order)), r


@pytest.mark.parametrize("N", [0, 1025])
def test_topn_rank_rejects_n(ops, N):
    from diffmm_b200._lib import DiffMMError
    s = torch.zeros((2, 2000), device=DEV)
    sel = torch.zeros((2, 1100), dtype=torch.int32, device=DEV)
    items = torch.zeros((2, 1100), dtype=torch.int32, device=DEV)
    out = torch.zeros((2, 1100), device=DEV)
    with pytest.raises(DiffMMError, match="1024"):
        ops.topn_rank(s, sel, N, items, out)


def test_topn_rank_zero_rows(ops):
    s = torch.zeros((0, 64), device=DEV)
    e = torch.zeros((0, 8), dtype=torch.int32, device=DEV)
    ops.topn_rank(s, e, 8, e.clone(), torch.zeros((0, 8), device=DEV))


# ------------------------------------------------------------------------------------------------ metrics at cutoffs
def _calc_res_literal(top, test_items, K):
    """Main.py:422-448 for one user and one list length K, literally (recall = ndcg = 0 without test items)."""
    tem_top = list(top)
    tst_num = len(test_items)
    max_dcg = np.sum([np.reciprocal(np.log2(loc + 2)) for loc in range(min(tst_num, K))])
    recall = dcg = precision = 0
    for val in test_items:
        if val in tem_top:
            recall += 1
            dcg = dcg + np.reciprocal(np.log2(tem_top.index(val) + 2))
            precision += 1
    if tst_num == 0:
        return 0.0, 0.0, precision / K
    return recall / tst_num, dcg / max_dcg, precision / K


@pytest.mark.parametrize("cutoffs", [(1,), (20,), (10, 20, 50), (1000,)])
def test_metrics_at_cutoffs(ops, cutoffs):
    from diffmm_b200 import recommend
    rng = np.random.default_rng(sum(cutoffs))
    N = cutoffs[-1] + 3
    I = N + 200
    U = 60
    train = [np.sort(rng.choice(I, int(rng.integers(0, 30)), replace=False)) for _ in range(U)]
    test = []
    for u in range(U):
        n_te = int(rng.integers(1, 6))
        if u % 5 == 1:
            n_te = min(cutoffs[-1] + 9, I)                  # more test items than the largest cutoff
        if u % 9 == 4:
            n_te = 0                                        # no test items
        te = list(rng.choice(I, n_te, replace=False))
        if u % 4 == 2 and n_te and len(train[u]):
            te[0] = int(train[u][0])                        # a test item that is a train item
        test.append(np.asarray(te, dtype=np.int32))
    rows = rng.permutation(np.concatenate([np.arange(U), rng.integers(0, U, 13)])).astype(np.int64)   # unsorted, repeated
    n = len(rows)
    ranked = np.empty((n, N), dtype=np.int32)
    for r, u in enumerate(rows):
        free = np.setdiff1d(np.arange(I), train[u])
        # bias the list towards the user's test items so that hits land at every depth
        pool = np.concatenate([rng.permutation(np.intersect1d(free, test[u])), rng.permutation(free)])
        lst = pool[np.sort(np.unique(pool, return_index=True)[1])]
        lst = rng.permutation(lst[:N]) if r % 2 else lst[:N]
        ranked[r, :len(lst)] = lst
        ranked[r, len(lst):] = -1
        if r % 7 == 0:
            ranked[r, N // 2:] = -1                         # a short list (-1 padding)
    rbuf = np.full((n, N + 4), -9, dtype=np.int32)
    rbuf[:, :N] = ranked
    inv, max_dcg = recommend.metric_tables(N)
    tptr = _ptr(test)
    titems = np.concatenate(test).astype(np.int32)
    out = torch.full((n, len(cutoffs), 3), float("nan"), dtype=torch.float64, device=DEV)
    ops.eval_metrics_cutoffs(T(rbuf)[:, :N], N, list(cutoffs), T(rows), T(tptr), T(titems), T(inv), T(max_dcg), out)
    got = out.cpu().numpy()
    for r, u in enumerate(rows):
        for j, c in enumerate(cutoffs):
            ref = np.array(_calc_res_literal(ranked[r, :c], test[u], c), dtype=np.float64)
            assert np.array_equal(got[r, j], ref), (r, u, c, got[r, j], ref)


def test_metrics_at_cutoffs_rejects(ops):
    from diffmm_b200._lib import DiffMMError
    ranked = torch.zeros((2, 40), dtype=torch.int32, device=DEV)
    ptr = torch.tensor([0, 1, 2], dtype=torch.int64, device=DEV)
    items = torch.zeros(2, dtype=torch.int32, device=DEV)
    rows = torch.tensor([0, 1], dtype=torch.int64, device=DEV)
    tab = torch.ones(1100, dtype=torch.float64, device=DEV)
    out = torch.empty((2, 4, 3), dtype=torch.float64, device=DEV)
    for N, cuts in ((40, [20, 10]), (40, [10, 10]), (40, [0]), (40, [41]), (0, [1]), (1025, [1])):
        with pytest.raises(DiffMMError):
            ops.eval_metrics_cutoffs(ranked, N, cuts, rows, ptr, items, tab, tab, out)
    ops.eval_metrics_cutoffs(ranked, 40, [1], rows[:0], ptr, items, tab, tab, out)      # zero rows: no-op
