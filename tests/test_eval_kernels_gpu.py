"""The device evaluation tail (csrc/eval.cu) against the reference's literal per-user loop (Main.py:390-448) in float64:
train mask (dmm_eval_mask_scores) -> top-K (dmm_topk_edges with k = K) -> rank + Recall / NDCG / Precision per user
(dmm_eval_metrics).  The reference ranks with torch.topk; its order among exactly equal scores is the kernels'
documented rule here: score descending, then column ascending."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FILL = -1e8


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


def _dataset(I, K, seed):
    """U users with train and test items; the evaluated rows are a shuffled selection with repeats, not a multiple of 8
    long.  Planted: users with more test items than K, users with fewer than K unmasked items (filled entries enter
    their top-K), a test item that is also a train item, and exact score ties straddling position K."""
    rng = np.random.default_rng(seed)
    U = 50
    train, test = [], []
    for u in range(U):
        n_tr = int(rng.integers(0, min(30, I // 2)))
        if u % 7 == 3:
            n_tr = I - max(K // 2, 1)                     # fewer than K unmasked items
        tr = rng.choice(I, n_tr, replace=False)
        n_te = int(rng.integers(1, 6))
        if u % 5 == 1:
            n_te = min(K + 7, I)                          # more test items than K
        te = list(rng.choice(I, n_te, replace=False))
        if u % 4 == 2 and n_tr:
            te[0] = int(tr[0])                            # a test item that is also a train item
        train.append(np.sort(tr).astype(np.int32))
        test.append(np.asarray(te, dtype=np.int32))
    rows = rng.permutation(np.concatenate([np.arange(U), rng.integers(0, U, 11)]))[:53]   # unsorted, repeated
    scores = rng.standard_normal((len(rows), I)).astype(np.float32)
    for r, u in enumerate(rows):
        mask = np.ones(I, dtype=bool)
        mask[train[u]] = False
        free = np.flatnonzero(mask)
        if r % 3 == 0 and len(free) > K + 3:
            # ties straddling position K: the K-th best unmasked score is shared by 5 columns, some of them test items
            order = free[np.lexsort((free, -scores[r, free]))]
            tied = order[max(K - 3, 0):K + 2]
            scores[r, tied] = scores[r, order[K - 1]]
            test[u] = np.unique(np.concatenate([test[u], tied[::2]])).astype(np.int32)
    return U, train, test, rows, scores


def _calc_res_literal(top, test_items, K):
    """Main.py:422-448 for one user, literally."""
    tem_top = list(top)
    tst_num = len(test_items)
    max_dcg = np.sum([np.reciprocal(np.log2(loc + 2)) for loc in range(min(tst_num, K))])
    recall = dcg = precision = 0
    for val in test_items:
        if val in tem_top:
            recall += 1
            dcg = dcg + np.reciprocal(np.log2(tem_top.index(val) + 2))
            precision += 1
    return recall / tst_num, dcg / max_dcg, precision / K


@pytest.mark.parametrize("I", [45, 1003])
@pytest.mark.parametrize("K", [1, 20, 32])
def test_eval_mask_topk_metrics(ops, I, K):
    U, train, test, rows, scores = _dataset(I, K, seed=I + K)
    n = len(rows)
    assert n % 8 != 0
    ld = I + 3
    sbuf = np.full((n, ld), 7.25, dtype=np.float32)
    sbuf[:, :I] = scores
    s_dev = T(sbuf)
    ops.eval_mask_scores(T(_ptr(train)), T(np.concatenate(train)), T(rows.astype(np.int64)), s_dev[:, :I], I, FILL)
    masked = s_dev.cpu().numpy()
    # exactly `fill` at the train items, every other score (and the padding) bit for bit as before
    want = sbuf.copy()
    for r, u in enumerate(rows):
        want[r, train[u]] = np.float32(FILL)
    assert np.array_equal(masked.view(np.int32), want.view(np.int32))

    kptr = torch.arange(n + 1, dtype=torch.int64, device=DEV) * K
    top = torch.empty(n * K, dtype=torch.int32, device=DEV)
    ops.topk_edges(s_dev[:, :I], I, kptr, 0, None, top)
    inv = np.array([np.reciprocal(np.log2(p + 2)) for p in range(K)], dtype=np.float64)
    max_dcg = np.array([np.sum([np.reciprocal(np.log2(loc + 2)) for loc in range(t)]) for t in range(K + 1)],
                       dtype=np.float64)
    out = torch.full((n, 3), float("nan"), dtype=torch.float64, device=DEV)
    ops.eval_metrics(s_dev[:, :I], top, K, T(rows.astype(np.int64)), T(_ptr(test)), T(np.concatenate(test)), T(inv),
                     T(max_dcg), out)
    got = out.cpu().numpy()
    top_np = top.view(n, K).cpu().numpy()
    n_filled = 0
    for r, u in enumerate(rows):
        m = want[r, :I]
        ranked = np.lexsort((np.arange(I), -m.astype(np.float64)))[:K]     # score desc, then column asc
        assert np.array_equal(top_np[r], np.sort(ranked)), r
        n_filled += int((m[ranked] == np.float32(FILL)).sum())
        ref = _calc_res_literal(ranked, test[u], K)
        assert np.array_equal(got[r], np.array(ref, dtype=np.float64)), (r, u, got[r], ref)
    assert n_filled > 0 or K == 1


def test_eval_metrics_rejects_k_above_32(ops):
    from diffmm_b200._lib import DiffMMError
    K = 33
    scores = torch.zeros((2, 64), device=DEV)
    top = torch.zeros(2 * K, dtype=torch.int32, device=DEV)
    ptr = torch.tensor([0, 1, 2], dtype=torch.int64, device=DEV)
    items = torch.zeros(2, dtype=torch.int32, device=DEV)
    rows = torch.tensor([0, 1], dtype=torch.int64, device=DEV)
    tab = torch.ones(K + 1, dtype=torch.float64, device=DEV)
    out = torch.empty((2, 3), dtype=torch.float64, device=DEV)
    with pytest.raises(DiffMMError):
        ops.eval_metrics(scores, top, K, rows, ptr, items, tab, tab, out)
