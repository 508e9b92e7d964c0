"""The public recommendation layer: ``recommend.score_topn`` against a numpy ranking of the library's own dense bf16x3
scores and against the same pipeline built from the whole-row kernels, and ``Coach.recommend`` / ``Coach.evaluate`` on a
trained Coach (built like tests/test_epoch_gpu.py builds it): evaluate((K,)) returns exactly testEpoch()'s floats, other
cutoffs equal a host literal loop on the same masked scores, and neither call draws random numbers or moves a
parameter."""
import json
import os
import random
import shutil

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "epoch_run")


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _rank_rows(s):
    """Per row: column order by score descending, then column ascending (no NaN in these scores)."""
    cols = np.broadcast_to(np.arange(s.shape[1]), s.shape)
    return np.lexsort((cols, -s.astype(np.float64)), axis=-1)


def _dense_scores(u, it, precision="bf16x3"):
    """The library's own contraction, dense, without the chunk maxima (the evaluation's linear_tn)."""
    from diffmm_b200.autograd import linear_tn
    return linear_tn(u, it, None, 0, precision)


def _case(B, I, D, seed, excl):
    rng = np.random.default_rng(seed)
    u = rng.standard_normal((B, D)).astype(np.float32)
    it = rng.standard_normal((I, D)).astype(np.float32) * 0.5
    U = B + 3
    if excl == "none":
        return u, it, None, None
    lists = []
    for r in range(U):
        if excl == "all":
            lists.append(np.arange(I))
        elif excl == "all_but_three":
            lists.append(np.setdiff1d(np.arange(I), rng.choice(I, 3, replace=False)))
        else:
            lists.append(np.sort(rng.choice(I, int(rng.integers(0, min(60, I))), replace=False)))
    ptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=ptr[1:])
    idx = np.concatenate(lists).astype(np.int32)
    rows = rng.permutation(U)[:B]
    return u, it, (ptr, idx, rows), lists


@pytest.mark.parametrize("B,I,n,excl", [
    (77, 1003, 20, "none"),
    (64, 7050, 100, "some"),
    (5, 300, 17, "all"),
    (33, 7050, 20, "all_but_three"),
    (40, 257, 257, "some"),                 # n = I
    (9000, 7050, 50, "some"),               # more users than one 1 GB score block (8192 rows at 7050 items)
])
def test_score_topn_against_reference_ranking(B, I, n, excl):
    from diffmm_b200 import recommend
    u, it, ex, lists = _case(B, I, 64, seed=B + I + n, excl=excl)
    exclude = None if ex is None else (T(ex[0]), T(ex[1]), ex[2])
    items, scores = recommend.score_topn(T(u), T(it), n, exclude=exclude)
    assert items.dtype == torch.int64 and scores.dtype == torch.float32 and items.shape == (B, n) == scores.shape
    dense = _dense_scores(T(u), T(it)).cpu().numpy()
    masked = dense.copy()
    if ex is not None:
        for b, r in enumerate(ex[2]):
            masked[b, lists[r]] = -np.inf
    order = _rank_rows(masked)[:, :n]
    want_s = np.take_along_axis(masked, order, axis=1)
    want_i = np.where(np.isneginf(want_s), -1, order)
    got_i, got_s = items.cpu().numpy(), scores.cpu().numpy()
    assert np.array_equal(got_i, want_i)
    assert np.array_equal(got_s.view(np.int32), want_s.view(np.int32))
    if excl == "all":
        assert np.all(got_i == -1) and np.all(np.isneginf(got_s))
    if excl == "all_but_three":
        assert np.all((got_i[:, :3] >= 0)) and np.all(got_i[:, 3:] == -1)
    # the scores are the bf16x3 product: within DESIGN §2's gate of the float64 product
    ref = u.astype(np.float64) @ it.astype(np.float64).T
    scale = np.abs(ref).max()
    fin = got_i >= 0
    err = np.abs(got_s[fin] - np.take_along_axis(ref, np.maximum(got_i, 0), axis=1)[fin]).max() if fin.any() else 0.0
    assert err <= 3e-5 * scale, err / scale


@pytest.mark.parametrize("I,n", [(7050, 20), (7050, 55), (33000, 100), (33000, 258), (7050, 1000), (256, 64)])
@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_score_topn_equals_whole_row_pipeline(I, n, precision):
    """score_topn against the same pipeline on the whole-row kernels: contraction without maxima, eval_mask_scores,
    topk_edges, topn_rank.  score_topn prunes at 4 n <= ceil(I / 32): (7050, 20), (7050, 55), (33000, 100) and (33000, 258)
    (the last two through the pruned kernel's deferred two-level pass, k > 64); the others are the whole-row path."""
    from diffmm_b200 import ops, recommend
    B = 300
    u, it, ex, _ = _case(B, I, 64, seed=I + n, excl="some")
    items, scores = recommend.score_topn(T(u), T(it), n, exclude=(T(ex[0]), T(ex[1]), ex[2]), precision=precision)
    dense = _dense_scores(T(u), T(it), precision)
    ops.eval_mask_scores(T(ex[0]), T(ex[1]), T(ex[2].astype(np.int64)), dense, I, float("-inf"))
    kptr = torch.arange(B + 1, dtype=torch.int64, device=DEV) * n
    sel = torch.empty(B * n, dtype=torch.int32, device=DEV)
    ops.topk_edges(dense, I, kptr, 0, None, sel)
    wi = torch.empty((B, n), dtype=torch.int32, device=DEV)
    ws = torch.empty((B, n), dtype=torch.float32, device=DEV)
    ops.topn_rank(dense, sel.view(B, n), n, wi, ws)
    assert torch.equal(items, wi.long())
    assert torch.equal(scores.view(torch.int32), ws.view(torch.int32))


# ------------------------------------------------------------------------------------------------ Coach
@pytest.fixture(scope="module")
def coach(tmp_path_factory):
    from diffmm_b200 import Main
    from diffmm_b200.Conf import Config
    gold = json.load(open(os.path.join(GOLD, "result.json")))
    tmp = tmp_path_factory.mktemp("rec")
    shutil.copytree(os.path.join(GOLD, "Datasets"), tmp / "Datasets")
    with pytest.MonkeyPatch.context() as mp:
        mp.chdir(tmp)
        mp.setenv("DIFFMM_CPU_RNG", "1")
        cfg = Config()
        cfg.data.name = "tiktok"
        for k, v in gold["overrides"].items():
            sec, key = k.split(".")
            setattr(getattr(cfg, sec), key, v)
        cfg.base.precision = "bf16x3"
        cfg.base.cuda_graph = False
        Main.seed_it(cfg.base.seed)
        handler = Main.DataHandler(cfg)
        handler.LoadData()
        c = Main.Coach(handler, cfg)
        c.run()
        yield c


def _state(c):
    params = [p for m in [c.model, *c._denoise_dict().values()] for p in m.parameters()]
    return (torch.get_rng_state(), torch.cuda.get_rng_state(), np.random.get_state(), random.getstate(),
            [p._version for p in params], [p.detach().clone() for p in params])


def _same_state(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert a[2][0] == b[2][0] and np.array_equal(a[2][1], b[2][1]) and a[2][2:] == b[2][2:]
    assert a[3] == b[3]
    assert a[4] == b[4]
    assert all(torch.equal(x, y) for x, y in zip(a[5], b[5]))


def test_evaluate_at_k_equals_test_epoch(coach):
    K = int(coach.config.base.topk)
    got = coach.evaluate((K,))
    want = coach.testEpoch()
    assert got == {f"Recall@{K}": want["Recall"], f"NDCG@{K}": want["NDCG"], f"Precision@{K}": want["Precision"]}
    assert want["Recall"] > 0


def test_evaluate_cutoffs_against_host_literal_loop(coach):
    from diffmm_b200 import ops
    cutoffs = (10, 20, 50)
    got = coach.evaluate((50, 20, 10, 20))          # unsorted, repeated: the same as (10, 20, 50)
    assert list(got) == [f"{m}@{c}" for c in cutoffs for m in ("Recall", "NDCG", "Precision")]
    h, cfg = coach.handler, coach.config
    I = cfg.data.item_num
    users = np.asarray(h.testData.test_users, dtype=np.int64)
    u_embs, i_embs = coach._final_embs()
    usr = T(users)
    scores = _dense_scores(u_embs[usr].contiguous(), i_embs)
    ops.eval_mask_scores(h.train_indptr, h.train_indices, usr, scores, I, -1e8)
    order = _rank_rows(scores.cpu().numpy())[:, :max(cutoffs)]
    tb = int(cfg.train.test_batch)
    for c in cutoffs:
        maxdcg = [np.sum([np.reciprocal(np.log2(loc + 2)) for loc in range(t)]) for t in range(c + 1)]
        tot = [0, 0, 0]
        for s in range(0, len(users), tb):
            part = [0, 0, 0]
            for b in range(s, min(s + tb, len(users))):
                top = list(order[b, :c])
                tst = h.testData.test_user_its[users[b]]
                hit, dcg = 0, 0
                for val in tst:
                    if val in top:
                        hit += 1
                        dcg = dcg + np.reciprocal(np.log2(top.index(val) + 2))
                vals = (hit / len(tst), dcg / maxdcg[min(len(tst), c)], hit / c)
                for m in range(3):
                    part[m] += vals[m]
            for m in range(3):
                tot[m] += part[m]
        n = len(users)
        assert got[f"Recall@{c}"] == tot[0] / n
        assert got[f"NDCG@{c}"] == tot[1] / n
        assert got[f"Precision@{c}"] == tot[2] / n


def test_recommend_excludes_train_items(coach):
    h = coach.handler
    U = coach.config.data.user_num
    ptr, idx = h.train_indptr.cpu().numpy(), h.train_indices.cpu().numpy()
    users = np.random.default_rng(0).permutation(U)[:100]
    items, scores = coach.recommend(users, 20)
    items, scores = items.cpu().numpy(), scores.cpu().numpy()
    items_all, _ = coach.recommend(list(users), 20, exclude_train=False)
    items_all = items_all.cpu().numpy()
    n_train_hits = 0
    for b, u in enumerate(users):
        tr = set(idx[ptr[u]:ptr[u + 1]].tolist())
        assert not tr.intersection(items[b].tolist())
        n_train_hits += len(tr.intersection(items_all[b].tolist()))
        assert np.all(np.diff(scores[b]) <= 0)
    assert n_train_hits > 0             # without the exclusion the train items are ranked like any other
    # the unmasked lists are the plain ranking of the same scores
    u_embs, i_embs = coach._final_embs()
    dense = _dense_scores(u_embs[T(users.astype(np.int64))].contiguous(), i_embs).cpu().numpy()
    assert np.array_equal(items_all, _rank_rows(dense)[:, :20])


def test_recommend_and_evaluate_leave_training_state_alone(coach):
    before = _state(coach)
    coach.evaluate()
    coach.recommend(np.arange(10), 5)
    _same_state(before, _state(coach))


def test_coach_rejects_bad_arguments(coach):
    I, U = coach.config.data.item_num, coach.config.data.user_num
    for cuts in ((), (0,), (1025,), (I + 1,)):
        with pytest.raises(ValueError):
            coach.evaluate(cuts)
    with pytest.raises(ValueError):
        coach.recommend([0, U], 5)
    with pytest.raises(ValueError):
        coach.recommend([0, 1], 0)
