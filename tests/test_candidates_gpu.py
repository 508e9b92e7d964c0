"""Pair scores, candidate ranking and the sampled-negative evaluation on a trained Coach (built like
tests/test_recommend_gpu.py builds it): ``Coach.score`` is ``recommend.score_pairs`` on ``_final_embs()``,
``Coach.rank_candidates`` a numpy ranking of those scores, ``Coach.evaluate_sampled`` a host literal loop over the same
``sampled_candidates`` rows and the library's pair scores, exactly; none of them draws random numbers from a global
generator or moves a parameter."""
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


def _order_key(x):
    """The library's total order as an unsigned key (-0.0 ties with +0.0, NaN by its bits)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).copy()
    u[u == 0x80000000] = 0
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.int64)


@pytest.fixture(scope="module")
def coach(tmp_path_factory):
    from diffmm_b200 import Main
    from diffmm_b200.Conf import Config
    gold = json.load(open(os.path.join(GOLD, "result.json")))
    tmp = tmp_path_factory.mktemp("cand")
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


def test_score_equals_score_pairs(coach):
    from diffmm_b200 import recommend
    U, I = coach.config.data.user_num, coach.config.data.item_num
    rng = np.random.default_rng(0)
    users, items = rng.integers(0, U, 5000), rng.integers(0, I, 5000)
    got = coach.score(users, items)
    u_embs, i_embs = coach._final_embs()
    want = recommend.score_pairs(u_embs, i_embs, users, items, precision="bf16x3")
    assert got.shape == (5000,) and got.dtype == torch.float32
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    # CUDA ids: the same scores
    dev = coach.score(T(users), T(items.astype(np.int32)))
    assert torch.equal(dev.view(torch.int32), got.view(torch.int32))
    # within the bound of tests/test_candidates_kernels_gpu.py of the float64 product
    prod = u_embs.double()[T(users)] * i_embs.double()[T(items)]
    D = u_embs.shape[1]
    bound = (3 * 2.0 ** -16 * (1 + 2.0 ** -6) + (3 * D + 8) * 2.0 ** -24 * (1 + 2.0 ** -5)) * prod.abs().sum(1)
    assert bool(((got.double() - prod.sum(1)).abs() <= bound).all())


def test_rank_candidates_equals_numpy_ranking(coach):
    U, I = coach.config.data.user_num, coach.config.data.item_num
    rng = np.random.default_rng(1)
    B, C, n = 64, 150, 40
    users = rng.integers(0, U, B)
    cand = rng.integers(-1, I, (B, C)).astype(np.int64)
    cand[5] = -1                                    # an empty row
    cand[6, 3:] = cand[6, :3].max()                 # fewer distinct candidates than n
    items, scores = coach.rank_candidates(users, cand, n)
    assert items.shape == (B, n) == scores.shape and items.dtype == torch.int64
    items, scores = items.cpu().numpy(), scores.cpu().numpy()
    for b in range(B):
        c = np.unique(cand[b][cand[b] >= 0])
        s = coach.score(np.full(c.size, users[b]), c).cpu().numpy() if c.size else np.zeros(0, np.float32)
        o = np.lexsort((c, -_order_key(s)))[:n]
        want_i = np.full(n, -1)
        want_s = np.full(n, -np.inf, dtype=np.float32)
        want_i[:o.size], want_s[:o.size] = c[o], s[o]
        assert np.array_equal(items[b], want_i), b
        assert np.array_equal(scores[b].view(np.int32), want_s.view(np.int32)), b
    # train items are not excluded: the caller chose the candidates
    h = coach.handler
    ptr, idx = h.train_indptr.cpu().numpy(), h.train_indices.cpu().numpy()
    u0 = int(np.flatnonzero(np.diff(ptr) > 0)[0])
    tr = idx[ptr[u0]:ptr[u0 + 1]]
    got, _ = coach.rank_candidates([u0], tr[None, :], len(tr))
    assert sorted(got[0].tolist()) == sorted(tr.tolist())


def _literal_sampled(coach, n_neg, cutoffs, seed):
    """The sampled protocol, literally: per instance the held-out item's position among its row's candidates under the
    library's pair scores (score desc, item asc), HR / NDCG added instance by instance in float64."""
    from diffmm_b200 import recommend
    h = coach.handler
    users = np.asarray(h.testData.test_users, dtype=np.int64)
    inst, cand = recommend.sampled_candidates(users, h.testData.test_user_its,
                                              (h.train_indptr.cpu().numpy(), h.train_indices.cpu().numpy()),
                                              coach.config.data.item_num, n_neg, seed)
    T_, C = cand.shape
    s = coach.score(np.repeat(inst, C), cand.ravel()).cpu().numpy().reshape(T_, C)
    res = {}
    for K in cutoffs:
        hr, ndcg = 0, 0
        for r in range(T_):
            key = _order_key(s[r])
            pos = int(np.sum((key > key[0]) | ((key == key[0]) & (cand[r] < cand[r, 0]))))
            if pos < K:
                hr += 1.0
                ndcg = ndcg + np.reciprocal(np.log2(pos + 2))
            else:
                hr += 0.0
                ndcg = ndcg + 0.0
        res[f"HR@{K}"], res[f"NDCG@{K}"] = hr / T_, ndcg / T_
    return res, cand


# n_neg = 118: the fewest eligible items of any test user, whose rows then hold every one of them
@pytest.mark.parametrize("n_neg,cutoffs", [(100, (1, 5, 10)), (20, (21, 3, 1)), (118, (50,))])
def test_evaluate_sampled_against_host_literal_loop(coach, n_neg, cutoffs):
    got = coach.evaluate_sampled(n_neg=n_neg, cutoffs=cutoffs, seed=3)
    want, _ = _literal_sampled(coach, n_neg, sorted(set(cutoffs)), seed=3)
    assert got == want
    assert list(got) == [f"{m}@{c}" for c in sorted(set(cutoffs)) for m in ("HR", "NDCG")]
    assert 0 < got[f"HR@{max(cutoffs)}"] <= 1


def test_evaluate_sampled_seeds(coach):
    from diffmm_b200 import recommend
    a = coach.evaluate_sampled(seed=11)
    assert coach.evaluate_sampled(seed=11) == a
    h = coach.handler
    users = np.asarray(h.testData.test_users, dtype=np.int64)
    csr = (h.train_indptr.cpu().numpy(), h.train_indices.cpu().numpy())
    I = coach.config.data.item_num
    _, c1 = recommend.sampled_candidates(users, h.testData.test_user_its, csr, I, 100, 11)
    _, c2 = recommend.sampled_candidates(users, h.testData.test_user_its, csr, I, 100, 12)
    assert np.array_equal(c1[:, 0], c2[:, 0]) and not np.array_equal(c1[:, 1:], c2[:, 1:])
    assert coach.evaluate_sampled(seed=12) == _literal_sampled(coach, 100, (1, 5, 10), 12)[0]


def test_candidate_calls_leave_training_state_alone(coach):
    before = _state(coach)
    coach.evaluate_sampled()
    coach.score([0, 1, 2], [3, 4, 5])
    coach.rank_candidates([0, 1], [[1, 2, 3], [4, -1, 4]], 2)
    _same_state(before, _state(coach))


def test_coach_candidate_calls_reject_bad_arguments(coach):
    I, U = coach.config.data.item_num, coach.config.data.user_num
    for kw in (dict(cutoffs=()), dict(cutoffs=(0,)), dict(n_neg=10, cutoffs=(12,)), dict(cutoffs=(1025,), n_neg=2000),
               dict(n_neg=-1), dict(n_neg=I)):
        with pytest.raises(ValueError):
            coach.evaluate_sampled(**kw)
    with pytest.raises(ValueError):
        coach.score([0, U], [0, 1])
    with pytest.raises(ValueError):
        coach.score([0, 1], [0, I])
    with pytest.raises(ValueError):
        coach.score(T(np.array([0, 1])), T(np.array([0, I])))        # CUDA ids are checked too
    with pytest.raises(ValueError):
        coach.rank_candidates([0, U], [[0], [1]], 1)
    with pytest.raises(ValueError):
        coach.rank_candidates([0, 1], [[0, I], [1, 2]], 1)
    with pytest.raises(ValueError):
        coach.rank_candidates([0, 1], [[0, 1], [1, 2]], 3)
