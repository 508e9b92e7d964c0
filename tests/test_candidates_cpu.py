"""Argument checks of the pair-score / candidate-ranking surface (recommend.score_pairs, recommend.rank_candidates) and
the host-side sampled-negative rows (recommend.sampled_candidates), without a GPU: every bad argument raises ValueError
before any device call (CPU tensors that pass every other check are refused last, for not being on a CUDA device)."""
import random

import numpy as np
import pytest
import torch

from diffmm_b200 import recommend


def _embs(B=4, I=50, D=8, dtype=torch.float32):
    return torch.zeros((B, D), dtype=dtype), torch.zeros((I, D), dtype=dtype)


# ------------------------------------------------------------------------------------------------ score_pairs
@pytest.mark.parametrize("case", ["user_f64", "item_bf16", "user_1d", "width", "no_items", "not_tensor"])
def test_score_pairs_rejects_bad_embeddings(case):
    u, i = _embs()
    if case == "user_f64":
        u = u.double()
    elif case == "item_bf16":
        i = i.bfloat16()
    elif case == "user_1d":
        u = u[0]
    elif case == "width":
        i = torch.zeros((50, 9))
    elif case == "no_items":
        i = torch.zeros((0, 8))
    else:
        u = u.numpy()
    with pytest.raises(ValueError):
        recommend.score_pairs(u, i, [0, 1], [0, 1])


@pytest.mark.parametrize("users,items,match", [
    ([0, 4], [0, 1], "users"),              # user id = B
    ([-1, 0], [0, 1], "users"),
    ([0, 1], [0, 50], "items"),             # item id = I
    ([0, 1], [-2, 0], "items"),
    ([0, 1, 2], [0, 1], "length"),
    ([[0, 1]], [[0, 1]], "users"),          # 2-D
    ([0.0, 1.0], [0, 1], "users"),          # float ids
    ([0, 1], np.array([0.5, 1.0]), "items"),
    (torch.tensor([0, 1], dtype=torch.float32), [0, 1], "users"),
    (torch.tensor([True, False]), [0, 1], "users"),
])
def test_score_pairs_rejects_bad_ids(users, items, match):
    u, i = _embs()
    with pytest.raises(ValueError, match=match):
        recommend.score_pairs(u, i, users, items)


def test_score_pairs_rejects_bad_precision():
    u, i = _embs()
    with pytest.raises(ValueError, match="precision"):
        recommend.score_pairs(u, i, [0], [0], precision="fp32")


def test_score_pairs_refuses_host_tensors_last():
    u, i = _embs()
    with pytest.raises(ValueError, match="CUDA"):
        recommend.score_pairs(u, i, torch.tensor([0, 3]), np.array([49, 0], dtype=np.uint16))


# ------------------------------------------------------------------------------------------------ rank_candidates
def test_rank_candidates_rejects_bad_embeddings():
    u, i = _embs()
    with pytest.raises(ValueError):
        recommend.rank_candidates(u.double(), i, np.zeros((4, 3), dtype=np.int32), 2)
    with pytest.raises(ValueError):
        recommend.rank_candidates(u, torch.zeros((50, 7)), np.zeros((4, 3), dtype=np.int32), 2)


@pytest.mark.parametrize("cand,match", [
    (np.zeros((3, 5), dtype=np.int32), "rows"),                 # B != user rows
    (np.zeros(5, dtype=np.int32), "2-D"),
    (np.zeros((4, 5), dtype=np.float32), "integer"),
    (np.zeros((4, 0), dtype=np.int32), "columns"),              # C = 0
    (np.zeros((4, 4097), dtype=np.int32), "columns"),           # C > MAX_CANDIDATES
    (np.full((4, 5), 50, dtype=np.int32), "candidates"),        # item id = I
    (np.full((4, 5), -2, dtype=np.int64), "candidates"),        # only -1 marks an empty slot
])
def test_rank_candidates_rejects_bad_candidates(cand, match):
    u, i = _embs()
    with pytest.raises(ValueError, match=match):
        recommend.rank_candidates(u, i, cand, 2)


@pytest.mark.parametrize("n", [0, -1, 6, 1025, 2.0, True, None])
def test_rank_candidates_rejects_bad_n(n):
    u, i = _embs()
    with pytest.raises(ValueError, match="n must"):
        recommend.rank_candidates(u, i, np.zeros((4, 5), dtype=np.int32), n)       # n > C = 5 among them


def test_rank_candidates_n_capped_at_1024():
    u, i = _embs(I=5000)
    cand = np.zeros((4, 2000), dtype=np.int32)
    with pytest.raises(ValueError, match="n must"):
        recommend.rank_candidates(u, i, cand, 1025)
    with pytest.raises(ValueError, match="CUDA"):          # n = 1024 <= C passes every check but the device one
        recommend.rank_candidates(u, i, cand, 1024)


def test_rank_candidates_rejects_bad_precision():
    u, i = _embs()
    with pytest.raises(ValueError, match="precision"):
        recommend.rank_candidates(u, i, np.zeros((4, 5), dtype=np.int32), 2, precision="x3")


def test_rank_candidates_refuses_host_tensors_last():
    u, i = _embs()
    cand = torch.tensor([[-1, 0, 49, 49]] * 4, dtype=torch.int64)
    with pytest.raises(ValueError, match="CUDA"):
        recommend.rank_candidates(u, i, cand, 4)


def test_max_candidates():
    assert recommend.MAX_CANDIDATES == 4096


# ------------------------------------------------------------------------------------------------ sampled_candidates
def _world(seed=0, U=40, I=300, n_test=(0, 1, 2, 5)):
    """A random train CSR and test lists (some test items are train items too; some users have no test items)."""
    rng = np.random.default_rng(seed)
    train = [np.sort(rng.choice(I, int(rng.integers(0, 60)), replace=False)) for _ in range(U)]
    test = []
    for u in range(U):
        k = int(n_test[u % len(n_test)])
        t = list(rng.choice(I, k, replace=False))
        if k and len(train[u]) and u % 3 == 0:
            t[0] = int(train[u][0])
        test.append(t if k else None)
    ptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum([len(x) for x in train], out=ptr[1:])
    idx = np.concatenate(train).astype(np.int32)
    users = np.array([u for u in rng.permutation(U) if test[u] is not None], dtype=np.int64)
    return users, test, (ptr, idx), I, train


def _rng_states():
    return (torch.get_rng_state(), np.random.get_state(), random.getstate())


@pytest.mark.parametrize("n_neg", [0, 1, 10, 100])
def test_sampled_candidates_rows(n_neg):
    users, test, csr, I, train = _world()
    before = _rng_states()
    inst, cand = recommend.sampled_candidates(users, test, csr, I, n_neg, seed=7)
    after = _rng_states()
    assert torch.equal(before[0], after[0])
    assert before[1][0] == after[1][0] and np.array_equal(before[1][1], after[1][1]) and before[1][2:] == after[1][2:]
    assert before[2] == after[2]
    assert inst.dtype == np.int64 and cand.dtype == np.int32 and cand.shape == (len(inst), 1 + n_neg)
    # instances in users order, then each user's stored test order; column 0 is the held-out item
    want_u = [u for u in users for _ in test[u]]
    want_p = [it for u in users for it in test[u]]
    assert inst.tolist() == want_u and cand[:, 0].tolist() == want_p
    for r, u in enumerate(inst):
        neg = cand[r, 1:]
        assert len(set(neg.tolist())) == n_neg                           # no duplicates
        assert np.all(np.diff(neg) > 0) if n_neg > 1 else True
        assert not set(neg.tolist()) & (set(train[u].tolist()) | set(test[u]))
        assert np.all((neg >= 0) & (neg < I))
    # deterministic for a seed, different for another
    inst2, cand2 = recommend.sampled_candidates(list(users), test, (torch.from_numpy(csr[0]), torch.from_numpy(csr[1])),
                                                I, n_neg, seed=7)
    assert np.array_equal(inst, inst2) and np.array_equal(cand, cand2)
    if n_neg:
        _, cand3 = recommend.sampled_candidates(users, test, csr, I, n_neg, seed=8)
        assert not np.array_equal(cand, cand3)


def test_sampled_candidates_takes_every_eligible_item():
    """n_neg = the number of eligible items: every row holds exactly the user's eligible items (the redraw loop ends)."""
    users, test, csr, I, train = _world(seed=3, U=12, I=90, n_test=(1, 3))
    n_ok = min(I - len(set(train[u].tolist()) | set(test[u])) for u in users)
    inst, cand = recommend.sampled_candidates(users, test, csr, I, n_ok, seed=1)
    for r, u in enumerate(inst):
        eligible = sorted(set(range(I)) - set(train[u].tolist()) - set(test[u]))
        if len(eligible) == n_ok:
            assert cand[r, 1:].tolist() == eligible
        else:
            assert set(cand[r, 1:].tolist()) <= set(eligible)


def test_sampled_candidates_uniform():
    """Every eligible item is drawn about equally often (a chi-square bound far beyond its 1e-6 quantile fails)."""
    I = 40
    test = [[10, 11]]
    csr = (np.array([0, 10], dtype=np.int64), np.arange(10, dtype=np.int32))
    counts = np.zeros(I, dtype=np.int64)
    for s in range(400):
        _, cand = recommend.sampled_candidates([0], test, csr, I, 7, seed=s)
        np.add.at(counts, cand[:, 1:].ravel(), 1)
    assert counts[:12].sum() == 0
    obs = counts[12:]
    exp = obs.sum() / obs.size
    chi2 = float(((obs - exp) ** 2 / exp).sum())
    assert chi2 < 80, chi2          # 27 degrees of freedom: P(chi2 > 80) < 1e-6


def test_sampled_candidates_rejects():
    users, test, csr, I, _ = _world()
    with pytest.raises(ValueError, match="fewer than"):
        recommend.sampled_candidates(users, test, csr, I, I - 1, seed=0)
    for n_neg in (-1, 4096, 2.0, True):
        with pytest.raises(ValueError, match="n_neg"):
            recommend.sampled_candidates(users, test, csr, I, n_neg, seed=0)
    with pytest.raises(ValueError, match="users"):
        recommend.sampled_candidates(np.array([len(test)]), test, csr, I, 5, seed=0)
    with pytest.raises(ValueError, match="users"):
        recommend.sampled_candidates(np.array([0.0]), test, csr, I, 5, seed=0)
    with pytest.raises(ValueError, match="n_items"):
        recommend.sampled_candidates(users, test, csr, 0, 5, seed=0)
    with pytest.raises(ValueError, match="train"):
        recommend.sampled_candidates(users, test, csr, 10, 5, seed=0)     # train ids beyond n_items
    bad = list(test)
    u0 = int(users[0])
    bad[u0] = [I]
    with pytest.raises(ValueError, match="test items"):
        recommend.sampled_candidates(users, bad, csr, I, 5, seed=0)
    with pytest.raises(ValueError, match="train_csr"):
        recommend.sampled_candidates(users, test, csr[0], I, 5, seed=0)
