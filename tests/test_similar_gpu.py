"""Similar items and MMR-diversified lists on a trained Coach (built like tests/test_candidates_gpu.py builds it, on the
tiktok golden data, which has an audio modality):
  * recommend.similar_items is score_topn(unit[q], unit, n, exclude = each query itself) bit for bit, unit = the rows
    normalised by ops.rownorm_fwd; its lists equal a float64 cosine ranking as sets except at near-ties; the query never
    appears and n = I - 1 fills every slot; Coach.similar_items is it on every view's vectors;
  * Coach.recommend_diverse at lam = 1 is Coach.recommend bit for bit; at lam < 1 it is recommend.mmr_rerank of the
    pool (score_topn with the train items excluded) in the view's cosine space, a subset of the pool, no train item;
  * none of them draws random numbers or moves a parameter."""
import json
import os
import random
import shutil

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "epoch_run")
VIEWS = ("final", "image", "text", "audio")


@pytest.fixture(scope="module")
def coach(tmp_path_factory):
    from diffmm_b200 import Main
    from diffmm_b200.Conf import Config
    gold = json.load(open(os.path.join(GOLD, "result.json")))
    tmp = tmp_path_factory.mktemp("similar")
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


def _bits(t):
    return t.view(torch.int32)


def _self_exclude(q):
    Q = q.shape[0]
    rows = torch.arange(Q + 1, dtype=torch.int64, device=q.device)
    return rows, q.to(torch.int32), np.arange(Q)


@pytest.mark.parametrize("view", VIEWS)
def test_similar_items_is_score_topn_with_self_excluded(coach, view):
    from diffmm_b200 import ops, recommend
    I = coach.config.data.item_num
    vecs = coach._view_embs(view)
    q = torch.arange(I, device=vecs.device)                      # every item as a query
    for n in (1, 10, I - 1):
        got_i, got_s = coach.similar_items(q.cpu().numpy(), n, view=view)
        unit, _ = ops.rownorm_fwd(vecs)
        want_i, want_s = recommend.score_topn(unit[q], unit, n, exclude=_self_exclude(q))
        assert torch.equal(got_i, want_i) and torch.equal(_bits(got_s), _bits(want_s)), (view, n)
        assert got_i.dtype == torch.int64 and got_i.shape == (I, n)
        assert not bool((got_i == q[:, None]).any())             # never the query
        assert bool((got_i >= 0).all())                           # n = I - 1 fills every slot
        if n == I - 1:
            assert torch.equal(torch.sort(got_i, 1).values.sum(1), torch.full((I,), I * (I - 1) // 2, device=q.device)
                               - q)
        # CUDA query ids: the same lists
        dev_i, dev_s = coach.similar_items(q, n, view=view)
        assert torch.equal(dev_i, got_i) and torch.equal(_bits(dev_s), _bits(got_s))


@pytest.mark.parametrize("view", VIEWS)
def test_similar_items_against_float64_cosines(coach, view):
    I = coach.config.data.item_num
    x = coach._view_embs(view).double().cpu().numpy()
    u = x / np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-12)
    cos = u @ u.T
    np.fill_diagonal(cos, -np.inf)
    n = 20
    items, scores = coach.similar_items(np.arange(I), n, view=view)
    items, scores = items.cpu().numpy(), scores.cpu().numpy()
    tol = 1e-5
    for q in range(I):
        row = cos[q]
        assert np.all(np.abs(scores[q] - row[items[q]]) <= tol), q
        want = np.argsort(-row, kind="stable")[:n]
        kth = row[want[-1]]
        diff = set(items[q].tolist()) ^ set(want.tolist())
        assert all(abs(row[i] - kth) <= tol for i in diff), (q, diff)     # differ only at near-ties with the n-th


def test_similar_items_fills_a_catalog_and_accepts_unnormalised_rows():
    from diffmm_b200 import recommend
    rng = np.random.default_rng(3)
    I, D = 700, 24
    v = torch.from_numpy(rng.standard_normal((I, D)).astype(np.float32) * 5).cuda()
    q = rng.integers(0, I, 33)
    items, cos = recommend.similar_items(v, q, I - 1)
    items = items.cpu().numpy()
    for r, qq in enumerate(q):
        assert sorted(items[r].tolist()) == [i for i in range(I) if i != qq]
    assert bool((cos[:, :-1] >= cos[:, 1:]).all()) and float(cos.abs().max()) <= 1 + 1e-5
    with pytest.raises(ValueError):
        recommend.similar_items(v, torch.tensor([0, I], device="cuda:0"), 3)     # CUDA ids are checked too


def test_recommend_diverse_lam1_is_recommend(coach):
    U = coach.config.data.user_num
    users = np.arange(0, U, 3)
    for n in (1, 10, 50):
        for view in ("final", "audio"):
            gi, gs = coach.recommend_diverse(users, n, lam=1.0, view=view)
            wi, ws = coach.recommend(users, n)
            assert torch.equal(gi, wi) and torch.equal(_bits(gs), _bits(ws)), (n, view)
            assert gi.dtype == torch.int64


@pytest.mark.parametrize("view", VIEWS)
@pytest.mark.parametrize("lam,n,pool", [(0.5, 10, None), (0.0, 5, 40), (0.3, 20, 200), (0.9, 50, 120)])
def test_recommend_diverse_is_mmr_of_the_pool(coach, view, lam, n, pool):
    from diffmm_b200 import recommend
    U = coach.config.data.user_num
    users = np.arange(U)
    gi, gs = coach.recommend_diverse(users, n, lam=lam, view=view, pool=pool)
    P = pool if pool is not None else min(4 * n, coach.config.data.item_num)
    pi, ps = coach.recommend(users, P)
    wi, ws = recommend.mmr_rerank(coach._item_view(view), pi, ps, n, lam)
    assert torch.equal(gi, wi) and torch.equal(_bits(gs), _bits(ws))
    gi_h, pi_h = gi.cpu().numpy(), pi.cpu().numpy()
    h = coach.handler
    ptr, idx = h.train_indptr.cpu().numpy(), h.train_indices.cpu().numpy()
    for u in users:
        got = gi_h[u][gi_h[u] >= 0]
        assert set(got.tolist()) <= set(pi_h[u].tolist())                    # from the pool
        assert not set(got.tolist()) & set(idx[ptr[u]:ptr[u + 1]].tolist())   # no train item
        assert got.size == min(n, int((pi_h[u] >= 0).sum()))
    # the first pick is the most relevant item at every lam
    assert torch.equal(gi[:, 0], pi[:, 0])


def test_item_view_is_unit_rows(coach):
    for view in VIEWS:
        u = coach._item_view(view)
        assert u.shape == (coach.config.data.item_num, coach.config.base.latdim) and u.dtype == torch.float32
        assert float((u.double().norm(dim=1) - 1).abs().max()) < 1e-5


def test_similarity_calls_leave_training_state_alone(coach):
    before = _state(coach)
    for view in VIEWS:
        coach.similar_items([0, 1, 2], 5, view=view)
        coach.recommend_diverse([0, 1], 5, lam=0.5, view=view)
    recommend_mod = __import__("diffmm_b200.recommend", fromlist=["mmr_rerank"])
    recommend_mod.mmr_rerank(coach._item_view("final"), torch.tensor([[0, 1, -1]], device="cuda:0"),
                             torch.tensor([[0.5, 0.25, 0.0]], device="cuda:0"), 2, 0.5)
    _same_state(before, _state(coach))


def test_mmr_rerank_checks_cuda_input(coach):
    from diffmm_b200 import recommend
    v = coach._item_view("final")
    I = v.shape[0]
    cand = torch.tensor([[0, 1, 2], [3, -1, 4]], device="cuda:0")
    rel = torch.tensor([[0.5, 0.25, 0.0], [1.0, float("nan"), 0.5]], device="cuda:0")
    items, out = recommend.mmr_rerank(v, cand, rel, 3, 0.5)                  # NaN at an empty slot: not read
    assert items[1, 2].item() == -1 and out[1, 2].item() == float("-inf")
    host_i, host_r = recommend.mmr_rerank(v, cand.cpu().numpy(), rel.cpu().numpy(), 3, 0.5)
    assert torch.equal(host_i, items) and torch.equal(_bits(host_r), _bits(out))
    with pytest.raises(ValueError, match="candidates"):
        recommend.mmr_rerank(v, torch.tensor([[0, I]], device="cuda:0"), rel[:1, :2], 1, 0.5)
    with pytest.raises(ValueError, match="relevance"):
        recommend.mmr_rerank(v, cand, torch.tensor([[0.5, float("inf"), 0.0], [1.0, 0.0, 0.5]], device="cuda:0"), 2, 0.5)
