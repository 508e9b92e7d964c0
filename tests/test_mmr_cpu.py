"""Argument checks of the item-similarity surface without a GPU: recommend.mmr_rerank, recommend.similar_items and the
Coach entry points (similar_items, recommend_diverse) raise ValueError for every bad argument before any device call;
CPU tensors that pass every other check are refused last, for not being on a CUDA device."""
import numpy as np
import pytest
import torch

from diffmm_b200 import recommend


def _mmr_args(I=50, D=8, B=3, C=6):
    rng = np.random.default_rng(0)
    return (torch.zeros((I, D)), rng.integers(-1, I, (B, C)).astype(np.int32),
            rng.standard_normal((B, C)).astype(np.float32))


# ------------------------------------------------------------------------------------------------ mmr_rerank
@pytest.mark.parametrize("lam", [-0.01, 1.01, float("nan"), float("inf"), True, "0.5", None])
def test_mmr_rejects_bad_lam(lam):
    v, c, r = _mmr_args()
    with pytest.raises(ValueError, match="lam"):
        recommend.mmr_rerank(v, c, r, 2, lam)


@pytest.mark.parametrize("C,D", [(1025, 8), (513, 64), (129, 256), (33, 1024)])
def test_mmr_rejects_rows_over_the_shared_memory_limit(C, D):
    v, c, r = _mmr_args(D=D, C=C)
    with pytest.raises(ValueError):
        recommend.mmr_rerank(v, c, r, 1, 0.5)


def test_mmr_accepts_the_largest_rows_up_to_the_device_check():
    for C, D in ((512, 64), (1024, 32), (128, 256)):
        v, c, r = _mmr_args(D=D, C=C)
        with pytest.raises(ValueError, match="CUDA"):
            recommend.mmr_rerank(v, c, r, C, 0.5)


@pytest.mark.parametrize("n", [0, 7, -1, 2.0, True])
def test_mmr_rejects_bad_n(n):
    v, c, r = _mmr_args()                               # C = 6
    with pytest.raises(ValueError, match="n must"):
        recommend.mmr_rerank(v, c, r, n, 0.5)


@pytest.mark.parametrize("case", ["vec_f64", "vec_1d", "vec_wide", "vec_empty", "vec_numpy", "cand_float", "cand_1d",
                                  "cand_empty_cols", "rel_f64", "rel_shape", "rel_int", "rel_list"])
def test_mmr_rejects_bad_dtypes_and_ranks(case):
    v, c, r = _mmr_args()
    if case == "vec_f64":
        v = v.double()
    elif case == "vec_1d":
        v = v[0]
    elif case == "vec_wide":
        v = torch.zeros((50, 257))
    elif case == "vec_empty":
        v = torch.zeros((0, 8))
    elif case == "vec_numpy":
        v = v.numpy()
    elif case == "cand_float":
        c = c.astype(np.float32)
    elif case == "cand_1d":
        c = c[0]
    elif case == "cand_empty_cols":
        c, r = c[:, :0], r[:, :0]
    elif case == "rel_f64":
        r = r.astype(np.float64)
    elif case == "rel_shape":
        r = r[:, :5]
    elif case == "rel_int":
        r = torch.zeros(c.shape, dtype=torch.int32)
    else:
        r = r.tolist()
    with pytest.raises(ValueError):
        recommend.mmr_rerank(v, c, r, 2, 0.5)


@pytest.mark.parametrize("bad", [50, -2, 2 ** 32 + 5, -2 ** 32 + 3, 2 ** 31])
def test_mmr_rejects_out_of_range_candidates(bad):
    v, c, r = _mmr_args()
    c = c.astype(np.int64)                              # ids outside the int32 range must not wrap into 0..I-1
    c[1, 2] = bad
    with pytest.raises(ValueError, match="candidates"):
        recommend.mmr_rerank(v, c, r, 2, 0.5)


@pytest.mark.parametrize("x", [np.nan, np.inf, -np.inf])
def test_mmr_rejects_non_finite_relevance_at_candidates_only(x):
    v, c, r = _mmr_args()
    c[0, 0] = 4
    r[0, 0] = x
    with pytest.raises(ValueError, match="relevance"):
        recommend.mmr_rerank(v, c, r, 2, 0.5)
    c[0, 0] = -1                                        # an empty slot's relevance is never read
    with pytest.raises(ValueError, match="CUDA"):
        recommend.mmr_rerank(v, c, r, 2, 0.5)


# ------------------------------------------------------------------------------------------------ similar_items
@pytest.mark.parametrize("n", [0, 50, 1025, 2.0, True])
def test_similar_items_rejects_bad_n(n):
    with pytest.raises(ValueError, match="n must"):
        recommend.similar_items(torch.zeros((50, 8)), [0, 1], n)          # n <= I - 1 = 49


def test_similar_items_n_capped_at_1024():
    v = torch.zeros((2000, 8))
    with pytest.raises(ValueError, match="n must"):
        recommend.similar_items(v, [0], 1025)
    with pytest.raises(ValueError, match="CUDA"):
        recommend.similar_items(v, [0], 1024)


@pytest.mark.parametrize("case", ["vec_f64", "vec_1d", "vec_empty", "items_2d", "items_float", "items_range",
                                  "items_negative", "precision"])
def test_similar_items_rejects_bad_arguments(case):
    v, items, kw = torch.zeros((50, 8)), [0, 3], {}
    if case == "vec_f64":
        v = v.double()
    elif case == "vec_1d":
        v = v[0]
    elif case == "vec_empty":
        v = torch.zeros((0, 8))
    elif case == "items_2d":
        items = [[0, 3]]
    elif case == "items_float":
        items = [0.0, 3.0]
    elif case == "items_range":
        items = [0, 50]
    elif case == "items_negative":
        items = [-1, 3]
    else:
        kw = dict(precision="fp32")
    with pytest.raises(ValueError):
        recommend.similar_items(v, items, 2, **kw)


# ------------------------------------------------------------------------------------------------ Coach
class _Handler:
    def __init__(self, has_audio):
        self.has_audio = has_audio


def _coach(has_audio):
    """A Coach shell with a config and a handler only: enough for every argument check, no model, no device."""
    from diffmm_b200 import Main
    from diffmm_b200.Conf import Config
    c = object.__new__(Main.Coach)
    c.config = Config()
    c.config.data.user_num, c.config.data.item_num = 30, 700
    c.handler = _Handler(has_audio)
    return c


@pytest.mark.parametrize("view", ["finale", "IMAGE", "", None, 0])
def test_coach_rejects_unknown_view(view):
    c = _coach(True)
    with pytest.raises(ValueError, match="view"):
        c.similar_items([0], 5, view=view)
    with pytest.raises(ValueError, match="view"):
        c.recommend_diverse([0], 5, view=view)


def test_coach_rejects_audio_without_audio_features():
    c = _coach(False)
    with pytest.raises(ValueError, match="audio"):
        c.similar_items([0], 5, view="audio")
    with pytest.raises(ValueError, match="audio"):
        c.recommend_diverse([0], 5, view="audio")
    with pytest.raises(ValueError, match="audio"):
        c._item_view("audio")


@pytest.mark.parametrize("kw", [dict(n=0), dict(n=513), dict(n=5, pool=4), dict(n=5, pool=513), dict(n=5, lam=-0.5),
                                dict(n=5, lam=float("nan")), dict(n=5, pool=10.0), dict(n=5.0)])
def test_coach_recommend_diverse_rejects_bad_sizes(kw):
    c = _coach(False)                                   # latdim 64: pool <= min(700, 32768 // 64, 1024) = 512
    with pytest.raises(ValueError):
        c.recommend_diverse([0, 1], **kw)


@pytest.mark.parametrize("users", [[0, 30], [-1], [[0]], [0.5]])
def test_coach_recommend_diverse_rejects_bad_users(users):
    with pytest.raises(ValueError, match="users"):
        _coach(False).recommend_diverse(users, 5)
