"""Argument checks of the recommendation surface (diffmm_b200.recommend): every bad argument raises ValueError before
any device call, so these run without a GPU (CPU tensors that pass every other check are refused last, for not being
on a CUDA device)."""
import numpy as np
import pytest
import torch

from diffmm_b200 import recommend


def _embs(B=4, I=50, D=8, dtype=torch.float32):
    return torch.zeros((B, D), dtype=dtype), torch.zeros((I, D), dtype=dtype)


def _csr(U=4, I=50):
    return torch.zeros(U + 1, dtype=torch.int64), torch.zeros(0, dtype=torch.int32)


@pytest.mark.parametrize("n", [0, -1, 1025, 51, 2.0, True, None])
def test_score_topn_rejects_bad_n(n):
    u, i = _embs()
    with pytest.raises(ValueError, match="n"):
        recommend.score_topn(u, i, n)


@pytest.mark.parametrize("case", ["user_f64", "item_bf16", "user_1d", "width", "no_items", "not_tensor"])
def test_score_topn_rejects_bad_embeddings(case):
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
        recommend.score_topn(u, i, 5)


def test_score_topn_rejects_bad_precision():
    u, i = _embs()
    with pytest.raises(ValueError, match="precision"):
        recommend.score_topn(u, i, 5, precision="fp32")


@pytest.mark.parametrize("rows", [[0, 1, 2, 4], [-1, 0, 1, 2], [0, 1, 2], [[0, 1, 2, 3]], [0.0, 1.0, 2.0, 3.0],
                                  "cuda_only"])
def test_score_topn_rejects_bad_exclusion_rows(rows):
    u, i = _embs()
    ptr, idx = _csr()
    if rows == "cuda_only":
        if not torch.cuda.is_available():
            pytest.skip("needs a CUDA tensor to pass")
        rows = torch.zeros(4, dtype=torch.int64, device="cuda")
    with pytest.raises(ValueError, match="row_ids"):
        recommend.score_topn(u, i, 5, exclude=(ptr, idx, rows))


def test_score_topn_rejects_bad_exclusion_csr():
    u, i = _embs()
    ptr, idx = _csr()
    with pytest.raises(ValueError, match="indptr"):
        recommend.score_topn(u, i, 5, exclude=(ptr.int(), idx, [0, 1, 2, 3]))
    with pytest.raises(ValueError, match="indices"):
        recommend.score_topn(u, i, 5, exclude=(ptr, idx.long(), [0, 1, 2, 3]))
    with pytest.raises(ValueError, match="tuple"):
        recommend.score_topn(u, i, 5, exclude=(ptr, idx))


def test_score_topn_refuses_host_tensors_last():
    u, i = _embs()
    ptr, idx = _csr()
    with pytest.raises(ValueError, match="CUDA"):
        recommend.score_topn(u, i, 5, exclude=(ptr, idx, np.arange(4)))


@pytest.mark.parametrize("cutoffs", [(), [0], [10, -2], [1025], [51], [10, 2.5], [True], 20, None])
def test_cutoffs_rejected(cutoffs):
    with pytest.raises(ValueError):
        recommend.check_cutoffs(cutoffs, 50)


def test_cutoffs_sorted_and_deduplicated():
    assert recommend.check_cutoffs((50, 10, 20, 10), 50) == [10, 20, 50]
    assert recommend.check_cutoffs([np.int64(3)], 50) == [3]
    assert recommend.check_cutoffs(range(1, 1025), 2000) == list(range(1, 1025))


def test_metric_tables_match_calcres_expressions():
    inv, max_dcg = recommend.metric_tables(40)
    assert inv.shape == (40,) and max_dcg.shape == (41,)
    for t in range(41):     # Coach.calcRes' table, expression for expression
        assert max_dcg[t] == np.sum([np.reciprocal(np.log2(loc + 2)) for loc in range(t)])
    assert np.array_equal(inv, np.array([np.reciprocal(np.log2(p + 2)) for p in range(40)]))
