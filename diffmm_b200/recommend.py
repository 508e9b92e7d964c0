"""Ranked top-N recommendation lists on the device.

``score_topn`` turns user and item embeddings into the N best items per user, in rank order, with their scores:
the score contraction of the evaluation (Main.py:410, bf16x3 on tcgen05) also writes the per-32-column chunk maxima,
the excluded items are overwritten with -inf and their chunk maxima refreshed (dmm_eval_mask_scores_cmax), the pruned
top-k selects the N best columns reading only the chunks that can hold them (for rows of at least 4 N chunks; shorter
rows take the whole-row top-k without chunk maxima), and dmm_topn_rank puts them into rank order: score descending,
then item id ascending (the tie order of the library's top-k).  Users are processed in chunks whose score block stays
under 1 GB, like ``Coach.testEpoch``.  Host data enters through pinned buffers with asynchronous copies, so the call
does not wait for work already queued on the stream.
"""
from __future__ import annotations

import numbers
from typing import Tuple

import numpy as np
import torch

from . import ops

MAX_N = 1024          # longest ranked list (dmm_topn_rank / dmm_eval_metrics_cutoffs)
# score_topn takes the pruned top-k when a row has at least PRUNE_RATIO * n chunks of 32 columns, the whole-row top-k
# otherwise.  Chosen from tools/bench_recommend.py on a B200 at 1000 W (DESIGN §7, profiles/r03_recommend.json): the
# pruned path lost at 0.22, 0.57 and 2.2 chunks per listed item, won at 5.7, 29 and 156, and was within the run-to-run
# spread at 11.  The value equals the PRUNE_RATIO of csrc/topk.cu below which the pruned kernel defers a row (k <= 64)
# to its slower second pass; keep the two together.
PRUNE_RATIO = 4


def to_device(a: np.ndarray, device) -> torch.Tensor:
    """Host array -> device tensor through a pinned staging buffer: the copy is queued on the current stream without
    waiting for the work before it (torch keeps the pinned buffer alive until the copy has run)."""
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().to(device, non_blocking=True)


def user_chunk(n_items: int) -> int:
    """Users per score block: 1 GB of fp32 scores, clamped to [256, 8192] (the rule of Coach.testEpoch)."""
    return int(max(256, min(8192, (1 << 30) // (4 * max(n_items, 1)))))


def check_n(n, n_items: int) -> int:
    if isinstance(n, bool) or not isinstance(n, numbers.Integral):
        raise ValueError(f"n must be an int, got {n!r}")
    n = int(n)
    if n < 1 or n > MAX_N:
        raise ValueError(f"n must be in 1..{MAX_N}, got {n}")
    if n > n_items:
        raise ValueError(f"n = {n} exceeds the number of items ({n_items})")
    return n


def check_cutoffs(cutoffs, n_items: int) -> list:
    """Sorted distinct cutoffs; each must be an int in 1..min(1024, n_items)."""
    try:
        cuts = list(cutoffs)
    except TypeError:
        raise ValueError(f"cutoffs must be a sequence of ints, got {cutoffs!r}") from None
    if not cuts:
        raise ValueError("cutoffs must not be empty")
    for c in cuts:
        if isinstance(c, bool) or not isinstance(c, numbers.Integral):
            raise ValueError(f"cutoffs must be ints, got {c!r}")
        if c < 1 or c > MAX_N or c > n_items:
            raise ValueError(f"cutoff {c} outside 1..{min(MAX_N, n_items)} (at most {MAX_N} and the number of items)")
    return sorted({int(c) for c in cuts})


def _check_embs(user_embs, item_embs):
    for name, t in (("user_embs", user_embs), ("item_embs", item_embs)):
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or t.dim() != 2:
            raise ValueError(f"{name} must be a 2-D float32 tensor, got "
                             f"{getattr(t, 'dtype', type(t).__name__)} {tuple(getattr(t, 'shape', ()))}")
    if user_embs.shape[1] != item_embs.shape[1]:
        raise ValueError(f"embedding widths differ: user_embs {tuple(user_embs.shape)}, item_embs {tuple(item_embs.shape)}")
    if item_embs.shape[0] < 1:
        raise ValueError("item_embs has no rows")


def _check_exclude(exclude, n_users: int, device):
    """(indptr, indices, row_ids) -> (indptr, indices, host int64 row ids); the row ids are checked on the host."""
    try:
        indptr, indices, row_ids = exclude
    except (TypeError, ValueError):
        raise ValueError("exclude must be an (indptr, indices, row_ids) tuple") from None
    if not isinstance(indptr, torch.Tensor) or indptr.dtype != torch.int64 or indptr.dim() != 1 or indptr.numel() < 1:
        raise ValueError("exclude indptr must be a 1-D int64 tensor with at least one entry")
    if not isinstance(indices, torch.Tensor) or indices.dtype != torch.int32 or indices.dim() != 1:
        raise ValueError("exclude indices must be a 1-D int32 tensor")
    if indptr.device != device or indices.device != device:
        raise ValueError(f"exclude indptr / indices must be on {device}")
    if isinstance(row_ids, torch.Tensor) and row_ids.is_cuda:
        raise ValueError("exclude row_ids must be host data (checked against the CSR before any launch)")
    rid = np.asarray(row_ids.numpy() if isinstance(row_ids, torch.Tensor) else row_ids)
    if rid.ndim != 1 or rid.shape[0] != n_users or (rid.size and rid.dtype.kind not in "iu"):
        raise ValueError(f"exclude row_ids must be {n_users} integers (one per user row)")
    n_rows = indptr.numel() - 1
    if rid.size and (rid.min() < 0 or rid.max() >= n_rows):
        raise ValueError(f"exclude row_ids out of range 0..{n_rows - 1}")
    return indptr, indices, torch.from_numpy(rid.astype(np.int64))


def score_topn(user_embs: torch.Tensor, item_embs: torch.Tensor, n: int, *, exclude=None,
               precision: str = "bf16x3") -> Tuple[torch.Tensor, torch.Tensor]:
    """The n best items of every user, in rank order.

    user_embs fp32 [B, D], item_embs fp32 [I, D] (CUDA); score = user . item in ``precision`` ("bf16x3": the evaluation's
    fp32-faithful split-bf16 contraction, or single-pass "bf16").  exclude = (indptr int64, indices int32, row_ids): a
    CSR whose row row_ids[b] lists the items user row b must not be recommended (e.g. its train items); row_ids is host
    data (list / numpy / CPU tensor).  Returns (items int64 [B, n], scores fp32 [B, n]) on the device, score descending
    then item id ascending; when fewer than n items are left, the tail holds item -1 with score -inf."""
    if precision not in ("bf16", "bf16x3"):
        raise ValueError(f"precision must be 'bf16' or 'bf16x3', got {precision!r}")
    _check_embs(user_embs, item_embs)
    n = check_n(n, item_embs.shape[0])
    if exclude is not None:
        exclude = _check_exclude(exclude, user_embs.shape[0], user_embs.device)
    if not (user_embs.is_cuda and item_embs.is_cuda) or user_embs.device != item_embs.device:
        raise ValueError(f"user_embs and item_embs must be CUDA tensors on one device, got {user_embs.device} and "
                         f"{item_embs.device}")
    with torch.cuda.device(user_embs.device):
        if exclude is not None:
            exclude = (exclude[0], exclude[1], to_device(exclude[2].numpy(), user_embs.device))
        items, scores = _topn(user_embs, item_embs, n, exclude, float("-inf"), precision)
        return items.long(), scores


def _topn(user_embs, item_embs, n, exclude, fill, precision):
    """score_topn without the argument checks: int32 items.  exclude = (indptr, indices, device int64 row ids)."""
    dev = user_embs.device
    B, D = user_embs.shape
    I = item_embs.shape[0]
    split = precision == "bf16x3"
    b_hi, b_lo = ops.pack_bf16(item_embs.contiguous(), split=split)       # once per call
    items = torch.empty((B, n), dtype=torch.int32, device=dev)
    scores = torch.empty((B, n), dtype=torch.float32, device=dev)
    if B == 0:
        return items, scores
    chunk = min(user_chunk(I), B)
    ld = ops.pad_to(I, 4)
    block = torch.empty((chunk, ld), dtype=torch.float32, device=dev)
    # The pruned top-k reads n chunks of 32 scores per row instead of the row: faster while those chunks are a small part
    # of the row, slower beyond (PRUNE_RATIO).  Both select the same columns, bit for bit.
    prune = PRUNE_RATIO * n <= (I + 31) // 32
    cmax = ops.cmax_buffer(chunk, I, dev) if prune else None
    sel = torch.empty(chunk * n, dtype=torch.int32, device=dev)
    kptr = torch.arange(chunk + 1, dtype=torch.int64, device=dev) * n        # k = n for every row
    for s in range(0, B, chunk):
        b = min(chunk, B - s)
        sc = block[:b, :I]
        cm = cmax[:b] if prune else None
        a_hi, a_lo = ops.pack_bf16(user_embs[s:s + b].contiguous(), split=split)
        ops.gemm_bf16_tn(a_hi, a_lo, b_hi, b_lo, b, I, D, out_f32=sc, cmax=cm)
        if exclude is not None:
            indptr, indices, rid = exclude
            if prune:
                ops.eval_mask_scores_cmax(indptr, indices, rid[s:s + b], sc, I, cm, fill)
            else:
                ops.eval_mask_scores(indptr, indices, rid[s:s + b], sc, I, fill)
        if prune:
            ops.topk_edges_pruned(sc, I, cm, kptr, 0, None, sel[:b * n])
        else:
            ops.topk_edges(sc, I, kptr, 0, None, sel[:b * n])
        ops.topn_rank(sc, sel[:b * n].view(b, n), n, items[s:s + b], scores[s:s + b])
    return items, scores


def metric_tables(n: int):
    """Host float64 tables of calcRes (Main.py:422-448) up to list length n: inv_log2[p] = 1 / log2(p + 2) (p < n) and
    max_dcg[t] = the sum of its first t entries (t <= n), evaluated with the same numpy expressions as Coach.calcRes."""
    inv = [np.reciprocal(np.log2(p + 2)) for p in range(n)]
    max_dcg = [float(np.sum(inv[:t])) for t in range(n + 1)]
    return np.array(inv, dtype=np.float64), np.array(max_dcg, dtype=np.float64)


def heldout_csr(users: np.ndarray, test_user_its, n_users: int):
    """(indptr int64 [n_users + 1], items int32): the test items of each of `users` (distinct ids) in stored order; every
    other user has none."""
    tptr = np.zeros(n_users + 1, dtype=np.int64)
    for u in users:
        tptr[u + 1] = len(test_user_its[u])
    np.cumsum(tptr, out=tptr)
    titems = np.fromiter((it for u in np.sort(users) for it in test_user_its[u]), dtype=np.int32, count=int(tptr[-1]))
    return tptr, titems
