"""Ranked top-N recommendation lists on the device.

``score_topn`` turns user and item embeddings into the N best items per user, in rank order, with their scores:
the score contraction of the evaluation (Main.py:410, bf16x3 on tcgen05) also writes the per-32-column chunk maxima,
the excluded items are overwritten with -inf and their chunk maxima refreshed (dmm_eval_mask_scores_cmax), the pruned
top-k selects the N best columns reading only the chunks that can hold them (for rows of at least 4 N chunks; shorter
rows take the whole-row top-k without chunk maxima), and dmm_topn_rank puts them into rank order: score descending,
then item id ascending (the tie order of the library's top-k).  Users are processed in chunks whose score block stays
under 1 GB, like ``Coach.testEpoch``.  Host data enters through pinned buffers with asynchronous copies, so the call
does not wait for work already queued on the stream.

``score_pairs`` scores given (user, item) pairs and ``rank_candidates`` ranks a given candidate list per user, both
without the full contraction (dmm_score_pairs / dmm_rank_candidates): the same split-bf16 terms, summed in fp32 in a
fixed order, so a pair gets the same bits from both, though not score_topn's bits (the contraction sums in another
order).  ``sampled_candidates`` builds the rows of the sampled-negative evaluation protocol (one held-out item against
n_neg sampled negatives) on the host.
"""
from __future__ import annotations

import numbers
from typing import Tuple

import numpy as np
import torch

from . import ops

MAX_N = 1024          # longest ranked list (dmm_topn_rank / dmm_eval_metrics_cutoffs)
MAX_CANDIDATES = 4096  # longest candidate row of rank_candidates (dmm_rank_candidates: one row's keys in 32 KB of shared memory)
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


def _check_precision(precision):
    if precision not in ("bf16", "bf16x3"):
        raise ValueError(f"precision must be 'bf16' or 'bf16x3', got {precision!r}")


def _check_on_device(user_embs, item_embs):
    if not (user_embs.is_cuda and item_embs.is_cuda) or user_embs.device != item_embs.device:
        raise ValueError(f"user_embs and item_embs must be CUDA tensors on one device, got {user_embs.device} and "
                         f"{item_embs.device}")


def _ids(a, name: str, ndim: int):
    """Integer ids as a host numpy array or a CUDA tensor (left where they are), checked for rank and dtype."""
    if isinstance(a, torch.Tensor):
        if a.dim() != ndim or a.dtype.is_floating_point or a.dtype.is_complex or a.dtype == torch.bool:
            raise ValueError(f"{name} must be a {ndim}-D integer array, got {a.dtype} {tuple(a.shape)}")
        return a if a.is_cuda else a.numpy()
    arr = np.asarray(a)
    if arr.ndim != ndim or (arr.size and arr.dtype.kind not in "iu"):
        raise ValueError(f"{name} must be a {ndim}-D integer array, got {arr.dtype} {arr.shape}")
    return arr


def _check_ranges(checks):
    """checks: [(ids, lo, hi, name)]: every id in [lo, hi].  Host arrays are checked on the host; the CUDA tensors are
    reduced on the device and read back together (one synchronisation)."""
    dev = [(a, lo, hi, name) for a, lo, hi, name in checks if isinstance(a, torch.Tensor) and a.numel()]
    host = [(a, lo, hi, name) for a, lo, hi, name in checks if not isinstance(a, torch.Tensor) and a.size]
    bounds = [(int(a.min()), int(a.max())) for a, *_ in host]
    if dev:
        mm = torch.stack([torch.stack([a.min(), a.max()]).long() for a, *_ in dev]).cpu().tolist()
        bounds += mm
    for (mn, mx), (_, lo, hi, name) in zip(bounds, host + dev):
        if mn < lo or mx > hi:
            raise ValueError(f"{name} out of range {lo}..{hi} (found {mn}..{mx})")


def _to(a, device, dtype) -> torch.Tensor:
    """Checked ids -> contiguous device tensor of `dtype` (host data through to_device)."""
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=dtype).contiguous()
    return to_device(a.astype({torch.int32: np.int32, torch.int64: np.int64}[dtype]), device)


def score_pairs(user_embs: torch.Tensor, item_embs: torch.Tensor, users, items, precision: str = "bf16x3") -> torch.Tensor:
    """Scores of given pairs: out[p] = user_embs[users[p]] . item_embs[items[p]] (fp32 [P] on the device).

    users, items: 1-D integer arrays of equal length, host data (list / numpy / CPU tensor) or CUDA tensors on the
    embeddings' device.  Every id is checked before any launch; for CUDA ids that costs one device synchronisation.
    precision: "bf16x3" = sum over d of hi_u hi_i + hi_u lo_i + lo_u hi_i with hi = bf16(x), lo = bf16(x - hi) (the
    evaluation's fp32-faithful split), "bf16" = sum of hi_u hi_i; fp32 sums in a fixed order, the same bits as
    ``rank_candidates`` gives the pair, but not bit-identical to ``score_topn`` (its contraction sums in another order)."""
    _check_precision(precision)
    _check_embs(user_embs, item_embs)
    u = _ids(users, "users", 1)
    i = _ids(items, "items", 1)
    if u.shape[0] != i.shape[0]:
        raise ValueError(f"users and items differ in length ({u.shape[0]} vs {i.shape[0]})")
    check = [(u, 0, user_embs.shape[0] - 1, "users"), (i, 0, item_embs.shape[0] - 1, "items")]
    on_dev = any(isinstance(a, torch.Tensor) for a in (u, i))
    if not on_dev:
        _check_ranges(check)
    _check_on_device(user_embs, item_embs)
    for name, a in (("users", u), ("items", i)):
        if isinstance(a, torch.Tensor) and a.device != user_embs.device:
            raise ValueError(f"{name} is on {a.device}, the embeddings on {user_embs.device}")
    with torch.cuda.device(user_embs.device):
        if on_dev:
            _check_ranges(check)
        dev = user_embs.device
        out = torch.empty(u.shape[0], dtype=torch.float32, device=dev)
        if u.shape[0]:
            ops.score_pairs(user_embs, item_embs, _to(u, dev, torch.int64), _to(i, dev, torch.int32),
                            precision == "bf16x3", out)
        return out


def rank_candidates(user_embs: torch.Tensor, item_embs: torch.Tensor, candidates, n: int,
                    precision: str = "bf16x3") -> Tuple[torch.Tensor, torch.Tensor]:
    """Row b's candidate items ranked for user row b: (items int64 [B, n], scores fp32 [B, n]) on the device.

    candidates: int [B, C] (host data or a CUDA tensor on the embeddings' device), 1 <= C <= MAX_CANDIDATES; every entry
    is -1 (an empty slot) or an item id, checked before any launch (one device synchronisation for CUDA input).  Rank
    order is score descending, then item id ascending; an item listed twice in a row is ranked once, and a candidate is
    listed with its score even if that is -inf.  Slots past the row's distinct candidates hold item -1, score -inf.
    1 <= n <= min(MAX_N, C).  Scores as ``score_pairs`` computes them, bit for bit (``precision`` likewise)."""
    _check_precision(precision)
    _check_embs(user_embs, item_embs)
    cand = _ids(candidates, "candidates", 2)
    B, C = cand.shape
    if B != user_embs.shape[0]:
        raise ValueError(f"candidates has {B} rows, user_embs {user_embs.shape[0]}")
    if C < 1 or C > MAX_CANDIDATES:
        raise ValueError(f"candidates must have 1..{MAX_CANDIDATES} columns, got {C}")
    if isinstance(n, bool) or not isinstance(n, numbers.Integral):
        raise ValueError(f"n must be an int, got {n!r}")
    n = int(n)
    if n < 1 or n > min(MAX_N, C):
        raise ValueError(f"n must be in 1..{min(MAX_N, C)} (at most {MAX_N} and the {C} candidates), got {n}")
    check = [(cand, -1, item_embs.shape[0] - 1, "candidates")]
    on_dev = isinstance(cand, torch.Tensor)
    if not on_dev:
        _check_ranges(check)
    _check_on_device(user_embs, item_embs)
    if on_dev and cand.device != user_embs.device:
        raise ValueError(f"candidates is on {cand.device}, the embeddings on {user_embs.device}")
    with torch.cuda.device(user_embs.device):
        if on_dev:
            _check_ranges(check)
        items, scores = _rank_candidates(user_embs, item_embs, _to(cand, user_embs.device, torch.int32), n, precision)
        return items.long(), scores


def _rank_candidates(user_embs, item_embs, cand, n, precision):
    """rank_candidates without the argument checks: cand int32 on the device, int32 items."""
    B = cand.shape[0]
    items = torch.empty((B, n), dtype=torch.int32, device=user_embs.device)
    scores = torch.empty((B, n), dtype=torch.float32, device=user_embs.device)
    if B:
        ops.rank_candidates(user_embs, item_embs, cand, n, precision == "bf16x3", items, scores)
    return items, scores


def check_n_neg(n_neg) -> int:
    """Negatives per held-out item: an int in 0..MAX_CANDIDATES - 1 (a row holds the held-out item and its negatives)."""
    if isinstance(n_neg, bool) or not isinstance(n_neg, numbers.Integral) or not 0 <= n_neg < MAX_CANDIDATES:
        raise ValueError(f"n_neg must be an int in 0..{MAX_CANDIDATES - 1}, got {n_neg!r}")
    return int(n_neg)


def sampled_candidates(users, test_user_its, train_csr, n_items: int, n_neg: int, seed):
    """Candidate rows of the sampled-negative evaluation: one row per (user, held-out item) instance, instances in the
    order of ``users`` and then of each user's stored test items.  Column 0 is the held-out item; columns 1 .. n_neg are
    negatives drawn uniformly without replacement (ascending) from the items in neither the user's train items
    (train_csr = (indptr, indices), host arrays) nor its test items.  Draws come from np.random.default_rng(seed) only:
    no global RNG state (torch, numpy, random) is read or moved.  Returns (instance users int64 [T], candidates int32
    [T, 1 + n_neg]).  A user with fewer than n_neg eligible items raises ValueError."""
    if isinstance(n_items, bool) or not isinstance(n_items, numbers.Integral) or n_items < 1:
        raise ValueError(f"n_items must be a positive int, got {n_items!r}")
    n_items, n_neg = int(n_items), check_n_neg(n_neg)
    try:
        indptr, indices = (np.asarray(a.cpu() if isinstance(a, torch.Tensor) else a) for a in train_csr)
    except (TypeError, ValueError):
        raise ValueError("train_csr must be an (indptr, indices) pair") from None
    if indptr.ndim != 1 or indptr.size < 1 or indices.ndim != 1 or (indices.size and indices.dtype.kind not in "iu") \
            or indptr.dtype.kind not in "iu":
        raise ValueError("train_csr must be 1-D integer (indptr, indices) arrays")
    usr = _ids(users.cpu() if isinstance(users, torch.Tensor) else users, "users", 1).astype(np.int64)
    n_rows = indptr.size - 1
    if usr.size and (usr.min() < 0 or usr.max() >= n_rows):
        raise ValueError(f"users out of range 0..{n_rows - 1}")
    if indices.size and (indices.min() < 0 or indices.max() >= n_items):
        raise ValueError(f"train items out of range 0..{n_items - 1}")
    tests = [np.asarray(test_user_its[u] if test_user_its[u] is not None else [], dtype=np.int64) for u in usr]
    for u, t in zip(usr, tests):
        if t.size and (t.min() < 0 or t.max() >= n_items):
            raise ValueError(f"test items of user {u} out of range 0..{n_items - 1}")
    counts = np.array([t.size for t in tests], dtype=np.int64)
    inst_users = np.repeat(usr, counts)
    pos = np.concatenate(tests) if tests else np.zeros(0, dtype=np.int64)
    T = inst_users.size
    cand = np.empty((T, 1 + n_neg), dtype=np.int32)
    cand[:, 0] = pos
    if T == 0 or n_neg == 0:
        return inst_users, cand
    # per user: its excluded items (train + test, sorted, distinct) and the number of eligible ones
    excl = [np.unique(np.concatenate([indices[indptr[u]:indptr[u + 1]].astype(np.int64), t]))
            for u, t in zip(usr, tests)]
    n_ok = np.array([n_items - e.size for e in excl], dtype=np.int64)
    short = np.flatnonzero((n_ok < n_neg) & (counts > 0))
    if short.size:
        u = int(usr[short[0]])
        raise ValueError(f"user {u} has {int(n_ok[short[0]])} items outside its train and test items, fewer than "
                         f"n_neg = {n_neg}")
    # ranks among the eligible items, uniform without replacement: draw with replacement, then redraw the surplus copies
    # of any repeated value until a row is distinct (every step treats all values alike, so the resulting set is uniform
    # over the n_neg-subsets)
    rng = np.random.default_rng(seed)
    m = np.repeat(n_ok, counts)
    ranks = np.sort(rng.integers(0, m[:, None], size=(T, n_neg)), axis=1)
    rows = np.flatnonzero((ranks[:, 1:] == ranks[:, :-1]).any(axis=1))
    while rows.size:
        sub = ranks[rows]
        dup = np.zeros(sub.shape, dtype=bool)
        dup[:, 1:] = sub[:, 1:] == sub[:, :-1]
        r_idx, c_idx = np.nonzero(dup)
        sub[r_idx, c_idx] = rng.integers(0, m[rows][r_idx])
        sub.sort(axis=1)
        ranks[rows] = sub
        rows = rows[(sub[:, 1:] == sub[:, :-1]).any(axis=1)]
    # rank k of a user -> its k-th eligible item: k + #{excluded <= item}, by one search over all users' excluded lists
    # (user j's list shifted by j * (n_items + 1) so the lists stay apart)
    lens = np.array([e.size for e in excl], dtype=np.int64)
    base = np.arange(usr.size, dtype=np.int64) * (n_items + 1)
    gaps = np.concatenate([e - np.arange(e.size) for e in excl]) + np.repeat(base, lens)
    off = np.concatenate([[0], np.cumsum(lens)[:-1]])
    j = np.repeat(np.arange(usr.size), counts)[:, None]
    shifted = ranks + base[j]
    cand[:, 1:] = ranks + np.searchsorted(gaps, shifted, side="right") - off[j]
    return inst_users, cand


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
