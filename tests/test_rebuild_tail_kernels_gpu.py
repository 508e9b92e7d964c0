"""Direct tests of the rebuild's tail, called through the C ABI: the per-user top-k (dmm_topk_edges,
dmm_topk_edges_pruned) on every route its dispatch can take, and the normalised adjacency build
(dmm_build_norm_adj_csr).

Every case is built to reach one route, named from the constants of csrc/topk.cu (32 keys per thread on the register
kernels, 8192-column segments, 2048 merge candidates, the pruned kernel's 64 / 4 / 512 limits, 20480 staged keys of the
deferred kernel).  Results are compared bit for bit with a numpy restatement of the kernels' total order.  Every output
is filled with a sentinel and padded on both sides, score rows are padded past n_cols with +inf or +NaN and chunk-maxima
rows past n_chunks with NaN, so a read or a write outside a call's own entries shows up as a wrong result.

The adjacency is compared bit for bit with a float64 restatement of the kernel's arithmetic (d^-1/2 = 1 / sqrt(deg) with
the self loop in the degree, val = fp32((d_r^-1/2 * 1) * d_c^-1/2)); fp64 sqrt and division are correctly rounded on
both sides, so the two agree exactly.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from diffmm_b200 import _lib
from oracle import diffmm_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PAD = 64                 # sentinel entries on each side of every output
SENT = -7                # int32 sentinel of item / user / column outputs
SENT_F = np.int32(-123456789).view(np.float32)   # fp32 sentinel of adjacency values (a NaN-free, unmistakable pattern)
WS_PAD = 256             # sentinel bytes behind every workspace

# csrc/topk.cu
PER_THREAD = 32          # keys per thread of the register kernels (TOPK_V4 float4 loads)
SEG_COLS = 8192          # TOPK_SEG_COLS
MERGE_CAP = 2048         # TOPK_MERGE_CAP
SMEM_KEYS = 20480        # staged keys of topk_deferred_kernel


# ------------------------------------------------------------------------------------------------ helpers
def order_key(a):
    """The kernels' order-preserving key of the fp32 bit pattern: -0 folded to +0, +NaN above +inf, -NaN below -inf."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32).astype(np.int64)
    u = np.where(u == 0x80000000, 0, u)
    return np.where(u & 0x80000000, (~u) & 0xFFFFFFFF, u | 0x80000000)


def ref_topk(row, k):
    """The k best columns of a row by (key descending, column ascending), in ascending column order."""
    k = min(int(k), row.size)
    if k <= 0:
        return np.zeros(0, dtype=np.int64)
    return np.sort(np.lexsort((np.arange(row.size), -order_key(row)))[:k])


def f32(bits):
    return np.uint32(bits).view(np.float32)


NEG_NAN = f32(0xFFC00000)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _vp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _seg(n_cols):
    """make_seg of topk.cu: (segments, columns per segment)."""
    S = -(-n_cols // SEG_COLS)
    return S, (-(-n_cols // S) + 3) // 4 * 4


def _smem_cap_cols():
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    return (optin - 20480) // 4 if optin > 40960 else 0


# ------------------------------------------------------------------------------------------------ special rows
def _row_pm_zero(rng, n, k):
    """k-th value is 0 shared by -0 and +0 (the -0 first): only the fold puts the lower columns first."""
    row = -1.0 - np.abs(rng.standard_normal(n)).astype(np.float32)
    cols = np.sort(rng.choice(n, 8, replace=False))
    row[cols[:2]] = 2.0
    row[cols[2::2]] = -0.0
    row[cols[3::2]] = 0.0
    return row, 2 + k


def _row_tail_max(rng, n):
    row = rng.standard_normal(n).astype(np.float32)
    t = n & 3
    if t:
        row[n - t:] = 5.0 + np.arange(t, dtype=np.float32)
    return row


def _row_masked(rng, n, finite):
    """Masked evaluation row: -inf except `finite` columns."""
    row = np.full(n, -np.inf, dtype=np.float32)
    if finite:
        row[rng.choice(n, finite, replace=False)] = rng.standard_normal(finite).astype(np.float32)
    return row


def _row_nan(rng, n, where=None):
    row = rng.standard_normal(n).astype(np.float32)
    cols = rng.choice(n, 3, replace=False) if where is None else np.asarray(where)
    row[cols[0]] = np.nan
    row[cols[1]] = NEG_NAN
    row[cols[2]] = np.inf
    return row


def _rows(n_cols, ks, specials, seed):
    """Continuous rows for `ks`, then the special rows [(row, k)]."""
    rng = np.random.default_rng(seed)
    rows = [rng.standard_normal(n_cols).astype(np.float32) for _ in ks] + [r for r, _ in specials]
    return np.stack(rows), np.array(list(ks) + [k for _, k in specials], dtype=np.int64)


# ------------------------------------------------------------------------------------------------ runners
def _scores_buffer(scores, ld, off, pad):
    n_rows, n_cols = scores.shape
    buf = torch.full((off + n_rows * ld + 64,), pad, dtype=torch.float32, device=DEV)
    buf[off:off + n_rows * ld].view(n_rows, ld)[:, :n_cols] = torch.from_numpy(scores).to(DEV)
    return buf, C.c_void_p(buf.data_ptr() + 4 * off)


def _workspace(nbytes):
    ws = torch.full((nbytes + WS_PAD,), 0xA5, dtype=torch.uint8, device=DEV)
    return ws


def _check_ws_tail(ws, nbytes, what):
    assert (ws[nbytes:].cpu().numpy() == 0xA5).all(), f"{what}: write past the end of the workspace"


# variants of every top-k case: (order, out_ptr[0], row_base, out_users given, pad of the score rows)
VARIANTS = [(False, 0, 0, True, float("inf")), (True, 0, 0, False, float("nan")), (True, 1000, 5000, True, float("inf"))]


def _expected(ptr, want, e0, E):
    items = np.full(PAD + e0 + E + PAD, SENT, dtype=np.int32)
    users = items.copy()
    for r, w in enumerate(want):
        o = PAD + int(ptr[r])
        items[o:o + w.size] = w
        users[o:o + w.size] = r
    return items, users


def _run(fn, scores, k, ld, off, want, variant, rng, ws_bytes_fn, cmax=None):
    use_order, e0, row_base, with_users, pad = variant
    n_rows, n_cols = scores.shape
    ptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(k, out=ptr[1:])
    ptr += e0
    E = int(ptr[-1] - ptr[0])
    buf, sp = _scores_buffer(scores, ld, off, pad)
    d_ptr = torch.from_numpy(ptr).to(DEV)
    items = torch.full((PAD + e0 + E + PAD,), SENT, dtype=torch.int32, device=DEV)
    users = torch.full_like(items, SENT) if with_users else None
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    order = torch.from_numpy(rng.permutation(n_rows).astype(np.int32)).to(DEV) if use_order else None
    out_i = C.c_void_p(items.data_ptr() + 4 * PAD)
    out_u = C.c_void_p(users.data_ptr() + 4 * PAD) if with_users else None
    ws_bytes = ws_bytes_fn(E)
    ws = _workspace(ws_bytes) if ws_bytes is not None else None
    if ws is not None and cmax is not None:
        ws[:4].view(torch.int32).fill_(-1)            # the deferred-row count: -1 until the pruned kernel writes it
    fn(sp, d_ptr, row_base, out_u, out_i, status, order, ws, ws_bytes, E)
    torch.cuda.synchronize()
    want_items, want_users = _expected(ptr, want, e0, E)
    tag = f"order={use_order} e0={e0} row_base={row_base} users={with_users} pad={pad}"
    np.testing.assert_array_equal(items.cpu().numpy(), want_items, err_msg=tag)
    if with_users:
        wu = np.where(want_users == SENT, SENT, want_users + row_base).astype(np.int32)
        np.testing.assert_array_equal(users.cpu().numpy(), wu, err_msg=tag)
    assert int(status.item()) == (1 if (k > n_cols).any() else 0), tag
    if ws is not None:
        _check_ws_tail(ws, ws_bytes, tag)
    return ws


def run_edges(scores, k, ld, off=0, use_ws=False):
    """dmm_topk_edges on every variant; use_ws: the segment workspace (else NULL: one CTA per whole row)."""
    n_rows, n_cols = scores.shape
    want = [ref_topk(scores[r], k[r]) for r in range(n_rows)]
    lib = _lib.load()
    rng = np.random.default_rng(n_cols)

    def ws_bytes_fn(E):
        return int(lib.dmm_topk_workspace_bytes(n_cols, E)) if use_ws else None

    def fn(sp, d_ptr, row_base, out_u, out_i, status, order, ws, ws_bytes, E):
        _lib.call("dmm_topk_edges", _lib.ctx(0), sp, ld, n_rows, n_cols, _vp(d_ptr), row_base, out_u, out_i, _vp(status),
                  _vp(order), _vp(ws), ws_bytes or 0, E, _stream())

    for v in VARIANTS:
        _run(fn, scores, k, ld, off, want, v, rng, ws_bytes_fn)


def chunk_max(scores):
    n_rows, n_cols = scores.shape
    nch = -(-n_cols // 32)
    pad = np.full((n_rows, nch * 32), -np.inf, dtype=np.float32)
    pad[:, :n_cols] = scores
    return pad.reshape(n_rows, nch, 32).max(axis=2)      # NaN-propagating, like the contraction epilogue


def run_pruned(scores, k, defer=(), control=(), fallback=False):
    """dmm_topk_edges_pruned on every variant.  defer / control: rows that must / must not be in the deferred list;
    fallback: the width takes the dmm_topk_edges kernels for the whole call (the count stays unwritten)."""
    n_rows, n_cols = scores.shape
    ld = (n_cols + 3) // 4 * 4 + 4
    nch = -(-n_cols // 32)
    ld_cmax = (nch + 3) // 4 * 4 + 4
    cm = torch.full((n_rows, ld_cmax), float("nan"), device=DEV)
    cm[:, :nch] = torch.from_numpy(chunk_max(scores)).to(DEV)
    want = [ref_topk(scores[r], k[r]) for r in range(n_rows)]
    lib = _lib.load()
    rng = np.random.default_rng(n_cols + 1)

    def ws_bytes_fn(E):
        return int(lib.dmm_topk_pruned_workspace_bytes(n_rows, n_cols, E))

    def fn(sp, d_ptr, row_base, out_u, out_i, status, order, ws, ws_bytes, E):
        _lib.call("dmm_topk_edges_pruned", _lib.ctx(0), sp, ld, n_rows, n_cols, _vp(cm), ld_cmax, _vp(d_ptr), row_base,
                  out_u, out_i, _vp(status), _vp(order), _vp(ws), ws_bytes, E, _stream())

    for v in VARIANTS:
        ws = _run(fn, scores, k, ld, 0, want, v, rng, ws_bytes_fn, cmax=cm)
        count = int(ws[:4].view(torch.int32).item())
        if fallback:
            assert count == -1, "the pruned kernel ran on a width outside its range"
            continue
        assert 0 <= count <= n_rows
        rows = ws[256:256 + 4 * count].view(torch.int32).cpu().numpy()
        assert len(set(rows.tolist())) == count and ((rows >= 0) & (rows < n_rows)).all()
        missing = set(defer) - set(rows.tolist())
        assert not missing, f"rows built to defer were ranked on the pruned path: {sorted(missing)}"
        wrong = set(control) & set(rows.tolist())
        assert not wrong, f"continuous control rows were deferred: {sorted(wrong)}"


# ------------------------------------------------------------------------------------------------ dmm_topk_edges
def _layout(n_cols, name):
    """(ld, offset of the base pointer): aligned rows, ld % 4 == 1 (aligned and unaligned rows in one launch), and both
    with a base pointer one column off."""
    ld4 = (n_cols + 3) // 4 * 4
    return {"aligned": (ld4, 0), "ld1": (ld4 + 1, 0), "off1": (ld4 + 1, 1)}[name]


@pytest.mark.parametrize("layout", ["aligned", "ld1", "off1"])
@pytest.mark.parametrize("NT,n_cols", [(256, 8191), (256, 8192), (512, 8193), (512, 16384), (1024, 16386), (1024, 32767),
                                       (1024, 32768)])
def test_topk_register_kernels(NT, n_cols, layout):
    """topk_rows_reg_kernel<NT> (NULL workspace): the q <= 8 bound, the bitonic bound (k > 8 * warps), the in-kernel
    generic fallback (k > NT, unaligned rows), a tail of 1 .. 3 columns that holds the maximum, +-0, NaN, masked rows."""
    assert (n_cols - 1) // PER_THREAD // NT == 0 and n_cols > NT * PER_THREAD // 2
    NW = NT // 32
    rng = np.random.default_rng(NT + n_cols)
    specials = [(_row_tail_max(rng, n_cols), 1), (_row_tail_max(rng, n_cols), 3), _row_pm_zero(rng, n_cols, 2),
                _row_pm_zero(rng, n_cols, 3), (_row_nan(rng, n_cols), 10), (_row_masked(rng, n_cols, 0), 5),
                (_row_masked(rng, n_cols, 10), 30),
                (rng.integers(-3, 4, n_cols).astype(np.float32), 8 * NW + 1)]   # crowded ties at the threshold
    scores, k = _rows(n_cols, [0, 1, 2, 8 * NW, 8 * NW + 1, NT - 1, NT, NT + 1, 17], specials, n_cols)
    ld, off = _layout(n_cols, layout)
    run_edges(scores, k, ld, off)


@pytest.mark.parametrize("n_cols,use_ws", [(5, False), (300, False), (8192, False), (20000, True)])
def test_topk_k_at_and_above_the_row_width(n_cols, use_ws):
    """k = n_cols takes the whole row; k = n_cols + 1 emits the row and sets status bit 0."""
    scores, k = _rows(n_cols, [n_cols, n_cols + 1, 1, min(n_cols, 3)], [], n_cols)
    run_edges(scores, k, (n_cols + 3) // 4 * 4, use_ws=use_ws)


@pytest.mark.parametrize("where", ["smem_first", "smem_cap", "global_first", "global"])
@pytest.mark.parametrize("layout", ["aligned", "ld1"])
def test_topk_whole_row_generic_kernels(where, layout):
    """topk_edges_kernel: in shared memory up to (smem_optin - 20480) / 4 columns (float4 loads for 16-byte aligned row
    starts, scalar loads otherwise), in global memory above.  Unaligned rows take them with a workspace too."""
    cap = _smem_cap_cols()
    n_cols = {"smem_first": 1024 * PER_THREAD + 1, "smem_cap": cap, "global_first": cap + 1, "global": 70001}[where]
    rng = np.random.default_rng(n_cols)
    specials = [(_row_nan(rng, n_cols), 7), _row_pm_zero(rng, n_cols, 3), (_row_masked(rng, n_cols, 20), 40),
                (rng.integers(-3, 4, n_cols).astype(np.float32), 1000)]
    scores, k = _rows(n_cols, [0, 1, 100, 256, 257, 3000], specials, n_cols)
    ld, off = _layout(n_cols, layout)
    run_edges(scores, k, ld, off, use_ws=layout == "ld1")


SEGMENT_CASES = [(2, 16384), (3, 20000), (9, 70001), (33, 262145), (62, 500000), (65, 530000)]   # (S, n_cols)


@pytest.mark.parametrize("S,n_cols", SEGMENT_CASES)
def test_topk_segment_pass_merge_and_mode2(S, n_cols):
    """Rows wider than 8192 columns with a workspace: segment pass + merge for k <= min(256, 2048 / S), the whole-row
    generic kernel (mode 2) for the rest.  Ties at the threshold straddle seg_cols multiples; a NaN sits in one
    segment; masked rows."""
    S_, seg_cols = _seg(n_cols)
    assert S_ == S
    edge = min(256, MERGE_CAP // S)
    rng = np.random.default_rng(S)
    tie = -np.abs(rng.standard_normal(n_cols)).astype(np.float32)
    tie_cols = np.array([m * seg_cols + d for m in range(1, S) for d in (-2, -1, 0, 1)])
    tie[tie_cols] = 1.0
    tie[rng.choice(seg_cols, 2, replace=False)] = 3.0                  # two scores above the tied value
    n_tie = min(edge, tie_cols.size + 2 - 1)
    nan_row = _row_nan(rng, n_cols, where=[seg_cols + 5, 2 * seg_cols - 1 if S > 2 else seg_cols + 9, 7])
    specials = [(tie, n_tie), (tie, 3), (tie.copy(), edge + 1), (nan_row, 4), (nan_row.copy(), edge),
                _row_pm_zero(rng, n_cols, 3), (_row_masked(rng, n_cols, 5), 12), (_row_masked(rng, n_cols, 0), 2)]
    scores, k = _rows(n_cols, [0, 1, edge, edge + 1, 256, 257], specials, n_cols)
    run_edges(scores, k, (n_cols + 3) // 4 * 4, use_ws=True)


# ------------------------------------------------------------------------------------------------ dmm_topk_edges_pruned
@pytest.mark.parametrize("n_cols,fallback", [(224, True), (225, False), (65536, False), (65537, False), (262144, False),
                                             (262145, False), (524288, False), (524289, True)])
def test_pruned_width_boundaries(n_cols, fallback):
    """64 / 256 / 512-thread pruned kernels at their width boundaries, and the whole-call fallbacks (fewer than 8 or
    more than 16384 chunks)."""
    nch = -(-n_cols // 32)
    small = [1, 2] if nch < 16 else [1, 4, 16, 25]
    big = [] if nch < 16 else [65, 300]
    rng = np.random.default_rng(n_cols)
    specials = [(_row_nan(rng, n_cols), 2), _row_pm_zero(rng, n_cols, 1), (_row_masked(rng, n_cols, 3), min(n_cols, 9))]
    scores, k = _rows(n_cols, [0] + small + big, specials, n_cols)
    control = list(range(1, 1 + len(small)))
    defer = [1 + len(small) + i for i in range(len(big))] + [len(k) - 3]    # k > 64; the NaN row
    if nch < 16:
        control, defer = [1], [len(k) - 3]
    run_pruned(scores, k, defer=defer, control=control, fallback=fallback)


def test_pruned_deferral_causes_at_100_chunks():
    """k * 4 == n_chunks is ranked on the pruned path, n_chunks + 4 is deferred; a NaN chunk maximum defers; tied scores
    inside the chosen chunks are ranked by column (mutation check of the final ranking)."""
    n_cols = 3200
    rng = np.random.default_rng(1)
    ties = (rng.standard_normal(n_cols) * 0.1).astype(np.float32)
    for c in (2, 5, 9, 11, 20, 33, 40):
        ties[[32 * c + 3, 32 * c + 20]] = 1.0                          # 7 chunks, two equal maxima each
    specials = [(ties, 5), (ties.copy(), 9), (_row_nan(rng, n_cols), 5), _row_pm_zero(rng, n_cols, 2)]
    scores, k = _rows(n_cols, [25, 26, 1, 7], specials, 2)
    run_pruned(scores, k, defer=[1, 6], control=[0, 2, 3, 4, 5])


def test_pruned_deferral_causes_k64_and_crowded_bounds():
    """k = 64 ranked, k = 65 deferred (260 chunks); more than 512 equal chunk maxima at the bound; more than 512 equal
    scores >= Lk in the chosen chunks (1024 chunks, 64-thread kernel)."""
    rng = np.random.default_rng(3)
    s1, k1 = _rows(8320, [64, 65, 3], [], 4)
    run_pruned(s1, k1, defer=[1], control=[0, 2])
    n_cols = 32768
    crowd_max = (rng.standard_normal(n_cols) * 0.1).astype(np.float32)
    crowd_max[np.arange(1024) * 32 + rng.integers(0, 32, 1024)] = 1.0           # every chunk maximum equals 1.0
    crowd_sc = (rng.standard_normal(n_cols) * 0.1).astype(np.float32)
    chunks = np.concatenate([4 * np.arange(10), 4 * np.arange(32, 42)])          # 10 threads of each warp hold one
    crowd_sc[(chunks[:, None] * 32 + np.arange(32)).ravel()] = 1.0               # 20 chunks x 32 equal scores
    specials = [(crowd_max, 10), (crowd_max.copy(), 40), (crowd_sc, 20), (crowd_sc.copy(), 20)]
    s2, k2 = _rows(n_cols, [1, 8, 16], specials, 5)
    run_pruned(s2, k2, defer=[3, 4, 5, 6], control=[0, 1, 2])


def test_pruned_deferred_kernel_routes():
    """Deferred rows of 2188 chunks: two-level select with phase B staged in shared memory (k * 32 <= 20480) and read
    from global memory (k > 640), up to 2k == n_chunks; the whole-row route above it."""
    n_cols = 70001
    nch = -(-n_cols // 32)
    kb = SMEM_KEYS // 32
    rng = np.random.default_rng(7)
    quant = np.round(rng.standard_normal(n_cols), 1).astype(np.float32)        # moderate ties
    specials = [(quant, kb + 1), (quant.copy(), 70)]
    scores, k = _rows(n_cols, [65, kb, kb + 1, 700, nch // 2, nch // 2 + 1, 1, 3], specials, 8)
    run_pruned(scores, k, defer=[0, 1, 2, 3, 4, 5, 8, 9], control=[6, 7])


# ------------------------------------------------------------------------------------------------ adjacency
def ref_adj(ptr, items, U, I):
    """float64 restatement of dmm_build_norm_adj_csr: rows users [self | items], items [users | self]."""
    deg = np.concatenate([np.diff(ptr), np.bincount(items, minlength=I)]).astype(np.float64) + 1.0
    dinv = 1.0 / np.sqrt(deg)
    N = U + I
    u = np.repeat(np.arange(U, dtype=np.int64), np.diff(ptr))
    it = items.astype(np.int64) + U
    rows = np.concatenate([u, it, np.arange(N)])
    cols = np.concatenate([it, u, np.arange(N)])
    o = np.lexsort((cols, rows))
    rows, cols = rows[o], cols[o]
    adj_ptr = np.zeros(N + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows, minlength=N), out=adj_ptr[1:])
    return adj_ptr, cols.astype(np.int32), ((dinv[rows] * 1.0) * dinv[cols]).astype(np.float32)


def run_adj(ptr, items, U, I):
    """dmm_build_norm_adj_csr into sentinel-filled outputs padded by PAD entries on both sides."""
    E, N = items.size, U + I
    lib = _lib.load()
    ws_bytes = int(lib.dmm_build_adj_workspace_bytes(U, I, E))
    ws = _workspace(ws_bytes)
    a_ptr = torch.full((N + 1 + 2 * PAD,), SENT, dtype=torch.int64, device=DEV)
    a_idx = torch.full((2 * E + N + 2 * PAD,), SENT, dtype=torch.int32, device=DEV)
    a_val = torch.full((2 * E + N + 2 * PAD,), float(SENT_F), dtype=torch.float32, device=DEV)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    d_ptr = torch.from_numpy(ptr).to(DEV)
    d_items = torch.from_numpy(items.astype(np.int32)).to(DEV) if E else None
    off = lambda t: C.c_void_p(t.data_ptr() + PAD * t.element_size())  # noqa: E731
    _lib.call("dmm_build_norm_adj_csr", _lib.ctx(0), _vp(d_ptr), _vp(d_items), U, I, E, off(a_ptr), off(a_idx), off(a_val),
              _vp(ws), ws_bytes, _vp(status), _stream())
    torch.cuda.synchronize()
    _check_ws_tail(ws, ws_bytes, "dmm_build_norm_adj_csr")
    p, i, v = a_ptr.cpu().numpy(), a_idx.cpu().numpy(), a_val.cpu().numpy()
    for arr, sent, what in ((p, SENT, "ptr"), (i, SENT, "idx"), (v.view(np.int32), SENT_F.view(np.int32), "val")):
        assert (arr[:PAD] == sent).all() and (arr[-PAD:] == sent).all(), f"adjacency {what}: write outside the array"
    return p[PAD:-PAD], i[PAD:-PAD], v[PAD:-PAD], int(status.item())


def _csr(rows_items, U):
    ptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum([len(r) for r in rows_items], out=ptr[1:])
    items = np.concatenate([np.asarray(r, dtype=np.int64) for r in rows_items]) if ptr[-1] else np.zeros(0, np.int64)
    return ptr, items


def _random_graph(U, I, E, seed, empty_ends=True):
    rng = np.random.default_rng(seed)
    key = np.unique(rng.integers(0, U, E).astype(np.int64) * I + rng.integers(0, I, E))
    u, i = key // I, key % I
    if empty_ends:
        keep = (u != 0) & (u != U - 1) & (i != 0) & (i != I - 1)
        u, i = u[keep], i[keep]
    ptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(np.bincount(u, minlength=U), out=ptr[1:])
    return ptr, i


def _graph(name):
    if name == "E0":
        return np.zeros(5, dtype=np.int64), np.zeros(0, np.int64), 4, 3
    if name == "U1_I1":
        return np.array([0, 1], dtype=np.int64), np.array([0]), 1, 1
    if name.startswith("items_"):                    # end_bit edges and offsets_dinv_kernel's 255-item blocks
        I = int(name.split("_")[1])
        return (*_random_graph(300, I, 6000, I), 300, I)
    if name == "hub_65537":                          # an item with more than 65 536 users, a user with every item
        U, I = 70000, 300
        rng = np.random.default_rng(9)
        rows = [[0] + sorted(rng.choice(np.arange(1, I), 2, replace=False).tolist()) for _ in range(U)]
        rows[5] = list(range(I))
        rows[0], rows[-1] = [], []
        ptr, items = _csr(rows, U)
        return ptr, items, U, I
    if name == "I_2p20":
        return (*_random_graph(5000, (1 << 20) + 3, 40000, 11), 5000, (1 << 20) + 3)
    if name == "E_6M":                               # beyond the former sort-scratch bound (about 4.7 M edges)
        U, I = 60000, 100000
        rng = np.random.default_rng(12)
        items = (np.arange(100) * 1000 + rng.integers(0, 1000, (U, 100))).ravel()
        return np.arange(U + 1, dtype=np.int64) * 100, items, U, I
    raise KeyError(name)


ADJ_GRAPHS = ["E0", "U1_I1", "items_255", "items_256", "items_257", "items_254", "items_511", "items_65536",
              "items_65537", "hub_65537", "I_2p20", "E_6M"]


@pytest.mark.parametrize("name", ADJ_GRAPHS)
def test_adj_bit_exact(name):
    ptr, items, U, I = _graph(name)
    got_p, got_i, got_v, status = run_adj(ptr, items, U, I)
    assert status == 0
    wp, wi, wv = ref_adj(ptr, items, U, I)
    np.testing.assert_array_equal(got_p, wp)
    np.testing.assert_array_equal(got_i, wi)
    np.testing.assert_array_equal(got_v.view(np.int32), wv.view(np.int32))
    if items.size <= 100000:                         # and within 1 ulp of the reference's deg ** -0.5
        op, oi, ov = O.normalized_adj_csr(np.repeat(np.arange(U), np.diff(ptr)), items, U, I)
        np.testing.assert_array_equal(got_p, op)
        np.testing.assert_array_equal(got_i.astype(np.int64), oi)
        assert np.abs(got_v.view(np.int32).astype(np.int64) - ov.view(np.int32).astype(np.int64)).max() <= 1


@pytest.mark.parametrize("ids", ["above", "below", "both"])
def test_adj_out_of_range_ids_stay_inside_the_arrays(ids):
    """Ids n_items .. n_items + 7 and / or -1 .. -8 set status bit 1; nothing outside the arrays is written (sentinel
    padding) and no stored column is outside [0, N).  With only the ids above n_items they sort last, where an unguarded
    item-side write lands up to 7 entries past 2E + N."""
    U, I = 16, 40
    rng = np.random.default_rng(13)
    rows = [sorted(rng.choice(I, 3, replace=False).tolist()) for _ in range(U)]
    for j in range(8):
        if ids != "below":
            rows[j] = sorted(rows[j] + [I + j])
        if ids != "above":
            rows[8 + j] = sorted(rows[8 + j] + [-1 - j])
    ptr, items = _csr(rows, U)
    _, idx, _, status = run_adj(ptr, items, U, I)
    assert status & 2
    stored = idx[idx != SENT]
    assert ((stored >= 0) & (stored < U + I)).all(), "a stored column lies outside [0, N)"
