"""The joint-training kernels (csrc/spmm.cu, csrc/prop.cu, csrc/loss.cu), one entry point at a time, against float64 or
bit-exact restatements of what each one computes: the CSR SpMM on its three D = 64 paths (planned fp32, unplanned,
separable bf16 table) and the generic-D kernel, spmm_replan, sign_noise_, the gcn_MM glue (rownorm_fwd / _bwd,
modal_mix_fwd / _bwd), BPR, InfoNCE (register-tiled D = 64 and warp-per-row D = 32 / 128 / 256) with scatter_add_rows,
and the fused bpr_infonce_fwd / _bwd of a whole joint step.

Conventions (those of test_chain_kernels_gpu.py):
- Every output buffer the caller provides is larger than the documented region (extra rows, leading dimensions beyond
  the width) and is filled with a sentinel first; after the call everything outside the region must still hold it.
- Exact work is compared bit for bit; everything else against float64 within a bound derived, in a comment next to it,
  from the order of the kernel's operations.  u = 2^-24 is the unit roundoff of fp32 and gamma(n) = n u / (1 - n u)
  bounds the relative error of n roundings in a chain (Higham, ch. 3).  The loss bounds are first-order; they are
  doubled (SLACK) to cover the second-order terms and the ulp-level error of expf / logf / sqrtf.
- CSR matrices are built by hand so that row lengths land exactly on the kernels' thresholds: PLAN_LONG_ROW = 64
  (rows with more entries are chunked), 16 vs 17 chunks (pass A vs pass B of the reduce: 1024 vs 1025 entries) and
  LONG_ROW = 1024 of the unplanned kernel.

Out of scope, as in torch's fp32 F.normalize: the fp32 sum of squares of rownorm / InfoNCE overflows for |x| above
about 1.8e19; no input here comes near it."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
SENT32 = float("nan")    # bits 0x7FC00000
NAN32_BITS = np.int32(0x7FC00000)
F32 = np.float32
SLACK = 2.0


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


def gamma(n):
    n = np.asarray(n, dtype=np.float64)
    return n * U / (1.0 - n * U)


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def f64(t):
    return t.detach().double().cpu().numpy()


def bits(t):
    """int16 / int32 bit view of a bf16 / fp32 tensor on the host (NaN-safe equality)."""
    return t.detach().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).cpu().numpy()


def bf16_rn(v):
    """Round-to-nearest-even bf16 bits (uint16) of a finite fp32 array."""
    b = np.ascontiguousarray(v, dtype=F32).view(np.uint32).astype(np.uint64)
    return ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint16)


def bf16_val(b):
    return (np.asarray(b).astype(np.uint16).astype(np.uint32) << 16).view(F32)


def sentinel_buf(rows, ld):
    return torch.full((rows, ld), SENT32, dtype=torch.float32, device=DEV)


def assert_sentinel(buf, rows, cols):
    """Everything of buf outside [rows, :cols] (rows: a slice or index array) still holds the sentinel."""
    b = bits(buf)
    mask = np.ones(b.shape, dtype=bool)
    mask[rows, :cols] = False
    assert (b[mask] == NAN32_BITS).all(), "a kernel wrote outside its documented region"


def padded(a, extra=8, fill=1e30):
    """fp32 device copy of the host array a [R, C] as a view with leading dimension C + extra (a multiple of 4 when C
    is); the padding holds `fill`."""
    R, C = a.shape
    buf = torch.full((max(R, 1), C + extra), fill, dtype=torch.float32, device=DEV)
    buf[:R, :C] = T(np.asarray(a, dtype=F32))
    return buf[:R, :C]


def assert_within(got, want, bound, what):
    got = np.asarray(got, dtype=np.float64)
    ok = np.abs(got - want) <= bound
    assert ok.all(), (f"{what}: {(~ok).sum()} of {ok.size} outside the bound; worst at {np.argwhere(~ok)[0]}: "
                      f"got {got[~ok][0]!r}, want {np.asarray(want)[~ok][0]!r}, bound {np.asarray(bound)[~ok][0]!r}")


# ================================================================================================ SpMM
THRESH_LENS = [0, 1, 7, 8, 9, 63, 64, 65, 128, 1023, 1024, 1025, 1100, 3000]
N_SP = 4096
# row -> length: a chunked row at 0 and at n - 1 (blocks starting / ending on one), every threshold length in between
SPECIAL = {0: 1025, 1: 0, 2: 1, 100: 7, 101: 8, 102: 9, 500: 63, 501: 64, 502: 65, 900: 128, 1500: 1023, 1501: 1024,
           1502: 1025, 2000: 1100, 2001: 0, 2500: 3000, 3000: 64, 3001: 65, N_SP - 1: 3000}
BLOCKS = [(0, N_SP), (0, 1), (2000, 2501), (1501, N_SP), (N_SP - 1, N_SP), (7, 7)]


def csr_lengths(rng, lens):
    """CSR with the given row lengths over len(lens) columns: distinct ascending columns, values uniform in
    +-[0.25, 1)."""
    n = len(lens)
    ptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=ptr[1:])
    idx = np.concatenate([np.sort(rng.choice(n, int(k), replace=False)) for k in lens] + [np.zeros(0, np.int64)])
    val = (rng.uniform(0.25, 1.0, idx.size) * rng.choice([-1.0, 1.0], idx.size)).astype(F32)
    return ptr, idx.astype(np.int32), val


def threshold_lens(rng):
    lens = rng.integers(0, 13, N_SP)
    lens[rng.choice(N_SP, 200, replace=False)] = rng.integers(13, 80, 200)       # mixed-length warps at every bin border
    for r, k in SPECIAL.items():
        lens[r] = k
    assert set(THRESH_LENS) <= set(lens.tolist())
    return lens


@pytest.fixture(scope="module")
def thresh_csr():
    rng = np.random.default_rng(11)
    return csr_lengths(rng, threshold_lens(rng))


def make_adj(ops, ptr, idx, val, separable=False):
    n = len(ptr) - 1
    return ops.CsrAdj(T(ptr), T(idx), T(val), n, 0, separable=separable)


def sp_ref(ptr, idx, val, x):
    """(A x, |A| |x|) in float64."""
    n = len(ptr) - 1
    A = sp.csr_matrix((val.astype(np.float64), idx, ptr), shape=(n, n))
    x = np.asarray(x, dtype=np.float64)
    return A @ x, abs(A) @ np.abs(x)


def spmm_bound(lens, absax, alpha, beta, z):
    """|y - (alpha A x + beta z)|: the row sum of len_r products is a chain of at most len_r + 1 roundings on every path
    (one fma chain per unit / half warp, the partial sums of a chunked row added in a fixed order: a deeper tree than
    len_r never forms), alpha * acc rounds once and fmaf(beta, z, o) once more: gamma(len_r + 3) |alpha| sum_j |a_rj x_j|
    plus u |beta z_r|."""
    b = gamma(np.asarray(lens)[:, None] + 3) * abs(alpha) * absax
    if z is not None:
        b = b + U * np.abs(beta * np.asarray(z, dtype=np.float64))
    return b


def spmm_raw(ops, adj, x, out, row0, row1, alpha=1.0, beta=0.0, z=None, plan=None):
    """dmm_spmm_csr straight through the C ABI (plan None: the documented unplanned D = 64 path)."""
    ws = adj.workspace if plan is not None else None
    ops._lib.call("dmm_spmm_csr", ops._ctx(x), ops._p(adj.ptr), ops._p(adj.idx), ops._p(adj.val), int(row0), int(row1),
                  ops._p(x), ops._row_major(x, "x"), x.shape[1], float(alpha), float(beta), ops._p(z),
                  ops._row_major(z, "z") if z is not None else 0, ops._p(out), ops._row_major(out, "out"), ops._p(plan),
                  int(adj.nnz), ops._p(ws), ws.numel() if ws is not None else 0, ops._stream())


EPIS = {"plain": (1.0, 0.0), "axpy": (float(F32(1.3)), float(F32(-0.7)))}      # the kernels receive fp32 alpha, beta


def run_spmm(ops, path, adj, x, out, row0, row1, alpha, beta, z):
    if path == "unplanned":
        spmm_raw(ops, adj, x, out, row0, row1, alpha, beta, z)
    else:
        ops.spmm(adj, x, alpha=alpha, beta=beta, z=z, out=out, row0=row0, row1=row1)


@pytest.mark.parametrize("epi", sorted(EPIS))
@pytest.mark.parametrize("path,D", [("planned", 64), ("unplanned", 64)] + [("generic", d) for d in (4, 36, 60, 68, 128, 252, 256)])
def test_spmm_row_lengths_on_every_threshold(ops, thresh_csr, path, D, epi):
    """Every path against float64 on rows of 0 .. 3000 entries, padded X / Y / Z, z = x as SpMMAxpy passes it, row
    blocks that begin and end on chunked rows (and an empty one): rows outside the block keep the sentinel."""
    ptr, idx, val = thresh_csr
    lens = np.diff(ptr)
    rng = np.random.default_rng(D)
    xh = rng.standard_normal((N_SP, D)).astype(F32)
    alpha, beta = EPIS[epi]
    adj = make_adj(ops, ptr, idx, val)
    x = padded(xh, extra=8)
    z = x if epi == "axpy" else None
    ax, absax = sp_ref(ptr, idx, val, xh)
    want = alpha * ax + (beta * xh.astype(np.float64) if z is not None else 0.0)
    bound = spmm_bound(lens, absax, alpha, beta, xh if z is not None else None)
    for row0, row1 in BLOCKS:
        buf = sentinel_buf(N_SP + 3, D + 12)
        run_spmm(ops, path, adj, x, buf[:N_SP, :D], row0, row1, alpha, beta, z)
        assert_sentinel(buf, slice(row0, row1), D)
        assert_within(f64(buf[row0:row1, :D]), want[row0:row1], bound[row0:row1], f"{path} D={D} rows {row0}:{row1}")


def bad_rows_case(rng, D, bad):
    xh = rng.standard_normal((N_SP, D)).astype(F32)
    xh[bad, : D // 2] = np.inf
    xh[bad, D // 2:] = np.nan
    return xh


@pytest.mark.parametrize("bad", [0, N_SP // 2])
@pytest.mark.parametrize("path,D", [("planned", 64), ("unplanned", 64), ("generic", 128), ("bf16", 64)])
def test_spmm_non_finite_row_reaches_only_its_neighbours(ops, thresh_csr, path, D, bad):
    """+inf / NaN in one row of X: only output rows that store that column may become non-finite; every other row is
    finite and as accurate as without it.  (The fp32 units kernel once gathered column 0 with value 0 for the padding
    entries of a mixed-length warp: 0 * inf made rows that never reference row 0 NaN.)"""
    ptr, idx, val = thresh_csr
    lens = np.diff(ptr)
    rng = np.random.default_rng(5 + bad)
    xh = bad_rows_case(rng, D, bad)
    reach = np.zeros(N_SP, dtype=bool)
    reach[np.repeat(np.arange(N_SP), lens)[idx == bad]] = True
    assert 0 < reach.sum() < N_SP // 10
    clean = xh.copy()
    clean[bad] = 0.0
    adj = make_adj(ops, ptr, idx, val, separable=True)
    buf = sentinel_buf(N_SP, D + 4)
    if path == "bf16":
        dinv = np.where(lens > 0, 1.0 / np.sqrt(np.maximum(lens, 1).astype(np.float64)), 0.0).astype(F32)
        ops.spmm_norm_bf16(adj, padded(xh), out=buf[:, :D])
        tab = bf16_val(bf16_rn(dinv[:, None] * clean)).astype(np.float64)
        ones = np.ones_like(val)
        s, sabs = sp_ref(ptr, idx, ones, tab)
        want, bound = dinv[:, None] * s, gamma(lens[:, None] + 4) * dinv[:, None] * sabs
    else:
        run_spmm(ops, path, adj, padded(xh), buf[:, :D], 0, N_SP, 1.0, 0.0, None)
        want, absax = sp_ref(ptr, idx, val, clean)
        bound = spmm_bound(lens, absax, 1.0, 0.0, None)
    got = f64(buf[:, :D])
    assert np.isfinite(got[~reach]).all(), \
        f"{path}: rows that do not store column {bad} became non-finite: {np.flatnonzero(~np.isfinite(got).all(1) & ~reach)[:10]}"
    assert_within(got[~reach], want[~reach], bound[~reach], f"{path} finite rows")


# ---------------------------------------------------------------------------------------- separable bf16 table
def bipartite_thresholds(rng):
    """User-item CSR whose normalised adjacency (build_norm_adj: a user with k items has a row of k + 1 entries with its
    self loop) has user rows on every threshold length; 3000 filler users all hold item 0 (an item row of > 3000
    entries: pass B)."""
    I = 1200
    targets = [1, 7, 8, 9, 63, 64, 65, 128, 1023, 1024, 1025, 1100]
    rows = [np.sort(rng.choice(I, k - 1, replace=False)) for k in targets]
    rows += [np.sort(np.concatenate([[0], 1 + rng.choice(I - 1, int(rng.integers(0, 12)), replace=False)]))
             for _ in range(3000)]
    ptr = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([len(r) for r in rows], out=ptr[1:])
    return ptr, np.concatenate(rows).astype(np.int32), len(rows), I


@pytest.fixture(scope="module")
def norm_adj_case(ops):
    ptr, items, Un, In = bipartite_thresholds(np.random.default_rng(3))
    adj = ops.build_norm_adj(T(ptr), T(items), Un, In)
    hp, hi = adj.ptr.cpu().numpy(), adj.idx.cpu().numpy()
    lens = np.diff(hp)
    assert {1, 7, 8, 9, 63, 64, 65, 128, 1023, 1024, 1025, 1100} <= set(lens[:12].tolist()) and lens.max() > 3000
    return adj, hp, hi, lens


@pytest.mark.parametrize("split", ["x2_only", "x_only", "interior"])
@pytest.mark.parametrize("epi", sorted(EPIS))
def test_spmm_bf16_table_and_product(ops, norm_adj_case, split, epi):
    """T = bf16_rn(d^-1/2 X) bit for bit (X = [x ; x2] with padded leading dimensions, split at n_first), then
    Y = alpha d_r^-1/2 sum_c T_c (+ beta z) against float64 on every row block."""
    adj, hp, hi, lens = norm_adj_case
    n = adj.n_nodes
    rng = np.random.default_rng(len(split))
    xh = rng.standard_normal((n, 64)).astype(F32)
    n_first = {"x2_only": 0, "x_only": n, "interior": 12 + 3000 // 2}[split]
    xb = torch.full((n + 1, 72), 1e30, dtype=torch.float32, device=DEV)
    xb[:n_first, :64] = T(xh[:n_first])
    x = xb[:n_first, :64]
    x2 = padded(xh[n_first:], extra=20) if n_first < n else None
    if n_first == 0:      # no rows from x: through the C ABI (the wrapper takes n_first from x, whose pointer must be valid)
        ops._ensure_plan(adj, x2.device)
        table = torch.empty((n, 64), dtype=torch.bfloat16, device=DEV)
        ops._lib.call("dmm_spmm_table_bf16", ops._ctx(x2), ops._p(x2), 64, 0, ops._p(x2), ops._row_major(x2, "x2"), n,
                      ops._p(adj.plan), int(adj.nnz), ops._p(table), ops._stream())
    else:
        table = ops.spmm_table_bf16(adj, x, x2)
    dinv = np.where(lens > 0, 1.0 / np.sqrt(np.maximum(lens, 1).astype(np.float64)), 0.0).astype(F32)
    tab16 = bf16_rn(dinv[:, None] * xh)          # one fp32 product, one bf16 rounding
    assert np.array_equal(bits(table).view(np.uint16), tab16)
    alpha, beta = EPIS[epi]
    zh = rng.standard_normal((n, 64)).astype(F32)
    z = padded(zh, extra=4) if epi == "axpy" else None
    tab = bf16_val(tab16).astype(np.float64)
    s, sabs = sp_ref(hp, hi, np.ones(hi.size, F32), tab)
    # the sum of len_r table rows (fp32 accumulator += bf16 operand) is a chain of len_r + 1 roundings (the chunks of a
    # long row added in a fixed order), alpha d_r^-1/2 rounds once, times the sum once, fmaf(beta, z, o) once
    bz = beta * zh.astype(np.float64) if z is not None else 0.0           # (a float32 array times a float stays float32)
    want = alpha * dinv[:, None] * s + bz
    bound = gamma(lens[:, None] + 4) * abs(alpha) * dinv[:, None] * sabs + U * np.abs(bz)
    for row0, row1 in [(0, n), (0, 1), (5, 13), (11, n), (n - 1, n), (3, 3)]:
        buf = sentinel_buf(n + 2, 76)
        ops.spmm_norm_bf16(adj, table=table, alpha=alpha, beta=beta, z=z, out=buf[:n, :64], row0=row0, row1=row1)
        assert_sentinel(buf, slice(row0, row1), 64)
        assert_within(f64(buf[row0:row1, :64]), want[row0:row1], bound[row0:row1], f"bf16 rows {row0}:{row1}")


# ------------------------------------------------------------------------------------------------- replan
def lens_with_total(rng, n, fixed, total):
    """Row lengths with the given {row: length} and short filler rows (0 .. 30) adding up to `total` entries."""
    lens = rng.integers(0, 31, n)
    for r, k in fixed.items():
        lens[r] = k
    free = np.array([r for r in range(n) if r not in fixed])
    diff = total - int(lens.sum())
    while diff != 0:
        r = free[rng.integers(0, free.size)]
        step = int(np.clip(diff, -lens[r], 30 - lens[r]))
        lens[r] += step
        diff -= step
    return lens


def test_spmm_replan_follows_a_new_degree_profile(ops):
    """The arrays of an adjacency are overwritten in place with a graph of the same nnz and another degree profile and
    spmm_replan rebuilds its plan (Main._bind_static_adjacencies in graph mode): short rows become rows of more than
    1024 entries, then the count of such rows drops to 0.  The fp32 and bf16 products must equal those of a freshly
    planned adjacency bit for bit, and float64."""
    rng = np.random.default_rng(17)
    n, total = 3000, 60000
    profiles = [{5: 1500, 2000: 2000},                 # two rows of > 16 chunks
                {5: 3, 2000: 0, 100: 1800, 101: 1100},    # those short, two short rows now > 1024
                {100: 1000, 101: 1000, 7: 65}]            # no row > 1024 any more
    xh = rng.standard_normal((n, 64)).astype(F32)
    x = padded(xh)
    adj = None
    for fixed in profiles:
        lens = lens_with_total(rng, n, fixed, total)
        ptr, idx, val = csr_lengths(rng, lens)
        if adj is None:
            adj = make_adj(ops, ptr, idx, val, separable=True)
            ops.spmm(adj, x)                                     # builds the plan that replan refreshes
        else:
            adj.ptr.copy_(T(ptr))
            adj.idx.copy_(T(idx))
            adj.val.copy_(T(val))
            ops.spmm_replan(adj)
        fresh = make_adj(ops, ptr, idx, val, separable=True)
        y, y_fresh = ops.spmm(adj, x), ops.spmm(fresh, x)
        b, b_fresh = ops.spmm_norm_bf16(adj, x), ops.spmm_norm_bf16(fresh, x)
        assert np.array_equal(bits(y), bits(y_fresh)) and np.array_equal(bits(b), bits(b_fresh))
        ax, absax = sp_ref(ptr, idx, val, xh)
        assert_within(f64(y), ax, spmm_bound(lens, absax, 1.0, 0.0, None), f"replanned fp32 {sorted(fixed.items())}")
        dinv = np.where(lens > 0, 1.0 / np.sqrt(np.maximum(lens, 1).astype(np.float64)), 0.0).astype(F32)
        tab = bf16_val(bf16_rn(dinv[:, None] * xh)).astype(np.float64)
        s, sabs = sp_ref(ptr, idx, np.ones(idx.size, F32), tab)
        assert_within(f64(b), dinv[:, None] * s, gamma(lens[:, None] + 4) * dinv[:, None] * sabs, "replanned bf16")


# ================================================================================================ sign_noise_
@pytest.mark.parametrize("D", [1, 31, 64, 100])
def test_sign_noise_against_float64(ops, D):
    """e += sign(e) rnd / max(||rnd||, 1e-12) * degree on a padded e: zero entries of e stay 0 exactly, a zero rnd row
    leaves its row unchanged and a rnd row of norm below 1e-12 is divided by the clamp."""
    rng = np.random.default_rng(D)
    n, deg = 777, 0.1
    eh = rng.standard_normal((n, D)).astype(F32)
    eh[rng.random((n, D)) < 0.1] = 0.0
    eh[3] = 0.0
    rh = rng.standard_normal((n, D)).astype(F32)
    rh[4] = 0.0
    rh[5] = (rh[5] * (1e-14 / np.sqrt(D))).astype(F32)           # norm < 1e-12: the clamp divides
    buf = sentinel_buf(n + 2, D + 5)
    buf[:n, :D] = T(eh)
    ops.sign_noise_(buf[:n, :D], padded(rh, extra=3), deg)
    assert_sentinel(buf, slice(0, n), D)
    got = f64(buf[:n, :D])
    assert np.array_equal(got[eh == 0], np.zeros((eh == 0).sum()))
    r64 = rh.astype(np.float64)
    nrm = np.sqrt((r64 ** 2).sum(1, keepdims=True))
    step = r64 * (deg / np.maximum(nrm, 1e-12))
    want = eh + np.sign(eh) * step
    # ss: a chain of ceil(D / 32) fmas per lane and a 5-level butterfly; sqrtf, the division and rnd * inv round once
    # each (the sign multiply is exact), the final add once
    k = -(-D // 32) + 5
    bound = np.abs(step) * (gamma(k) / 2 + 4 * U) + U * np.abs(want)
    assert_within(got, want, bound, "sign_noise_")
    assert np.array_equal(got[4], eh[4].astype(np.float64))


# ================================================================================================ gcn_MM glue
@pytest.mark.parametrize("D", [1, 31, 33, 64, 100, 1500])
def test_rownorm_fwd_bwd_against_float64(ops, D):
    """y = x / max(||x||, eps), inv = +-1 / den (negative: clamped), gx = (g - y (y . g)) |inv| (plain g |inv| for a
    clamped row): padded inputs, zero rows and rows just below / above eps."""
    eps = 1e-12
    rng = np.random.default_rng(D)
    n = 300
    xh = rng.standard_normal((n, D))
    unit = xh / np.linalg.norm(xh, axis=1, keepdims=True)
    xh[0] = 0.0
    xh[1] = unit[1] * eps * 0.97          # below eps: clamped, y = x / eps is not 0
    xh[2] = unit[2] * eps * 1.03          # above eps: a true norm
    xh[3] = unit[3] * 1e-30 if D > 1 else 0.0
    xh = xh.astype(F32)
    y, inv = ops.rownorm_fwd(padded(xh, extra=7), eps)
    x64 = xh.astype(np.float64)
    nrm = np.sqrt((x64 ** 2).sum(1))
    clamped = ~(nrm > eps)
    assert clamped[[0, 1, 3]].all() and not clamped[2]
    den = np.where(clamped, eps, nrm)
    # ss: a chain of ceil(D / 32) fmas per lane + 5 butterfly levels; sqrtf and the division round once each
    k = -(-D // 32) + 5
    assert_within(f64(y), x64 / den[:, None], np.abs(x64 / den[:, None]) * (gamma(k) / 2 + 3 * U), "rownorm y")
    ih = inv.cpu().numpy()
    assert np.array_equal(ih[clamped], np.full(clamped.sum(), -(F32(1) / F32(eps)), F32))       # one IEEE division
    assert_within(ih[~clamped], 1.0 / nrm[~clamped], (gamma(k) / 2 + 3 * U) / nrm[~clamped], "rownorm inv")
    gh = rng.standard_normal((n, D)).astype(F32)
    gx = ops.rownorm_bwd(y, inv, padded(gh, extra=3))
    y64, s = f64(y), np.abs(ih.astype(np.float64))[:, None]
    g64 = gh.astype(np.float64)
    dot = np.where(clamped, 0.0, (y64 * g64).sum(1))[:, None]
    want = (g64 - y64 * dot) * s
    # the dot: ceil(D / 32) fmas per lane + 5 levels; g - y dot at most two roundings, times |inv| one
    dabs = np.where(clamped, 0.0, np.abs(y64 * g64).sum(1))[:, None]
    bound = s * (np.abs(y64) * gamma(k) * dabs + 2 * U * (np.abs(g64) + np.abs(y64 * dot))) + U * np.abs(want)
    assert_within(f64(gx), want, bound, "rownorm_bwd")
    # a clamped row skips the projection: g * |inv| exactly
    assert np.array_equal(bits(gx)[clamped], (gh[clamped] * np.abs(ih[clamped])[:, None]).astype(F32).view(np.int32))


MIX_N = [4, 1020, 1024, 1028, 4096 + 1024 + 12]


@pytest.mark.parametrize("lam", [0.0, 0.6, -1.3])
@pytest.mark.parametrize("M", [1, 2, 3, 4])
def test_modal_mix_fwd_bwd_against_float64(ops, M, lam):
    """out = sum_m w_m (y + lam z_m) bit for bit with the eager expression; gy, gz_m = lam w_m g and gw_m = sum g . (y +
    lam z_m) (per-CTA partials added in a fixed order) against float64, at element counts around the 1024-element CTA."""
    for n_el in MIX_N:
        rng = np.random.default_rng(n_el + M)
        shp = (n_el // 4, 4)
        yh, gh = rng.standard_normal(shp).astype(F32), rng.standard_normal(shp).astype(F32)
        zh = [rng.standard_normal(shp).astype(F32) for _ in range(M)]
        wh = rng.uniform(0.1, 1.0, M).astype(F32)
        y, g, zs, w = T(yh), T(gh), [T(z) for z in zh], T(wh)
        out = ops.modal_mix_fwd(y, zs, w, lam)
        lam32 = F32(lam)
        acc = None
        for m in range(M):
            t = wh[m] * (yh + lam32 * zh[m])                    # numpy fp32: every operation rounds once, as the kernel's
            acc = t if acc is None else acc + t
        assert np.array_equal(bits(out), acc.view(np.int32)), f"modal_mix_fwd n={n_el}"
        ref = None
        for m in range(M):
            t = w[m] * (y + lam * zs[m])
            ref = t if ref is None else ref + t
        assert torch.equal(out, ref)
        for need_gz in (True, False):
            gy, gzs, gw = ops.modal_mix_bwd(g, y, zs, w, lam, need_gz=need_gz)
            g64, w64 = gh.astype(np.float64), wh.astype(np.float64)
            # gy = sum_m (w_m g): M products and M - 1 additions (fused or not)
            assert_within(f64(gy), w64.sum() * g64, gamma(2 * M) * w64.sum() * np.abs(g64), f"gy n={n_el}")
            for m in range(M):
                if need_gz:
                    assert np.array_equal(bits(gzs[m]), (lam32 * (wh[m] * gh)).view(np.int32)), f"gz n={n_el}"
                else:
                    assert gzs[m] is None
                aw = yh.astype(np.float64) + lam * zh[m].astype(np.float64)
                absaw = np.abs(yh) + abs(lam) * np.abs(zh[m]).astype(np.float64)
                n_cta = -(-n_el // 1024)
                # y + lam z: two roundings; the 4 products of a thread, 5 warp levels, 8 warps, then the CTA partials:
                # a tree no deeper than 2 + 4 + 5 + 8 + n_cta
                b = gamma(19 + n_cta) * (np.abs(g64) * absaw).sum()
                assert_within(float(gw[m]), (g64 * aw).sum(), b, f"gw[{m}] n={n_el}")


@pytest.mark.parametrize("M", [0, 5])
def test_modal_mix_rejects_modality_counts_outside_1_to_4(ops, M):
    y = torch.zeros((8, 4), device=DEV)
    with pytest.raises(ValueError, match="modalities"):
        ops.modal_mix_fwd(y, [y.clone() for _ in range(M)], torch.ones(M, device=DEV), 0.5)
    with pytest.raises(ValueError, match="modalities"):
        ops.modal_mix_bwd(y, y, [y.clone() for _ in range(M)], torch.ones(M, device=DEV), 0.5)


# ================================================================================================ losses
def bpr_ref(u, p, q, gs):
    """BPR of rows u, p, q (float64 [B, D]): row losses -log(1e-5 + s), s = sigmoid(u.p - u.q), gradients of gs * mean,
    and their bounds.  The kernels: per-lane fma chains of ceil(D / 32) and a 5-level butterfly for u.p and u.q (the
    fused kernel: u.(p - q), the difference rounding once), x = dp - dq once; s = 1 / (1 + expf(-x)) moves by
    s (1 - s) dx plus expf's 2 ulp and two roundings; the loss by ds / (1e-5 + s) plus logf's ulp; the gradient factor
    d = -f(s) gs / B, f = s (1 - s) / (1e-5 + s), by |f'(s)| ds and four roundings."""
    B, D = u.shape
    x = (u * p).sum(1) - (u * q).sum(1)
    s = 1.0 / (1.0 + np.exp(-x))
    row = -np.log(1e-5 + s)
    dx = gamma(-(-D // 32) + 8) * (np.abs(u) * (np.abs(p) + np.abs(q))).sum(1)
    ds = s * ((1 - s) * (dx + 4 * U) + 3 * U) + 2.0 ** -126
    drow = ds / (1e-5 + s) + 2 * U + 2 * U * np.abs(row)
    f = s * (1 - s) / (1e-5 + s)
    fp = np.abs(((1 - 2 * s) * (1e-5 + s) - s * (1 - s)) / (1e-5 + s) ** 2)
    c = gs / B
    d = -f * c
    dd = abs(c) * (fp * ds + 6 * U * f)
    gu, gp, gq = d[:, None] * (p - q), d[:, None] * u, -d[:, None] * u
    bu = dd[:, None] * np.abs(p - q) + 3 * U * np.abs(gu)
    bp = dd[:, None] * np.abs(u) + 2 * U * np.abs(gp)
    return row, drow, (gu, gp, gq), (bu, bp, bp)


def mean_bound(row, drow):
    """mean_reduce_kernel / the fused combine: 1024 strided per-thread sums, two 5-level butterflies, one scaling."""
    B = row.size
    return (drow.sum() + gamma(-(-B // 1024) + 12) * np.abs(row).sum()) / B + 2 * U * abs(row.mean())


LOSS_B = [1, 2, 31, 32, 33, 255, 256, 257, 511, 512, 513, 767, 768, 769, 1024, 1025, 4096]


def loss_tables(rng, D, n=3000):
    a = rng.standard_normal((n, D)).astype(F32)
    b = (a + 0.7 * rng.standard_normal((n, D))).astype(F32)
    a[0] = 0.0                                             # zero rows: the 1e-12 clamp of the normalisation
    b[1] = 0.0
    return a, b


def batch_idx(rng, B, n=3000):
    idx = rng.integers(0, n, B)
    idx[: min(B, 4)] = [0, 1, 7, 7][: min(B, 4)]          # zero rows and a repeated index in every batch
    return idx.astype(np.int64)


@pytest.mark.parametrize("B", LOSS_B)
@pytest.mark.parametrize("D", [1, 32, 64, 100, 128, 256])
def test_bpr_against_float64(ops, D, B):
    """Loss and row gradients on padded tables, repeated indices, saturated margins (+-100)."""
    rng = np.random.default_rng(D * 7919 + B)
    NU, NI = 500, 800
    uh, ih = rng.standard_normal((NU, D)).astype(F32), rng.standard_normal((NI, D)).astype(F32)
    uh[0], ih[0], ih[1] = 0.0, 0.0, 0.0
    uh[0, 0], ih[0, 0] = 10.0, 10.0                         # u0.i0 - u0.i1 = 100
    users, pos, neg = rng.integers(0, NU, B), rng.integers(0, NI, B), rng.integers(0, NI, B)
    users[:2], pos[:2], neg[:2] = 0, [0, 1][:B], [1, 0][:B]  # margins +100 and -100
    gs = 0.37
    loss, (gu, gp, gn) = ops.bpr_fwd_bwd(padded(uh, 3), padded(ih, 5), T(users), T(pos), T(neg), gs)
    u, p, q = (uh[users].astype(np.float64), ih[pos].astype(np.float64), ih[neg].astype(np.float64))
    row, drow, grads, bounds = bpr_ref(u, p, q, gs)
    assert_within(float(loss), row.mean(), SLACK * mean_bound(row, drow), "bpr loss")
    for got, want, b, name in zip((gu, gp, gn), grads, bounds, ("g_u", "g_p", "g_n")):
        assert_within(f64(got), want, SLACK * b, f"bpr {name}")


def test_bpr_accepts_D_up_to_256_only(ops):
    t = torch.zeros((4, 257), device=DEV)
    i = torch.zeros(2, dtype=torch.int64, device=DEV)
    with pytest.raises(ops._lib.DiffMMError, match="bad shape"):
        ops.bpr_fwd_bwd(t, t, i, i, i)


def nce_ref(x1, x2, temp, gs):
    """In-batch InfoNCE of the gathered raw rows x1, x2 (float64 [B, D]): lse, row losses, the row gradients of
    gs * mean, and bounds on each.  The kernels normalise with fp32 (ceil(D / 32) fmas per lane + 5 levels, sqrtf, one
    division, one product: relative en per component), form each logit from unit vectors (D products in a tree, then
    times fl(1 / T): ds absolute), sum exp(s - m) online (s - m rounds, |s - m| <= 2 / T; every step of the chain over
    the stream rows, tiles, splits and the merge costs at most expf's 2 ulp of a rescale and two roundings: 6 B + 40)
    and take logf; the gradient weights w = exp(s - lse) - [i == j] carry p (ds + dlse + 4 u + u |s - lse|) + u |w|,
    are accumulated against the stream rows (depth B + 16), projected with
    g_x = inv (G - n (n . G)) (a dot of depth D / 16 + 8, three roundings) and scaled by gs / (B T) (four roundings)."""
    B, D = x1.shape
    n1n, n2n = np.sqrt((x1 ** 2).sum(1)), np.sqrt((x2 ** 2).sum(1))
    inv1, inv2 = 1.0 / np.maximum(n1n, 1e-12), 1.0 / np.maximum(n2n, 1e-12)
    n1, n2 = x1 * inv1[:, None], x2 * inv2[:, None]
    s = n1 @ n2.T / temp
    m = s.max(1, keepdims=True)
    l = np.exp(s - m).sum(1, keepdims=True)
    lse = (m + np.log(l))[:, 0]
    P = np.exp(s - lse[:, None])
    row = lse - np.diag(s)
    kd = -(-D // 32) + 5
    en = gamma(kd) / 2 + 4 * U
    ds = (gamma(D) + 2 * en + 3 * U) / temp
    el = gamma(6 * B + 40) + 2 * U * 2 / temp
    dlse = ds + el + 2 * U * np.abs(lse)
    drow = dlse + ds + U * np.abs(row)
    W = P - np.eye(B)
    dW = P * (ds + dlse[:, None] + 4 * U + U * np.abs(s - lse[:, None])) + U * np.abs(W)
    c = gs / (B * temp)
    out = []
    for n, nb, inv, Wm, dWm in ((n1, n2, inv1, W, dW), (n2, n1, inv2, W.T, dW.T)):
        G = Wm @ nb
        dG = dWm @ np.abs(nb) + (np.abs(Wm) @ np.abs(nb)) * (en + gamma(B + 16))
        nG = (n * G).sum(1, keepdims=True)
        g = c * inv[:, None] * (G - n * nG)
        an = np.abs(n)
        dg = abs(c) * inv[:, None] * (dG + an * (an * dG).sum(1, keepdims=True)
                                      + (gamma(D // 16 + 8) + 2 * en) * an * (an * np.abs(G)).sum(1, keepdims=True)
                                      + 3 * U * (np.abs(G) + an * np.abs(nG))) + (gamma(6) + en) * np.abs(g)
        out.append((g, dg))
    return lse, dlse, row, drow, inv1, inv2, en, out


class Scatter:
    """Sum of row gradients per destination row and its bound: the bounds of the terms add, and the atomic adds (any
    order) of k terms into one entry add gamma(k) sum |terms|."""

    def __init__(self, n, D):
        self.acc, self.bnd, self.mag, self.cnt = (np.zeros((n, D)) for _ in range(4))

    def add(self, rows, g, dg):
        np.add.at(self.acc, rows, g)
        np.add.at(self.bnd, rows, dg)
        np.add.at(self.mag, rows, np.abs(g))
        np.add.at(self.cnt, rows, 1.0)
        return self

    def bound(self, slack=1.0):
        return slack * self.bnd + gamma(self.cnt) * self.mag


NCE_TEMPS = [0.05, 0.2, 0.5]


@pytest.mark.parametrize("B", LOSS_B)
@pytest.mark.parametrize("D", [32, 64, 128, 256])
def test_infonce_against_float64(ops, D, B):
    """Loss, lse, inv1 / inv2 and the scattered gradients of both views (tiled D = 64 kernels and the warp-per-row
    kernels of D = 32 / 128 / 256) at batch sizes across every split / tile edge, repeated indices, zero rows."""
    temp = NCE_TEMPS[(LOSS_B.index(B) + D) % 3]
    rng = np.random.default_rng(D * 131 + B)
    n = 3000
    ah, bh = loss_tables(rng, D, n)
    idx = batch_idx(rng, B, n)
    v1, v2, ti = padded(ah, 4), padded(bh, 12), T(idx)
    loss, (lse, inv1, inv2) = ops.infonce_fwd(v1, v2, ti, temp)
    gs = 1.7
    g1, g2 = ops.infonce_bwd(v1, v2, ti, temp, (lse, inv1, inv2), gs)
    d1, d2 = sentinel_buf(n + 2, D + 4), sentinel_buf(n + 2, D + 4)
    d1[:n, :D] = 0.0
    d2[:n, :D] = 0.0
    ops.scatter_add_rows(g1, ti, d1[:n, :D])
    ops.scatter_add_rows(g2, ti, d2[:n, :D])
    x1, x2 = ah[idx].astype(np.float64), bh[idx].astype(np.float64)
    lse_r, dlse, row, drow, i1, i2, en, ((gr1, db1), (gr2, db2)) = nce_ref(x1, x2, temp, gs)
    assert_within(f64(lse), lse_r, SLACK * dlse, "lse")
    assert_within(float(loss), row.mean(), SLACK * mean_bound(row, drow), "infonce loss")
    assert_within(f64(inv1), i1, i1 * en, "inv1")
    assert_within(f64(inv2), i2, i2 * en, "inv2")
    assert_within(f64(g1), gr1, SLACK * db1, "g1 rows")
    assert_within(f64(g2), gr2, SLACK * db2, "g2 rows")
    for d, gr, db, name in ((d1, gr1, db1, "d v1"), (d2, gr2, db2, "d v2")):
        assert_sentinel(d, slice(0, n), D)
        sc = Scatter(n, D).add(idx, gr, db)
        assert_within(f64(d[:n, :D]), sc.acc, sc.bound(SLACK), name)


def test_infonce_rejects_unsupported_D(ops):
    v = torch.zeros((10, 48), device=DEV)
    with pytest.raises(ops._lib.DiffMMError, match="D must be 32, 64, 128 or 256"):
        ops.infonce_fwd(v, v, torch.zeros(4, dtype=torch.int64, device=DEV), 0.2)


# ---------------------------------------------------------------------------------------- fused BPR + InfoNCE
FUSED = [  # P, B, (g_cl, g_bpr), index of a table without a gradient (or None)
    (1, 1, (0.37, -2.0), None),
    (2, 300, (0.0, 0.37), None),
    (8, 1024, (-2.0, 0.0), 3),
    (12, 769, (0.37, -2.0), 2),
]


@pytest.mark.parametrize("P,B,gg,null_tab", FUSED)
def test_bpr_infonce_against_float64(ops, P, B, gg, null_tab):
    """dmm_bpr_infonce_fwd / _bwd against a float64 restatement of the whole joint loss: per-problem temperatures and
    weights (one 0), user and item problems (row_offset U), one problem with the same table as both views, padded views
    and gradient tables (ld > 64), a table without a gradient; losses[P + 1] = sum_p weight_p losses[p]."""
    rng = np.random.default_rng(P * 1000 + B)
    Un, In, n_tab = 900, 1300, 4
    N = Un + In
    tabs_h = [rng.standard_normal((N, 64)).astype(F32) for _ in range(n_tab)]
    tabs_h[1][3] = 0.0
    users, pos, neg = rng.integers(0, Un, B), rng.integers(0, In, B), rng.integers(0, In, B)
    users[: min(B, 2)] = 3                               # a zero row (clamp) and a repeat
    problems_h = []
    for k in range(P):
        i1, i2 = (int(v) for v in rng.choice(n_tab, 2, replace=False))
        if k == 1:
            i2 = i1                                      # the same table as v1 and v2
        kind = "u" if k % 2 == 0 else "i"
        problems_h.append((i1, i2, kind, float(rng.choice(NCE_TEMPS)), 0.0 if k == P - 1 and P > 1 else float(rng.uniform(0.2, 1.5))))
    tabs = [padded(t, 16 * (k % 2)) if k % 2 else T(t) for k, t in enumerate(tabs_h)]
    tu, tp, tn = T(users), T(pos), T(neg)
    problems = [(i1, i2, tu if kind == "u" else tp, 0 if kind == "u" else Un, temp, w) for i1, i2, kind, temp, w in problems_h]
    bpr_tab = 0
    bpr = (bpr_tab, Un, tu, tp, tn)
    losses, saved = ops.bpr_infonce_fwd(tabs, problems, bpr, B)
    grads, bufs = [], []
    for k in range(n_tab):
        if k == null_tab:
            grads.append(None)
            bufs.append(None)
            continue
        buf = sentinel_buf(N + 1, 64 + 8 * k)
        buf[:N, :64] = 0.0
        grads.append(buf[:N, :64])
        bufs.append(buf)
    g_cl, g_bpr = gg
    ops.bpr_infonce_bwd(tabs, problems, bpr, B, saved, torch.tensor(g_cl, device=DEV), torch.tensor(g_bpr, device=DEV), grads)

    lh = losses.cpu().numpy()
    want = [Scatter(N, 64) for _ in range(n_tab)]
    means = []
    for p, (i1, i2, kind, temp, w) in enumerate(problems_h):
        rows = (users if kind == "u" else Un + pos)
        x1, x2 = tabs_h[i1][rows].astype(np.float64), tabs_h[i2][rows].astype(np.float64)
        lse_r, dlse, row, drow, inv1, inv2, en, ((g1, b1), (g2, b2)) = nce_ref(x1, x2, temp, w * g_cl)
        assert_within(lh[p], row.mean(), SLACK * mean_bound(row, drow), f"losses[{p}]")
        assert_within(f64(saved[0][p]), lse_r, SLACK * dlse, f"lse[{p}]")
        assert_within(f64(saved[1][p, 0]), inv1, inv1 * en, f"inv[{p}, 0]")
        assert_within(f64(saved[1][p, 1]), inv2, inv2 * en, f"inv[{p}, 1]")
        means.append(row.mean())
        want[i1].add(rows, g1, b1)
        want[i2].add(rows, g2, b2)
    u = tabs_h[bpr_tab][users].astype(np.float64)
    p_, q_ = tabs_h[bpr_tab][Un + pos].astype(np.float64), tabs_h[bpr_tab][Un + neg].astype(np.float64)
    row, drow, (gu, gp, gq), (bu, bp, bq) = bpr_ref(u, p_, q_, g_bpr)
    assert_within(lh[P], row.mean(), SLACK * mean_bound(row, drow), "losses[P] (BPR)")
    # the weighted total: P products and P additions of the kernel's own means
    wl = np.array([w for *_r, w in problems_h]) * lh[:P].astype(np.float64)
    assert_within(lh[P + 1], wl.sum(), gamma(2 * P) * np.abs(wl).sum(), "losses[P + 1]")
    for rows, g, b in ((users, gu, bu), (Un + pos, gp, bp), (Un + neg, gq, bq)):
        want[bpr_tab].add(rows, g, b)
    for k in range(n_tab):
        if bufs[k] is None:
            continue
        assert_sentinel(bufs[k], slice(0, N), 64)
        assert_within(f64(bufs[k][:N, :64]), want[k].acc, want[k].bound(SLACK), f"gradient table {k}")


def test_bpr_infonce_rejects_more_than_12_problems(ops):
    t = torch.zeros((10, 64), device=DEV)
    i = torch.zeros(4, dtype=torch.int64, device=DEV)
    with pytest.raises(ValueError, match="problems"):
        ops.bpr_infonce_fwd([t], [(0, 0, i, 0, 0.2, 1.0)] * 13, (0, 0, i, i, i), 4)
