"""GPU parity tests of the non-GEMM kernels against the numpy oracle and the golden vectors
(bit-exact for index work, stated tolerances for fp32).  Everything goes through the C ABI."""
import os

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import diffmm_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def T(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(DEV)


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


# ------------------------------------------------------------------------------------------- top-k
def _csr_ptr(k):
    p = np.zeros(len(k) + 1, dtype=np.int64)
    np.cumsum(k, out=p[1:])
    return p


def _run_topk(ops, scores, k, ld=None):
    n_rows, n_cols = scores.shape
    ld = n_cols if ld is None else ld
    buf = torch.full((n_rows, ld), float("nan"), device=DEV)
    buf[:, :n_cols] = T(scores)
    ptr = _csr_ptr(k)
    E = int(ptr[-1])
    users = torch.full((max(E, 1),), -1, dtype=torch.int32, device=DEV)
    items = torch.full((max(E, 1),), -1, dtype=torch.int32, device=DEV)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    ops.topk_edges(buf[:, :n_cols], n_cols, T(ptr), 100, users, items, status)
    torch.cuda.synchronize()
    return ptr, users.cpu().numpy()[:E], items.cpu().numpy()[:E], int(status.item())


def test_topk_golden_rebuild(ops):
    g = load_golden("rebuild")
    ptr, users, items, status = _run_topk(ops, g["scores"], g["deg"])
    assert status == 0
    want = O.topk_edges(g["scores"], g["deg"])
    for r, w in enumerate(want):
        np.testing.assert_array_equal(items[ptr[r]:ptr[r + 1]], w)
        assert (users[ptr[r]:ptr[r + 1]] == 100 + r).all()
        # against the reference's own torch.topk output (as a set)
        np.testing.assert_array_equal(np.sort(g["edge_i"][g["edge_u"] == r]), w)


@pytest.mark.parametrize("n_cols,ld", [(1, 4), (33, 36), (6710, 6720), (7050, 7104), (18357, 18368), (70001, 70004)])
def test_topk_random_vs_oracle(ops, n_cols, ld):
    rng = np.random.default_rng(n_cols)
    n_rows = 64
    scores = (rng.standard_normal((n_rows, n_cols)) * 0.05).astype(np.float32)
    k = np.minimum(rng.integers(0, 40, n_rows), n_cols)
    k[0], k[1], k[2] = 0, n_cols, min(n_cols, 603)
    ptr, _, items, status = _run_topk(ops, scores, k, ld)
    assert status == 0
    want = O.topk_edges(scores, k)
    for r, w in enumerate(want):
        np.testing.assert_array_equal(items[ptr[r]:ptr[r + 1]], w, err_msg=f"row {r} k={k[r]}")


def test_topk_generic_kernels_forced():
    """The register path covers every shipped row width, so the generic kernels (bucket histogram + radix
    select; rows wider than 32768 columns) are also forced onto small and mid-sized rows in a subprocess, on the
    widths of the register kernels' and the shared-memory kernel's boundaries (tests/test_rebuild_tail_kernels_gpu.py),
    with aligned rows and with ld % 4 == 1."""
    import subprocess
    import sys
    env = dict(os.environ, DMM_TOPK_GENERIC="1")
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    cap = (optin - 20480) // 4                       # widest row the shared-memory generic kernel stages
    args = ["500:500:0", "7050:7104:1", "33:36:1", "40000:40000:1"]
    for n in (8191, 8192, 8193, 16384, 16386, 32767, 32768, 32769, cap, cap + 1):
        ld4 = (n + 3) // 4 * 4
        args += [f"{n}:{ld4}:1", f"{n}:{ld4 + 1}:1"]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "dbg_topk.py"), *args], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == len(args) and all(ln.endswith("OK") for ln in lines), r.stdout + r.stderr


def test_topk_ties_and_signed_zero(ops):
    # heavy ties: quantised scores, +-0, duplicates of the k-th value -> value desc, index asc
    rng = np.random.default_rng(3)
    scores = rng.integers(-3, 4, (32, 500)).astype(np.float32)
    scores[0, :] = 0.0
    scores[1, ::2] = -0.0
    scores[1, 1::2] = 0.0
    k = rng.integers(1, 200, 32)
    ptr, _, items, _ = _run_topk(ops, scores, k)
    want = O.topk_edges(scores, k)
    for r, w in enumerate(want):
        np.testing.assert_array_equal(items[ptr[r]:ptr[r + 1]], w, err_msg=f"row {r}")


def test_topk_nan_and_inf_scores_follow_key_order(ops):
    # +NaN above +inf, -NaN below -inf (bit-pattern order), ties by column: register path hands NaN rows to the generic path
    rng = np.random.default_rng(8)
    scores = rng.standard_normal((16, 300)).astype(np.float32)
    scores[0, [5, 17]] = np.nan
    scores[1, 7] = np.float32(np.inf)
    scores[1, 9] = -np.float32(np.inf)
    scores[2, :] = np.nan
    neg_nan = np.frombuffer(np.uint32(0xFFC00000).tobytes(), dtype=np.float32)[0]
    scores[3, [1, 2, 3]] = neg_nan
    scores[3, 4] = np.nan
    k = rng.integers(1, 30, 16)
    k[3] = 299
    ptr, _, items, _ = _run_topk(ops, scores, k)
    # the kernel's stated total order (the oracle never sees NaN): order-preserving key of the fp32 bit pattern
    u = scores.view(np.uint32).astype(np.uint64)
    u = np.where(u == 0x80000000, 0, u)
    key = np.where(u & 0x80000000, (~u) & 0xFFFFFFFF, u | 0x80000000).astype(np.int64)
    for r in range(scores.shape[0]):
        order = np.lexsort((np.arange(scores.shape[1]), -key[r]))
        np.testing.assert_array_equal(items[ptr[r]:ptr[r + 1]], np.sort(order[:k[r]]), err_msg=f"row {r}")


def test_topk_k_larger_than_row_sets_status(ops):
    scores = np.zeros((2, 8), dtype=np.float32)
    _, _, _, status = _run_topk(ops, scores, np.array([9, 1]))
    assert status == 1


# ------------------------------------------------------------------------------------------- adjacency
def _edges_csr(u, i, U):
    order = np.lexsort((i, u))
    u, i = u[order], i[order]
    ptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(np.bincount(u, minlength=U), out=ptr[1:])
    return ptr, i.astype(np.int32)


def _check_adj(ops, u, i, U, I):
    ptr, items = _edges_csr(u, i, U)
    adj = ops.build_norm_adj(T(ptr), T(items), U, I)
    torch.cuda.synchronize()
    wp, wi, wv = O.normalized_adj_csr(u, i, U, I)
    np.testing.assert_array_equal(adj.ptr.cpu().numpy(), wp)
    np.testing.assert_array_equal(adj.idx.cpu().numpy().astype(np.int64), wi)
    got = adj.val.cpu().numpy()
    ulp = np.abs(got.view(np.int32).astype(np.int64) - wv.view(np.int32).astype(np.int64))
    assert ulp.max() <= 1, f"adjacency values differ by {ulp.max()} ulp"
    return adj


def test_adj_golden(ops):
    g = load_golden("rebuild")
    adj = _check_adj(ops, g["edge_u"], g["edge_i"], 40, 120)
    # against the reference's makeTorchAdj output (coalesced COO, row-major sorted)
    idx, val = g["adj_idx"], g["adj_val"]
    order = np.lexsort((idx[1], idx[0]))
    np.testing.assert_array_equal(adj.idx.cpu().numpy(), idx[1][order])
    np.testing.assert_array_equal(adj.val.cpu().numpy(), val[order])
    _check_adj(ops, g["trn_u"], g["trn_i"], 40, 120)


def test_adj_random_with_empty_rows_and_hub_item(ops):
    rng = np.random.default_rng(5)
    U, I = 3000, 1700
    u = rng.integers(0, U, 20000)
    i = np.where(rng.random(20000) < 0.2, 7, rng.integers(0, I, 20000))   # item 7 is a hub (>1024 users)
    key = np.unique(u.astype(np.int64) * I + i)
    u, i = key // I, key % I
    keep = (u % 17 != 0) & (i % 13 != 0)                                  # users / items without any edge
    _check_adj(ops, u[keep], i[keep], U, I)


# ------------------------------------------------------------------------------------------- SpMM
@pytest.mark.parametrize("D", [64, 32, 128])
def test_spmm_vs_oracle(ops, D):
    rng = np.random.default_rng(D)
    U, I = 2500, 1500
    u = rng.integers(0, U, 15000)
    i = np.where(rng.random(15000) < 0.25, 3, rng.integers(0, I, 15000))  # hub row > LONG_ROW
    key = np.unique(u.astype(np.int64) * I + i)
    u, i = key // I, key % I
    ptr, items = _edges_csr(u, i, U)
    adj = ops.build_norm_adj(T(ptr), T(items), U, I)
    x = rng.standard_normal((U + I, D)).astype(np.float32)
    z = rng.standard_normal((U + I, D)).astype(np.float32)
    want = O.spmm_csr(*O.normalized_adj_csr(u, i, U, I), x)
    got = ops.spmm(adj, T(x)).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=2e-5, atol=2e-6)
    got2 = ops.spmm(adj, T(x), alpha=0.5, beta=2.0, z=T(z)).cpu().numpy()
    np.testing.assert_allclose(got2, 0.5 * want + 2.0 * z, rtol=2e-5, atol=4e-6)
    # row-block form used by the row-partitioned propagation
    out = torch.zeros(U + I, D, device=DEV)
    ops.spmm(adj, T(x), out=out, row0=100, row1=2600)
    o = out.cpu().numpy()
    np.testing.assert_allclose(o[100:2600], want[100:2600], rtol=2e-5, atol=2e-6)
    assert not o[:100].any() and not o[2600:].any()


def test_cl_propagate_golden(ops):
    g = load_golden("cl_propagate")
    U, I = 40, 120
    ptr, items = _edges_csr(g["trn_u"], g["trn_i"], U)
    adj = ops.build_norm_adj(T(ptr), T(items), U, I)
    e = T(np.concatenate([g["u"], g["i"]]))
    outs = []
    for k in range(3):
        e = ops.spmm(adj, e)
        ops.sign_noise_(e, T(g["rand"][k]), float(g["noise_degree"]))
        outs.append(e)
    np.testing.assert_allclose(outs[0].cpu().numpy(), g["layer1"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(torch.stack(outs).mean(0).cpu().numpy(), g["mean"], rtol=2e-5, atol=2e-6)


# ------------------------------------------------------------------------------------------- losses
def test_bpr_golden(ops):
    g = load_golden("losses")
    B = g["u"].shape[0]
    ar = torch.arange(B, device=DEV)
    loss, (gu, gp, gn) = ops.bpr_fwd_bwd(T(g["u"]), T(np.concatenate([g["p"], g["n"]])), ar, ar, ar + B)
    np.testing.assert_allclose(loss.item(), g["bpr"], rtol=1e-5)
    np.testing.assert_allclose(gu.cpu().numpy(), g["g_u"], rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(gp.cpu().numpy(), g["g_p"], rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(gn.cpu().numpy(), g["g_n"], rtol=1e-4, atol=1e-7)


def test_infonce_golden(ops):
    g = load_golden("losses")
    v1, v2, idx = T(g["v1"]), T(g["v2"]), T(g["idx"])
    loss, saved = ops.infonce_fwd(v1, v2, idx, float(g["temp"]))
    np.testing.assert_allclose(loss.item(), g["infonce"], rtol=1e-5)
    g1, g2 = ops.infonce_bwd(v1, v2, idx, float(g["temp"]), saved)
    d1 = ops.scatter_add_rows(g1, idx, torch.zeros_like(v1))
    d2 = ops.scatter_add_rows(g2, idx, torch.zeros_like(v2))
    np.testing.assert_allclose(d1.cpu().numpy(), g["g_v1"], rtol=1e-4, atol=2e-7)
    np.testing.assert_allclose(d2.cpu().numpy(), g["g_v2"], rtol=1e-4, atol=2e-7)


def test_infonce_b1024_vs_oracle(ops):
    rng = np.random.default_rng(0)
    v1 = rng.standard_normal((5000, 64)).astype(np.float32)
    v2 = (v1 + 0.5 * rng.standard_normal((5000, 64))).astype(np.float32)
    idx = rng.integers(0, 5000, 1024)
    loss, _ = ops.infonce_fwd(T(v1), T(v2), T(idx), 0.5)
    np.testing.assert_allclose(loss.item(), O.info_nce(v1, v2, idx, 0.5), rtol=2e-5)


@pytest.mark.parametrize("B", [1, 31, 64, 257, 1000, 1024, 1500])
def test_infonce_tiled_fwd_bwd_vs_torch(ops, B):
    """Tiled D = 64 kernels (anchor tiles x column splits, cp.async double buffering) against torch fp32 autograd of
    Utils/Utils.py:57-75, ragged batch sizes, repeated indices."""
    rng = np.random.default_rng(B)
    n = 700
    v1 = torch.tensor(rng.standard_normal((n, 64)).astype(np.float32), device=DEV, requires_grad=True)
    v2 = torch.tensor((v1.detach().cpu().numpy() + 0.7 * rng.standard_normal((n, 64))).astype(np.float32), device=DEV,
                      requires_grad=True)
    idx = T(rng.integers(0, n, B))
    a = torch.nn.functional.normalize(v1[idx], dim=1)
    b = torch.nn.functional.normalize(v2[idx], dim=1)
    want = -torch.diag(torch.log_softmax(a @ b.T / 0.2, dim=1)).mean()
    want.backward()
    loss, saved = ops.infonce_fwd(v1.detach(), v2.detach(), idx, 0.2)
    np.testing.assert_allclose(loss.item(), want.item(), rtol=2e-5)
    g1, g2 = ops.infonce_bwd(v1.detach(), v2.detach(), idx, 0.2, saved, grad_scale=1.0)
    d1 = ops.scatter_add_rows(g1, idx, torch.zeros_like(v1))
    d2 = ops.scatter_add_rows(g2, idx, torch.zeros_like(v2))
    scale = float(v1.grad.abs().max())
    np.testing.assert_allclose(d1.cpu().numpy(), v1.grad.cpu().numpy(), rtol=2e-4, atol=2e-5 * scale)
    np.testing.assert_allclose(d2.cpu().numpy(), v2.grad.cpu().numpy(), rtol=2e-4, atol=2e-5 * scale)


@pytest.mark.parametrize("n_out", [1024, 200])
def test_csr_gather_act_vs_dense_and_scheduling_order(ops, n_out):
    """First Denoise layer on binary CSR rows (dmm_csr_gather_act) against the dense product on the same bf16 weights;
    the scheduling order (longest rows first, or any permutation) must not change a single bit."""
    rng = np.random.default_rng(n_out)
    U, I = 300, 900
    deg = rng.integers(0, 12, U)
    deg[[5, 77, 200]] = [400, 650, 129]                      # users with hundreds of interactions
    indptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(deg, out=indptr[1:])
    indices = np.concatenate([np.sort(rng.choice(I, d, replace=False)) for d in deg]).astype(np.int32)
    w = (rng.standard_normal((n_out, I)) * 0.05).astype(np.float32)          # first layer [H, I]
    bias = (rng.standard_normal(n_out) * 0.1).astype(np.float32)
    wt_hi, _ = ops.pack_bf16(T(w), transpose=True, split=False)              # W^T [I, pad(H)]
    ld = ops.pad_to(n_out, 8)

    def run(order):
        h = torch.full((U, ld), 3.0, dtype=torch.bfloat16, device=DEV)
        z = torch.full((U, ld), float("nan"), device=DEV)
        ops.csr_gather_act(T(indptr), T(indices), U, I, wt_hi, None, T(bias), 1, n_out, h[:, :n_out], None, z_f32=z[:, :n_out],
                           order=order)
        return h, z

    h0, z0 = run(None)
    x0 = np.zeros((U, I), dtype=np.float32)
    for u in range(U):
        x0[u, indices[indptr[u]:indptr[u + 1]]] = 1.0
    want_z = x0.astype(np.float64) @ wt_hi[:, :n_out].float().cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(z0[:, :n_out].cpu().numpy(), want_z, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(h0[:, :n_out].float().cpu().numpy(), np.tanh(want_z + bias), rtol=2 ** -8, atol=1e-5)
    from diffmm_b200.rebuild import longest_rows_first
    order = longest_rows_first(T(indptr), 0, U)
    assert order.dtype == torch.int32 and sorted(order.tolist()) == list(range(U))
    assert sorted(order[:3].tolist()) == [5, 77, 200]          # the users with more than 32 interactions come first
    for o in (order, T(rng.permutation(U).astype(np.int32))):
        h1, z1 = run(o)
        assert torch.equal(h1, h0) and torch.equal(z1[:, :n_out], z0[:, :n_out])


@pytest.mark.parametrize("split,weighted", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("n_out", [1024, 516, 260, 96])
def test_csr_gather_act_rows_divided_by_length_is_bit_identical(ops, n_out, split, weighted):
    """dmm_csr_gather_act_split (one warp per short row over all its columns, one warp per (row, slice) for the long rows,
    one launch) against dmm_csr_gather_act: same bits in h (hi, lo), z and the untouched padding -- binary and weighted
    rows, single-pass and split-bf16 weights, a row subset selected through row_ids, ragged last 8-column piece."""
    rng = np.random.default_rng(n_out + 2 * split + weighted)
    U, I = 700, 1200
    deg = rng.integers(0, 14, U)
    deg[[0, 13, 300, 699]] = [33, 640, 32, 257]              # around the threshold of 32 and far beyond it
    indptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(deg, out=indptr[1:])
    indices = np.concatenate([np.sort(rng.choice(I, d, replace=False)) for d in deg]).astype(np.int32)
    vals = T(rng.standard_normal(len(indices)).astype(np.float32)) if weighted else None
    w = (rng.standard_normal((n_out, I)) * 0.05).astype(np.float32)
    bias = T((rng.standard_normal(n_out) * 0.1).astype(np.float32))
    wt_hi, wt_lo = ops.pack_bf16(T(w), transpose=True, split=split)
    ld = ops.pad_to(n_out, 8)
    row0, n_rows = 100, 550                                    # a block of the users
    d_ptr, d_idx = T(indptr), T(indices)
    order = ops.rows_long_first(d_ptr, row0, n_rows, 32)
    assert int(order._dmm_counters[0]) == int((deg[row0:row0 + n_rows] > 32).sum())
    plain = order.clone()                                      # same permutation without the counters: the per-slice kernel

    def run(o):
        h = torch.full((n_rows, ld), 3.0, dtype=torch.bfloat16, device=DEV)
        hl = torch.full((n_rows, ld), 5.0, dtype=torch.bfloat16, device=DEV) if split else None
        z = torch.full((n_rows, ld), float("nan"), device=DEV)
        ops.csr_gather_act(d_ptr, d_idx, n_rows, I, wt_hi, wt_lo, bias, 1, n_out, h[:, :n_out],
                           hl[:, :n_out] if split else None, row0=row0, z_f32=z[:, :n_out], order=o, vals=vals)
        return h, hl, z

    h0, l0, z0 = run(plain)
    h1, l1, z1 = run(order)
    assert torch.equal(h1.view(torch.int16), h0.view(torch.int16))
    assert torch.equal(z1[:, :n_out], z0[:, :n_out]) and torch.isnan(z1[:, n_out:]).all()
    if split:
        assert torch.equal(l1.view(torch.int16), l0.view(torch.int16))
    assert not torch.isnan(z1[:, :n_out]).any()


# ------------------------------------------------------------------------------------------- staging kernels
def test_pack_bf16_split_and_transpose(ops):
    rng = np.random.default_rng(1)
    x = rng.standard_normal((70, 45)).astype(np.float32)
    hi, lo = ops.pack_bf16(T(x))
    assert hi.shape == (70, 64)
    rec = (hi.float() + lo.float()).cpu().numpy()
    np.testing.assert_allclose(rec[:, :45], x, rtol=2 ** -15)
    assert not rec[:, 45:].any()
    np.testing.assert_array_equal(hi[:, :45].cpu().float().numpy(), T(x).to(torch.bfloat16).float().cpu().numpy())
    hit, lot = ops.pack_bf16(T(x), transpose=True)
    assert hit.shape == (45, 128)
    np.testing.assert_array_equal(hit[:, :70].float().cpu().numpy(), hi[:, :45].float().cpu().numpy().T)
    np.testing.assert_array_equal(lot[:, :70].float().cpu().numpy(), lo[:, :45].float().cpu().numpy().T)
    assert not hit[:, 70:].float().cpu().numpy().any()


@pytest.mark.parametrize("shape", [(70, 45), (1024, 7060), (130, 64), (64, 130), (1, 9)])
@pytest.mark.parametrize("split", [True, False])
def test_pack_bf16_pair_equals_separate_packs(ops, shape, split):
    """Both orientations from one read (dmm_pack_bf16_pair) == the two separate dmm_pack_bf16 calls, bit for bit,
    including the zero padding."""
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    x = T(rng.standard_normal(shape).astype(np.float32))
    (n_hi, n_lo), (t_hi, t_lo) = ops.pack_bf16_pair(x, split=split)
    w_hi, w_lo = ops.pack_bf16(x, split=split)
    wt_hi, wt_lo = ops.pack_bf16(x, transpose=True, split=split)
    assert n_hi.shape == w_hi.shape and t_hi.shape == wt_hi.shape
    assert torch.equal(n_hi.view(torch.int16), w_hi.view(torch.int16)) and torch.equal(t_hi.view(torch.int16), wt_hi.view(torch.int16))
    if split:
        assert torch.equal(n_lo.view(torch.int16), w_lo.view(torch.int16)) and torch.equal(t_lo.view(torch.int16), wt_lo.view(torch.int16))
    else:
        assert n_lo is None and t_lo is None


def test_csr_rows_to_dense(ops):
    g = load_golden("generate_view")
    U, I = g["x0"].shape
    x = torch.full((U, 128), 7.0, device=DEV)
    a = torch.full((U, 192), 7.0, dtype=torch.bfloat16, device=DEV)
    ops.csr_rows_to_dense(T(g["indptr"]), T(g["indices"], torch.int32), U, I, x_f32=x, a_bf16=a)
    np.testing.assert_array_equal(x[:, :I].cpu().numpy(), g["x0"])
    np.testing.assert_array_equal(a[:, :I].float().cpu().numpy(), g["x0"])
    assert (x[:, I:] == 7).all() and (a[:, I:].float() == 7).all()
    ids = T(np.array([5, 0, 39, 5], dtype=np.int64))
    x2 = torch.empty((4, I), device=DEV)
    ops.csr_rows_to_dense(T(g["indptr"]), T(g["indices"], torch.int32), 4, I, row_ids=ids, x_f32=x2)
    np.testing.assert_array_equal(x2.cpu().numpy(), g["x0"][[5, 0, 39, 5]])


def test_time_embedding_and_q_sample(ops):
    g = load_golden("denoise_forward")
    q = load_golden("q_sample")
    w, b = g["p.emb_w"], g["p.emb_b"]
    t = g["t"]
    want = O.time_embedding(t, 10) @ w.T + b
    out = torch.empty((len(t), 10), device=DEV)
    ops.time_embedding(T(w), T(b), len(t), t=T(t), temb_f32=out)
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=1e-5, atol=1e-6)
    s = O.make_schedule(0.5, 1e-4, 0.02, 5)
    ca = T(s["sqrt_alphas_cumprod"][q["t"]].astype(np.float32))
    cb = T(s["sqrt_one_minus_alphas_cumprod"][q["t"]].astype(np.float32))
    xt = torch.empty_like(T(q["x0"]))
    ops.q_sample(T(q["x0"]), T(q["noise"]), ca, cb, 0, x_t=xt)
    np.testing.assert_allclose(xt.cpu().numpy(), q["xt_explicit"], rtol=1e-6, atol=1e-7)
    ops.q_sample(T(q["x0"]), T(q["randn"]), ca, cb, 1, x_t=xt)
    np.testing.assert_allclose(xt.cpu().numpy(), q["xt_default"], rtol=1e-5, atol=1e-7)
