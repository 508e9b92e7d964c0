"""GPU parity tests of the round-2 kernels, all through the C ABI:
  * chunk maxima written by the contraction epilogue (dmm_gemm_epilogue.cmax) == max over the written scores;
  * dmm_topk_edges_pruned == dmm_topk_edges == numpy oracle, bit for bit (widths 256 .. 500 000 columns, ties, NaN);
  * the sparse q_sample'd start of the reverse chain (dmm_csr_qsample_values + weighted dmm_csr_gather_act) == the dense
    q_sample + dense first layer of the reference formulation (Model.py:300-341);
  * device-side status bits; accurate tanh in the fp32-faithful (bf16x3) training forward."""
import numpy as np
import pytest
import torch

from oracle import diffmm_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(DEV)


@pytest.fixture(scope="module")
def ops():
    from diffmm_b200 import ops as o
    return o


def _ptr(k):
    p = np.zeros(len(k) + 1, dtype=np.int64)
    np.cumsum(k, out=p[1:])
    return p


def _chunk_max(scores_t):
    """torch restatement of the side array: NaN-propagating max over 32-column chunks (tail chunk over its valid columns)."""
    n_rows, n_cols = scores_t.shape
    nch = (n_cols + 31) // 32
    pad = torch.full((n_rows, nch * 32), float("-inf"), device=scores_t.device)
    pad[:, :n_cols] = scores_t
    return pad.view(n_rows, nch, 32).amax(dim=2)


def _run_pruned(ops, scores, k, order=None):
    n_rows, n_cols = scores.shape
    ld = ops.pad_to(n_cols, 4)
    buf = torch.zeros((n_rows, ld), device=DEV)
    buf[:, :n_cols] = T(scores)
    sc = buf[:, :n_cols]
    cm = ops.cmax_buffer(n_rows, n_cols, DEV)
    cm.fill_(float("nan"))
    cm[:, :(n_cols + 31) // 32] = _chunk_max(sc)
    ptr = _ptr(k)
    E = int(ptr[-1])
    users = torch.full((max(E, 1),), -1, dtype=torch.int32, device=DEV)[:E]
    items = torch.full((max(E, 1),), -1, dtype=torch.int32, device=DEV)[:E]
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    d_ptr = T(ptr)
    ops.topk_edges_pruned(sc, n_cols, cm, d_ptr, 7, users, items, status=status, order=order)
    items2 = torch.full((max(E, 1),), -1, dtype=torch.int32, device=DEV)[:E]
    ops.topk_edges(sc, n_cols, d_ptr, 7, None, items2)
    torch.cuda.synchronize()
    return ptr, users.cpu().numpy(), items.cpu().numpy(), items2.cpu().numpy(), int(status.item())


@pytest.mark.parametrize("n_cols", [256, 1000, 7050, 18357, 70001, 262144 + 37, 500000])
def test_pruned_topk_equals_full_topk_and_oracle(ops, n_cols):
    rng = np.random.default_rng(n_cols)
    n_rows = 48 if n_cols <= 70001 else 12
    scores = (rng.standard_normal((n_rows, n_cols)) * 0.05).astype(np.float32)
    k = np.minimum(rng.integers(0, 30, n_rows), n_cols)
    k[0], k[1], k[2], k[3], k[4] = 0, 1, min(n_cols, 64), min(n_cols, 65), min(n_cols, 603)
    k[5] = max(1, min(64, n_cols // 128))
    k[6] = max(1, min(700, n_cols // 64))        # deferred rows: two-level select, keys beyond the shared-memory staging
    ptr, users, items, items_full, status = _run_pruned(ops, scores, k)
    assert status == 0
    np.testing.assert_array_equal(items, items_full)
    want = O.topk_edges(scores, k)
    for r, w in enumerate(want):
        np.testing.assert_array_equal(items[ptr[r]:ptr[r + 1]], w, err_msg=f"row {r} k={k[r]}")
        assert (users[ptr[r]:ptr[r + 1]] == 7 + r).all()


def test_pruned_topk_ties_signed_zero_nan_and_order(ops):
    """Quantised scores (the k-th value is shared by hundreds of columns and by many chunk maxima), +-0, NaN rows: the
    pruned kernel must defer what it cannot rank exactly and agree with the whole-row kernels everywhere."""
    rng = np.random.default_rng(5)
    n_rows, n_cols = 40, 7050
    scores = rng.integers(-3, 4, (n_rows, n_cols)).astype(np.float32)
    scores[0, :] = 0.0
    scores[1, ::2] = -0.0
    scores[1, 1::2] = 0.0
    scores[2] = (rng.standard_normal(n_cols) * 0.1).astype(np.float32)
    scores[2, [40, 4000]] = np.nan
    scores[3] = (rng.standard_normal(n_cols) * 0.1).astype(np.float32)
    scores[3, 7] = np.inf
    scores[3, 6999] = -np.inf
    scores[4] = np.round(rng.standard_normal(n_cols), 1).astype(np.float32)      # moderate ties
    for r in range(5, 12):                                                       # the same maximum in many chunks
        scores[r] = (rng.standard_normal(n_cols) * 0.01).astype(np.float32)
        scores[r, rng.choice(n_cols, 300, replace=False)] = 1.0
    k = rng.integers(1, 50, n_rows)
    order = T(rng.permutation(n_rows).astype(np.int32))
    ptr, _, items, items_full, _ = _run_pruned(ops, scores, k, order=order)
    np.testing.assert_array_equal(items, items_full)
    u = scores.view(np.uint32).astype(np.uint64)
    u = np.where(u == 0x80000000, 0, u)
    key = np.where(u & 0x80000000, (~u) & 0xFFFFFFFF, u | 0x80000000).astype(np.int64)
    for r in range(n_rows):
        o = np.lexsort((np.arange(n_cols), -key[r]))
        np.testing.assert_array_equal(items[ptr[r]:ptr[r + 1]], np.sort(o[:k[r]]), err_msg=f"row {r}")


def test_pruned_topk_full_size_matches_torch_topk(ops):
    """baby-shape block through the pruned path vs torch.topk sets (continuous scores: no ties)."""
    g = torch.Generator(device=DEV).manual_seed(11)
    n_rows, n_cols = 19445, 7050
    buf = torch.randn((n_rows, ops.pad_to(n_cols, 4)), device=DEV, generator=g)
    sc = buf[:, :n_cols]
    rng = np.random.default_rng(2)
    k = np.clip(np.round(rng.lognormal(1.4, 0.9, n_rows)), 1, 600).astype(np.int64)
    ptr = _ptr(k)
    cm = ops.cmax_buffer(n_rows, n_cols, DEV)
    cm[:, :(n_cols + 31) // 32] = _chunk_max(sc)
    items = torch.empty(int(ptr[-1]), dtype=torch.int32, device=DEV)
    ops.topk_edges_pruned(sc, n_cols, cm, T(ptr), 0, None, items)
    got = items.cpu().numpy()
    for kk in np.unique(k):
        rows = np.nonzero(k == kk)[0]
        want = torch.topk(sc[T(rows)], int(kk), dim=1).indices.sort(dim=1).values.cpu().numpy()
        have = np.stack([got[ptr[r]:ptr[r + 1]] for r in rows])
        np.testing.assert_array_equal(have, want)


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
@pytest.mark.parametrize("M,N,K", [(300, 7050, 256), (129, 100, 64), (1000, 18357, 128)])
def test_gemm_chunk_maxima_match_the_written_scores(ops, precision, M, N, K):
    g = torch.Generator(device=DEV).manual_seed(M + N)
    a = torch.randn((M, K), device=DEV, generator=g)
    b = torch.randn((N, K), device=DEV, generator=g) * 0.1
    bias = torch.randn(N, device=DEV, generator=g)
    split = precision == "bf16x3"
    a_hi, a_lo = ops.pack_bf16(a, split=split)
    b_hi, b_lo = ops.pack_bf16(b, split=split)
    out = torch.zeros((M, ops.pad_to(N, 4)), device=DEV)[:, :N]
    cm = ops.cmax_buffer(M, N, DEV)
    cm.fill_(float("nan"))
    ops.gemm_bf16_tn(a_hi, a_lo, b_hi, b_lo, M, N, K, bias=bias, alpha=0.5, out_f32=out, cmax=cm)
    torch.cuda.synchronize()
    nch = (N + 31) // 32
    want = _chunk_max(out)
    assert torch.equal(cm[:, :nch], want)        # the maxima of exactly the values that were written


def test_sparse_qsample_start_equals_dense_qsample_start(ops):
    """rebuild from a q_sample'd start (conf/baby.toml: sampling_step 5): CSR rows + weighted gather vs the dense
    formulation of the reference (Model.py:300-341) on the same noise."""
    from diffmm_b200 import rebuild
    from diffmm_b200.Conf import Config
    from diffmm_b200.Model import Denoise, GaussianDiffusion
    U, I, H = 257, 1000, 128
    rng = np.random.default_rng(4)
    k = rng.integers(0, 12, U)
    k[3] = 300
    ptr = _ptr(k)
    idx = np.concatenate([np.sort(rng.choice(I, kk, replace=False)) for kk in k]).astype(np.int32)
    cfg = Config()
    cfg.base.precision = "bf16x3"
    cfg.base.denoise_dim = f"[{H}]"
    cfg.data.user_num, cfg.data.item_num = U, I
    torch.manual_seed(0)
    gd = GaussianDiffusion(cfg).to(DEV)
    den = Denoise([I, H], [H, I], cfg).to(DEV)
    x0 = np.zeros((U, I), dtype=np.float32)
    x0[np.repeat(np.arange(U), k), idx] = 1.0
    noise = torch.randn((U, I), device=DEV)
    for ss in (1, 5):
        dense = rebuild.denoise_chain(gd, den, x_dense=T(x0), sampling_step=ss, noise=noise).clone()
        sparse = rebuild.denoise_chain(gd, den, csr=(T(ptr), T(idx)), row0=0, n_rows=U, sampling_step=ss, noise=noise).clone()
        scale = float(dense.abs().max())
        assert float((dense - sparse).abs().max()) <= 2e-5 * max(scale, 1.0), ss
        # and against the numpy oracle's generate_view on the explicit x_t
        t = ss - 1
        nn = noise.cpu().numpy().astype(np.float64)
        nrm = np.maximum(np.sqrt((nn ** 2).sum(1, keepdims=True)), 1e-12)
        sched = O.make_schedule(cfg.hyper.noise_scale, cfg.hyper.noise_min, cfg.hyper.noise_max, cfg.hyper.steps)
        f = lambda p: p.detach().cpu().numpy()  # noqa: E731
        params = dict(emb_w=f(den.emb_layer.weight), emb_b=f(den.emb_layer.bias), w1=f(den.in_layers[0].weight),
                      b1=f(den.in_layers[0].bias), w2=f(den.out_layers[0].weight), b2=f(den.out_layers[0].bias),
                      gate_w=f(den.gate_layer.weight), gate_b=f(den.gate_layer.bias))
        a = np.float32(gd.sqrt_alphas_cumprod[t].item())
        b = np.float32(gd.sqrt_one_minus_alphas_cumprod[t].item())
        x_t = (a * x0 + b * (np.sign(x0) * (nn / nrm))).astype(np.float32)
        want = O.generate_view(sched, params, x_t, 0)
        assert float(np.abs(sparse.cpu().numpy() - want).max()) <= 5e-5 * max(float(np.abs(want).max()), 1.0), ss


def test_rebuild_status_bits(ops):
    # status bit 1 of the adjacency build (out-of-range item ids): tests/test_rebuild_tail_kernels_gpu.py
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    scores = torch.zeros((1, 8), device=DEV)
    out = torch.zeros(9, dtype=torch.int32, device=DEV)
    ops.topk_edges(scores, 8, T(np.array([0, 9], dtype=np.int64)), 0, None, out, status)
    assert int(status.item()) & 1


def test_bf16x3_training_forward_uses_the_accurate_tanh():
    """ADVICE r1: with lo operands the fp32-faithful instantiation (and its accurate tanh) must be selected."""
    from diffmm_b200.autograd import linear_tn
    g = torch.Generator(device=DEV).manual_seed(0)
    x = torch.randn((300, 200), device=DEV, generator=g)
    w = torch.nn.Parameter(torch.randn((96, 200), device=DEV, generator=g) * 0.1)
    b = torch.nn.Parameter(torch.randn(96, device=DEV, generator=g) * 0.1)
    y = linear_tn(x, w, b, 1, "bf16x3")
    z = linear_tn(x, w, b, 0, "bf16x3")                      # the same contraction without the activation
    assert float((y - torch.tanh(z.double()).float()).abs().max()) < 5e-7      # tanh.approx would be ~5e-4 off
    want = torch.tanh(x.double() @ w.double().t() + b.double()).float()
    assert float((y - want).abs().max()) < 5e-5                                # split-bf16 contraction error at |z| ~ 5


# ---------------------------------------------------------------------------------------------- fused training step
def _denoise_from_golden(cfg, g):
    from diffmm_b200.Model import Denoise
    I, H = g["w2"].shape
    den = Denoise([I, H], [H, I], cfg).to(DEV)
    with torch.no_grad():
        den.emb_layer.weight.copy_(T(g["emb_w"])); den.emb_layer.bias.copy_(T(g["emb_b"]))
        den.in_layers[0].weight.copy_(T(g["w1"])); den.in_layers[0].bias.copy_(T(g["b1"]))
        den.out_layers[0].weight.copy_(T(g["w2"])); den.out_layers[0].bias.copy_(T(g["b2"]))
        den.gate_layer.weight.copy_(T(g["gate_w"])); den.gate_layer.bias.copy_(T(g["gate_b"]))
    return den


def _grads(den):
    return {"w1": den.in_layers[0].weight.grad, "b1": den.in_layers[0].bias.grad, "w2": den.out_layers[0].weight.grad,
            "b2": den.out_layers[0].bias.grad, "emb_w": den.emb_layer.weight.grad, "emb_b": den.emb_layer.bias.grad,
            "gate_w": den.gate_layer.weight.grad, "gate_b": den.gate_layer.bias.grad}


def _rel(got, want):
    want = np.asarray(want, dtype=np.float64)
    got = got.detach().double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, dtype=np.float64)
    return float(np.abs(got - want).max() / (np.abs(want).max() + 1e-30))


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_fused_training_step_matches_the_reference_golden(precision, monkeypatch):
    """training_losses on the hand-scheduled step (train_step.py) against the tensors the UNMODIFIED reference produced
    (tests/golden/training_losses.npz): per-row float64 losses and all eight Denoise gradients."""
    from conftest import load_golden
    from diffmm_b200 import train_step
    from diffmm_b200.Conf import Config
    from diffmm_b200.Model import GaussianDiffusion
    from conftest import params_of
    g = load_golden("training_losses")
    calls = []
    orig = train_step.denoise_loss
    monkeypatch.setattr(train_step, "denoise_loss", lambda *a, **k: (calls.append(1), orig(*a, **k))[1])
    cfg = Config()
    pp = params_of(g)
    cfg.base.denoise_dim, cfg.base.precision = f"[{pp['w2'].shape[1]}]", precision
    cfg.hyper.noise_scale, cfg.hyper.sim_weight, cfg.train.reg = 0.5, 0.01, 1e-4
    den = _denoise_from_golden(cfg, pp)
    gd = GaussianDiffusion(cfg).to(DEV)
    losses = gd.training_losses(den, T(g["x0"]), T(g["i_embs"]), T(g["feat"]), timesteps=T(g["t"]), noise=T(g["noise"]))
    assert calls, "the fused step was not selected"
    assert losses.dtype == torch.float64 and losses.shape == (g["x0"].shape[0],)
    assert _rel(losses, g["losses"]) <= (2e-4 if precision == "bf16x3" else 1e-1)
    losses.mean().backward()
    for k, v in _grads(den).items():
        assert _rel(v, g[f"g.{k}"]) <= (1e-3 if precision == "bf16x3" else 1e-1), k


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_fused_training_step_equals_the_per_op_path(precision, monkeypatch):
    """Mid-size problem with ragged dimensions (B = 300, I = 1003, H = 136): fused step vs the per-op autograd path
    (LinearTN + ATen glue) on the same inputs."""
    from diffmm_b200.Conf import Config
    from diffmm_b200.Model import Denoise, GaussianDiffusion
    B, I, H = 300, 1003, 136
    rng = np.random.default_rng(1)
    cfg = Config()
    cfg.base.denoise_dim, cfg.base.precision = f"[{H}]", precision
    cfg.hyper.noise_scale = 0.5
    cfg.data.item_num = I
    torch.manual_seed(5)
    gd = GaussianDiffusion(cfg).to(DEV)
    den = Denoise([I, H], [H, I], cfg).to(DEV)
    x0 = (rng.random((B, I)) < 0.01).astype(np.float32)
    feat = T(rng.standard_normal((I, 64)).astype(np.float32) * 0.1)
    i_embs = T(rng.standard_normal((I, 64)).astype(np.float32) * 0.1)
    t = T(rng.integers(0, 5, B))
    noise = T(rng.standard_normal((B, I)).astype(np.float32))
    out = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("DIFFMM_FUSED_TRAIN", mode)
        den.zero_grad(set_to_none=True)
        losses = gd.training_losses(den, T(x0), i_embs, feat, timesteps=t, noise=noise)
        losses.mean().backward()
        out[mode] = (losses.detach().clone(), {k: v.detach().clone() for k, v in _grads(den).items()})
    tol_l, tol_g = (1e-4, 2e-3) if precision == "bf16x3" else (3e-2, 1.5e-1)
    assert _rel(out["1"][0], out["0"][0].cpu().numpy()) <= tol_l
    for k in out["1"][1]:
        assert _rel(out["1"][1][k], out["0"][1][k].cpu().numpy()) <= tol_g, k


# ---------------------------------------------------------------------------------------------- fused BPR + InfoNCE
@pytest.mark.parametrize("B,n_mod,cl_method", [(1024, 3, 0), (700, 2, 1), (33, 2, 0)])
def test_fused_joint_losses_equal_the_per_term_losses(B, n_mod, cl_method):
    """dmm_bpr_infonce_fwd / _bwd (all terms of a joint step in one call) vs bpr_loss + InfoNCE term by term
    (Utils/Utils.py:57-98, themselves golden-tested against the reference): values and table gradients."""
    from diffmm_b200.autograd import joint_losses
    from diffmm_b200.Utils.Utils import InfoNCE, bpr_loss
    U, I = 900, 500
    N = U + I
    g = torch.Generator(device=DEV).manual_seed(B)
    tabs = [torch.randn((N, 64), device=DEV, generator=g).requires_grad_(True) for _ in range(n_mod + 3)]
    users = torch.randint(0, U, (B,), device=DEV, generator=g)
    pos = torch.randint(0, I, (B,), device=DEV, generator=g)
    neg = torch.randint(0, I, (B,), device=DEV, generator=g)
    Tc, Rc, T, R = 0.2, 0.5, 0.5, 0.01
    i_mean, i_first = 1 + n_mod, 2 + n_mod
    problems = [(i_mean, i_first, "u", Tc, Rc), (i_mean, i_first, "i", Tc, Rc)]
    if cl_method == 1:
        for a, b in [(0, 1)] + ([(0, 2), (1, 2)] if n_mod == 3 else []):
            problems += [(1 + a, 1 + b, "u", T, R), (1 + a, 1 + b, "i", T, R)]
    else:
        for m in range(n_mod):
            problems += [(0, 1 + m, "u", T, R), (0, 1 + m, "i", T, R)]
    rec, cl = joint_losses(problems, 0, U, users, pos, neg, tabs)
    (rec * 1.7 + cl * 0.9).backward()
    got = [t.grad.clone() for t in tabs]
    for t in tabs:
        t.grad = None
    fin = tabs[0]
    rec_w = bpr_loss(fin[:U][users], fin[U:][pos], fin[U:][neg])
    cl_w = 0.0
    for (i1, i2, kind, temp, w) in problems:
        a, b = tabs[i1], tabs[i2]
        if kind == "u":
            cl_w = cl_w + InfoNCE(a[:U], b[:U], users, temp) * w
        else:
            cl_w = cl_w + InfoNCE(a[U:], b[U:], pos, temp) * w
    (rec_w * 1.7 + cl_w * 0.9).backward()
    assert float((rec - rec_w).abs()) <= 2e-6 * max(1.0, float(rec_w.abs()))
    assert float((cl - cl_w).abs()) <= 1e-5 * max(1.0, float(cl_w.abs()))
    for k, t in enumerate(tabs):
        scale = float(t.grad.abs().max()) + 1e-30
        assert float((got[k] - t.grad).abs().max()) <= 2e-5 * scale, k


# ---------------------------------------------------------------------------------------------- SpMM variants
def test_spmm_units_kernel_row_ranges(ops):
    """Round-2 SpMM (length-sorted units, chunked long rows, fixed-order reduce) on a graph with heavy rows: whole product,
    row-block calls and the alpha / beta epilogue vs the numpy oracle."""
    from diffmm_b200 import synth
    U, I = 3000, 800
    inter = synth.interactions(U, I, seed=5, mean_deg=7.0, heavy_frac=0.03)
    ptr, idx = T(inter.indptr), T(inter.indices)
    adj = ops.build_norm_adj(ptr, idx, U, I)
    N = U + I
    rng = np.random.default_rng(0)
    x = rng.standard_normal((N, 64)).astype(np.float32)
    want = O.spmm_csr(adj.ptr.cpu().numpy(), adj.idx.cpu().numpy(), adj.val.cpu().numpy(), x)
    xd = T(x)
    y = ops.spmm(adj, xd).cpu().numpy()
    np.testing.assert_allclose(y, want, rtol=2e-5, atol=2e-6)
    out = torch.full((N, 64), float("nan"), device=DEV)
    for a, b in [(0, 1000), (1000, U), (U, U + 300), (U + 300, N)]:
        ops.spmm(adj, xd, out=out, row0=a, row1=b)
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=2e-5, atol=2e-6)
    z = T(rng.standard_normal((N, 64)).astype(np.float32))
    y2 = ops.spmm(adj, xd, alpha=0.5, beta=2.0, z=z).cpu().numpy()
    np.testing.assert_allclose(y2, 0.5 * want + 2.0 * z.cpu().numpy(), rtol=3e-5, atol=3e-6)


def test_spmm_norm_bf16_exact_on_the_rounded_table(ops):
    """dmm_spmm_table_bf16 + dmm_spmm_norm_bf16 (separable normalisation, bf16 gather table, units sorted by length):
      * the table is bf16_rn(d^-1/2 x) exactly (d from the row pointers, [x ; x2] never concatenated);
      * Y = alpha d_r^-1/2 sum_c T[c] (+ beta Z) against the same sum in float64 on the very table the kernel read
        (fp32 accumulation: 2e-6 relative), whole product and row blocks, rows with 0 .. 3000 entries;
      * against the fp32 product it stays within bf16 rounding of the gathered operand (the stated bf16 tolerance)."""
    from diffmm_b200 import synth
    U, I = 3000, 800
    inter = synth.interactions(U, I, seed=5, mean_deg=7.0, heavy_frac=0.03)
    adj = ops.build_norm_adj(T(inter.indptr), T(inter.indices), U, I)
    assert adj.separable
    N = U + I
    rng = np.random.default_rng(1)
    x = rng.standard_normal((N, 64)).astype(np.float32)
    xu, xi = T(x[:U]), T(x[U:])
    ptr, idx, val = adj.ptr.cpu().numpy(), adj.idx.cpu().numpy(), adj.val.cpu().numpy()
    deg = np.diff(ptr)
    assert deg.max() > 500 and deg.min() >= 1
    dinv = (1.0 / np.sqrt(deg.astype(np.float64))).astype(np.float32)
    table = ops.spmm_table_bf16(adj, xu, xi)
    want_t = torch.from_numpy(dinv[:, None] * x).bfloat16()
    assert torch.equal(table.cpu(), want_t)
    tf = table.float().cpu().numpy().astype(np.float64)
    rows = np.repeat(np.arange(N), deg)
    ref = np.zeros((N, 64))
    np.add.at(ref, rows, tf[idx])
    ref *= dinv[:, None].astype(np.float64)
    y = ops.spmm_norm_bf16(adj, xu, x2=xi).cpu().numpy()
    np.testing.assert_allclose(y, ref, rtol=3e-6, atol=3e-6 * np.abs(ref).max())
    out = torch.full((N, 64), float("nan"), device=DEV)
    for a, b in [(0, 1000), (1000, U), (U, U + 300), (U + 300, N)]:
        ops.spmm_norm_bf16(adj, table=table, out=out, row0=a, row1=b)
    assert np.array_equal(out.cpu().numpy(), y)                      # row blocks: same units, same sums, bit for bit
    z = T(rng.standard_normal((N, 64)).astype(np.float32))
    y2 = ops.spmm_norm_bf16(adj, T(x), alpha=0.5, beta=2.0, z=z).cpu().numpy()
    np.testing.assert_allclose(y2, 0.5 * ref + 2.0 * z.cpu().numpy(), rtol=1e-5, atol=1e-5 * np.abs(ref).max())
    full = O.spmm_csr(ptr, idx, val, x)                              # fp32 values, fp32 table
    assert np.abs(y - full).max() <= 4e-3 * np.abs(full).max()
    assert np.linalg.norm(y - full) <= 2e-3 * np.linalg.norm(full)
    # the separability the kernel relies on: val == d_r^-1/2 d_c^-1/2 to fp32 rounding
    assert np.abs(val - dinv[rows] * dinv[idx]).max() <= 2e-7 * val.max()
    # deterministic
    assert np.array_equal(ops.spmm_norm_bf16(adj, table=table).cpu().numpy(), y)


def test_spmm_bf16_autograd_path_matches_fp32_within_tolerance(ops, monkeypatch):
    """autograd.spmm under set_spmm_precision("bf16"): value and gradient (A symmetric: the same product on g) within the
    bf16 tolerance of the fp32 path; non-separable adjacencies keep the fp32 kernel."""
    from diffmm_b200 import autograd as ag, synth
    from diffmm_b200.DataHandler import csr_from_torch_sparse
    monkeypatch.setenv("DIFFMM_SPMM_BF16_MIN_NNZ", "0")
    U, I = 2000, 600
    inter = synth.interactions(U, I, seed=2, mean_deg=6.0, heavy_frac=0.02)
    adj = ops.build_norm_adj(T(inter.indptr), T(inter.indices), U, I)
    x = torch.randn(U + I, 64, device=DEV)
    w = torch.randn(U + I, 64, device=DEV)
    res = {}
    for prec in ("bf16x3", "bf16"):
        xx = x.clone().requires_grad_(True)
        yy = ag.spmm(adj, ag.spmm_cat(adj, xx[:U], xx[U:], prec), prec)
        (yy * w).sum().backward()
        res[prec] = (yy.detach(), xx.grad.detach())
    for a, b in zip(res["bf16"], res["bf16x3"]):
        assert float((a - b).norm() / b.norm()) <= 3e-3
        assert float((a - b).abs().max() / b.abs().max()) <= 6e-3
    assert torch.equal(res["bf16x3"][0], ops.spmm(adj, ops.spmm(adj, x)))          # bf16x3: the fp32 kernel, untouched
    generic = csr_from_torch_sparse(adj.to_torch_coo())
    assert not generic.separable
    assert torch.equal(ag.spmm(generic, x, "bf16"), ops.spmm(generic, x))


def test_chi2_rng_qsample_values_are_standard_normal_and_counter_based(ops):
    """dmm_csr_qsample_values_rng: (vals - a) / b = n_c / ||n|| for i.i.d. N(0, 1) rows generated in the kernel.  Checked:
    moments of sqrt(I) (vals - a) / b (mean 0, variance 1, kurtosis 3), row norms through the identity
    sum_c (n_c / ||n||)^2 over a FULL row = 1, determinism per seed, independence of blocking (element (r, c) is a pure
    function of (seed, r, c)), and a different stream for a different seed."""
    U, I = 600, 4093
    rng = np.random.default_rng(0)
    k = rng.integers(0, 40, U)
    k[0], k[1] = I, 0                                   # one full row (identity check), one empty row
    ptr = _ptr(k)
    idx = np.concatenate([np.sort(rng.choice(I, kk, replace=False)) for kk in k]).astype(np.int32)
    d_ptr, d_idx = T(ptr), T(idx)
    a, b = 0.9, 0.4
    seed = torch.tensor([1234567], dtype=torch.int64, device=DEV)
    ref = torch.empty(idx.size, dtype=torch.float32, device=DEV)
    ops.csr_qsample_values_rng(d_ptr, d_idx, U, I, seed, a, b, ref)
    z = (ref.cpu().numpy().astype(np.float64) - a) / b   # n_c / ||n||
    assert abs((z[:I] ** 2).sum() - 1.0) < 1e-4          # row 0 holds every column: the rest of the norm is empty
    s = z[I:] * np.sqrt(I)
    assert abs(s.mean()) < 0.03 and abs(s.var() - 1.0) < 0.05 and abs((s ** 4).mean() / s.var() ** 2 - 3.0) < 0.25
    # deterministic, and independent of how the rows are blocked / addressed
    vals2 = torch.empty_like(ref)
    ops.csr_qsample_values_rng(d_ptr, d_idx, 300, I, seed, a, b, vals2)
    ops.csr_qsample_values_rng(d_ptr, d_idx, U - 300, I, seed, a, b, vals2, row0=300)
    assert torch.equal(ref, vals2)
    vals3 = torch.full_like(ref, float("nan"))
    ids = torch.arange(U - 1, -1, -1, device=DEV)
    ops.csr_qsample_values_rng(d_ptr, d_idx, U, I, seed, a, b, vals3, row_ids=ids)
    assert torch.equal(ref, vals3)
    vals4 = torch.empty_like(ref)
    ops.csr_qsample_values_rng(d_ptr, d_idx, U, I, seed + 1, a, b, vals4)
    assert float((vals4 - ref).abs().max()) > 1e-3


@pytest.mark.parametrize("n_cols", [40, 70, 7050])
def test_chi2_qsample_values_follow_the_exact_beta_law(ops, n_cols):
    """One interaction per user: z^2 = n_c^2 / ||n||^2 ~ Beta(1/2, (I - 1)/2) exactly.  Checks mean and variance over
    40 000 rows for the generator of support normals + one chi-square(I - 1) variate (explicit normals for I - 1 <= 64,
    Marsaglia-Tsang above)."""
    U = 40000
    rng = np.random.default_rng(n_cols)
    ptr = np.arange(U + 1, dtype=np.int64)
    idx = rng.integers(0, n_cols, U).astype(np.int32)
    seed = torch.tensor([99], dtype=torch.int64, device=DEV)
    al, be = 0.5, 0.5 * (n_cols - 1)
    mean = al / (al + be)
    var = al * be / ((al + be) ** 2 * (al + be + 1))
    vals = torch.empty(U, dtype=torch.float32, device=DEV)
    ops.csr_qsample_values_rng(T(ptr), T(idx), U, n_cols, seed, 0.0, 1.0, vals)
    z2 = vals.cpu().numpy().astype(np.float64) ** 2
    assert abs(z2.mean() - mean) < 5.0 * np.sqrt(var / U), (z2.mean(), mean)
    assert abs(z2.var() - var) < 0.08 * var, (z2.var(), var)


@pytest.mark.parametrize("n_cols", [50, 7050])
def test_chi2_qsample_short_row_path_equals_general_path(ops, n_cols):
    """Rows of fewer than 32 entries take the one-round path of the sufficient-statistics generator (one entry per lane, the
    chi-square draw in lockstep on the free lane).  The values are a pure function of (seed, row, column, support size):
    the same rows padded to >= 32 entries with out-of-range columns (ignored by contract) go through the general path and
    must give the same bits."""
    rng = np.random.default_rng(n_cols + 1)
    U = 3000
    deg = rng.integers(0, 32, U)
    deg[:4] = [0, 1, 31, 30]
    rows = [np.sort(rng.choice(n_cols, d, replace=False)).astype(np.int32) for d in deg]
    ptr_a = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(deg, out=ptr_a[1:])
    idx_a = np.concatenate(rows) if ptr_a[-1] else np.zeros(0, dtype=np.int32)
    padded = [np.concatenate([r, np.full(40 - len(r), n_cols, dtype=np.int32)]) if len(r) else r for r in rows]
    ptr_b = np.zeros(U + 1, dtype=np.int64)
    np.cumsum([len(r) for r in padded], out=ptr_b[1:])
    idx_b = np.concatenate(padded)
    seed = torch.tensor([1234567], dtype=torch.int64, device=DEV)
    va = torch.zeros(len(idx_a), dtype=torch.float32, device=DEV)
    vb = torch.zeros(len(idx_b), dtype=torch.float32, device=DEV)
    ops.csr_qsample_values_rng(T(ptr_a), T(idx_a), U, n_cols, seed, 0.25, 0.75, va)
    ops.csr_qsample_values_rng(T(ptr_b), T(idx_b), U, n_cols, seed, 0.25, 0.75, vb)
    keep = torch.from_numpy(idx_b < n_cols).to(DEV)
    assert torch.equal(va, vb[keep])
    assert float((va - 0.25).abs().max()) > 0.0
