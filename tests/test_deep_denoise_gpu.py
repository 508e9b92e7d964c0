"""denoise_dim with more than one entry (reference Model.py:160-162,211-218) on the B200: the reverse chain in both modes
(hidden-space and literal), the rebuild's top-k on its scores, the fused training step's loss and every gradient, an
epoch in graph mode and the drop-in generate_view.

For denoise_dim = [d_1, ..., d_L] the network is in_layers ([x_t, temb] -> d_L -> ... -> d_1) and out_layers
(d_1 -> ... -> d_L -> items): 2L Linear layers, 2L - 1 hidden activations.  The parametrization covers L = 2 and 3,
widths that are not multiples of 64, a 1024-wide hidden-space operator P and the row-divided CSR gather."""
import ast

import numpy as np
import pytest
import torch

from oracle import diffmm_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DIMS = ["[1000, 200]", "[512, 1024]", "[96, 160, 136]"]
PRECISIONS = ["bf16x3", "bf16"]


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _ptr(k):
    p = np.zeros(len(k) + 1, dtype=np.int64)
    np.cumsum(k, out=p[1:])
    return p


def _model(denoise_dim, I, precision, seed=0, noise_scale=None):
    """GaussianDiffusion + Denoise built the way Main.py:155-156 builds them."""
    from diffmm_b200.Conf import Config
    from diffmm_b200.Model import Denoise, GaussianDiffusion
    cfg = Config()
    cfg.base.denoise_dim, cfg.base.precision = denoise_dim, precision
    cfg.data.item_num = I
    if noise_scale is not None:
        cfg.hyper.noise_scale = noise_scale
    torch.manual_seed(seed)
    gd = GaussianDiffusion(cfg).to(DEV)
    out_dims = ast.literal_eval(denoise_dim) + [I]
    den = Denoise(out_dims[::-1], out_dims, cfg).to(DEV)
    return cfg, gd, den


def _layers(den):
    return list(den.in_layers) + list(den.out_layers)


def _params(den):
    f = lambda t: t.detach().cpu().numpy()  # noqa: E731
    return dict(emb_w=f(den.emb_layer.weight), emb_b=f(den.emb_layer.bias),
                w1=[f(m.weight) for m in den.in_layers], b1=[f(m.bias) for m in den.in_layers],
                w2=[f(m.weight) for m in den.out_layers], b2=[f(m.bias) for m in den.out_layers],
                gate_w=f(den.gate_layer.weight), gate_b=f(den.gate_layer.bias))


def _csr_rows(U, I, seed):
    rng = np.random.default_rng(seed)
    k = rng.integers(0, 12, U)
    k[3], k[10] = 300, 64                      # rows longer than 32 entries: the row-divided gather
    idx = np.concatenate([np.sort(rng.choice(I, kk, replace=False)) for kk in k]).astype(np.int32)
    x0 = np.zeros((U, I), dtype=np.float32)
    x0[np.repeat(np.arange(U), k), idx] = 1.0
    return k, _ptr(k), idx, x0


def _tol(precision):
    # (vs the oracle, hidden vs full), relative to the score scale
    return (5e-5, 2e-5) if precision == "bf16x3" else (1e-2, 1e-2)


# ---------------------------------------------------------------------------------------------- 1. chain vs oracle
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("denoise_dim", DIMS)
def test_deep_chain_matches_the_oracle_in_both_modes(denoise_dim, precision):
    from diffmm_b200 import rebuild
    U, I = 257, 1000
    cfg, gd, den = _model(denoise_dim, I, precision)
    k, ptr, idx, x0 = _csr_rows(U, I, 4)
    d_ptr, d_idx = T(ptr), T(idx)
    order = rebuild.longest_rows_first(d_ptr, 0, U)
    sched = O.make_schedule(cfg.hyper.noise_scale, cfg.hyper.noise_min, cfg.hyper.noise_max, cfg.hyper.steps)
    params = _params(den)
    noise = torch.randn((U, I), device=DEV)
    nn = noise.cpu().numpy().astype(np.float64)
    nrm = np.maximum(np.sqrt((nn ** 2).sum(1, keepdims=True)), 1e-12)
    tol_o, tol_m = _tol(precision)
    with torch.no_grad():
        # dense start
        res = {m: rebuild.denoise_chain(gd, den, x_dense=T(x0), sampling_step=0, mode=m).clone() for m in ("hidden", "full")}
        want = O.generate_view(sched, params, x0, 0)
        scale = max(float(np.abs(want).max()), 1.0)
        for m, got in res.items():
            assert float(np.abs(got.cpu().numpy() - want).max()) <= tol_o * scale, ("dense", m)
        assert float((res["hidden"] - res["full"]).abs().max()) <= tol_m * scale, "dense"
        # CSR rows, binary start and q_sample'd starts (injected noise)
        for ss in (0, 1, 5):
            res = {m: rebuild.denoise_chain(gd, den, csr=(d_ptr, d_idx), row0=0, n_rows=U, sampling_step=ss, noise=noise,
                                            mode=m, order=order).clone() for m in ("hidden", "full")}
            if ss == 0:
                x_t = x0
            else:
                a = np.float32(gd.sqrt_alphas_cumprod[ss - 1].item())
                b = np.float32(gd.sqrt_one_minus_alphas_cumprod[ss - 1].item())
                x_t = (a * x0 + b * (np.sign(x0) * (nn / nrm))).astype(np.float32)
            want = O.generate_view(sched, params, x_t, 0)
            scale = max(float(np.abs(want).max()), 1.0)
            for m, got in res.items():
                err = float(np.abs(got.cpu().numpy() - want).max())
                assert err <= tol_o * scale, (ss, m, err / scale)
            assert float((res["hidden"] - res["full"]).abs().max()) <= tol_m * scale, ss


# ---------------------------------------------------------------------------------------------- 2. full size
def _ref_chain64(gd, den, x0):
    """The reference's literal chain (Model.py:183-220,300-322,357-378) in float64 on the device."""
    D = lambda p: p.detach().double()  # noqa: E731
    n = x0.shape[0]
    x = x0.double()
    half = den.time_emb_dim // 2
    freqs = torch.exp(-np.log(10000.0) * torch.arange(half, device=DEV, dtype=torch.float32) / half).double()
    for i in range(gd.steps - 1, -1, -1):
        ang = torch.full((n, 1), float(i), device=DEV, dtype=torch.float64) * freqs[None]
        temb = torch.cat([torch.cos(ang), torch.sin(ang)], -1) @ D(den.emb_layer.weight).t() + D(den.emb_layer.bias)
        h = torch.cat([x, temb], -1)
        for m in den.in_layers:
            h = torch.tanh(h @ D(m.weight).t() + D(m.bias))
        for j, m in enumerate(den.out_layers):
            h = h @ D(m.weight).t() + D(m.bias)
            if j != len(den.out_layers) - 1:
                h = torch.tanh(h)
        x = float(np.float32(gd._h_coef1[i])) * h + float(np.float32(gd._h_coef2[i])) * x
    return x


def test_deep_chain_precision_at_the_baby_shape():
    """Every user of the baby shape (19445 x 7050) with denoise_dim [1024, 1024], both precisions, against float64:
    the same gates as the one-layer chain (tests/test_precision_fullsize_gpu.py)."""
    from diffmm_b200 import ops, synth
    from diffmm_b200.rebuild import denoise_chain
    U, I, _ = synth.SHAPES["baby"]
    inter = synth.interactions(U, I, seed=0)
    ptr, idx = T(inter.indptr), T(inter.indices)
    deg = np.diff(inter.indptr)
    cfg, gd, den = _model("[1024, 1024]", I, "bf16")
    stats = {p: dict(max_err=0.0, hit=0) for p in PRECISIONS}
    scale = 0.0
    B = 2048
    with torch.no_grad():
        for b0 in range(0, U, B):
            n = min(B, U - b0)
            x0 = torch.zeros((n, ops.pad_to(I, 4)), device=DEV)[:, :I]
            ops.csr_rows_to_dense(ptr, idx, n, I, row0=b0, x_f32=x0)
            want = _ref_chain64(gd, den, x0)
            scale = max(scale, float(want.abs().max()))
            kb = T(deg[b0:b0 + n])
            kmax = int(kb.max())
            ar = torch.arange(kmax, device=DEV)[None, :] < kb[:, None]
            top_w = torch.topk(want, kmax, dim=1).indices
            for p in stats:
                got = denoise_chain(gd, den, csr=(ptr, idx), row0=b0, n_rows=n, precision=p)
                stats[p]["max_err"] = max(stats[p]["max_err"], float((got.double() - want).abs().max()))
                top_g = torch.topk(got, kmax, dim=1).indices
                mask = torch.zeros((n, I), dtype=torch.bool, device=DEV)
                mask.scatter_(1, torch.where(ar, top_w, top_w[:, :1]), True)
                stats[p]["hit"] += int((mask.gather(1, top_g) & ar).sum())
    E = int(deg.sum())
    out = {p: dict(max_err_over_score_scale=s["max_err"] / scale, topk_edge_overlap=s["hit"] / E) for p, s in stats.items()}
    print("baby [1024, 1024]", out, "score scale", scale)
    assert out["bf16x3"]["max_err_over_score_scale"] <= 3e-5, out
    assert out["bf16x3"]["topk_edge_overlap"] >= 0.9999, out
    assert out["bf16"]["max_err_over_score_scale"] <= 1e-2, out
    assert out["bf16"]["topk_edge_overlap"] >= 0.97, out


# ---------------------------------------------------------------------------------------------- 3. rebuild
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("denoise_dim", DIMS)
def test_deep_rebuild_edges_pruned_unpruned_and_chain_topk_agree(denoise_dim, precision, monkeypatch):
    from diffmm_b200 import ops, rebuild
    U, I = 700, 1000
    _, gd, den = _model(denoise_dim, I, precision, seed=1)
    _, _, den2 = _model(denoise_dim, I, precision, seed=2)
    k, ptr, idx, _ = _csr_rows(U, I, 6)
    d_ptr, d_idx = T(ptr), T(idx)
    dens = {"image": den, "text": den2}
    out = {}
    for prune in ("1", "0"):
        monkeypatch.setenv("DIFFMM_TOPK_PRUNE", prune)
        items = rebuild.rebuild_edges(gd, dens, d_ptr, d_idx, U, I, sampling_step=0, block_rows=256)
        out[prune] = {m: v.clone() for m, v in items.items()}
    for m, d in dens.items():
        assert torch.equal(out["1"][m], out["0"][m]), m
        want = torch.empty_like(out["1"][m])
        with torch.no_grad():
            for b0 in range(0, U, 256):
                n = min(256, U - b0)
                sc = rebuild.denoise_chain(gd, d, csr=(d_ptr, d_idx), row0=b0, n_rows=n, sampling_step=0,
                                           order=rebuild.longest_rows_first(d_ptr, b0, n))
                ops.topk_edges(sc, I, d_ptr[b0:], b0, None, want)
        assert torch.equal(out["1"][m], want), m


# ---------------------------------------------------------------------------------------------- 4. fused training step
def _train_inputs(B, I, seed=1):
    rng = np.random.default_rng(seed)
    x0 = T((rng.random((B, I)) < 0.01).astype(np.float32))
    feat = T(rng.standard_normal((I, 64)).astype(np.float32) * 0.1)
    i_embs = T(rng.standard_normal((I, 64)).astype(np.float32) * 0.1)
    t = T(rng.integers(0, 5, B))
    noise = T(rng.standard_normal((B, I)).astype(np.float32))
    return x0, feat, i_embs, t, noise


def _all_grads(den):
    g = {n: p.grad for n, p in den.named_parameters()}
    assert all(v is not None for v in g.values()), [n for n, v in g.items() if v is None]
    return g


def _rel(got, want):
    return float((got.double() - want.double()).abs().max() / (want.double().abs().max() + 1e-30))


def _training_losses64(cfg, gd, den, x0, i_embs, feat, t, noise):
    """Model.py:385-428 with Denoise.forward (Model.py:183-220) in float64 torch autograd; returns the loss and the
    float64 leaf copies of the Denoise parameters (by name)."""
    P = {n: p.detach().double().requires_grad_(True) for n, p in den.named_parameters()}
    L = len(den.in_layers)
    x0d, f = x0.double(), feat.double()
    x_t = gd.sqrt_alphas_cumprod[t].float().double()[:, None] * x0d + \
        gd.sqrt_one_minus_alphas_cumprod[t].float().double()[:, None] * noise.double()
    half = den.time_emb_dim // 2
    freqs = torch.exp(-np.log(10000.0) * torch.arange(half, device=DEV, dtype=torch.float32) / half)
    temp = t[:, None].float() * freqs[None]
    temb = torch.cat([torch.cos(temp), torch.sin(temp)], -1).double() @ P["emb_layer.weight"].t() + P["emb_layer.bias"]
    proj = x_t @ f
    gate = torch.sigmoid(proj @ P["gate_layer.weight"].t() + P["gate_layer.bias"])
    h = torch.cat([x_t + (proj * gate) @ f.t(), temb], -1)
    for k in range(L):
        h = torch.tanh(h @ P[f"in_layers.{k}.weight"].t() + P[f"in_layers.{k}.bias"])
    for k in range(L):
        h = h @ P[f"out_layers.{k}.weight"].t() + P[f"out_layers.{k}.bias"]
        if k != L - 1:
            h = torch.tanh(h)
    mse = ((h - x0d) ** 2).mean(-1)
    ac = gd.alphas_cumprod
    snr = lambda tt: ac[tt] / (1 - ac[tt] + 1e-8)  # noqa: E731
    w = torch.where(t == 0, 1.0, snr(torch.clamp(t - 1, min=0)) - snr(t))
    um, ui = h @ f, x0d @ i_embs.double()
    sim = 1 - torch.nn.functional.cosine_similarity(um, ui, dim=-1)
    reg = (i_embs.double() ** 2).sum() * cfg.train.reg
    return w * mse + sim * cfg.hyper.sim_weight + reg * cfg.train.reg, P


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("denoise_dim", DIMS)
def test_deep_fused_training_step(denoise_dim, precision, monkeypatch):
    """Ragged sizes (B = 300, I = 1003): the fused step (selected: counted through train_step.denoise_loss) vs the
    per-op path (DIFFMM_FUSED_TRAIN=0) and vs float64 autograd, loss and the gradient of every Denoise parameter."""
    from diffmm_b200 import train_step
    B, I = 300, 1003
    cfg, gd, den = _model(denoise_dim, I, precision, seed=5, noise_scale=0.5)
    x0, feat, i_embs, t, noise = _train_inputs(B, I)
    calls = []
    orig = train_step.denoise_loss
    monkeypatch.setattr(train_step, "denoise_loss", lambda *a, **k: (calls.append(1), orig(*a, **k))[1])
    out = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("DIFFMM_FUSED_TRAIN", mode)
        den.zero_grad(set_to_none=True)
        n_calls = len(calls)
        losses = gd.training_losses(den, x0, i_embs, feat, timesteps=t, noise=noise)
        assert len(calls) == n_calls + (1 if mode == "1" else 0), "the fused step was not selected"
        losses.mean().backward()
        out[mode] = (losses.detach().clone(), {k: v.detach().clone() for k, v in _all_grads(den).items()})
    assert len(out["1"][1]) == 4 + 4 * len(den.in_layers)
    tol_l, tol_g = (1e-4, 2e-3) if precision == "bf16x3" else (3e-2, 1.5e-1)
    assert _rel(out["1"][0], out["0"][0]) <= tol_l
    for k in out["1"][1]:
        assert _rel(out["1"][1][k], out["0"][1][k]) <= tol_g, k
    want, P = _training_losses64(cfg, gd, den, x0, i_embs, feat, t, noise)
    want.mean().backward()
    tol_l, tol_g = (2e-4, 1e-3) if precision == "bf16x3" else (1e-1, 1e-1)
    assert _rel(out["1"][0], want.detach()) <= tol_l
    for k, p in P.items():
        assert _rel(out["1"][1][k], p.grad) <= tol_g, (k, _rel(out["1"][1][k], p.grad))


# every extra entry of denoise_dim adds two hidden-to-hidden layers; per layer the fused step issues, with the packed
# weights rebuilt (first step after an update): forward 1 contraction + 1 two-orientation pack, backward 2 contractions
# (dh, dW) + dmm_hidden_bwd + dmm_colsum (db)
LAUNCHES_PER_EXTRA_ENTRY = 2 * (1 + 1 + 2 + 1 + 1)


def test_deep_fused_step_adds_only_library_launches():
    from collections import Counter

    from torch.profiler import ProfilerActivity, profile

    from diffmm_b200 import autograd as ag
    B, I = 256, 1003
    x0, feat, i_embs, t, noise = _train_inputs(B, I, seed=2)

    def kernels(denoise_dim):
        _, gd, den = _model(denoise_dim, I, "bf16", seed=3)

        def step():
            ag._PACK_CACHE.clear()
            den.zero_grad(set_to_none=True)
            gd.training_losses(den, x0, i_embs, feat, timesteps=t, noise=noise).mean().backward()
        step()                                   # warm-up (feature operand copies, tables)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        c = Counter()
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in ev.name.lower() \
                    and "memset" not in ev.name.lower():
                c[ev.name] += 1
        return c

    c = [kernels(dd) for dd in ("[128]", "[128, 96]", "[128, 96, 160]")]
    for lo, hi in zip(c[:-1], c[1:]):
        assert not (lo - hi), lo - hi                       # nothing disappears
        extra = hi - lo
        assert sum(extra.values()) == LAUNCHES_PER_EXTRA_ENTRY, extra
        foreign = [n for n in extra if "at::" in n or "cublas" in n.lower() or "cutlass" in n.lower() or "nvjet" in n]
        assert not foreign, foreign


# ---------------------------------------------------------------------------------------------- 5. epoch
def _coach(tmp_path, monkeypatch, cuda_graph, epochs):
    from diffmm_b200 import Main, synth
    from diffmm_b200.Conf import Config
    U, I = 700, 300
    synth.write_dataset(str(tmp_path), "tiktok", synth.interactions(U, I, seed=3, mean_deg=6.0, heavy_frac=0.02),
                        synth.features(I, dict(image=16, text=24, audio=8), seed=3))
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("DIFFMM_CPU_RNG", "0")
    cfg = Config()
    cfg.data.name = "tiktok"
    cfg.base.denoise_dim, cfg.base.cuda_graph, cfg.base.precision = "[96, 64]", cuda_graph, "bf16"
    cfg.train.batch, cfg.train.test_batch, cfg.train.epoch = 128, 128, epochs
    Main.seed_it(7)
    handler = Main.DataHandler(cfg)
    handler.LoadData()
    return Main.Coach(handler, cfg), handler, cfg, U, I


def _check_packs(dens):
    from diffmm_b200 import autograd as ag, ops
    for den in dens:
        for m in _layers(den):
            ent = ag._PACK_CACHE.get(id(m.weight))
            if ent is None or ent[0]() is not m.weight:
                continue
            for tr, (hi, _) in ent[2].items():
                assert torch.equal(hi, ops.pack_bf16(m.weight.detach(), transpose=tr, split=False)[0]), tr


def test_deep_epoch_in_graph_mode_keeps_every_layer_fresh(tmp_path, monkeypatch):
    from diffmm_b200 import autograd as ag, ops, rebuild
    coach, handler, cfg, U, I = _coach(tmp_path, monkeypatch, True, 3)
    assert len(handler.diffusionLoader) == 6 and U % 128 != 0
    coach.run()
    assert coach._use_graph() and coach._diff_graph is not None and coach._joint_graph is not None
    assert all(np.isfinite(list(h["train"].values())).all() for h in coach.history)
    dens = list(coach._denoise_dict().values())
    assert all(len(d.in_layers) == 2 for d in dens)
    _check_packs(dens)                                      # whatever the run left cached is current
    ag._PACK_CACHE.clear()
    for den in dens:
        den._dmm_hidden_ops = None
    fresh = rebuild.rebuild_modal_adj(coach.diffusion_model, coach._denoise_dict(), handler.train_indptr,
                                      handler.train_indices, U, I, cfg.hyper.sampling_step, "bf16")
    for name, adj in (("image", coach.image_adj), ("text", coach.text_adj), ("audio", coach.audio_adj)):
        assert torch.equal(adj.ptr, fresh[name].ptr) and torch.equal(adj.idx, fresh[name].idx), name
        assert torch.equal(adj.val, fresh[name].val), name
        x = torch.randn((U + I, 64), device=adj.val.device)
        assert torch.equal(ops.spmm(adj, x), ops.spmm(fresh[name], x)), name
    # every layer's packs (both orientations) vs fresh packs of the current weights
    for den in dens:
        for m in _layers(den):
            for tr in (False, True):
                hi, _ = ag.packed_weight(m.weight, tr, False)
                assert torch.equal(hi, ops.pack_bf16(m.weight.detach(), transpose=tr, split=False)[0])


def test_deep_eager_epoch_takes_the_fused_step(tmp_path, monkeypatch):
    from diffmm_b200 import train_step
    coach, *_ = _coach(tmp_path, monkeypatch, False, 1)
    calls = []
    orig = train_step.denoise_loss
    monkeypatch.setattr(train_step, "denoise_loss", lambda *a, **k: (calls.append(1), orig(*a, **k))[1])
    coach.run()
    assert calls, "the fused step was not selected"
    assert all(np.isfinite(list(h["train"].values())).all() for h in coach.history)


# ---------------------------------------------------------------------------------------------- 6. drop-in
@pytest.mark.parametrize("denoise_dim", DIMS)
def test_dropin_generate_view_on_a_deep_denoise(denoise_dim):
    from diffmm_b200 import rebuild
    U, I = 129, 1000
    _, gd, den = _model(denoise_dim, I, "bf16x3")
    _, _, _, x0 = _csr_rows(U, I, 8)
    for ss in (0, 2):
        torch.manual_seed(11)
        got = gd.generate_view(den, T(x0), ss).clone()
        torch.manual_seed(11)
        with torch.no_grad():
            want = rebuild.denoise_chain(gd, den, x_dense=T(x0), sampling_step=ss)
        assert torch.equal(got, want), ss
