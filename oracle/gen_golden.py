"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by executing the UNMODIFIED
reference (/root/reference) on CPU through oracle/ref_shim.py.

Run in the build container (the reference does not travel to the GPU box):
    python oracle/gen_golden.py
The committed .npz files are the pins for oracle/diffmm_oracle.py and for the CUDA
parity tests.  Every RNG draw the reference makes is replayed and stored so the
kernels can be fed identical noise / timesteps.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import ref_shim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
U, I, H, D = 40, 120, 32, 64
FEAT = dict(image=16, text=24, audio=8)


def np32(t):
    return t.detach().cpu().numpy().astype(np.float32)


def synth_interactions(rng, n_users, n_items, mean_deg=4, heavy=(0, 30)):
    rows, cols = [], []
    for u in range(n_users):
        k = int(np.clip(rng.poisson(mean_deg), 0, n_items))
        if u == heavy[0]:
            k = heavy[1]
        if u == 1:
            k = 0                                  # a user with no interactions (tiktok has 10)
        its = rng.choice(n_items, size=k, replace=False)
        rows += [u] * k
        cols += list(its)
    return np.array(rows, dtype=np.int64), np.array(cols, dtype=np.int64)


def denoise_params(m):
    return dict(
        emb_w=np32(m.emb_layer.weight), emb_b=np32(m.emb_layer.bias),
        w1=np32(m.in_layers[0].weight), b1=np32(m.in_layers[0].bias),
        w2=np32(m.out_layers[0].weight), b2=np32(m.out_layers[0].bias),
        gate_w=np32(m.gate_layer.weight), gate_b=np32(m.gate_layer.bias),
    )


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = ref_shim.load_reference()
    rng = np.random.default_rng(20261018)
    torch.manual_seed(1818)

    # ---------------------------------------------------------------- schedules (a3)
    sched = {}
    for name, (ns, nmin, nmax, steps) in dict(tiktok=(0.5, 1e-4, 0.02, 5), sports=(0.1, 1e-4, 0.02, 5),
                                              wide=(1.0, 1e-3, 0.05, 8)).items():
        cfg = ref_shim.make_config(ref, **{"hyper.noise_scale": ns, "hyper.noise_min": nmin,
                                           "hyper.noise_max": nmax, "hyper.steps": steps})
        gd = ref.Model.GaussianDiffusion(cfg)
        for k in ("betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod",
                  "sqrt_one_minus_alphas_cumprod", "posterior_variance", "posterior_mean_coef1",
                  "posterior_mean_coef2"):
            sched[f"{name}.{k}"] = getattr(gd, k).numpy().astype(np.float64)
        t = torch.arange(steps)
        sched[f"{name}.snr"] = gd.SNR(t).numpy()
        sched[f"{name}.args"] = np.array([ns, nmin, nmax, steps], dtype=np.float64)
    np.savez(os.path.join(OUT, "schedule.npz"), **sched)

    # ---------------------------------------------------------------- the reference's conf/*.toml, parsed (f4)
    import json
    import tomllib
    conf_dir = os.path.join(ref_shim.REFERENCE_ROOT, "conf")
    confs = {}
    for f in sorted(os.listdir(conf_dir)):
        if f.endswith(".toml"):
            with open(os.path.join(conf_dir, f), "rb") as fh:
                confs[f] = tomllib.load(fh)
    with open(os.path.join(OUT, "reference_conf.json"), "w") as fh:
        json.dump(confs, fh, indent=1, sort_keys=True)
        fh.write("\n")

    # ---------------------------------------------------------------- common small problem
    cfg = ref_shim.make_config(ref, "tiktok", **{
        "base.denoise_dim": f"[{H}]", "hyper.noise_scale": 0.5, "hyper.sim_weight": 0.01,
        "train.reg": 1e-4, "hyper.noise_degree": 1.5, "hyper.residual_weight": 0.5,
        "hyper.modal_adj_weight": 0.2})
    cfg.data.user_num, cfg.data.item_num = U, I
    cfg.data.image_feat_dim, cfg.data.text_feat_dim, cfg.data.audio_feat_dim = FEAT["image"], FEAT["text"], FEAT["audio"]
    ref.Main.config = cfg
    rows, cols = synth_interactions(rng, U, I)
    x_dense = np.zeros((U, I), dtype=np.float32)
    x_dense[rows, cols] = 1.0
    order = np.lexsort((cols, rows))
    rows, cols = rows[order], cols[order]
    indptr = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows, minlength=U), out=indptr[1:])

    gd = ref.Model.GaussianDiffusion(cfg)
    den = ref.Model.Denoise([I, H], [H, I], cfg)
    with torch.no_grad():                                # move away from init so every term matters
        for prm in den.parameters():
            prm.add_(0.05 * torch.randn_like(prm))
    P = denoise_params(den)
    x = torch.from_numpy(x_dense)

    # ---------------------------------------------------------------- Denoise.forward (a2)
    B = 24
    xt_in = torch.randn(B, I) * 0.3 + x[:B]
    ts = torch.randint(0, 5, (B,))
    feat = torch.randn(I, D) * 0.2
    with torch.no_grad():
        out_nogate = den(xt_in, ts)
        out_gate = den(xt_in, ts, modal_feat=feat)
    np.savez(os.path.join(OUT, "denoise_forward.npz"), x_t=np32(xt_in), t=ts.numpy(), feat=np32(feat),
             out_nogate=np32(out_nogate), out_gate=np32(out_gate), **{f"p.{k}": v for k, v in P.items()})

    # ---------------------------------------------------------------- q_sample (a4)
    noise = torch.randn(B, I)
    with torch.no_grad():
        xt_explicit = gd.forward_cal_xt(x[:B], ts, noise)
        torch.manual_seed(7)
        g = torch.randn(B, I)                            # replay of the draw made inside :337
        torch.manual_seed(7)
        xt_default = gd.forward_cal_xt(x[:B], ts)
    np.savez(os.path.join(OUT, "q_sample.npz"), x0=x_dense[:B], t=ts.numpy(), noise=np32(noise),
             xt_explicit=np32(xt_explicit), randn=np32(g), xt_default=np32(xt_default))

    # ---------------------------------------------------------------- training_losses (a5) value + grads
    i_embs = torch.nn.Parameter(torch.randn(I, D) * 0.1)
    torch.manual_seed(11)
    t_replay = torch.randint(0, 5, (B,)).long()          # :397
    n_replay = torch.randn(B, I)                         # :400
    torch.manual_seed(11)
    den.zero_grad()
    losses = gd.training_losses(den, x[:B], i_embs, feat)
    losses.mean().backward()
    grads = {f"g.{k}": np32(v) for k, v in dict(
        emb_w=den.emb_layer.weight.grad, emb_b=den.emb_layer.bias.grad,
        w1=den.in_layers[0].weight.grad, b1=den.in_layers[0].bias.grad,
        w2=den.out_layers[0].weight.grad, b2=den.out_layers[0].bias.grad,
        gate_w=den.gate_layer.weight.grad, gate_b=den.gate_layer.bias.grad).items()}
    np.savez(os.path.join(OUT, "training_losses.npz"), x0=x_dense[:B], t=t_replay.numpy(), noise=np32(n_replay),
             i_embs=np32(i_embs), feat=np32(feat), losses=losses.detach().numpy().astype(np.float64),
             reg=np.float64(cfg.train.reg), sim_weight=np.float64(cfg.hyper.sim_weight),
             g_i_embs=np32(i_embs.grad), **grads, **{f"p.{k}": v for k, v in P.items()})

    # ---------------------------------------------------------------- generate_view (a7)
    with torch.no_grad():
        view0 = gd.generate_view(den, x, 0)
        torch.manual_seed(13)
        g2 = torch.randn(U, I)
        torch.manual_seed(13)
        view2 = gd.generate_view(den, x, 2)
    np.savez(os.path.join(OUT, "generate_view.npz"), x0=x_dense, view0=np32(view0), randn=np32(g2),
             view2=np32(view2), indptr=indptr, indices=cols)

    # ---------------------------------------------------------------- rebuild loop (a8) + adjacency (a9)
    deg = np.asarray(x_dense.sum(1), dtype=int)
    u_list, i_list = [], []
    for r in range(U):                                   # Main.py:224-230 verbatim in behaviour
        _, idxs = torch.topk(view0[r], k=int(deg[r]))
        for j in range(idxs.shape[0]):
            u_list.append(r)
            i_list.append(int(idxs[j]))
    from scipy.sparse import coo_matrix
    mat = coo_matrix((np.ones(len(u_list)), (np.array(u_list), np.array(i_list))), shape=(U, I), dtype=np.float32)
    adj = ref.DataHandler.DataHandler.makeTorchAdj(mat, U, I, torch.device("cpu")).coalesce()
    trn = coo_matrix((np.ones(len(rows)), (rows, cols)), shape=(U, I), dtype=np.float32)
    bi = ref.DataHandler.DataHandler.makeTorchAdj(trn, U, I, torch.device("cpu")).coalesce()
    np.savez(os.path.join(OUT, "rebuild.npz"), scores=np32(view0), deg=deg.astype(np.int64),
             edge_u=np.array(u_list, dtype=np.int64), edge_i=np.array(i_list, dtype=np.int64),
             adj_idx=adj.indices().numpy(), adj_val=adj.values().numpy(),
             trn_u=rows, trn_i=cols, bi_idx=bi.indices().numpy(), bi_val=bi.values().numpy())

    # ---------------------------------------------------------------- gcn_MM (a10) value + grads, 3 and 2 modalities
    feats = {m: torch.randn(I, d) for m, d in FEAT.items()}
    # modality graphs: perturb the train graph deterministically
    madj = {}
    for s, m in enumerate(FEAT):
        keep = rng.random(len(rows)) > 0.3
        extra_u = rng.integers(0, U, 25)
        extra_i = rng.integers(0, I, 25)
        mu = np.concatenate([rows[keep], extra_u])
        mi = np.concatenate([cols[keep], extra_i])
        mm = coo_matrix((np.ones(len(mu)), (mu, mi)), shape=(U, I), dtype=np.float32)
        madj[m] = (mu, mi, ref.DataHandler.DataHandler.makeTorchAdj(mm, U, I, torch.device("cpu")))
    for tag, mods in (("3", ["image", "text", "audio"]), ("2", ["image", "text"])):
        torch.manual_seed(5)
        model = ref.Model.Model(cfg, feats["image"], feats["text"], feats["audio"] if tag == "3" else None)
        with torch.no_grad():
            model.modal_weight.add_(torch.tensor([0.2, -0.1, 0.05][:len(mods)]))
        args = [madj[m][2] for m in mods]
        out = model.gcn_MM(bi, *args)
        probe = torch.randn(U + I, D)
        cat = lambda a, b: torch.cat([a, b])  # noqa: E731
        scal = (cat(out.u_final_embs, out.i_final_embs) * probe).sum()
        zs = [cat(out.u_image_embs, out.i_image_embs), cat(out.u_text_embs, out.i_text_embs)]
        if tag == "3":
            zs.append(cat(out.u_audio_embs, out.i_audio_embs))
        for k, z in enumerate(zs):
            scal = scal + (z * probe * (0.5 + k)).sum()
        scal.backward()
        d = dict(u_embs=np32(model.u_embs), i_embs=np32(model.i_embs), modal_weight=np32(model.modal_weight),
                 probe=np32(probe), final=np32(cat(out.u_final_embs, out.i_final_embs)),
                 g_u=np32(model.u_embs.grad), g_i=np32(model.i_embs.grad), g_mw=np32(model.modal_weight.grad),
                 modal_adj_weight=np.float64(cfg.hyper.modal_adj_weight),
                 residual_weight=np.float64(cfg.hyper.residual_weight))
        for k, m in enumerate(mods):
            lin = getattr(model, f"{m}_layer")
            d[f"feat.{m}"] = np32(feats[m])
            d[f"lin_w.{m}"], d[f"lin_b.{m}"] = np32(lin.weight), np32(lin.bias)
            d[f"g_lin_w.{m}"], d[f"g_lin_b.{m}"] = np32(lin.weight.grad), np32(lin.bias.grad)
            d[f"z.{m}"] = np32(zs[k])
            d[f"adj_u.{m}"], d[f"adj_i.{m}"] = madj[m][0], madj[m][1]
        np.savez(os.path.join(OUT, f"gcn_mm_{tag}.npz"), trn_u=rows, trn_i=cols, **d)

    # ---------------------------------------------------------------- InfoNCE / BPR / l2 (a12, a13) value + grads
    Bn = 48
    v1 = torch.nn.Parameter(torch.randn(U, D))
    v2 = torch.nn.Parameter(torch.randn(U, D))
    idx = torch.randint(0, U, (Bn,))                     # repeats on purpose (Bn > U)
    l = ref.Utils.InfoNCE(v1, v2, idx, 0.2)
    l.backward()
    ue = torch.nn.Parameter(torch.randn(Bn, D) * 0.5)
    pe = torch.nn.Parameter(torch.randn(Bn, D) * 0.5)
    ne = torch.nn.Parameter(torch.randn(Bn, D) * 0.5)
    b = ref.Utils.bpr_loss(ue, pe, ne)
    b.backward()
    r = ref.Utils.l2_reg_loss(1e-4, [v1.detach(), v2.detach()], torch.device("cpu"))
    np.savez(os.path.join(OUT, "losses.npz"), v1=np32(v1), v2=np32(v2), idx=idx.numpy(), temp=np.float64(0.2),
             infonce=np32(l), g_v1=np32(v1.grad), g_v2=np32(v2.grad),
             u=np32(ue), p=np32(pe), n=np32(ne), bpr=np32(b), g_u=np32(ue.grad), g_p=np32(pe.grad), g_n=np32(ne.grad),
             l2=np32(r), l2_reg=np.float64(1e-4))

    # ---------------------------------------------------------------- cross-layer CL block (a11), Main.py:315-330
    torch.manual_seed(17)
    rs = [torch.rand(U + I, D) for _ in range(3)]        # replay of the three rand_like draws
    torch.manual_seed(17)
    ue0 = torch.randn(U, D) * 0.1
    ie0 = torch.randn(I, D) * 0.1
    torch.manual_seed(17)
    joint = torch.cat([ue0, ie0], dim=0)
    all_embs = []
    all_cl = joint
    import torch.nn.functional as F
    for k in range(3):
        joint = torch.sparse.mm(bi, joint)
        random_noise = torch.rand_like(joint)
        joint = joint + torch.sign(joint) * F.normalize(random_noise) * cfg.hyper.noise_degree
        all_embs.append(joint)
        if k == 0:
            all_cl = joint
    final = torch.mean(torch.stack(all_embs), dim=0)
    np.savez(os.path.join(OUT, "cl_propagate.npz"), u=np32(ue0), i=np32(ie0), rand=np.stack([np32(r_) for r_ in rs]),
             mean=np32(final), layer1=np32(all_cl), noise_degree=np.float64(cfg.hyper.noise_degree),
             trn_u=rows, trn_i=cols)
    print("golden vectors written to", OUT)
    for f in sorted(os.listdir(OUT)):
        print(f"  {f}: {os.path.getsize(os.path.join(OUT, f)) / 1024:.1f} KiB")


if __name__ == "__main__":
    main()
