"""Deeper Denoise networks (denoise_dim with more than one entry) at the baby shape: rebuild step, per-contraction times
and the diffusion-training batch, one JSON object per configuration.

    python tools/bench_deep_denoise.py [--out profiles/r03_deep_denoise_baby.json] [--dims "[1024]" "[1000, 200]" ...]

Workload: bench.py's baby workload (19445 users x 7050 items, 2 modalities, 5 reverse steps from sampling_step 5,
synthetic interactions and the weights drawn the way bench.build_workload draws them) with the Denoise of each
denoise_dim.  For "[1024]" the step is bench.py's step (same weights, same call), which makes that row the check of the
one-layer path.  Reported per configuration:
  * rebuild ms/step and users/s: CUDA events on the launching stream, 256 MiB written between timed steps (the L2 holds
    nothing of the previous step), as many steps as fill >= 1 s; packed weights and P, q are rebuilt inside every step;
  * every contraction of one step (DIFFMM_STREAMS=1, events around each launch, same flush), grouped by shape, with the
    FLOPs from the shapes (3 passes in bf16x3) -- per user, modality and intermediate reverse step the hidden-space chain
    costs 2 (sum_inner w_k w_{k+1} + d_L^2) FLOPs;
  * diffusion training, forward + backward of training_losses for both modalities on a 1024-row batch, fused vs per-op
    (DIFFMM_FUSED_TRAIN=0), packs rebuilt every batch as after an optimiser step, >= 1 s windows;
  * the card's name and power limit, read in the same run."""
import argparse
import ast
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # pragma: no cover
        q = f"nvidia-smi unavailable ({e})"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": q}


def build(dims, dev, precision, seed=0):
    """bench.build_workload('baby') with the Denoise of `dims` (the same draws in the same order)."""
    from diffmm_b200 import synth
    from diffmm_b200.Conf import Config
    from diffmm_b200.Model import Denoise, GaussianDiffusion
    w = bench.WORKLOADS["baby"]
    hyper = bench.workload_hyper("baby")
    cfg = Config()
    cfg.base.precision, cfg.base.denoise_dim = precision, dims
    cfg.hyper.steps, cfg.hyper.sampling_step = hyper["steps"], hyper["sampling_step"]
    cfg.hyper.noise_scale, cfg.hyper.noise_min, cfg.hyper.noise_max = hyper["noise"]
    cfg.data.user_num, cfg.data.item_num = w["users"], w["items"]
    inter = synth.interactions(w["users"], w["items"], seed=seed)
    torch.manual_seed(seed)
    diff = GaussianDiffusion(cfg).to(dev)
    out_dims = ast.literal_eval(dims) + [w["items"]]
    dens = {m: Denoise(out_dims[::-1], out_dims, cfg).to(dev) for m in w["modalities"]}
    return cfg, inter, diff, dens


def timed(fn, flush, min_s=1.0, warm=3):
    """(ms per call, calls): events on the launching stream, the flush written (untimed) before every call."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    n = max(10, int(np.ceil(min_s / max(time.perf_counter() - t0, 1e-4))))
    while True:
        ev = []
        for _ in range(n):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            ev.append((a, b))
        torch.cuda.synchronize()
        total = sum(a.elapsed_time(b) for a, b in ev)
        if total >= min_s * 1e3:
            return total / n, n, total
        n = int(np.ceil(n * 1.1 * min_s * 1e3 / total))     # the host-timed estimate undercounted: time a longer window


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dims", nargs="+", default=["[1024]", "[1000, 200]", "[512, 1024]"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "bf16x3"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_deep_denoise_baby.json"))
    args = ap.parse_args()
    from diffmm_b200 import autograd as ag, ops, rebuild, train_step
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"card": card(), "precision": args.precision, "configs": {}}
    for dims in args.dims:
        cfg, inter, diff, dens = build(dims, dev, args.precision)
        U, I = cfg.data.user_num, cfg.data.item_num
        SS = cfg.hyper.sampling_step
        ip, ix = torch.from_numpy(inter.indptr).to(dev), torch.from_numpy(inter.indices).to(dev)

        def step():
            ag._PACK_CACHE.clear()
            for dn in dens.values():
                dn._dmm_hidden_ops = None
            res = {}
            rebuild.rebuild_edges(diff, dens, ip, ix, U, I, SS, args.precision,
                                  per_modality=lambda v: ops.build_norm_adj(ip, v, U, I), per_modality_out=res)
            return res

        ms, n, total = timed(step, flush)
        entry = {"rebuild_ms_per_step": ms, "users_per_s": U / (ms * 1e-3), "timed_steps": n, "timed_ms": total}

        # every contraction of one step, on the caller's stream
        den0 = next(iter(dens.values()))
        widths = rebuild.hidden_widths(den0)
        dL = widths[0]
        inner = [(m.weight.shape[0], m.weight.shape[1]) for m in rebuild._layers(den0)[1]]
        entry["hidden_widths"] = list(widths)
        entry["flop_per_user_modality_intermediate_step"] = 2 * (sum(a * b for a, b in inner) + dL * dL)
        orig = ops.gemm_bf16_tn
        calls = []

        def gemm(a_hi, a_lo, b_hi, b_lo, M, N, K, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            orig(a_hi, a_lo, b_hi, b_lo, M, N, K, **kw)
            e1.record()
            calls.append((M, N, K, 1 + (a_lo is not None) + (b_lo is not None), e0, e1))
        os.environ["DIFFMM_STREAMS"] = "1"
        ops.gemm_bf16_tn = gemm
        try:
            step()
            torch.cuda.synchronize()
            calls.clear()
            flush.fill_(1)
            step()
            torch.cuda.synchronize()
        finally:
            ops.gemm_bf16_tn = orig
            del os.environ["DIFFMM_STREAMS"]
        by = {}
        for M, N, K, passes, e0, e1 in calls:
            k = f"{M}x{N}x{K}"
            b = by.setdefault(k, {"launches": 0, "ms": 0.0, "flop": 0.0})
            b["launches"] += 1
            b["ms"] += e0.elapsed_time(e1)
            b["flop"] += 2.0 * M * N * K * passes
        for b in by.values():
            b["tflop_per_s"] = b["flop"] / (b["ms"] * 1e-3) / 1e12
        entry["contractions_by_shape_MxNxK"] = by
        entry["contraction_ms_per_step"] = sum(b["ms"] for b in by.values())

        # diffusion training: forward + backward for every modality on one batch
        B = cfg.train.batch
        rng = np.random.default_rng(0)
        rows = rng.choice(U, B, replace=False)
        x0 = torch.zeros((B, I), device=dev)
        for r, u in enumerate(rows):
            x0[r, inter.indices[inter.indptr[u]:inter.indptr[u + 1]]] = 1.0
        feat = torch.randn((I, 64), device=dev) * 0.1
        i_embs = torch.randn((I, 64), device=dev) * 0.1
        t = torch.randint(0, cfg.hyper.steps, (B,), device=dev)
        noise = torch.randn((B, I), device=dev)

        def train():
            ag._PACK_CACHE.clear()
            for dn in dens.values():
                dn.zero_grad(set_to_none=True)
                diff.training_losses(dn, x0, i_embs, feat, timesteps=t, noise=noise).mean().backward()
        for mode in ("1", "0"):
            os.environ["DIFFMM_FUSED_TRAIN"] = mode
            ms_t, n_t, _ = timed(train, flush)
            entry["train_ms_per_batch_" + ("fused" if mode == "1" else "per_op")] = ms_t
            entry["train_batches_timed_" + ("fused" if mode == "1" else "per_op")] = n_t
        del os.environ["DIFFMM_FUSED_TRAIN"]
        train_step.clear_caches()
        result["configs"][dims] = entry
        print(dims, json.dumps(entry), flush=True)
        del dens, diff
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
