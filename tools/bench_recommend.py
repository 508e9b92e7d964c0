"""Times recommend.score_topn (every user's n best unseen items, in rank order) against a torch baseline, one JSON object
per shape.

    python tools/bench_recommend.py [--out profiles/r03_recommend.json] [--min-s 1.0]

Workload: synthetic seeded embeddings (D = 64, the model's latdim) and a train CSR with the shape's degree profile
(synth.interactions: log-normal degrees, 1 % heavy tail), every user excluded from its train items.  Shapes: baby
(19445 x 7050) and sports (35598 x 18357) with n in {20, 100, 1000}, and a wide case, 16384 users x 500 000 items with
n = 100.  Reported per shape:
  * ms per full pass over all users and users/s: CUDA events on the launching stream, 256 MiB written between timed passes
    (the L2 holds nothing of the previous pass), passes of the new path and the baseline alternating, >= min-s each;
  * each stage's time in one extra pass (events around every launch): item pack, user pack + contraction with chunk
    maxima, mask + maxima refresh, pruned top-k, rank;
  * the same pipeline forced onto the pruned top-k and forced onto the whole-row top-k (score_topn picks one of the two by
    recommend.PRUNE_RATIO), in the same rotation: the measurement behind that choice;
  * the torch baseline: fp32 torch.mm, -inf index_put_ of the train items, torch.topk(sorted=True), per user block of
    the same size, and the overlap of its lists with ours (bf16x3 scores vs fp32 scores: near-ties can swap);
  * the card's name, power limit and max SM clock, read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SHAPES = [("baby", 19445, 7050, 20), ("baby", 19445, 7050, 100), ("baby", 19445, 7050, 1000),
          ("sports", 35598, 18357, 20), ("sports", 35598, 18357, 100), ("sports", 35598, 18357, 1000),
          ("wide", 16384, 500000, 100)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # pragma: no cover
        q = f"nvidia-smi unavailable ({e})"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": q}


def torch_topn(u, it, n, ptr_host, idx_dev, deg_dev, neg_inf, chunk):
    """The baseline: fp32 torch.mm, -inf at the train items, torch.topk(sorted=True), block by block (the block's entry
    range comes from the host indptr: no host synchronisation inside the loop)."""
    B = u.shape[0]
    out = torch.empty((B, n), dtype=torch.int64, device=u.device)
    for s in range(0, B, chunk):
        b = min(chunk, B - s)
        sc = torch.mm(u[s:s + b], it.t())
        e0, e1 = int(ptr_host[s]), int(ptr_host[s + b])
        rows = torch.repeat_interleave(torch.arange(b, device=u.device), deg_dev[s:s + b], output_size=e1 - e0)
        sc.index_put_((rows, idx_dev[e0:e1].long()), neg_inf)
        out[s:s + b] = torch.topk(sc, n, dim=1, sorted=True).indices
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_recommend.json"))
    ap.add_argument("--min-s", type=float, default=1.0)
    ap.add_argument("--shapes", nargs="*", default=None, help="subset, e.g. baby:20 wide:100")
    args = ap.parse_args()
    from diffmm_b200 import ops, recommend, synth
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"card": card(), "precision": "bf16x3", "D": 64, "shapes": {}}
    for name, U, I, n in SHAPES:
        if args.shapes and f"{name}:{n}" not in args.shapes:
            continue
        inter = synth.interactions(U, I, seed=0)
        rng = np.random.default_rng(1)
        u = torch.from_numpy((rng.standard_normal((U, 64)) * 0.1).astype(np.float32)).to(dev)
        it = torch.from_numpy((rng.standard_normal((I, 64)) * 0.1).astype(np.float32)).to(dev)
        ptr, idx = torch.from_numpy(inter.indptr).to(dev), torch.from_numpy(inter.indices).to(dev)
        deg = ptr[1:] - ptr[:-1]
        rows = np.arange(U)
        chunk = recommend.user_chunk(I)

        def ours():
            return recommend.score_topn(u, it, n, exclude=(ptr, idx, rows))

        neg_inf = torch.tensor(float("-inf"), device=dev)

        def base():
            return torch_topn(u, it, n, inter.indptr, idx, deg, neg_inf, chunk)

        def forced(ratio):
            # score_topn with its top-k choice fixed: ratio 0 always prunes, a huge ratio never does
            def f():
                saved = recommend.PRUNE_RATIO
                recommend.PRUNE_RATIO = ratio
                try:
                    return ours()
                finally:
                    recommend.PRUNE_RATIO = saved
            return f
        pruned, whole_row = forced(0), forced(1 << 40)
        arms = (("ours", ours), ("torch", base), ("pruned_topk", pruned), ("whole_row_topk", whole_row))

        for f in [f for _, f in arms] * 2:    # warm-up of every shape each path uses
            f()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ours()
        torch.cuda.synchronize()
        reps = max(3, int(np.ceil(args.min_s / max(time.perf_counter() - t0, 1e-4))))
        times = {k: [] for k, _ in arms}
        for _ in range(reps):
            for key, f in arms:
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                f()
                b.record()
                torch.cuda.synchronize()
                times[key].append(a.elapsed_time(b))
        ms = {k: float(np.median(v)) for k, v in times.items()}
        got_items = ours()[0]
        want_items = base()
        overlap = float(np.mean([len(np.intersect1d(g, w)) / n for g, w in
                                 zip(got_items.cpu().numpy(), want_items.cpu().numpy())]))

        # stages of one pass: events around every launch of the pipeline
        stages = {}
        wrapped = {}
        for nm in ("pack_bf16", "gemm_bf16_tn", "eval_mask_scores_cmax", "eval_mask_scores", "topk_edges_pruned", "topk_edges",
                   "topn_rank"):
            orig = getattr(ops, nm)
            wrapped[nm] = orig

            def timed(*a, _o=orig, _n=nm, **k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = _o(*a, **k)
                e1.record()
                stages.setdefault(_n, []).append((e0, e1))
                return r
            setattr(ops, nm, timed)
        try:
            flush.fill_(1)
            ours()
            torch.cuda.synchronize()
        finally:
            for nm, orig in wrapped.items():
                setattr(ops, nm, orig)
        stage_ms = {k: sum(a.elapsed_time(b) for a, b in v) for k, v in stages.items()}
        entry = {"users": U, "items": I, "n": n, "pruned": recommend.PRUNE_RATIO * n <= (I + 31) // 32,
                 "train_entries": int(inter.indptr[-1]), "user_block": chunk,
                 "passes_timed_each": reps, "ms_per_pass": ms["ours"], "users_per_s": U / (ms["ours"] * 1e-3),
                 "torch_ms_per_pass": ms["torch"], "torch_users_per_s": U / (ms["torch"] * 1e-3),
                 "speedup_vs_torch": ms["torch"] / ms["ours"], "pruned_topk_ms_per_pass": ms["pruned_topk"],
                 "whole_row_topk_ms_per_pass": ms["whole_row_topk"], "chunks_per_listed_item": ((I + 31) // 32) / n,
                 "stage_ms_one_pass": stage_ms,
                 "overlap_with_torch_fp32_lists": overlap,
                 "ms_all_passes": {k: [round(x, 4) for x in v] for k, v in times.items()}}
        key = f"{name}_{U}x{I}_n{n}"
        result["shapes"][key] = entry
        print(key, json.dumps({k: v for k, v in entry.items() if k != "ms_all_passes"}), flush=True)
        del u, it, ptr, idx
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
