"""Times recommend MMR re-ranking (dmm_mmr_rerank) and similar_items against torch fp32 baselines with the same math, one
JSON object per shape.

    python tools/bench_mmr.py [--out profiles/r05_similar_mmr.json] [--min-s 1.0]

Workload: synthetic seeded embeddings (D = 64, the model's latdim, N(0, 0.1^2)).
  * mmr: every user of the shape gets its pool = score_topn(user, items, C) (C best items, bf16x3 relevance: the pool
    Coach.recommend_diverse builds), re-ranked to n items at lam = 0.5 over the unit item rows; baby (19445 users x 7050
    items) and sports (35598 x 18357) with (C, n) in {(100, 10), (200, 20), (512, 50)}.  Arms: the kernel path
    (recommend._mmr_rerank: one launch), the public call on device input (adds the id range and finiteness checks: one
    synchronisation), and a batched torch fp32 greedy with the same math (the pool's vectors gathered once, then per
    step: obj = lam rel - (1 - lam) m, masked arg-max, one batched product against the picked vectors, m = max(m, sim)).
  * similar: n = 10 and 100 most similar items of every item of baby and sports, and of 16 384 queries in a 500 000-item
    catalog.  Arms: recommend.similar_items and torch fp32 (F.normalize, query rows @ unit.T in row chunks of the same
    1 GB rule, the query's own column set to -inf, torch.topk(sorted=True)).
Reported per shape: ms per call (CUDA events on the launching stream; 256 MiB written before every timed call, so the
L2 holds nothing of the previous one; the arms alternate, each until it has >= min-s of timed calls; the median, and each
arm's min / median / max in ms_spread), the work per call, and agreement with torch (fp32 sums in other orders:
near-ties can swap, and in MMR one swapped pick changes the later ones).  The card's name, power limit and max SM clock
are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

D = 64
LAM = 0.5
MMR_CASES = [(name, U, I, C, n) for name, U, I in (("baby", 19445, 7050), ("sports", 35598, 18357))
             for C, n in ((100, 10), (200, 20), (512, 50))]
SIM_CASES = [("baby", 7050, 7050, n) for n in (10, 100)] + [("sports", 18357, 18357, n) for n in (10, 100)] + \
            [("wide", 500000, 16384, n) for n in (10, 100)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # pragma: no cover
        q = f"nvidia-smi unavailable ({e})"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": q}


def time_arms(arms, flush, min_s):
    """Round robin over the arms (L2 overwritten before every call), each arm leaving the rotation once it has >= min_s
    of timed calls and >= 3 calls.  Returns {arm: [ms, ...]}."""
    for _, f in arms * 2:                 # warm-up of every shape each arm uses
        f()
    torch.cuda.synchronize()
    times = {k: [] for k, _ in arms}
    while True:
        todo = [(k, f) for k, f in arms if len(times[k]) < 3 or sum(times[k]) < min_s * 1e3]
        if not todo:
            return times
        for key, f in todo:
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            torch.cuda.synchronize()
            times[key].append(a.elapsed_time(b))


def spread(times):
    return {k: {"calls": len(v), "min": round(min(v), 4), "median": round(float(np.median(v)), 4), "max": round(max(v), 4)}
            for k, v in times.items()}


def torch_mmr(unit, cand, rel, n, lam):
    """Batched fp32 MMR greedy with the kernel's math (distinct candidates in relevance order: torch's first arg-max is
    the kernel's tie rule)."""
    B, C = cand.shape
    X = unit[cand.long()]                                        # [B, C, D], gathered once
    lr = lam * rel
    mu = 1.0 - lam
    m = torch.full_like(rel, float("-inf"))
    picked = torch.zeros_like(rel, dtype=torch.bool)
    out = []
    for s in range(n):
        obj = lr if s == 0 else lr - mu * m
        p = obj.masked_fill(picked, float("-inf")).argmax(1, keepdim=True)
        picked.scatter_(1, p, True)
        out.append(p)
        if s + 1 < n:
            x = X.gather(1, p.unsqueeze(2).expand(B, 1, X.shape[2]))
            m = torch.maximum(m, torch.bmm(X, x.transpose(1, 2)).squeeze(2))
    idx = torch.cat(out, 1)
    return cand.gather(1, idx), rel.gather(1, idx)


def torch_similar(v, q, n, chunk):
    unit = F.normalize(v)
    items, vals = [], []
    for s in range(0, q.shape[0], chunk):
        qs = q[s:s + chunk]
        sc = unit[qs] @ unit.T
        sc[torch.arange(qs.shape[0], device=v.device), qs] = float("-inf")
        top = torch.topk(sc, n, dim=1, sorted=True)
        items.append(top.indices)
        vals.append(top.values)
    return torch.cat(items), torch.cat(vals)


def overlap(a, b):
    return float((torch.sort(a, 1).values.unsqueeze(2) == torch.sort(b, 1).values.unsqueeze(1)).any(2).float().mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_similar_mmr.json"))
    ap.add_argument("--min-s", type=float, default=1.0)
    args = ap.parse_args()
    from diffmm_b200 import ops, recommend
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"card": card(), "D": D, "lam": LAM, "mmr": {}, "similar": {}}
    gen = torch.Generator(device=dev)

    for name, U, I, C, n in MMR_CASES:
        key = f"{name}_{U}x{I}_C{C}_n{n}"
        gen.manual_seed(0)
        u = torch.randn((U, D), generator=gen, device=dev) * 0.1
        it = torch.randn((I, D), generator=gen, device=dev) * 0.1
        cand, rel = recommend.score_topn(u, it, C)
        cand = cand.int()
        unit, _ = ops.rownorm_fwd(it)

        def ours():
            return recommend._mmr_rerank(unit, cand, rel, n, LAM)

        def public():
            return recommend.mmr_rerank(unit, cand, rel, n, LAM)

        def torch_ref():
            return torch_mmr(unit, cand, rel, n, LAM)

        times = time_arms([("ours", ours), ("public", public), ("torch", torch_ref)], flush, args.min_s)
        ms = {k: float(np.median(v)) for k, v in times.items()}
        gi, _ = ours()
        ti, _ = torch_ref()
        entry = {"users": U, "items": I, "C": C, "n": n, "multiply_adds": U * (n - 1) * C * D,
                 "gathered_bytes": U * C * D * 4, "ms": ms["ours"], "public_call_ms": ms["public"],
                 "torch_fp32_ms": ms["torch"], "speedup_vs_torch": ms["torch"] / ms["ours"],
                 "list_overlap_with_torch_fp32": overlap(gi, ti),
                 "rows_in_same_order_as_torch_fp32": float((gi == ti).all(1).float().mean()),
                 "ms_spread": spread(times)}
        result["mmr"][key] = entry
        print(key, json.dumps(entry), flush=True)
        del u, it, cand, rel, unit
        torch.cuda.empty_cache()

    for name, I, Q, n in SIM_CASES:
        key = f"{name}_{I}items_{Q}queries_n{n}"
        gen.manual_seed(1)
        v = torch.randn((I, D), generator=gen, device=dev) * 0.1
        q = torch.arange(I, device=dev) if Q == I else torch.randint(0, I, (Q,), generator=gen, device=dev)
        chunk = recommend.user_chunk(I)

        def ours():
            return recommend.similar_items(v, q, n)

        def torch_ref():
            return torch_similar(v, q, n, chunk)

        times = time_arms([("ours", ours), ("torch", torch_ref)], flush, args.min_s)
        ms = {k: float(np.median(v_)) for k, v_ in times.items()}
        gi, _ = ours()
        ti, _ = torch_ref()
        entry = {"items": I, "queries": Q, "n": n, "multiply_adds": Q * I * D, "ms": ms["ours"],
                 "torch_fp32_ms": ms["torch"], "speedup_vs_torch": ms["torch"] / ms["ours"],
                 "list_overlap_with_torch_fp32": overlap(gi, ti),
                 "rows_in_same_order_as_torch_fp32": float((gi == ti).all(1).float().mean()),
                 "ms_spread": spread(times)}
        result["similar"][key] = entry
        print(key, json.dumps(entry), flush=True)
        del v, q
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
        f.write("\n")
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
