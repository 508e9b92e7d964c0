"""Times recommend.rank_candidates (each user's caller-supplied candidate row, scored and ranked in one launch) and
recommend.score_pairs (scores of given pairs) against torch fp32 baselines, one JSON object per shape.

    python tools/bench_candidates.py [--out profiles/r04_candidates.json] [--min-s 1.0]

Workload: synthetic seeded embeddings (D = 64, the model's latdim, N(0, 0.1^2)).
  * rank: every user of the shape gets one row of C distinct uniform candidates; baby (19445 x 7050) and sports
    (35598 x 18357) with C in {101, 1001} and n in {10, 100}, and 16384 users x 500 000 items with C = 1000, n = 100.
    Arms: the kernel path (recommend._rank_candidates: one dmm_rank_candidates launch), the public call on device
    candidates (adds the id range check: two reductions and one synchronisation), the torch fp32 baseline (gather of
    the candidates' item rows, einsum, torch.topk(sorted=True), gather of the ids), and for context score_topn over the
    full catalog with the same n (no exclusion).
  * pairs: 10 M uniform random (user, item) pairs at baby and at 16384 x 500 000.  Arms: the kernel path
    (ops.score_pairs), the public call on device ids, and the torch fp32 baseline (two row gathers, einsum).
Reported per shape: ms per call (CUDA events on the launching stream; 256 MiB written before every timed call, so the
L2 holds nothing of the previous one; the arms alternate, each until it has >= min-s of timed calls; the median, and
each arm's min / median / max in ms_spread), the
algorithmic bytes moved (gathered rows, ids, outputs) per second, and agreement with the baseline (bf16x3 vs fp32
scores: near-ties can swap).  The card's name, power limit and max SM clock are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

D = 64
RANK_CASES = [("baby", 19445, 7050, C, n) for C in (101, 1001) for n in (10, 100)] + \
             [("sports", 35598, 18357, C, n) for C in (101, 1001) for n in (10, 100)] + \
             [("wide", 16384, 500000, 1000, 100)]
PAIR_CASES = [("baby", 19445, 7050, 10_000_000), ("wide", 16384, 500000, 10_000_000)]


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
    """Per arm: calls timed and the min / median / max ms of a call."""
    return {k: {"calls": len(v), "min": round(min(v), 4), "median": round(float(np.median(v)), 4), "max": round(max(v), 4)}
            for k, v in times.items()}


def distinct_candidates(B, I, C, gen, dev):
    """C distinct uniform items per row (top-C of uniform keys), in blocks of <= 2^28 keys."""
    out = torch.empty((B, C), dtype=torch.int32, device=dev)
    rows = max(1, (1 << 28) // I)
    for s in range(0, B, rows):
        b = min(rows, B - s)
        out[s:s + b] = torch.rand((b, I), generator=gen, device=dev).topk(C, dim=1).indices.int()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_candidates.json"))
    ap.add_argument("--min-s", type=float, default=1.0)
    ap.add_argument("--cases", nargs="*", default=None, help="subset, e.g. rank:baby:101:10 pairs:wide")
    args = ap.parse_args()
    from diffmm_b200 import ops, recommend
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"card": card(), "precision": "bf16x3", "D": D, "rank": {}, "pairs": {}}
    gen = torch.Generator(device=dev)

    def embs(U, I, seed):
        gen.manual_seed(seed)
        u = torch.randn((U, D), generator=gen, device=dev) * 0.1
        it = torch.randn((I, D), generator=gen, device=dev) * 0.1
        return u, it

    for name, U, I, C, n in RANK_CASES:
        key = f"{name}_{U}x{I}_C{C}_n{n}"
        if args.cases and f"rank:{name}:{C}:{n}" not in args.cases:
            continue
        u, it = embs(U, I, 0)
        gen.manual_seed(1)
        cand = distinct_candidates(U, I, C, gen, dev)

        def ours():
            return recommend._rank_candidates(u, it, cand, n, "bf16x3")

        def public():
            return recommend.rank_candidates(u, it, cand, n)

        def torch_ref():
            s = torch.einsum("bd,bcd->bc", u, it[cand.long()])
            top = torch.topk(s, n, dim=1, sorted=True)
            return cand.gather(1, top.indices), top.values

        def full_catalog():
            return recommend.score_topn(u, it, n)

        times = time_arms([("ours", ours), ("public", public), ("torch", torch_ref), ("score_topn_full", full_catalog)],
                          flush, args.min_s)
        ms = {k: float(np.median(v)) for k, v in times.items()}
        gi, _ = ours()
        ti, _ = torch_ref()
        overlap = float((torch.sort(gi, 1).values.unsqueeze(2) == torch.sort(ti, 1).values.unsqueeze(1))
                        .any(2).float().mean())
        same_order = float((gi == ti).all(1).float().mean())
        nbytes = U * C * D * 4 + U * D * 4 + U * C * 4 + U * n * 8
        entry = {"users": U, "items": I, "C": C, "n": n, "algorithmic_bytes": nbytes,
                 "ms": ms["ours"], "GB_per_s": nbytes / (ms["ours"] * 1e-3) / 1e9,
                 "public_call_ms": ms["public"],
                 "torch_fp32_ms": ms["torch"], "torch_GB_per_s": nbytes / (ms["torch"] * 1e-3) / 1e9,
                 "speedup_vs_torch": ms["torch"] / ms["ours"],
                 "score_topn_full_catalog_ms": ms["score_topn_full"],
                 "list_overlap_with_torch_fp32": overlap, "rows_in_same_order_as_torch_fp32": same_order,
                 "ms_spread": spread(times)}
        result["rank"][key] = entry
        print(key, json.dumps(entry), flush=True)
        del u, it, cand
        torch.cuda.empty_cache()

    for name, U, I, P in PAIR_CASES:
        key = f"{name}_{U}x{I}_P{P}"
        if args.cases and f"pairs:{name}" not in args.cases:
            continue
        u, it = embs(U, I, 2)
        gen.manual_seed(3)
        pu = torch.randint(0, U, (P,), generator=gen, device=dev)
        pi = torch.randint(0, I, (P,), generator=gen, device=dev).int()
        out = torch.empty(P, device=dev)

        def ours():
            return ops.score_pairs(u, it, pu, pi, True, out)

        def public():
            return recommend.score_pairs(u, it, pu, pi)

        def torch_ref():
            return torch.einsum("pd,pd->p", u[pu], it[pi.long()])

        times = time_arms([("ours", ours), ("public", public), ("torch", torch_ref)], flush, args.min_s)
        ms = {k: float(np.median(v)) for k, v in times.items()}
        got, ref = ours().double(), torch_ref().double()
        mag = (u[pu].double().abs() * it[pi.long()].double().abs()).sum(1)
        nbytes = P * (2 * D * 4 + 8 + 4 + 4)
        entry = {"users": U, "items": I, "pairs": P, "algorithmic_bytes": nbytes,
                 "ms": ms["ours"], "GB_per_s": nbytes / (ms["ours"] * 1e-3) / 1e9, "public_call_ms": ms["public"],
                 "torch_fp32_ms": ms["torch"], "torch_GB_per_s": nbytes / (ms["torch"] * 1e-3) / 1e9,
                 "speedup_vs_torch": ms["torch"] / ms["ours"],
                 "max_abs_diff_vs_torch_fp32_over_sum_abs_terms": float(((got - ref).abs() / mag).max()),
                 "ms_spread": spread(times)}
        result["pairs"][key] = entry
        print(key, json.dumps(entry), flush=True)
        del u, it, pu, pi, out
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
