#!/usr/bin/env python
"""Benchmark of the DiffMM hot path on B200: denoise/top-k graph rebuild users per second.

    python bench.py --gpus N --steps K --warmup W          # our arm (1 process per GPU under torchrun for N > 1)
    python bench.py --impl reference ...                   # the unmodified reference (oracle/_ref) on the host cores

A "step" is one full pass of phase 2 (reference Main.py:195-253) over the workload's users: for every
modality the S-step reverse-diffusion chain (tcgen05 GEMMs), the per-user top-k (k = deg(u)) and the
normalised-adjacency build.  Workload (N = 1): conf/baby.toml (19445 users x 7050 items, 2 modalities,
hidden 1024, 5 steps, sampling_step 5: the rebuild starts from a q_sample'd x_5), synthetic interactions +
random-init weights of that architecture (same seed in both arms).  For N > 1 every rank owns a shard of the
same size (weak scaling: N x 19445 users); the only data-path collective is the edge all-gather.  One JSON
line is printed by rank 0; besides the contract's keys it carries `variants` (sampling_step 0, bf16x3),
`long_run` (a >= 1 s timed region), `other_workloads` (N > 1: sports strong scaling, 2M x 500k slice),
`propagation` (row-partitioned SpMM + all-gather at the ifashion shape), `aux_rooflines`, `epoch_sec`.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: users, items, modalities, hidden; the hyper-parameters (noise schedule, steps, sampling_step) come from the
    # matching conf/*.toml (workload_hyper)
    "tiktok": dict(users=9308, items=6710, modalities=["image", "text", "audio"], hidden=1024, conf="tiktok.toml"),
    "baby": dict(users=19445, items=7050, modalities=["image", "text"], hidden=1024, conf="baby.toml"),
    "sports": dict(users=35598, items=18357, modalities=["image", "text"], hidden=1024, conf="sports.toml"),
    # BASELINE.json configs[4] (2M users x 500k items, 3 modalities): one GPU's slice of the user rows per step
    "scaleout": dict(users=16384, items=500000, modalities=["image", "text", "audio"], hidden=1024, conf="sports.toml"),
}


def workload_hyper(name, sampling_step=None):
    """Hyper-parameters of the workload from its conf/*.toml (through the repo's tolerant loader): conf/baby.toml gives
    sampling_step 5 (the rebuild starts from a q_sample'd x_5), tiktok / sports 0.  --sampling-step overrides."""
    from diffmm_b200.Conf import load_config
    cfg = load_config(os.path.join(ROOT, "conf", WORKLOADS[name]["conf"]))
    ss = cfg.hyper.sampling_step if sampling_step is None else int(sampling_step)
    return dict(noise=(cfg.hyper.noise_scale, cfg.hyper.noise_min, cfg.hyper.noise_max), steps=int(cfg.hyper.steps),
                sampling_step=int(ss), conf="conf/" + WORKLOADS[name]["conf"])


def config_dict(name, w, hyper, precision):
    """The `config` object of the JSON line: identical for the GPU arm and the reference arm of the same workload."""
    return {"workload": f"{name}-shape rebuild phase (Main.py:195-253) with the hyper-parameters of {hyper['conf']}: "
                        f"{w['users']} users x {w['items']} items per GPU, {len(w['modalities'])} modalities, hidden "
                        f"{w['hidden']}, {hyper['steps']} reverse steps from sampling_step {hyper['sampling_step']}, "
                        f"top-k k=deg(u), adjacency build",
            "users_per_gpu": w["users"], "items": w["items"], "modalities": len(w["modalities"]), "hidden": w["hidden"],
            "diffusion_steps": hyper["steps"], "sampling_step": hyper["sampling_step"], "conf": hyper["conf"]}


METRIC = "denoise_topk_rebuild_users_per_sec"
UNIT = "users/s"
KERNELS_PER_CALL = {   # hand-written kernels launched per C-ABI call (CUB's sort kernels are not counted)
    "dmm_pack_bf16": 1, "dmm_csr_rows_to_dense": 1, "dmm_time_embedding": 1, "dmm_q_sample": 1, "dmm_gemm_bf16_tn": 1,
    "dmm_gemm_f32_tn": 1, "dmm_topk_edges": 1, "dmm_topk_edges_pruned": 2, "dmm_csr_qsample_values": 1,
    "dmm_build_norm_adj_csr": 3, "dmm_sign_noise_": 1,
    "dmm_bpr_fwd_bwd": 2, "dmm_infonce_fwd": 3, "dmm_infonce_bwd": 3, "dmm_scatter_add_rows": 1,
    "dmm_spmm_csr": 2, "dmm_spmm_plan": 6, "dmm_spmm_table_bf16": 1, "dmm_spmm_norm_bf16": 2, "dmm_gemm_bf16_tn_splitk": 2,
}


_RESULT_FD = 1


def emit(line):
    """Writes the result line to the process's original stdout (see main)."""
    sys.stdout.flush()
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------ workload
def build_workload(name, device, seed, precision, world=1, hyper=None, users_total=None, init_on_device=False):
    """Synthetic interactions + random-init Denoise weights of the workload's architecture.  The default workload draws
    its weights on the CPU generator in the reference's construction order (the reference arm draws the same ones);
    init_on_device draws them with the device generator instead (the 500k-item models are 6 GB of normals)."""
    import torch
    from diffmm_b200 import synth
    from diffmm_b200.Conf import Config
    from diffmm_b200.Model import Denoise, GaussianDiffusion
    w = WORKLOADS[name]
    hyper = hyper or workload_hyper(name)
    users_total = w["users"] * world if users_total is None else users_total
    cfg = Config()
    cfg.base.precision = precision
    cfg.base.denoise_dim = f"[{w['hidden']}]"
    cfg.hyper.steps = hyper["steps"]
    cfg.hyper.sampling_step = hyper["sampling_step"]
    cfg.hyper.noise_scale, cfg.hyper.noise_min, cfg.hyper.noise_max = hyper["noise"]
    cfg.data.user_num, cfg.data.item_num = users_total, w["items"]
    inter = synth.interactions(users_total, w["items"], seed=seed)      # same global dataset on every rank
    torch.manual_seed(seed)
    diff = GaussianDiffusion(cfg).to(device)
    if init_on_device and str(device) != "cpu":
        torch.cuda.manual_seed(seed)
        with torch.device(device):
            dens = {m: Denoise([w["items"], w["hidden"]], [w["hidden"], w["items"]], cfg) for m in w["modalities"]}
    else:
        dens = {m: Denoise([w["items"], w["hidden"]], [w["hidden"], w["items"]], cfg).to(device) for m in w["modalities"]}
    return cfg, inter, diff, dens


def oracle_params(den):
    f = lambda t: t.detach().cpu().numpy()  # noqa: E731
    return dict(emb_w=f(den.emb_layer.weight), emb_b=f(den.emb_layer.bias), w1=f(den.in_layers[0].weight),
                b1=f(den.in_layers[0].bias), w2=f(den.out_layers[0].weight), b2=f(den.out_layers[0].bias),
                gate_w=f(den.gate_layer.weight), gate_b=f(den.gate_layer.bias))


def cpu_rebuild_sample(inter, w, params_by_mod, n_sample, hyper, seed=0):
    """The reference's phase 2 restated in numpy (oracle/diffmm_oracle.py) on `n_sample` users; returns seconds.
    Only used when oracle/_ref is absent (the port leg; always sampling_step 0)."""
    from oracle import diffmm_oracle as O
    sched = O.make_schedule(*hyper["noise"], hyper["steps"])
    users = np.arange(min(n_sample, w["users"]))
    ptr, idx = inter.indptr, inter.indices
    t0 = time.perf_counter()
    x = np.zeros((len(users), w["items"]), dtype=np.float32)
    for r, u in enumerate(users):
        x[r, idx[ptr[u]:ptr[u + 1]]] = 1.0
    deg = np.diff(ptr)[users]
    edges = 0
    for m, p in params_by_mod.items():
        for b0 in range(0, len(users), 1024):                       # the reference's batch of 1024 (Main.py:211)
            view = O.generate_view(sched, p, x[b0:b0 + 1024], 0)
            edges += sum(len(e) for e in O.topk_edges(view, deg[b0:b0 + 1024]))
    dt = time.perf_counter() - t0
    return dt, len(users), edges


def epoch_seconds(name, seed, precision, epochs=3, cuda_graph=True):
    """One full training epoch + eval (phases 1-3 of Coach.trainEpoch + testEpoch) on the synthetic
    `name`-shape dataset written in the reference's on-disk format; returns the last epoch's phase seconds."""
    import tempfile
    import torch
    from diffmm_b200 import Main, synth
    from diffmm_b200.Conf import Config
    U, I, dims = synth.SHAPES[name]
    root = tempfile.mkdtemp(prefix="diffmm_bench_")
    synth.write_dataset(root, name, synth.interactions(U, I, seed=seed), synth.features(I, dims, seed=seed))
    cwd = os.getcwd()
    os.chdir(root)
    try:
        cfg = Config()
        cfg.data.name = name
        cfg.base.precision = precision
        cfg.train.epoch = epochs
        cfg.base.cuda_graph = cuda_graph
        cfg.train.test_batch = 1024
        Main.seed_it(seed)
        h = Main.DataHandler(cfg)
        h.LoadData()
        coach = Main.Coach(h, cfg)
        coach.prepareModel()
        out = {}
        for ep in range(epochs):
            coach.phase_seconds = {}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            coach.trainEpoch()
            res = coach.testEpoch()
            torch.cuda.synchronize()
            out = dict(coach.phase_seconds)
            out["epoch_total"] = time.perf_counter() - t0
            out["recall_at_20"] = float(res["Recall"])
        out["steps"] = {"diffusion_batches": len(h.diffusionLoader), "joint_batches": len(h.trainLoader)}
        return out
    finally:
        os.chdir(cwd)
        import shutil
        shutil.rmtree(root, ignore_errors=True)


def aux_rooflines(dev, breakdown, U, I, E, n_mod, pk, seed, precision="bf16"):
    """HBM-bound kernels of the path against the measured copy bandwidth: top-k (from the step breakdown) and the
    CSR SpMM at the ifashion-shaped graph of BASELINE.json configs[3] (300k users x 80k items; the shipped
    shapes are L2 resident, SURVEY.md 8d), each timed with CUDA events on the launching stream."""
    import torch
    from diffmm_b200 import ops, synth
    out = {}
    tk = "dmm_topk_edges_pruned" if "dmm_topk_edges_pruned" in breakdown else "dmm_topk_edges"
    if tk in breakdown:
        ms = breakdown[tk]["ms_per_step"] / max(breakdown[tk]["calls_per_step"], 1)
        by = 4.0 * I * U + 4.0 * E + 8.0 * (U + 1)
        out["topk_edges"] = {"bound": "hbm", "bytes_per_launch": by, "avg_launch_ms": ms, "achieved": by / (ms * 1e-3) / 1e9,
                             "peak": pk["hbm"], "unit": "GB/s", "frac": by / (ms * 1e-3) / 1e9 / pk["hbm"],
                             "entry_point": tk,
                             "shape": f"{U} rows x {I} fp32 scores, k = deg(u)",
                             "note": "against the algorithmic 4*I bytes per row (SURVEY 8d); the pruned kernel reads the chunk "
                                     "maxima the scores contraction wrote (4*I/32 bytes per row) plus k 128-byte chunks, so "
                                     "its DRAM traffic is ~1/20 of that figure and the fraction can exceed 1"}
    Ui, Ii, _ = synth.SHAPES["ifashion"]
    inter = synth.interactions(Ui, Ii, seed=seed)
    ptr = torch.from_numpy(inter.indptr).to(dev)
    idx = torch.from_numpy(inter.indices).to(dev)
    adj = ops.build_norm_adj(ptr, idx, Ui, Ii)
    N, D = Ui + Ii, 64
    x = torch.randn((N, D), device=dev)
    y = torch.empty_like(x)
    def _time_product(fn, reps=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        evs = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / len(evs)

    by = 8.0 * adj.nnz + 8.0 * (N + 1) + 2.0 * N * D * 4
    table = ops.spmm_table_bf16(adj, x)
    ms_fp32 = _time_product(lambda: ops.spmm(adj, x, out=y))
    ms_b16 = _time_product(lambda: ops.spmm_norm_bf16(adj, x, out=y, table=None))
    ms_b16_given = _time_product(lambda: ops.spmm_norm_bf16(adj, table=table, out=y))
    ms = ms_b16 if precision == "bf16" else ms_fp32
    out["spmm_csr"] = {"bound": "hbm", "bytes_per_launch": by, "avg_launch_ms": ms, "achieved": by / (ms * 1e-3) / 1e9,
                       "peak": pk["hbm"], "unit": "GB/s", "frac": by / (ms * 1e-3) / 1e9 / pk["hbm"],
                       "shape": f"ifashion-shaped graph: N = {N} nodes, nnz = {adj.nnz}, D = 64 (working set > L2)",
                       "entry_point": ("dmm_spmm_table_bf16 + dmm_spmm_norm_bf16 (the propagation product of precision bf16: "
                                       "table pass included)" if precision == "bf16" else "dmm_spmm_csr (fp32 gather table)"),
                       "variants_ms": {"fp32_table_dmm_spmm_csr": ms_fp32, "bf16_table_pass_included": ms_b16,
                                       "bf16_table_given": ms_b16_given},
                       "note": "bytes_per_launch is the fp32 product's compulsory traffic 8 nnz + 8 (N + 1) + 2 N D 4 (SURVEY 8d) "
                               "for every variant"}
    for _ in range(2):                      # allocator warm-up: a cudaMalloc between the events would be timed as well
        ops.build_norm_adj(ptr, idx, Ui, Ii)
    torch.cuda.synchronize()
    evs = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.build_norm_adj(ptr, idx, Ui, Ii)
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
    Ei = int(idx.numel())
    by = 8.0 * Ei + 8.0 * (2 * Ei + N) + 8.0 * (N + 1)
    out["build_norm_adj_csr"] = {"bound": "hbm", "bytes_per_launch": by, "avg_launch_ms": ms,
                                 "achieved": by / (ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                                 "frac": by / (ms * 1e-3) / 1e9 / pk["hbm"],
                                 "shape": f"ifashion-shaped: E = {Ei} edges, N = {N} (includes the CUB sort passes)"}
    return out


# ------------------------------------------------------------------------------------------------ reference arm
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def reference_rebuild_step(ref, diff, dens, x_rows, deg, sampling_step):
    """The reference's phase 2 for one set of users (Main.py:211-231 verbatim in structure): per modality and batch of
    1024 users ``generate_view`` (Model.py:300-322) on torch-CPU, then the per-user ``torch.topk`` loop with one
    ``int(tensor)`` per emitted edge.  Returns (seconds, edges)."""
    import torch
    edges = 0
    t0 = time.perf_counter()
    with torch.no_grad():
        for m, den in dens.items():
            i_list = []
            for b0 in range(0, x_rows.shape[0], 1024):
                batch = x_rows[b0:b0 + 1024]
                view = diff.generate_view(den, batch, sampling_step)
                for i in range(batch.shape[0]):
                    _, indices = torch.topk(view[i], k=int(deg[b0 + i]))
                    for j in range(indices.shape[0]):
                        i_list.append(int(indices[j]))
            edges += len(i_list)
    return time.perf_counter() - t0, edges


def load_reference_arm(w, seed, hyper, force_cpu=True):
    """Unmodified reference modules from oracle/_ref (never /root/reference at run time), forced onto the CPU (or left on
    their own ``cuda:0`` path: force_cpu=False), with Denoise weights drawn exactly like the GPU arm's (same seed, same
    construction order)."""
    import torch
    os.environ["DIFFMM_REFERENCE_ROOT"] = REF_DIR
    from oracle import ref_shim
    ref = ref_shim.load_reference(force_cpu=force_cpu)
    cfg = ref_shim.make_config(ref, "tiktok" if len(w["modalities"]) == 3 else "sports")
    cfg.base.denoise_dim = f"[{w['hidden']}]"
    cfg.hyper.steps = hyper["steps"]
    cfg.hyper.noise_scale, cfg.hyper.noise_min, cfg.hyper.noise_max = hyper["noise"]
    cfg.data.user_num, cfg.data.item_num = w["users"], w["items"]
    torch.manual_seed(seed)
    diff = ref.Model.GaussianDiffusion(cfg)
    dens = {m: ref.Model.Denoise([w["items"], w["hidden"]], [w["hidden"], w["items"]], cfg) for m in w["modalities"]}
    return ref, diff, dens


def run_reference(args):
    """CPU arm: the reference's own implementation of the rebuild phase on the box's host cores, on the SAME workload,
    weights (seed) and users as the GPU arm; each step is a bounded sample of `--ref-sample` users (the first ones)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from diffmm_b200 import synth
    w = WORKLOADS[args.workload]
    hyper = workload_hyper(args.workload, args.sampling_step)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)              # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host core
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)
    except Exception:
        pass
    inter = synth.interactions(w["users"], w["items"], seed=args.seed)
    n_sample = min(args.ref_sample, w["users"])
    ptr, idx = inter.indptr, inter.indices
    deg = np.diff(ptr)[:n_sample]
    kind = "reference"
    on_gpu = args.ref_device == "cuda"
    if on_gpu and not (os.path.isfile(os.path.join(REF_DIR, "Model.py")) and torch.cuda.is_available()):
        emit({"impl": "reference", "unavailable": "stock-torch GPU leg needs oracle/_ref and a GPU"})
        return
    if os.path.isfile(os.path.join(REF_DIR, "Model.py")):
        ref, diff, dens = load_reference_arm(w, args.seed, hyper, force_cpu=not on_gpu)
        x = torch.zeros((n_sample, w["items"]), dtype=torch.float32)
        for u in range(n_sample):
            x[u, torch.from_numpy(idx[ptr[u]:ptr[u + 1]].astype(np.int64))] = 1.0
        if on_gpu:
            # the reference's own device path (Main.py:60-77 moves the models with .cuda(), DataHandler the rows): stock
            # torch kernels (cuBLAS fp32 GEMMs, torch.topk per user, one int(tensor) device->host sync per emitted edge)
            x = x.cuda()
            dens = {m: d.cuda() for m, d in dens.items()}
            kind = "reference-on-gpu"

        def step(n):
            dt, e = reference_rebuild_step(ref, diff, dens, x[:n], deg, hyper["sampling_step"])
            return dt, e
    else:   # oracle/_ref not built on this machine: numpy restatement of the same path (oracle/diffmm_oracle.py)
        kind = "port"
        _, _, _, dens_t = build_workload(args.workload, "cpu", args.seed, "bf16", 1, hyper)
        params = {m: oracle_params(d) for m, d in dens_t.items()}

        def step(n):
            dt, _, e = cpu_rebuild_sample(inter, w, params, n, hyper)
            return dt, e
    for _ in range(args.warmup):
        step(min(n_sample, 128))
    total, users = 0.0, 0
    for _ in range(args.steps):
        dt, _ = step(n_sample)
        total += dt
        users += n_sample
    val = users / total
    sample = (f"first {n_sample} of {w['users']} users x {len(w['modalities'])} modalities per step, {args.steps} steps, "
              f"{total:.1f} s; " + ("unmodified reference modules (oracle/_ref: GaussianDiffusion.generate_view + the "
                                    "Main.py:224-230 per-user torch.topk loop) on torch-CPU" if kind.startswith("reference") else
                                    "numpy port (oracle/diffmm_oracle.py)") + f", same seed-{args.seed} weights as the GPU arm")
    if on_gpu:
        sample = sample.replace("on torch-CPU", "on cuda:0 through stock torch (the reference's own .cuda() path)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.workload, w, hyper, args.precision),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def cpu_baseline_subprocess(args, w):
    """The reference arm on a bounded sample, in its own process (it patches torch onto the CPU path and must not share
    a process with GPU work): same workload, seed and hyper-parameters; ~10-20 s of host-core time."""
    import subprocess
    n_cpu = max(64, int(args.cpu_sample * min(1.0, 7050.0 / w["items"])))
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload, "--seed", str(args.seed),
           "--steps", "1", "--warmup", "1", "--ref-sample", str(n_cpu)]
    if args.sampling_step is not None:
        cmd += ["--sampling-step", str(args.sampling_step)]
    env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "MKL_NUM_THREADS")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        ref_line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        return ref_line["cpu_baseline"]
    except Exception as e:
        return {"error": repr(e)[:300]}


def stock_torch_gpu_subprocess(args, w):
    """SURVEY 8(d) "stock library" comparison: the UNMODIFIED reference's rebuild phase on the same B200 through stock
    torch (its own .cuda() path), on a bounded sample of the same workload, in its own process."""
    import subprocess
    n = max(64, int(2048 * min(1.0, 7050.0 / w["items"])))
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-device", "cuda", "--workload", args.workload,
           "--seed", str(args.seed), "--steps", "1", "--warmup", "1", "--ref-sample", str(n)]
    if args.sampling_step is not None:
        cmd += ["--sampling-step", str(args.sampling_step)]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        ref_line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        if "unavailable" in ref_line:
            return {"unavailable": ref_line["unavailable"]}
        cb = ref_line["cpu_baseline"]
        return {"value": cb["value"], "unit": cb["unit"], "kind": cb["kind"], "sample": cb["sample"]}
    except Exception as e:
        return {"error": repr(e)[:300]}


# ------------------------------------------------------------------------------------------------ our arm
class RebuildJob:
    """One rebuild workload on this rank: the synthetic train CSR (global, replicated: it is small), replicated Denoise
    weights, the rank's user block, pinned host buffers for the end-to-end leg, and the step functions.

    scaling 'weak': the job is world x users (each rank owns `users` rows); 'strong': `users` rows split over the ranks.
    N > 1: chain + top-k on the rank's block, ONE NCCL all-gather of the edge lists per modality straight into the final
    buffers (dist.allgather_edges), then the whole-graph adjacencies on every rank."""

    def __init__(self, name, precision, sampling_step, dev, seed, world, rank, scaling="weak", init_on_device=False):
        import torch
        from diffmm_b200 import dist as ddist
        self.name, self.precision, self.dev, self.world, self.rank = name, precision, dev, world, rank
        self.w = w = WORKLOADS[name]
        self.hyper = workload_hyper(name, sampling_step)
        self.users_total = w["users"] * world if scaling == "weak" else w["users"]
        self.cfg, self.inter, self.diff, self.dens = build_workload(name, dev, seed, precision, world, self.hyper,
                                                                    users_total=self.users_total, init_on_device=init_on_device)
        self.I, self.mods = w["items"], w["modalities"]
        self.r0, self.r1 = ddist.row_blocks(self.users_total, world)[rank]
        self.plan = ddist.EdgeGatherPlan(torch.from_numpy(self.inter.indptr), self.users_total, world) if world > 1 else None
        ptr = self.inter.indptr
        self.e0, self.e1 = int(ptr[self.r0]), int(ptr[self.r1])
        self.E = int(self.inter.indices.size)
        self.h_indptr = torch.from_numpy(ptr).pin_memory()
        self.h_indices_local = torch.from_numpy(self.inter.indices[self.e0:self.e1].copy()).pin_memory()
        self.d_indptr = self.h_indptr.to(dev)
        self.d_indices = torch.from_numpy(self.inter.indices).to(dev)
        self.d_indices_e2e = torch.zeros_like(self.d_indices)          # only the rank's slice is ever uploaded into it
        self.h_edges = {m: torch.empty(self.e1 - self.e0, dtype=torch.int32).pin_memory() for m in self.mods}

    def step(self, ip, ix, edges_to_host=False):
        import torch  # noqa: F401
        from diffmm_b200 import autograd as _ag, ops, rebuild
        # everything that depends on the Denoise weights is rebuilt inside the step, as after an epoch of training:
        # bf16 operand copies of W1 / W2 (and their transposes) and the hidden-space operators P = W1x W2, q = W1x b2
        _ag._PACK_CACHE.clear()
        for dn in self.dens.values():
            dn._dmm_hidden_ops = None
        U, I, SS = self.users_total, self.I, self.hyper["sampling_step"]
        if self.world > 1:
            full = {}
            hook = None
            if edges_to_host:     # the rank's slice of every edge list leaves from inside the modality's pipeline
                host = iter(self.h_edges.values())

                def hook(v):
                    next(host).copy_(v[self.e0:self.e1], non_blocking=True)
            adjs = rebuild.rebuild_sharded(self.diff, self.dens, ip, ix, U, I, SS, self.precision, (self.r0, self.r1),
                                           group=None, plan=self.plan, full_items=full, local_hook=hook)
            return adjs, full
        res = {}
        if edges_to_host:
            # end-to-end leg: every modality's edge list leaves for its pinned host buffer from inside its own pipeline, as
            # soon as its top-k has emitted it (the per_modality hook of the public API runs on the pipeline's stream), so
            # the copy overlaps the adjacency build instead of following the join
            host = iter(self.h_edges.values())

            def tail(v):
                next(host).copy_(v[self.e0:self.e1], non_blocking=True)
                return ops.build_norm_adj(ip, v, U, I), v
        else:
            def tail(v):
                return ops.build_norm_adj(ip, v, U, I), v
        rebuild.rebuild_edges(self.diff, self.dens, ip, ix, U, I, SS, self.precision, row_range=(self.r0, self.r1),
                              per_modality=tail, per_modality_out=res)
        return {m: r[0] for m, r in res.items()}, {m: r[1] for m, r in res.items()}

    def step_device(self):
        return self.step(self.d_indptr, self.d_indices)

    def step_e2e(self):
        """Public-API call with HOST inputs and outputs: the train CSR offsets and the rank's slice of the item ids come
        from pinned host memory, the rank's slice of every rebuilt edge list goes back to pinned host memory."""
        ip = self.h_indptr.to(self.dev, non_blocking=True)
        self.d_indices_e2e[self.e0:self.e1].copy_(self.h_indices_local, non_blocking=True)
        adjs, items = self.step(ip, self.d_indices_e2e, edges_to_host=True)
        return adjs

    def h2d_bytes(self):
        return int(self.world * self.h_indptr.numel() * 8 + self.E * 4)          # summed over the ranks

    def d2h_bytes(self):
        return int(len(self.mods) * self.E * 4)


def run_ours(args):
    import torch
    import torch.distributed as td
    from diffmm_b200 import _lib, ops, rebuild

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        td.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warm=2):
        """Sum of the per-step device times (CUDA events on the launching stream, L2 flushed before every step, untimed),
        max over the ranks."""
        for _ in range(warm):
            fn()
        barrier()
        ev = []
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            ev.append((e0, e1))
        barrier()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=dev)
        if world > 1:
            td.all_reduce(t, op=td.ReduceOp.MAX)
        return float(t[0])

    job = RebuildJob(args.workload, args.precision, args.sampling_step, dev, args.seed, world, rank, "weak",
                     init_on_device=args.workload == "scaleout")
    w, hyper = job.w, job.hyper
    U, I, H, S, mods, E = w["users"], w["items"], w["hidden"], hyper["steps"], job.mods, job.E

    # per-launch instrumentation of the dominant kernel (events on the launching stream)
    gemm_events = []
    orig_gemm = ops.gemm_bf16_tn

    def timed_gemm(a_hi, a_lo, b_hi, b_lo, M, N, K, **kw):
        if not timed_gemm.on:
            return orig_gemm(a_hi, a_lo, b_hi, b_lo, M, N, K, **kw)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_gemm(a_hi, a_lo, b_hi, b_lo, M, N, K, **kw)
        e1.record()
        passes = 1 + (a_lo is not None) + (b_lo is not None)
        # compulsory HBM bytes of the call: operands once, every epilogue tensor once
        nbytes = 2.0 * M * K * (1 + (a_lo is not None)) + 2.0 * N * K * (1 + (b_lo is not None))
        nbytes += 4.0 * M * N * ((kw.get("residual") is not None) + (kw.get("out_f32") is not None))
        nbytes += 2.0 * M * N * sum(kw.get(k) is not None for k in ("out_hi", "out_lo", "res_hi", "res_lo"))
        gemm_events.append((2.0 * M * N * K, e0, e1, (M, N, K, passes), nbytes))
    timed_gemm.on = False
    ops.gemm_bf16_tn = timed_gemm
    rebuild.ops.gemm_bf16_tn = timed_gemm
    orig_splitk = ops.gemm_bf16_tn_splitk

    def timed_splitk(a_hi, b_hi, M, N, K, **kw):        # contraction + slab reduce: both launches inside the event pair
        if not timed_gemm.on:
            return orig_splitk(a_hi, b_hi, M, N, K, **kw)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_splitk(a_hi, b_hi, M, N, K, **kw)
        e1.record()
        nbytes = 2.0 * M * K + 2.0 * N * K + 4.0 * M * N * (kw.get("out_f32") is not None) + 2.0 * M * N * (
            (kw.get("out_hi") is not None) + (kw.get("out_lo") is not None))
        gemm_events.append((2.0 * M * N * K, e0, e1, (M, N, K, "1+splitK"), nbytes))
    ops.gemm_bf16_tn_splitk = timed_splitk
    rebuild.ops.gemm_bf16_tn_splitk = timed_splitk

    counts = {}
    orig_call = _lib.call

    def counting_call(name, *a):
        counts[name] = counts.get(name, 0) + 1
        return orig_call(name, *a)
    _lib.call = counting_call
    ops._lib.call = counting_call

    # ---- the timed region of the contract: W warm-up steps, then exactly K steps, device-resident inputs
    for _ in range(max(args.warmup, 3)):
        job.step_device()
    sampler = ClockSampler(local)
    sampler.start()
    counts.clear()
    t_wall0 = time.perf_counter()
    ms = timed(job.step_device, args.steps, warm=0)
    t_wall = time.perf_counter() - t_wall0
    launches = sum(KERNELS_PER_CALL.get(k, 1) * v for k, v in counts.items())

    pk = peaks()

    def gemm_stats(events):
        tot_ms = sum(a.elapsed_time(b) for _, a, b, _, _ in events)
        flops = sum(f for f, _, _, _, _ in events)
        shapes = {}
        for f, a, b, shape, nb in events:
            d = shapes.setdefault("x".join(map(str, shape[:3])) + f"/p{shape[3]}", [0, 0.0, 0.0, 0.0])
            d[0] += 1
            d[1] += a.elapsed_time(b)
            d[2] += f
            d[3] += nb
        out = {}
        for k, v in shapes.items():
            tf, gbs = v[2] / (v[1] * 1e-3) / 1e12, v[3] / (v[1] * 1e-3) / 1e9
            # the roofline that bounds the shape: tensor pipe above the ridge (peak FLOP/s / peak B/s), HBM below it
            intensity, ridge = v[2] / max(v[3], 1.0), pk["tf_burst"] * 1e12 / (pk["hbm"] * 1e9)
            out[k] = {"launches": v[0], "avg_ms": v[1] / v[0], "tflops": tf, "compulsory_GBps": gbs,
                      "flop_per_byte": intensity, "bound": "tensor" if intensity >= ridge else "hbm",
                      "frac_of_its_bound": tf / pk["tf_burst"] if intensity >= ridge else gbs / pk["hbm"]}
            # Third bound, the one that binds the 256 x 256 pair tiles in practice (DESIGN.md section 4, tools/gemm_l2_model.py):
            # bytes a CTA pulls through the L2 per tile (its 128 rows of A + its 128-row half of B per k-block, and its
            # 128 x 256 part of the epilogue tensors) against the measured L2 slice throughput of the chip
            # (B300_MICROARCH "LTS throughput cap" ~6300 B/clk), in waves of 74 pair tiles.
            Ms, Ns, Ks = (int(t) for t in k.split("/")[0].split("x"))
            if Ms >= 256 and Ns > 256 and "splitK" not in k:
                passes = int(k.split("/p")[1][0])
                ep_b = max(v[3] / v[0] - (Ms + Ns) * Ks * 2.0 * (2 if passes > 1 else 1), 0.0) / (Ms * Ns)
                tiles = -(-Ms // 256) * -(-Ns // 256)
                full_w, rem = divmod(tiles, 74)
                waves = full_w + (max(rem / 74.0, 0.25) if rem else 0.0)
                cta_bytes = 2 * 128 * Ks * 2.0 * passes + 128 * 256 * ep_b
                l2_ms = waves * cta_bytes / (6300.0 / 148) / (1.965e9) * 1e3
                out[k].update({"l2_bytes_per_cta_tile": cta_bytes, "l2_bound_ms": l2_ms,
                               "measured_over_l2_bound": (v[1] / v[0]) / l2_ms})
        return tot_ms, flops, out

    # The modalities run as concurrent pipelines on two streams (rebuild.rebuild_edges), so an event pair around a
    # contraction inside the timed region also spans whatever the other stream ran meanwhile.  The kernel's own launch
    # durations therefore come from a second pass of the same K steps with the pipelines serialised on one stream
    # (DIFFMM_STREAMS=1, same inputs, same L2 flush, events on the launching stream).
    n_streams = int(os.environ.get("DIFFMM_STREAMS", "2"))
    os.environ["DIFFMM_STREAMS"] = "1"
    for _ in range(2):
        job.step_device()
    timed_gemm.on = True
    serial_ms = timed(job.step_device, args.steps, warm=0)
    timed_gemm.on = False
    gemm_ms, gemm_flops, by_shape = gemm_stats(gemm_events)

    # per-entry-point device time inside a step (one stream: every call's events see only that call)
    per_call = []

    def timing_call(name, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_call(name, *a)
        e1.record()
        per_call.append((name, e0, e1))
    _lib.call = timing_call
    ops._lib.call = timing_call
    n_bd = 2
    for _ in range(n_bd):
        flush.fill_(1)
        job.step_device()
    barrier()
    _lib.call = orig_call
    ops._lib.call = orig_call
    os.environ["DIFFMM_STREAMS"] = str(n_streams)
    breakdown = {}
    for name, a, b in per_call:
        d = breakdown.setdefault(name, [0, 0.0])
        d[0] += 1
        d[1] += a.elapsed_time(b)
    breakdown = {k: {"calls_per_step": v[0] // n_bd, "ms_per_step": round(v[1] / n_bd, 4)} for k, v in breakdown.items()}

    # ---- end to end through the public call with host buffers (the headline against the reference arm)
    ms_e2e = timed(job.step_e2e, args.steps)
    sampler.stop_flag = True
    sampler.join(timeout=1.0)

    # ---- a >= 1 s timed region of the same step (K steps of ~2 ms are a short sample)
    n_long = int(min(2000, max(args.steps, np.ceil(1000.0 / max(ms / args.steps, 1e-3)))))
    ms_long = timed(job.step_device, n_long, warm=0) if not args.no_long else None

    # the literal chain (2 item-space contractions per reverse step) timed the same way, for the record
    ms_full = None
    if not args.no_variants:
        os.environ["DIFFMM_CHAIN"] = "full"
        ms_full = timed(job.step_device, max(2, args.steps // 2)) / max(2, args.steps // 2)
        os.environ.pop("DIFFMM_CHAIN", None)

    # ---- variants of the same workload: sampling_step 0 (rebuild from the binary rows) and the fp32-faithful precision
    variants = {}
    if not args.no_variants and args.workload != "scaleout":
        k_var = min(args.steps, 10)
        ops.gemm_bf16_tn = orig_gemm
        rebuild.ops.gemm_bf16_tn = orig_gemm
        todo = []
        if hyper["sampling_step"] != 0:
            todo.append(("sampling_step_0", args.precision, 0))
        if args.precision != "bf16x3":
            todo.append(("bf16x3", "bf16x3", args.sampling_step))
        for label, prec, ss in todo:
            vj = RebuildJob(args.workload, prec, ss, dev, args.seed, world, rank, "weak")
            v_ms = timed(vj.step_device, k_var, warm=3)
            v_e2e = timed(vj.step_e2e, k_var, warm=2)
            variants[label] = {"dtype": prec, "sampling_step": vj.hyper["sampling_step"], "steps": k_var,
                               "ms_per_step": v_ms / k_var, "value": world * U * k_var / (v_ms * 1e-3),
                               "e2e_value": world * U * k_var / (v_e2e * 1e-3), "unit": UNIT}
            del vj
            torch.cuda.empty_cache()

    # ---- N > 1: the other configurations BASELINE.json names for the multi-GPU runs
    others = {}
    if world > 1 and not args.no_others and args.workload == "baby":
        for label, name, scaling, k_o in (("sports_strong", "sports", "strong", 6), ("scaleout_slice_weak", "scaleout", "weak", 3)):
            try:
                oj = RebuildJob(name, args.precision, None, dev, args.seed, world, rank, scaling, init_on_device=True)
                o_ms = timed(oj.step_device, k_o, warm=3)
                o_e2e = timed(oj.step_e2e, k_o, warm=1)
                users = oj.users_total
                others[label] = {"workload": config_dict(name, oj.w, oj.hyper, args.precision)["workload"], "scaling": scaling,
                                 "users_total": users, "steps": k_o, "ms_per_step": o_ms / k_o,
                                 "value": users * k_o / (o_ms * 1e-3), "e2e_value": users * k_o / (o_e2e * 1e-3), "unit": UNIT}
                del oj
                torch.cuda.empty_cache()
            except Exception as e:      # the headline line must survive a failure of an auxiliary measurement
                others[label] = {"error": repr(e)[:300]}

    # ---- row-partitioned propagation (BASELINE.json configs[3]): ifashion-shaped graph, per-layer SpMM + all-gather
    prop = None
    if not args.no_prop:
        try:
            prop = propagation_bench(dev, world, rank, args.seed, timed)
        except Exception as e:
            prop = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            td.destroy_process_group()
        return

    # DRAM traffic per launch of the dominant kernel from the committed ncu capture (profiles/ncu_traffic.json),
    # averaged over this run's launch mix; null when a shape has no capture
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["gemm_bf16_tn_kernel"]
        tot, cnt = 0.0, 0
        for _, _, _, shape, _ in gemm_events:
            if shape[3] == "1+splitK":      # captured as the plain launch only: left out of the average
                continue
            ent = tr.get("x".join(map(str, shape[:3])))
            if ent is None or shape[3] != 1:
                tot, cnt = 0.0, 0
                break
            tot += ent["dram_read_bytes"] + ent["dram_write_bytes"]
            cnt += 1
        traffic = tot / cnt if cnt else None
    except Exception:
        traffic = None
    n_gemm = max(len(gemm_events), 1)
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    value = world * U * args.steps / (ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.precision, "data": "synthetic",
        "config": config_dict(args.workload, w, hyper, args.precision),
        "run": {"edges": E, "precision": args.precision, "l2": "256 MiB flush write between timed steps; per-step working set > L2",
                "streams": n_streams if len(mods) > 1 else 1,
                "parallelism": (f"user-sharded x{world}: {job.users_total} users in total, one NCCL all-gather of the edge lists "
                                f"per modality into the final buffers, adjacency of the whole graph on every rank")
                if world > 1 else "single GPU"},
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": pk["tf_burst"], "unit": "TFLOP/s",
                     "frac": achieved / pk["tf_burst"], "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram read + write)",
                     "kernel": "gemm_bf16_tn_kernel (tcgen05)",
                     "launches": len(gemm_events), "avg_launch_ms": gemm_ms / n_gemm, "share_of_step": gemm_ms / serial_ms,
                     "peak_source": f"{pk['source']} bf16_tflops (burst: the timed region is tens of ms at full clocks); "
                                    f"sustained {pk['tf_sustained']}",
                     "frac_of_sustained": achieved / pk["tf_sustained"], "by_shape_MxNxK": by_shape,
                     "frac_of_binding_roofline_time_weighted": (
                         sum(v["frac_of_its_bound"] * v["avg_ms"] * v["launches"] for v in by_shape.values()) /
                         max(sum(v["avg_ms"] * v["launches"] for v in by_shape.values()), 1e-9)),
                     "algorithmic_flops_per_launch": gemm_flops / n_gemm,
                     "measured_in": f"second pass of the same {args.steps} steps with the modality pipelines serialised on one "
                                    f"stream ({serial_ms / args.steps:.3f} ms/step); in the timed region they overlap on "
                                    f"{n_streams} streams and an event pair would also span the other stream's kernels"},
        "e2e": {"value": world * U * args.steps / (ms_e2e * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": job.h2d_bytes(), "d2h_bytes_per_step": job.d2h_bytes()},
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        "wall_s_timed_region": t_wall,
        "chain": {"mode": rebuild.chain_mode(),
                  "note": "hidden-space chain: z_t = x_t W1^T carried in fp32, one [rows,H]x[H,H] contraction per intermediate "
                          "step, item space only for the first gather and the last step; P = W1x W2, q = W1x b2 and all "
                          "operand packs are rebuilt inside every timed step; the scores contraction also writes the chunk "
                          "maxima the pruned top-k reads",
                  "full_chain_ms_per_step": ms_full,
                  "full_chain_users_per_s": (world * U / (ms_full * 1e-3)) if ms_full else None},
        "breakdown_ms_per_step": breakdown,
    }
    if ms_long is not None:
        line["long_run"] = {"steps": n_long, "ms_per_step": ms_long / n_long, "value": world * U * n_long / (ms_long * 1e-3),
                            "timed_region_s": ms_long * 1e-3, "unit": UNIT}
    if variants:
        line["variants"] = variants
    if others:
        line["other_workloads"] = others
    if prop is not None:
        line["propagation"] = prop
    if world == 1 and not args.no_cpu_baseline:          # reported on rank 0 at N = 1 only (a bounded host-core sample)
        line["cpu_baseline"] = cpu_baseline_subprocess(args, w)
        line["stock_torch_gpu"] = stock_torch_gpu_subprocess(args, w)
    if world == 1 and not args.no_aux:
        try:
            line["aux_rooflines"] = aux_rooflines(dev, breakdown, U, I, E, len(mods), pk, args.seed, args.precision)
        except Exception as e:
            line["aux_rooflines"] = {"error": repr(e)[:300]}
    if world == 1 and not args.no_epoch and args.workload in ("tiktok", "baby", "sports"):
        # restore the un-instrumented entry points before running the trainer
        ops.gemm_bf16_tn = orig_gemm
        rebuild.ops.gemm_bf16_tn = orig_gemm
        try:
            # the default configuration (phases 1 and 3 replayed from CUDA graphs) and the eager loop
            line["epoch_sec"] = epoch_seconds(args.workload, args.seed, args.precision, cuda_graph=True)
            line["epoch_sec_eager"] = epoch_seconds(args.workload, args.seed, args.precision, cuda_graph=False)
        except Exception as e:  # the headline number must survive a failure of the auxiliary measurement
            line["epoch_sec"] = {"error": repr(e)[:300]}
    emit(line)
    if world > 1:
        td.destroy_process_group()


def propagation_bench(dev, world, rank, seed, timed):
    """Row-partitioned propagation at the ifashion shape (300k users x 80k items, D = 64): one product Y = A X as the
    product path runs it (autograd.spmm -> dist.PropPartition: local row blocks on the CSR SpMM kernel + in-place NCCL
    all-gather), its two halves timed separately, and the un-partitioned product for comparison."""
    import torch
    import torch.distributed as td
    from diffmm_b200 import autograd as ag, dist as ddist, ops, synth
    Ui, Ii, _ = synth.SHAPES["ifashion"]
    inter = synth.interactions(Ui, Ii, seed=seed)
    ptr = torch.from_numpy(inter.indptr).to(dev)
    idx = torch.from_numpy(inter.indices).to(dev)
    adj = ops.build_norm_adj(ptr, idx, Ui, Ii)
    N, D = Ui + Ii, 64
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn((N, D), device=dev, generator=g)
    y = torch.empty_like(x)
    k = 10
    full_ms = timed(lambda: ops.spmm(adj, x, out=y), k, warm=3) / k
    full_b16_ms = timed(lambda: ops.spmm_norm_bf16(adj, x, out=y), k, warm=3) / k
    out = {"shape": f"ifashion-shaped graph: N = {N} nodes, nnz = {adj.nnz}, D = 64 fp32", "n_gpus": world,
           "full_product_ms": full_ms, "full_product_bf16_ms": full_b16_ms,
           "bytes_per_product": 8.0 * adj.nnz + 8.0 * (N + 1) + 2.0 * N * D * 4}
    if world > 1:
        part = ddist.PropPartition(Ui, Ii, td.group.WORLD)

        def local():
            for r0, r1 in part.row_ranges():
                ops.spmm(adj, x, out=y, row0=r0, row1=r1)
        local_ms = timed(local, k, warm=3) / k
        gather_ms = timed(lambda: part.gather_(y), k, warm=3) / k
        ag.set_partition(part)
        part_ms = timed(lambda: ag.spmm(adj, x), k, warm=3) / k
        ag.set_partition(None)
        # the partitioned product equals the full one
        want = ops.spmm(adj, x)
        ag.set_partition(part)
        got = ag.spmm(adj, x)
        ag.set_partition(None)
        ag.set_partition(part)
        ag.set_spmm_precision("bf16")
        part_b16_ms = timed(lambda: ag.spmm(adj, x), k, warm=3) / k
        ag.set_spmm_precision("bf16x3")
        ag.set_partition(None)
        out["partitioned_product_bf16_ms"] = part_b16_ms
        out.update({"local_row_blocks_ms": local_ms, "allgather_ms": gather_ms, "partitioned_product_ms": part_ms,
                    "allgather_bytes_per_rank": float(N * D * 4) * (world - 1) / world,
                    "allgather_GBps_per_rank": float(N * D * 4) * (world - 1) / world / (gather_ms * 1e-3) / 1e9,
                    "matches_full_product": bool(torch.equal(got, want)),
                    "speedup_vs_full": full_ms / part_ms})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="baby", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "bf16x3"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=8192, help="users of the cpu_baseline sample (scaled down with the row width)")
    ap.add_argument("--ref-sample", type=int, default=1024, help="users per step of the reference (CPU) arm")
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"],
                    help="--impl reference: cpu = the driver's reference arm (host cores); cuda = the same unmodified reference "
                         "through stock torch on the GPU (the stock_torch_gpu leg of the main line)")
    ap.add_argument("--sampling-step", type=int, default=None,
                    help="override the workload's conf/*.toml hyper.sampling_step (0 = rebuild from the binary rows)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true", help="skip the top-k / SpMM / adjacency roofline measurements")
    ap.add_argument("--no-epoch", action="store_true", help="skip the full-epoch (phases 1-3 + eval) timing")
    ap.add_argument("--no-variants", action="store_true", help="skip the sampling_step-0 / bf16x3 / literal-chain variants")
    ap.add_argument("--no-others", action="store_true", help="N > 1: skip the sports strong-scaling and scale-out slice runs")
    ap.add_argument("--no-prop", action="store_true", help="skip the row-partitioned propagation measurement")
    ap.add_argument("--no-long", action="store_true", help="skip the >= 1 s timed region of the same step")
    ap.add_argument("--quick", action="store_true", help="headline only: implies every --no-* switch")
    args = ap.parse_args()
    if args.quick:
        args.no_cpu_baseline = args.no_aux = args.no_epoch = args.no_variants = args.no_others = args.no_prop = args.no_long = True
    # stdout carries exactly ONE JSON line: native libraries (NCCL prints its version banner on fd 1) write to stderr
    # while the run is in progress; the saved descriptor is restored for the result line
    global _RESULT_FD
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    _RESULT_FD = real_stdout
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        _RESULT_FD = 1
        os.close(real_stdout)


if __name__ == "__main__":
    main()
