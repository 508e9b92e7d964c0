"""CPU-only tests of the host logic around the kernels: the stream-exact negative sampler, the vectorised
train loader and the vectorised Recall/NDCG arithmetic must reproduce the reference's Python loops exactly
(reference DataHandler.py:145-179, Main.py:422-448)."""
import numpy as np
import torch
from scipy.sparse import coo_matrix
from torch.utils.data import DataLoader

from diffmm_b200 import Main, synth
from diffmm_b200.Conf import Config
from diffmm_b200.DataHandler import TrainData, TrainLoader


def _train_data(U, I, mean_deg, seed):
    inter = synth.interactions(U, I, seed=seed, mean_deg=mean_deg)
    rows = np.repeat(np.arange(U), np.diff(inter.indptr))
    m = coo_matrix((np.ones(len(rows)), (rows, inter.indices)), shape=(U, I))
    cfg = Config()
    cfg.data.item_num, cfg.data.user_num = I, U
    return TrainData(m, cfg)


def test_neg_sampling_replays_the_reference_loop_and_rng_state():
    for U, I, md, seed in [(600, 150, 25, 3), (3000, 2000, 6.4, 0), (200, 4000, 35, 9)]:
        td = _train_data(U, I, md, seed)
        np.random.seed(7)
        td.negSamplingLoop()
        want, want_next = td.negs.copy(), np.random.randint(1 << 30)
        np.random.seed(7)
        td.negSampling()
        got, got_next = td.negs.copy(), np.random.randint(1 << 30)
        assert got.dtype == np.int32
        np.testing.assert_array_equal(got, want)
        assert got_next == want_next                     # the global generator is left where the loop leaves it
        keys = set(zip(td.rows.tolist(), td.cols.tolist()))
        assert not any((u, n) in keys for u, n in zip(td.rows.tolist(), got.tolist()))


def test_train_loader_matches_torch_dataloader():
    td = _train_data(500, 300, 8, 1)
    np.random.seed(0)
    td.negSampling()
    torch.manual_seed(123)
    ref = [tuple(t.clone() for t in b) for b in DataLoader(td, batch_size=128, shuffle=True, num_workers=0)]
    nxt_ref = torch.rand(1)
    torch.manual_seed(123)
    loader = TrainLoader(td, 128)
    got = list(loader)
    nxt = torch.rand(1)
    assert len(loader) == len(ref) == len(got)
    for a, b in zip(ref, got):
        for x, y in zip(a, b):
            assert x.dtype == y.dtype and torch.equal(x, y)
    assert torch.equal(nxt, nxt_ref)                      # same CPU-generator consumption


def _calc_res_reference(top_idxs, test_u_its, users, topk):
    allRecall = allNdcg = allPrecision = 0
    for i in range(len(users)):
        u_rec_list = list(top_idxs[i])
        u_its = test_u_its[users[i]]
        tstNum = len(u_its)
        maxDcg = np.sum([np.reciprocal(np.log2(loc + 2)) for loc in range(min(tstNum, topk))])
        recall_hits = dcg = 0
        for item in u_its:
            if item in u_rec_list:
                recall_hits += 1
                dcg += np.reciprocal(np.log2(u_rec_list.index(item) + 2))
        allRecall += recall_hits / tstNum
        allNdcg += dcg / maxDcg
        allPrecision += recall_hits / topk
    return allRecall, allNdcg, allPrecision


def test_calc_res_is_bit_identical_to_the_reference_loop():
    class NS:
        pass
    coach = Main.Coach.__new__(Main.Coach)
    coach.config = NS()
    coach.config.base = NS()
    coach.config.base.topk = 20
    rng = np.random.default_rng(0)
    B, I = 257, 400
    top = np.stack([rng.permutation(I)[:20] for _ in range(B)])
    test = [list(rng.choice(I, size=rng.integers(1, 35), replace=False)) for _ in range(B)]
    users = torch.arange(B)
    want = _calc_res_reference(top, test, users.tolist(), 20)
    got = coach.calcRes(top, test, users)
    assert tuple(float(x) for x in got) == tuple(float(x) for x in want)


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference: stdout carries exactly one JSON line (native banners go to stderr) with the contract's
    keys; the arm runs the CPU oracle port on a bounded sample (no GPU, no reference checkout needed)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-sample", "32"], capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "denoise_topk_rebuild_users_per_sec" and d["unit"] == "users/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


# ---------------------------------------------------------------------------------------------- configuration (f4)
import os
import pytest
from diffmm_b200.Conf import load_config

_CONF = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "conf")
_EXPECT = {   # file -> (data.name, seed, sampling_step, cl_method, residual_weight, stale keys the loader must drop)
    "tiktok.toml": ("tiktok", 1818, 0, 0, 0.5, []),
    "sports.toml": ("sports", 2233, 0, 1, 0.5, []),
    "yelp.toml": ("yelp", 125, 0, 1, 0.5, []),
    "baby.toml": ("baby", 999, 5, 1, 0.2, ["base.trans", "hyper.keepRate", "hyper.e_loss", "hyper.rebuild_k", "train.norm",
                                           "train.sampling_noise"]),
    "ifashion.toml": ("ifashion", 1818, 1, 1, 0.5, ["base.trans", "hyper.keepRate", "hyper.e_loss", "train.norm",
                                                    "train.sampling_noise"]),
    "test.toml": ("tiktok", 1818, 1, 0, 0.5, ["base.trans", "hyper.keepRate", "hyper.e_loss", "train.norm",
                                              "train.sampling_noise"]),
}


@pytest.mark.parametrize("name", sorted(_EXPECT))
def test_load_config_accepts_every_shipped_toml(name):
    """All six conf/*.toml of the reference load (three of them carry stale keys its own loader rejects, Conf.py:69-77)."""
    cfg = load_config(os.path.join(_CONF, name))
    data_name, seed, sstep, clm, rw, stale = _EXPECT[name]
    assert (cfg.data.name, cfg.base.seed, cfg.hyper.sampling_step, cfg.base.cl_method) == (data_name, seed, sstep, clm)
    assert cfg.hyper.residual_weight == rw and cfg.hyper.steps == 5 and cfg.base.denoise_dim == "[1024]"
    assert sorted(cfg.ignored_keys) == sorted(stale)
    assert cfg.base.precision == "bf16"


@pytest.mark.parametrize("name", sorted(_EXPECT))
def test_shipped_tomls_carry_the_reference_values(name):
    """tests/golden/reference_conf.json holds the reference's conf/*.toml, parsed (oracle/gen_golden.py)."""
    import json
    import tomllib
    from conftest import GOLDEN
    with open(os.path.join(GOLDEN, "reference_conf.json")) as f, open(os.path.join(_CONF, name), "rb") as g:
        assert tomllib.load(g) == json.load(f)[name]


def test_load_config_rejects_a_sampling_step_beyond_the_schedule(tmp_path):
    p = tmp_path / "bad.toml"
    p.write_text("[hyper]\nsteps = 5\nsampling_step = 6\n")
    with pytest.raises(ValueError):
        load_config(str(p))


def test_reference_arm_and_gpu_arm_draw_identical_denoise_weights(monkeypatch):
    """bench.py's two arms must time the same model: the GPU arm's Denoise models and GaussianDiffusion
    (bench.build_workload) draw the reference's weights and noise schedule from the same seed.  The reference's side is
    golden data of oracle/gen_golden.py: its Denoise (I = 120, H = 32) drawn right after torch.manual_seed(1818), then
    moved by 0.05 * randn_like of every parameter, and its schedules for the noise of conf/tiktok.toml and of
    conf/sports.toml (which conf/baby.toml shares).  Replaying those moves on the first modality gives the same tensors
    bit for bit only if its construction drew exactly the reference's numbers, in the reference's order and count; the
    second modality must then be the same construction from where the first one left the generator, as in the
    reference arm (bench.load_reference_arm)."""
    import bench
    from conftest import load_golden, params_of
    from diffmm_b200.Model import Denoise
    g, sched = load_golden("denoise_forward"), load_golden("schedule")
    for name, golden_noise in (("tiktok", "tiktok"), ("baby", "sports")):
        hyper = bench.workload_hyper(name)
        assert hyper["noise"] + (hyper["steps"],) == tuple(sched[f"{golden_noise}.args"]), name
        monkeypatch.setitem(bench.WORKLOADS, name, dict(users=40, items=120, modalities=["image", "text"], hidden=32,
                                                        conf=f"{name}.toml"))
        _, _, diff, _ = bench.build_workload(name, "cpu", 1818, "bf16", 1, hyper)
        np.testing.assert_array_equal(diff.posterior_mean_coef1.cpu().numpy(),
                                      sched[f"{golden_noise}.posterior_mean_coef1"], err_msg=name)
    hyper = bench.workload_hyper("baby")
    cfg, _, _, dens = bench.build_workload("baby", "cpu", 1818, "bf16", 1, hyper)
    # the first modality: the reference's draws (golden replay)
    monkeypatch.setitem(bench.WORKLOADS, "baby", dict(users=40, items=120, modalities=["image"], hidden=32,
                                                      conf="baby.toml"))
    _, _, _, first = bench.build_workload("baby", "cpu", 1818, "bf16", 1, hyper)
    after_first = torch.get_rng_state()
    moved = {k: v.clone() for k, v in first["image"].state_dict().items()}
    for k in moved:                                   # parameters() order == state_dict() order for Denoise
        moved[k].add_(0.05 * torch.randn_like(moved[k]))
    want = params_of(g)
    names = dict(emb_w="emb_layer.weight", emb_b="emb_layer.bias", w1="in_layers.0.weight", b1="in_layers.0.bias",
                 w2="out_layers.0.weight", b2="out_layers.0.bias", gate_w="gate_layer.weight", gate_b="gate_layer.bias")
    assert sorted(names.values()) == sorted(moved)
    for k, sd in names.items():
        np.testing.assert_array_equal(moved[sd].numpy(), want[k], err_msg=k)
    # both modalities of the two-modality workload: the first as above, the second drawn where the first left off
    torch.set_rng_state(after_first)
    second = Denoise([120, 32], [32, 120], cfg)
    for m, ref in (("image", first["image"]), ("text", second)):
        so, sr = dens[m].state_dict(), ref.state_dict()
        assert list(so) == list(sr)
        for k in so:
            assert torch.equal(so[k], sr[k]), (m, k)


def test_bench_dump_outputs_writes_float_arrays_within_the_budget(tmp_path):
    """bench.py --dump-outputs: integer outputs become exact float64, fp32 stays fp32; over the byte budget every array
    keeps the same seeded sample of its elements, the same from run to run."""
    import bench
    ids = np.arange(5000, dtype=np.int32) * 7
    vals = torch.linspace(0, 1, 3000)
    bench.dump_outputs(str(tmp_path / "all"), {"ids": ids, "vals": vals})
    a, v = np.load(tmp_path / "all" / "ids.npy"), np.load(tmp_path / "all" / "vals.npy")
    assert a.dtype == np.float64 and np.array_equal(a, ids) and v.dtype == np.float32 and np.array_equal(v, vals.numpy())
    budget = 3 * bench.NPY_HEADER_BYTES + 20000
    for run in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / run), {"ids": ids, "vals": vals, "one": np.ones(10, np.float64)}, budget=budget)
    files = sorted((tmp_path / "s1").iterdir())
    assert sum(f.stat().st_size for f in files) <= budget
    for f in files:
        s1, s2 = np.load(f), np.load(tmp_path / "s2" / f.name)
        assert 0 < s1.size and np.array_equal(s1, s2)
    s = np.load(tmp_path / "s1" / "ids.npy")
    assert np.all(np.diff(s) > 0) and np.all(np.isin(s, ids))


def test_fused_step_adam_falls_back_to_torch_on_unsupported_configurations():
    """optim.FusedStepAdam only takes the one-launch path for the graph-mode configuration (CUDA fp32 parameters, capturable,
    tensor lr, no weight decay); everything else -- here CPU parameters -- is torch's own step, bit for bit."""
    import torch
    from torch.optim.adam import Adam
    from diffmm_b200.optim import FusedStepAdam
    torch.manual_seed(0)
    a = [torch.randn(7, 3, requires_grad=True), torch.randn(5, requires_grad=True)]
    b = [t.detach().clone().requires_grad_(True) for t in a]
    oa, ob = FusedStepAdam(a, lr=1e-2, weight_decay=0.1), Adam(b, lr=1e-2, weight_decay=0.1)
    for _ in range(5):
        for x, y in zip(a, b):
            g = torch.randn_like(x)
            x.grad, y.grad = g.clone(), g.clone()
        oa.step()
        ob.step()
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert oa.state_dict()["param_groups"][0]["lr"] == ob.state_dict()["param_groups"][0]["lr"]


def test_bench_rejects_dump_outputs_for_the_reference_arm(tmp_path):
    """--dump-outputs writes what our timed path computed; the reference arm has nothing to write, so the combination is
    an argument error instead of an empty directory."""
    import subprocess
    import sys
    root = os.path.dirname(_CONF)
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--dump-outputs",
                        str(tmp_path / "out")], capture_output=True, text=True, timeout=120, cwd=root)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr, r.stderr[-1000:]
    assert not (tmp_path / "out").exists()
