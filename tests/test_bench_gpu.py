"""bench.py --dump-outputs: the headline run writes what its last timed step computed, and with the same arguments two
runs write the same arrays (inputs, weights and noise all come from --seed), so two builds can be compared output for
output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--quick", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    return json.loads(lines[0])


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from diffmm_b200 import ops, synth
    line = _bench(tmp_path / "a")
    assert line["steps"] == 2
    w = bench.WORKLOADS["baby"]
    U, I, mods = w["users"], w["items"], w["modalities"]
    names = sorted(f"{m}_{k}.npy" for m in mods for k in ("items", "adj_ptr", "adj_idx", "adj_val"))
    assert sorted(os.listdir(tmp_path / "a")) == names
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES
    inter = synth.interactions(U, I, seed=0)
    ptr = torch.from_numpy(inter.indptr).cuda()
    for m in mods:
        got = {k: np.load(tmp_path / "a" / f"{m}_{k}.npy") for k in ("items", "adj_ptr", "adj_idx", "adj_val")}
        assert got["items"].dtype == np.float64 and got["adj_val"].dtype == np.float32
        items = got["items"].astype(np.int32)
        assert np.array_equal(items, got["items"]) and len(items) == inter.indices.size
        assert items.min() >= 0 and items.max() < I
        # k = deg(u) distinct items per user, and the adjacency is the one built from exactly this edge list
        u = np.repeat(np.arange(U), np.diff(inter.indptr))
        assert np.unique(u.astype(np.int64) * I + items).size == items.size
        adj = ops.build_norm_adj(ptr, torch.from_numpy(items).cuda(), U, I)
        assert np.array_equal(adj.ptr.cpu().numpy(), got["adj_ptr"])
        assert np.array_equal(adj.idx.cpu().numpy(), got["adj_idx"])
        assert np.array_equal(adj.val.cpu().numpy(), got["adj_val"])
    _bench(tmp_path / "b")
    for f in names:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
