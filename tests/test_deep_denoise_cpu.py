"""denoise_dim with more than one entry (reference Model.py:160-162,211-218, Main.py:155-156) on the host: the config check,
the deep Denoise's parameter names and shapes, and the numpy oracle's multi-layer forward against a float64 torch
restatement of the reference's Denoise.forward (and against the reference's own Denoise where its sources are present)."""
import ast
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import diffmm_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg(denoise_dim="[1000, 200]", I=300):
    from diffmm_b200.Conf import Config
    cfg = Config()
    cfg.base.denoise_dim = denoise_dim
    cfg.data.item_num = I
    return cfg


def _deep_denoise(denoise_dim, I, seed=0):
    """Denoise built the way Main.py:155-156 builds it."""
    from diffmm_b200.Model import Denoise
    cfg = _cfg(denoise_dim, I)
    out_dims = ast.literal_eval(denoise_dim) + [I]
    torch.manual_seed(seed)
    return Denoise(out_dims[::-1], out_dims, cfg), cfg


def test_conf_accepts_deep_denoise_dim():
    from diffmm_b200.Conf import validate
    for ok in ("[1000, 200]", "[1024]", "[96, 160, 136]"):
        validate(_cfg(ok))


@pytest.mark.parametrize("bad", ["[]", "[0]", "[-4, 8]", "abc", "[1.5]", "1024", "[True]", "(8, 8)"])
def test_conf_rejects_bad_denoise_dim(bad):
    from diffmm_b200.Conf import validate
    with pytest.raises(ValueError, match="denoise_dim"):
        validate(_cfg(bad))


@pytest.mark.parametrize("bad", [0, 1, 65, 1000, -10, 10.0, "10", True, None])
def test_conf_rejects_bad_d_emb_size(bad):
    """The time-embedding kernels take widths 2 ... 64; load_config must say so instead of the first kernel call."""
    from diffmm_b200.Conf import validate
    cfg = _cfg("[1024]")
    cfg.base.d_emb_size = bad
    with pytest.raises(ValueError, match="d_emb_size"):
        validate(cfg)


def test_conf_accepts_d_emb_size_range(tmp_path):
    from diffmm_b200.Conf import load_config, validate
    for ok in (2, 9, 10, 64):
        cfg = _cfg("[1024]")
        cfg.base.d_emb_size = ok
        validate(cfg)
    p = tmp_path / "x.toml"
    p.write_text('[base]\nd_emb_size = 65\n')
    with pytest.raises(ValueError, match="d_emb_size"):
        load_config(str(p))
    p.write_text('[base]\nd_emb_size = 64\n')
    assert load_config(str(p)).base.d_emb_size == 64


def test_load_config_rejects_bad_denoise_dim(tmp_path):
    from diffmm_b200.Conf import load_config
    p = tmp_path / "x.toml"
    p.write_text('[base]\ndenoise_dim = "[]"\n')
    with pytest.raises(ValueError, match="denoise_dim"):
        load_config(str(p))
    p.write_text('[base]\ndenoise_dim = "[1000, 200]"\n')
    assert load_config(str(p)).base.denoise_dim == "[1000, 200]"


@pytest.mark.parametrize("denoise_dim", ["[1000, 200]", "[96, 160, 136]"])
def test_deep_denoise_has_the_reference_state_dict(denoise_dim):
    I, d = 300, 10
    den, _ = _deep_denoise(denoise_dim, I)
    dims = ast.literal_eval(denoise_dim)
    out_dims = dims + [I]
    in_dims = out_dims[::-1]
    in_tmp = [in_dims[0] + d] + in_dims[1:]
    want = {"emb_layer.weight": (d, d), "emb_layer.bias": (d,), "gate_layer.weight": (64, 64), "gate_layer.bias": (64,)}
    for k, (a, b) in enumerate(zip(in_tmp[:-1], in_tmp[1:])):
        want[f"in_layers.{k}.weight"], want[f"in_layers.{k}.bias"] = (b, a), (b,)
    for k, (a, b) in enumerate(zip(out_dims[:-1], out_dims[1:])):
        want[f"out_layers.{k}.weight"], want[f"out_layers.{k}.bias"] = (b, a), (b,)
    got = {k: tuple(v.shape) for k, v in den.state_dict().items()}
    assert got == want
    assert len(den.in_layers) == len(den.out_layers) == len(dims)
    from diffmm_b200.rebuild import hidden_widths
    L = len(dims)
    assert hidden_widths(den) == tuple(dims[::-1] + dims[1:])           # d_L .. d_1 .. d_L: 2L - 1 activations
    assert len(hidden_widths(den)) == 2 * L - 1


def _params(den):
    f = lambda t: t.detach().numpy().astype(np.float32)  # noqa: E731
    return dict(emb_w=f(den.emb_layer.weight), emb_b=f(den.emb_layer.bias),
                w1=[f(m.weight) for m in den.in_layers], b1=[f(m.bias) for m in den.in_layers],
                w2=[f(m.weight) for m in den.out_layers], b2=[f(m.bias) for m in den.out_layers],
                gate_w=f(den.gate_layer.weight), gate_b=f(den.gate_layer.bias))


def _torch_forward64(den, x_t, t, feat=None):
    """Model.py:183-220 in float64 torch: time embedding, optional gate, in_layers with tanh, out_layers with tanh
    between them."""
    D = lambda p: p.detach().double()  # noqa: E731
    x = x_t.double()
    d = den.time_emb_dim
    half = d // 2
    freqs = torch.exp(-np.log(10000.0) * torch.arange(half, dtype=torch.float32) / half).double()
    ang = t[:, None].double() * freqs[None]
    temb = torch.cat([torch.cos(ang), torch.sin(ang)], -1) @ D(den.emb_layer.weight).t() + D(den.emb_layer.bias)
    if feat is not None:
        f = feat.double()
        proj = x @ f
        gate = torch.sigmoid(proj @ D(den.gate_layer.weight).t() + D(den.gate_layer.bias))
        x = x + (proj * gate) @ f.t()
    h = torch.cat([x, temb], -1)
    for m in den.in_layers:
        h = torch.tanh(h @ D(m.weight).t() + D(m.bias))
    for i, m in enumerate(den.out_layers):
        h = h @ D(m.weight).t() + D(m.bias)
        if i != len(den.out_layers) - 1:
            h = torch.tanh(h)
    return h


@pytest.mark.parametrize("denoise_dim", ["[1000, 200]", "[96, 160, 136]", "[64]"])
@pytest.mark.parametrize("gated", [False, True])
def test_oracle_list_forward_matches_float64_restatement(denoise_dim, gated):
    I, B = 300, 17
    den, _ = _deep_denoise(denoise_dim, I, seed=3)
    rng = np.random.default_rng(1)
    x_t = (rng.random((B, I)) < 0.05).astype(np.float32) + rng.standard_normal((B, I)).astype(np.float32) * 0.1
    t = rng.integers(0, 5, B)
    feat = (rng.standard_normal((I, 64)) * 0.1).astype(np.float32) if gated else None
    got = O.denoise_forward(_params(den), x_t, t, feat)
    want = _torch_forward64(den, torch.from_numpy(x_t), torch.from_numpy(t),
                            torch.from_numpy(feat) if gated else None).numpy()
    assert got.shape == (B, I)
    assert np.abs(got - want).max() <= 1e-5 * max(1.0, np.abs(want).max())


_REF_SCRIPT = r"""
import ast, sys
import numpy as np
import torch
sys.path.insert(0, {root!r})
from oracle import ref_shim
ref = ref_shim.load_reference(force_cpu=True)
from oracle import diffmm_oracle as O
I, B, d = 300, 17, 10
cfg = ref_shim.make_config(ref, "tiktok", **{{"base.denoise_dim": {dims!r}}})
cfg.data.item_num = I
out_dims = ast.literal_eval({dims!r}) + [I]
torch.manual_seed(3)
den = ref.Model.Denoise(out_dims[::-1], out_dims, cfg)
rng = np.random.default_rng(1)
x_t = (rng.random((B, I)) < 0.05).astype(np.float32) + rng.standard_normal((B, I)).astype(np.float32) * 0.1
t = rng.integers(0, 5, B)
feat = (rng.standard_normal((I, 64)) * 0.1).astype(np.float32)
f = lambda p: p.detach().numpy().astype(np.float32)
p = dict(emb_w=f(den.emb_layer.weight), emb_b=f(den.emb_layer.bias),
         w1=[f(m.weight) for m in den.in_layers], b1=[f(m.bias) for m in den.in_layers],
         w2=[f(m.weight) for m in den.out_layers], b2=[f(m.bias) for m in den.out_layers],
         gate_w=f(den.gate_layer.weight), gate_b=f(den.gate_layer.bias))
with torch.no_grad():
    want = den(torch.from_numpy(x_t), torch.from_numpy(t), torch.from_numpy(feat)).numpy()
got = O.denoise_forward(p, x_t, t, feat)
err = float(np.abs(got - want).max() / max(1.0, np.abs(want).max()))
assert err <= 1e-5, err
print("ok", err)
"""


@pytest.mark.parametrize("denoise_dim", ["[1000, 200]", "[96, 160, 136]"])
def test_reference_deep_denoise_matches_the_oracle(denoise_dim):
    """The reference's own Denoise (run in a child process: the shim forces its CPU path for the whole process)."""
    sys.path.insert(0, ROOT)
    from oracle import ref_shim
    if not ref_shim.available():
        pytest.skip("reference sources not present (oracle/_ref)")
    r = subprocess.run([sys.executable, "-c", _REF_SCRIPT.format(root=ROOT, dims=denoise_dim)], capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
