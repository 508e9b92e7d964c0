"""Configuration dataclasses + TOML loader with the reference's names (Conf.py:9-77).

Differences, all on purpose (SURVEY.md §0):
  * nested dataclasses use default_factory (the reference's instance defaults raise on Python >= 3.11);
  * load_config ignores keys the dataclasses do not know (conf/baby.toml, conf/ifashion.toml and
    conf/test.toml carry stale keys that make the reference's loader raise TypeError) and maps the
    stale spelling ``sampling_steps`` to ``sampling_step`` (so conf/baby.toml runs the rebuild from a q_sample'd
    start at step 5, conf/ifashion.toml and conf/test.toml at step 1: the dense-start path of rebuild.denoise_chain);
  * ``base.precision`` ("bf16" | "bf16x3") selects the tensor-pipe mode of the Denoise contractions.
"""
from __future__ import annotations

import ast
import dataclasses
from dataclasses import dataclass, field

try:  # Python >= 3.11
    import tomllib as _toml

    def _load(path):
        with open(path, "rb") as f:
            return _toml.load(f)
except ModuleNotFoundError:  # pragma: no cover
    import toml as _toml

    def _load(path):
        with open(path, "r") as f:
            return _toml.load(f)


@dataclass
class BaseConfig:
    latdim: int = 64
    topk: int = 20
    gpu: str = "0"
    seed: int = 8888
    denoise_dim: str = "[1024]"
    d_emb_size: int = 10
    cl_method: int = 0
    precision: str = "bf16"     # not in the reference: tensor-pipe mode of the Denoise GEMMs
    cuda_graph: bool = True     # not in the reference: phases 1 and 3 replayed from CUDA graphs (single GPU, device RNG)


@dataclass
class DataConfig:
    name: str = "tiktok"
    # updated by DataHandler.LoadData()
    user_num: int = 0
    item_num: int = 0
    image_feat_dim: int = 0
    text_feat_dim: int = 0
    audio_feat_dim: int = 0


@dataclass
class HyperConfig:
    modal_cl_temp: float = 0.5
    modal_cl_rate: float = 0.01
    cross_cl_temp: float = 0.2
    cross_cl_rate: float = 0.2
    noise_degree: float = 0.2

    noise_scale: float = 0.1
    noise_min: float = 0.0001
    noise_max: float = 0.02
    steps: int = 5

    sim_weight: float = 0.1
    residual_weight: float = 0.5
    modal_adj_weight: float = 0.2

    sampling_step: int = 0

    knn_topk: int = 10


@dataclass
class TrainConfig:
    lr: float = 0.001
    batch: int = 1024
    test_batch: int = 256
    reg: float = 1e-5
    epoch: int = 50
    tstEpoch: int = 1
    gnn_layer: int = 1
    use_lr_scheduler: bool = True


@dataclass
class Config:
    base: BaseConfig = field(default_factory=BaseConfig)
    data: DataConfig = field(default_factory=DataConfig)
    hyper: HyperConfig = field(default_factory=HyperConfig)
    train: TrainConfig = field(default_factory=TrainConfig)


_RENAMES = {"sampling_steps": "sampling_step"}


def _build(cls, raw: dict, ignored: list, section: str):
    known = {f.name for f in dataclasses.fields(cls)}
    kwargs = {}
    for k, v in raw.items():
        k2 = _RENAMES.get(k, k)
        if k2 in known:
            kwargs[k2] = v
        else:
            ignored.append(f"{section}.{k}")
    return cls(**kwargs)


def load_config(path: str) -> Config:
    raw = _load(path)
    ignored: list = []
    cfg = Config(
        base=_build(BaseConfig, raw.get("base", {}), ignored, "base"),
        data=_build(DataConfig, raw.get("data", {}), ignored, "data"),
        hyper=_build(HyperConfig, raw.get("hyper", {}), ignored, "hyper"),
        train=_build(TrainConfig, raw.get("train", {}), ignored, "train"),
    )
    cfg.ignored_keys = ignored  # type: ignore[attr-defined]
    validate(cfg)
    return cfg


def validate(cfg: Config) -> None:
    """Range checks the reference leaves to an IndexError deep inside the diffusion tables (Model.py:305-306 indexes
    the schedule with sampling_step - 1)."""
    if not (0 <= int(cfg.hyper.sampling_step) <= int(cfg.hyper.steps)):
        raise ValueError(f"hyper.sampling_step must lie in [0, steps = {cfg.hyper.steps}], got {cfg.hyper.sampling_step}")
    if int(cfg.hyper.steps) < 1:
        raise ValueError(f"hyper.steps must be >= 1, got {cfg.hyper.steps}")
    if cfg.base.precision not in ("bf16", "bf16x3"):
        raise ValueError(f"base.precision must be 'bf16' or 'bf16x3', got {cfg.base.precision!r}")
    # Main.py:155-156 literal_eval's the hidden widths of the Denoise; an empty list builds a Denoise without layers
    # (the loss shapes fail in the reference too)
    try:
        dims = ast.literal_eval(cfg.base.denoise_dim) if isinstance(cfg.base.denoise_dim, str) else None
    except (ValueError, SyntaxError, TypeError, MemoryError, RecursionError):
        dims = None
    if not (isinstance(dims, list) and dims and all(type(w) is int and w > 0 for w in dims)):
        raise ValueError(f"base.denoise_dim must be a non-empty list of positive ints such as \"[1024]\", "
                         f"got {cfg.base.denoise_dim!r}")
    # the time-embedding kernels (dmm_train_prep, dmm_time_embedding, dmm_time_bias) take widths 2 ... 64 and would
    # reject any other one only at their first launch
    d = cfg.base.d_emb_size
    if not (type(d) is int and 2 <= d <= 64):
        raise ValueError(f"base.d_emb_size must be an int in [2, 64], got {d!r}")
