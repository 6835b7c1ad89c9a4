"""Stand-ins for the reference's absent dependencies, so that ITS OWN hot-path code runs unmodified in this container.

Test infrastructure only. The reference (a read-only checkout of ml-jku/LRAM, named by LRAM_REFERENCE_ROOT) imports
`gym`, `stable_baselines3`, `omegaconf`, `dacite`, `torchmetrics`, `h5py` and the third-party `xlstm`; none is installed and none can be fetched. `install()`:
  * registers small functional stubs for the handful of symbols the path really executes (gym spaces, SB3's
    `is_image_space` / `get_obs_shape` / `get_action_dim` / `BaseFeaturesExtractor`, `OmegaConf.to_container`,
    `dacite.from_dict`),
  * auto-stubs everything else those packages are asked for (imported names become inert placeholder classes),
  * auto-stubs the reference's own sub-packages that are NOT on the path (buffers, optimizers, envs, schedulers,
    augmentations, utils, callbacks.builder ...) while the modules ON the path are imported from the real files,
  * registers `oracle.xlstm_shim` as `xlstm` (module layout of v1.0.x as the reference imports it).
After that `from src.algos.models.decision_xlstm import MultiDomainDiscreteDecisionXLSTMModel`,
`from src.algos.decision_xlstm import DiscreteDecisionXLSTM` and
`from src.callbacks.evaluation import custom_evaluate_policy` are the reference's real code.

Used by tests/golden/make_ref_golden.py (fixture generator) and by CPU tests that skip unless LRAM_REFERENCE_ROOT
names such a checkout (the reference is not part of this repository).
"""
from __future__ import annotations

import dataclasses
import importlib.abc
import importlib.machinery
import os
import sys
import types
import typing

import numpy as np
import torch
import torch.nn as nn

REFERENCE_ROOT = os.environ.get("LRAM_REFERENCE_ROOT", "")
SKIP_REASON = "needs a checkout of the reference (ml-jku/LRAM): set LRAM_REFERENCE_ROOT"

# third-party packages that are absent here
_STUB_TOPLEVEL = ("gym", "stable_baselines3", "omegaconf", "dacite", "torchmetrics", "h5py", "xlstm", "wandb_stub")
# reference sub-packages off the hot path (prefix match), auto-stubbed instead of imported
_STUB_SRC_PREFIXES = (
    "src.buffers", "src.optimizers", "src.envs", "src.utils", "src.schedulers", "src.augmentations", "src.data",
    "src.callbacks.builder", "src.callbacks.custom_eval_callback", "src.callbacks.validation_callback",
    "src.algos.models.custom_critic", "src.algos.models.extractors",
)
# ... except these, which the path executes and which import cleanly once the stubs are in
_REAL_SRC = ("src.buffers.buffer_utils", "src.envs.env_utils")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "algos", "models"))


class _AutoStub(types.ModuleType):
    """A module every attribute of which is an inert placeholder class (cached by name)."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        cls = type(name, (), {"__init__": lambda self, *a, **k: None, "__module__": self.__name__})
        setattr(self, name, cls)
        return cls


class _Finder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path=None, target=None):
        top = fullname.split(".")[0]
        if top in _STUB_TOPLEVEL and fullname not in sys.modules:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        if fullname in _REAL_SRC:
            return None
        if any(fullname == p or fullname.startswith(p + ".") for p in _STUB_SRC_PREFIXES):
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        m = _AutoStub(spec.name)
        # a stubbed reference package keeps its real directory so that the _REAL_SRC modules below it still import
        real = os.path.join(REFERENCE_ROOT, *spec.name.split("."))
        m.__path__ = [real] if (spec.name.startswith("src.") and os.path.isdir(real)) else []
        return m

    def exec_module(self, module):
        return None


# ---- gym ---------------------------------------------------------------------------------------------------------------
class _Space:
    shape: tuple = ()
    dtype = None


class Box(_Space):
    def __init__(self, low, high, shape=None, dtype=np.float32, seed=None):
        self.shape = tuple(shape) if shape is not None else tuple(np.shape(low))
        self.dtype = np.dtype(dtype)
        self.low = np.broadcast_to(np.asarray(low, dtype=self.dtype), self.shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=self.dtype), self.shape).copy()
        self._rng = np.random.default_rng(0 if seed is None else seed)

    def sample(self):
        if np.issubdtype(self.dtype, np.integer):
            return self._rng.integers(self.low, self.high.astype(np.int64) + 1, size=self.shape).astype(self.dtype)
        return self._rng.uniform(self.low, self.high, size=self.shape).astype(self.dtype)


class Discrete(_Space):
    def __init__(self, n, seed=None):
        self.n = int(n)
        self.shape = ()
        self.dtype = np.dtype(np.int64)
        self._rng = np.random.default_rng(0 if seed is None else seed)

    def sample(self):
        return int(self._rng.integers(self.n))


def _is_image_space(observation_space, check_channels: bool = False, normalized_image: bool = False) -> bool:
    # stable_baselines3.common.preprocessing.is_image_space: uint8 Box in [0, 255] with 3 dims
    if isinstance(observation_space, Box) and len(observation_space.shape) == 3:
        if observation_space.dtype != np.uint8:
            return False
        return bool(np.all(observation_space.low == 0) and np.all(observation_space.high == 255))
    return False


def _get_obs_shape(space):
    if isinstance(space, Box):
        return space.shape
    if isinstance(space, Discrete):
        return (1,)
    raise NotImplementedError(type(space))


def _get_action_dim(space) -> int:
    if isinstance(space, Box):
        return int(np.prod(space.shape))
    if isinstance(space, Discrete):
        return 1
    raise NotImplementedError(type(space))


class _BaseFeaturesExtractor(nn.Module):
    def __init__(self, observation_space, features_dim: int = 0):
        super().__init__()
        self._observation_space = observation_space
        self._features_dim = features_dim

    @property
    def features_dim(self):
        return self._features_dim


# ---- omegaconf / dacite ----------------------------------------------------------------------------------------------
class _OmegaConf:
    @staticmethod
    def to_container(cfg, resolve=True, throw_on_missing=False):
        return cfg


def _from_dict(data_class, data, config=None):
    """dacite.from_dict for nested dataclasses with Optional[...] / List[...] fields, strict on unknown keys."""
    hints = typing.get_type_hints(data_class)
    names = {f.name for f in dataclasses.fields(data_class)}
    unknown = set(data) - names
    if unknown and getattr(config, "strict", False):
        raise ValueError(f"unknown keys for {data_class.__name__}: {sorted(unknown)}")
    kw = {}
    for k, v in data.items():
        t = hints[k]
        args = [a for a in typing.get_args(t) if a is not type(None)]
        inner = args[0] if (typing.get_origin(t) is typing.Union and args) else t
        if dataclasses.is_dataclass(inner) and isinstance(v, dict):
            v = _from_dict(inner, v, config)
        kw[k] = v
    return data_class(**kw)


@dataclasses.dataclass
class _DaciteConfig:
    strict: bool = False


_installed = False


def install() -> None:
    """Idempotent. Puts the stubs in sys.modules / sys.meta_path and the reference checkout on sys.path."""
    global _installed
    if _installed:
        return
    if not reference_available():
        raise RuntimeError(f"reference tree not found at LRAM_REFERENCE_ROOT={REFERENCE_ROOT!r}")
    repo_root = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    for p in (repo_root, REFERENCE_ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    sys.meta_path.insert(0, _Finder())

    import gym  # noqa: E402  (auto-stub created by the finder; now give it the functional bits)
    spaces = importlib.import_module("gym.spaces")
    for mod in (gym, spaces):
        mod.Box, mod.Discrete, mod.Space = Box, Discrete, _Space
    gym.spaces = spaces
    gym.Env = type("Env", (), {})

    pre = importlib.import_module("stable_baselines3.common.preprocessing")
    pre.is_image_space = _is_image_space
    pre.is_image_space_channels_first = lambda space: True
    pre.get_obs_shape = _get_obs_shape
    pre.get_action_dim = _get_action_dim
    tl = importlib.import_module("stable_baselines3.common.torch_layers")
    tl.BaseFeaturesExtractor = _BaseFeaturesExtractor
    vec = importlib.import_module("stable_baselines3.common.vec_env")
    vec.is_vecenv_wrapped = lambda env, cls: False

    oc = importlib.import_module("omegaconf")
    oc.OmegaConf = _OmegaConf
    dc = importlib.import_module("dacite")
    dc.from_dict, dc.Config = _from_dict, _DaciteConfig

    # the xlstm stand-in, laid out as the reference imports it (decision_xlstm.py:8-12,33)
    from oracle import xlstm_shim as S
    x = importlib.import_module("xlstm")
    x.xLSTMBlockStack, x.xLSTMBlockStackConfig = S.xLSTMBlockStack, S.xLSTMBlockStackConfig
    ln = importlib.import_module("xlstm.components.ln")
    ln.MultiHeadLayerNorm, ln.LayerNorm = S.MultiHeadLayerNorm, S.LayerNorm
    importlib.import_module("xlstm.components.linear_headwise").LinearHeadwiseExpand = S.LinearHeadwiseExpand
    importlib.import_module("xlstm.blocks.slstm.cell").sLSTMCell_cuda = S.sLSTMCell_cuda
    importlib.import_module("xlstm.blocks.mlstm.cell").mLSTMCell = S.mLSTMCell

    importlib.import_module("src.envs.target_returns").ALL_TARGETS = {}
    importlib.import_module("src.envs.env_names").ID_TO_DOMAIN = {}
    _installed = True


# ---- a deterministic VecEnv for the reference's rollout loop ------------------------------------------------------------
class ScriptedVecEnv:
    """One env (evaluation.py:80 asserts num_envs == 1) replaying a pre-generated observation stream; reward 1 per
    step, `done` after `ep_len` steps (then the returned observation is the next episode's reset observation, as SB3's
    VecEnv does). Mirrors `src/envs/dummy_env_utils.py:8-36` with a fixed stream instead of `space.sample()`."""

    num_envs = 1

    def __init__(self, observations: np.ndarray, action_space, observation_space, ep_len: int, name: str = "dummy",
                 reward: float = 1.0):
        self.obs = observations
        self.action_space, self.observation_space = action_space, observation_space
        self.ep_len, self.reward = ep_len, reward
        self.cursor, self.t = 0, 0
        self.envs = [types.SimpleNamespace(name=name)]
        self.actions_seen = []

    def env_is_wrapped(self, cls):
        return [False]

    def reset(self):
        o = self.obs[self.cursor]
        self.cursor += 1
        self.t = 0
        return o[None]

    def step(self, action):
        self.actions_seen.append(np.array(action).copy())
        self.t += 1
        done = self.t >= self.ep_len
        o = self.obs[self.cursor]
        self.cursor += 1
        if done:
            self.t = 0
        return o[None], np.array([self.reward], dtype=np.float32), np.array([done]), [{}]

    def render(self):
        return None
