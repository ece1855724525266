"""CPU-only stand-ins for the third-party packages the reference (liuzuxin/FSRL) imports and that are absent
here: ``tianshou`` (setup.py:16, ~=0.5.0), ``gymnasium``, ``bullet_safety_gym``, ``safety_gymnasium``, ``pyrallis``,
``h5py``.  Test / baseline infrastructure: ``install()`` lets ``import fsrl`` resolve to the UNMODIFIED reference
package (a checkout of it, or its install under ``oracle/_ref``) in a process that never
imports ``fsrl_b200`` -- so the reference arm of bench.py maps no product code.

Only what ``fsrl`` touches on the measured path is provided (SURVEY.md 2.3, Appendix C [UNVERIFIED restatements of
tianshou 0.5 semantics]): the ``Batch`` container, space classes, the MLP / ActorProb / Critic / Actor modules
(plain ``torch.nn``, oracle/shims/nets.py), ``RunningMeanStd``, noise classes and inert base classes for vector
envs and buffers.  The three dependency-free host modules shared with the product (``fsrl_b200/data/batch.py``,
``fsrl_b200/spaces.py``, ``fsrl_b200/utils/optim_util.py``: pure numpy/torch containers, no device code) are loaded
BY FILE PATH, which does not import the ``fsrl_b200`` package and therefore does not load libfsrl_b200.so."""
from __future__ import annotations

import importlib.util
import os
import sys
import types
from typing import List

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _load_file(name: str, rel: str):
    full = "oracle.shims._shared_" + name
    if full in sys.modules:
        return sys.modules[full]
    spec = importlib.util.spec_from_file_location(full, os.path.join(ROOT, rel))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[full] = mod
    spec.loader.exec_module(mod)
    return mod


def _mod(name: str, **attrs) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []
    sys.modules[name] = m
    return m


def _missing(name: str) -> bool:
    if name in sys.modules:
        return False
    try:
        return importlib.util.find_spec(name) is None
    except (ImportError, ValueError):
        return True


def install() -> List[str]:
    """Register the stand-ins for every absent package; returns the names that were installed."""
    import numpy as np
    import torch

    from . import nets as _nets
    batch = _load_file("batch", "fsrl_b200/data/batch.py")
    spaces = _load_file("spaces", "fsrl_b200/spaces.py")
    optim_util = _load_file("optim_util", "fsrl_b200/utils/optim_util.py")
    done = []
    if _missing("gymnasium"):
        class Env:                                          # type annotation target only (base_agent.py:39)
            pass

        def make(*a, **k):
            raise RuntimeError("gymnasium is absent: the CPU arm steps oracle/envs.py through oracle/subproc_env.py")
        sp = _mod("gymnasium.spaces", Box=spaces.Box, Discrete=spaces.Discrete, MultiBinary=spaces.MultiBinary,
                  MultiDiscrete=spaces.MultiDiscrete, Space=spaces.Space)
        _mod("gymnasium", make=make, Env=Env, Space=spaces.Space, spaces=sp)
        done.append("gymnasium")
    for name in ("bullet_safety_gym", "safety_gymnasium", "h5py"):
        if _missing(name):
            _mod(name)
            done.append(name)
    if _missing("pyrallis"):
        _mod("pyrallis", wrap=lambda *a, **k: (lambda fn: fn))
        done.append("pyrallis")
    if _missing("tianshou"):
        class BaseVectorEnv:
            pass

        class ReplayBuffer:
            pass

        class ReplayBufferManager(ReplayBuffer):
            pass

        class MovAvg:
            def __init__(self, size=100):
                self.size, self.cache = size, []

            def add(self, x):
                self.cache = (self.cache + list(np.atleast_1d(x)))[-self.size:]
                return self.get()

            def get(self):
                return float(np.mean(self.cache)) if self.cache else 0.0

        class DummyTqdm:
            def __init__(self, total, **kw):
                self.total, self.n = total, 0

            def set_postfix(self, **kw):
                pass

            def update(self, n=1):
                self.n += n

            def __enter__(self):
                return self

            def __exit__(self, *a):
                pass

        class BaseNoise:
            def reset(self):
                pass

        class GaussianNoise(BaseNoise):
            def __init__(self, mu: float = 0.0, sigma: float = 1.0):
                self._mu, self._sigma = mu, sigma

            def __call__(self, size):
                return np.random.normal(self._mu, self._sigma, size)

        def to_hdf5(*a, **k):
            raise NotImplementedError("HDF5 export needs h5py and tianshou, both absent")

        t_env = _mod("tianshou.env", BaseVectorEnv=BaseVectorEnv, DummyVectorEnv=BaseVectorEnv,
                     ShmemVectorEnv=BaseVectorEnv, SubprocVectorEnv=BaseVectorEnv)
        conv = _mod("tianshou.data.utils.converter", to_hdf5=to_hdf5)
        d_utils = _mod("tianshou.data.utils", converter=conv)
        t_data = _mod("tianshou.data", Batch=batch.Batch, ReplayBuffer=ReplayBuffer, ReplayBufferManager=ReplayBufferManager,
                      VectorReplayBuffer=ReplayBufferManager, to_numpy=batch.to_numpy, to_torch_as=batch.to_torch_as,
                      utils=d_utils)
        n_common = _mod("tianshou.utils.net.common", Net=_nets.Net, MLP=_nets.MLP)
        n_cont = _mod("tianshou.utils.net.continuous", ActorProb=_nets.ActorProb, Critic=_nets.Critic, Actor=_nets.Actor)
        t_net = _mod("tianshou.utils.net", common=n_common, continuous=n_cont)
        t_utils = _mod("tianshou.utils", RunningMeanStd=optim_util.RunningMeanStd, MovAvg=MovAvg, DummyTqdm=DummyTqdm,
                       MultipleLRSchedulers=object, tqdm_config={"dynamic_ncols": True, "ascii": True},
                       deprecation=lambda msg: None, net=t_net)
        t_expl = _mod("tianshou.exploration", BaseNoise=BaseNoise, GaussianNoise=GaussianNoise)
        _mod("tianshou", env=t_env, data=t_data, utils=t_utils, exploration=t_expl)
        done.append("tianshou")
    return done
