"""Run the UNMODIFIED reference policy classes on the CPU (test / baseline infrastructure).

The reference (liuzuxin/FSRL) is pure Python but imports ``tianshou`` and ``gymnasium``, which are
absent here (no network).  ``bootstrap(ref_dir)`` registers the repo's thin shims for exactly those
packages (attribute containers, spaces, plain ``torch.nn`` modules -- fsrl_b200.compat; no device
code is involved), puts ``ref_dir`` first on ``sys.path`` so that ``import fsrl`` IS the reference,
and adds the one missing tianshou method the learners call, ``Batch.split`` (restated in
oracle/ppo.py::split_indices, SURVEY.md 2.3 [UNVERIFIED]).

ref_dir is a checkout of the reference (golden-vector generation) or ``oracle/_ref``
(``refarm.install``: ``pip install --no-deps --target``) for ``bench.py --impl reference`` / ``cpu_baseline``.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_BOOTED = None


def bootstrap(ref_dir: str):
    """Returns the shim ``Batch`` class after making ``fsrl`` importable from ref_dir."""
    global _BOOTED
    if _BOOTED is not None:
        if _BOOTED[0] != os.path.abspath(ref_dir):
            raise RuntimeError(f"reference already loaded from {_BOOTED[0]}")
        return _BOOTED[1]
    ref_dir = os.path.abspath(ref_dir)
    if not os.path.isdir(os.path.join(ref_dir, "fsrl")):
        raise FileNotFoundError(f"no fsrl package under {ref_dir}")
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    sys.path.insert(0, ref_dir)           # `fsrl` must resolve to the reference, not to a shim
    import fsrl_b200.compat as compat
    done = compat.install()
    if "fsrl" in done:
        raise RuntimeError("the compat layer shadowed the reference package")
    import importlib.util
    import types
    for absent in ("h5py",):              # imported at module top by fsrl.data.traj_buf (offline-dataset export); unused here
        if absent not in sys.modules and importlib.util.find_spec(absent) is None:
            sys.modules[absent] = types.ModuleType(absent)
    if "tianshou.data.utils.converter" not in sys.modules:            # same module: HDF5 export helper, unused here
        def to_hdf5(*a, **k):
            raise NotImplementedError("HDF5 export needs h5py and tianshou, both absent")
        conv = types.ModuleType("tianshou.data.utils.converter"); conv.to_hdf5 = to_hdf5
        utils = types.ModuleType("tianshou.data.utils"); utils.converter = conv
        sys.modules["tianshou.data.utils"], sys.modules["tianshou.data.utils.converter"] = utils, conv
    import fsrl
    if not os.path.abspath(fsrl.__file__).startswith(ref_dir):
        raise RuntimeError(f"fsrl resolved to {fsrl.__file__}, expected {ref_dir}")
    from tianshou.data import Batch
    from oracle.ppo import split_indices

    def split(self, size, shuffle=True, merge_last=False):
        for idx in split_indices(len(self), size, shuffle=shuffle, merge_last=merge_last):
            yield self[idx]

    Batch.split = split
    _BOOTED = (ref_dir, Batch)
    return Batch


class Capture:
    """Stands in for fsrl.utils.BaseLogger: keeps every stored scalar in call order."""

    def __init__(self):
        self.rows = {}

    def store(self, tab=None, **kw):
        for k, v in kw.items():
            key = k if tab is None else f"{tab}/{k}"
            self.rows.setdefault(key, []).append(float(v))

    def print(self, *a, **k):
        pass

    def write(self, *a, **k):
        pass


class RingView:
    """What BasePolicy.compute_*_returns asks of a tianshou buffer, served from an OracleBuffer: the
    ring semantics (next / unfinished_index) are OUR restatement [tianshou absent]; everything the
    reference then does with them (masks, end flags, dtype flow, the numba kernels) is its own code."""

    def __init__(self, buf, Batch):
        from oracle import offpolicy as ooff
        self._b, self._next = buf, ooff.buffer_next
        self.terminated, self.truncated = buf.terminated, buf.truncated
        self.done = buf.terminated | buf.truncated
        self.rew = buf.rew.astype(np.float64)                 # tianshou stores rew as float64
        self.info = Batch(cost=buf.cost.astype(np.float64))

    def next(self, idx):
        return self._next(self._b, idx)

    def unfinished_index(self):
        return self._b.unfinished_index()


def box_spaces(D: int, A: int):
    from gymnasium.spaces import Box
    return (Box(low=-np.ones(A, np.float32), high=np.ones(A, np.float32)),
            Box(low=-np.ones(D, np.float32) * 10, high=np.ones(D, np.float32) * 10))


def independent_normal(*logits):
    return torch.distributions.Independent(torch.distributions.Normal(*logits), 1)


def ppo_lag_policy(D: int, A: int, hidden, lr: float = 5e-4, **kw):
    """The reference's PPOLagAgent recipe (fsrl/agent/ppo_lag_agent.py:128-200) with its own policy class:
    orthogonal init, log sigma = -0.5, one Adam over actor + critics."""
    from fsrl.policy.ppo_lag import PPOLagrangian
    from tianshou.utils.net.common import Net
    from tianshou.utils.net.continuous import ActorProb, Critic
    actor = ActorProb(Net(D, hidden_sizes=tuple(hidden)), A, max_action=1.0)
    critics = [Critic(Net(D, hidden_sizes=tuple(hidden))) for _ in range(2)]
    torch.nn.init.constant_(actor.sigma_param, -0.5)
    for m in list(actor.modules()) + [mm for c in critics for mm in c.modules()]:
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.orthogonal_(m.weight)
            torch.nn.init.zeros_(m.bias)
    optim = torch.optim.Adam([p for m in [actor] + critics for p in m.parameters()], lr=lr)
    act_space, obs_space = box_spaces(D, A)
    pol = PPOLagrangian(actor, critics, optim, independent_normal, logger=Capture(), observation_space=obs_space,
                        action_space=act_space, **kw)
    pol.train()
    return pol, actor, critics
