"""The CPU arm of bench.py (test / baseline infrastructure): the UNMODIFIED reference classes from ``oracle/_ref``
(``install()``: ``pip install --no-deps --target`` from a checkout of liuzuxin/FSRL) run the whole collect + update
cycle on the host cores --

* ``fsrl.data.FastCollector.collect`` (fast_collector.py:192-408) drives a vector env whose every env lives in its
  OWN worker process behind a pipe: tianshou's ``SubprocVectorEnv`` protocol (send the action to each worker, then
  wait for all of them), restated here because tianshou is absent.  The physics inside a worker is the numpy twin of
  the device env model (oracle/envs.py) -- pybullet / mujoco are absent too -- so the per-step IPC, Python and Batch
  overhead of the reference path are real, the simulator cost is a lower bound;
* ``fsrl.policy.PPOLagrangian.process_fn`` / ``learn`` (ppo_lag.py:134-257: numba GAE, eager autograd, Adam).

Nothing here imports ``fsrl_b200``: the third-party packages the reference needs come from oracle/shims."""
from __future__ import annotations

import multiprocessing as mp
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
# the checkout of liuzuxin/FSRL the install is made from; FSRL_REFERENCE names another one
REF_SRC = os.environ.get("FSRL_REFERENCE", "/root/reference")
_REF = None


def install(src: str = REF_SRC, dst: str = REF_DIR) -> None:
    """Install the reference package from the checkout ``src`` into ``dst`` unless it is there already or ``src``
    holds no checkout.  No dependencies are installed: ``bootstrap`` supplies the third-party packages from
    oracle/shims.  pip writes build files beside the sources, so it builds from a copy and ``src`` may be read-only."""
    if os.path.isdir(os.path.join(dst, "fsrl")) or not os.path.isdir(os.path.join(src, "fsrl")):
        return
    with tempfile.TemporaryDirectory() as tmp:
        work = os.path.join(tmp, "reference")
        shutil.copytree(src, work, ignore=shutil.ignore_patterns(".git"), copy_function=shutil.copyfile)
        for d, _, _ in os.walk(work):
            os.chmod(d, 0o755)                  # copytree keeps the directories' modes, and pip writes into them
        subprocess.check_call([sys.executable, "-m", "pip", "install", "--quiet", "--no-index", "--no-build-isolation",
                               "--no-deps", "--no-cache-dir", "--target", dst, work])


def bootstrap(ref_dir: str):
    """Make ``import fsrl`` resolve to the reference under ref_dir; returns the shim Batch class."""
    global _REF
    ref_dir = os.path.abspath(ref_dir)
    if _REF is not None:
        if _REF[0] != ref_dir:
            raise RuntimeError("reference already loaded from " + _REF[0])
        return _REF[1]
    if not os.path.isdir(os.path.join(ref_dir, "fsrl")):
        raise FileNotFoundError("no fsrl package under " + ref_dir)
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from oracle import shims
    shims.install()
    sys.path.insert(0, ref_dir)
    import fsrl
    if not os.path.abspath(fsrl.__file__).startswith(ref_dir):
        raise RuntimeError("fsrl resolved to %s, expected %s" % (fsrl.__file__, ref_dir))
    from tianshou.data import Batch
    from oracle.ppo import split_indices

    def split(self, size, shuffle=True, merge_last=False):          # tianshou Batch.split (SURVEY 2.3 [UNVERIFIED])
        for idx in split_indices(len(self), size, shuffle=shuffle, merge_last=merge_last):
            yield self[idx]

    Batch.split = split
    _REF = (ref_dir, Batch)
    return Batch


# ---- one env per worker process --------------------------------------------------------------------------
def _worker(conn, kind, n_env, index, seed):
    from oracle.envs import OracleVecEnv
    torch.set_num_threads(1)
    env = OracleVecEnv(kind, n_env, seed)            # env `index` of the vector: same RNG streams as the in-process twin
    ids = np.array([index])
    try:
        while True:
            cmd, data = conn.recv()
            if cmd == "step":
                conn.send(env.step(np.asarray(data, np.float32)[None], ids))
            elif cmd == "reset":
                conn.send(env.reset(ids))
            else:
                break
    except (EOFError, KeyboardInterrupt):
        pass
    conn.close()


class SubprocVecEnv:
    """``len``, ``action_space`` per env, ``reset(ids) -> (obs, info)``, ``step(action, id) -> 5-tuple`` with
    ``info["cost"]`` -- what FastCollector asks of a tianshou vector env (fast_collector.py:134,172,259-262,286-303)."""

    def __init__(self, kind, n_env: int, seed: int, workers: bool = True):
        from gymnasium.spaces import Box
        from oracle.envs import DIMS, KINDS, OracleVecEnv
        k = KINDS[kind] if isinstance(kind, str) else int(kind)
        self.D, self.A, _, self.T = DIMS[k]
        self.E = n_env
        self.action_space = [Box(low=-np.ones(self.A, np.float32), high=np.ones(self.A, np.float32))] * n_env
        self.workers = workers
        if workers:
            ctx = mp.get_context("fork")
            self.conns, self.procs = [], []
            for i in range(n_env):
                parent, child = ctx.Pipe()
                p = ctx.Process(target=_worker, args=(child, k, n_env, i, seed), daemon=True)
                p.start()
                child.close()
                self.conns.append(parent); self.procs.append(p)
        else:
            self.e = OracleVecEnv(k, n_env, seed)

    def __len__(self):
        return self.E

    def reset(self, ids=None, **kw):
        ids = np.arange(self.E) if ids is None else np.asarray(ids)
        if self.workers:
            for i in ids:
                self.conns[i].send(("reset", None))
            obs = np.concatenate([self.conns[i].recv() for i in ids], axis=0)
        else:
            obs = self.e.reset(ids)
        return obs, {"cost": np.zeros(len(obs))}

    def step(self, action, id=None):
        ids = np.arange(self.E) if id is None else np.asarray(id)
        action = np.asarray(action, np.float32)
        if self.workers:
            for k, i in enumerate(ids):
                self.conns[i].send(("step", action[k]))
            parts = [self.conns[i].recv() for i in ids]
            obs_next, rew, cost, term, trunc = (np.concatenate([p[q] for p in parts], axis=0) for q in range(5))
        else:
            obs_next, rew, cost, term, trunc = self.e.step(action, ids)
        trunc = trunc & ~term
        return obs_next, rew.astype(np.float64), term, trunc, {"cost": cost.astype(np.float64)}

    def close(self):
        if self.workers:
            for c in self.conns:
                try:
                    c.send(("close", None))
                except (BrokenPipeError, OSError):
                    pass
            for p in self.procs:
                p.join(timeout=2)


def make_buffer(total, n_env, D, A):
    """Ring storage FastCollector.collect writes into (``buffer.add(batch, buffer_ids)`` -> ptr, ep_rew, ep_len, ep_idx):
    tianshou's VectorReplayBuffer restated over oracle/collector.OracleBuffer [tianshou absent]."""
    from tianshou.data import ReplayBufferManager
    from oracle.collector import OracleBuffer

    class RecBuffer(ReplayBufferManager):
        def __init__(self):
            self.b = OracleBuffer(total, n_env, D, A)
            self.buffer_num, self.maxsize = n_env, total
            self.run_rew, self.run_len = np.zeros(n_env), np.zeros(n_env, np.int64)

        def reset(self, keep_statistics=False):
            self.b.reset()

        def add(self, batch, buffer_ids=None):
            ids = np.asarray(buffer_ids)
            ptr = ids * self.b.cap + self.b.ptr[ids]
            self.b.add(ids, batch.obs, batch.act, batch.rew.astype(np.float32), np.asarray(batch.cost, np.float32),
                       np.zeros(len(ids), np.float32), batch.terminated, batch.truncated, batch.obs_next)
            self.run_rew[ids] += batch.rew; self.run_len[ids] += 1
            done = np.asarray(batch.done, bool)
            ep_rew = np.where(done, self.run_rew[ids], 0.0); ep_len = np.where(done, self.run_len[ids], 0)
            fin = ids[done]
            self.run_rew[fin] = 0; self.run_len[fin] = 0
            return ptr, ep_rew, ep_len, ptr

    return RecBuffer()


class _Capture:
    def store(self, tab=None, **kw):
        pass

    def print(self, *a, **k):
        pass

    def write(self, *a, **k):
        pass


class _RingView:
    """What BasePolicy.compute_gae_returns asks of the buffer (next / unfinished_index / rew / info)."""

    def __init__(self, buf, Batch):
        from oracle import offpolicy as ooff
        self._b, self._next = buf, ooff.buffer_next
        self.terminated, self.truncated = buf.terminated, buf.truncated
        self.done = buf.terminated | buf.truncated
        self.rew = buf.rew.astype(np.float64)
        self.info = Batch(cost=buf.cost.astype(np.float64))

    def next(self, idx):
        return self._next(self._b, idx)

    def unfinished_index(self):
        return self._b.unfinished_index()


def ppo_lag_cycle_runner(ref_dir, task_kind, n_env, hidden, batch_size, repeat, threads, workers=True, seed=10, lr=5e-4):
    """Build the reference's PPO-Lagrangian stack (ppo_lag_agent.py:128-200 recipe) and return ``cycle()``: one
    collect (n_env episodes) + process_fn + learn, returning (env steps, collect seconds, update seconds)."""
    Batch = bootstrap(ref_dir)
    from fsrl.data import FastCollector
    from fsrl.policy.ppo_lag import PPOLagrangian
    from gymnasium.spaces import Box
    from tianshou.utils.net.common import Net
    from tianshou.utils.net.continuous import ActorProb, Critic
    torch.set_num_threads(threads)
    torch.manual_seed(seed); np.random.seed(seed)
    env = SubprocVecEnv(task_kind, n_env, seed, workers=workers)
    D, A, T = env.D, env.A, env.T
    actor = ActorProb(Net(D, hidden_sizes=tuple(hidden)), A, max_action=1.0)
    critics = [Critic(Net(D, hidden_sizes=tuple(hidden))) for _ in range(2)]
    torch.nn.init.constant_(actor.sigma_param, -0.5)
    for m in list(actor.modules()) + [mm for c in critics for mm in c.modules()]:
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.orthogonal_(m.weight)
            torch.nn.init.zeros_(m.bias)
    optim = torch.optim.Adam([p for m in [actor] + critics for p in m.parameters()], lr=lr)
    dist = lambda *logits: torch.distributions.Independent(torch.distributions.Normal(*logits), 1)
    pol = PPOLagrangian(actor, critics, optim, dist, logger=_Capture(), target_kl=float("inf"), max_grad_norm=0.5,
                        cost_limit=10.0, gamma=0.99,
                        observation_space=Box(low=-np.ones(D, np.float32) * 10, high=np.ones(D, np.float32) * 10),
                        action_space=env.action_space[0])
    pol.train()
    buf = make_buffer(n_env * T, n_env, D, A)
    col = FastCollector(pol, env, buf, exploration_noise=True)

    def cycle():
        t0 = time.time()
        col.reset_buffer()
        st = col.collect(n_episode=n_env)
        t1 = time.time()
        pol.pre_update_fn(stats_train=st)
        b = buf.b
        idx = b.sample_all()
        view = _RingView(b, Batch)
        batch = Batch(obs=torch.from_numpy(b.obs[idx]), obs_next=torch.from_numpy(b.obs_next[idx]),
                      act=torch.from_numpy(b.act[idx]), rew=view.rew[idx], terminated=b.terminated[idx],
                      truncated=b.truncated[idx], info=Batch(cost=b.cost[idx].astype(np.float64)))
        batch = pol.process_fn(batch, view, idx)
        pol.learn(batch, batch_size, repeat)
        t2 = time.time()
        return int(st["n/st"]), t1 - t0, t2 - t1

    cycle.close = env.close
    cycle.T = T
    return cycle
