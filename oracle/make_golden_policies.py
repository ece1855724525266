"""Golden vectors for the UPDATE paths, produced by the reference's OWN policy classes.

Run in the build container only (needs /root/reference; never on the GPU box):

    python oracle/make_golden_policies.py

The reference (fsrl.policy.*) cannot normally be imported here: tianshou / gymnasium are absent.
This script registers the repo's thin shims for exactly those two packages (fsrl_b200.compat --
attribute containers, spaces, plain torch.nn modules; none of the device code is involved), puts
/root/reference on sys.path so that ``fsrl`` IS the reference, and then drives the reference's
``learn()`` on CPU with torch autograd + torch.optim.Adam on small seeded batches.  What it
records -- inputs, initial weights, the per-minibatch statistics the reference logs and the final
weights -- pins ``oracle/{ppo,cpo,trpo,focops}.py`` (tests/test_oracle_golden.py replays them on
CPU); the CUDA path is then compared with the oracle in the -m gpu tests.

The only non-reference ingredient is ``Batch.split`` (tianshou 0.5.0 source is absent): it is the
restatement in oracle/ppo.py::split_indices [SURVEY.md 2.3, UNVERIFIED] -- permutation order is
therefore shared by construction, the arithmetic of every update step is the reference's.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")

D, A, H, N, BS, REPEAT = 8, 2, 16, 200, 64, 2


def _bootstrap():
    sys.path.insert(0, ROOT)
    from oracle import refrun
    return refrun.bootstrap(REF)


def _Capture():
    from oracle import refrun
    return refrun.Capture()


def _nets(seed):
    from tianshou.utils.net.common import Net
    from tianshou.utils.net.continuous import ActorProb, Critic
    torch.manual_seed(seed)
    actor = ActorProb(Net(D, hidden_sizes=(H, H)), A, max_action=1.0)
    critics = [Critic(Net(D, hidden_sizes=(H, H))) for _ in range(2)]
    torch.nn.init.constant_(actor.sigma_param, -0.5)
    for m in list(actor.modules()) + [mm for c in critics for mm in c.modules()]:
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.orthogonal_(m.weight)
            torch.nn.init.zeros_(m.bias)
    return actor, critics


def _data(seed, actor):
    rng = np.random.default_rng(seed)
    obs = rng.normal(size=(N, D)).astype(np.float32)
    with torch.no_grad():
        (mu, sigma), _ = actor(torch.from_numpy(obs))
        act = (mu + sigma * torch.from_numpy(rng.normal(size=(N, A)).astype(np.float32)))
        # the behaviour policy is a slightly older one: shift the stored log-prob a little
        logp = torch.distributions.Independent(torch.distributions.Normal(mu, sigma), 1).log_prob(act)
        logp = logp + torch.from_numpy(rng.normal(scale=0.05, size=N).astype(np.float32))
    advs = rng.normal(size=(N, 2)).astype(np.float32) * np.array([1.0, 0.5], np.float32)
    rets = rng.normal(size=(N, 2)).astype(np.float32)
    values = rets + rng.normal(scale=0.3, size=(N, 2)).astype(np.float32)
    mean_old = (mu + 0.02 * torch.from_numpy(rng.normal(size=(N, A)).astype(np.float32))).numpy()
    std_old = (sigma * 1.03).numpy()
    return dict(obs=obs, act=act.numpy(), logp_old=logp.numpy(), advs=advs, rets=rets, values=values,
                mean_old=mean_old, std_old=std_old)


def _batch(Batch, d):
    t = lambda k: torch.from_numpy(d[k].copy())
    return Batch(obs=t("obs"), act=t("act"), logp_old=t("logp_old"), advs=t("advs"), rets=t("rets"),
                 values=t("values"), mean_old=t("mean_old"), std_old=t("std_old"), info=Batch())


def _state(mods):
    out = {}
    for name, m in mods:
        for k, v in m.state_dict().items():
            out[f"{name}.{k}"] = v.detach().numpy().copy()
    return out


def _space():
    from gymnasium.spaces import Box
    return Box(low=-np.ones(A, np.float32), high=np.ones(A, np.float32)), Box(low=-np.ones(D, np.float32) * 10, high=np.ones(D, np.float32) * 10)


def _dist(*logits):
    return torch.distributions.Independent(torch.distributions.Normal(*logits), 1)


def golden_ppo(Batch):
    from fsrl.policy.ppo_lag import PPOLagrangian
    cases = {}
    for name, kw, lag in (("base", dict(), 0.7), ("dualclip_vclip", dict(dual_clip=3.0, value_clip=True, reward_normalization=True), 0.3),
                          ("nolag", dict(use_lagrangian=False), 0.0)):
        actor, critics = _nets(3)
        d = _data(11, actor)
        init = _state([("actor", actor)] + [(f"critics.{i}", c) for i, c in enumerate(critics)])
        params = [p for m in [actor] + critics for p in m.parameters()]
        optim = torch.optim.Adam(params, lr=5e-4)
        act_space, obs_space = _space()
        log = _Capture()
        pol = PPOLagrangian(actor, critics, optim, _dist, logger=log, target_kl=1e9, max_grad_norm=0.5,
                            cost_limit=10.0, observation_space=obs_space, action_space=act_space, **kw)
        if pol.use_lagrangian:
            pol.lag_optims[0].lagrangian = lag
        pol.train()
        np.random.seed(21)
        torch.manual_seed(5)
        pol.learn(_batch(Batch, d), BS, REPEAT)
        final = _state([("actor", actor)] + [(f"critics.{i}", c) for i, c in enumerate(critics)])
        cases[name] = dict(kw=kw, lag=lag, data=d, init=init, final=final, stats=log.rows)
    return cases


def _crit_optim(critics, lr):
    return torch.optim.Adam([p for c in critics for p in c.parameters()], lr=lr)


def _mods(actor, critics):
    return [("actor", actor)] + [(f"critics.{i}", c) for i, c in enumerate(critics)]


def golden_cpo(Batch):
    """cpo.py:353-370 on one full batch: cost_limit / ave_cost pairs that reach different dual cases."""
    from fsrl.policy.cpo import CPO
    cases = {}
    for name, cost_limit, ave_cost in (("feasible", 1000.0, 12.0), ("infeasible", 0.0, 35.0), ("case2", 10.0, 9.99),
                                       ("case1_then_2", 10.0, 10.05), ("case0_then_1", 10.0, 10.1)):
        actor, critics = _nets(4)
        d = _data(12, actor)
        for i in range(2):                       # process_fn standardises the advantages (:127-131)
            a = d["advs"][:, i]
            d["advs"][:, i] = (a - a.mean()) / a.std(ddof=1)
        init = _state(_mods(actor, critics))
        act_space, obs_space = _space()
        log = _Capture()
        pol = CPO(actor, critics, _crit_optim(critics, 1e-3), _dist, logger=log, target_kl=0.01, max_backtracks=10,
                  optim_critic_iters=3, l2_reg=0.001, cost_limit=cost_limit, observation_space=obs_space,
                  action_space=act_space)
        pol.pre_update_fn(stats_train={"cost": ave_cost})
        pol.train()
        np.random.seed(22)
        torch.manual_seed(6)
        pol.learn(_batch(Batch, d), 99999, 2)
        cases[name] = dict(kw=dict(cost_limit=cost_limit, ave_cost=ave_cost), lag=0.0, data=d, init=init,
                           final=_state(_mods(actor, critics)), stats=log.rows,
                           extra=dict(cost_limit=cost_limit, ave_cost=ave_cost))
    return cases


def golden_trpo(Batch):
    from fsrl.policy.trpo_lag import TRPOLagrangian
    cases = {}
    for name, lag in (("lag06", 0.6), ("lag0", 0.0)):
        actor, critics = _nets(5)
        d = _data(13, actor)
        for i in range(2):
            a = d["advs"][:, i]
            d["advs"][:, i] = (a - a.mean()) / a.std(ddof=1)
        init = _state(_mods(actor, critics))
        act_space, obs_space = _space()
        log = _Capture()
        pol = TRPOLagrangian(actor, critics, _crit_optim(critics, 5e-4), _dist, logger=log, target_kl=0.001,
                             optim_critic_iters=3, cost_limit=10.0, observation_space=obs_space,
                             action_space=act_space)
        pol.lag_optims[0].lagrangian = lag
        pol.train()
        np.random.seed(23)
        torch.manual_seed(7)
        pol.learn(_batch(Batch, d), 99999, 2)
        cases[name] = dict(kw={}, lag=lag, data=d, init=init, final=_state(_mods(actor, critics)), stats=log.rows)
    return cases


def golden_focops(Batch):
    from fsrl.policy.focops import FOCOPS
    cases = {}
    for name, eta, ave_cost in (("eta02", 0.02, 31.5), ("eta_tiny", 1e-4, 4.0)):
        actor, critics = _nets(6)
        d = _data(14, actor)
        init = _state(_mods(actor, critics))
        act_space, obs_space = _space()
        log = _Capture()
        nu = (2.0, 1e-2, torch.zeros(1))
        pol = FOCOPS(actor, critics, torch.optim.Adam(actor.parameters(), lr=5e-4), _crit_optim(critics, 1e-3), _dist,
                     logger=log, cost_limit=10.0, nu=nu, l2_reg=1e-3, delta=1e9, eta=eta, tem_lambda=0.95,
                     max_grad_norm=0.5, observation_space=obs_space, action_space=act_space)
        pol.pre_update_fn(stats_train={"cost": ave_cost})
        pol.train()
        np.random.seed(24)
        torch.manual_seed(8)
        pol.learn(_batch(Batch, d), BS, REPEAT)
        cases[name] = dict(kw={}, lag=0.0, data=d, init=init, final=_state(_mods(actor, critics)), stats=log.rows,
                           extra=dict(eta=eta, ave_cost=ave_cost))
    return cases


class _NoiseTape:
    """Records every standard-normal draw torch.distributions makes (Normal.rsample), so that the
    oracle replay injects exactly the reference's reparameterisation noise."""

    def __init__(self):
        import torch.distributions.normal as tn
        self._tn, self._orig, self.draws = tn, tn._standard_normal, []

    def __enter__(self):
        def tapped(shape, dtype, device):
            e = self._orig(shape, dtype=dtype, device=device)
            self.draws.append(e.detach().numpy().copy())
            return e
        self._tn._standard_normal = tapped
        return self

    def __exit__(self, *a):
        self._tn._standard_normal = self._orig


def _q_nets(seed, double):
    from tianshou.utils.net.common import Net
    from tianshou.utils.net.continuous import Actor, ActorProb, Critic
    from fsrl.utils.net.continuous import DoubleCritic
    torch.manual_seed(seed)
    if double:
        actor = ActorProb(Net(D, hidden_sizes=(H, H)), A, max_action=1.0, unbounded=True, conditioned_sigma=True)
        critics = [DoubleCritic(Net(D, A, hidden_sizes=(H, H), concat=True), Net(D, A, hidden_sizes=(H, H), concat=True))
                   for _ in range(2)]
    else:
        actor = Actor(Net(D, hidden_sizes=(H, H)), A, max_action=1.0)
        critics = [Critic(Net(D, A, hidden_sizes=(H, H), concat=True)) for _ in range(2)]
    for m in list(actor.modules()) + [mm for c in critics for mm in c.modules()]:
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.orthogonal_(m.weight)
            torch.nn.init.zeros_(m.bias)
    return actor, critics


def _off_data(seed):
    rng = np.random.default_rng(seed)
    return dict(obs=rng.normal(size=(BS, D)).astype(np.float32),
                act=np.tanh(rng.normal(size=(BS, A))).astype(np.float32),
                rets=rng.normal(size=(BS, 2)).astype(np.float32) * np.array([2.0, 1.0], np.float32))


def golden_sac(Batch):
    """sac_lag.py:185-269: three consecutive learn() calls on given n-step targets (`rets`)."""
    from fsrl.policy.sac_lag import SACLagrangian
    cases = {}
    for name, auto_alpha, lag in (("auto_alpha", True, 0.8), ("fixed_alpha", False, 0.0)):
        actor, critics = _q_nets(7, True)
        init = _state(_mods(actor, critics))
        if auto_alpha:
            log_alpha = torch.zeros(1, requires_grad=True)
            alpha = (-float(A), log_alpha, torch.optim.Adam([log_alpha], lr=3e-4))
        else:
            alpha = 0.2
        act_space, obs_space = _space()
        log = _Capture()
        pol = SACLagrangian(actor, critics, torch.optim.Adam(actor.parameters(), lr=5e-4),
                            torch.optim.Adam(torch.nn.ModuleList(critics).parameters(), lr=1e-3), logger=log,
                            alpha=alpha, tau=0.05, gamma=0.97, n_step=2, cost_limit=10.0,
                            observation_space=obs_space, action_space=act_space)
        pol.lag_optims[0].lagrangian = lag
        pol.train()
        torch.manual_seed(9)
        data, eps = {}, []
        for k in range(3):
            d = _off_data(30 + k)
            with _NoiseTape() as tape:
                pol.learn(Batch(obs=torch.from_numpy(d["obs"]), act=torch.from_numpy(d["act"]),
                                rets=torch.from_numpy(d["rets"]), info=Batch()))
            assert len(tape.draws) == 1
            for kk, v in d.items():
                data[f"{kk}{k}"] = v
            data[f"eps{k}"] = tape.draws[0]
        final = _state(_mods(actor, critics) + [(f"critics_old.{i}", c) for i, c in enumerate(pol.critics_old)])
        cases[name] = dict(kw={}, lag=lag, data=data, init=init, final=final, stats=log.rows,
                           extra=dict(auto_alpha=float(auto_alpha)))
    return cases


def golden_ddpg(Batch):
    """ddpg_lag.py:165-223: three consecutive learn() calls on given n-step targets."""
    from fsrl.policy.ddpg_lag import DDPGLagrangian
    cases = {}
    for name, lag in (("lag05", 0.5), ("lag0", 0.0)):
        actor, critics = _q_nets(8, False)
        init = _state(_mods(actor, critics))
        act_space, obs_space = _space()
        log = _Capture()
        pol = DDPGLagrangian(actor, critics, torch.optim.Adam(actor.parameters(), lr=5e-4),
                             torch.optim.Adam(torch.nn.ModuleList(critics).parameters(), lr=1e-3), logger=log,
                             tau=0.05, gamma=0.97, n_step=2, cost_limit=10.0, observation_space=obs_space,
                             action_space=act_space)
        pol.lag_optims[0].lagrangian = lag
        pol.train()
        data = {}
        for k in range(3):
            d = _off_data(40 + k)
            pol.learn(Batch(obs=torch.from_numpy(d["obs"]), act=torch.from_numpy(d["act"]),
                            rets=torch.from_numpy(d["rets"]), info=Batch()))
            for kk, v in d.items():
                data[f"{kk}{k}"] = v
        final = _state(_mods(actor, critics) + [("actor_old", pol.actor_old)] +
                       [(f"critics_old.{i}", c) for i, c in enumerate(pol.critics_old)])
        cases[name] = dict(kw={}, lag=lag, data=data, init=init, final=final, stats=log.rows)
    return cases


def _RingView(buf, Batch):
    from oracle import refrun
    return refrun.RingView(buf, Batch)


def _ring(seed, E=3, T=40, p_term=0.08):
    from oracle.collector import OracleBuffer
    rng = np.random.default_rng(seed)
    buf = OracleBuffer(E * T, E, D, A)
    lens = [T, T - 7, T - 15]                                # ragged: two envs stop mid-episode (unfinished)
    for t in range(T):
        ids = np.array([e for e in range(E) if t < lens[e]])
        n = len(ids)
        trunc = np.array([(t + 1) % 13 == 0 for _ in ids])
        buf.add(ids, rng.normal(size=(n, D)).astype(np.float32), np.tanh(rng.normal(size=(n, A))).astype(np.float32),
                rng.normal(0.5, 1.0, size=n).astype(np.float32), (rng.random(n) < 0.1).astype(np.float32),
                np.zeros(n, np.float32), rng.random(n) < p_term, trunc, rng.normal(size=(n, D)).astype(np.float32))
    return buf


def golden_returns_glue(Batch):
    """base_policy.py:384-451 (compute_gae_returns, with and without reward normalisation) and :453-512
    (compute_nstep_returns) executed by the reference on a ragged 3-env ring."""
    from fsrl.policy.ppo_lag import PPOLagrangian
    cases = {}
    buf = _ring(50)
    view = _RingView(buf, Batch)
    idx = buf.sample_all()
    ring = dict(obs=buf.obs, obs_next=buf.obs_next, act=buf.act, rew=buf.rew, cost=buf.cost,
                terminated=buf.terminated, truncated=buf.truncated, ptr=buf.ptr, len=buf.len, idx=idx)
    for name, rew_norm in (("gae", False), ("gae_rew_norm", True)):
        actor, critics = _nets(9)
        init = _state(_mods(actor, critics))
        act_space, obs_space = _space()
        pol = PPOLagrangian(actor, critics, torch.optim.Adam(actor.parameters()), _dist, logger=_Capture(),
                            reward_normalization=rew_norm, gamma=0.99, observation_space=obs_space,
                            action_space=act_space)
        out = {}
        for call in range(2):                                 # the second call sees the updated running std
            batch = Batch(obs=torch.from_numpy(buf.obs[idx]), obs_next=torch.from_numpy(buf.obs_next[idx]),
                          rew=view.rew[idx], terminated=buf.terminated[idx], truncated=buf.truncated[idx],
                          info=Batch(cost=buf.cost[idx].astype(np.float64)))
            batch = pol.compute_gae_returns(batch, view, idx, 0.95)
            out[f"values{call}"] = batch.values.numpy(); out[f"rets{call}"] = batch.rets.numpy()
            out[f"advs{call}"] = batch.advs.numpy()
            out[f"rms_var{call}"] = np.array([float(r.var) for r in pol.ret_rms])
        cases[name] = dict(kw={}, lag=0.0, data=ring, init=init, final=out, stats={})
    # n-step targets with a fixed target-Q function
    rng = np.random.default_rng(51)
    actor, critics = _nets(9)
    act_space, obs_space = _space()
    pol = PPOLagrangian(actor, critics, torch.optim.Adam(actor.parameters()), _dist, logger=_Capture(), gamma=0.97,
                        observation_space=obs_space, action_space=act_space)
    sel = rng.choice(idx, size=48).astype(np.int64)
    out = {"sel": sel}
    for n_step in (1, 2, 3, 5):
        tq = [rng.normal(size=(48, 1)).astype(np.float32) for _ in range(2)]
        b = pol.compute_nstep_returns(Batch(), view, sel, lambda _buf, _term: [torch.from_numpy(t) for t in tq], n_step)
        out[f"tq{n_step}"] = np.stack([t[:, 0] for t in tq])
        out[f"rets{n_step}"] = b.rets.numpy()
    cases["nstep"] = dict(kw={}, lag=0.0, data=ring, init={}, final=out, stats={})
    return cases


def golden_trainers():
    """fsrl/trainer/{base_trainer,onpolicy,offpolicy}.py + fsrl.utils.BaseLogger driven by scripted fakes."""
    import json
    from fsrl.trainer import OffpolicyTrainer, OnpolicyTrainer
    from fsrl.utils import BaseLogger
    from oracle import trainer_scenario
    rec = trainer_scenario.run(OnpolicyTrainer, OffpolicyTrainer, BaseLogger)
    import tempfile
    from fsrl.utils.exp_util import load_config_and_model
    with tempfile.TemporaryDirectory() as tmp:
        rec["logger_files"] = trainer_scenario.logger_files(BaseLogger, tmp)
    # cross-read: a run directory written by fsrl_b200's logger must load with the REFERENCE's loader
    from fsrl_b200.utils.logger import BaseLogger as OurLogger
    with tempfile.TemporaryDirectory() as tmp:
        trainer_scenario.logger_files(OurLogger, tmp)
        cfg, model = load_config_and_model(os.path.join(tmp, "run"))
        assert cfg["task"] == "SafetyCarCircle-v0" and tuple(cfg["hidden_sizes"]) == (128, 128) and "model" in model
        cfg_b, model_b = load_config_and_model(os.path.join(tmp, "run"), best=True)
        assert torch.equal(model_b["model"]["w"], torch.arange(3.0))
    path = os.path.join(OUT, "trainer_golden.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
    print("wrote", path, {k: (len(v["trace"]), len(v["epochs"])) for k, v in rec.items() if "trace" in v})


def golden_configs_and_names():
    """fsrl/config/*_cfg.py defaults (every TrainCfg / Bullet* / Mujoco* dataclass) and
    fsrl.utils.exp_util.{to_string, auto_name} on a handful of inputs."""
    import importlib
    import json
    from dataclasses import asdict
    from fsrl.utils.exp_util import auto_name, to_string
    rec = {"configs": {}, "to_string": [], "auto_name": []}
    for key in ("ppol", "cpo", "sacl", "ddpgl", "trpol", "focosp"):
        mod = importlib.import_module(f"fsrl.config.{key}_cfg")
        for cls in ("TrainCfg", "Bullet1MCfg", "Bullet5MCfg", "Bullet10MCfg", "MujocoBaseCfg", "Mujoco2MCfg",
                    "Mujoco10MCfg", "Mujoco20MCfg"):
            d = asdict(getattr(mod, cls)())
            rec["configs"][f"{key}.{cls}"] = {k: (list(v) if isinstance(v, tuple) else v) for k, v in d.items()}
    for v in (3, 2.5, 1e-4, 0.00037, 123456.789, True, None, "abc", [1, 2.5, "x"], (64, 64), {"a": 1, "b": [2, 3]}, 1e9, 10):
        rec["to_string"].append([repr(v), to_string(v)])
    base = asdict(importlib.import_module("fsrl.config.ppol_cfg").TrainCfg())
    for changes, prefix, suffix, skip in (({}, "ppol", "", []), ({"lr": 1e-3, "seed": 5}, "ppol", "", []),
                                          ({"hidden_sizes": (256, 256), "cost_limit": 25, "task": "SafetyAntCircle-v0"}, "x", "s1", []),
                                          ({"gamma": 0.995, "unbounded": True}, "", "end", ["gamma"])):
        cur = dict(base); cur.update(changes)
        rec["auto_name"].append({"changes": {k: (list(v) if isinstance(v, tuple) else v) for k, v in changes.items()},
                                 "prefix": prefix, "suffix": suffix, "skip": skip,
                                 # the last 5 characters are a random "-uuid4[:4]" tag
                                 "name": (auto_name(base, cur, prefix, suffix, skip_keys=skip) if skip
                                          else auto_name(base, cur, prefix, suffix))[:-5]})
    path = os.path.join(OUT, "config_names_golden.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
    print("wrote", path, len(rec["configs"]), "config classes")


def golden_action_maps():
    """BasePolicy.map_action / map_action_inverse (base_policy.py:226-283) of the reference on sample actions."""
    import json
    from fsrl.policy.ppo_lag import PPOLagrangian
    from gymnasium.spaces import Box
    rng = np.random.default_rng(60)
    acts = (rng.normal(scale=1.5, size=(6, 3))).astype(np.float32)
    lows, highs = np.array([-2.0, 0.0, -1.0], np.float32), np.array([2.0, 0.0, 3.0], np.float32)   # one degenerate dim
    rec = {"act": acts.tolist(), "low": lows.tolist(), "high": highs.tolist(), "cases": []}
    for method in ("clip", "tanh", ""):
        for scaling in (True, False):
            actor, critics = _nets(2)
            pol = PPOLagrangian(actor, critics, torch.optim.Adam(actor.parameters()), _dist, logger=_Capture(),
                                action_scaling=scaling, action_bound_method=method,
                                observation_space=_space()[1], action_space=Box(low=lows.copy(), high=highs.copy()))
            src = np.clip(acts, -1, 1) if (method == "" and scaling) else acts
            fwd = pol.map_action(src.copy())
            env_acts = (lows + (highs - lows) * rng.random(size=(6, 3))).astype(np.float32)
            inv = pol.map_action_inverse(env_acts.copy())
            rec["cases"].append({"method": method, "scaling": scaling, "src": src.tolist(),
                                 "mapped": np.asarray(fwd, np.float64).tolist(), "env_acts": env_acts.tolist(),
                                 "inverse": np.nan_to_num(np.asarray(inv, np.float64), nan=1e30, posinf=1e30, neginf=-1e30).tolist()})
    path = os.path.join(OUT, "action_map_golden.json")
    with open(path, "w") as f:
        json.dump(rec, f)
    print("wrote", path, len(rec["cases"]), "cases")


def golden_collector():
    """fsrl/data/fast_collector.py:192-408 executed by the reference: its FastCollector drives a numpy twin of
    our env model through a minimal vector-env facade and a recording buffer (deterministic eval-mode
    policy), for several (env count, n_episode) pairs that exercise the surplus-env rule.  The recorded
    buffers / statistics are what oracle/collector.py::collect must reproduce."""
    from fsrl.data import FastCollector
    from fsrl.policy.ppo_lag import PPOLagrangian
    from gymnasium.spaces import Box
    from tianshou.data import ReplayBufferManager
    from oracle.collector import OracleBuffer
    from oracle.envs import OracleVecEnv
    KIND, SEED_ENV = "ball_run", 77                      # T = 100, terminates when the ball leaves the track

    from oracle.trainer_scenario import TerminatingEnv

    class VecEnv:
        def __init__(self, n, period=0):
            self.e = TerminatingEnv(KIND, n, SEED_ENV, period) if period else OracleVecEnv(KIND, n, SEED_ENV)
            self.action_space = [Box(low=-np.ones(self.e.A, np.float32), high=np.ones(self.e.A, np.float32))] * n

        def __len__(self):
            return self.e.E

        def reset(self, ids=None, **kw):
            obs = self.e.reset(ids)
            return obs, {"cost": np.zeros(len(obs))}

        def step(self, action, id=None):
            ids = np.arange(self.e.E) if id is None else np.asarray(id)
            obs_next, rew, cost, term, trunc = self.e.step(np.asarray(action, np.float32), ids)
            trunc = trunc & ~term
            return obs_next, rew.astype(np.float64), term, trunc, {"cost": cost.astype(np.float64)}

    class RecBuffer(ReplayBufferManager):
        def __init__(self, total, n, D, A):                 # deliberately NOT calling the device buffer's __init__
            self.b = OracleBuffer(total, n, D, A)
            self.buffer_num, self.maxsize = n, total
            self.run_rew, self.run_len = np.zeros(n), np.zeros(n, np.int64)

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

    cases = {}
    for E, n_ep, period in ((4, 4, 0), (4, 9, 0), (3, 7, 0), (5, 2, 0), (2, 1, 0),
                            (4, 11, 41), (5, 13, 29), (3, 5, 41), (6, 4, 17)):
        torch.manual_seed(15)
        env = VecEnv(E, period)
        D, A = env.e.D, env.e.A
        from tianshou.utils.net.common import Net
        from tianshou.utils.net.continuous import ActorProb, Critic
        actor = ActorProb(Net(D, hidden_sizes=(H, H)), A, max_action=1.0)
        critics = [Critic(Net(D, hidden_sizes=(H, H))) for _ in range(2)]
        torch.nn.init.constant_(actor.sigma_param, -0.5)
        pol = PPOLagrangian(actor, critics, torch.optim.Adam(actor.parameters()), _dist, logger=_Capture(),
                            observation_space=Box(low=-np.ones(D, np.float32) * 10, high=np.ones(D, np.float32) * 10),
                            action_space=env.action_space[0])
        pol.eval()
        buf = RecBuffer(E * 100 * 4, E, D, A)
        col = FastCollector(pol, env, buf, exploration_noise=False)
        st = col.collect(n_episode=n_ep)
        b = buf.b
        cases[f"E{E}_n{n_ep}" + (f"_term{period}" if period else "")] = dict(
            kw={}, lag=0.0, init=_state([("actor", actor)]), stats={},
            data=dict(E=np.array(E), n_episode=np.array(n_ep), period=np.array(period)),
            final=dict(obs=b.obs, obs_next=b.obs_next, act=b.act, rew=b.rew, cost=b.cost, terminated=b.terminated,
                       truncated=b.truncated, ptr=b.ptr, len=b.len,
                       stats=np.array([st[k] for k in ("n/ep", "n/st", "rew", "len", "total_cost", "cost", "truncated", "terminated")],
                                      dtype=np.float64),
                       collect_step=np.array(col.collect_step), collect_episode=np.array(col.collect_episode)))
    return cases


def golden_state_dicts():
    """Checkpoint surface of every learner: state_dict keys / shapes (incl. the PID `_extra_state`,
    lagrangian_base.py:122-143) and the PID state after a scripted cost sequence."""
    import json
    from copy import deepcopy
    from fsrl.policy import CPO, FOCOPS, DDPGLagrangian, PPOLagrangian, SACLagrangian, TRPOLagrangian
    act_space, obs_space = _space()
    common = dict(observation_space=obs_space, action_space=act_space)
    rec = {}

    def describe(pol):
        sd = pol.state_dict()
        out = {"keys": {k: (list(v.shape) if torch.is_tensor(v) else "object") for k, v in sd.items()}}
        if hasattr(pol, "lag_optims"):
            for cost in (25.0, 14.0, 3.0, 40.0):
                pol.pre_update_fn(stats_train={"cost": cost})
            ex = pol.get_extra_state()
            out["extra_state"] = [{k: (list(v) if isinstance(v, (tuple, list)) else float(v)) for k, v in e.items()} for e in ex]
            out["lagrangian"] = [float(o.get_lag()) for o in pol.lag_optims]
            clone = deepcopy(pol)
            for o in clone.lag_optims:
                o.lagrangian = 0.0
            clone.load_state_dict(pol.state_dict())
            out["restored"] = [float(o.get_lag()) for o in clone.lag_optims]
        return out

    actor, critics = _nets(1)
    rec["ppol"] = describe(PPOLagrangian(actor, critics, torch.optim.Adam(actor.parameters()), _dist, logger=_Capture(),
                                         cost_limit=10.0, **common))
    actor, critics = _nets(1)
    rec["trpol"] = describe(TRPOLagrangian(actor, critics, _crit_optim(critics, 1e-3), _dist, logger=_Capture(),
                                           cost_limit=10.0, **common))
    actor, critics = _nets(1)
    rec["cpo"] = describe(CPO(actor, critics, _crit_optim(critics, 1e-3), _dist, logger=_Capture(), cost_limit=10.0, **common))
    actor, critics = _nets(1)
    rec["focops"] = describe(FOCOPS(actor, critics, torch.optim.Adam(actor.parameters()), _crit_optim(critics, 1e-3), _dist,
                                    logger=_Capture(), cost_limit=10.0, nu=(2.0, 1e-2, torch.zeros(1)), **common))
    actor, critics = _q_nets(1, True)
    log_alpha = torch.zeros(1, requires_grad=True)
    rec["sacl"] = describe(SACLagrangian(actor, critics, torch.optim.Adam(actor.parameters()),
                                         torch.optim.Adam(torch.nn.ModuleList(critics).parameters()), logger=_Capture(),
                                         alpha=(-2.0, log_alpha, torch.optim.Adam([log_alpha])), cost_limit=10.0, **common))
    actor, critics = _q_nets(1, False)
    rec["ddpgl"] = describe(DDPGLagrangian(actor, critics, torch.optim.Adam(actor.parameters()),
                                           torch.optim.Adam(torch.nn.ModuleList(critics).parameters()), logger=_Capture(),
                                           cost_limit=10.0, **common))
    path = os.path.join(OUT, "state_dict_golden.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
    print("wrote", path, {k: len(v["keys"]) for k, v in rec.items()})


def golden_signatures():
    """Public call signatures of the drop-in surface (SURVEY.md 8b): parameter names, order and defaults of the
    reference's agents, policies, collector, trainers and loggers."""
    import inspect
    import json
    import fsrl.agent as A_
    import fsrl.data as D_
    import fsrl.policy as P_
    import fsrl.trainer as T_
    import fsrl.utils as U_

    def sig(fn):
        out = []
        for name, p in inspect.signature(fn).parameters.items():
            if name == "self":
                continue
            d = p.default
            if d is inspect.Parameter.empty:
                rep = "<required>"
            elif isinstance(d, (int, float, str, bool, tuple, list, type(None))):
                rep = repr(d)
            else:
                rep = "<object:%s>" % type(d).__name__
            out.append([name, str(p.kind), rep])
        return out

    rec = {}
    for mod, names, methods in (
            (A_, ["PPOLagAgent", "CPOAgent", "SACLagAgent", "DDPGLagAgent", "TRPOLagAgent", "FOCOPSAgent"],
             ["__init__", "learn", "evaluate"]),
            (P_, ["PPOLagrangian", "CPO", "SACLagrangian", "DDPGLagrangian", "TRPOLagrangian", "FOCOPS"],
             ["__init__", "learn", "process_fn", "pre_update_fn", "update", "forward", "map_action", "map_action_inverse"]),
            (D_, ["FastCollector"], ["__init__", "collect", "reset_env", "reset_buffer", "reset_stat"]),
            (T_, ["OnpolicyTrainer", "OffpolicyTrainer"], ["__init__", "policy_update_fn", "train_step", "test_step", "run"]),
            (U_, ["BaseLogger", "TensorboardLogger", "WandbLogger", "DummyLogger"],
             ["__init__", "store", "write", "save_checkpoint", "save_config", "get_mean", "print"])):
        for cn in names:
            cls = getattr(mod, cn)
            for m in methods:
                if hasattr(cls, m):
                    rec[f"{cn}.{m}"] = sig(getattr(cls, m))
    path = os.path.join(OUT, "signatures_golden.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
    print("wrote", path, len(rec), "signatures")


def golden_agent_inits():
    """Initial weights the reference's agent presets produce for a given seed (seed_all -> net construction ->
    orthogonal init -> optional last-layer scaling; e.g. ppo_lag_agent.py:128-162): the torch RNG is consumed in a
    fixed order, so a drop-in must build the same nets in the same order to start from the same point."""
    import types
    from fsrl.agent import CPOAgent, DDPGLagAgent, FOCOPSAgent, PPOLagAgent, SACLagAgent, TRPOLagAgent
    from fsrl.utils import BaseLogger
    act_space, obs_space = _space()
    env = types.SimpleNamespace(observation_space=obs_space, action_space=act_space)
    cases = {}
    for name, cls, kw in (("ppol", PPOLagAgent, {}), ("ppol_scaled", PPOLagAgent, dict(last_layer_scale=True)),
                          ("cpo", CPOAgent, {}), ("trpol", TRPOLagAgent, {}), ("focops", FOCOPSAgent, {}),
                          ("sacl", SACLagAgent, {}), ("sacl_fixed_sigma", SACLagAgent, dict(conditioned_sigma=False)),
                          ("ddpgl", DDPGLagAgent, {})):
        agent = cls(env, logger=BaseLogger(), device="cpu", seed=7, hidden_sizes=(H, H), **kw)
        sd = {k: v.detach().numpy().copy() for k, v in agent.policy.state_dict().items() if torch.is_tensor(v)}
        cases[name] = dict(kw=kw, lag=0.0, data={}, init=sd, final={}, stats={})
    return cases


def golden_public_attrs_and_safety_loss():
    """Public (non-nn.Module) attribute names of each learner instance, and LagrangianPolicy.safety_loss /
    BasePolicy.get_metrics on sample inputs."""
    import json
    from fsrl.policy import CPO, FOCOPS, DDPGLagrangian, PPOLagrangian, SACLagrangian, TRPOLagrangian
    base = set(dir(torch.nn.Module()))
    act_space, obs_space = _space()
    sp = dict(observation_space=obs_space, action_space=act_space)

    def pub(o):
        return sorted(n for n in dir(o) if not n.startswith("_") and n not in base)

    rec = {"attrs": {}}
    actor, critics = _nets(1)
    ppo = PPOLagrangian(actor, critics, torch.optim.Adam(actor.parameters()), _dist, logger=_Capture(), cost_limit=10.0, **sp)
    rec["attrs"]["PPOLagrangian"] = pub(ppo)
    actor, critics = _nets(1)
    rec["attrs"]["CPO"] = pub(CPO(actor, critics, _crit_optim(critics, 1e-3), _dist, logger=_Capture(), cost_limit=10.0, **sp))
    actor, critics = _nets(1)
    rec["attrs"]["TRPOLagrangian"] = pub(TRPOLagrangian(actor, critics, _crit_optim(critics, 1e-3), _dist, logger=_Capture(),
                                                         cost_limit=10.0, **sp))
    actor, critics = _nets(1)
    rec["attrs"]["FOCOPS"] = pub(FOCOPS(actor, critics, torch.optim.Adam(actor.parameters()), _crit_optim(critics, 1e-3), _dist,
                                         logger=_Capture(), cost_limit=10.0, nu=(2.0, 1e-2, torch.zeros(1)), **sp))
    actor, critics = _q_nets(1, True)
    la = torch.zeros(1, requires_grad=True)
    rec["attrs"]["SACLagrangian"] = pub(SACLagrangian(actor, critics, torch.optim.Adam(actor.parameters()),
                                                       torch.optim.Adam(torch.nn.ModuleList(critics).parameters()),
                                                       logger=_Capture(), alpha=(-2.0, la, torch.optim.Adam([la])), cost_limit=10.0, **sp))
    actor, critics = _q_nets(1, False)
    rec["attrs"]["DDPGLagrangian"] = pub(DDPGLagrangian(actor, critics, torch.optim.Adam(actor.parameters()),
                                                         torch.optim.Adam(torch.nn.ModuleList(critics).parameters()),
                                                         logger=_Capture(), cost_limit=10.0, **sp))
    # safety_loss (lagrangian_base.py:145-166) with and without rescaling
    rng = np.random.default_rng(70)
    vals = rng.normal(size=50).astype(np.float32)
    cases = []
    for lag, resc in ((0.0, True), (0.7, True), (2.5, False)):
        ppo.lag_optims[0].lagrangian = lag
        ppo.rescaling = resc
        loss, st = ppo.safety_loss([torch.from_numpy(vals)])
        cases.append({"lag": lag, "rescaling": resc, "loss": float(loss), "stats": {k: float(v) for k, v in st.items()}})
    rec["safety_loss"] = {"values": vals.tolist(), "cases": cases}
    path = os.path.join(OUT, "public_attrs_golden.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
    print("wrote", path, {k: len(v) for k, v in rec["attrs"].items()})


def golden_cvpo(Batch):
    """cvpo.py:248-430: three consecutive CVPO.learn() calls (SingleCritic and DoubleCritic variants) on given
    n-step targets; the K action particles each call draws from the old policy are recorded."""
    import torch.distributions as td
    from fsrl.policy.cvpo import CVPO
    from fsrl.utils.net.continuous import DoubleCritic, SingleCritic
    from tianshou.utils.net.common import Net
    from tianshou.utils.net.continuous import ActorProb
    cases = {}
    for name, double in (("single", False), ("double", True)):
        torch.manual_seed(11)
        actor = ActorProb(Net(D, hidden_sizes=(H, H)), A, max_action=1.0, conditioned_sigma=True)
        critics = []
        for _ in range(2):
            if double:
                critics.append(DoubleCritic(Net(D, A, hidden_sizes=(H, H), concat=True), Net(D, A, hidden_sizes=(H, H), concat=True)))
            else:
                critics.append(SingleCritic(Net(D, A, hidden_sizes=(H, H), concat=True)))
        for m in list(actor.modules()) + [mm for c in critics for mm in c.modules()]:
            if isinstance(m, torch.nn.Linear):
                torch.nn.init.orthogonal_(m.weight)
                torch.nn.init.zeros_(m.bias)
        init = _state(_mods(actor, critics))
        act_space, obs_space = _space()
        log = _Capture()
        pol = CVPO(actor, critics, torch.optim.Adam(actor.parameters(), lr=5e-4),
                   torch.optim.Adam(torch.nn.ModuleList(critics).parameters(), lr=1e-3), act_space, _dist, 300, logger=log,
                   cost_limit=10.0, tau=0.05, gamma=0.98, n_step=2, sample_act_num=8)
        pol.train()
        pol.pre_update_fn()
        torch.manual_seed(12)
        data = {}
        orig_sample = td.Independent.sample
        for k in range(3):
            d = _off_data(80 + k)
            drawn = []

            def tapped(self, sample_shape=torch.Size()):
                out = orig_sample(self, sample_shape)
                if len(sample_shape):
                    drawn.append(out.detach().numpy().copy())
                return out

            td.Independent.sample = tapped
            try:
                pol.learn(Batch(obs=torch.from_numpy(d["obs"]), act=torch.from_numpy(d["act"]),
                                rets=torch.from_numpy(d["rets"]), info=Batch()))
            finally:
                td.Independent.sample = orig_sample
            assert len(drawn) == 1 and drawn[0].shape == (8, BS, A)
            for kk, v in d.items():
                data[f"{kk}{k}"] = v
            data[f"particles{k}"] = drawn[0]
        final = _state(_mods(actor, critics) + [(f"critics_old.{i}", c) for i, c in enumerate(pol.critics_old)])
        final["estep_dual"] = pol.estep_dual.detach().numpy().copy()
        cases[name] = dict(kw={}, lag=0.0, data=data, init=init, final=final, stats=log.rows,
                           extra=dict(double=float(double), qc_thres=pol.qc_thres[0]))
    return cases


def golden_exports():
    """The reference packages' ``__all__`` lists."""
    import importlib
    import json
    rec = {m: sorted(getattr(importlib.import_module(f"fsrl.{m}"), "__all__", []))
           for m in ("agent", "policy", "data", "trainer", "utils")}
    path = os.path.join(OUT, "exports_golden.json")
    with open(path, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
    print("wrote", path, {k: len(v) for k, v in rec.items()})


def _save(name, cases):
    flat = {}
    for cname, c in cases.items():
        for grp in ("data", "init", "final"):
            for k, v in c[grp].items():
                flat[f"{cname}|{grp}|{k}"] = np.asarray(v)
        for k, v in c["stats"].items():
            flat[f"{cname}|stats|{k}"] = np.asarray(v, dtype=np.float64)
        flat[f"{cname}|lag"] = np.asarray(c["lag"], dtype=np.float64)
        for k, v in c.get("extra", {}).items():
            flat[f"{cname}|{k}"] = np.asarray(v, dtype=np.float64)
    path = os.path.join(OUT, name)
    np.savez_compressed(path, **flat)
    print("wrote", path, f"{os.path.getsize(path) / 1024:.1f} KiB", {k: len(v["stats"]) for k, v in cases.items()})


def check(ref_dir, rtol=2e-5):
    """Re-run the PPO cases with the reference found in `ref_dir` (e.g. the oracle/_ref install) and
    compare with the committed fixture: the installed copy must behave like the source tree."""
    global REF
    REF = ref_dir
    B = _bootstrap()
    fresh = golden_ppo(B)
    raw = np.load(os.path.join(OUT, "policy_ppo_golden.npz"))
    worst = 0.0
    for cname, c in fresh.items():
        for k, v in c["stats"].items():
            want = raw[f"{cname}|stats|{k}"]
            got = np.asarray(v, dtype=np.float64)
            assert got.shape == want.shape, (cname, k)
            err = np.abs(got - want).max() / (np.abs(want).max() + 1e-12)
            worst = max(worst, err)
            assert err <= rtol, (cname, k, err)
    print(f"reference in {ref_dir} reproduces tests/golden/policy_ppo_golden.npz (max rel err {worst:.2e})")


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--check":
        check(os.path.abspath(sys.argv[2]))
        sys.exit(0)
    B = _bootstrap()
    _save("policy_ppo_golden.npz", golden_ppo(B))
    _save("policy_cpo_golden.npz", golden_cpo(B))
    _save("policy_trpo_golden.npz", golden_trpo(B))
    _save("policy_focops_golden.npz", golden_focops(B))
    _save("policy_sac_golden.npz", golden_sac(B))
    _save("policy_ddpg_golden.npz", golden_ddpg(B))
    _save("policy_cvpo_golden.npz", golden_cvpo(B))
    _save("policy_returns_glue_golden.npz", golden_returns_glue(B))
    _save("collector_golden.npz", golden_collector())
    golden_trainers()
    golden_configs_and_names()
    golden_action_maps()
    golden_state_dicts()
    golden_signatures()
    golden_exports()
    golden_public_attrs_and_safety_loss()
    _save("agent_init_golden.npz", golden_agent_inits())
