"""The oracle against the reference's own outputs (fixtures made by oracle/make_golden.py
from the AST-extracted /root/reference/fsrl/policy/base_policy.py:524-567 and the imported
/root/reference/fsrl/utils/optim_util.py) and SURVEY.md Appendix B's literal vectors."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import cport, returns
from oracle.lagrangian import PIDLagrangian


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "returns_golden.npz"))


def test_gae_numpy_and_c_match_reference_bitwise(gold):
    n = int(gold["gae_count"])
    assert n >= 10
    for k in range(n):
        v, vn, r, e = (gold[f"gae{k}_{s}"] for s in ("v", "vn", "r", "e"))
        g, l = gold[f"gae{k}_gl"]
        want = gold[f"gae{k}_out"]
        got_c = cport.gae_return(v, vn, r, e, g, l)
        assert got_c.dtype == np.float64
        assert np.array_equal(got_c, want), f"C port differs on case {k}"
        if len(r) <= 5000:
            got = returns.gae_return(v, vn, r, e, g, l)
            assert np.array_equal(got, want), f"numpy port differs on case {k}"


def test_gae_appendix_b_literals():
    out = returns.gae_return(np.array([1, 2, 3, 4], np.float32), np.array([2, 3, 4, 0], np.float32),
                             np.ones(4), np.array([0, 0, 0, 1], bool), 0.99, 0.95)
    np.testing.assert_allclose(out, [3.07075357, 1.15975925, -0.8615, -3.0], rtol=0, atol=1e-8)
    out = returns.gae_return(np.array([0, 1], np.float32), np.array([0, 1], np.float32),
                             np.array([0., 1.]), np.array([False, True]), 0.1, 0.1)
    np.testing.assert_allclose(out, [0.001, 0.1], rtol=0, atol=1e-12)


def test_nstep_matches_reference(gold):
    n = int(gold["ns_count"])
    for k in range(n):
        m, e, tq, idx = (gold[f"ns{k}_{s}"] for s in ("m", "e", "tq", "idx"))
        g, ns = gold[f"ns{k}_gn"]
        want = gold[f"ns{k}_out"]
        got = returns.nstep_return(m, e, tq, idx, float(g), int(ns))
        np.testing.assert_allclose(got, want, rtol=1e-15, atol=0)
        got_c = cport.nstep_return(m, e, tq, idx, float(g), int(ns))
        np.testing.assert_allclose(got_c, want, rtol=1e-15, atol=0)


def test_nstep_appendix_b_literal():
    out = returns.nstep_return(np.array([1., 2, 3, 4, 5]), np.array([0, 0, 1, 0, 0], bool),
                               np.array([[10], [20], [0], [40]], np.float32),
                               np.array([[0, 1, 2, 3], [1, 2, 2, 4]]), 0.99, 2)
    np.testing.assert_allclose(out.ravel(), [12.781, 24.572, 3.0, 48.154], atol=1e-9)


def test_pid_matches_reference(golden_dir):
    cases = json.load(open(os.path.join(golden_dir, "pid_golden.json")))
    assert len(cases) >= 4
    for c in cases:
        o = PIDLagrangian(c["pid"])
        for cost, lam, integ, eold in zip(c["costs"], c["lagrangian"], c["error_integral"],
                                          c["error_old"]):
            o.step(cost, c["limit"])
            assert o.lagrangian == lam and o.error_integral == integ and o.error_old == eold
    # Appendix B literal
    o = PIDLagrangian((0.05, 0.0005, 0.1))
    lams = [o.step(c, 10) for c in (25, 18, 12, 8, 9, 14)]
    np.testing.assert_allclose(lams, [2.2575, 0.4115, 0.1125, 0.0, 0.061, 0.713], atol=1e-12)


def test_dual_gae_layout():
    rng = np.random.default_rng(0)
    N = 50
    v = rng.standard_normal((2, N)).astype(np.float32)
    vn = rng.standard_normal((2, N)).astype(np.float32)
    term = rng.random(N) < 0.1
    trunc = np.zeros(N, bool); trunc[24] = True
    unf = np.zeros(N, bool); unf[-1] = True
    vals, rets, advs = returns.dual_gae(v, vn, rng.random(N), rng.random(N) < 0.2, term, trunc,
                                        unf, 0.99, 0.95)
    assert vals.shape == rets.shape == advs.shape == (N, 2) and advs.dtype == np.float32
    np.testing.assert_allclose(rets, advs + vals, rtol=0, atol=1e-5)
    # a terminated step does not bootstrap: adv = r - v
    i = int(np.flatnonzero(term)[0])
    assert abs(advs[i, 0] - (np.float32(0) + 0)) >= 0  # smoke


# ---------------------------------------------------------------------------------------------------
# update paths: the oracle restatements replay golden vectors produced by the reference's OWN
# policy classes (oracle/make_golden_policies.py drives fsrl.policy.*.learn on CPU in the build
# container; tianshou / gymnasium are supplied by thin shims, the arithmetic is the reference's)
# ---------------------------------------------------------------------------------------------------
def _load_policy_golden(golden_dir, fname):
    raw = np.load(os.path.join(golden_dir, fname))
    cases = {}
    for key in raw.files:
        parts = key.split("|")
        c = cases.setdefault(parts[0], {"data": {}, "init": {}, "final": {}, "stats": {}})
        if len(parts) == 2:
            c[parts[1]] = float(raw[key])
        else:
            c[parts[1]][parts[2]] = raw[key]
    return cases


def _oracle_nets_from(init, D, A, H):
    from oracle import nets as onets
    sd = {k: torch.from_numpy(v) for k, v in init.items()}
    actor = onets.load_from_state_dict(onets.GaussActor(D, A, [H, H]), sd, "actor.")
    critics = [onets.load_from_state_dict(onets.ValueNet(D, [H, H]), sd, f"critics.{i}.") for i in range(2)]
    return actor, critics


def _assert_final_params(final, actor, critics, atol):
    pairs = [("actor.preprocess.model.model.0.weight", actor.body.layers[0].weight),
             ("actor.preprocess.model.model.0.bias", actor.body.layers[0].bias),
             ("actor.preprocess.model.model.2.weight", actor.body.layers[1].weight),
             ("actor.mu.model.0.weight", actor.mu.weight), ("actor.mu.model.0.bias", actor.mu.bias),
             ("actor.sigma_param", actor.sigma_param)]
    for i, c in enumerate(critics):
        pairs += [(f"critics.{i}.preprocess.model.model.0.weight", c.body.layers[0].weight),
                  (f"critics.{i}.preprocess.model.model.2.weight", c.body.layers[1].weight),
                  (f"critics.{i}.last.model.0.weight", c.last.weight), (f"critics.{i}.last.model.0.bias", c.last.bias)]
    for key, p in pairs:
        want = final[key]
        got = p.detach().numpy().reshape(want.shape)
        assert np.abs(got - want).max() <= atol, (key, np.abs(got - want).max())


@pytest.mark.parametrize("case,kw", [("base", {}), ("dualclip_vclip", dict(dual_clip=3.0, value_clip=True)),
                                     ("nolag", dict(use_lagrangian=False))])
def test_ppo_oracle_replays_reference_learn(golden_dir, case, kw):
    from oracle import ppo as oppo
    g = _load_policy_golden(golden_dir, "policy_ppo_golden.npz")[case]
    d = g["data"]
    D, A, H = d["obs"].shape[1], d["act"].shape[1], g["init"]["actor.mu.model.0.weight"].shape[1]
    actor, critics = _oracle_nets_from(g["init"], D, A, H)
    opt = torch.optim.Adam([p for m in [actor] + critics for p in m.parameters()], lr=5e-4)
    np.random.seed(21)
    stats = oppo.learn(actor, critics, opt, d, 64, 2, g["lag"], max_grad_norm=0.5, target_kl=1e9, **kw)
    ref = g["stats"]
    assert len(stats) == len(ref["loss/kl"])
    for key in ("loss/actor_rew", "loss/actor_total", "loss/kl", "loss/vf0", "loss/vf1", "loss/vf_total",
                "loss/total", "loss/entropy"):
        got = np.array([s[key] for s in stats])
        np.testing.assert_allclose(got, ref[key], rtol=2e-5, atol=2e-7, err_msg=key)
    if kw.get("use_lagrangian", True):
        np.testing.assert_allclose([s["loss/actor_safety"] for s in stats], ref["loss/actor_safety"], rtol=2e-5, atol=2e-7)
        np.testing.assert_allclose(ref["loss/lagrangian"], g["lag"])
    _assert_final_params(g["final"], actor, critics, atol=2e-6)


def _cmp_stats(stats, ref, keys, rtol, atol):
    for key in keys:
        assert key in ref, (key, sorted(ref))
        got = np.array([float(s[key]) for s in stats])
        want = np.asarray(ref[key])
        assert len(got) == len(want), (key, len(got), len(want))
        np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=key)


@pytest.mark.parametrize("case,dual_cases", [("feasible", [3, 3]), ("infeasible", [0, 0]), ("case2", [2, 2]),
                                            ("case1_then_2", [1, 2]), ("case0_then_1", [0, 1])])
def test_cpo_oracle_replays_reference_learn(golden_dir, case, dual_cases):
    """cpo.py:147-370 (critic regression, CG, dual case analysis, line search) run by the reference itself."""
    from oracle import cpo as ocpo
    g = _load_policy_golden(golden_dir, "policy_cpo_golden.npz")[case]
    d = g["data"]
    D, A, H = d["obs"].shape[1], d["act"].shape[1], g["init"]["actor.mu.model.0.weight"].shape[1]
    actor, critics = _oracle_nets_from(g["init"], D, A, H)
    opt = torch.optim.Adam([p for c in critics for p in c.parameters()], lr=1e-3)
    np.random.seed(22)
    stats = ocpo.learn(actor, critics, opt, d, 99999, 2, g["ave_cost"], g["cost_limit"], optim_critic_iters=3,
                       l2_reg=0.001, delta=0.01, max_backtracks=10)
    ref = g["stats"]
    assert [int(s["loss/optim_case"]) for s in stats] == [int(x) for x in ref["loss/optim_case"]] == dual_cases
    _cmp_stats(stats, ref, ("loss/kl", "loss/entropy", "loss/rew_loss", "loss/cost_loss", "loss/vf0", "loss/vf1",
                            "loss/vf_total", "loss/step_size"), rtol=2e-3, atol=2e-6)
    _cmp_stats(stats, ref, ("loss/optim_Q", "loss/optim_R", "loss/optim_S", "loss/optim_lam", "loss/optim_nu"),
               rtol=5e-3, atol=1e-5)
    _assert_final_params(g["final"], actor, critics, atol=5e-5)


@pytest.mark.parametrize("case", ["lag06", "lag0"])
def test_trpo_oracle_replays_reference_learn(golden_dir, case):
    from oracle import trpo as otrpo
    g = _load_policy_golden(golden_dir, "policy_trpo_golden.npz")[case]
    d = g["data"]
    D, A, H = d["obs"].shape[1], d["act"].shape[1], g["init"]["actor.mu.model.0.weight"].shape[1]
    actor, critics = _oracle_nets_from(g["init"], D, A, H)
    opt = torch.optim.Adam([p for c in critics for p in c.parameters()], lr=5e-4)
    np.random.seed(23)
    stats = otrpo.learn(actor, critics, opt, d, 99999, 2, g["lag"], optim_critic_iters=3, delta=0.001)
    ref = g["stats"]
    _cmp_stats(stats, ref, ("loss/actor_rew", "loss/actor_total", "loss/kl", "loss/step_size", "loss/vf0", "loss/vf1"),
               rtol=2e-3, atol=2e-6)
    _assert_final_params(g["final"], actor, critics, atol=5e-5)


@pytest.mark.parametrize("case", ["eta02", "eta_tiny"])
def test_focops_oracle_replays_reference_learn(golden_dir, case):
    from oracle import focops as ofoc
    g = _load_policy_golden(golden_dir, "policy_focops_golden.npz")[case]
    d = g["data"]
    D, A, H = d["obs"].shape[1], d["act"].shape[1], g["init"]["actor.mu.model.0.weight"].shape[1]
    actor, critics = _oracle_nets_from(g["init"], D, A, H)
    aopt = torch.optim.Adam(actor.parameters(), lr=5e-4)
    copt = torch.optim.Adam([p for c in critics for p in c.parameters()], lr=1e-3)
    nu, loss_nu = ofoc.nu_step(0.0, 1e-2, 2.0, 10.0, g["ave_cost"])
    ref = g["stats"]
    assert ref["loss/nu_value"][0] == pytest.approx(nu, abs=1e-7) and ref["loss/nu_loss"][0] == pytest.approx(loss_nu)
    np.random.seed(24)
    stats = ofoc.learn(actor, critics, aopt, copt, d, 64, 2, nu, eta=g["eta"], delta=1e9)
    _cmp_stats(stats, ref, ("loss/actor_loss", "loss/kl", "loss/entropy", "loss/vf0", "loss/vf1", "loss/vf_total"),
               rtol=2e-5, atol=2e-7)
    _assert_final_params(g["final"], actor, critics, atol=2e-6)


def _load_q(net, sd, prefix, k=None):
    from oracle import nets as onets
    pre = "preprocess" if k is None else f"preprocess{k}"
    last = "last" if k is None else f"last{k}"
    g = lambda key: sd[prefix + key]
    onets.load_linear(net.body.layers[0], g(pre + ".model.model.0.weight"), g(pre + ".model.model.0.bias"))
    onets.load_linear(net.body.layers[1], g(pre + ".model.model.2.weight"), g(pre + ".model.model.2.bias"))
    onets.load_linear(net.last, g(last + ".model.0.weight"), g(last + ".model.0.bias"))
    return net


def _assert_q(final, prefix, net, k, atol):
    pre = "preprocess" if k is None else f"preprocess{k}"
    last = "last" if k is None else f"last{k}"
    for key, p in ((pre + ".model.model.0.weight", net.body.layers[0].weight),
                   (pre + ".model.model.2.weight", net.body.layers[1].weight),
                   (pre + ".model.model.2.bias", net.body.layers[1].bias),
                   (last + ".model.0.weight", net.last.weight), (last + ".model.0.bias", net.last.bias)):
        want = final[prefix + key]
        assert np.abs(p.detach().numpy().reshape(want.shape) - want).max() <= atol, (prefix + key)


@pytest.mark.parametrize("case", ["auto_alpha", "fixed_alpha"])
def test_sac_oracle_replays_reference_learn(golden_dir, case):
    """sac_lag.py:185-269 (twin-Q critics, tanh-squashed actor loss, alpha step, Polyak) run by the reference
    itself; the reparameterisation noise it drew is replayed from the golden file."""
    from oracle import nets as onets, offpolicy as ooff
    g = _load_policy_golden(golden_dir, "policy_sac_golden.npz")[case]
    d, init = g["data"], {k: torch.from_numpy(v) for k, v in g["init"].items()}
    D, A = d["obs0"].shape[1], d["act0"].shape[1]
    H = g["init"]["actor.mu.model.0.weight"].shape[1]
    actor = onets.load_from_state_dict(onets.GaussActor(D, A, [H, H], unbounded=True, conditioned_sigma=True), init, "actor.")
    crit = [[_load_q(onets.ValueNet(D + A, [H, H]), init, f"critics.{i}.", k) for k in (1, 2)] for i in range(2)]
    crit_old = [[_load_q(onets.ValueNet(D + A, [H, H]), init, f"critics.{i}.", k) for k in (1, 2)] for i in range(2)]
    a_opt = torch.optim.Adam(actor.parameters(), lr=5e-4)
    c_opt = torch.optim.Adam([p for pair in crit for q in pair for p in q.parameters()], lr=1e-3)
    auto, alpha = None, 0.2
    if g["auto_alpha"]:
        log_alpha = torch.zeros(1, requires_grad=True)
        auto = (-float(A), log_alpha, torch.optim.Adam([log_alpha], lr=3e-4))
        alpha = 1.0
    stats = []
    for k in range(3):
        t = lambda name: torch.from_numpy(d[f"{name}{k}"])
        st, alpha = ooff.sac_update(actor, crit, crit_old, a_opt, c_opt, t("obs"), t("act"), t("rets"), t("eps"),
                                    alpha=alpha, tau=0.05, lagrangian=g["lag"], auto_alpha=auto)
        stats.append(st)
    ref = g["stats"]
    keys = ["loss/q0", "loss/q1", "loss/q_total", "loss/actor_rew", "loss/actor_safety", "loss/actor_total"]
    if g["auto_alpha"]:
        keys += ["loss/alpha_loss", "loss/alpha_value"]
    _cmp_stats(stats, ref, keys, rtol=2e-5, atol=2e-7)
    final = g["final"]
    for key, p in (("actor.mu.model.0.weight", actor.mu.weight), ("actor.sigma.model.0.weight", actor.sigma.weight),
                   ("actor.preprocess.model.model.0.weight", actor.body.layers[0].weight)):
        assert np.abs(p.detach().numpy() - final[key]).max() <= 2e-6, key
    for i in range(2):
        for k in (1, 2):
            _assert_q(final, f"critics.{i}.", crit[i][k - 1], k, 2e-6)
            _assert_q(final, f"critics_old.{i}.", crit_old[i][k - 1], k, 2e-6)      # Polyak-averaged targets


@pytest.mark.parametrize("case", ["lag05", "lag0"])
def test_ddpg_oracle_replays_reference_learn(golden_dir, case):
    from oracle import nets as onets, offpolicy as ooff
    g = _load_policy_golden(golden_dir, "policy_ddpg_golden.npz")[case]
    d, init = g["data"], {k: torch.from_numpy(v) for k, v in g["init"].items()}
    D, A = d["obs0"].shape[1], d["act0"].shape[1]
    H = g["init"]["actor.last.model.0.weight"].shape[1]

    def det_actor():
        a = onets.DetActor(D, A, [H, H])
        onets.load_linear(a.body.layers[0], init["actor.preprocess.model.model.0.weight"], init["actor.preprocess.model.model.0.bias"])
        onets.load_linear(a.body.layers[1], init["actor.preprocess.model.model.2.weight"], init["actor.preprocess.model.model.2.bias"])
        onets.load_linear(a.last, init["actor.last.model.0.weight"], init["actor.last.model.0.bias"])
        return a

    actor, actor_old = det_actor(), det_actor()
    crit = [_load_q(onets.ValueNet(D + A, [H, H]), init, f"critics.{i}.") for i in range(2)]
    crit_old = [_load_q(onets.ValueNet(D + A, [H, H]), init, f"critics.{i}.") for i in range(2)]
    a_opt = torch.optim.Adam(actor.parameters(), lr=5e-4)
    c_opt = torch.optim.Adam([p for q in crit for p in q.parameters()], lr=1e-3)
    stats = []
    for k in range(3):
        t = lambda name: torch.from_numpy(d[f"{name}{k}"])
        stats.append(ooff.ddpg_update(actor, actor_old, crit, crit_old, a_opt, c_opt, t("obs"), t("act"), t("rets"),
                                      tau=0.05, lagrangian=g["lag"]))
    _cmp_stats(stats, g["stats"], ["loss/q0", "loss/q1", "loss/q_total", "loss/actor_rew", "loss/actor_safety",
                                   "loss/actor_total"], rtol=2e-5, atol=2e-7)
    final = g["final"]
    for prefix, a in (("actor.", actor), ("actor_old.", actor_old)):
        for key, p in (("preprocess.model.model.0.weight", a.body.layers[0].weight), ("last.model.0.weight", a.last.weight),
                       ("last.model.0.bias", a.last.bias)):
            assert np.abs(p.detach().numpy() - final[prefix + key]).max() <= 2e-6, prefix + key
    for i in range(2):
        _assert_q(final, f"critics.{i}.", crit[i], None, 2e-6)
        _assert_q(final, f"critics_old.{i}.", crit_old[i], None, 2e-6)


def _ring_from(d):
    from oracle.collector import OracleBuffer
    E = len(d["ptr"])
    cap = d["obs"].shape[0] // E
    buf = OracleBuffer(cap * E, E, d["obs"].shape[1], d["act"].shape[1])
    for k in ("obs", "obs_next", "act", "rew", "cost"):
        setattr(buf, k, d[k])
    buf.terminated, buf.truncated = d["terminated"].astype(bool), d["truncated"].astype(bool)
    buf.ptr, buf.len = d["ptr"].astype(np.int64), d["len"].astype(np.int64)
    return buf


@pytest.mark.parametrize("case", ["gae", "gae_rew_norm"])
def test_gae_glue_replays_reference_compute_gae_returns(golden_dir, case):
    """base_policy.py:384-451 executed by the reference on a ragged ring (unfinished episodes, terminations,
    truncations): value mask, end flags, dtype flow, optional running-std normalisation."""
    from fsrl_b200.utils.optim_util import RunningMeanStd
    g = _load_policy_golden(golden_dir, "policy_returns_glue_golden.npz")[case]
    d, out = g["data"], g["final"]
    buf = _ring_from(d)
    idx = d["idx"].astype(np.int64)
    D, A, H = d["obs"].shape[1], d["act"].shape[1], g["init"]["actor.mu.model.0.weight"].shape[1]
    _, critics = _oracle_nets_from(g["init"], D, A, H)
    with torch.no_grad():
        v = np.stack([c(torch.from_numpy(buf.obs[idx])).flatten().numpy() for c in critics])
        vn = np.stack([c(torch.from_numpy(buf.obs_next[idx])).flatten().numpy() for c in critics])
    unfinished = np.isin(idx, buf.unfinished_index())
    assert unfinished.sum() == 2                       # two of the three envs stop mid-episode
    rms = [RunningMeanStd(), RunningMeanStd()]
    for call in range(2):
        if case == "gae":
            vals, rets, advs = returns.dual_gae(v, vn, buf.rew[idx], buf.cost[idx], buf.terminated[idx], buf.truncated[idx],
                                                unfinished, 0.99, 0.95)
        else:
            vals, rets, advs, moments = returns.dual_gae_rew_norm(
                v, vn, buf.rew[idx], buf.cost[idx], buf.terminated[idx], buf.truncated[idx], unfinished, 0.99, 0.95,
                [r.var for r in rms])
            for r, (m, var, cnt) in zip(rms, moments):
                r.update_moments(m, var, cnt)
            np.testing.assert_allclose([r.var for r in rms], out[f"rms_var{call}"], rtol=1e-6)
        np.testing.assert_allclose(vals, out[f"values{call}"], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(advs, out[f"advs{call}"], rtol=2e-6, atol=2e-6)
        np.testing.assert_allclose(rets, out[f"rets{call}"], rtol=2e-6, atol=2e-6)


def test_nstep_glue_replays_reference_compute_nstep_returns(golden_dir):
    """base_policy.py:453-512 executed by the reference (n = 1, 2, 3, 5) with a fixed target-Q function."""
    from oracle import offpolicy as ooff
    g = _load_policy_golden(golden_dir, "policy_returns_glue_golden.npz")["nstep"]
    buf = _ring_from(g["data"])
    out = g["final"]
    sel = out["sel"].astype(np.int64)
    for n_step in (1, 2, 3, 5):
        tq = [out[f"tq{n_step}"][i] for i in range(2)]
        rets, _ = ooff.nstep_targets(buf, sel, tq, 0.97, n_step)
        want = out[f"rets{n_step}"]                      # the reference keeps target_q's (bsz, 1) shape: (bsz, 1, C)
        assert want.shape == (len(sel), 1, 2)
        np.testing.assert_allclose(rets, want[:, 0, :], rtol=1e-6, atol=1e-6, err_msg=f"n_step={n_step}")


def test_installed_reference_reproduces_golden():
    """oracle/_ref (the --no-deps pip install used by `bench.py --impl reference`) runs through the same
    shims and reproduces the committed PPO fixture.  Runs in a subprocess: loading the reference rewires
    sys.modules (tianshou / gymnasium shims, `fsrl` = the reference)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = os.path.join(root, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref, "fsrl")):
        pytest.skip("oracle/_ref not installed (build() installs it where a checkout of liuzuxin/FSRL is present)")
    out = subprocess.run([sys.executable, os.path.join(root, "oracle", "make_golden_policies.py"), "--check", ref],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "reproduces" in out.stdout


def test_trainers_and_logger_match_reference_trace(golden_dir):
    """a15 (drivers + the train_speed bookkeeping): fsrl_b200's On/OffpolicyTrainer + BaseLogger, driven by
    the scripted fakes of oracle/trainer_scenario.py, make the same calls in the same order and return /
    log the same values as the reference's trainers did (tests/golden/trainer_golden.json)."""
    from fsrl_b200.trainer import OffpolicyTrainer, OnpolicyTrainer
    from fsrl_b200.utils.logger import BaseLogger
    from oracle import trainer_scenario
    want = json.load(open(os.path.join(golden_dir, "trainer_golden.json")))
    got = json.loads(json.dumps(trainer_scenario.run(OnpolicyTrainer, OffpolicyTrainer, BaseLogger)))
    for kind in ("onpolicy", "offpolicy"):
        w, g = want[kind], got[kind]
        assert g["trace"] == w["trace"], next((i, a, b) for i, (a, b) in enumerate(zip(g["trace"], w["trace"])) if a != b)
        np.testing.assert_allclose(np.array(g["stops"]), np.array(w["stops"]), rtol=1e-9)
        assert (g["env_step"], g["cum_episode"]) == (w["env_step"], w["cum_episode"])
        assert g["cum_cost"] == pytest.approx(w["cum_cost"])
        assert len(g["epochs"]) == len(w["epochs"]) == 3
        for ge, we in zip(g["epochs"], w["epochs"]):
            assert ge["epoch"] == we["epoch"]
            assert set(ge["stats"]) == set(we["stats"]), set(ge["stats"]) ^ set(we["stats"])
            for k in we["stats"]:
                assert ge["stats"][k] == pytest.approx(we["stats"][k], rel=1e-9), k
            assert set(ge["info"]) == set(we["info"]), set(ge["info"]) ^ set(we["info"])
            for k in we["info"]:
                assert ge["info"][k] == pytest.approx(we["info"][k], rel=1e-9), k


def test_config_defaults_and_run_names_match_reference(golden_dir):
    """Every config dataclass of the reference (fsrl/config/*_cfg.py: TrainCfg, Bullet*, Mujoco*) has the same
    fields and defaults in fsrl_b200.config, and exp_util.to_string / auto_name produce the same run names."""
    import dataclasses
    from fsrl_b200 import config as cfg
    from fsrl_b200.utils.exp_util import auto_name, to_string
    want = json.load(open(os.path.join(golden_dir, "config_names_golden.json")))
    norm = lambda d: {k: (list(v) if isinstance(v, tuple) else v) for k, v in d.items()}
    assert len(want["configs"]) == 48
    for name, fields in want["configs"].items():
        key, cls = name.split(".")
        got = norm(dataclasses.asdict(getattr(getattr(cfg, key + "_cfg"), cls)()))
        assert list(got) == list(fields) or set(got) == set(fields), (name, set(got) ^ set(fields))
        for k, v in fields.items():
            assert got[k] == v, (name, k, got[k], v)
    samples = (3, 2.5, 1e-4, 0.00037, 123456.789, True, None, "abc", [1, 2.5, "x"], (64, 64), {"a": 1, "b": [2, 3]}, 1e9, 10)
    for v, (rep, s) in zip(samples, want["to_string"]):
        assert repr(v) == rep and to_string(v) == s, (v, to_string(v), s)
    base = dataclasses.asdict(cfg.ppol_cfg.TrainCfg())
    for case in want["auto_name"]:
        cur = dict(base)
        cur.update({k: (tuple(v) if isinstance(v, list) else v) for k, v in case["changes"].items()})
        got = (auto_name(base, cur, case["prefix"], case["suffix"], skip_keys=case["skip"]) if case["skip"]
               else auto_name(base, cur, case["prefix"], case["suffix"]))
        assert got[:-5] == case["name"] and got[-5] == "-", (got, case["name"])


def test_action_maps_match_reference(golden_dir):
    """BasePolicy.map_action / map_action_inverse (a4) against the reference's own methods: clip / tanh / no
    bounding, with and without scaling, including a degenerate (low == high) action dimension."""
    import types
    import warnings
    from fsrl_b200.policy.base_policy import BasePolicy
    from fsrl_b200.spaces import Box
    g = json.load(open(os.path.join(golden_dir, "action_map_golden.json")))
    low, high = np.array(g["low"], np.float32), np.array(g["high"], np.float32)
    assert len(g["cases"]) == 6
    for c in g["cases"]:
        stub = types.SimpleNamespace(action_space=Box(low=low.copy(), high=high.copy()), action_scaling=c["scaling"],
                                     action_bound_method=c["method"])
        mapped = BasePolicy.map_action(stub, np.array(c["src"], np.float32))
        np.testing.assert_allclose(np.asarray(mapped, np.float64), np.array(c["mapped"]), rtol=0, atol=0)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")           # atanh of values outside (-1, 1): nan / inf like the reference
            inv = BasePolicy.map_action_inverse(stub, np.array(c["env_acts"], np.float32))
        inv = np.nan_to_num(np.asarray(inv, np.float64), nan=1e30, posinf=1e30, neginf=-1e30)
        np.testing.assert_allclose(inv, np.array(c["inverse"]), rtol=0, atol=0)


def test_logger_files_match_reference_byte_for_byte(golden_dir, tmp_path):
    """f3: config.yaml, progress.txt and the checkpoint file names written by fsrl_b200's BaseLogger equal what
    the reference's BaseLogger wrote for the same calls; our loader reads the reference's files."""
    from fsrl_b200.utils.exp_util import load_config_and_model
    from fsrl_b200.utils.logger import BaseLogger
    from oracle import trainer_scenario
    want = json.load(open(os.path.join(golden_dir, "trainer_golden.json")))["logger_files"]
    got = trainer_scenario.logger_files(BaseLogger, str(tmp_path / "ours"))
    assert got["progress.txt"] == want["progress.txt"]
    assert got["config.yaml"] == want["config.yaml"]
    assert got["checkpoints"] == want["checkpoints"] == ["model.pt", "model_7.pt", "model_best.pt"]
    assert got["cfg_after"] == want["cfg_after"]                      # the reference writes `name` into the caller's dict
    # a run directory as the REFERENCE wrote it (texts from the golden file) loads with our loader
    ref_run = tmp_path / "theirs" / "run"
    (ref_run / "checkpoint").mkdir(parents=True)
    (ref_run / "config.yaml").write_text(want["config.yaml"])
    torch.save({"model": {"w": torch.arange(3.0)}}, ref_run / "checkpoint" / "model.pt")
    cfg, model = load_config_and_model(str(ref_run))
    assert cfg["hidden_sizes"] == (128, 128) and cfg["lagrangian_pid"] == (0.05, 0.0005, 0.1) and cfg["name"] == "run"
    assert torch.equal(model["model"]["w"], torch.arange(3.0))


@pytest.mark.parametrize("case", ["E4_n4", "E4_n9", "E3_n7", "E5_n2", "E2_n1", "E4_n11_term41", "E5_n13_term29",
                                  "E3_n5_term41", "E6_n4_term17"])
def test_collector_oracle_replays_reference_fast_collector(golden_dir, case):
    """a1: fsrl/data/fast_collector.py:192-408 was executed by the reference's own FastCollector on the numpy env
    twin (deterministic eval-mode policy); oracle/collector.py::collect must fill the same buffer slots with the
    same transitions and return the same statistics -- episode counting, the surplus-env rule, reset order."""
    from oracle import collector as ocol, nets as onets
    from oracle.envs import OracleVecEnv
    g = _load_policy_golden(golden_dir, "collector_golden.npz")[case]
    E, n_ep = int(g["data"]["E"]), int(g["data"]["n_episode"])
    want = g["final"]
    period = int(g["data"]["period"])          # > 0: scripted terminations, episodes end at different times per env
    from oracle.trainer_scenario import TerminatingEnv
    env = TerminatingEnv("ball_run", E, 77, period) if period else OracleVecEnv("ball_run", E, 77)
    env.reset()
    D, A = env.D, env.A
    H = g["init"]["actor.mu.model.0.weight"].shape[1]
    actor = onets.load_from_state_dict(onets.GaussActor(D, A, [H, H]), {k: torch.from_numpy(v) for k, v in g["init"].items()}, "actor.")
    buf = ocol.OracleBuffer(E * 100 * 4, E, D, A)
    st = ocol.collect(env, actor, n_ep, 0, np.zeros(E, np.uint32), buf, mode="eval")
    got_stats = np.array([st[k] for k in ("n/ep", "n/st", "rew", "len", "total_cost", "cost", "truncated", "terminated")])
    np.testing.assert_allclose(got_stats, want["stats"], rtol=1e-6, atol=1e-9)
    assert int(want["collect_episode"]) == n_ep == st["n/ep"] and int(want["collect_step"]) == st["n/st"]
    np.testing.assert_array_equal(buf.ptr, want["ptr"]); np.testing.assert_array_equal(buf.len, want["len"])
    for k in ("terminated", "truncated"):
        np.testing.assert_array_equal(getattr(buf, k), want[k].astype(bool), err_msg=k)
    for k in ("obs", "obs_next", "act", "rew", "cost"):
        np.testing.assert_allclose(getattr(buf, k), want[k], rtol=1e-6, atol=1e-6, err_msg=k)


def _our_policy(kind):
    """fsrl_b200 learners built on the CPU (the device arena is created lazily, so the host-side surface --
    state_dict, PID bookkeeping -- can be inspected without a GPU)."""
    from torch.distributions import Independent, Normal
    from fsrl_b200 import nets
    from fsrl_b200.optim import FusedAdam
    from fsrl_b200.policy import CPO, FOCOPS, DDPGLagrangian, PPOLagrangian, SACLagrangian, TRPOLagrangian
    from fsrl_b200.spaces import Box
    D, A, H = 8, 2, 16
    sp = dict(observation_space=Box(low=-np.ones(D, np.float32) * 10, high=np.ones(D, np.float32) * 10),
              action_space=Box(low=-np.ones(A, np.float32), high=np.ones(A, np.float32)))
    dist = lambda *l: Independent(Normal(*l), 1)
    if kind in ("ppol", "trpol", "cpo", "focops"):
        actor = nets.ActorProb(nets.Net(D, hidden_sizes=(H, H)), A, max_action=1.0)
        critics = [nets.Critic(nets.Net(D, hidden_sizes=(H, H))) for _ in range(2)]
        if kind == "ppol":
            return PPOLagrangian(actor, critics, FusedAdam(lr=5e-4), dist, cost_limit=10.0, **sp)
        if kind == "trpol":
            return TRPOLagrangian(actor, critics, FusedAdam(lr=1e-3), dist, cost_limit=10.0, **sp)
        if kind == "cpo":
            return CPO(actor, critics, FusedAdam(lr=1e-3), dist, cost_limit=10.0, **sp)
        return FOCOPS(actor, critics, FusedAdam(lr=5e-4), FusedAdam(lr=1e-3), dist, cost_limit=10.0, nu=(2.0, 1e-2, 0.0), **sp)
    if kind == "sacl":
        actor = nets.ActorProb(nets.Net(D, hidden_sizes=(H, H)), A, max_action=1.0, unbounded=True, conditioned_sigma=True)
        critics = [nets.DoubleCritic(nets.Net(D, A, hidden_sizes=(H, H), concat=True), nets.Net(D, A, hidden_sizes=(H, H), concat=True))
                   for _ in range(2)]
        log_alpha = torch.zeros(1, requires_grad=True)
        return SACLagrangian(actor, critics, FusedAdam(lr=5e-4), FusedAdam(lr=1e-3),
                             alpha=(-2.0, log_alpha, torch.optim.Adam([log_alpha])), cost_limit=10.0, **sp)
    actor = nets.Actor(nets.Net(D, hidden_sizes=(H, H)), A, max_action=1.0)
    critics = [nets.Critic(nets.Net(D, A, hidden_sizes=(H, H), concat=True)) for _ in range(2)]
    return DDPGLagrangian(actor, critics, FusedAdam(lr=5e-4), FusedAdam(lr=1e-3), cost_limit=10.0, **sp)


@pytest.mark.parametrize("kind", ["ppol", "trpol", "cpo", "focops", "sacl", "ddpgl"])
def test_checkpoint_surface_matches_reference(golden_dir, kind):
    """f3: `{"model": policy.state_dict()}` is the checkpoint both sides exchange -- same keys, same shapes (incl.
    the PID `_extra_state`), and the PID multiplier after a scripted cost sequence and a state_dict round trip."""
    want = json.load(open(os.path.join(golden_dir, "state_dict_golden.json")))[kind]
    pol = _our_policy(kind)
    sd = pol.state_dict()
    got_keys = {k: (list(v.shape) if torch.is_tensor(v) else "object") for k, v in sd.items()}
    assert set(got_keys) == set(want["keys"]), sorted(set(got_keys) ^ set(want["keys"]))
    for k, shape in want["keys"].items():
        assert got_keys[k] == shape, (k, got_keys[k], shape)
    if "extra_state" in want:
        for cost in (25.0, 14.0, 3.0, 40.0):
            pol.pre_update_fn(stats_train={"cost": cost})
        ex = pol.get_extra_state()
        assert len(ex) == len(want["extra_state"])
        for e, w in zip(ex, want["extra_state"]):
            assert set(e) == set(w)
            for k in w:
                np.testing.assert_allclose(np.asarray(e[k], np.float64), np.asarray(w[k], np.float64), rtol=1e-12)
        np.testing.assert_allclose(pol.lagrangians(), want["lagrangian"], rtol=1e-12)
        # restoring: the reference goes through load_state_dict -> set_extra_state; ours would first build the
        # device arena in load_state_dict, so the CPU test exercises the same hook directly
        clone = _our_policy(kind)
        assert clone.lagrangians() != pol.lagrangians()
        clone.set_extra_state(pol.state_dict()["_extra_state"])
        # Reference quirk, pinned here: its set_extra_state looks for an "_extra_state" KEY inside what torch
        # hands it -- which is the list itself -- so load_state_dict leaves the PID at zero
        # (lagrangian_base.py:139-143; the golden records 0.0).  fsrl_b200 restores the state (the evident
        # intent; resume continues the dual variable) and still accepts the wrapped form.
        assert want["restored"] == [0.0] * len(want["restored"])
        np.testing.assert_allclose(clone.lagrangians(), want["lagrangian"], rtol=1e-12)
        wrapped = _our_policy(kind)
        wrapped.set_extra_state({"_extra_state": pol.state_dict()["_extra_state"]})
        np.testing.assert_allclose(wrapped.lagrangians(), want["lagrangian"], rtol=1e-12)
        for cost in (5.0, 30.0):                      # and the restored PID continues identically
            clone.pre_update_fn(stats_train={"cost": cost}); pol.pre_update_fn(stats_train={"cost": cost})
        np.testing.assert_allclose(clone.lagrangians(), pol.lagrangians(), rtol=1e-12)


def test_public_signatures_match_reference(golden_dir):
    """(b) drop-in boundary: every parameter of the reference's agents / policies / collector / trainers / loggers
    (names, order, defaults; tests/golden/signatures_golden.json, extracted with inspect from the reference) exists
    on the fsrl_b200 class with the same default.  Deliberate deviations are listed here, nothing else may differ."""
    import inspect
    import fsrl_b200.agent as A_
    import fsrl_b200.data as D_
    import fsrl_b200.policy as P_
    import fsrl_b200.trainer as T_
    from fsrl_b200.utils import logger as U_
    want = json.load(open(os.path.join(golden_dir, "signatures_golden.json")))
    allowed = {
        # the engine only runs on CUDA devices ("cpu" is accepted and mapped to "cuda")
        **{(f"{a}.__init__", "device"): "'cuda'" for a in ("PPOLagAgent", "CPOAgent", "SACLagAgent", "DDPGLagAgent",
                                                           "TRPOLagAgent", "FOCOPSAgent")},
        # dist_fn is optional: the device kernels implement Independent(Normal) directly
        **{(f"{p}.__init__", "dist_fn"): "None" for p in ("PPOLagrangian", "CPO", "TRPOLagrangian", "FOCOPS")},
    }
    home = {**{n: A_ for n in ("PPOLagAgent", "CPOAgent", "SACLagAgent", "DDPGLagAgent", "TRPOLagAgent", "FOCOPSAgent")},
            **{n: P_ for n in ("PPOLagrangian", "CPO", "SACLagrangian", "DDPGLagrangian", "TRPOLagrangian", "FOCOPS")},
            "FastCollector": D_, "OnpolicyTrainer": T_, "OffpolicyTrainer": T_,
            **{n: U_ for n in ("BaseLogger", "TensorboardLogger", "WandbLogger", "DummyLogger")}}

    def rep(d):
        if d is inspect.Parameter.empty:
            return "<required>"
        return repr(d) if isinstance(d, (int, float, str, bool, tuple, list, type(None))) else "<object:%s>" % type(d).__name__

    assert len(want) == 109
    problems = []
    for key, ref_params in sorted(want.items()):
        cn, m = key.split(".")
        cls = getattr(home[cn], cn)
        assert hasattr(cls, m), key
        ours = inspect.signature(getattr(cls, m)).parameters
        has_kwargs = any(p.kind is inspect.Parameter.VAR_KEYWORD for p in ours.values())
        for name, kind, default in ref_params:
            if kind in ("VAR_KEYWORD", "VAR_POSITIONAL"):
                continue
            if name not in ours:
                if not has_kwargs:
                    problems.append(f"{key}: parameter {name} missing")
                continue
            got = rep(ours[name].default)
            if got != default and not (default.startswith("<object") or got.startswith("<object")):
                if allowed.get((key, name)) != got:
                    problems.append(f"{key}: {name} default {got} != reference {default}")
        ref_order = [n for n, k, _ in ref_params if k == "POSITIONAL_OR_KEYWORD"]
        our_order = [n for n, p in ours.items() if p.kind is inspect.Parameter.POSITIONAL_OR_KEYWORD and n != "self"]
        if [n for n in our_order if n in ref_order] != [n for n in ref_order if n in our_order]:
            problems.append(f"{key}: positional order differs {our_order} vs {ref_order}")
    assert not problems, "\n".join(problems)


@pytest.mark.parametrize("case,agent,kw", [("ppol", "PPOLagAgent", {}), ("ppol_scaled", "PPOLagAgent", dict(last_layer_scale=True)),
                                           ("cpo", "CPOAgent", {}), ("trpol", "TRPOLagAgent", {}), ("focops", "FOCOPSAgent", {}),
                                           ("sacl", "SACLagAgent", {}), ("ddpgl", "DDPGLagAgent", {})])
def test_agent_presets_start_from_the_reference_weights(golden_dir, monkeypatch, case, agent, kw):
    """Same seed -> same initial parameters as the reference's agent presets (bit for bit): seed_all, the order in
    which the nets are built (default torch init consumes the RNG), orthogonal re-initialisation order, sigma_param
    constant, last-layer scaling, deep-copied target nets.  The device arena is patched out: only the host recipe
    is under test, so this runs without a GPU."""
    import types
    import fsrl_b200.agent as A_
    from fsrl_b200.policy.base_policy import BasePolicy
    from fsrl_b200.spaces import Box
    monkeypatch.setattr(BasePolicy, "_build_arena",
                        lambda self, device=None: setattr(self, "_arena", types.SimpleNamespace(device="cpu")) or self._arena)
    want = _load_policy_golden(golden_dir, "agent_init_golden.npz")[case]["init"]
    env = types.SimpleNamespace(observation_space=Box(low=-np.ones(8, np.float32) * 10, high=np.ones(8, np.float32) * 10),
                                action_space=Box(low=-np.ones(2, np.float32), high=np.ones(2, np.float32)))
    a = getattr(A_, agent)(env, seed=7, hidden_sizes=(16, 16), **kw)
    got = {k: v.detach().cpu().numpy() for k, v in a.policy.state_dict().items() if torch.is_tensor(v)}
    assert set(got) == set(want), sorted(set(got) ^ set(want))
    for k in want:
        np.testing.assert_array_equal(got[k], want[k], err_msg=k)


def test_package_exports_cover_the_reference(golden_dir):
    """Every name in the reference's ``fsrl.{agent,policy,data,trainer,utils}.__all__`` is importable from the
    matching fsrl_b200 package, except the documented out-of-scope components (DESIGN.md section 7)."""
    import importlib
    want = json.load(open(os.path.join(golden_dir, "exports_golden.json")))
    out_of_scope = {"CVPOAgent", "CVPO", "BasicCollector", "TrajectoryBuffer",
                    "BasicLogger"}          # listed in fsrl.utils.__all__ but defined nowhere in the reference
    for pkg, names in want.items():
        mod = importlib.import_module(f"fsrl_b200.{pkg}")
        missing = [n for n in names if not hasattr(mod, n) and n not in out_of_scope]
        assert not missing, (pkg, missing)


def test_public_attributes_and_safety_loss_match_reference(golden_dir):
    """Every public attribute / method name a reference learner instance exposes exists on the fsrl_b200 learner
    (the per-piece loss methods are the documented exception: they are fused into the device update), and
    LagrangianPolicy.safety_loss returns the reference's value and statistics."""
    g = json.load(open(os.path.join(golden_dir, "public_attrs_golden.json")))
    fused = {"critics_loss", "policy_loss"}          # no per-piece host methods: one fused kernel chain does both
    kinds = {"PPOLagrangian": "ppol", "CPO": "cpo", "TRPOLagrangian": "trpol", "FOCOPS": "focops",
             "SACLagrangian": "sacl", "DDPGLagrangian": "ddpgl"}
    for cls, kind in kinds.items():
        pol = _our_policy(kind)
        # PPOLagrangian carries eager-autograd versions of the per-piece hooks; the other learners' pieces are fused
        missing = [n for n in g["attrs"][cls] if not hasattr(pol, n) and (n not in fused or kind == "ppol")]
        # compute_nstep_returns lives on the off-policy learners (it needs their replay descriptor)
        missing = [n for n in missing if not (n == "compute_nstep_returns" and kind in ("ppol", "cpo", "trpol", "focops"))]
        assert not missing, (cls, missing)
    pol = _our_policy("ppol")
    vals = torch.tensor(g["safety_loss"]["values"], dtype=torch.float32)
    for c in g["safety_loss"]["cases"]:
        pol.lag_optims[0].lagrangian = c["lag"]
        pol.rescaling = c["rescaling"]
        loss, st = pol.safety_loss([vals])
        assert float(loss) == pytest.approx(c["loss"], rel=1e-6, abs=1e-9)
        assert set(st) == set(c["stats"])
        for k, v in c["stats"].items():
            assert float(st[k]) == pytest.approx(v, rel=1e-6, abs=1e-9), k


@pytest.mark.parametrize("case", ["single", "double"])
def test_cvpo_oracle_replays_reference_learn(golden_dir, case):
    """Groundwork for SURVEY 8(f4): oracle/cvpo.py reproduces three consecutive CVPO.learn() calls of the reference
    (critic regression, E-step dual Adam + softmax weights over the recorded action particles, M-step with the
    decoupled KL multipliers, Polyak targets) -- SingleCritic and DoubleCritic variants."""
    from oracle import cvpo as ocvpo, nets as onets
    g = _load_policy_golden(golden_dir, "policy_cvpo_golden.npz")[case]
    d, init = g["data"], {k: torch.from_numpy(v) for k, v in g["init"].items()}
    D, A = d["obs0"].shape[1], d["act0"].shape[1]
    H = g["init"]["actor.mu.model.0.weight"].shape[1]
    double = bool(g["double"])

    def build():
        actor = onets.load_from_state_dict(onets.GaussActor(D, A, [H, H], conditioned_sigma=True), init, "actor.")
        if double:
            crit = [[_load_q(onets.ValueNet(D + A, [H, H]), init, f"critics.{i}.", k) for k in (1, 2)] for i in range(2)]
        else:
            crit = [_load_q(onets.ValueNet(D + A, [H, H]), init, f"critics.{i}.") for i in range(2)]
        return actor, crit

    actor, crit = build()
    actor_old, crit_old = build()
    flat = lambda cs: [p for c in cs for q in (c if isinstance(c, list) else [c]) for p in q.parameters()]
    a_opt = torch.optim.Adam(actor.parameters(), lr=5e-4)
    c_opt = torch.optim.Adam(flat(crit), lr=1e-3)
    estep_dual = torch.tensor([1.0, 0.0], requires_grad=True, dtype=torch.float32)
    e_opt = torch.optim.Adam([estep_dual], lr=0.02)
    mduals = (torch.zeros(1, requires_grad=True), torch.zeros(1, requires_grad=True))      # pre_update_fn (:172-181)
    m_opt = torch.optim.Adam(list(mduals), lr=0.1)
    stats = []
    for k in range(3):
        t = lambda name: torch.from_numpy(d[f"{name}{k}"])
        stats.append(ocvpo.cvpo_update(actor, actor_old, crit, crit_old, a_opt, c_opt, estep_dual, e_opt, mduals, m_opt,
                                       t("obs"), t("act"), t("rets"), t("particles"), qc_thres=[g["qc_thres"]], tau=0.05))
    assert g["qc_thres"] == pytest.approx(ocvpo.qc_thresholds(10.0, 0.98, 300)[0], rel=1e-12)
    ref = g["stats"]
    keys = ["loss/loss_q0", "loss/loss_q1", "loss/q_total", "loss/estep_loss", "estep/dual0", "estep/dual1",
            "estep/val_q0", "estep/val_q1", "mstep/mstep_kl_mu", "mstep/mstep_kl_std", "mstep/mstep_loss_mle",
            "mstep/mstep_loss_kl", "mstep/mstep_loss_total", "mstep/mstep_dual_mu", "mstep/mstep_dual_std", "mstep/entropy"]
    _cmp_stats(stats, ref, keys, rtol=5e-5, atol=1e-6)
    final = g["final"]
    np.testing.assert_allclose(estep_dual.detach().numpy(), final["estep_dual"], rtol=1e-5, atol=1e-7)
    for key, p in (("actor.mu.model.0.weight", actor.mu.weight), ("actor.sigma.model.0.weight", actor.sigma.weight),
                   ("actor.preprocess.model.model.2.weight", actor.body.layers[1].weight)):
        assert np.abs(p.detach().numpy() - final[key]).max() <= 5e-6, key
    for i in range(2):
        if double:
            for k in (1, 2):
                _assert_q(final, f"critics.{i}.", crit[i][k - 1], k, 5e-6)
                _assert_q(final, f"critics_old.{i}.", crit_old[i][k - 1], k, 5e-6)
        else:
            _assert_q(final, f"critics.{i}.", crit[i], None, 5e-6)
            _assert_q(final, f"critics_old.{i}.", crit_old[i], None, 5e-6)
