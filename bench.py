"""bench.py -- BASELINE.json's metric on its configurations.

metric : env-steps/sec over collect+update (the reference's ``train_speed``, fsrl/trainer/base_trainer.py:345-347)
step   : ONE collect + update cycle (trainer.train_step + policy_update_fn)
configs: --config c1 | c2 (default, the headline) | c3 | c4 | c5   (BASELINE.json "configs", in order)

  python bench.py [--config c2] [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Prints one JSON line (rank 0).  See DESIGN.md "Measurement" for how every field is derived.  --dump-outputs writes what
the last timed step computed as DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 10
# BASELINE.json configs.  `envs` is per GPU (weak scaling); hyper-parameters are the reference's cfg files
# (fsrl/config/{ppol,cpo,sacl}_cfg.py, SURVEY.md Appendix E) except the widths / env counts BASELINE.json overrides.
CONFIGS = {
    "c1": dict(algo="ppol", task="SafetyCarCircle-v0", kind="car_circle", envs=4, hidden=(64, 64), batch=256, repeat=4,
               desc="c1: PPO-Lagrangian SafetyCarCircle-v0, 4 envs x 300 steps, 2x64 MLP, batch_size 256, repeat 4"),
    "c2": dict(algo="ppol", task="SafetyCarCircle-v0", kind="car_circle", envs=2048, hidden=(256, 256), batch=256, repeat=4,
               desc="c2: PPO-Lagrangian SafetyCarCircle-v0, 2048 envs/GPU x 300 steps, 2x256 MLP, batch_size 256, repeat 4, "
                    "max_grad_norm 0.5"),
    "c3": dict(algo="cpo", task="SafetyPointGoal1Gymnasium-v0", kind="point_goal", envs=2048, hidden=(128, 128), batch=99999,
               repeat=4, desc="c3: CPO SafetyPointGoal1-v0, 2048 envs/GPU x 1000 steps, 2x128 MLP, CG iters 10, "
                              "max_backtracks 100, optim_critic_iters 10, repeat 4"),
    "c4": dict(algo="sacl", task="SafetyCarRun-v0", kind="car_run", envs=4096, hidden=(128, 128), batch=256, ups=0.2,
               desc="c4: SAC-Lagrangian SafetyCarRun-v0, 4096 envs/GPU x 200 steps, 2x128 MLP, replay on device, "
                    "update_per_step 0.2, batch 256, n_step 2"),
    "c5": dict(algo="ppol", task="SafetyAntCircle-v0", kind="ant_circle", envs=1024, hidden=(512, 512), batch=256, repeat=4,
               desc="c5: PPO-Lagrangian SafetyAntCircle-v0, 1024 envs/GPU (8192 on 8 GPUs) x 500 steps, 2x512 MLP, "
                    "batch_size 256, repeat 4, max_grad_norm 0.5"),
}
METRIC = {"ppol": "PPO-Lag", "cpo": "CPO", "sacl": "SAC-Lag"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# -------------------------------------------------------------------------------------------------
# our arm
# -------------------------------------------------------------------------------------------------
def build(cfg, device, rank):
    from fsrl_b200 import envs as fenvs
    from fsrl_b200.agent import CPOAgent, PPOLagAgent, SACLagAgent
    from fsrl_b200.data import FastCollector, VectorReplayBuffer
    from fsrl_b200.parallel import shard_seed
    from fsrl_b200.trainer import OffpolicyTrainer, OnpolicyTrainer
    from fsrl_b200.utils.logger import BaseLogger
    demo = fenvs.make(cfg["task"])
    logger = BaseLogger()
    envs, T = cfg["envs"], demo.spec.max_episode_steps
    algo = cfg["algo"]
    if algo == "ppol":
        agent = PPOLagAgent(demo, logger=logger, cost_limit=10, device=device, seed=SEED, lr=5e-4,
                            hidden_sizes=cfg["hidden"], max_grad_norm=0.5)      # ppol_cfg.py:14-33
        # fixed work per step: the KL early stop (ppo_lag.py:251-255) is disabled so that EVERY step runs all
        # `repeat` passes over the batch (the most work the config can do)
        agent.policy._target_kl = float("inf")
    elif algo == "cpo":
        agent = CPOAgent(demo, logger=logger, cost_limit=10, device=device, seed=SEED, hidden_sizes=cfg["hidden"],
                         max_backtracks=100, optim_critic_iters=10)            # cpo_cfg.py:19-26
    else:
        agent = SACLagAgent(demo, logger=logger, cost_limit=10, device=device, seed=SEED, hidden_sizes=cfg["hidden"],
                            unbounded=False, n_step=2, tau=0.05, gamma=0.97)   # sacl_cfg.py:14-30
    train_envs = fenvs.DeviceVectorEnv(cfg["task"], envs, device=device, seed=shard_seed(SEED + 1, rank))
    agent.policy.set_action_seed(shard_seed(SEED + 7, rank))
    buf = VectorReplayBuffer(envs * T, envs, device=device)
    col = FastCollector(agent.policy, train_envs, buf, exploration_noise=True)
    common = dict(max_epoch=1, batch_size=cfg["batch"], cost_limit=10, step_per_epoch=envs * T, episode_per_collect=envs,
                  episode_per_test=1, logger=logger, verbose=False, show_progress=False)
    if algo == "sacl":
        trainer = OffpolicyTrainer(agent.policy, col, None, update_per_step=cfg["ups"], **common)
    else:
        trainer = OnpolicyTrainer(agent.policy, col, None, repeat_per_collect=cfg["repeat"], **common)
    return agent, trainer, col, buf, T


def one_cycle(trainer):
    stats = trainer.train_step()
    trainer.policy_update_fn(stats)
    return stats


def ev_time(fn, stream_sync=True):
    """CUDA-event duration [ms] of fn() on the current (launching) stream, synchronised on both sides."""
    torch.cuda.synchronize()
    s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
    s.record(); out = fn(); e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e), out


def net_flops(D, H, A, rows):
    """Algorithmic flops (2 x MAC) of forward + backward-data + weight-gradient of actor + 2 critics on `rows` rows."""
    def net(out):
        fwd = 2 * rows * (D * H + H * H + H * out)
        bwd = 2 * rows * (H * out + H * H)
        wgr = 2 * rows * (D * H + H * H + H * out)
        return fwd + bwd + wgr
    return net(A) + 2 * net(1)


def ppo_rooflines(cfg, agent, col, buf, T, device, pk, how):
    """Dominant kernel of the PPO configs = the minibatch update (one persistent launch per repeat, or the three-launch
    chain where the persistent gate does not apply): algorithmic flops / CUDA-event time of one repeat.  Second object:
    the HBM roofline BASELINE.json names, collect + GAE, from event-timed collect / process_fn passes."""
    import ctypes
    from fsrl_b200 import _lib
    pol = agent.policy
    envs = cfg["envs"]
    col.reset_buffer()
    ms_collect, _ = ev_time(lambda: col.collect(envs))
    idx = buf.sample_indices(0)
    ms_gae, batch = ev_time(lambda: pol.process_fn(None, buf, idx))
    n = batch.n
    s0 = pol.arena.slots[0]
    D, H, A = s0.D, s0.H, s0.out
    pol._ensure_update_state(cfg["batch"], n, 1)
    u = pol._descriptor(batch, torch.zeros(n, dtype=torch.int32, device=device))
    persistent = bool(_lib.lib.fsrl_ppo_persist_active(ctypes.byref(u), n, cfg["batch"]))
    # one repeat = one fsrl_ppo_lag_epoch call (gather + advantage statistics + the update launch(es)); the permutation is
    # uploaded before the timed region so that the host's draw of it is not counted as kernel time
    perm = torch.randperm(n, device=device).to(torch.int32)
    pol._dp_batch = int(cfg["batch"])
    u = pol._descriptor(batch, perm)
    pol._stats_dev.zero_()
    n_mb_c = ctypes.c_int(0)
    stream = pol._stream()

    def one_repeat():
        _lib.check(_lib.lib.fsrl_ppo_lag_epoch(ctypes.byref(u), n, int(cfg["batch"]), 0, pol.optim.step_count,
                                               ctypes.byref(n_mb_c), stream))
        pol.optim.step_count += n_mb_c.value
    one_repeat()                                                   # warm
    l0 = int(_lib.lib.fsrl_launch_count())
    ms_rep, _ = ev_time(one_repeat)
    launches_rep = int(_lib.lib.fsrl_launch_count()) - l0
    n_mb = max(n // cfg["batch"], 1)
    fl = net_flops(D, H, A, cfg["batch"]) * n_mb
    ach = fl / (ms_rep * 1e-3) / 1e12
    peak = pk["bf16_tflops_sustained"]
    traffic_file = os.path.join(ROOT, "profiles", "r2_ppo_persist_traffic.json")
    # the captured DRAM traffic belongs to the persistent launch; the chain's (H != 256) is in profiles/r1_ppo_update_ncu_summary.txt
    traffic = json.load(open(traffic_file)) if (persistent and os.path.exists(traffic_file)) else None
    roof = {"kernel": "ppo_persist_kernel (one launch per repeat: tcgen05 kind::tf32 3-term split, TMEM accumulators, bulk-copy "
                      "operand images)" if persistent else "ppo_fwd/bwd/wgrad_adam chain (three launches per minibatch)",
            "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
            "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
            "traffic_unit": "DRAM bytes read+written per launch (ncu --set full --cache-control none, "
                            "profiles/r2_ppo_persist_ncu_summary.txt)" if traffic else None,
            "peak_source": how + " bf16 sustained (kernel timed inside a long step)",
            "ms_per_launch": ms_rep, "minibatch_steps_per_launch": n_mb, "us_per_minibatch_step": ms_rep * 1e3 / n_mb,
            "launches_per_repeat": launches_rep, "persistent": persistent,
            "algorithmic_flops_per_minibatch_step": net_flops(D, H, A, cfg["batch"]),
            "note": "fp32-faithful 3xTF32 (3 tensor-core MMAs per fp32 product; the algorithmic flop count is NOT tripled); a chain of "
                    "dependent optimiser steps of 256 rows: latency- and synchronisation-bound, far from the tensor peak"}
    bstep = 12 * D + 4 * A + 28 + 12 * 2                        # SURVEY.md 8d: algorithmic bytes per env step, collect + GAE
    hbm = {"kernel": "rollout_step_kernel x T + mlp_forward_kernel + gae_dual_kernel (collect + dual GAE)", "bound": "hbm",
           "achieved": bstep * n / ((ms_collect + ms_gae) * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
           "bytes_per_env_step": bstep, "ms_collect": ms_collect, "ms_process_fn": ms_gae, "transitions": n,
           "peak_source": how}
    hbm["frac"] = hbm["achieved"] / hbm["peak"]
    hbm["note"] = ("one fused launch per vector step moves %d B per env: the collect is a chain of T dependent launches, not a bandwidth "
                   "problem at this env count" % (8 * D + 4 * A + 18))
    return roof, hbm


def gae_time(buf, policy, iters=20):
    from fsrl_b200 import ops
    n = buf.maxsize
    v = torch.randn(2, n, device=policy.device); vn = torch.randn(2, n, device=policy.device)
    end = (buf.terminated | buf.truncated)
    adv = torch.empty_like(v); ret = torch.empty_like(v)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=policy.device)
    ts = []
    for i in range(iters + 3):
        flush.zero_()
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(); ops.gae_dual(v, vn, buf.rew, buf.cost, end, buf.terminated, 0.99, 0.95, out=(adv, ret)); e.record()
        torch.cuda.synchronize()
        if i >= 3:
            ts.append(s.elapsed_time(e))
    return float(np.mean(ts)), n


def run_ours(args):
    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(device))
    agent, trainer, col, buf, T = build(cfg, device, rank)
    if world > 1:
        from fsrl_b200 import parallel
        parallel.attach(agent.policy, dist, device=device)
    envs = cfg["envs"]
    steps_per_cycle = envs * T

    for _ in range(args.warmup):
        one_cycle(trainer)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- device-timed region: K collect+update cycles ---------------------------------------------
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    from fsrl_b200 import _lib as _fl
    launches0 = int(_fl.lib.fsrl_launch_count())
    ev0.record()
    collect_s = 0.0
    for _ in range(args.steps):
        c0 = col.collect_time
        stats = one_cycle(trainer)
        collect_s += col.collect_time - c0
    ev1.record()
    torch.cuda.synchronize()
    launches = int(_fl.lib.fsrl_launch_count()) - launches0
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, agent.policy, stats, buf)
    if dist is not None:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    total_steps = steps_per_cycle * args.steps * world
    value = total_steps / (ms * 1e-3)
    # ---- e2e: a SECOND region of K cycles through the public trainer API, wall clock, synchronised on both sides.  Every
    # cycle uploads the minibatch permutations / sampled indices from pinned host memory and downloads the per-minibatch
    # statistics + collect statistics the trainer logs; observations never exist on the host (the environment model runs on
    # the device, SURVEY 8-a2), so these ARE the path's copies.
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t_e2e0 = time.time()
    for _ in range(args.steps):
        one_cycle(trainer)
    torch.cuda.synchronize()
    t_e2e = time.time() - t_e2e0
    if dist is not None:
        t = torch.tensor([t_e2e], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_e2e = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    ranks_identical = None
    if dist is not None:
        # lock-step check: every rank must hold bit-identical parameters after the K + K cycles
        th = agent.policy.arena.theta.detach().contiguous()
        allth = [torch.empty_like(th) for _ in range(world)]
        dist.all_gather(allth, th)
        ranks_identical = all(bool(torch.equal(allth[0].view(torch.int32), x.view(torch.int32))) for x in allth)
        if not ranks_identical and rank == 0:
            for r in range(1, world):
                bad = (allth[0].view(torch.int32) != allth[r].view(torch.int32)).nonzero().flatten()
                if bad.numel():
                    print("rank 0 vs rank %d: %d of %d parameters differ, max |diff| %.3e, first offsets %s; slots %s" % (
                        r, bad.numel(), th.numel(), float((allth[0] - allth[r]).abs().max()), bad[:8].tolist(),
                        [(sl.offset, sl.D, sl.H, sl.out) for sl in agent.policy.arena.slots]), file=sys.stderr, flush=True)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    algo = cfg["algo"]
    if algo == "sacl":
        n_upd = round(cfg["ups"] * steps_per_cycle)
        h2d = n_upd * cfg["batch"] * 4                             # int32 replay indices per gradient step
        d2h = n_upd * 8 * 4 + 64
    else:
        n_mb = max(steps_per_cycle // cfg["batch"], 1)
        h2d = cfg["repeat"] * steps_per_cycle * 4                  # int32 permutation per repeat
        d2h = cfg["repeat"] * n_mb * 8 * 4 + 64                    # per-minibatch stats + collect stats
    e2e_value = total_steps / t_e2e
    pk, how = peaks()
    out = {
        "metric": f"env-steps/sec (collect+update) {cfg['task']} {METRIC[algo]}",
        "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["desc"] + " (analytic on-device env model, random-init weights)",
                   "name": args.config, "envs_per_gpu": envs, "transitions_per_step": steps_per_cycle * world,
                   "parallelism": f"dp{world}",
                   "kl_early_stop": "disabled (fixed work per step)" if algo == "ppol" else "n/a",
                   "l2": "working set per cycle (rollout buffers + per-repeat gathers over all rows) cycles through more "
                         "distinct data than L2 holds between reuses; no explicit flush"},
        "collect_s_per_step": collect_s / args.steps,
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "how": "separate region: K more collect+update cycles through Trainer.train_step / policy_update_fn, wall clock, "
                       "max over ranks; H2D = pinned minibatch permutations (replay indices), D2H = per-minibatch + collect statistics"},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if ranks_identical is not None:
        out["ranks_bit_identical_parameters"] = ranks_identical
    if world > 1:
        # the other ranks are gone: the per-kernel measurements below run on this GPU alone, without the exchange
        agent.policy._dp = None
    if algo == "ppol":
        roof, hbm = ppo_rooflines(cfg, agent, col, buf, T, device, pk, how)
        out["roofline"], out["roofline_hbm"] = roof, hbm
        gms, gn = gae_time(buf, agent.policy)
        out["roofline_gae"] = {"kernel": "gae_dual_kernel<2,true>", "bound": "hbm", "achieved": gn * 42 / (gms * 1e-3) / 1e9,
                               "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gn * 42 / (gms * 1e-3) / 1e9 / pk["hbm_gbs"], "ms": gms,
                               "bytes_per_transition": 42, "transitions": gn, "peak_source": how,
                               "note": "the scan alone, L2 flushed before every launch"}
    else:
        out["roofline"] = other_roofline(cfg, agent, steps_per_cycle, ms / args.steps, collect_s / args.steps, pk, how)
    if world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_reference(args.config, sample_envs=args.cpu_envs, cycles=1)
    print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


DUMP_ROWS = 1 << 16                 # replay rows sampled for --dump-outputs
DUMP_LIMIT = 64 << 20               # bytes


def dump_outputs(out_dir, policy, stats, buf):
    """What a caller of the timed path holds after its last step, as float32 / float64 arrays: the collect statistics
    (collect_*), the update's per-step losses (update_*), the Lagrange multipliers, every network parameter (params)
    and the replay rows the collect wrote (buffer_*; a fixed, seeded sample of DUMP_ROWS rows, the same in every run)."""
    arrays = {"collect_" + k: np.float64(v) for k, v in stats.items()}
    for k, v in policy.last_stats.items():
        v = np.asarray(v)
        arrays["update_" + k] = v if v.dtype == np.float32 else v.astype(np.float64)
    if hasattr(policy, "lagrangians"):
        arrays["lagrangians"] = np.asarray(policy.lagrangians(), np.float64)
    arrays["params"] = policy.arena.theta.detach().float().cpu().numpy()
    rows = np.random.default_rng(0).choice(buf.maxsize, min(DUMP_ROWS, buf.maxsize), replace=False)
    rows = torch.from_numpy(np.sort(rows)).to(buf.device)
    for k in ("obs", "obs_next", "act", "rew", "cost", "logp", "terminated", "truncated"):
        arrays["buffer_" + k] = getattr(buf, k)[rows].float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name.replace("/", "_") + ".npy"), a)


def other_roofline(cfg, agent, steps_per_cycle, ms_cycle, collect_s, pk, how):
    """CPO: Fisher/Hessian-vector products dominate (~ 4 x 2 N P flops each, SURVEY.md 8d); SAC: latency of a gradient step."""
    s0 = agent.policy.arena.slots[0]
    if cfg["algo"] == "cpo":
        P, N = s0.size, steps_per_cycle
        n_hvp = 22 * cfg["repeat"]
        fl = 4 * 2 * N * P * n_hvp
        upd_s = ms_cycle * 1e-3 - collect_s
        ach = fl / upd_s / 1e12
        return {"kernel": "cpo_rfwd/rbwd/rhead (exact KL Hessian-vector products) + CG + line search", "bound": "tensor",
                "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops_sustained"],
                "traffic": None, "peak_source": how + " bf16 sustained",
                "note": f"algorithmic flops = 4 x 2 N P per product, {n_hvp} products per cycle over the whole update time "
                        f"({upd_s * 1e3:.1f} ms; critic regression and line-search forwards included in the time, not in the flops)"}
    n_upd = round(cfg["ups"] * steps_per_cycle)
    upd_s = ms_cycle * 1e-3 - collect_s
    return {"kernel": "fsrl_offpolicy_steps (generic engine, ~22 launches per gradient step)", "bound": "tensor",
            "achieved": None, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": None, "traffic": None,
            "gradient_steps_per_cycle": n_upd, "us_per_gradient_step": upd_s * 1e6 / max(n_upd, 1),
            "note": "latency-bound chain of dependent 256-row gradient steps; reported as time per step"}


# -------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own classes on the host cores (oracle/refarm.py)
# -------------------------------------------------------------------------------------------------
REF_MISSING = "oracle/_ref is missing: __graft_entry__.build() installs it where a checkout of liuzuxin/FSRL is present (FSRL_REFERENCE)"


def _reference_dir():
    from oracle.refarm import REF_DIR
    return REF_DIR if os.path.isdir(os.path.join(REF_DIR, "fsrl")) else None


def cpu_reference(config="c2", sample_envs=32, cycles=1, threads=None, runner=None):
    """One or more collect+update cycles of the UNMODIFIED reference (oracle/_ref): fsrl.data.FastCollector over one worker
    PROCESS per env (tianshou SubprocVectorEnv protocol; the simulator inside a worker is the numpy twin of the device env
    model, pybullet / mujoco being absent), fsrl.policy.PPOLagrangian.process_fn + learn.  c1 runs verbatim (4 envs); the other
    PPO configs run their network / batch shapes on a bounded sample of `sample_envs` envs (one process per env does not
    scale to thousands of envs on any host -- the reference itself tops out at its core count).  CPO / SAC configs report the
    PPO arm of c2's shapes is NOT substituted: they time the oracle port of their own update (kind = "port")."""
    cfg = CONFIGS[config]
    if cfg["algo"] != "ppol":
        return cpu_port_other(cfg, sample_envs)
    ref_dir = _reference_dir()
    if ref_dir is None:
        return {"value": None, "unit": "env-steps/s", "kind": "reference", "unavailable": REF_MISSING}
    from oracle import refarm
    n_env = cfg["envs"] if config == "c1" else min(sample_envs, cfg["envs"])
    threads = threads or 4                                        # the reference's default (ppol_cfg.py:11 thread = 4)
    own = runner is None
    if own:
        runner = refarm.ppo_lag_cycle_runner(ref_dir, cfg["kind"], n_env, cfg["hidden"], cfg["batch"], cfg["repeat"], threads,
                                             workers=True, seed=SEED)
    n = tc = tu = 0.0
    for _ in range(cycles):
        a, b, c = runner()
        n += a; tc += b; tu += c
    if own:
        runner.close()
    return {"value": n / (tc + tu), "unit": "env-steps/s", "cores": os.cpu_count(), "env_worker_processes": n_env,
            "torch_threads": threads, "kind": "reference", "collect_s": tc, "update_s": tu,
            "same_config": config == "c1",
            "sample": f"{n_env} envs x {runner.T} steps x {cycles} cycle(s), {cfg['hidden'][0]}-wide MLPs, batch {cfg['batch']}, "
                      f"repeat {cfg['repeat']}: unmodified fsrl.data.FastCollector + fsrl.policy.PPOLagrangian from oracle/_ref "
                      f"(no fsrl_b200 import), one env worker process per env, torch.set_num_threads({threads}) (reference default); "
                      f"collect {tc:.1f} s + update {tu:.1f} s"}


def cpu_port_other(cfg, sample_envs):
    """CPO / SAC configs: the oracle restatement of the reference update (oracle/cpo.py, oracle/offpolicy.py) on the host
    cores; the reference classes themselves are pinned against these ports in tests/test_oracle_golden.py."""
    return {"value": None, "unit": "env-steps/s", "cores": os.cpu_count(), "kind": "port",
            "sample": "not timed in this run: use --config c1/c2/c5 for the reference arm (PPO-Lagrangian)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    if cfg["algo"] != "ppol":
        print(json.dumps({"impl": "reference", "unavailable": "the CPU reference arm covers the PPO-Lagrangian configs (c1, c2, c5)"}))
        return
    from oracle import refarm
    ref_dir = _reference_dir()
    if ref_dir is None:
        print(json.dumps({"impl": "reference", "unavailable": REF_MISSING}))
        return
    n_env = cfg["envs"] if args.config == "c1" else min(args.cpu_envs, cfg["envs"])
    threads = 4
    runner = refarm.ppo_lag_cycle_runner(ref_dir, cfg["kind"], n_env, cfg["hidden"], cfg["batch"], cfg["repeat"], threads,
                                         workers=True, seed=SEED)
    for _ in range(args.warmup):
        runner()
    t0 = time.time()
    last = None
    for _ in range(args.steps):
        last = cpu_reference(args.config, sample_envs=args.cpu_envs, cycles=1, threads=threads, runner=runner)
    dt = time.time() - t0
    runner.close()
    n = args.steps * n_env * runner.T
    v = n / dt
    cb = dict(last); cb["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": f"env-steps/sec (collect+update) {cfg['task']} {METRIC[cfg['algo']]}",
        "value": v, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["desc"] + f" -- on the host cores: {n_env} envs per step"
                               + (" (verbatim)" if args.config == "c1" else " (bounded sample of the config's env count; same networks, "
                                  "batch size and repeats)"), "name": args.config},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--cpu-envs", type=int, default=32,
                    help="envs (= worker processes) of the bounded CPU sample for configs other than c1")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    a = ap.parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
