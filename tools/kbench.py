"""Kernel micro-benchmarks (CUDA events on the launching stream, L2 flushed between
iterations).  Usage: python tools/kbench.py gae [--envs 2048 --T 300]"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsrl_b200 import ops  # noqa: E402
from fsrl_b200.utils.synth import synth_gae_inputs  # noqa: E402


def peaks():
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def time_kernel(fn, iters=20, warmup=5, flush=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    return float(np.mean(ts)), float(np.min(ts))


def bench_gae(envs, T):
    d = synth_gae_inputs(envs, T, seed=10)
    N = envs * T
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    v, vn, r, c = dev(d["v"]), dev(d["vnext"]), dev(d["rew"]), dev(d["cost"])
    end = dev((d["terminated"] | d["truncated"]).astype(np.uint8))
    term = dev(d["terminated"].astype(np.uint8))
    adv = torch.empty_like(v); ret = torch.empty_like(v)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    fn = lambda: ops.gae_dual(v, vn, r, c, end, term, 0.99, 0.95, out=(adv, ret))
    mean_ms, min_ms = time_kernel(fn, flush=flush)
    alg_bytes = N * (16 * 2 + 10)   # SURVEY.md 8(d): 16*C + 10 B / transition (+1 B terminated)
    pk, how = peaks()
    gbs = alg_bytes / (mean_ms * 1e-3) / 1e9
    print(json.dumps({"kernel": "gae_dual", "N": N, "ms_mean": mean_ms, "ms_min": min_ms,
                      "alg_bytes": alg_bytes, "GBps": gbs, "frac_of_%s_hbm" % how: gbs / pk["hbm_gbs"]}))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["gae"])
    ap.add_argument("--envs", type=int, default=2048)
    ap.add_argument("--T", type=int, default=300)
    a = ap.parse_args()
    if a.what == "gae":
        bench_gae(a.envs, a.T)
        bench_gae(a.envs * 16, a.T)
