#!/usr/bin/env python
"""Environments at different points of their episodes (m3pc_plan env_horizons, evaluate_plan refill), walker2d shapes,
critic_lambda_guiding, 1024 candidates, bf16.

1. Plan latency of E = 8 environments: uniform h = 4 against the horizon patterns of environments in their first T - h steps
   (graph replay, CUDA events around each call), with launches per plan.
2. evaluate_plan wall time for 32 episodes on 8 slots: LinearEnv stand-ins whose lengths spread over 100..1000 steps, each
   step costing `step_cost_s` of host time like a physics step; lock-step rounds (refill=False) against refilled slots.

    python tools/episode_slots_bench.py [--plans 200] [--episodes 32] [--step-cost-us 100] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from m3pc_b200 import rollout as ro  # noqa: E402
from test_rollout import _gpu_learner  # noqa: E402  (the Learner construction the rollout tests use)

PATTERNS = {"uniform h=4": [4] * 8, "[8,4,4,4,4,4,4,4]": [8, 4, 4, 4, 4, 4, 4, 4], "[8,7,6,5,4,4,4,4]": [8, 7, 6, 5, 4, 4, 4, 4]}


def plan_latency(n_plans):
    E, N = 8, 1024
    shape, L = _gpu_learner("bf16", N, E)
    eng = L._engine()
    T = shape.traj_length
    g = torch.Generator(device="cuda").manual_seed(0)
    ws = torch.randn(E, T, shape.obs_dim, device="cuda", generator=g)
    wa = torch.rand(E, T, shape.act_dim, device="cuda", generator=g) * 2 - 1
    wr, wt = torch.randn(E, T, device="cuda", generator=g), torch.randn(E, T, device="cuda", generator=g)
    out = {}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, hz in PATTERNS.items():
        h = max(hz)
        call = lambda s: eng.plan(guidance="critic_lambda_guiding", horizon=h, n_cand=N, win_states=ws, win_actions=wa, win_rewards=wr,  # noqa: E731
                                  win_returns_tok=wt, discount=0.99, temperature=1.0, lmbda=0.6, seed=s, n_env=E,
                                  env_horizons=None if min(hz) == h else hz)
        for s in range(10):  # eager, capture, replays
            call(s)
        torch.cuda.synchronize()
        times = []
        for s in range(n_plans):
            ev0.record()
            call(100 + s)
            ev1.record()
            ev1.synchronize()
            times.append(ev0.elapsed_time(ev1))
        t = np.array(times)
        out[name] = {"p50_ms": float(np.median(t)), "p10_ms": float(np.percentile(t, 10)), "p90_ms": float(np.percentile(t, 90)),
                     "launches": eng.last_launch_count()}
        print(f"plan E=8 {name:>20}: p50 {out[name]['p50_ms']:.3f} ms (p10 {out[name]['p10_ms']:.3f}, p90 {out[name]['p90_ms']:.3f}), "
              f"{out[name]['launches']} launches", flush=True)
    return out


def rollout_wall(n_episodes, step_cost_s, groups):
    E = 8
    shape, L = _gpu_learner("bf16", 1024, E)
    rs = np.random.RandomState(0)
    lengths = rs.randint(100, 1001, size=n_episodes).tolist()
    res = {"episode_lengths": lengths}
    ro.evaluate_plan(L, lambda: ro.LinearEnv(shape.obs_dim, shape.act_dim, seed=1, horizon=12), num_episodes=E, episode_rtg_ref=np.full(1000, 3.0),
                     n_envs=E, groups=groups, max_path_length=1000, refill=True)  # warm-up: captures the graphs of the early patterns
    for refill in (False, True):
        count = [0]

        def make_env():
            i = count[0]
            count[0] += 1
            return ro.LinearEnv(shape.obs_dim, shape.act_dim, seed=i, horizon=lengths[i], step_cost_s=step_cost_s)

        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = ro.evaluate_plan(L, make_env, num_episodes=n_episodes, episode_rtg_ref=np.full(1000, 3.0), n_envs=E, groups=groups,
                               max_path_length=1000, refill=refill)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        steps = int(sum(out["lengths"]))
        key = "refill" if refill else "lock_step"
        res[key] = {"wall_s": dt, "env_steps": steps, "steps_per_s": steps / dt}
        print(f"evaluate_plan {n_episodes} episodes on {E} slots ({groups} groups), refill={refill}: {dt:.2f} s, {steps} env steps, "
              f"{steps / dt:.0f} steps/s", flush=True)
    res["speedup"] = res["lock_step"]["wall_s"] / res["refill"]["wall_s"]
    rounds = [lengths[i:i + E] for i in range(0, n_episodes, E)]
    res["ideal_speedup"] = sum(max(r) for r in rounds) * E / sum(lengths)  # slot-steps of lock-step rounds over env steps
    print(f"refill speedup {res['speedup']:.2f}x (slot-step bound {res['ideal_speedup']:.2f}x)", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--plans", type=int, default=200)
    ap.add_argument("--episodes", type=int, default=32)
    ap.add_argument("--step-cost-us", type=float, default=100.0, help="host time per environment step (emulated physics)")
    ap.add_argument("--groups", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    print(f"device: {gpu}", flush=True)
    res = {"device": gpu, "plan": plan_latency(args.plans),
           "rollout": rollout_wall(args.episodes, args.step_cost_us * 1e-6, args.groups), "step_cost_us": args.step_cost_us}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
