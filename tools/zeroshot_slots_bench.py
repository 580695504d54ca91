#!/usr/bin/env python
"""Zero-shot (backward) planners on environments at different points of their episodes: hopper shapes, E = 256 environments,
id and piid, bf16 (BASELINE.json config 4).

1. Device time per call (CUDA events around each call) and launches per call (m3pc_last_launch_count) at C = 512 action draws and
   at C = 1: a lock-step batch (every environment at h = 4) against a batch where a quarter of the environments are in their
   first T - h steps (horizons 8, 7, 6, 5; five horizon classes in all).
2. A refill run (evaluate_plan, refill=True, device-resident histories, one group) over LinearEnv stand-ins with waypoint tables:
   every plan of the run timed the same way (one action per environment, C = 1), with the horizon classes it held.

    python tools/zeroshot_slots_bench.py [--calls 50] [--episodes 768] [--out FILE.json]
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
from test_zeroshot_slots import _zs_learner  # noqa: E402  (the Learner construction the zero-shot slot tests use)

E, C = 256, 512
QUARTER = [8, 7, 6, 5] * (E // 16) + [4] * (3 * E // 4)  # a quarter of the slots in their first T - h steps (T = 8, h = 4)


def _stats(times):
    t = np.array(times)
    return {"p50_ms": float(np.median(t)), "p10_ms": float(np.percentile(t, 10)), "p90_ms": float(np.percentile(t, 90)), "calls": len(t)}


def per_call(L, n_calls):
    eng = L._engine()
    shape_T, obs, act = L.cfg.traj_length, eng.obs, eng.act
    g = torch.Generator(device="cuda").manual_seed(0)
    ws = torch.randn(E, shape_T, obs, device="cuda", generator=g)
    wa = torch.rand(E, shape_T, act, device="cuda", generator=g) * 2 - 1
    wr, wt = torch.randn(E, shape_T, device="cuda", generator=g), torch.randn(E, shape_T, device="cuda", generator=g)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = {}
    for mode in ("id", "piid"):
        for n_draws in (C, None):
            for name, hz in (("lock-step h=4", [4] * E), ("quarter in first T-h steps", QUARTER)):
                h = max(hz)
                call = lambda s: eng.backward_plan(mode=mode, horizon=h, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt,  # noqa: E731
                                                   n_draws=n_draws, seed=s, env_horizons=None if min(hz) == h else hz)
                for s in range(5):
                    call(s)
                torch.cuda.synchronize()
                times = []
                for s in range(n_calls):
                    ev0.record()
                    call(100 + s)
                    ev1.record()
                    ev1.synchronize()
                    times.append(ev0.elapsed_time(ev1))
                key = f"{mode} C={n_draws or 1} {name}"
                out[key] = dict(_stats(times), launches=eng.last_launch_count(), classes=len(set(hz)))
                print(f"{key:>40}: p50 {out[key]['p50_ms']:.3f} ms (p10 {out[key]['p10_ms']:.3f}, p90 {out[key]['p90_ms']:.3f}), "
                      f"{out[key]['launches']} launches, {out[key]['classes']} horizon classes", flush=True)
    return out


def refill_run(L, n_episodes):
    """evaluate_plan over LinearEnv stand-ins whose lengths spread over 20..80 steps, waypoints from a seeded table per episode;
    every backward plan of the run bracketed by CUDA events (read after the run)."""
    eng = L._engine()
    obs, act = eng.obs, eng.act
    lengths = np.random.RandomState(0).randint(20, 81, size=n_episodes).tolist()
    res = {}
    for mode in ("id", "piid"):
        marks = []
        inner = L._backward_device

        def timed(mode_, horizons, *a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = inner(mode_, horizons, *a, **kw)
            e1.record()
            marks.append((e0, e1, eng.last_launch_count(), len(set(horizons))))
            return r

        L._backward_device = timed
        count = [0]

        def make_env():
            i = count[0]
            count[0] += 1
            return ro.LinearEnv(obs, act, seed=i, horizon=lengths[i])

        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = ro.evaluate_plan(L, make_env, num_episodes=n_episodes, episode_rtg_ref=np.full(1000, 3.0), n_envs=E, groups=1,
                                   max_path_length=1000, refill=True, device_histories=True,
                                   waypoints=lambda i: np.random.RandomState(10_000 + i).randn(1000, obs).astype(np.float32), zeroshot_mode=mode)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
        finally:
            del L._backward_device
        steps = int(sum(out["lengths"]))
        by = {}
        for e0, e1, n, k in marks[3:]:  # the first plans load modules
            by.setdefault(k, []).append((e0.elapsed_time(e1), n))
        res[mode] = {"wall_s": wall, "env_steps": steps, "plans": len(marks), "episodes": n_episodes,
                     "by_classes": {str(k): dict(_stats([t for t, _ in v]), launches_max=max(n for _, n in v)) for k, v in sorted(by.items())}}
        print(f"refill {mode}: {n_episodes} episodes on {E} slots, {len(marks)} plans, {steps} env steps, {wall:.2f} s wall", flush=True)
        for k, v in res[mode]["by_classes"].items():
            print(f"    {k} horizon classes: {v['calls']} plans, p50 {v['p50_ms']:.3f} ms (p90 {v['p90_ms']:.3f}), up to {v['launches_max']} launches",
                  flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--episodes", type=int, default=768)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    print(f"device: {gpu}", flush=True)
    _, L = _zs_learner("bf16", E)
    res = {"device": gpu, "E": E, "C": C, "per_call": per_call(L, args.calls), "refill": refill_run(L, args.episodes)}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
