#!/usr/bin/env python
"""bench.py -- M^3PC plans/sec on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--mode env|cand] [--envs E]
                    [--dump-outputs DIR]

A plan is one pass of the hot path (pass 1, candidate sampling, pass 2 at B=candidates, critic / return scoring, softmax
selection) for one environment state.  A "step" plans ``--envs`` E lock-step environments (default 8, each with its own
history window and its own 1024 candidates) in ONE ``m3pc_plan`` launch sequence -- E plans per step; ``value`` counts plans.
The reference's call shape (one window per call, E = 1) is always measured too and reported under ``single_env`` with its
p50 latency.  Default workload = BASELINE.json configs[1]: walker2d shapes (obs 17 / act 6), critic_lambda_guiding, 1024
candidates per plan, horizon 4, shipped MTM (D=512, 4 heads, 2+1 layers, T=8), random-init weights, synthetic histories.

  value     device-resident throughput: window already in HBM, K plans timed with CUDA events (one event pair per plan on
            the launching stream; a 256 MiB L2 flush between plans sits outside the pairs), max over ranks.
  e2e       the same K steps through the public API ``Learner.action_sample_batch`` (``action_sample`` at E = 1) with HOST numpy
            histories: window building, one pinned H2D of the E windows and a D2H read of the E actions inside the timed
            region (host wall clock, max over ranks).
  roofline  tensor-core GEMMs (the dominant kernel): algorithmic FLOPs of the GEMM launches / their summed per-launch
            CUDA-event time in a profiling pass of the same plan, against MEASURED_PEAKS.json (sustained bf16).
  cpu_baseline  the oracle port of the reference planner (torch CPU fp32, all host threads), same workload, bounded sample.

``--dump-outputs DIR`` writes what the timed device-resident path returned in its last timed step -- the eval and sample
actions, (E, A) -- as ``DIR/<name>.npy`` (float32; the one-window call's under ``single_env_*``).  Weights, histories and
noise seeds are fixed, so two builds run with the same arguments can be compared output for output.

Multi-GPU (launched by torchrun, one rank per GPU): ``--mode env`` (default) gives every rank its own environment --
independent plans, no data-path collective, weak scaling; ``--mode cand`` shards the candidates of ONE plan across
ranks (BASELINE.json configs[2]) with one NCCL all-gather of a 72-float record per plan.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: env, guidance, candidates, temperature, model
    "walker2d_critic_1024": dict(env="walker2d", guidance="critic_lambda_guiding", n_cand=1024, temperature=1.0, model="shipped"),
    "hopper_rtg_625": dict(env="hopper", guidance="rtg_guiding", n_cand=625, temperature=0.01, model="shipped"),
    "hopper_rtg_1024": dict(env="hopper", guidance="rtg_guiding", n_cand=1024, temperature=0.01, model="shipped"),
    "halfcheetah_rtg_16384": dict(env="halfcheetah", guidance="rtg_guiding", n_cand=16384, temperature=0.01, model="shipped"),
    "scaled_rtg_4096": dict(env="hopper", guidance="rtg_guiding", n_cand=4096, temperature=0.01, model="scaled"),
}
METRIC = "plans_per_sec"
_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's real stdout (everything else -- NCCL's version banner, library
    chatter -- was redirected to stderr in main())."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()
UNIT = "plans/s"


def model_shape(w):
    from m3pc_b200 import synthetic as syn
    return syn.scaled_shape(w["env"]) if w["model"] == "scaled" else syn.shipped_shape(w["env"])


def flops_per_plan(shape, n_cand, guidance, h):
    """Dense algorithmic FLOPs of one plan (SURVEY.md 8d): pass-2 rows (fd mask) + one pass-1 row (rcbc mask) + critic."""
    D, T, F = shape.n_embd, shape.traj_length, 4 * shape.n_embd
    idx = T - h

    def block(S):
        return 2 * S * D * 3 * D + 4 * S * S * D + 2 * S * D * D + 4 * S * D * F

    def fwd(S_enc):
        emb = 2 * sum(shape.feature_dims.values()) * D * T
        dec_embed = 2 * 4 * T * D * D
        heads = 3 * T * (2 * D * D) + 2 * T * D * (shape.obs_dim + 2) + 2 * 2 * T * D * shape.act_dim
        return emb + shape.n_enc_layer * block(S_enc) + dec_embed + shape.n_dec_layer * block(4 * T) + heads

    s_fd, s_rcbc = (idx + 1) + T, (idx + 1) + idx + T
    total = n_cand * fwd(s_fd) + fwd(s_rcbc)
    if guidance != "rtg_guiding":
        total += n_cand * h * 2 * 2 * ((shape.obs_dim + shape.act_dim) * 256 + 256 * 256 + 256)
    return float(total), float(fwd(s_fd))


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip().split(", "))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        busy = [c for c in sm if c > 0.5 * mx] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arms
def cpu_planner(w, shape):
    """(planner, kind): the UNMODIFIED reference ``Learner`` (oracle/_ref staged by oracle/stage_ref.py, or /root/reference in
    the dev container) -> kind "reference"; only if neither exists, the oracle port -> kind "port"."""
    import torch
    from m3pc_b200 import synthetic as syn
    from oracle import ref_harness as rh
    if rh.available():
        return rh.build_learner(shape, guidance=w["guidance"], n_cand=w["n_cand"], temperature=w["temperature"], device="cpu"), "reference"
    from oracle import planner_oracle as po
    crit = w["guidance"] != "rtg_guiding"
    P = po.from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), dtype=torch.float32,
                          critic_np=syn.make_critic_state_dict(shape) if crit else None, obs_norm=syn.make_obs_norm(shape) if crit else None,
                          action_samples=w["n_cand"], temperature=w["temperature"], plan_guidance=w["guidance"])
    return P, "port"


def time_cpu(w, shape, steps, warmup, budget_s=None):
    """``Learner.action_sample(history, plan=True, eval=True, rtg=3.0)`` (research/finetune_omtm/learner.py:329-417) on the host
    cores, all threads; returns (plans/s, per-plan seconds, threads, kind)."""
    import numpy as np
    import torch
    from m3pc_b200 import synthetic as syn
    torch.set_num_threads(os.cpu_count() or 1)
    P, kind = cpu_planner(w, shape)
    T, A, N = shape.traj_length, shape.act_dim, w["n_cand"]
    rs = np.random.RandomState(7)
    times = []
    t_start = time.perf_counter()
    for i in range(warmup + steps):
        hist = syn.make_history(shape, seed=100 + i, path_length=50)
        if kind == "port":
            kw = dict(eps=torch.from_numpy(rs.randn(N, 1, T, 1, A).astype(np.float32)), q=torch.from_numpy(rs.exponential(1.0, N).astype(np.float32)))
        else:
            kw = {}  # the reference draws its own noise from torch's generator
        t0 = time.perf_counter()
        with torch.no_grad():
            P.action_sample(hist, plan=True, eval=True, rtg=3.0, **kw)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        if budget_s is not None and i >= warmup and time.perf_counter() - t_start > budget_s:
            break
    return len(times) / sum(times), times, torch.get_num_threads(), kind


def _kind_text(kind):
    return ("UNMODIFIED reference Learner.action_sample from oracle/_ref" if kind == "reference" else
            "oracle port of Learner.action_sample (the reference is not staged on this box)")


def time_gpu_library(w, shape, dev, steps=12, warmup=3):
    """The "stock PyTorch on the same B200" bar (SURVEY.md section 8d "Also time"): the UNMODIFIED reference objects moved to
    the GPU (``cfg.device = "cuda"``, finetune.py:154) -- cuBLAS / ATen library kernels, one plan per call as the reference
    runs it -- in fp32, with TF32 matmuls allowed, and under bf16 autocast.  CUDA events around each plan (the call ends in
    the device-side selection; the host sync the caller's ``.cpu()`` adds is not counted).  Returns None when the reference
    is not staged."""
    import torch
    from m3pc_b200 import synthetic as syn
    from oracle import ref_harness as rh
    if not rh.available():
        return None
    L = rh.build_learner(shape, guidance=w["guidance"], n_cand=w["n_cand"], temperature=w["temperature"], device=str(dev))
    hists = [syn.make_history(shape, seed=100 + i, path_length=50) for i in range(steps + warmup)]
    out = {"api": "research.finetune_omtm.learner.Learner.action_sample(device='cuda'), one plan per call (the reference has no "
                  "multi-environment call)", "unit": UNIT, "plans_timed": steps}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)

    def run(mode):
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = mode == "tf32"
        ms = []
        for i, hist in enumerate(hists):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=mode == "bf16_autocast"):
                L.action_sample(hist, plan=True, eval=True, rtg=3.0)
            e1.record()
            torch.cuda.synchronize()
            if i >= warmup:
                ms.append(e0.elapsed_time(e1))
        return {"value": 1e3 * len(ms) / sum(ms), "p50_ms": statistics.median(ms)}

    try:
        for mode in ("fp32", "tf32", "bf16_autocast"):
            try:
                out[mode] = run(mode)
            except Exception as exc:  # a library path that does not run under this mode is reported, not hidden
                out[mode] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    return out


def run_reference(args, w, shape, rank):
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    val, times, threads, kind = time_cpu(w, shape, steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times), "warmup": warmup,
        "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": args.workload, "candidates": w["n_cand"], "horizon": 4, "guidance": w["guidance"], "env_shapes": w["env"],
                   "model": f"D={shape.n_embd},heads={shape.n_head},enc={shape.n_enc_layer},dec={shape.n_dec_layer},T={shape.traj_length}",
                   "plans_per_step": 1, "step": "one window per plan (Learner.action_sample), the reference's only call shape"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"{len(times)} full plans ({_kind_text(kind)}, torch CPU fp32, {threads} threads of {os.cpu_count()} host cpus)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "p50_ms": 1e3 * statistics.median(times),
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ ours
def dump_outputs(out_dir, arrays):
    """``out_dir/<name>.npy`` (float32) for every tensor of ``arrays``."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def build_learner(w, shape, n_local, E, dev, args, cand_offset=0):
    import torch
    from m3pc_b200 import synthetic as syn
    from m3pc_b200.learner import Learner
    from m3pc_b200.mtm_model import omtmConfig
    from m3pc_b200.tokenizers import manager_from_stats
    crit = w["guidance"] != "rtg_guiding"
    cfg = SimpleNamespace(traj_length=shape.traj_length, device=str(dev), action_samples=n_local, discount=0.99, temperature=w["temperature"],
                          horizon=4, plan_guidance=w["guidance"], lmbda=0.6)
    mcfg = omtmConfig(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer, dropout=0.1,
                      norm="none", precision=args.precision, max_batch=n_local * max(1, E), chunk=args.chunk)
    om, os_ = syn.make_obs_norm(shape)
    L = Learner(cfg, None, shape.data_shapes, mcfg, None, om, os_, manager_from_stats(syn.make_tokenizer_stats(shape, 1)),
                {k: False for k in shape.data_shapes}, max_envs=max(1, E))
    L.mtm.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 0).items()})
    if crit:
        L.iql.qf.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_critic_state_dict(shape).items()})
    L.seed, L.cand_offset = 1234, cand_offset
    return L


def measure(L, w, shape, E, K, W, dev, flush, barrier, hist_base=1000, shard=None):
    """K timed steps of E lock-step environments each (E = 1: the reference's one-window call), device-resident and e2e.
    ``shard = (lo, hi)``: this rank plans candidates [lo, hi) of ONE shared plan and the select kernel exchanges + merges the
    shard records over peer memory (``exchange=True``)."""
    import torch
    from m3pc_b200 import synthetic as syn
    eng = L._engine()
    h, T, A, obs = 4, shape.traj_length, shape.act_dim, shape.obs_dim
    n_local = int(L.cfg.action_samples)
    lo = shard[0] if shard else 0
    pool = [syn.make_history(shape, seed=hist_base + j) for j in range(61)]  # distinct episodes; every (step, env) reads a different window of one
    hists = [[dict(pool[(i * E + e) % 61], path_length=50 + (i * E + e) % 900) for e in range(E)] for i in range(K + W)]
    windows = []  # windows resident in HBM (built by the same host code the public API uses)
    for hs in hists:
        ring, slot = L._window_buffers(obs, A, n_env=E)
        for e, hist in enumerate(hs):
            v = (slot.h_states, slot.h_actions, slot.h_rewards, slot.h_returns) if E == 1 else \
                (slot.h_states[e], slot.h_actions[e], slot.h_rewards[e], slot.h_returns[e])
            L._fill_window(*v, hist, h, 1.0, 3.0)
        windows.append(slot.host.to(dev))
    cur = torch.empty_like(windows[0])
    o = [0, E * T * obs, E * T * (obs + A), E * T * (obs + A + 1), cur.numel()]
    lead = (E,) if E > 1 else ()
    cur_views = (cur[o[0]:o[1]].view(*lead, T, obs), cur[o[1]:o[2]].view(*lead, T, A), cur[o[2]:o[3]].view(*lead, T), cur[o[3]:o[4]].view(*lead, T))

    def plan_resident(i):
        # the windows are already in HBM; they are copied (E x 800 B, device to device) into the buffer the engine's CUDA graph reads
        cur.copy_(windows[i % len(windows)], non_blocking=True)
        ws, wa, wr, wt = cur_views
        ev, sm, _ = eng.plan(guidance=w["guidance"], horizon=h, n_cand=n_local, win_states=ws, win_actions=wa, win_rewards=wr,
                             win_returns_tok=wt, discount=0.99, temperature=w["temperature"], lmbda=0.6, seed=7 + i, cand_offset=lo,
                             n_env=E, exchange=shard is not None)
        return ev, sm

    # ---- device-resident timing: K steps, one CUDA-event pair each, L2 flushed between steps ----
    for i in range(W):
        plan_resident(i)
    torch.cuda.synchronize(); barrier()
    pairs = []
    t_wall0 = time.perf_counter()
    for i in range(K):
        flush.fill_(float(i))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = plan_resident(W + i)
        e1.record()
        pairs.append((e0, e1))
    torch.cuda.synchronize(); barrier()
    wall_resident = time.perf_counter() - t_wall0
    outputs = {"eval_action": last[0].clone(), "sample_action": last[1].clone()}  # engine-owned: the next plan overwrites them
    per_step_ms = [a.elapsed_time(b) for a, b in pairs]
    launches = eng.last_launch_count()

    # ---- e2e: public API with host histories (pinned H2D + D2H inside the timed region) ----
    def api_step(i):
        if shard is not None:
            ring, slot = L._window_buffers(obs, A)
            L._fill_window(slot.h_states, slot.h_actions, slot.h_rewards, slot.h_returns, hists[i][0], h, 1.0, 3.0)
            L._upload_window(ring, slot)
            ev, _, _ = eng.plan(guidance=w["guidance"], horizon=h, n_cand=n_local, win_states=ring.d_states, win_actions=ring.d_actions,
                                win_rewards=ring.d_rewards, win_returns_tok=ring.d_returns, discount=0.99, temperature=w["temperature"],
                                lmbda=0.6, seed=7 + i, cand_offset=lo, exchange=True)
            return ev.cpu()
        if E == 1:
            return L.action_sample(hists[i][0], plan=True, eval=True, rtg=3.0).cpu()
        return L.action_sample_batch(hists[i], plan=True, eval=True, rtg=3.0).cpu()

    for i in range(W):
        api_step(i)
    torch.cuda.synchronize(); barrier()
    t0 = time.perf_counter()
    lat = []
    for i in range(K):
        t1 = time.perf_counter()
        api_step(W + i)
        lat.append(time.perf_counter() - t1)
    torch.cuda.synchronize(); barrier()
    e2e_s = time.perf_counter() - t0
    return SimpleNamespace(E=E, dev_s=sum(per_step_ms) / 1e3, per_step_ms=per_step_ms, wall=wall_resident, launches=launches, e2e_s=e2e_s,
                           lat=lat, plan_resident=plan_resident, outputs=outputs)


def measure_cand_shard(args, dev, rank, world, flush, barrier, reduce_max, K, W):
    """BASELINE.json configs[2] on the driver's own scaling run: ONE halfcheetah rtg plan of 16 384 candidates sharded over the
    `world` GPUs of the node (rank g owns [lo, hi); pass 1 replicated; Philox noise keyed by global candidate id), the shard
    records exchanged + merged inside the select kernel over NVLink peer memory.  Strong scaling; rank 0 also times the same
    plan unsharded on its GPU alone so the line carries its own denominator."""
    import torch
    from m3pc_b200 import dist as mdist
    name = "halfcheetah_rtg_16384"
    w = WORKLOADS[name]
    shape = model_shape(w)
    n_total = w["n_cand"]
    lo, hi = mdist.shard_range(n_total, rank, world)
    L = build_learner(w, shape, hi - lo, 1, dev, args, cand_offset=lo)
    nbytes = mdist.broadcast_parameters(L.mtm) if world > 1 else 0
    if world > 1:
        mdist.connect_exchange(L._engine())
    m = measure(L, w, shape, 1, K, W, dev, flush, barrier, hist_base=5000, shard=(lo, hi) if world > 1 else None)
    dev_s, e2e_s = reduce_max([m.dev_s, m.e2e_s])
    out = {"workload": name, "candidates": n_total, "ranks": world, "scaling": "strong", "value": K / dev_s, "unit": UNIT,
           "ms_per_step": 1e3 * dev_s / K, "e2e_value": K / e2e_s, "p50_latency_ms_e2e": 1e3 * statistics.median(m.lat),
           "launches_per_plan": m.launches, "steps": K,
           "collective": ("none (one GPU)" if world == 1 else
                          "in-kernel: select_kernel stores the 8+2A-float shard record into every rank's exchange buffer over NVLink peer "
                          "memory (CUDA IPC), release/acquire flags, log-sum-exp merge -- inside the plan's CUDA graph, no NCCL launch"),
           "weights": f"one flat broadcast of {nbytes} bytes from rank 0 at load" if world > 1 else "loaded locally"}
    if world > 1:
        ep, bad = L._engine().exchange_status()
        out["exchange_epochs"], out["exchange_timeouts"] = ep, int(bad != 0)
        # the same plan, unsharded, on rank 0's GPU alone (the other ranks idle at the barrier): the denominator of the efficiency
        n1 = None
        if rank == 0:
            L1 = build_learner(w, shape, n_total, 1, dev, args)
            m1 = measure(L1, w, shape, 1, min(K, 20), 3, dev, flush, lambda: None, hist_base=5000)
            n1 = min(K, 20) / m1.dev_s
        barrier()
        if rank == 0:
            out["n1_value_same_run"] = n1
            out["efficiency_vs_n1_same_run"] = out["value"] / (world * n1)
    return out, m.outputs


def run_ours(args, w, shape, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from m3pc_b200 import dist as mdist

    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    h, T, A = 4, shape.traj_length, shape.act_dim
    n_total = w["n_cand"]
    cand_mode = args.mode == "cand" and world > 1
    K, W = args.steps, args.warmup
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)

    def reduce_max(vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    if cand_mode:  # explicit --mode cand: the candidate-sharded plan IS the headline of this run
        cs, outputs = measure_cand_shard(args, dev, rank, world, flush, barrier, reduce_max, K, W)
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        if rank == 0:
            emit({"metric": METRIC, "value": cs["value"], "unit": UNIT, "n_gpus": world, "steps": cs["steps"], "warmup": W,
                  "ms_per_step": cs["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
                  "data": "synthetic", "config": {"workload": cs["workload"], "parallelism": f"cand-shard x{world}", "collective": cs["collective"]},
                  "e2e": {"value": cs["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": 4 * 8 * (17 + 6 + 2), "d2h_bytes_per_step": 4 * 6},
                  "gpu_launches": cs["launches_per_plan"] * cs["steps"], "cand_shard": cs})
        return

    E_head = max(1, args.envs)
    L = build_learner(w, shape, n_total, E_head, dev, args)
    weights_note = "random-init (numpy seed 0), reference state_dict layout"
    if world > 1:
        nb = mdist.broadcast_parameters(L.mtm)
        weights_note += f"; one flat NCCL broadcast of {nb} bytes from rank 0 at load"
    eng = L._engine()
    torch.cuda.synchronize(); barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    base = 1000 + rank * 10007  # every rank plans for its own environment(s)
    single = measure(L, w, shape, 1, K, W, dev, flush, barrier, hist_base=base)  # the reference's call shape: one window per plan
    head = measure(L, w, shape, E_head, K, W, dev, flush, barrier, hist_base=base) if E_head > 1 else single
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        outputs = dict(head.outputs)
        if E_head > 1:
            outputs.update({f"single_env_{k}": v for k, v in single.outputs.items()})
        dump_outputs(args.dump_outputs, outputs)

    # ---- roofline pass: same step with one event pair per GEMM launch ----
    eng.set_profile(True)
    g_ms, g_fl, g_n = 0.0, 0.0, 0
    for i in range(3):
        head.plan_resident(W + i)
        torch.cuda.synchronize()
        ms, fl, n = eng.get_profile()
        g_ms, g_fl, g_n = g_ms + ms, g_fl + fl, g_n + n
    eng.set_profile(False)

    dev_s, e2e_s, wall_resident, single_dev_s, single_e2e_s = reduce_max([head.dev_s, head.e2e_s, head.wall, single.dev_s, single.e2e_s])
    plans_per_step = E_head * world
    value = plans_per_step * K / dev_s
    e2e_value = plans_per_step * K / e2e_s

    # ---- the north-star's own target config (BASELINE configs[0] shapes): hopper, rtg_guiding, the shipped 625 candidates ----
    ns = None
    if args.workload != "hopper_rtg_625" and not args.lean:
        wn = WORKLOADS["hopper_rtg_625"]
        shn = model_shape(wn)
        Ln = build_learner(wn, shn, wn["n_cand"], E_head, dev, args)
        Kn = min(K, 50)
        s1 = measure(Ln, wn, shn, 1, Kn, 3, dev, flush, barrier, hist_base=base + 77)
        s8 = measure(Ln, wn, shn, E_head, Kn, 3, dev, flush, barrier, hist_base=base + 77) if E_head > 1 else s1
        r = reduce_max([s1.dev_s, s1.e2e_s, s8.dev_s, s8.e2e_s])
        ns = {"workload": "hopper_rtg_625", "candidates": 625, "guidance": "rtg_guiding", "unit": UNIT,
              "single_env": {"value": world * Kn / r[0], "e2e_value": world * Kn / r[1], "p50_ms_device": statistics.median(s1.per_step_ms),
                             "p50_latency_ms_e2e": 1e3 * statistics.median(s1.lat)},
              "envs_per_gpu": E_head, "value": world * E_head * Kn / r[2], "e2e_value": world * E_head * Kn / r[3]}
        del Ln

    # ---- candidate-sharded config 3 rides along on every multi-GPU run, so the driver's scaling file records the collective ----
    cs = None
    if not args.lean and (world > 1 or args.cand_shard):
        del L, eng  # free the workspaces of the head workload first
        torch.cuda.empty_cache()
        cs, _ = measure_cand_shard(args, dev, rank, world, flush, barrier, reduce_max, min(K, 50), 5)  # bounded side measurement
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback (B200_PROFILING.md sustained)"
    gemm_kernel = "gemm_bf16_2sm_kernel + gemm_ln_2sm_kernel (tcgen05 cta_group::2; the latter carries the residual add and the LayerNorm)"
    if args.precision == "fp32":
        # the fp32 mode runs its GEMMs on the FFMA pipe (sgemm.cu): its ceiling is SMs x 128 lanes x 2 flop x the SM clock under load
        mhz = float((clocks or {}).get("sm_mhz") or 1965.0)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        peak_tf = sms * 128 * 2 * mhz * 1e6 / 1e12
        peak_src = f"computed: {sms} SMs x 128 FFMA lanes x 2 x {mhz:.0f} MHz (the fp32 path does not use tensor cores)"
        gemm_kernel = "sgemm128_kernel (fp32 FFMA, 128x128x16 tiles, 8x8 outputs per thread; reference-grade precision mode, not the headline path)"
    ach_tf = g_fl / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    fl_plan, fl_row = flops_per_plan(shape, n_total, w["guidance"], h)
    traffic, traffic_src = None, None
    try:
        if args.precision != "bf16":
            raise KeyError("the committed DRAM-traffic capture is of the bf16 GEMMs")
        tj = json.load(open(os.path.join(ROOT, "profiles", "gemm_traffic.json")))
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
    except Exception:
        pass
    cpu = gpu_lib = None
    if world == 1 and not args.no_cpu_baseline:
        cval, ctimes, threads, kind = time_cpu(w, shape, steps=8, warmup=1, budget_s=25.0)
        cpu = {"value": cval, "unit": UNIT, "cores": threads, "kind": kind,
               "sample": f"{len(ctimes)} full plans of the same workload ({_kind_text(kind)}, torch CPU fp32, {threads} threads of {os.cpu_count()} host cpus)"}
        if ns is not None:
            wn = WORKLOADS["hopper_rtg_625"]
            nval, ntimes, _, nkind = time_cpu(wn, model_shape(wn), steps=6, warmup=1, budget_s=12.0)
            ns["cpu_reference"] = {"value": nval, "kind": nkind, "cores": threads, "plans_timed": len(ntimes)}
            ns["speedup_e2e_single_env_vs_cpu_reference"] = ns["single_env"]["e2e_value"] / nval
        if not args.lean:
            gpu_lib = time_gpu_library(w, shape, dev)
            if gpu_lib is not None:
                best = max((v["value"] for v in gpu_lib.values() if isinstance(v, dict) and "value" in v), default=None)
                if best:
                    gpu_lib["speedup_single_env_device_vs_best_library_mode"] = (K / single_dev_s) / best
    win_bytes = 4 * T * (shape.obs_dim + A + 2) * E_head
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": 1e3 * dev_s / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": args.workload, "candidates": n_total, "horizon": h, "guidance": w["guidance"], "env_shapes": w["env"],
                   "model": f"D={shape.n_embd},heads={shape.n_head},enc={shape.n_enc_layer},dec={shape.n_dec_layer},T={shape.traj_length}",
                   "parallelism": f"env-parallel x{world} (independent plans, no collective)",
                   "envs_per_gpu": E_head, "plans_per_step": plans_per_step,
                   "step": (f"{E_head} lock-step environments x {n_total} candidates planned by ONE m3pc_plan launch sequence per GPU "
                            f"(Learner.action_sample_batch); the one-window call of the reference is reported under single_env") if E_head > 1 else
                           "one window per plan (Learner.action_sample)", "l2": "256 MiB flush write between timed plans (outside the per-plan event pairs)",
                   "weights": weights_note, "chunk": args.chunk, "options": args.option},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": win_bytes, "d2h_bytes_per_step": 4 * A * E_head,
                "p50_latency_ms": 1e3 * statistics.median(head.lat),
                "api": ("Learner.action_sample_batch(E host numpy histories) -> .cpu()" if E_head > 1 else "Learner.action_sample(host numpy history) -> .cpu()")},
        "single_env": {"value": world * K / single_dev_s, "e2e_value": world * K / single_e2e_s, "unit": UNIT,
                       "p50_ms_device": statistics.median(single.per_step_ms), "p50_latency_ms_e2e": 1e3 * statistics.median(single.lat),
                       "launches_per_plan": single.launches, "api": "Learner.action_sample(host numpy history) -> .cpu()"},
        "gpu_launches": head.launches * K,
        "roofline": {"bound": "tensor" if args.precision == "bf16" else "fp32_ffma", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf if peak_tf else None,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": gemm_kernel,
                     "launches_per_step": g_n // 3, "gemm_ms_per_step": g_ms / 3,
                     "gemm_flops_per_step": g_fl / 3, "gemm_flops_per_plan": g_fl / 3 / E_head, "peak_source": peak_src,
                     "whole_step_executed_frac": (g_fl / 3) / (dev_s / K) / (peak_tf * 1e12) if dev_s > 0 else None,
                     "dense_equivalent_speed_frac": fl_plan * value / (world * peak_tf * 1e12),
                     "note": "achieved = executed GEMM FLOPs / summed per-launch GEMM event time; whole_step_executed_frac divides the same FLOPs by "
                             "the whole step; dense_equivalent_speed_frac counts FLOPs the restricted decoder and the shared-history block do NOT "
                             "execute -- a speed in dense-plan units, not a roofline fraction"},
        "flops_per_plan_dense": fl_plan, "flops_per_candidate_row": fl_row,
        "candidate_rollouts_per_sec": value * n_total,  # SURVEY.md section 8(d): plans/s x candidates per plan
        "p50_ms": statistics.median(head.per_step_ms), "wall_s_resident_loop": wall_resident,
        "clocks": clocks,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if gpu_lib is not None:
        line["gpu_library_baseline"] = gpu_lib
    if ns is not None:
        line["north_star_hopper_rtg_625"] = ns
    if cs is not None:
        line["cand_shard"] = cs
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="walker2d_critic_1024", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="env", choices=["env", "cand"])
    ap.add_argument("--envs", type=int, default=8, help="lock-step environments planned per step on each GPU (one m3pc_plan launch sequence)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--option", action="append", default=[], metavar="NAME=VALUE",
                    help="m3pc_set_option applied to every engine (A/B between result-equivalent launch sequences), e.g. fused_mlp=0")
    ap.add_argument("--lean", action="store_true", help="headline workload only: no north-star hopper key, no library baseline, no cand_shard")
    ap.add_argument("--cand-shard", action="store_true", help="also run the candidate-sharded config (halfcheetah 16384) on a single GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the actions of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")  # keep the real stdout for the JSON line ...
    os.dup2(2, 1)                              # ... and send every other write to fd 1 (NCCL prints its version there) to stderr
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    w = WORKLOADS[args.workload]
    shape = model_shape(w)
    rank, local_rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, w, shape, rank)
        return
    from m3pc_b200 import dist as mdist
    if args.option:
        from m3pc_b200.engine import PlanEngine
        for kv in args.option:
            k, v = kv.split("=")
            PlanEngine.default_options[k] = int(v)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # a box-level NCCL_DEBUG=VERSION would otherwise print to stdout, next to the JSON line
    mdist.init_from_env("nccl")
    try:
        run_ours(args, w, shape, rank, local_rank, world)
    finally:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
