"""The three precision modes side by side on the bench.py default workload (walker2d, critic_lambda_guiding, 8 environments x
1024 candidates per step), in one process, and the pass-2 GEMM shapes of that step for the two fp32-grade GEMMs.

  * plan steps: the modes alternate (fp32, tf32x3, bf16, fp32, ...) over --rounds rounds of --steps steps each, every mode's
    shapes warmed up first (CUDA graphs captured); per step the device time (CUDA events, L2 flushed before every step) and
    plans/s = environments / step time; then one profiled step per mode (m3pc_set_profile: eager launches, an event pair per GEMM)
    for the GEMM time and FLOPs of a step.
  * GEMMs at M = 106 496 rows (8 x 1024 candidates x 13 decoder rows): QKV, out-projection, linear1, linear2 and the decoder K/V
    projection of the step, m3pc_gemm_tf32x3 against m3pc_gemm_fp32, alternating, the L2 overwritten before every timed launch.
    Achieved TFLOP/s = 2 M N K / kernel time, reported against 1 125 TFLOP/s (data-sheet dense TF32 of one B200) / 3: the
    3xTF32 split issues three TF32 MMAs per product, so a third of the TF32 rate is its ceiling.  On the same inputs, the error of
    both kernels against the float64 product: max |C - C64| / max(1, max |C64|).

Writes one JSON document (the card's name and power limit beside the numbers) to --out and prints a summary.
Usage: python tools/precision_modes.py --out profiles/r2t_precision_modes.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TF32_DENSE_TFLOPS = 1125.0  # NVIDIA HGX B200 data sheet, one GPU, dense
MODES = ("fp32", "tf32x3", "bf16")


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def plan_steps(args, out):
    import torch
    import bench
    from m3pc_b200 import synthetic as syn
    w = bench.WORKLOADS["walker2d_critic_1024"]
    shape = syn.shipped_shape(w["env"])
    E, N, h = args.envs, w["n_cand"], 4
    dev = torch.device("cuda:0")
    flush = torch.empty(64 * 1024 * 1024, device=dev)  # 256 MB > 126 MB of L2
    runs = {}
    for mode in MODES:
        L = bench.build_learner(w, shape, N, E, dev, SimpleNamespace(precision=mode, chunk=0))
        eng = L._engine()
        hists = [syn.make_history(shape, seed=1000 + e, path_length=50 + 37 * e) for e in range(E)]
        ring, slot = L._window_buffers(shape.obs_dim, shape.act_dim, n_env=E)
        for e, hist in enumerate(hists):
            L._fill_window(slot.h_states[e], slot.h_actions[e], slot.h_rewards[e], slot.h_returns[e], hist, h, 1.0, 3.0)
        win = slot.host.to(dev)
        T, A, obs = shape.traj_length, shape.act_dim, shape.obs_dim
        o = [0, E * T * obs, E * T * (obs + A), E * T * (obs + A + 1), win.numel()]
        views = (win[o[0]:o[1]].view(E, T, obs), win[o[1]:o[2]].view(E, T, A), win[o[2]:o[3]].view(E, T), win[o[3]:o[4]].view(E, T))

        def step(i, eng=eng, views=views):
            return eng.plan(guidance=w["guidance"], horizon=h, n_cand=N, win_states=views[0], win_actions=views[1], win_rewards=views[2],
                            win_returns_tok=views[3], discount=0.99, temperature=w["temperature"], lmbda=0.6, seed=7 + i, n_env=E)
        for i in range(args.warmup):
            step(i)
        runs[mode] = (eng, step)
    torch.cuda.synchronize()
    ms = {m: [] for m in MODES}
    for r in range(args.rounds):
        for mode in MODES:
            eng, step = runs[mode]
            for i in range(args.steps):
                flush.fill_(float(i))
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                step(i)
                e1.record()
                e1.synchronize()
                ms[mode].append(e0.elapsed_time(e1))
    res = {}
    for mode in MODES:
        eng, step = runs[mode]
        eng.set_profile(True)
        flush.fill_(0.0)
        step(0)
        torch.cuda.synchronize()
        gemm_ms, gemm_flops, n_gemm = eng.get_profile()
        eng.set_profile(False)
        p50 = statistics.median(ms[mode])
        res[mode] = {"step_ms_p50": p50, "step_ms_min": min(ms[mode]), "step_ms_max": max(ms[mode]), "steps": len(ms[mode]),
                     "plans_per_s": E / (p50 * 1e-3),
                     "profiled_step": {"gemm_ms": gemm_ms, "gemm_gflop": gemm_flops / 1e9, "gemm_launches": n_gemm,
                                       "gemm_tflops": gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms else None}}
    res["speedup_tf32x3_over_fp32"] = res["fp32"]["step_ms_p50"] / res["tf32x3"]["step_ms_p50"]
    out["plan_steps"] = res
    out["workload"] = {"name": "walker2d_critic_1024", "envs": E, "n_cand": N, "horizon": h,
                       "timing": "CUDA events around m3pc_plan (CUDA-graph replay), L2 overwritten before every step; modes alternate by round"}
    return shape


def gemm_shapes(args, out, D):
    import torch
    from m3pc_b200 import _native as nat
    lib = nat.lib()
    M = args.rows
    shapes = [("qkv", 3 * D, D, 0), ("out_proj", D, D, 2), ("linear1", 4 * D, D, 1), ("linear2", D, 4 * D, 2), ("dec_kv", 2 * D, D, 0)]
    flush = torch.empty(64 * 1024 * 1024, device="cuda")
    rows = []
    for name, N, K, flags in shapes:
        g = torch.Generator(device="cuda").manual_seed(N + K)
        A = torch.randn(M, K, device="cuda", generator=g)
        W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
        b = torch.randn(N, device="cuda", generator=g)
        C = torch.zeros(M, N, device="cuda")
        fns = {"tf32x3": lib.m3pc_gemm_tf32x3, "fp32": lib.m3pc_gemm_fp32}
        for fn in fns.values():  # warm-up
            nat.check(fn(A.data_ptr(), W.data_ptr(), b.data_ptr(), C.data_ptr(), M, N, K, flags, None))
        t = {k: [] for k in fns}
        for _ in range(args.gemm_reps):
            for k, fn in fns.items():
                flush.fill_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                nat.check(fn(A.data_ptr(), W.data_ptr(), b.data_ptr(), C.data_ptr(), M, N, K, flags, None))
                e1.record()
                e1.synchronize()
                t[k].append(e0.elapsed_time(e1))
        flop = 2.0 * M * N * K
        row = {"name": name, "M": M, "N": N, "K": K, "flags": flags}
        C0 = torch.randn(M, N, device="cuda", generator=g)
        ref = A.double() @ W.double().T + b.double()
        if flags & 1:
            ref = torch.nn.functional.gelu(ref)
        if flags & 2:
            ref += C0.double()
        for k, fn in fns.items():
            m = statistics.median(t[k])
            C.copy_(C0)
            nat.check(fn(A.data_ptr(), W.data_ptr(), b.data_ptr(), C.data_ptr(), M, N, K, flags, None))
            torch.cuda.synchronize()
            err = float((C.double() - ref).abs().max() / max(1.0, float(ref.abs().max())))
            row[k] = {"ms_p50": m, "tflops": flop / (m * 1e-3) / 1e12, "max_rel_err_vs_fp64": err}
        row["tf32x3"]["frac_of_tf32_rate_over_3"] = row["tf32x3"]["tflops"] / (TF32_DENSE_TFLOPS / 3)
        row["speedup"] = row["fp32"]["ms_p50"] / row["tf32x3"]["ms_p50"]
        rows.append(row)
        del A, W, C, C0, ref
    out["gemms"] = {"rows": rows, "ceiling_tflops": TF32_DENSE_TFLOPS / 3,
                    "ceiling": "1125 TFLOP/s dense TF32 (data sheet, one B200) / 3: the split runs three TF32 MMAs per product",
                    "timing": f"CUDA events around one launch, median of {args.gemm_reps}, the two kernels alternating, L2 overwritten before each"}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--envs", type=int, default=8)
    ap.add_argument("--steps", type=int, default=10, help="timed steps per mode per round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--rows", type=int, default=106496)
    ap.add_argument("--gemm-reps", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("precision_modes.py measures on a GPU; none is visible")
    out = {"card": card()}
    shape = plan_steps(args, out)
    gemm_shapes(args, out, shape.n_embd)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["card"]))
    for m in MODES:
        r = out["plan_steps"][m]
        print(f"{m:7s} step p50 {r['step_ms_p50']:.3f} ms  {r['plans_per_s']:.1f} plans/s  GEMMs {r['profiled_step']['gemm_ms']:.3f} ms "
              f"{r['profiled_step']['gemm_gflop']:.0f} GFLOP ({r['profiled_step']['gemm_launches']} launches)")
    print(f"tf32x3 / fp32 step speed-up: {out['plan_steps']['speedup_tf32x3_over_fp32']:.2f}x")
    for r in out["gemms"]["rows"]:
        print(f"{r['name']:9s} M={r['M']} N={r['N']} K={r['K']}: tf32x3 {r['tf32x3']['ms_p50']:.3f} ms {r['tf32x3']['tflops']:.1f} TFLOP/s "
              f"({r['tf32x3']['frac_of_tf32_rate_over_3']:.2f} of TF32/3)  fp32 {r['fp32']['ms_p50']:.3f} ms {r['fp32']['tflops']:.1f} TFLOP/s  x{r['speedup']:.2f}  "
              f"err vs fp64: tf32x3 {r['tf32x3']['max_rel_err_vs_fp64']:.2e} fp32 {r['fp32']['max_rel_err_vs_fp64']:.2e}")


if __name__ == "__main__":
    main()
