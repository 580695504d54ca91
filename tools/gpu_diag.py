#!/usr/bin/env python
"""Exploratory GPU diagnostics (run under gpurun): each section in its own subprocess with a timeout, so that a
hung kernel cannot take the other sections down.  Writes gpurun_out/diag_<section>.log.

    python tools/gpu_diag.py all
"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "gpurun_out")
SECTIONS = ["sgemm", "small", "gemm_bf16", "fwd_fp32", "fwd_bf16", "plan_fp32", "plan_bf16", "timing"]


def rel_err(a, b):
    import torch
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30)), float((a - b).abs().max())


def sec_sgemm():
    import ctypes as C
    import torch
    from m3pc_b200 import _native as nat
    L = nat.lib()
    torch.manual_seed(0)
    for (M, N, K, flags) in [(17, 1536, 512, 0), (200, 512, 2048, 1), (333, 256, 23, 4), (64, 1, 256, 0), (1000, 512, 512, 2)]:
        A = torch.randn(M, K, device="cuda"); W = torch.randn(N, K, device="cuda") / K ** 0.5; b = torch.randn(N, device="cuda")
        Cm = torch.randn(M, N, device="cuda"); C0 = Cm.clone()
        nat.check(L.m3pc_gemm_fp32(A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, flags, None))
        torch.cuda.synchronize()
        ref = A.double() @ W.double().T + b.double()
        if flags & 1: ref = torch.nn.functional.gelu(ref)
        if flags & 4: ref = torch.relu(ref)
        if flags & 2: ref = ref + C0.double()
        print("sgemm", (M, N, K, flags), "rel/abs err", rel_err(Cm, ref), flush=True)


def sec_small():
    import torch
    from m3pc_b200 import _native as nat
    L = nat.lib()
    torch.manual_seed(0)
    for D in (512, 1024):
        x = torch.randn(1000, D, device="cuda") * 3 + 1; g = torch.rand(D, device="cuda") + 0.5; b = torch.randn(D, device="cuda")
        ref = torch.nn.functional.layer_norm(x.double(), (D,), g.double(), b.double(), 1e-5)
        y = torch.empty(1000, D, device="cuda")
        nat.check(L.m3pc_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), y.data_ptr(), 1000, D, 0, None))
        y16 = torch.empty(1000, D, device="cuda", dtype=torch.bfloat16)
        nat.check(L.m3pc_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), y16.data_ptr(), 1000, D, 1, None))
        torch.cuda.synchronize()
        print("layernorm D", D, "fp32", rel_err(y, ref), "bf16", rel_err(y16, ref), flush=True)
    for (B, S, H) in [(5, 13, 4), (3, 32, 4), (2, 64, 8), (70, 17, 4)]:
        D = H * 128
        qkv = torch.randn(S * B, 3 * D, device="cuda")
        q, k, v = [t.reshape(S, B, H, 128).permute(1, 2, 0, 3).double() for t in qkv.split(D, dim=1)]
        att = torch.softmax(q @ k.transpose(-1, -2) / 128 ** 0.5, -1) @ v  # (B,H,S,128)
        ref = att.permute(2, 0, 1, 3).reshape(S * B, D)
        out = torch.empty(S * B, D, device="cuda")
        nat.check(L.m3pc_attention(qkv.data_ptr(), out.data_ptr(), B, S, H, 0, None))
        qkv16 = qkv.bfloat16(); out16 = torch.empty(S * B, D, device="cuda", dtype=torch.bfloat16)
        nat.check(L.m3pc_attention(qkv16.data_ptr(), out16.data_ptr(), B, S, H, 1, None))
        torch.cuda.synchronize()
        q, k, v = [t.reshape(S, B, H, 128).permute(1, 2, 0, 3).double() for t in qkv16.split(D, dim=1)]
        ref16 = (torch.softmax(q @ k.transpose(-1, -2) / 128 ** 0.5, -1) @ v).permute(2, 0, 1, 3).reshape(S * B, D)
        print("attention", (B, S, H), "fp32", rel_err(out, ref), "bf16", rel_err(out16, ref16), flush=True)


def sec_gemm_bf16():
    import torch
    from m3pc_b200 import _native as nat
    L = nat.lib()
    torch.manual_seed(0)
    cases = [(128, 128, 64, 0), (128, 128, 512, 0), (256, 256, 512, 0), (17, 1536, 512, 0), (8125, 512, 512, 2), (1000, 2048, 512, 1),
             (333, 512, 2048, 2), (4096, 1536, 512, 0), (130, 128, 128, 4)]
    for (M, N, K, flags) in cases:
        A = torch.randn(M, K, device="cuda").bfloat16(); W = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16()
        b = torch.randn(N, device="cuda")
        ref = A.double() @ W.double().T + b.double()
        if flags & 1: ref = torch.nn.functional.gelu(ref)
        if flags & 4: ref = torch.relu(ref)
        if flags & 2:
            Cm = torch.randn(M, N, device="cuda"); ref = ref + Cm.double()
        else:
            Cm = torch.zeros(M, N, device="cuda", dtype=torch.bfloat16)
        nat.check(L.m3pc_gemm_bf16(A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, flags, None))
        torch.cuda.synchronize()
        e = rel_err(Cm, ref)
        bad = (Cm.double() - ref).abs() > 0.05 * ref.abs().max()
        print("gemm_bf16", (M, N, K, flags), "rel/abs err", e, "bad elems", int(bad.sum()), "of", bad.numel(), flush=True)
        if bad.any():
            rows = bad.any(dim=1).nonzero().flatten()[:10].tolist(); cols = bad.any(dim=0).nonzero().flatten()[:10].tolist()
            print("   first bad rows", rows, "cols", cols, flush=True)


def sec_gemm_bench():
    """Time the tensor-core GEMM on the plan's shapes (CUDA events, warm L2, 20 reps)."""
    import torch
    from m3pc_b200 import _native as nat
    L = nat.lib()
    torch.manual_seed(0)
    shapes = [("enc qkv", 13312, 1536, 512, 0), ("enc out", 13312, 512, 512, 2), ("enc ffn1", 13312, 2048, 512, 1), ("enc ffn2", 13312, 512, 2048, 2),
              ("dec kv", 13312, 1024, 512, 0), ("dec ffn1", 7168, 2048, 512, 1), ("dec ffn2", 7168, 512, 2048, 2), ("full dec qkv", 32768, 1536, 512, 0),
              ("big ffn1", 65536, 2048, 512, 1), ("odd", 625 * 13, 1536, 512, 0)]
    for name, M, N, K, flags in shapes:
        A = torch.randn(M, K, device="cuda").bfloat16(); W = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16(); b = torch.randn(N, device="cuda")
        Cm = torch.randn(M, N, device="cuda") if flags & 2 else torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        ref = A.double() @ W.double().T + b.double()
        if flags & 1: ref = torch.nn.functional.gelu(ref)
        if flags & 2: ref = ref + Cm.double()
        nat.check(L.m3pc_gemm_bf16(A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, flags, None))
        torch.cuda.synchronize()
        err = rel_err(Cm, ref)[0]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if flags & 2: Cm.zero_()
        e0.record()
        for _ in range(20):
            L.m3pc_gemm_bf16(A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, flags, None)
        e1.record(); torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1000 / 20
        print(f"gemm {name:12s} M={M:6d} N={N:5d} K={K:5d} flags={flags}: {us:7.1f} us  {2.0*M*N*K/us/1e6:7.1f} TFLOP/s  err={err:.1e}", flush=True)


def sec_pass1():
    """Device time of pass 1 alone (B = 1): mtm_sampling = pass 1 + a 1-thread tail."""
    import torch
    from m3pc_b200 import synthetic as syn
    for prec in ("bf16", "fp32"):
        shape, sd, stats, csd, on, eng = _setup("walker2d", prec, 16)
        T = shape.traj_length
        ws = torch.randn(T, shape.obs_dim, device="cuda"); wa = torch.rand(T, shape.act_dim, device="cuda") * 2 - 1
        wr = torch.randn(T, device="cuda"); wt = torch.full((T,), 1.0, device="cuda")
        ts = []
        for i in range(10):
            eng.plan(guidance="mtm_sampling", horizon=4, n_cand=1, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt,
                     discount=0.99, temperature=1.0, lmbda=0.6, seed=i)
            torch.cuda.synchronize()
            ts.append(eng.last_device_ms())
        print(f"pass1[{prec}] launches={eng.last_launch_count()} ms median={sorted(ts)[5]:.3f} min={min(ts):.3f}", flush=True)


def _setup(env, precision, max_batch, critic=False, chunk=0):
    import torch
    from m3pc_b200 import synthetic as syn
    from m3pc_b200.engine import engine_from_synthetic
    shape = syn.shipped_shape(env)
    sd, stats = syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1)
    csd = syn.make_critic_state_dict(shape) if critic else None
    on = syn.make_obs_norm(shape) if critic else None
    eng = engine_from_synthetic(shape, sd, stats, precision=precision, max_batch=max_batch, critic_sd=csd, obs_norm=on, chunk=chunk)
    return shape, sd, stats, csd, on, eng


def _fwd(precision):
    import torch
    from m3pc_b200 import synthetic as syn
    from oracle import mtm_oracle as mo, planner_oracle as po
    shape, sd, stats, _, _, eng = _setup("hopper", precision, 64)
    sd64, st64 = mo.to_torch(sd, torch.float64), mo.stats_to_torch(stats, torch.float64)
    traj = {k: torch.from_numpy(v) for k, v in syn.make_trajectories(shape, 5, 5).items()}
    enc64 = mo.encode_all({k: v.double() for k, v in traj.items()}, st64)
    enc32 = mo.encode_all(traj, mo.stats_to_torch(stats))
    toks = {k: v.squeeze(2).cuda() for k, v in enc32.items()}
    for name, fn in [("fd", po.create_fd_mask), ("rcbc", po.create_rcbc_mask), ("pi", po.create_pi_mask), ("fid", po.create_fid_mask)]:
        for idx in (4, 0):
            m = fn(shape.traj_length, idx)
            ref = mo.mtm_forward(sd64, enc64, {k: torch.from_numpy(v) for k, v in m.items()}, shape.n_head, shape.n_enc_layer, shape.n_dec_layer)
            out = eng.forward(toks, m)
            torch.cuda.synchronize()
            msg = [f"fwd[{precision}] {name} idx{idx} launches={eng.last_launch_count()} ms={eng.last_device_ms():.3f}"]
            for k in ("states", "rewards", "returns"):
                msg.append(f"{k}={rel_err(out[k], ref[k].squeeze(2))[0]:.2e}")
            msg.append(f"mu={rel_err(out['act_mu'], ref['actions']['mu'].squeeze(2))[0]:.2e}")
            msg.append(f"std={rel_err(out['act_std'], ref['actions']['std'].squeeze(2))[0]:.2e}")
            print(" ".join(msg), flush=True)


def sec_fwd_fp32():
    _fwd("fp32")


def sec_fwd_bf16():
    _fwd("bf16")


def _plan(precision):
    import numpy as np
    import torch
    from m3pc_b200 import synthetic as syn
    from oracle import planner_oracle as po
    for env, guidance, temp, N, pl in [("hopper", "rtg_guiding", 0.01, 64, 50), ("hopper", "rtg_guiding", 0.01, 200, 2),
                                        ("walker2d", "critic_lambda_guiding", 1.0, 64, 50), ("walker2d", "noise_adding_lambda", 1.0, 96, 50)]:
        crit = guidance != "rtg_guiding"
        shape, sd, stats, csd, on, eng = _setup(env, precision, 256, critic=crit)
        P = po.from_synthetic(shape, sd, stats, dtype=torch.float64, critic_np=csd, obs_norm=on, action_samples=N, temperature=temp,
                              plan_guidance=guidance)
        hist = syn.make_history(shape, seed=4, path_length=pl)
        T, A = shape.traj_length, shape.act_dim
        rs = np.random.RandomState(7)
        traj, h = P.build_window(hist, rtg=3.0)
        if guidance == "noise_adding_lambda":
            eps = torch.from_numpy(rs.randn(N, h, A)); eps_dev = eps.float().cuda()
        else:
            eps = torch.from_numpy(rs.randn(N, 1, T, 1, A)); eps_dev = eps[:, 0, T - h:, 0, :].float().contiguous().cuda()
        q = torch.from_numpy(rs.exponential(1.0, N))
        act, dbg = P.action_sample(hist, plan=True, eval=True, rtg=3.0, eps=eps, q=q)
        ret_tok = ((traj["returns"].double() - float(stats["returns"]["mean"][0])) / float(stats["returns"]["std"][0])).float()
        ev, sm, d = eng.plan(guidance=guidance, horizon=h, n_cand=N, win_states=traj["states"][0].float().cuda(),
                             win_actions=traj["actions"][0].float().cuda(), win_rewards=traj["rewards"][0, :, 0].float().cuda(),
                             win_returns_tok=ret_tok[0, :, 0].cuda(), discount=0.99, temperature=temp, lmbda=0.6, eps=eps_dev,
                             expq=q.float().cuda(), debug=True)
        torch.cuda.synchronize()
        J, Jr = d["expect_return"].double().cpu(), dbg["expect_return"]
        print(f"plan[{precision}] {env} {guidance} N={N} h={h} launches={eng.last_launch_count()} ms={eng.last_device_ms():.3f}",
              "cand", rel_err(d["candidates"], dbg["candidates"]), "J", rel_err(J, Jr), "J spread", float(Jr.max() - Jr.min()),
              "eval", rel_err(ev, dbg["eval_action"]), "sample", rel_err(sm, dbg["sample_action"]),
              "idx", d["indices"].tolist(), int(dbg["argmax"]), int(dbg["sample_idx"]), flush=True)


def sec_plan_fp32():
    _plan("fp32")


def sec_plan_bf16():
    _plan("bf16")


def sec_timing():
    import torch
    from m3pc_b200 import synthetic as syn
    for env, guidance, N in [("walker2d", "critic_lambda_guiding", 1024), ("hopper", "rtg_guiding", 1024), ("hopper", "rtg_guiding", 4096)]:
        for chunk in (256, 1024, 4096):
            if chunk > N:
                continue
            shape, sd, stats, csd, on, eng = _setup(env, "bf16", N, critic=True, chunk=chunk)
            hist = syn.make_history(shape)
            T = shape.traj_length
            ws = torch.randn(T, shape.obs_dim, device="cuda"); wa = torch.rand(T, shape.act_dim, device="cuda") * 2 - 1
            wr = torch.randn(T, device="cuda"); wt = torch.full((T,), 1.0, device="cuda")
            ts = []
            for i in range(8):
                eng.plan(guidance=guidance, horizon=4, n_cand=N, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt,
                         discount=0.99, temperature=1.0, lmbda=0.6, seed=i)
                torch.cuda.synchronize()
                ts.append(eng.last_device_ms())
            print(f"timing {env} {guidance} N={N} chunk={chunk} launches={eng.last_launch_count()} ms={sorted(ts)[len(ts)//2]:.3f} (min {min(ts):.3f})", flush=True)
            del eng


if __name__ == "__main__":
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    if which == "all":
        os.makedirs(OUT, exist_ok=True)
        for s in SECTIONS:
            t0 = time.time()
            log = os.path.join(OUT, f"diag_{s}.log")
            with open(log, "w") as f:
                try:
                    rc = subprocess.run([sys.executable, __file__, s], stdout=f, stderr=subprocess.STDOUT, timeout=240).returncode
                except subprocess.TimeoutExpired:
                    rc = "TIMEOUT"
            print(f"=== {s}: rc={rc} ({time.time() - t0:.1f}s)")
            print(open(log).read()[-6000:])
    else:
        globals()["sec_" + which]()
