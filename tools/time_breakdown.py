#!/usr/bin/env python
"""Device-time breakdown of a plan (CUDA events, graph replay path) and a warm GEMM microbenchmark.

    python tools/time_breakdown.py plan            # pass-1-only vs full plan at several candidate counts
    python tools/time_breakdown.py gemm [BNxCL]    # the pass-2 GEMM shapes, warm, 50 reps each
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402


def med(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def time_calls(fn, reps=30, warm=5, flush=None):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return med(ts), min(ts)


def sec_plan():
    import bench
    from m3pc_b200 import synthetic as syn
    from m3pc_b200.engine import engine_from_synthetic
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda")
    for name in ("walker2d_critic_1024", "hopper_rtg_1024", "scaled_rtg_4096"):
        w = bench.WORKLOADS[name]
        shape = bench.model_shape(w)
        crit = w["guidance"] != "rtg_guiding"
        T = shape.traj_length
        h = T // 2
        g = torch.Generator(device="cuda").manual_seed(0)
        ws, wa = torch.randn(T, shape.obs_dim, device="cuda", generator=g), torch.rand(T, shape.act_dim, device="cuda", generator=g) * 2 - 1
        wr, wt = torch.randn(T, device="cuda", generator=g), torch.full((T,), 0.7, device="cuda")
        for N in (1, 256, 1024, 4096, 16384):
            if w["model"] == "scaled" and N > 4096:
                continue
            eng = engine_from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), precision="bf16", max_batch=N,
                                        critic_sd=syn.make_critic_state_dict(shape) if crit else None, obs_norm=syn.make_obs_norm(shape) if crit else None)
            guid = "mtm_sampling" if N == 1 else w["guidance"]
            seed = [0]

            def fn():
                seed[0] += 1
                eng.plan(guidance=guid, horizon=h, n_cand=N, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt,
                         discount=0.99, temperature=w["temperature"], lmbda=0.6, seed=seed[0])

            m_warm, mn_warm = time_calls(fn)
            m_cold, mn_cold = time_calls(fn, flush=flush)
            print(f"plan {name} N={N} guidance={guid} launches={eng.last_launch_count()} warm-L2 med {m_warm:.1f} us (min {mn_warm:.1f}) | L2-flushed med {m_cold:.1f} us (min {mn_cold:.1f})",
                  flush=True)
            del eng


def sec_envs():
    """pass 1 alone (mtm_sampling) and the whole plan at E lock-step environments x 1024 candidates"""
    import bench
    from m3pc_b200 import synthetic as syn
    from m3pc_b200.engine import engine_from_synthetic
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda")
    name = "walker2d_critic_1024"
    w = bench.WORKLOADS[name]
    shape = bench.model_shape(w)
    T, N, h = shape.traj_length, 1024, 4
    g = torch.Generator(device="cuda").manual_seed(0)
    for E in (1, 2, 4, 8, 16, 32):
        ws, wa = torch.randn(E, T, shape.obs_dim, device="cuda", generator=g), torch.rand(E, T, shape.act_dim, device="cuda", generator=g) * 2 - 1
        wr, wt = torch.randn(E, T, device="cuda", generator=g), torch.full((E, T), 0.7, device="cuda")
        eng = engine_from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), precision="bf16", max_batch=N * E,
                                    critic_sd=syn.make_critic_state_dict(shape), obs_norm=syn.make_obs_norm(shape))
        for guid in ("mtm_sampling", w["guidance"]):
            seed = [0]

            def fn():
                seed[0] += 1
                eng.plan(guidance=guid, horizon=h, n_cand=N, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt,
                         discount=0.99, temperature=w["temperature"], lmbda=0.6, seed=seed[0], n_env=E)

            m_warm, mn_warm = time_calls(fn)
            m_cold, mn_cold = time_calls(fn, flush=flush)
            print(f"envs {name} E={E} N={N} guidance={guid} launches={eng.last_launch_count()} warm-L2 med {m_warm:.1f} us (min {mn_warm:.1f}) | "
                  f"L2-flushed med {m_cold:.1f} us (min {mn_cold:.1f}) = {m_cold / E:.1f} us per plan", flush=True)
        del eng


def sec_gemm():
    from m3pc_b200 import _native as nat
    L = nat.lib()
    shapes = [(13312, 1536, 512, 0, "enc qkv"), (13312, 512, 512, 2, "enc out-proj +res"), (13312, 2048, 512, 1, "enc lin1 gelu"),
              (13312, 512, 2048, 2, "enc lin2 +res"), (13312, 1024, 512, 0, "dec kv"), (7168, 2048, 512, 1, "dec lin1"), (7168, 512, 2048, 2, "dec lin2"),
              (4096, 256, 256, 4, "critic l2"), (65536, 2048, 512, 1, "big lin1"), (65536, 512, 2048, 2, "big lin2"), (8192, 8192, 8192, 0, "square 8k")]
    for (M, N, K, flags, what) in shapes:
        A = torch.randn(M, K, device="cuda").bfloat16()
        W = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16()
        b = torch.randn(N, device="cuda")
        C = torch.zeros(M, N, device="cuda") if flags & 2 else torch.empty(M, N, device="cuda", dtype=torch.bfloat16)

        def fn():
            nat.check(L.m3pc_gemm_bf16(A.data_ptr(), W.data_ptr(), b.data_ptr(), C.data_ptr(), M, N, K, flags, None))

        m, mn = time_calls(fn, reps=20 if M * N * K > 1e11 else 50)
        fl = 2.0 * M * N * K
        # cuBLAS bf16 on the same shape as the library bar
        Cb = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        mb, mnb = time_calls(lambda: torch.matmul(A, W.t(), out=Cb), reps=20 if M * N * K > 1e11 else 50)
        print(f"gemm {what:18s} M={M} N={N} K={K} flags={flags}: med {m:.1f} us (min {mn:.1f}) = {fl / m / 1e6:.0f} TF/s | cuBLAS plain {mb:.1f} us = {fl / mb / 1e6:.0f} TF/s",
              flush=True)


if __name__ == "__main__":
    globals()["sec_" + sys.argv[1]]()
