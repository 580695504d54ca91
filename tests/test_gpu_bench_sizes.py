"""Oracle parity AT THE SIZES bench.py measures (BASELINE.json configs[0..4]) -- not only self-consistency.

Every case runs the product path at the bench's own launch configuration (default chunk, default options: fused residual
GEMM + LayerNorm kernels, shared-history first block, shared-key decoder attention, CUDA-graph replay with on-device
Philox noise where the bench uses it) and compares candidates, per-candidate scores J, the arg-max / sampled index
(gap-conditioned) and the eval action with the float64 oracle (oracle/planner_oracle.py, pinned against the live reference
by tests/golden).  J of a candidate depends only on that candidate and the window, so the oracle may score a SLICE of the
candidates where the full set would take minutes (16 384 candidates, the scaled model).

Error measure (same as tests/test_gpu_parity.py): ``rel(a, ref) = max|a - ref| / max(1, max|ref|)`` -- the worst
element against the SCALE of the reference tensor, not an element-wise ratio (an element-wise ratio is meaningless for the
rewards / returns / actions of this model, which cross zero).  Bar: 1e-2 at bf16 (north_star); measured values are printed
(``pytest -s``) and tabulated in DESIGN.md.
"""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from m3pc_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

TOL = 1e-2
REPORT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "bench_size_parity.jsonl")


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(1.0, float(b.abs().max())))


def _report(**kw):
    print("PARITY", json.dumps(kw))
    try:
        os.makedirs(os.path.dirname(REPORT), exist_ok=True)
        with open(REPORT, "a") as f:
            f.write(json.dumps(kw) + "\n")
    except OSError:
        pass


def _learner(env, guidance, n_cand, temperature, scaled=False, max_envs=1, horizon=4, cls=None):
    from m3pc_b200.learner import Learner
    from m3pc_b200.mtm_model import omtmConfig
    from m3pc_b200.tokenizers import manager_from_stats
    shape = syn.scaled_shape(env) if scaled else syn.shipped_shape(env)
    cfg = SimpleNamespace(traj_length=shape.traj_length, device="cuda", action_samples=n_cand, discount=0.99, temperature=temperature,
                          horizon=horizon, plan_guidance=guidance, lmbda=0.6)
    mcfg = omtmConfig(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer, dropout=0.1,
                      norm="none", precision="bf16", max_batch=n_cand * max_envs, chunk=0)
    om, os_ = syn.make_obs_norm(shape)
    L = (cls or Learner)(cfg, None, shape.data_shapes, mcfg, None, om, os_, manager_from_stats(syn.make_tokenizer_stats(shape, 1)),
                         {k: False for k in shape.data_shapes}, max_envs=max_envs)
    L.mtm.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 0).items()})
    if hasattr(L, "iql"):
        L.iql.qf.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_critic_state_dict(shape).items()})
    return shape, L


def _oracle(shape, guidance, n, temperature, horizon=4):
    from oracle import planner_oracle as po
    crit = guidance != "rtg_guiding"
    return po.from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), dtype=torch.float64,
                             critic_np=syn.make_critic_state_dict(shape) if crit else None, obs_norm=syn.make_obs_norm(shape) if crit else None,
                             action_samples=n, temperature=temperature, plan_guidance=guidance, horizon=horizon)


def _check_indices(J, Jr, q, temp, amax, sidx, ref_amax, ref_sidx, errJ):
    """Device indices are consistent with the device scores, and equal the oracle's wherever its gap exceeds twice the error."""
    assert amax == int(torch.argmax(J))
    w = torch.exp((J - J.max()) * temp)
    if q is not None:
        assert sidx == int(torch.argmax(w / q))
    top2 = torch.topk(Jr, 2).values
    checked = 0
    if float(top2[0] - top2[1]) > 2 * errJ:
        assert amax == int(ref_amax)
        checked += 1
    if q is not None:
        key = torch.exp((Jr - Jr.max()) * temp) / q
        k2 = torch.topk(key, 2).values
        if float(torch.log(k2[0]) - torch.log(k2[1])) > 2 * temp * 2 * errJ:
            assert sidx == int(ref_sidx)
            checked += 1
    return checked


# ------------------------------------------------------------------------------------------------ configs[1]: the bench default step
def test_bench_default_step_walker2d_critic_8_envs_x_1024(monkeypatch):
    """BASELINE configs[1] exactly as bench.py runs it: 8 lock-step environments x 1024 candidates in ONE launch sequence
    (pass 2 at 8192 batch rows = 106 496 encoder rows, one chunk, fused-LN kernels, shared-history block, shared-key decoder
    attention).  (a) injected noise: every environment's candidates / J / indices / eval action vs the fp64 oracle;
    (b) the production path -- CUDA-graph replay with on-device Philox noise: the replayed actions equal the eager run with
    the same key, and that run's own candidates scored by the oracle reproduce its J."""
    E, N, temp, guidance = 8, 1024, 1.0, "critic_lambda_guiding"
    shape, L = _learner("walker2d", guidance, N, temp, max_envs=E)
    T, A, h = shape.traj_length, shape.act_dim, 4
    P = _oracle(shape, guidance, N, temp)
    hists = [dict(syn.make_history(shape, seed=1000 + e), path_length=50 + 37 * e) for e in range(E)]
    rs = np.random.RandomState(5)
    eps = torch.from_numpy(rs.randn(E, N, 1, T, 1, A))
    q = torch.from_numpy(rs.exponential(1.0, (E, N)))
    L.injected_noise = (eps[:, :, 0, T - h:, 0, :].reshape(E * N, h, A).float().contiguous().cuda(), q.reshape(-1).float().cuda())
    L.debug_plans = True
    ev = L.action_sample_batch(hists, plan=True, eval=True, rtg=3.0).double().cpu()
    dbg = L.last_plan_debug
    Jd, Cd, idx = dbg["expect_return"].double().cpu().reshape(E, N), dbg["candidates"].double().cpu().reshape(E, N, h, A), dbg["indices"].cpu().reshape(E, 2)
    worst = dict(J=0.0, cand=0.0, ev=0.0)
    n_idx = 0
    for e in range(E):
        _, ref = P.action_sample(hists[e], plan=True, eval=True, rtg=3.0, eps=eps[e], q=q[e])
        Jr = ref["expect_return"]
        errJ = float((Jd[e] - Jr).abs().max())
        worst["J"] = max(worst["J"], errJ / max(1.0, float(Jr.abs().max())))
        worst["cand"] = max(worst["cand"], rel(Cd[e], ref["candidates"]))
        worst["ev"] = max(worst["ev"], rel(ev[e], ref["eval_action"]))
        n_idx += _check_indices(Jd[e], Jr, q[e], temp, int(idx[e, 0]), int(idx[e, 1]), ref["argmax"], ref["sample_idx"], errJ)
    _report(case="walker2d_critic E=8 x N=1024 (bench default step), injected noise", **worst, index_checks=n_idx)
    assert worst["J"] < TOL and worst["cand"] < 3.5 * TOL and worst["ev"] < 2 * TOL
    # (b) production path: graph replay + Philox
    L.injected_noise, L.debug_plans, L.seed = None, False, 11
    acts = []
    for _ in range(4):  # eager, capture + replay, replay, replay -- same Philox key every time
        L.__dict__["_plan_counter"] = 0
        acts.append(L.action_sample_batch(hists, plan=True, eval=True, rtg=3.0).double().cpu())
    launches = L.mtm.sync_engine().last_launch_count()
    assert launches > 30
    for a in acts[1:]:
        np.testing.assert_allclose(a.numpy(), acts[0].numpy(), rtol=0, atol=1e-6)
    L.debug_plans = True
    L.__dict__["_plan_counter"] = 0
    ev2 = L.action_sample_batch(hists, plan=True, eval=True, rtg=3.0).double().cpu()
    np.testing.assert_allclose(ev2.numpy(), acts[0].numpy(), rtol=0, atol=1e-6)
    d2 = L.last_plan_debug
    J2, C2 = d2["expect_return"].double().cpu().reshape(E, N), d2["candidates"].double().cpu().reshape(E, N, h, A)
    assert float(C2.abs().max()) <= 1.0 and float(C2.std()) > 0.01
    wj = wev = 0.0
    for e in (0, 5):
        P.cand_override = C2[e]
        _, ref = P.action_sample(hists[e], plan=True, eval=True, rtg=3.0, eps=None, q=None)
        wj = max(wj, rel(J2[e], ref["expect_return"]))
        wev = max(wev, rel(ev2[e], ref["eval_action"]))
    P.cand_override = None
    _report(case="walker2d_critic E=8 x N=1024, CUDA-graph replay + Philox (own candidates scored by the oracle)", J=wj, ev=wev, launches=launches)
    assert wj < TOL and wev < 2 * TOL


# ------------------------------------------------------------------------------------------------ configs[0]: hopper rtg 625
@pytest.mark.parametrize("E", [1, 8])
def test_hopper_rtg_625(E):
    """BASELINE configs[0] shapes (hopper, rtg_guiding, the reference's shipped action_samples = 625, temperature 0.01) in the
    reference's one-window call and as the 8-environment step."""
    N, temp, guidance = 625, 0.01, "rtg_guiding"
    shape, L = _learner("hopper", guidance, N, temp, max_envs=E)
    T, A, h = shape.traj_length, shape.act_dim, 4
    P = _oracle(shape, guidance, N, temp)
    hists = [dict(syn.make_history(shape, seed=300 + e), path_length=60 + 11 * e) for e in range(E)]
    rs = np.random.RandomState(9)
    eps = torch.from_numpy(rs.randn(E, N, 1, T, 1, A))
    q = torch.from_numpy(rs.exponential(1.0, (E, N)))
    L.injected_noise = (eps[:, :, 0, T - h:, 0, :].reshape(E * N, h, A).float().contiguous().cuda(), q.reshape(-1).float().cuda())
    L.debug_plans = True
    ev = (L.action_sample(hists[0], plan=True, eval=True, rtg=3.0).reshape(1, A) if E == 1 else
          L.action_sample_batch(hists, plan=True, eval=True, rtg=3.0)).double().cpu()
    dbg = L.last_plan_debug
    Jd, Cd, idx = dbg["expect_return"].double().cpu().reshape(E, N), dbg["candidates"].double().cpu().reshape(E, N, h, A), dbg["indices"].cpu().reshape(E, 2)
    worst = dict(J=0.0, cand=0.0, ev=0.0)
    n_idx = 0
    for e in range(E):
        _, ref = P.action_sample(hists[e], plan=True, eval=True, rtg=3.0, eps=eps[e], q=q[e])
        Jr = ref["expect_return"]
        errJ = float((Jd[e] - Jr).abs().max())
        worst["J"] = max(worst["J"], errJ / max(1.0, float(Jr.abs().max())))
        worst["cand"] = max(worst["cand"], rel(Cd[e], ref["candidates"]))
        worst["ev"] = max(worst["ev"], rel(ev[e], ref["eval_action"]))
        n_idx += _check_indices(Jd[e], Jr, q[e], temp, int(idx[e, 0]), int(idx[e, 1]), ref["argmax"], ref["sample_idx"], errJ)
    _report(case=f"hopper_rtg E={E} x N=625", **worst, index_checks=n_idx)
    assert worst["J"] < TOL and worst["cand"] < 3.5 * TOL and worst["ev"] < 2e-2


# ------------------------------------------------------------------------------------------------ configs[2]: halfcheetah 16 384 on 4 shards
def test_halfcheetah_rtg_16384_four_shard_merge():
    """BASELINE configs[2]: 16 384 candidates split over 4 candidate shards (each a ``m3pc_plan`` with ``cand_offset`` and a
    partial record), merged by ``m3pc_merge_partials``.  The oracle scores two 1024-candidate slices (shard 0 and shard 3);
    the merged eval action and indices are checked against a float64 softmax over the device's own J."""
    from m3pc_b200 import dist as mdist
    N, G, temp, guidance, S = 16384, 4, 0.01, "rtg_guiding", 1024
    shape, L = _learner("halfcheetah", guidance, N // G, temp)
    eng = L._engine()
    T, A, h = shape.traj_length, shape.act_dim, 4
    hist = dict(syn.make_history(shape, seed=77), path_length=123)
    P = _oracle(shape, guidance, S, temp)
    traj, hh = P.build_window(hist, 1.0, 3.0)
    assert hh == h
    dev = "cuda"
    ws, wa = traj["states"][0].float().to(dev), traj["actions"][0].float().to(dev)
    wr = traj["rewards"][0, :, 0].float().to(dev)
    st = syn.make_tokenizer_stats(shape, 1)["returns"]
    wt = torch.from_numpy(((3.0 * np.ones(T) - np.asarray(st["mean"], np.float64).reshape(-1)[0]) / np.asarray(st["std"], np.float64).reshape(-1)[0]).astype(np.float32)).to(dev)
    rs = np.random.RandomState(21)
    eps = torch.from_numpy(rs.randn(N, 1, T, 1, A))
    q = torch.from_numpy(rs.exponential(1.0, N))
    eps_d, q_d = eps[:, 0, T - h:, 0, :].float().contiguous().cuda(), q.float().cuda()
    recs, Js, Cs = [], [], []
    for r in range(G):
        lo, hi = mdist.shard_range(N, r, G)
        _, _, d = eng.plan(guidance=guidance, horizon=h, n_cand=hi - lo, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt,
                           discount=0.99, temperature=temp, lmbda=0.6, eps=eps_d[lo:hi].contiguous(), expq=q_d[lo:hi].contiguous(), cand_offset=lo,
                           debug=True)
        recs.append(d["partials"].clone()); Js.append(d["expect_return"].double().cpu()); Cs.append(d["candidates"].double().cpu())
    ev_m, sm_m, idx_m = eng.merge_partials(torch.stack(recs), temp)
    J, Cn = torch.cat(Js), torch.cat(Cs)
    worst = dict(J=0.0, cand=0.0)
    for lo in (0, 3 * (N // G) + 1500):
        _, ref = P.action_sample(hist, plan=True, eval=True, rtg=3.0, eps=eps[lo:lo + S], q=q[lo:lo + S])
        worst["J"] = max(worst["J"], rel(J[lo:lo + S], ref["expect_return"]))
        worst["cand"] = max(worst["cand"], rel(Cn[lo:lo + S], ref["candidates"]))
    w = torch.exp((J - J.max()) * temp)
    ev_host = (w[:, None] * Cn[:, 0]).sum(0) / w.sum()
    worst["ev_merge_vs_fp64_softmax_of_device_J"] = rel(ev_m, ev_host)
    assert int(idx_m[0]) == int(torch.argmax(J)) and int(idx_m[1]) == int(torch.argmax(w / q))
    assert torch.equal(sm_m.double().cpu(), Cn[int(idx_m[1]), 0])
    _report(case="halfcheetah_rtg N=16384, 4 candidate shards + merge (oracle on two 1024-candidate slices)", **worst)
    assert worst["J"] < TOL and worst["cand"] < 3.5 * TOL and worst["ev_merge_vs_fp64_softmax_of_device_J"] < 1e-4


# ------------------------------------------------------------------------------------------------ configs[3]: zero-shot 256 envs x 512 draws
def test_zeroshot_piid_256_envs_x_512_draws():
    """BASELINE configs[3]: backward (waypoint) planner, 256 lock-step environments x 512 action draws in one call
    (``action_piid_draws_batch`` -> ``m3pc_backward_plan_draws``).  Rows are compared with the oracle's B = 1
    ``action_piid_sample`` (zeroshot_omtm/learner.py:151-261) on a spread of 24 environments: the mean action and, through
    eps = 0 / +1 / -1 oracle calls, the mu / std every one of the 512 injected-noise draws of that row must follow."""
    from m3pc_b200.zeroshot_learner import Learner as ZL
    from oracle import planner_oracle as po
    E, Cn = 256, 512
    shape, L = _learner("hopper", "rtg_guiding", 1, 0.01, max_envs=E, cls=ZL)
    T, A, h = shape.traj_length, shape.act_dim, 4
    P = po.from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), dtype=torch.float64, action_samples=1)
    hists = [dict(syn.make_history(shape, seed=500 + e % 61), path_length=100 + e) for e in range(E)]
    rs = np.random.RandomState(2)
    eps = torch.from_numpy(rs.randn(E, Cn, A)).float()
    L.injected_eps = eps.cuda()
    ev, draws = L.action_piid_draws_batch(hists, Cn, rtg=2.0)
    ev, draws = ev.double().cpu(), draws.double().cpu()
    assert ev.shape == (E, A) and draws.shape == (E, Cn, A) and bool(torch.isfinite(draws).all())
    w_ev = w_dr = 0.0
    for e in range(0, E, 11):
        m0, _ = P.action_piid_sample(hists[e], eval=True, rtg=2.0)
        sp, _ = P.action_piid_sample(hists[e], eval=False, rtg=2.0, eps1=torch.ones(1, T, 1, A, dtype=torch.float64))
        mu = torch.atanh(m0)
        std = torch.atanh(sp) - mu
        ref = torch.tanh(mu[None, :] + std[None, :] * eps[e].double())
        w_ev = max(w_ev, rel(ev[e], m0))
        w_dr = max(w_dr, rel(draws[e], ref))
    _report(case="zeroshot piid E=256 x C=512 draws (24 environments vs oracle B=1 calls)", ev=w_ev, draws=w_dr)
    assert w_ev < 2e-2 and w_dr < 3.5e-2


# ------------------------------------------------------------------------------------------------ configs[4]: scaled model, 1024 candidates
def test_scaled_model_1024_candidates():
    """BASELINE configs[4] shapes (D=1024, 8 heads, 4+2 layers, T=16, h=8) at 1024 candidates; the oracle scores a
    96-candidate slice (6 GFLOP per candidate row in float64 on the host)."""
    N, S, temp, guidance, h = 1024, 96, 0.01, "rtg_guiding", 8
    shape, L = _learner("hopper", guidance, N, temp, scaled=True, horizon=h)
    T, A = shape.traj_length, shape.act_dim
    P = _oracle(shape, guidance, S, temp, horizon=h)
    hist = dict(syn.make_history(shape, seed=9), path_length=50)
    rs = np.random.RandomState(3)
    eps = torch.from_numpy(rs.randn(N, 1, T, 1, A))
    q = torch.from_numpy(rs.exponential(1.0, N))
    L.injected_noise = (eps[:, 0, T - h:, 0, :].float().contiguous().cuda(), q.float().cuda())
    L.debug_plans = True
    L.action_sample(hist, plan=True, eval=True, rtg=3.0)
    dbg = L.last_plan_debug
    J, Cd = dbg["expect_return"].double().cpu(), dbg["candidates"].double().cpu()
    lo = 517
    _, ref = P.action_sample(hist, plan=True, eval=True, rtg=3.0, eps=eps[lo:lo + S], q=q[lo:lo + S])
    eJ, eC = rel(J[lo:lo + S], ref["expect_return"]), rel(Cd[lo:lo + S], ref["candidates"])
    # per-head errors of the decoded predictions that enter J (returns x 1000 dominate J: J ~ 1000 * returns)
    _report(case="scaled model (D=1024, 4+2 layers, T=16, h=8) N=1024, oracle on a 96-candidate slice", J=eJ, cand=eC,
            J_scale=float(ref["expect_return"].abs().max()))
    assert eJ < TOL and eC < 3.5 * TOL


# ------------------------------------------------------------------------------------------------ bench.py --dump-outputs
def test_bench_dumps_the_actions_of_the_last_timed_step(tmp_path):
    """``bench.py --steps K --dump-outputs DIR`` times K steps and writes the actions the timed path returned in the last one:
    they equal a fresh plan of the last timed step's windows and seed, and differ from the step before it."""
    import subprocess
    import sys
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    K, W = 3, 3
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", str(K), "--warmup", str(W), "--lean", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == K
    dumped = {f.name: np.load(f) for f in tmp_path.glob("*.npy")}
    assert sorted(dumped) == ["eval_action.npy", "sample_action.npy", "single_env_eval_action.npy", "single_env_sample_action.npy"]
    assert all(a.dtype == np.float32 for a in dumped.values())
    # the same learner, windows and seeds as the bench's default workload (rank 0)
    w = bench.WORKLOADS["walker2d_critic_1024"]
    shape = bench.model_shape(w)
    dev = torch.device("cuda:0")
    L = bench.build_learner(w, shape, w["n_cand"], 8, dev, SimpleNamespace(precision="bf16", chunk=0))
    flush = torch.empty(1024, device=dev)
    for E, prefix in ((1, "single_env_"), (8, "")):
        m = bench.measure(L, w, shape, E, K, W, dev, flush, lambda: None, hist_base=1000)
        last = [t.cpu().numpy() for t in m.plan_resident(W + K - 1)]
        before = [t.cpu().numpy() for t in m.plan_resident(W + K - 2)]
        assert dumped[prefix + "eval_action.npy"].shape == ((E, shape.act_dim) if E > 1 else (shape.act_dim,))
        np.testing.assert_array_equal(dumped[prefix + "eval_action.npy"], last[0])
        np.testing.assert_array_equal(dumped[prefix + "sample_action.npy"], last[1])
        assert not np.array_equal(last[0], before[0])
