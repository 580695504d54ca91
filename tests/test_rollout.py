"""The vectorised / pipelined caller loop (m3pc_b200/rollout.py; reference loops: replay_buffer.py:167-232, learner.py:648-720).
CPU tests drive it with a stand-in planner; the GPU tests with the real one."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from m3pc_b200 import rollout as ro
from m3pc_b200 import synthetic as syn


class _FakeTicket:
    def __init__(self, a):
        self.a = a

    def result(self):
        return self.a


class _FakePlanner:
    """action = tanh of the first act_dim features of the latest observation, scaled by the rtg; records every call."""

    def __init__(self, act_dim):
        self.mtm = SimpleNamespace(data_shapes={"actions": (1, act_dim)})
        self.max_envs = 64
        self.calls = []

    def action_sample_async(self, histories, percentage=1.0, plan=True, eval=False, rtg=None):
        pls = {h["path_length"] for h in histories}
        assert len(pls) == 1, "a group must stay in lock-step"
        self.calls.append((len(histories), pls.pop(), rtg))
        A = self.mtm.data_shapes["actions"][1]
        return _FakeTicket(np.stack([2.0 * np.tanh(h["observations"][h["path_length"], :A]) * (1.0 if rtg is None else rtg) for h in histories]))


def _reference_loop(planner, env, rtg, max_path_length):
    """The reference's single-environment loop (learner.py:663-696), verbatim in structure."""
    obs_dim, A = env.x0.shape[0], planner.mtm.data_shapes["actions"][1]
    tr = ro.new_trajectory(obs_dim, A, max_path_length)
    observation, done, t = env.reset(), False, 0
    while not done and t < max_path_length:
        tr["observations"][t] = observation
        action = np.clip(planner.action_sample_async([tr], plan=True, eval=True, rtg=rtg(t)).result()[0], -1, 1)
        observation, reward, done, _ = env.step(action)
        tr["actions"][t] = action
        tr["rewards"][t] = reward
        t += 1
        tr["path_length"] += 1
    return tr


@pytest.mark.parametrize("groups", [1, 2, 3, 7])
def test_run_episodes_equals_the_reference_loop_per_environment(groups):
    E, obs, A, H = 7, 5, 2, 13
    horizons = [H, H, 6, H, 9, H, H]  # two environments terminate early
    envs = [ro.LinearEnv(obs, A, seed=e, horizon=horizons[e]) for e in range(E)]
    P = _FakePlanner(A)
    rtg = lambda t: 1.0 - 0.01 * t  # noqa: E731
    out = ro.run_episodes(P, envs, rtg=rtg, max_path_length=H, groups=groups)
    assert out["lengths"].tolist() == horizons
    assert all(n >= 1 for n, _, _ in P.calls)
    for e in range(E):
        ref = _reference_loop(_FakePlanner(A), ro.LinearEnv(obs, A, seed=e, horizon=horizons[e]), rtg, H)
        tr = out["trajectories"][e]
        assert tr["path_length"] == ref["path_length"]
        for k in ("observations", "actions", "rewards"):
            np.testing.assert_array_equal(tr[k], ref[k], err_msg=f"env {e} {k}")
        assert abs(out["returns"][e] - float(ref["rewards"].sum())) < 1e-5
        assert float(np.abs(tr["actions"]).max()) <= 1.0  # clipped like learner.py:688


def test_evaluate_plan_batches_episodes():
    P = _FakePlanner(2)
    ref = np.linspace(1.0, 0.5, 10)
    res = ro.evaluate_plan(P, lambda: ro.LinearEnv(4, 2, seed=3, horizon=10), num_episodes=5, episode_rtg_ref=ref, n_envs=2, groups=2, max_path_length=10)
    assert res["episodes"] == 5 and res["length_mean"] == 10 and np.isfinite(res["return_mean"]) and res["return_std"] < 1e-9
    assert {c[2] for c in P.calls} == set(float(v) for v in ref)  # rtg = episode_rtg_ref[timestep]


@pytest.mark.parametrize("groups", [1, 3])
def test_run_episodes_is_the_refill_loop_with_one_episode_per_slot(groups):
    """run_episodes(envs) and evaluate_plan(refill=True) with as many slots as episodes are one loop: the same planner calls
    (sizes, lock-step path_length, rtg) in the same order and the same trajectories."""
    E, obs, A, H = 5, 4, 2, 9
    horizons = [H, 4, H, 7, H]
    ref = np.linspace(1.0, 0.5, H)
    mk = lambda: [ro.LinearEnv(obs, A, seed=20 + e, horizon=horizons[e]) for e in range(E)]  # noqa: E731
    P, Q = _FakePlanner(A), _FakePlanner(A)
    out = ro.run_episodes(P, mk(), rtg=lambda t: ref[min(t, H - 1)], max_path_length=H, groups=groups)
    envs = iter(mk())
    res = ro.evaluate_plan(Q, lambda: next(envs), num_episodes=E, episode_rtg_ref=ref, n_envs=E, groups=groups, max_path_length=H, refill=True)
    assert P.calls == Q.calls and len(P.calls) >= H
    assert out["lengths"].tolist() == res["lengths"] == horizons
    for a, b in zip(out["trajectories"], res["trajectories"]):
        for k in ("observations", "actions", "rewards", "values", "total_return", "path_length"):
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)


# ------------------------------------------------------------------------------------------------ GPU
def _gpu_learner(precision, n_cand, max_envs, guidance="critic_lambda_guiding"):
    from m3pc_b200.learner import Learner
    from m3pc_b200.mtm_model import omtmConfig
    from m3pc_b200.tokenizers import manager_from_stats
    shape = syn.shipped_shape("walker2d")
    cfg = SimpleNamespace(traj_length=shape.traj_length, device="cuda", action_samples=n_cand, discount=0.99, temperature=1.0, horizon=4,
                          plan_guidance=guidance, lmbda=0.6)
    mcfg = omtmConfig(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer, dropout=0.1,
                      norm="none", precision=precision, max_batch=n_cand * max_envs)
    om, os_ = syn.make_obs_norm(shape)
    L = Learner(cfg, None, shape.data_shapes, mcfg, None, om, os_, manager_from_stats(syn.make_tokenizer_stats(shape, 1)),
                {k: False for k in shape.data_shapes}, max_envs=max_envs)
    L.mtm.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 0).items()})
    L.iql.qf.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_critic_state_dict(shape).items()})
    return shape, L


@pytest.mark.gpu
def test_pipelined_rollout_matches_blocking_single_env_loop():
    """plan=False / eval=True is noise-free (tanh(mu)), so the pipelined E-environment rollout must reproduce the reference-style
    blocking loop of each environment (fp32 engine; contracting dynamics keep rounding differences from growing)."""
    shape, L = _gpu_learner("fp32", 8, 6)
    E, H = 6, 11  # crosses the horizon-clamp regime change at path_length + 4 >= 8
    mk = lambda e: ro.LinearEnv(shape.obs_dim, shape.act_dim, seed=40 + e, horizon=H if e != 2 else 7)  # noqa: E731
    out = ro.run_episodes(L, [mk(e) for e in range(E)], rtg=lambda t: 3.0, plan=False, eval=True, max_path_length=H, groups=3)
    assert out["lengths"].tolist() == [H, H, 7, H, H, H]
    for e in (0, 2, 5):
        env, tr = mk(e), ro.new_trajectory(shape.obs_dim, shape.act_dim, H)
        observation, done, t = env.reset(), False, 0
        while not done and t < H:
            tr["observations"][t] = observation
            action = np.clip(L.action_sample(tr, plan=False, eval=True, rtg=3.0).cpu().numpy()[0], -1, 1)
            observation, reward, done, _ = env.step(action)
            tr["actions"][t] = action
            tr["rewards"][t] = reward
            t += 1
            tr["path_length"] += 1
        np.testing.assert_allclose(out["trajectories"][e]["actions"], tr["actions"], atol=2e-4)
        np.testing.assert_allclose(out["trajectories"][e]["observations"], tr["observations"], atol=2e-4)


@pytest.mark.gpu
def test_evaluate_plan_with_the_planner_and_tickets():
    shape, L = _gpu_learner("bf16", 64, 4)
    res = ro.evaluate_plan(L, lambda: ro.LinearEnv(shape.obs_dim, shape.act_dim, seed=1, horizon=10), num_episodes=6,
                           episode_rtg_ref=np.full(10, 3.0), n_envs=4, groups=2, max_path_length=10)
    assert res["episodes"] == 6 and res["length_mean"] == 10 and np.isfinite(res["return_mean"])
    # a ticket delivers exactly what the blocking call returns (same seed, same window)
    hist = syn.make_history(shape, seed=2, path_length=30)
    L.__dict__["_plan_counter"] = 100
    a = L.action_sample_batch([hist, hist], plan=True, eval=True, rtg=3.0).cpu().numpy()
    L.__dict__["_plan_counter"] = 100
    t = L.action_sample_async([hist, hist], plan=True, eval=True, rtg=3.0)
    b = t.result()
    np.testing.assert_array_equal(a, b)
    with pytest.raises(RuntimeError):
        t.result()


@pytest.mark.gpu
def test_device_resident_episodes_build_the_same_windows_and_actions():
    """DeviceEpisodes on m3pc_ring_reset / _append_slots / _windows_slots (SURVEY.md section 8f rank 1), every slot at the same
    step: windows cut on the device from HBM-resident histories are bit-identical to the host window builder (learner.py:346-366
    semantics) at every step, across the horizon-clamp regime change, and the plans on them return the same actions."""
    E, H = 5, 13
    shape, L = _gpu_learner("bf16", 32, E)
    envs = [ro.LinearEnv(shape.obs_dim, shape.act_dim, seed=70 + e, horizon=H) for e in range(E)]
    trajs = [ro.new_trajectory(shape.obs_dim, shape.act_dim, 1000) for _ in range(E)]
    ep = ro.DeviceEpisodes(L, n_env=E, max_path_length=1000)
    obs = np.stack([env.reset() for env in envs])
    ep.start(obs)
    for e in range(E):
        trajs[e]["observations"][0] = obs[e]
    T = shape.traj_length
    for t in range(H):
        rtg = [3.0 - 0.1 * t + 0.01 * e for e in range(E)]
        L.__dict__["_plan_counter"] = 500 + t
        host = L.action_sample_batch(trajs, plan=True, eval=True, rtg=rtg).cpu().numpy()
        ring = L.__dict__["_win"][(shape.obs_dim, shape.act_dim, T, E)]
        hs, ha, hr, ht = ring.d_states.clone(), ring.d_actions.clone(), ring.d_rewards.clone(), ring.d_returns.clone()
        L.__dict__["_plan_counter"] = 500 + t
        dev = ep.plan_async(plan=True, eval=True, rtg=rtg).result()
        assert torch.equal(ep.win_states, hs) and torch.equal(ep.win_actions, ha), f"step {t}"
        assert torch.equal(ep.win_rewards, hr) and torch.equal(ep.win_returns, ht), f"step {t}"
        np.testing.assert_array_equal(dev, host)
        actions = np.clip(dev, -1, 1)
        nxt, rew = np.zeros_like(obs), np.zeros(E, np.float32)
        for e in range(E):
            o, r, _, _ = envs[e].step(actions[e])
            nxt[e], rew[e] = o, r
            trajs[e]["actions"][t], trajs[e]["rewards"][t] = actions[e], r
            trajs[e]["path_length"] += 1
            if t + 1 < 1000:
                trajs[e]["observations"][t + 1] = o
        ep.step(actions, rew, nxt)
    with pytest.raises(ValueError):
        ro.DeviceEpisodes(L, n_env=E + 1)
