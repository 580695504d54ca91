"""Environments at different points of their episodes: ``m3pc_plan`` with one horizon per environment, per-slot clocks in the
device-resident histories (``m3pc_ring_reset`` / ``_append_slots`` / ``_windows_slots``) and ``evaluate_plan(refill=True)``.
The CPU tests drive the refilling loop with a stand-in planner; the GPU tests check the mixed plan bit for bit against the
uniform plan of each horizon class."""
import itertools
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from m3pc_b200 import rollout as ro
from m3pc_b200 import synthetic as syn


# ------------------------------------------------------------------------------------------------ CPU: refilling slots
class _Ticket:
    def __init__(self, a):
        self.a = a

    def result(self):
        return self.a


class _AnyStepPlanner:
    """action = 2 tanh(first act_dim features of the latest observation) * rtg of that environment; accepts environments at any
    path_length and records (environments per call, episodes started so far) for every call."""

    def __init__(self, act_dim, started):
        self.mtm = SimpleNamespace(data_shapes={"actions": (1, act_dim)})
        self.max_envs = 64
        self.calls = []
        self.started = started

    def action_sample_async(self, histories, percentage=1.0, plan=True, eval=False, rtg=None):
        self.calls.append((len(histories), self.started[0]))
        A = self.mtm.data_shapes["actions"][1]
        r = rtg if isinstance(rtg, (list, tuple)) else [rtg] * len(histories)
        return _Ticket(np.stack([2.0 * np.tanh(h["observations"][h["path_length"], :A]) * r[i] for i, h in enumerate(histories)]))


def _reference_episode(env, act_dim, rtg, max_path_length):
    """The reference's single-environment loop (learner.py:663-696) with the stand-in planner's rule."""
    tr = ro.new_trajectory(env.x0.shape[0], act_dim, max_path_length)
    observation, done, t = env.reset(), False, 0
    while not done and t < max_path_length:
        tr["observations"][t] = observation
        action = np.clip(2.0 * np.tanh(observation[:act_dim]) * float(rtg(t)), -1, 1)
        observation, reward, done, _ = env.step(action)
        tr["actions"][t] = action
        tr["rewards"][t] = reward
        tr["total_return"] += float(reward)
        t += 1
        tr["path_length"] += 1
    return tr


@pytest.mark.parametrize("n_envs,groups", [(3, 1), (3, 2), (4, 3), (16, 2)])
def test_refill_runs_every_episode_as_the_reference_loop(n_envs, groups):
    obs, A, H = 5, 2, 14
    lengths = [9, 3, 14, 5, 11, 2, 7, 14, 4, 6]  # episodes end at different steps; 14 = max_path_length
    started = [0]

    def make_env():
        i = started[0]
        started[0] += 1
        return ro.LinearEnv(obs, A, seed=100 + i, horizon=lengths[i])

    ref_rtg = np.linspace(1.0, 0.3, H)
    P = _AnyStepPlanner(A, started)
    out = ro.evaluate_plan(P, make_env, num_episodes=len(lengths), episode_rtg_ref=ref_rtg, n_envs=n_envs, groups=groups, max_path_length=H,
                           refill=True)
    assert out["episodes"] == len(lengths) and out["lengths"] == lengths
    rtg = lambda t: ref_rtg[min(t, H - 1)]  # noqa: E731
    for i, n in enumerate(lengths):
        ref = _reference_episode(ro.LinearEnv(obs, A, seed=100 + i, horizon=n), A, rtg, H)
        tr = out["trajectories"][i]
        assert tr["path_length"] == ref["path_length"] == n
        for k in ("observations", "actions", "rewards"):
            np.testing.assert_array_equal(tr[k], ref[k], err_msg=f"episode {i} {k}")
        assert out["returns"][i] == pytest.approx(ref["total_return"], abs=1e-6)
    # while episodes are still queued, every plan covers all slots of its group
    slots = min(n_envs, len(lengths))
    sizes = [len(r) for r in ro._split(slots, groups)]
    for k, (n, started_then) in enumerate(P.calls):
        if started_then < len(lengths):
            assert n == sizes[k % len(sizes)], (k, n, started_then)


def test_refill_keeps_the_lock_step_default_and_rejects_device_histories_without_refill():
    started = [0]
    P = _AnyStepPlanner(2, started)
    with pytest.raises(ValueError):
        ro.evaluate_plan(P, lambda: ro.LinearEnv(4, 2), num_episodes=2, episode_rtg_ref=np.ones(3), n_envs=2, device_histories=True)


# ------------------------------------------------------------------------------------------------ GPU: engine level
def _engine(precision, max_batch, chunk=0):
    from m3pc_b200.engine import engine_from_synthetic
    shape = syn.shipped_shape("walker2d")
    eng = engine_from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), precision=precision,
                                max_batch=max_batch, chunk=chunk, critic_sd=syn.make_critic_state_dict(shape), obs_norm=syn.make_obs_norm(shape))
    return shape, eng


def _windows(shape, E, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    T = shape.traj_length
    return (torch.randn(E, T, shape.obs_dim, device="cuda", generator=g), torch.rand(E, T, shape.act_dim, device="cuda", generator=g) * 2 - 1,
            torch.randn(E, T, device="cuda", generator=g), torch.randn(E, T, device="cuda", generator=g))


def _plan(eng, guidance, h, N, win, E, **kw):
    ws, wa, wr, wt = (w if E > 1 else w[0] for w in win)
    ev, sm, dbg = eng.plan(guidance=guidance, horizon=h, n_cand=N, win_states=ws.contiguous(), win_actions=wa.contiguous(),
                           win_rewards=wr.contiguous(), win_returns_tok=wt.contiguous(), discount=0.99, temperature=1.0, lmbda=0.6, n_env=E, **kw)
    ev, sm = ev.reshape(E, -1).clone(), sm.reshape(E, -1).clone()
    return ev, sm, {k: v.clone() for k, v in dbg.items()}


def _classes(hz):
    return [(h, [e for e in range(len(hz)) if hz[e] == h]) for h in sorted(set(hz))]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("guidance", ["rtg_guiding", "critic_lambda_guiding", "noise_adding_lambda"])
def test_mixed_horizon_plan_equals_the_uniform_plan_of_each_class(precision, guidance):
    E, N, hz = 5, 96, [4, 8, 4, 6, 4]
    hmax = max(hz)
    shape, eng = _engine(precision, E * N, chunk=200)  # a chunk that does not divide the pass-2 rows
    A = shape.act_dim
    win = _windows(shape, E)
    g = torch.Generator(device="cuda").manual_seed(1)
    eps = torch.randn(E * N, hmax, A, device="cuda", generator=g)
    q = -torch.log(torch.rand(E * N, device="cuda", generator=g))
    ev, sm, dbg = _plan(eng, guidance, hmax, N, win, E, eps=eps, expq=q, debug=True, env_horizons=hz)
    for h, members in _classes(hz):
        Ec = len(members)
        rows = torch.cat([torch.arange(e * N, (e + 1) * N, device="cuda") for e in members])
        cwin = tuple(w[members] for w in win)
        uev, usm, ud = _plan(eng, guidance, h, N, cwin, Ec, eps=eps[rows, :h].contiguous(), expq=q[rows].contiguous(), debug=True)
        for i, e in enumerate(members):
            assert torch.equal(ev[e], uev[i]) and torch.equal(sm[e], usm[i]), (h, e)
            assert torch.equal(dbg["expect_return"][e * N:(e + 1) * N], ud["expect_return"][i * N:(i + 1) * N]), (h, e)
            assert torch.equal(dbg["candidates"][e * N:(e + 1) * N, :h], ud["candidates"][i * N:(i + 1) * N]), (h, e)
            assert torch.equal(dbg["indices"].reshape(E, 2)[e], ud["indices"].reshape(Ec, 2)[i]), (h, e)
    # plan = False (mtm_sampling): eps (E, A)
    eps3 = torch.randn(E, A, device="cuda", generator=g)
    ev, sm, _ = _plan(eng, "mtm_sampling", hmax, N, win, E, eps=eps3, env_horizons=hz)
    for h, members in _classes(hz):
        uev, usm, _ = _plan(eng, "mtm_sampling", h, N, tuple(w[members] for w in win), len(members), eps=eps3[members].contiguous())
        for i, e in enumerate(members):
            assert torch.equal(ev[e], uev[i]) and torch.equal(sm[e], usm[i]), (h, e)


@pytest.mark.gpu
@pytest.mark.parametrize("injected", [False, True])
def test_equal_horizons_are_exactly_the_uniform_plan(injected):
    E, N, h = 8, 128, 4
    kw = {}
    if injected:
        g = torch.Generator(device="cuda").manual_seed(2)
        kw = dict(eps=torch.randn(E * N, h, 6, device="cuda", generator=g), expq=-torch.log(torch.rand(E * N, device="cuda", generator=g)),
                  debug=True)
    for guidance in ("critic_lambda_guiding", "mtm_sampling"):
        if injected and guidance == "mtm_sampling":
            continue
        runs = {}
        for hz in (None, [h] * E):
            shape, eng = _engine("bf16", E * N)  # one engine each: the graph cache starts empty for both
            assert shape.act_dim == 6
            win = _windows(shape, E, seed=3)
            out = []
            for _ in range(3):  # eager, captured, replayed
                ev, sm, dbg = _plan(eng, guidance, h, N, win, E, seed=11, env_horizons=hz, **kw)
                out.append((ev, sm, dbg, eng.last_launch_count()))
            runs[hz is None] = out
            eng.close()
        for (a, b) in zip(runs[True], runs[False]):
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and a[3] == b[3]
            for k in a[2]:
                assert torch.equal(a[2][k], b[2][k]), k


@pytest.mark.gpu
def test_mixed_plan_philox_graphs_and_independence_from_other_environments():
    E, N = 4, 256
    shape, eng = _engine("fp32", E * N)
    win = _windows(shape, E, seed=5)
    pa, pb = [8, 4, 4, 4], [8, 7, 6, 5]
    seq = []
    for hz in (pa, pb, pa, pb, pa, pb, pa):  # two patterns alternate: each must keep replaying its own graph
        ev, sm, _ = _plan(eng, "critic_lambda_guiding", 8, N, win, E, seed=21, env_horizons=hz)
        seq.append((hz, ev, sm, eng.last_launch_count()))
    assert torch.isfinite(seq[0][2]).all()
    for k, (hz, ev, sm, n) in enumerate(seq[2:]):
        ref, rep_ = (seq[0], seq[2]) if hz is pa else (seq[1], seq[3])  # first sighting runs eagerly; then captured and replayed
        assert torch.equal(ev, ref[1]) and torch.equal(sm, ref[2]) and n == rep_[3], k
    eng.set_option("graphs", 0)
    for hz, ev, sm, n in seq[:2]:
        e2, s2, _ = _plan(eng, "critic_lambda_guiding", 8, N, win, E, seed=21, env_horizons=hz)
        assert torch.equal(e2, ev) and torch.equal(s2, sm)
        assert eng.last_launch_count() == n
    # an environment's candidates do not depend on the horizons of the others (same class sizes, different other horizons)
    _, _, d1 = _plan(eng, "critic_lambda_guiding", 8, N, win, E, seed=21, env_horizons=[8, 4, 4, 4], debug=True)
    _, _, d2 = _plan(eng, "critic_lambda_guiding", 8, N, win, E, seed=21, env_horizons=[8, 5, 5, 5], debug=True)
    _, _, d3 = _plan(eng, "critic_lambda_guiding", 6, N, win, E, seed=21, env_horizons=[6, 4, 4, 4], debug=True)
    assert torch.equal(d1["candidates"][:N], d2["candidates"][:N])          # environment 0 at h = 8 alone in its class
    assert torch.equal(d1["candidates"][N:, :4], d3["candidates"][N:, :4])  # environments 1..3 at h = 4, three in their class
    assert not torch.equal(d1["candidates"][N:2 * N, :4], d1["candidates"][2 * N:3 * N, :4])  # different environments, different draws


@pytest.mark.gpu
def test_mixed_plan_rejects_invalid_horizons():
    E, N = 3, 64
    shape, eng = _engine("bf16", E * N)
    win = _windows(shape, E)
    T = shape.traj_length
    for hz, h in (([4, 0, 4], 4), ([4, T + 1, 4], T + 1), ([4, 6, 5], 5), ([4, 6, 5], 8), ([4, 4], 4)):
        with pytest.raises(ValueError):
            _plan(eng, "critic_lambda_guiding", h, N, win, E, env_horizons=hz)
    with pytest.raises(ValueError):  # candidate sharding (exchange) plans one uniform environment
        _plan(eng, "critic_lambda_guiding", 4, N, win, 1, env_horizons=[4], exchange=True)
    ev, _, _ = _plan(eng, "critic_lambda_guiding", 6, N, win, E, env_horizons=[4, 6, 5])  # still usable
    assert torch.isfinite(ev).all()


# ------------------------------------------------------------------------------------------------ GPU: slots and rollouts
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
def test_slots_with_resets_build_host_windows_and_actions():
    """Slots at different clocks, episodes that end and restart mid-run, a slot that goes idle: the device windows of the active
    slots are bit-identical to the host window builder on each slot's own history, and the plans return the same actions as
    ``action_sample_batch`` on those histories (same seeds)."""
    E, steps = 4, 24
    shape, L = _gpu_learner("bf16", 32, E)
    T = shape.traj_length
    lengths = itertools.cycle([5, 11, 3, 9, 13, 2, 6, 7, 4, 8, 3, 5, 10])
    ep = ro.DeviceEpisodes(L, n_env=E, max_path_length=1000)
    envs, trajs = [None] * E, [None] * E

    def fresh(s):
        envs[s] = ro.LinearEnv(shape.obs_dim, shape.act_dim, seed=200 + s + 10 * sum(t is not None for t in trajs), horizon=next(lengths))
        o = envs[s].reset()
        trajs[s] = ro.new_trajectory(shape.obs_dim, shape.act_dim, 1000)
        trajs[s]["observations"][0] = o
        return o

    ep.start(np.stack([fresh(s) for s in range(E)]))
    for step in range(steps):
        act = ep.active
        if step == 15:  # slot 1 goes idle for good
            ep.release([1])
            act = ep.active
        rtg = [3.0 - 0.05 * trajs[s]["path_length"] + 0.01 * s for s in act]
        L.__dict__["_plan_counter"] = 900 + step
        host = L.action_sample_batch([trajs[s] for s in act], plan=True, eval=False, rtg=rtg).cpu().numpy()
        ring = L.__dict__["_win"][(shape.obs_dim, shape.act_dim, T, len(act))]
        hw = [x.reshape(len(act), T, -1).clone() for x in (ring.d_states, ring.d_actions, ring.d_rewards, ring.d_returns)]
        L.__dict__["_plan_counter"] = 900 + step
        dev = ep.plan_async(plan=True, eval=False, rtg=rtg).result()
        n = len(act)
        dw = [ep.win_states[:n], ep.win_actions[:n], ep.win_rewards[:n, :, None], ep.win_returns[:n, :, None]]
        for a, b in zip(dw, hw):
            assert torch.equal(a, b), f"step {step}"
        np.testing.assert_array_equal(dev, host, err_msg=f"step {step}")
        acts = np.clip(dev, -1, 1)
        going, ended, nxt, rew = [], [], [], []
        for row, s in enumerate(act):
            o, r, done, _ = envs[s].step(acts[row])
            t = trajs[s]["path_length"]
            trajs[s]["actions"][t], trajs[s]["rewards"][t] = acts[row], r
            trajs[s]["path_length"] += 1
            if done:
                ended.append(s)
            else:
                trajs[s]["observations"][t + 1] = o
                going.append(row)
                nxt.append(o)
                rew.append(r)
        if going:
            ep.step(acts[going], np.array(rew, np.float32), np.stack(nxt), slots=[act[r_] for r_ in going])
        for s in ended:
            ep.reset([s], fresh(s)[None])
    assert ep.active.tolist() == [0, 2, 3]


@pytest.mark.gpu
@pytest.mark.parametrize("device_histories", [False, True])
def test_refill_rollout_matches_blocking_single_env_loop(device_histories):
    """plan=False / eval=True is noise-free (tanh(mu)), so every episode of the refilling rollout must reproduce the blocking
    single-environment loop (fp32 engine; contracting dynamics keep rounding differences from growing)."""
    shape, L = _gpu_learner("fp32", 8, 3)
    H, lengths = 12, [7, 12, 4, 9, 5, 11]
    count = [0]

    def make_env():
        i = count[0]
        count[0] += 1
        return ro.LinearEnv(shape.obs_dim, shape.act_dim, seed=60 + i, horizon=lengths[i])

    out = ro.evaluate_plan(L, make_env, num_episodes=len(lengths), episode_rtg_ref=np.full(H, 3.0), n_envs=3, groups=2, max_path_length=H,
                           refill=True, device_histories=device_histories, plan=False, eval=True)
    assert out["lengths"] == lengths
    for i in range(len(lengths)):
        env, tr = ro.LinearEnv(shape.obs_dim, shape.act_dim, seed=60 + i, horizon=lengths[i]), ro.new_trajectory(shape.obs_dim, shape.act_dim, H)
        observation, done, t = env.reset(), False, 0
        while not done and t < H:
            tr["observations"][t] = observation
            action = np.clip(L.action_sample(tr, plan=False, eval=True, rtg=3.0).cpu().numpy()[0], -1, 1)
            observation, reward, done, _ = env.step(action)
            tr["actions"][t] = action
            tr["rewards"][t] = reward
            t += 1
            tr["path_length"] += 1
        np.testing.assert_allclose(out["trajectories"][i]["actions"], tr["actions"], atol=2e-4)
        np.testing.assert_allclose(out["trajectories"][i]["observations"], tr["observations"], atol=2e-4)
