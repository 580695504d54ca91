"""Zero-shot (backward, goal-reaching) planners on environments at different points of their episodes: ``m3pc_backward_plan_env``
(one horizon per environment), waypoint tables in the device-resident histories (``m3pc_ring_write_obs``), the ``*_async`` tickets
of the zero-shot Learner and zero-shot episodes through ``rollout.run_episodes`` / ``evaluate_plan``.  The CPU tests drive the
loop with stand-in planners; the GPU tests check the mixed plan bit for bit against the uniform plan of each horizon class, and
against the float64 oracle."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from m3pc_b200 import rollout as ro
from m3pc_b200 import synthetic as syn

MODES = {"id": 0, "piid": 1}
ERR_INVALID = -1  # M3PC_ERR_INVALID, include/m3pc.h


# ------------------------------------------------------------------------------------------------ CPU: the rollout surface
class _Ticket:
    def __init__(self, a):
        self.a = a

    def result(self):
        return self.a


class _ZeroShotStandIn:
    """Marks itself zero-shot like ``zeroshot_learner.Learner``.  action = tanh of the waypoint two steps ahead, so the actions
    show which rows the planner was handed."""
    _future_obs_windows = True
    zeroshot_mode = "piid"

    def __init__(self, act_dim):
        self.mtm = SimpleNamespace(data_shapes={"actions": (1, act_dim)})
        self.max_envs = 8

    def _plan(self, histories):
        A = self.mtm.data_shapes["actions"][1]
        return _Ticket(np.stack([np.tanh(h["observations"][h["path_length"] + 2, :A]) for h in histories]))

    def action_piid_sample_async(self, histories, percentage=1.0, eval=False, rtg=None):
        return self._plan(histories)

    def action_id_sample_async(self, histories, percentage=1.0, eval=False, rtg=None):
        raise AssertionError("mode piid was asked for")


class _ForwardStandIn:
    def __init__(self, act_dim):
        self.mtm = SimpleNamespace(data_shapes={"actions": (1, act_dim)})
        self.max_envs = 8

    def action_sample_async(self, histories, percentage=1.0, plan=True, eval=False, rtg=None):
        return _Ticket(np.zeros((len(histories), self.mtm.data_shapes["actions"][1]), np.float32))


def _table(i, obs, rows=1000):
    return np.random.RandomState(1000 + i).randn(rows, obs).astype(np.float32)


def test_run_episodes_rejects_missing_or_misplaced_waypoints():
    obs, A = 5, 2
    with pytest.raises(ValueError, match="waypoints"):
        ro.run_episodes(_ZeroShotStandIn(A), [ro.LinearEnv(obs, A)], rtg=lambda t: 1.0, max_path_length=5)
    with pytest.raises(ValueError, match="waypoints"):
        ro.run_episodes(_ForwardStandIn(A), [ro.LinearEnv(obs, A)], rtg=lambda t: 1.0, max_path_length=5, waypoints=lambda i: _table(i, obs))
    with pytest.raises(ValueError, match="waypoints"):
        ro.evaluate_plan(_ZeroShotStandIn(A), lambda: ro.LinearEnv(obs, A), num_episodes=2, episode_rtg_ref=np.ones(5), n_envs=2, refill=True)
    with pytest.raises(ValueError, match="mode"):
        ro.run_episodes(_ZeroShotStandIn(A), [ro.LinearEnv(obs, A)], rtg=lambda t: 1.0, max_path_length=5, waypoints=lambda i: _table(i, obs),
                        zeroshot_mode="forward")


@pytest.mark.parametrize("refill", [False, True])
def test_host_histories_hold_the_waypoints_ahead_of_the_episode(refill):
    """Rows 0 .. path_length of the history a zero-shot planner sees are the episode's observations, the rows after it the
    episode's own waypoint table (episode order also across evaluate_plan rounds)."""
    obs, A, H = 5, 2, 9
    lengths = [4, 9, 6, 2, 7]
    count = [0]

    def make_env():
        i = count[0]
        count[0] += 1
        return ro.LinearEnv(obs, A, seed=30 + i, horizon=lengths[i])

    P = _ZeroShotStandIn(A)
    out = ro.evaluate_plan(P, make_env, num_episodes=len(lengths), episode_rtg_ref=np.ones(H), n_envs=2, groups=1, max_path_length=H,
                           refill=refill, waypoints=lambda i: _table(i, obs, rows=40 + i))
    assert out["lengths"] == lengths
    for i, tr in enumerate(out["trajectories"]):
        wp = _table(i, obs, rows=40 + i)
        n = tr["path_length"]
        assert tr["observations"].shape[0] == ro.WAYPOINT_ROWS
        np.testing.assert_array_equal(tr["observations"][n + 1:40 + i], wp[n + 1:])
        assert not tr["observations"][40 + i:].any()
        env = ro.LinearEnv(obs, A, seed=30 + i, horizon=lengths[i])
        o = env.reset()
        for t in range(n):  # the actions are tanh of waypoint t + 2, so the replayed observations are the episode's own
            np.testing.assert_array_equal(tr["observations"][t], o)
            np.testing.assert_array_equal(tr["actions"][t], np.clip(np.tanh(wp[t + 2, :A]), -1, 1))
            o, _, _, _ = env.step(tr["actions"][t])


# ------------------------------------------------------------------------------------------------ GPU: engine level
def _engine(precision, max_batch=256):
    from m3pc_b200.engine import engine_from_synthetic
    shape = syn.shipped_shape("hopper")
    eng = engine_from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), precision=precision, max_batch=max_batch)
    return shape, eng


def _windows(shape, E, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    T = shape.traj_length
    return (torch.randn(E, T, shape.obs_dim, device="cuda", generator=g), torch.rand(E, T, shape.act_dim, device="cuda", generator=g) * 2 - 1,
            torch.randn(E, T, device="cuda", generator=g), torch.randn(E, T, device="cuda", generator=g))


def _uniform(eng, mode, h, win, eps=None, n_draws=None, seed=0):
    ev, sm, _ = eng.backward_plan(mode=mode, horizon=h, win_states=win[0].contiguous(), win_actions=win[1].contiguous(),
                                  win_rewards=win[2].contiguous(), win_returns_tok=win[3].contiguous(), eps=eps, n_draws=n_draws, seed=seed)
    return ev.clone(), sm.clone()


def _env_call(eng, mode, hz, win, eps=None, n_draws=1, seed=0):
    """m3pc_backward_plan_env straight through the C ABI: (rc, eval (E, A), draws (E, C, A), launches)."""
    from m3pc_b200 import _native as nat
    E, A = win[0].shape[0], eng.act
    hz = np.ascontiguousarray(np.asarray(hz, dtype=np.int32))
    ev = torch.full((E, A), float("nan"), device="cuda")
    sm = torch.full((E, n_draws, A), float("nan"), device="cuda")
    ws, wa, wr, wt = (w.contiguous() for w in win)
    rc = nat.lib().m3pc_backward_plan_env(eng._h, MODES[mode], E, hz.ctypes.data_as(C.c_void_p), n_draws, ws.data_ptr(), wa.data_ptr(), wr.data_ptr(),
                                          wt.data_ptr(), None if eps is None else eps.contiguous().data_ptr(), seed, ev.data_ptr(), sm.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, ev, sm, eng.last_launch_count()


def _classes(hz):
    return [(h, [e for e in range(len(hz)) if hz[e] == h]) for h in sorted(set(hz))]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("mode", ["id", "piid"])
def test_mixed_horizon_backward_plan_equals_the_uniform_plan_of_each_class(precision, mode):
    """Path lengths 0 .. 3 (horizons 8, 7, 6, 5 at T = 8, h = 4) mixed with steady-state windows (h = 4); injected noise."""
    shape, eng = _engine(precision)
    T, A = shape.traj_length, shape.act_dim
    hz = [4, 8, 4, 7, 6, 5, 4, 8, 4, 5, 4]
    E = len(hz)
    win = _windows(shape, E)
    g = torch.Generator(device="cuda").manual_seed(1)
    eps = torch.randn(E, A, device="cuda", generator=g)
    ev, sm, _ = eng.backward_plan(mode=mode, horizon=max(hz), win_states=win[0], win_actions=win[1], win_rewards=win[2], win_returns_tok=win[3],
                                  eps=eps, env_horizons=hz)
    assert ev.shape == (E, A) and sm.shape == (E, A) and torch.isfinite(sm).all()
    for h, members in _classes(hz):
        uev, usm = _uniform(eng, mode, h, tuple(w[members] for w in win), eps=eps[members].contiguous())
        for i, e in enumerate(members):
            assert torch.equal(ev[e], uev[i]) and torch.equal(sm[e], usm[i]), (h, e)
    # the draws variant at the config-4 shape: C = 512 draws per environment, E = 256
    E, Cn = 256, 512
    hz = [[4, 8, 7, 6, 5][e % 5] if e % 3 == 0 else 4 for e in range(E)]
    win = _windows(shape, E, seed=2)
    eps = torch.randn(E, Cn, A, device="cuda", generator=g)
    ev, sm, _ = eng.backward_plan(mode=mode, horizon=max(hz), win_states=win[0], win_actions=win[1], win_rewards=win[2], win_returns_tok=win[3],
                                  eps=eps, n_draws=Cn, env_horizons=hz)
    assert sm.shape == (E, Cn, A)
    for h, members in _classes(hz):
        uev, usm = _uniform(eng, mode, h, tuple(w[members] for w in win), eps=eps[members].contiguous(), n_draws=Cn)
        idx = torch.tensor(members, device="cuda")
        assert torch.equal(ev[idx], uev) and torch.equal(sm[idx], usm), h


@pytest.mark.gpu
@pytest.mark.parametrize("injected", [False, True])
def test_equal_horizons_are_exactly_the_existing_entry(injected):
    shape, eng = _engine("bf16")
    E, Cn, h, A = 12, 16, 5, shape.act_dim
    win = _windows(shape, E, seed=3)
    eps = torch.randn(E, Cn, A, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4)) if injected else None
    for mode in MODES:
        uev, usm = _uniform(eng, mode, h, win, eps=eps, n_draws=Cn, seed=77)
        n_uniform = eng.last_launch_count()
        rc, ev, sm, n = _env_call(eng, mode, [h] * E, win, eps=eps, n_draws=Cn, seed=77)
        assert rc == 0 and n == n_uniform
        assert torch.equal(ev, uev) and torch.equal(sm, usm)
        # C = 1 with eps (E, A): exactly m3pc_backward_plan
        if injected:
            e1 = eps[:, 0].contiguous()
            uev, usm = _uniform(eng, mode, h, win, eps=e1)
            rc, ev, sm, _ = _env_call(eng, mode, [h] * E, win, eps=e1, n_draws=1)
            assert rc == 0 and torch.equal(ev, uev) and torch.equal(sm[:, 0], usm)


@pytest.mark.gpu
def test_mixed_backward_plan_philox_is_keyed_by_the_callers_environment():
    """Same seed, same caller index: a row's draws stay bit-identical when the other rows change their horizons and windows (the
    horizon classes of the call change, a row's own class keeps its size); another seed draws differently."""
    shape, eng = _engine("fp32")
    Cn = 64
    win = _windows(shape, 4, seed=5)
    other = _windows(shape, 4, seed=6)
    mixed = tuple(torch.cat([w[:1], o[1:]]) for w, o in zip(win, other))  # row 0 kept, rows 1..3 replaced
    for mode in MODES:
        _, _, a, _ = _env_call(eng, mode, [4, 8, 8, 8], win, n_draws=Cn, seed=9)
        _, _, b, _ = _env_call(eng, mode, [4, 6, 6, 6], mixed, n_draws=Cn, seed=9)
        _, _, c, _ = _env_call(eng, mode, [5, 8, 8, 8], tuple(torch.cat([o[:1], w[1:]]) for w, o in zip(win, other)), n_draws=Cn, seed=9)
        _, _, d, _ = _env_call(eng, mode, [4, 8, 8, 8], win, n_draws=Cn, seed=10)
        assert torch.isfinite(a).all()
        assert torch.equal(a[0], b[0])      # environment 0 at h = 4 alone in its class in both calls
        assert torch.equal(a[1:], c[1:])    # environments 1..3 at h = 8 in a class of three in both calls
        assert not torch.equal(a[1], a[2])  # different environments, different draws
        assert not torch.equal(a[0, 0], a[0, 1])
        assert not torch.equal(a, d)        # another seed
        # the same windows as a lock-step call keyed by the same caller indices: row 0 of the uniform call at h = 4
        _, _, u, _ = _env_call(eng, mode, [4], tuple(w[:1] for w in win), n_draws=Cn, seed=9)
        assert torch.equal(u[0], a[0])


@pytest.mark.gpu
def test_invalid_env_horizons_are_rejected_before_any_launch():
    from m3pc_b200 import _native as nat
    shape, eng = _engine("bf16")
    T = shape.traj_length
    win = _windows(shape, 257)
    for hz, n in (([4, 0, 4], 3), ([4, T + 1, 4], 3), ([4] * 257, 257), ([4, 5] * 128 + [6], 257)):
        rc, _, _, launches = _env_call(eng, "piid", hz, tuple(w[:n] for w in win))
        assert rc == ERR_INVALID and launches == 0, hz[:4]
        assert nat.lib().m3pc_last_error().decode()
    with pytest.raises(ValueError):  # horizon must be the largest entry
        eng.backward_plan(mode="id", horizon=6, win_states=win[0][:3], win_actions=win[1][:3], win_rewards=win[2][:3],
                          win_returns_tok=win[3][:3], env_horizons=[4, 5, 7])
    rc, ev, _, _ = _env_call(eng, "piid", [4, 5, 6], tuple(w[:3] for w in win))  # still usable
    assert rc == 0 and torch.isfinite(ev).all()


# ------------------------------------------------------------------------------------------------ GPU: Learner level
def _zs_learner(precision, max_envs):
    from m3pc_b200.mtm_model import omtmConfig
    from m3pc_b200.tokenizers import manager_from_stats
    from m3pc_b200.zeroshot_learner import Learner as ZL
    shape = syn.shipped_shape("hopper")
    cfg = SimpleNamespace(traj_length=shape.traj_length, device="cuda", action_samples=1, discount=0.99, temperature=0.01, horizon=4,
                          plan_guidance="rtg_guiding", lmbda=0.6)
    mcfg = omtmConfig(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer, dropout=0.1,
                      norm="none", precision=precision, max_batch=max_envs)
    om, os_ = syn.make_obs_norm(shape)
    L = ZL(cfg, None, shape.data_shapes, mcfg, None, om, os_, manager_from_stats(syn.make_tokenizer_stats(shape, 1)),
           {k: False for k in shape.data_shapes}, max_envs=max_envs)
    L.mtm.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 0).items()})
    return shape, L


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_mixed_batch_rows_match_the_fp64_oracle_at_their_own_horizon(precision):
    """Every row of a mixed batch (path_length 0 .. 3, steady state, and p + h > 1000 where the waypoints run out) equals the
    oracle's B = 1 zero-shot planner on its history, eval and injected-noise sample, id and piid."""
    from oracle import planner_oracle as po
    shape, L = _zs_learner(precision, 16)
    T, A = shape.traj_length, shape.act_dim
    P = po.from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), dtype=torch.float64, action_samples=1)
    pls = [0, 1, 2, 3, 40, 997, 998, 999, 2, 500]
    hists = [syn.make_history(shape, seed=70 + i, path_length=p) for i, p in enumerate(pls)]
    assert len({L._clamped_horizon(h) for h in hists}) == 5
    eps = torch.from_numpy(np.random.RandomState(8).randn(len(pls), A)).float()
    L.injected_eps = eps.cuda()
    atol = 1e-4 if precision == "fp32" else 2e-2
    for mode, fn in (("id", P.action_id_sample), ("piid", P.action_piid_sample)):
        batch = getattr(L, f"action_{mode}_sample_batch")
        ev = batch(hists, eval=True, rtg=2.0).cpu().numpy()
        sm = batch(hists, eval=False, rtg=2.0).cpu().numpy()
        for e, hist in enumerate(hists):
            h = L._clamped_horizon(hist)
            e1 = torch.zeros(1, T, 1, A, dtype=torch.float64)
            e1[0, T - h, 0] = eps[e].double()
            ref_ev, _ = fn(hist, eval=True, rtg=2.0)
            ref_sm, _ = fn(hist, eval=False, rtg=2.0, eps1=e1)
            np.testing.assert_allclose(ev[e], ref_ev.numpy().reshape(-1), atol=atol, err_msg=f"{mode} p={pls[e]}")
            np.testing.assert_allclose(sm[e], ref_sm.numpy().reshape(-1), atol=atol, err_msg=f"{mode} p={pls[e]}")
        ticket = getattr(L, f"action_{mode}_sample_async")(hists, eval=True, rtg=2.0)
        np.testing.assert_array_equal(ticket.result(), ev)


@pytest.mark.gpu
def test_device_windows_with_waypoints_equal_the_host_builder_around_the_clamp():
    """reset + waypoints, then appends: the device windows (future_obs) of every active slot are bit-identical to the host
    builder on a history whose observations hold the waypoints, step by step up to p = 999 (p + h > 1000), across resets with
    new tables (one shorter than the episode) and an idle slot."""
    shape, L = _zs_learner("bf16", 4)
    E, T, obs, A = 4, shape.traj_length, shape.obs_dim, shape.act_dim
    rs = np.random.RandomState(3)
    ep = ro.DeviceEpisodes(L, n_env=E, max_path_length=1000)
    assert ep.L == 1000
    trajs = [None] * E

    def fresh(s, rows):
        tab = rs.randn(rows, obs).astype(np.float32)
        tr = ro.new_trajectory(obs, A, 1000)
        tr["observations"][:rows] = tab
        tr["observations"][0] = rs.randn(obs).astype(np.float32)
        trajs[s] = tr
        return tab, tr["observations"][0]

    tabs, firsts = zip(*[fresh(s, 1000) for s in range(E)])
    ep.start(np.stack(firsts), waypoints=list(tabs))
    win = np.zeros((T, obs), np.float32), np.zeros((T, A), np.float32), np.zeros(T, np.float32), np.zeros(T, np.float32)
    checked = 0
    for step in range(1000):
        if step == 7:  # slot 1 starts a new episode with a short table
            tab, o = fresh(1, 12)
            ep.reset([1], o[None], waypoints=[tab])
        if step == 30:
            ep.release([2])
        act = ep.active
        if step < 16 or step > 980 or step % 97 == 0:
            rtg = [2.0 + 0.1 * s for s in act]
            ep.windows(act, rtg=rtg)
            n = len(act)
            dev = [x[:n].cpu().numpy() for x in (ep.win_states, ep.win_actions, ep.win_rewards, ep.win_returns)]
            for k, s in enumerate(act):
                L._fill_window(*win, trajs[s], L._clamped_horizon(trajs[s]), 1.0, rtg[k], future_obs=True)
                for d, hst in zip(dev, win):
                    np.testing.assert_array_equal(d[k], hst, err_msg=f"step {step} slot {s}")
                checked += 1
        if step == 999:
            break
        a = rs.uniform(-1, 1, size=(len(act), A)).astype(np.float32)
        r = rs.randn(len(act)).astype(np.float32)
        nxt = rs.randn(len(act), obs).astype(np.float32)
        for k, s in enumerate(act):
            t = trajs[s]["path_length"]
            trajs[s]["actions"][t], trajs[s]["rewards"][t] = a[k], r[k]
            trajs[s]["path_length"] += 1
            trajs[s]["observations"][t + 1] = nxt[k]
        ep.step(a, r, nxt, slots=act)
    assert trajs[0]["path_length"] == 999 and checked > 60


@pytest.mark.gpu
@pytest.mark.parametrize("device_histories", [False, True])
def test_zeroshot_refill_rollout_matches_blocking_single_env_loop(device_histories):
    """eval=True is noise-free (tanh(mu)), so every episode of the refilling zero-shot rollout must reproduce the blocking
    single-environment loop that calls ``action_piid_sample`` each step on the history holding the episode's waypoints (fp32)."""
    shape, L = _zs_learner("fp32", 3)
    obs, A = shape.obs_dim, shape.act_dim
    H, lengths = 12, [7, 12, 4, 9, 5, 11]
    count = [0]

    def make_env():
        i = count[0]
        count[0] += 1
        return ro.LinearEnv(obs, A, seed=60 + i, horizon=lengths[i])

    def waypoints(i):
        return np.random.RandomState(90 + i).randn(20 + i, obs).astype(np.float32)

    out = ro.evaluate_plan(L, make_env, num_episodes=len(lengths), episode_rtg_ref=np.full(H, 3.0), n_envs=3, groups=2, max_path_length=H,
                           refill=True, device_histories=device_histories, eval=True, waypoints=waypoints, zeroshot_mode="piid")
    assert out["lengths"] == lengths
    for i in range(len(lengths)):
        env, tr = ro.LinearEnv(obs, A, seed=60 + i, horizon=lengths[i]), ro.new_trajectory(obs, A, 1000)
        wp = waypoints(i)
        tr["observations"][:len(wp)] = wp
        observation, done, t = env.reset(), False, 0
        while not done and t < H:
            tr["observations"][t] = observation
            action = np.clip(L.action_piid_sample(tr, eval=True, rtg=3.0).cpu().numpy()[0], -1, 1)
            observation, reward, done, _ = env.step(action)
            tr["actions"][t] = action
            tr["rewards"][t] = reward
            t += 1
            tr["path_length"] += 1
        np.testing.assert_allclose(out["trajectories"][i]["actions"], tr["actions"], atol=2e-4)
        np.testing.assert_allclose(out["trajectories"][i]["observations"], tr["observations"], atol=2e-4)
