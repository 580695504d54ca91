"""The caller loops around the planning path, vectorised and pipelined (SURVEY.md section 8f rank 3).

Reference loops (one environment, one blocking plan per step):

  ReplayBuffer.online_rollout(sample_func=learner.action_sample)    finetune_omtm/replay_buffer.py:167-232
  Learner.evaluate_plan(num_episodes, episode_rtg_ref)              finetune_omtm/learner.py:648-720

Both build ``current_trajectory`` (zero-filled (1000, d) arrays + ``path_length``), call ``action_sample`` on it, clip the
action, ``env.step`` it and write action / reward back.  Here one loop (``_run``) runs episodes through E environment slots split
into G groups: while group g's environments step on the host, the plans of the other groups run on the GPU
(``Learner.action_sample_async`` tickets), so neither side waits for the other.  When an episode ends and more are queued, the
next one starts in that slot at once, so a plan may cover environments at different points of their episodes.
``run_episodes`` queues exactly one episode per slot, so its groups stay in lock-step; with G = 1 and E = 1 it degenerates to the
reference's loop.  ``evaluate_plan`` runs rounds of ``run_episodes`` or, with ``refill=True``, streams all its episodes through
the slots.  Environments use the reference's (old gym) protocol: ``reset() -> obs``, ``step(a) -> (obs, r, done, info)``.

Zero-shot (goal-reaching) learners (``m3pc_b200.zeroshot_learner``) run through the same loop: each episode gets a waypoint table
(``waypoints(episode) -> (L, obs)``) that fills its history's ``observations`` before the episode's own observations overwrite
rows 0 .. path_length (zeroshot_omtm/learner.py:75-79 reads the future rows), and each step calls the backward planner
(``zeroshot_mode`` "piid" or "id") instead of ``action_sample``.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Any, Callable, Dict, List, Optional, Sequence

import numpy as np


def new_trajectory(obs_dim: int, act_dim: int, max_path_length: int = 1000) -> Dict[str, Any]:
    """``current_trajectory`` of replay_buffer.py:192-205 / learner.py:663-675."""
    return {
        "observations": np.zeros((max_path_length, obs_dim), dtype=np.float32),
        "actions": np.zeros((max_path_length, act_dim), dtype=np.float32),
        "rewards": np.zeros((max_path_length, 1), dtype=np.float32),
        "values": np.zeros((max_path_length, 1), dtype=np.float32),
        "total_return": 0,
        "path_length": 0,
    }


#: rows of a zero-shot history: the waypoint windows read up to step 1000 (zeroshot_omtm/learner.py:77-79 clamps them there)
WAYPOINT_ROWS = 1000


def _is_zeroshot(learner) -> bool:
    return bool(getattr(learner, "_future_obs_windows", False))


def _history_rows(learner, max_path_length: int) -> int:
    """Rows of an episode's history arrays: ``max_path_length``, and for a zero-shot learner at least the 1000 rows its waypoint
    windows read, so that a window near the end of an episode still finds the rows the reference slices."""
    return max(int(max_path_length), WAYPOINT_ROWS) if _is_zeroshot(learner) else int(max_path_length)


def _split(n: int, groups: int) -> List[range]:
    groups = max(1, min(groups, n))
    cuts = [n * g // groups for g in range(groups + 1)]
    return [range(cuts[g], cuts[g + 1]) for g in range(groups)]


def run_episodes(learner, envs: Sequence[Any], *, rtg: Optional[Callable[[int], float]] = None, percentage: float = 1.0, plan: bool = True,
                 eval: bool = True, max_path_length: int = 1000, clip=(-1.0, 1.0), groups: int = 2,
                 on_step: Optional[Callable[[int, int, np.ndarray, float, bool], None]] = None,
                 waypoints: Optional[Callable[[int], np.ndarray]] = None, zeroshot_mode: Optional[str] = None) -> Dict[str, Any]:
    """One episode in each of ``envs`` (all reset now, stepped in lock-step).

    rtg(timestep) is the return-to-go handed to the planner at that step (``episode_rtg_ref[timestep]`` in evaluate_plan,
    learner.py:685); None -> the ``percentage`` rule of learner.py:368-385.  An environment that reports ``done`` leaves its
    group (the others keep their lock-step).  Returns per-environment ``returns`` / ``lengths`` and the trajectories.

    A zero-shot learner needs ``waypoints(i)``, the (L, obs) waypoint table of the episode in ``envs[i]``, and plans with
    ``zeroshot_mode`` ("piid" / "id"; default: the learner's ``zeroshot_mode``); ``plan`` does not apply to it.  A forward learner
    takes no waypoints.
    """
    trajs = _run(learner, lambda i: envs[i], len(envs), len(envs), rtg=rtg, plan=plan, eval=eval, max_path_length=max_path_length,
                 groups=groups, percentage=percentage, clip=clip, on_step=on_step, waypoints=waypoints, zeroshot_mode=zeroshot_mode)
    return {"returns": np.array([tr["total_return"] for tr in trajs], dtype=np.float64),
            "lengths": np.array([tr["path_length"] for tr in trajs], dtype=np.int64), "trajectories": trajs}


def evaluate_plan(learner, make_env: Callable[[], Any], num_episodes: int, episode_rtg_ref: np.ndarray, *, n_envs: Optional[int] = None,
                  groups: int = 2, max_path_length: int = 1000, refill: bool = False, device_histories: bool = False, plan: bool = True,
                  eval: bool = True, waypoints: Optional[Callable[[int], np.ndarray]] = None, zeroshot_mode: Optional[str] = None) -> Dict[str, Any]:
    """``Learner.evaluate_plan`` (learner.py:648-720) over ``num_episodes`` episodes on ``n_envs`` environment slots (default:
    the Learner's ``max_envs``): rtg = episode_rtg_ref[timestep of the episode], actions clipped to [-1, 1].

    refill=False: rounds of ``n_envs`` episodes that start together; a round lasts as long as its longest episode.
    refill=True: the episodes stream through the slots -- when an episode ends, the next one (``make_env()`` is called in
    episode order) starts in its slot at once, so no slot idles while episodes are queued.  Every episode runs exactly as it
    would alone (its own timestep, its own clamped horizon); only the batching changes.  ``device_histories=True`` keeps the
    histories in HBM (``DeviceEpisodes``) instead of re-slicing host arrays every step (refill only).  A zero-shot learner needs
    ``waypoints(episode)``, the (L, obs) waypoint table of each episode (episode order), and plans with ``zeroshot_mode``.

    Returns the means plus per-episode ``returns`` / ``lengths`` / ``trajectories`` in episode order."""
    n_envs = int(n_envs or getattr(learner, "max_envs", 1))
    rtg = lambda t: episode_rtg_ref[min(t, len(episode_rtg_ref) - 1)]  # noqa: E731
    if device_histories and not refill:
        raise ValueError("device_histories needs refill=True")
    _check_waypoints(learner, waypoints)
    if refill:
        trajs = _run(learner, lambda i: make_env(), num_episodes, n_envs, rtg=rtg, plan=plan, eval=eval, max_path_length=max_path_length,
                     groups=groups, device=device_histories, waypoints=waypoints, zeroshot_mode=zeroshot_mode)
    else:
        trajs = []
        while len(trajs) < num_episodes:
            k, base = min(n_envs, num_episodes - len(trajs)), len(trajs)
            wp = None if waypoints is None else (lambda i, b=base: waypoints(b + i))
            trajs += run_episodes(learner, [make_env() for _ in range(k)], rtg=rtg, plan=plan, eval=eval, max_path_length=max_path_length,
                                  groups=groups, waypoints=wp, zeroshot_mode=zeroshot_mode)["trajectories"]
    rets = [float(tr["total_return"]) for tr in trajs]
    lens = [int(tr["path_length"]) for tr in trajs]
    return {"return_mean": float(np.mean(rets)), "return_std": float(np.std(rets)), "length_mean": float(np.mean(lens)), "episodes": len(rets),
            "returns": rets, "lengths": lens, "trajectories": trajs}


def _check_waypoints(learner, waypoints) -> None:
    if _is_zeroshot(learner) and waypoints is None:
        raise ValueError("a zero-shot learner plans towards waypoints: pass waypoints(episode) -> (L, obs) array")
    if not _is_zeroshot(learner) and waypoints is not None:
        raise ValueError("waypoints are for zero-shot learners; this learner plans forward and takes none")


def _zeroshot_mode(learner, mode: Optional[str]) -> str:
    mode = mode if mode is not None else getattr(learner, "zeroshot_mode", "piid")
    if mode not in ("id", "piid"):
        raise ValueError(f"zero-shot mode {mode!r}: one of 'id', 'piid'")
    return mode


def _run(learner, env_of: Callable[[int], Any], num_episodes: int, n_slots: int, *, rtg: Optional[Callable[[int], float]], plan: bool,
         eval: bool, max_path_length: int, groups: int, percentage: float = 1.0, clip=(-1.0, 1.0), device: bool = False,
         on_step: Optional[Callable[[int, int, np.ndarray, float, bool], None]] = None, waypoints: Optional[Callable[[int], np.ndarray]] = None,
         zeroshot_mode: Optional[str] = None) -> List[Dict[str, Any]]:
    """The episode loop of every entry point: ``num_episodes`` episodes (``env_of(i)`` is the environment of episode i, asked for
    in episode order) through min(n_slots, num_episodes) slots split into G groups.  While group g's environments step on the
    host, the plans of the other groups run on the GPU.  A slot whose episode ends takes the next queued one before its group
    plans again; with as many slots as episodes none is refilled and every group stays in lock-step.  ``device`` keeps the
    histories in a ``DeviceEpisodes``.  ``on_step(episode, t, action, reward, done)`` follows every environment step.  Returns the
    trajectories in episode order.  ``waypoints`` / ``zeroshot_mode``: see ``run_episodes``."""
    _check_waypoints(learner, waypoints)
    zs = _is_zeroshot(learner)
    mode = _zeroshot_mode(learner, zeroshot_mode) if zs else None
    E = min(int(n_slots), int(num_episodes))
    if E < 1:
        raise ValueError("need at least one episode and one environment slot")
    act_dim = int(learner.mtm.data_shapes["actions"][1])
    hist_rows = _history_rows(learner, max_path_length)
    tables: List[Optional[np.ndarray]] = [None] * E  # waypoint table of each slot's episode
    done_trajs: List[Optional[Dict[str, Any]]] = [None] * num_episodes
    episode: List[Optional[int]] = [None] * E  # episode index running in each slot (None: idle)
    envs: List[Any] = [None] * E
    trajs: List[Optional[Dict[str, Any]]] = [None] * E
    queued = [0]  # next episode to start

    def begin(s: int) -> Optional[np.ndarray]:
        """Start the next queued episode in slot s; its first observation, or None when the queue is empty."""
        if queued[0] >= num_episodes:
            episode[s] = None
            return None
        episode[s], queued[0] = queued[0], queued[0] + 1
        envs[s] = env_of(episode[s])
        obs = np.asarray(envs[s].reset(), dtype=np.float32)
        trajs[s] = new_trajectory(obs.shape[-1], act_dim, hist_rows)
        if waypoints is not None:
            tables[s] = np.asarray(waypoints(episode[s]), dtype=np.float32).reshape(-1, obs.shape[-1])[:hist_rows]
            trajs[s]["observations"][:len(tables[s])] = tables[s]
        trajs[s]["observations"][0] = obs
        return obs

    first = [begin(s) for s in range(E)]
    ep = None
    if device:
        ep = DeviceEpisodes(learner, n_env=E, max_path_length=max_path_length)
        ep.start(np.stack(first), waypoints=tables if waypoints is not None else None)
    parts = [list(r) for r in _split(E, groups)]
    members: List[List[int]] = [[] for _ in parts]
    tickets: List[Any] = [None] * len(parts)

    def submit(g: int) -> None:
        members[g] = [s for s in parts[g] if episode[s] is not None]
        if not members[g]:
            tickets[g] = None
            return
        steps = [trajs[s]["path_length"] for s in members[g]]
        r = None  # a group in lock-step shares one return-to-go; otherwise one per member
        if rtg is not None:
            r = float(rtg(steps[0])) if len(set(steps)) == 1 else [float(rtg(t)) for t in steps]
        if ep is not None:
            tickets[g] = ep.plan_async(percentage=percentage, plan=plan, eval=eval, rtg=r, slots=members[g], mode=mode)
        elif zs:
            plan_zs = learner.action_piid_sample_async if mode == "piid" else learner.action_id_sample_async
            tickets[g] = plan_zs([trajs[s] for s in members[g]], percentage=percentage, eval=eval, rtg=r)
        else:
            tickets[g] = learner.action_sample_async([trajs[s] for s in members[g]], percentage=percentage, plan=plan, eval=eval, rtg=r)

    for g in range(len(parts)):
        submit(g)
    while any(t is not None for t in tickets):
        for g in range(len(parts)):
            if tickets[g] is None:
                continue
            actions = np.clip(tickets[g].result(), clip[0], clip[1])  # waits for THIS group's plan only
            going, ended = [], []
            for row, s in enumerate(members[g]):
                tr = trajs[s]
                t = tr["path_length"]
                new_obs, reward, done, _info = envs[s].step(actions[row])
                tr["actions"][t] = actions[row]
                tr["rewards"][t] = reward
                tr["total_return"] += float(reward)
                tr["path_length"] += 1
                if on_step is not None:
                    on_step(episode[s], t, actions[row], float(reward), bool(done))
                if done or t + 1 >= max_path_length:
                    done_trajs[episode[s]] = tr
                    ended.append(s)
                else:
                    tr["observations"][t + 1] = np.asarray(new_obs, dtype=np.float32)
                    going.append((row, s))
            if ep is not None and going:
                rows = [r_ for r_, _ in going]
                ep.step(actions[rows], np.array([trajs[s]["rewards"][trajs[s]["path_length"] - 1, 0] for _, s in going], np.float32),
                        np.stack([trajs[s]["observations"][trajs[s]["path_length"]] for _, s in going]), slots=[s for _, s in going])
            for s in ended:
                obs = begin(s)
                if ep is not None:
                    if obs is None:
                        ep.release([s])
                    else:
                        ep.reset([s], obs[None], waypoints=None if waypoints is None else [tables[s]])
            submit(g)  # queued behind the other groups' plans; runs while the next group's environments step
    return done_trajs


class DeviceEpisodes:
    """Device-resident histories of E episode slots (SURVEY.md section 8f rank 1; ``m3pc_ring_*`` in include/m3pc.h).

    The reference keeps each episode as zero-filled (1000, d) numpy arrays and re-slices a window out of them on the host at
    every step (learner.py:346-366).  Here the arrays live in HBM: a step uploads only the new observations and the actions /
    rewards just taken (obs + act + 1 floats per slot), and the planner's (E, T, .) windows are cut on the device.

    Every slot has its own clock ``t[slot]`` (its episode's ``path_length``; -1 = idle), so the slots need not be in lock-step:
    when an episode ends, ``reset`` starts the next one in its slot (or ``release`` leaves the slot idle) while the other slots
    carry on.  Per-slot arguments and results are in the order of the slot list they come with; without a list, that is every
    active slot in ascending order.

        ep = DeviceEpisodes(learner, n_env=E); ep.start(obs0)                     # obs0: (E, obs)
        a = ep.plan_async(rtg=3.0, plan=True, eval=True).result()                 # (n_active, act)
        ep.step(a, rewards, next_obs)                                             # then plan again
        ep.reset([2], obs)                                                        # slot 2 starts a new episode
        ep.release([5])                                                           # slot 5 stays idle

    With a zero-shot learner, ``start`` / ``reset`` take each new episode's waypoint table, uploaded once into the observation
    columns of its history (``m3pc_ring_write_obs``), and ``plan_async`` runs the backward planner on windows that carry the future
    waypoints; the history then holds max(max_path_length, 1000) rows, as the host histories of ``run_episodes`` do.
    """

    def __init__(self, learner, n_env: int, max_path_length: int = 1000):
        import ctypes as C

        import torch

        from . import _native as nat
        self.learner, self.E, self.max_path_length = learner, int(n_env), int(max_path_length)
        self.L = _history_rows(learner, max_path_length)  # ring rows
        if self.E < 1 or self.E > int(getattr(learner, "max_envs", 1)):
            raise ValueError(f"{n_env} environments but the Learner was built with max_envs={getattr(learner, 'max_envs', 1)}")
        learner._engine()
        self._nat, self._C, self._torch = nat, C, torch
        self.obs = int(learner.mtm.data_shapes["states"][1])
        self.act = int(learner.mtm.data_shapes["actions"][1])
        self.T = int(learner.cfg.traj_length)
        dev = learner.mtm.pos_embed.device
        w = self.obs + self.act + 1
        self.ring = torch.zeros(self.E, self.L, w, device=dev)
        self.t = np.full(self.E, -1, dtype=np.int64)  # path_length of each slot's current step; -1 = idle
        # staging: [clocks (E int32) | per-slot payload], one H2D copy per call
        n_stage = self.E * (w + 2)
        self._stage = [SimpleNamespace(host=torch.zeros(n_stage).pin_memory(), event=torch.cuda.Event(), used=False) for _ in range(2)]
        self._turn = 0
        self._dev_stage = torch.zeros(n_stage, device=dev)
        self._clock = self._dev_stage[:self.E].view(torch.int32)
        E, T = self.E, self.T
        self.win_states = torch.zeros(E, T, self.obs, device=dev)
        self.win_actions = torch.zeros(E, T, self.act, device=dev)
        self.win_rewards = torch.zeros(E, T, device=dev)
        self.win_returns = torch.zeros(E, T, device=dev)

    @property
    def active(self) -> np.ndarray:
        """Slots with a running episode, ascending."""
        return np.flatnonzero(self.t >= 0)

    def _slot(self):
        s = self._stage[self._turn]
        self._turn ^= 1
        if s.used:
            s.event.synchronize()
        return s

    def _upload(self, slot, n: int):
        self._dev_stage[:n].copy_(slot.host[:n], non_blocking=True)
        slot.event.record()
        slot.used = True

    def _stream(self):
        return self._torch.cuda.current_stream().cuda_stream

    def _slots(self, slots, need_active: bool) -> np.ndarray:
        s = self.active if slots is None else np.asarray(list(slots), dtype=np.int64).reshape(-1)
        if s.size and (s.min() < 0 or s.max() >= self.E or len(set(s.tolist())) != s.size):
            raise ValueError(f"slots {s.tolist()} must be distinct and in [0, {self.E})")
        if need_active and s.size and (self.t[s] < 0).any():
            raise RuntimeError(f"slots {s[self.t[s] < 0].tolist()} have no running episode (start() / reset() first)")
        return s.astype(np.int32)

    def _stage_clocks(self):
        slot = self._slot()
        h = slot.host.numpy()
        h[:self.E].view(np.int32)[:] = self.t
        return slot, h

    def start(self, obs0, waypoints=None) -> None:
        """Begin E episodes, one per slot: clears the histories and stores the first observations (E, obs) (and waypoint tables,
        see ``reset``)."""
        self.reset(range(self.E), obs0, waypoints)

    def reset(self, slots, obs, waypoints=None) -> None:
        """Start a new episode in each of ``slots``: zero its history (nothing of the previous episode may reach the windows of
        the next) and store its first observation (one row of ``obs`` per listed slot).  ``waypoints``: one (L_k, obs) waypoint
        table per listed slot, stored in the observation rows 0 .. L_k - 1 of its history (rows past the history are dropped)."""
        s = self._slots(slots, need_active=False)
        obs = np.asarray(obs, dtype=np.float32).reshape(len(s), -1)
        nat, C = self._nat, self._C
        nat.check(nat.lib().m3pc_ring_reset(self.ring.data_ptr(), self.E, self.L, self.obs, self.act, s.ctypes.data_as(C.c_void_p), len(s),
                                            self._stream()), "m3pc_ring_reset")
        if waypoints is not None:
            if len(waypoints) != len(s):
                raise ValueError(f"{len(waypoints)} waypoint tables for {len(s)} slots")
            tabs = [np.asarray(w, dtype=np.float32).reshape(-1, self.obs)[:self.L] for w in waypoints]
            n_rows = max(len(w) for w in tabs)
            rows = np.zeros((len(s), n_rows, self.obs), dtype=np.float32)  # shorter tables: zero rows, as the reset left them
            for k, w in enumerate(tabs):
                rows[k, :len(w)] = w
            d_rows = self._torch.from_numpy(rows).to(self.ring.device)
            nat.check(nat.lib().m3pc_ring_write_obs(self.ring.data_ptr(), self.E, self.L, self.obs, self.act, s.ctypes.data_as(C.c_void_p), len(s),
                                                    0, n_rows, d_rows.data_ptr(), self._stream()), "m3pc_ring_write_obs")
        self.t[s] = 0
        self._append(s, obs, None, None)

    def release(self, slots) -> None:
        """Leave ``slots`` idle: they are skipped by ``step`` and ``plan_async`` until ``reset``."""
        self.t[self._slots(slots, need_active=False)] = -1

    def step(self, actions, rewards, next_obs, slots=None) -> None:
        """Record the actions taken at the current step of ``slots`` (default: every active slot) and their rewards, and the
        observations of the next step; one row per listed slot."""
        s = self._slots(slots, need_active=True)
        if not s.size:
            raise RuntimeError("DeviceEpisodes.step() without a running episode")
        if (self.t[s] + 1 >= self.max_path_length).any():
            raise RuntimeError("episode longer than max_path_length")
        self.t[s] += 1
        self._append(s, np.asarray(next_obs, dtype=np.float32), np.asarray(actions, dtype=np.float32), np.asarray(rewards, dtype=np.float32))

    def _append(self, s: np.ndarray, obs, act, rew) -> None:
        n, o, a = len(s), self.obs, self.act
        if obs.shape != (n, o):
            raise ValueError(f"observations have shape {obs.shape}, expected {(n, o)}")
        slot, h = self._stage_clocks()
        base = self.E
        h[base:base + n * o] = obs.reshape(-1)
        m = base + n * o
        pa = pr = None
        if act is not None:
            h[m:m + n * a] = act.reshape(n * a)
            h[m + n * a:m + n * a + n] = rew.reshape(n)
            pa = self._dev_stage.data_ptr() + 4 * m
            pr = pa + 4 * n * a
            m += n * a + n
        self._upload(slot, m)
        nat, C = self._nat, self._C
        nat.check(nat.lib().m3pc_ring_append_slots(self.ring.data_ptr(), self.E, self.L, o, a, self._clock.data_ptr(), s.ctypes.data_as(C.c_void_p),
                                                   n, self._dev_stage.data_ptr() + 4 * base, pa, pr, self._stream()), "m3pc_ring_append_slots")

    def plan_async(self, percentage: float = 1.0, plan: bool = True, eval: bool = False, rtg=None, slots=None, mode: Optional[str] = None):
        """``Learner.action_sample_async`` on the device-resident histories of ``slots`` (default: every active slot): returns a
        ticket for their (n, act) actions, row k for slot k of the list.  Each slot plans at its own clock with its own clamped
        horizon (learner.py:342-345); ``rtg`` is a scalar or one value per listed slot.  A zero-shot learner runs its backward
        planner instead (``mode`` "piid" / "id", default: the learner's ``zeroshot_mode``; ``plan`` does not apply)."""
        L = self.learner
        if eval == True:  # noqa: E712
            assert rtg is not None
        s = self._slots(slots, need_active=True)
        n = len(s)
        if n == 0:
            raise RuntimeError("DeviceEpisodes.plan_async() without a running episode (start() / reset() first)")
        horizons = self.windows(s, percentage, rtg)
        T = self.T
        if _is_zeroshot(L):
            ev, sm = L._backward_device(_zeroshot_mode(L, mode), horizons.tolist(), self.win_states[:n], self.win_actions[:n], self.win_rewards[:n],
                                        self.win_returns[:n])
            return L._ticket(ev if eval else sm, n)
        guidance, lmbda = L._guidance(plan)
        lead = (n,) if n > 1 else ()
        ev, sm = L._plan_device(guidance, horizons.tolist(), lmbda, self.win_states[:n].view(*lead, T, self.obs),
                                self.win_actions[:n].view(*lead, T, self.act), self.win_rewards[:n].view(*lead, T), self.win_returns[:n].view(*lead, T))
        return L._ticket(ev if eval else sm, n)

    def windows(self, slots, percentage: float = 1.0, rtg=None) -> np.ndarray:
        """Cut the planner windows of ``slots`` on the device into ``win_states`` .. ``win_returns`` (row k for slot k of the list),
        each at its slot's clock with its clamped horizon; returns those horizons."""
        L = self.learner
        s = self._slots(slots, need_active=True)
        n = len(s)
        horizons = np.array([L._clamped_horizon({"path_length": int(self.t[k])}) for k in s], dtype=np.int32)
        slot, h = self._stage_clocks()
        h[self.E:self.E + n] = [L._rtg_token(percentage, L._rtg_of(rtg, k)) for k in range(n)]
        self._upload(slot, self.E + n)
        nat, C = self._nat, self._C
        nat.check(nat.lib().m3pc_ring_windows_slots(self.ring.data_ptr(), self.E, self.L, self.obs, self.act, self._clock.data_ptr(),
                                                    s.ctypes.data_as(C.c_void_p), horizons.ctypes.data_as(C.c_void_p), n, self.T,
                                                    1 if _is_zeroshot(L) else 0, self._dev_stage.data_ptr() + 4 * self.E,
                                                    self.win_states.data_ptr(), self.win_actions.data_ptr(), self.win_rewards.data_ptr(),
                                                    self.win_returns.data_ptr(), self._stream()), "m3pc_ring_windows_slots")
        return horizons


class LinearEnv:
    """A deterministic stand-in for the gym environments (none are installed): contracting linear dynamics with a bounded reward.
    Only for tests and the pipeline benchmark -- the reference's MuJoCo tasks are outside this path."""

    def __init__(self, obs_dim: int, act_dim: int, seed: int = 0, horizon: int = 1000, step_cost_s: float = 0.0):
        rs = np.random.RandomState(seed)
        a = rs.randn(obs_dim, obs_dim).astype(np.float32)
        self.A = (0.9 * a / max(1e-6, float(np.linalg.norm(a, 2)))).astype(np.float32)
        self.B = (0.3 * rs.randn(obs_dim, act_dim)).astype(np.float32)
        self.w = rs.randn(obs_dim).astype(np.float32) / np.sqrt(obs_dim)
        self.x0 = rs.randn(obs_dim).astype(np.float32)
        self.horizon, self.t, self.x = horizon, 0, self.x0.copy()
        self.step_cost_s = step_cost_s

    def reset(self):
        self.t, self.x = 0, self.x0.copy()
        return self.x.copy()

    def step(self, action):
        if self.step_cost_s > 0:  # emulate a physics step
            import time
            t_end = time.perf_counter() + self.step_cost_s
            while time.perf_counter() < t_end:
                pass
        a = np.asarray(action, dtype=np.float32).reshape(-1)  # the reference hands (1, act) exploration actions to env.step
        self.x = (self.A @ self.x + self.B @ a).astype(np.float32)
        self.t += 1
        reward = float(np.tanh(self.w @ self.x))
        return self.x.copy(), reward, self.t >= self.horizon, {}
