"""Backward M^3PC (zero-shot goal reaching) planners -- drop-in for research/zeroshot_omtm/learner.py:60-370.

  Learner.action_id_sample          zeroshot_omtm/learner.py:60-149   one pass, gid mask -> action at T-h
  Learner.action_piid_sample        zeroshot_omtm/learner.py:151-261  pi mask -> fill inferred states -> fid mask
  Learner.action_piid_list_sample   zeroshot_omtm/learner.py:263-370  same, stores ``self.action_list``

The reference plans one environment at a time (B = 1).  The ``*_batch`` variants plan E environments in one call (BASELINE.json
config 4); row e of their result equals the B=1 call on history e.  The environments need not be in lock-step: each is planned
with its own clamped horizon (``m3pc_backward_plan_env`` when the horizons differ).  The ``*_async`` variants return a
``PlanTicket`` instead of waiting for the actions (``m3pc_b200.rollout``).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch

from .learner import PlannerMixin, PlanTicket
from .mtm_model import omtm
from .tokenizers import TokenizerManager


class Learner(PlannerMixin):
    _future_obs_windows = True  # the states window holds future waypoints (zeroshot_omtm/learner.py:97-106, :188-197)
    #: backward planner the rollout loops use: "piid" (action_piid_sample) or "id" (action_id_sample)
    zeroshot_mode: str = "piid"

    def __init__(self, cfg, env, data_shapes, model_config, pretrain_model_path, obs_mean, obs_std,
                 tokenizer_manager: TokenizerManager, discrete_map: Dict[str, bool], max_envs: int = 1):
        self.cfg = cfg
        self.max_envs = int(max_envs)  # largest E the *_batch planners will be given
        self.env = env
        self.mtm: omtm = model_config.create(data_shapes, cfg.traj_length, discrete_map)
        if pretrain_model_path is not None:
            self.mtm.load_state_dict(torch.load(pretrain_model_path, map_location="cpu")["model"])
        self.mtm.to(cfg.device)
        self.tokenizer_manager = tokenizer_manager
        self.discrete_map = discrete_map
        self.action_list: List[torch.Tensor] = []

    #: eps (E, A) consumed by ``action_dist.sample()`` instead of the device Philox stream (parity tests)
    injected_eps: Optional[torch.Tensor] = None

    def _backward(self, mode: str, histories: Sequence[dict], percentage, rtg, n_draws: Optional[int] = None):
        if len(histories) < 1:
            raise ValueError("need at least one history")
        self._engine()
        horizons = [self._clamped_horizon(h) for h in histories]
        E, T = len(histories), self.cfg.traj_length
        wb = self._stage_windows(histories, horizons, percentage, rtg, future_obs=True)
        return self._backward_device(mode, horizons, wb.d_states.view(E, T, -1), wb.d_actions.view(E, T, -1), wb.d_rewards.view(E, T),
                                     wb.d_returns.view(E, T), n_draws)

    def _backward_device(self, mode: str, horizons: Sequence[int], ws, wa, wr, wt, n_draws: Optional[int] = None):
        """One backward plan on the (E, T, .) device windows, window e planned with horizon ``horizons[e]``."""
        h = max(horizons)
        ev, sm, dbg = self._engine().backward_plan(mode=mode, horizon=h, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt,
                                                   eps=self.injected_eps, debug=self.debug_plans, n_draws=n_draws, seed=self._next_seed(),
                                                   env_horizons=list(horizons) if min(horizons) != h else None)
        if self.debug_plans:
            self.last_plan_debug = dbg
        return ev, sm

    @torch.no_grad()
    def action_id_sample(self, sequence_history, percentage=1.0, horizon=4, plan=True, eval=False, rtg=None):
        if eval == True:  # noqa: E712
            assert rtg is not None
        ev, sm = self._backward("id", [sequence_history], percentage, rtg)
        return ev if eval else sm

    @torch.no_grad()
    def action_piid_sample(self, sequence_history, percentage=1.0, horizon=4, plan=True, eval=False, rtg=None):
        if eval == True:  # noqa: E712
            assert rtg is not None
        ev, sm = self._backward("piid", [sequence_history], percentage, rtg)
        return ev if eval else sm

    @torch.no_grad()
    def action_piid_list_sample(self, sequence_history, percentage=1.0, horizon=4, plan=True, eval=False, rtg=None):
        if eval == True:  # noqa: E712
            assert rtg is not None
        ev, _ = self._backward("piid", [sequence_history], percentage, rtg)
        self.action_list = [ev]

    # ---- E environments, each at its own step (extension; the reference is B = 1) ----------------------------
    @torch.no_grad()
    def action_id_sample_batch(self, histories: Sequence[dict], percentage=1.0, eval=False, rtg=None):
        ev, sm = self._backward("id", histories, percentage, rtg)
        return ev if eval else sm

    @torch.no_grad()
    def action_piid_draws_batch(self, histories: Sequence[dict], n_draws: int, percentage=1.0, rtg=None, mode: str = "piid"):
        """BASELINE.json config 4 (E environments x C candidate actions): the piid (or id) passes run once per environment and
        C actions are drawn from the resulting distribution -- what C calls of the reference's ``action_piid_sample`` on the same
        history draw (zeroshot_omtm/learner.py:248-259).  Returns (mean action (E, A), draws (E, C, A))."""
        return self._backward(mode, histories, percentage, rtg, n_draws=int(n_draws))

    @torch.no_grad()
    def action_piid_sample_batch(self, histories: Sequence[dict], percentage=1.0, eval=False, rtg=None):
        ev, sm = self._backward("piid", histories, percentage, rtg)
        return ev if eval else sm

    @torch.no_grad()
    def action_id_sample_async(self, histories: Sequence[dict], percentage=1.0, eval=False, rtg=None) -> PlanTicket:
        """``action_id_sample_batch`` without the host synchronisation: a ticket for the (E, A) actions, as
        ``PlannerMixin.action_sample_async``."""
        ev, sm = self._backward("id", histories, percentage, rtg)
        return self._ticket(ev if eval else sm, len(histories))

    @torch.no_grad()
    def action_piid_sample_async(self, histories: Sequence[dict], percentage=1.0, eval=False, rtg=None) -> PlanTicket:
        """``action_piid_sample_batch`` without the host synchronisation: a ticket for the (E, A) actions."""
        ev, sm = self._backward("piid", histories, percentage, rtg)
        return self._ticket(ev if eval else sm, len(histories))
