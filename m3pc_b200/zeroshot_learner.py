"""Backward M^3PC (zero-shot goal reaching) planners -- drop-in for research/zeroshot_omtm/learner.py:60-370.

  Learner.action_id_sample          zeroshot_omtm/learner.py:60-149   one pass, gid mask -> action at T-h
  Learner.action_piid_sample        zeroshot_omtm/learner.py:151-261  pi mask -> fill inferred states -> fid mask
  Learner.action_piid_list_sample   zeroshot_omtm/learner.py:263-370  same, stores ``self.action_list``

The reference plans one environment at a time (B = 1).  The ``*_batch`` variants plan E lock-step environments in one
``m3pc_backward_plan`` call (BASELINE.json config 4); row e of their result equals the B=1 call on history e.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch

from .learner import PlannerMixin
from .mtm_model import omtm
from .tokenizers import TokenizerManager


class Learner(PlannerMixin):
    _future_obs_windows = True  # the states window holds future waypoints (zeroshot_omtm/learner.py:97-106, :188-197)

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
        eng = self._engine()
        horizons = {self._clamped_horizon(h) for h in histories}
        if len(horizons) != 1:
            raise ValueError("lock-step environments must share the planning horizon (same path_length regime)")
        horizon = horizons.pop()
        E = len(histories)
        wb = self._stage_windows(histories, [horizon] * E, percentage, rtg, future_obs=True)
        T = self.cfg.traj_length
        ev, sm, dbg = eng.backward_plan(mode=mode, horizon=horizon, win_states=wb.d_states.view(E, T, -1), win_actions=wb.d_actions.view(E, T, -1),
                                        win_rewards=wb.d_rewards.view(E, T), win_returns_tok=wb.d_returns.view(E, T), eps=self.injected_eps,
                                        debug=self.debug_plans, n_draws=n_draws, seed=self._next_seed())
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

    # ---- E lock-step environments (extension; the reference is B = 1) ---------------------------------------
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
