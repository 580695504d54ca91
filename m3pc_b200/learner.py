"""Forward M^3PC planners -- drop-in for the planning half of research/finetune_omtm/learner.py.

Same entry points, argument meaning and return shapes as the reference:

  Learner.action_sample(sequence_history, percentage, horizon, plan, eval, rtg)   learner.py:329-417
  Learner.rtg_guiding(trajectory, h, lmbda=0.6)                                   learner.py:271-327
  Learner.critic_lambda_guiding(trajectory, h, lmbda)                             learner.py:211-268
  Learner.noise_adding_lambda(trajectory, h, lmbda)                               learner.py:142-208
  Learner.mtm_sampling(trajectory, h)                                             learner.py:103-115

but one call is ONE ``m3pc_plan`` launch sequence on the device (pass 1 at B=1, candidate sampling, pass 2 at
B=action_samples, critic / return scoring, softmax selection) with no host round trip in between; the host builds the
(T, obs+act+2) window in pinned memory, copies it once, and reads back ``act_dim`` floats.

``PlannerMixin`` carries the planners; a maintainer can mix it into the reference's own ``Learner`` (INTEGRATION.md).
The training / evaluation halves of the reference class (``mtm_update``, ``critic_update``, ``evaluate*``) are outside
this path and are not provided.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from .critic import TwinQ
from .mtm_model import omtm
from .tokenizers import TokenizerManager

class PlannerMixin:
    """Needs: self.cfg (traj_length, device, action_samples, discount, temperature, horizon, plan_guidance, lmbda),
    self.mtm (m3pc_b200.omtm), self.tokenizer_manager, and for the critic planners self.iql.qf (m3pc_b200.TwinQ)."""

    # -- noise control ---------------------------------------------------------------------------------
    #: (eps, q) to consume instead of the on-device Philox stream: eps (N,h,A) [or (A,) for mtm_sampling], q (N,).
    injected_noise: Optional[Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]] = None
    #: filled by every plan when ``debug_plans`` is True (expect_return, candidates, indices, partials)
    debug_plans: bool = False
    last_plan_debug: Optional[dict] = None
    seed: int = 0
    #: True on the zero-shot Learner: the states window also carries the stored future waypoints
    #: (zeroshot_omtm/learner.py:97-106); read by rollout.DeviceEpisodes when it cuts windows on the device
    _future_obs_windows: bool = False
    #: global candidate id of this process's first candidate / total (candidate sharding across ranks)
    cand_offset: int = 0

    #: precision of the shadow engine when ``self.mtm`` is the REFERENCE's trainable omtm (hybrid drop-in, INTEGRATION.md):
    #: "bf16", "fp32" or "tf32x3" (fp32-grade on the tensor cores)
    planner_precision: str = "bf16"

    @staticmethod
    def _versions(module) -> int:
        """Sum of the parameters' in-place version counters: moves on every optimiser step / ``load_state_dict`` / ``.mul_()``."""
        return sum(p._version for p in module.parameters()) if module is not None else 0

    def _planner_model(self):
        """The engine-backed ``omtm`` the planners run on.  ``self.mtm`` itself when it is this package's module; otherwise
        (``self.mtm`` is the REFERENCE's trainable omtm, mtm_model.py:324 -- the Learner keeps training it with its own
        ``compute_mtm_loss`` / ``mtm_update``, learner.py:419-538) an inference-only shadow with the same config whose
        parameters are re-copied from ``self.mtm.state_dict()`` whenever a parameter's version counter has moved, i.e. after
        every optimiser step.  No ``mark_dirty`` call is needed in that mode."""
        m = self.mtm
        if isinstance(m, omtm):
            return m
        d = self.__dict__
        if d.get("_shadow_of") is not m:
            from .mtm_model import omtmConfig
            c = m.config
            cfg = omtmConfig(n_embd=c.n_embd, n_head=c.n_head, n_enc_layer=c.n_enc_layer, n_dec_layer=c.n_dec_layer, dropout=c.dropout,
                             norm=c.norm, latent_dim=getattr(c, "latent_dim", None), precision=self.planner_precision)
            shadow = cfg.create(dict(m.data_shapes), m.max_len, {k: False for k in m.data_shapes})
            d["_shadow"], d["_shadow_of"], d["_shadow_version"] = shadow.to(m.pos_embed.device), m, None
        ver = self._versions(m)
        if d["_shadow_version"] != ver:
            d["_shadow"].load_state_dict(m.state_dict())
            d["_shadow_version"] = ver
        return d["_shadow"]

    def _engine(self):
        model = self._planner_model()
        critic = getattr(getattr(self, "iql", None), "qf", None)
        if model is not self.mtm:  # hybrid mode: the reference's TwinQ is trained in place by iql.update (model.py:286-308)
            cver = self._versions(critic)
            if self.__dict__.get("_critic_version") != cver:
                self.__dict__["_critic_version"] = cver
                model.mark_dirty()
        if self.__dict__.get("_planner_bound") is not model:
            # forward planners batch max_envs windows x action_samples candidates; the backward planners batch max_envs rows
            max_envs = int(getattr(self, "max_envs", 1))
            max_batch = int(getattr(self.cfg, "action_samples", 1)) * (max_envs if getattr(self, "_envs_times_candidates", False) else 1)
            max_batch = max(max_batch, max_envs)
            model.bind_planner(self.tokenizer_manager, critic, max_batch=max_batch)
            self.__dict__["_planner_bound"] = model
            self.__dict__["_plan_counter"] = 0
            self.__dict__.pop("_rtg_tok", None)  # cached return-to-go tokens were normalised with the previous statistics
            rt = self.tokenizer_manager.tokenizers["returns"]
            self.__dict__["_rt_norm"] = (rt._data_mean.detach().double().cpu().numpy(), rt._data_std.detach().double().cpu().numpy(), bool(rt.normalize))
        return model.sync_engine()

    def _returns_tok(self, returns: np.ndarray) -> np.ndarray:
        """Tokenise the return-to-go exactly like the reference: float64 arithmetic, one rounding to fp32
        (learner.py:368-385 builds a float64 tensor; continuous.py:74-79 normalises then casts)."""
        mean, std, normalize = self.__dict__["_rt_norm"]
        r = np.asarray(returns, dtype=np.float64)
        if normalize:
            r = (r - mean) / std
        return r.astype(np.float32)

    def _next_seed(self) -> int:
        c = self.__dict__.get("_plan_counter", 0)
        self.__dict__["_plan_counter"] = c + 1
        return (int(self.seed) << 32) ^ c

    def _guidance(self, plan: bool) -> Tuple[str, float]:
        """learner.py:388-412: (guidance, lmbda) of a plan; ``plan=False`` samples the model (``mtm_sampling``)."""
        if not plan:
            return "mtm_sampling", 0.0
        assert self.cfg.plan_guidance in ("critic_lambda_guiding", "rtg_guiding", "noise_adding_lambda")
        return self.cfg.plan_guidance, (0.6 if self.cfg.plan_guidance == "rtg_guiding" else self.cfg.lmbda)  # learner.py:405-407 drops cfg.lmbda

    def _plan_device(self, guidance: str, horizons: Sequence[int], lmbda: float, ws, wa, wr, wt):
        """One ``m3pc_plan`` on len(horizons) windows, window e planned with horizon ``horizons[e]``."""
        eng = self._engine()
        h = max(horizons)
        eps, q = self.injected_noise if self.injected_noise is not None else (None, None)
        ev, sm, dbg = eng.plan(guidance=guidance, horizon=h, n_cand=int(self.cfg.action_samples), win_states=ws, win_actions=wa,
                               win_rewards=wr, win_returns_tok=wt, discount=float(self.cfg.discount), temperature=float(self.cfg.temperature),
                               lmbda=float(lmbda), eps=eps, expq=q, seed=self._next_seed(), cand_offset=int(self.cand_offset),
                               debug=self.debug_plans, n_env=len(horizons), env_horizons=horizons if min(horizons) != h else None)
        if self.debug_plans:
            self.last_plan_debug = {k: v.clone() for k, v in dbg.items()}
        return ev, sm

    def _ticket(self, actions: torch.Tensor, n_env: int) -> "PlanTicket":
        """A pooled ``PlanTicket`` that receives the (n_env, act) ``actions`` once the work queued before them is done."""
        free = self.__dict__.setdefault("_tickets", {}).setdefault(n_env, [])
        ticket = free.pop() if free else PlanTicket(n_env, actions.shape[-1], free)
        ticket._submit(actions)
        return ticket

    def _plan_from_trajectory(self, guidance: str, trajectory: Dict[str, torch.Tensor], h: int, lmbda: float):
        self._engine()
        T = self.cfg.traj_length
        dev = self.mtm.pos_embed.device
        ws = trajectory["states"].reshape(T, -1).to(dev, torch.float32)
        wa = trajectory["actions"].reshape(T, -1).to(dev, torch.float32)
        wr = trajectory["rewards"].reshape(T).to(dev, torch.float32)
        wt = torch.from_numpy(self._returns_tok(trajectory["returns"].detach().reshape(T).cpu().numpy())).to(dev)
        return self._plan_device(guidance, [h], lmbda, ws, wa, wr, wt)

    # -- the reference's planner entry points -------------------------------------------------------------
    @torch.no_grad()
    def mtm_sampling(self, trajectory: Dict[str, torch.Tensor], h):
        ev, sm = self._plan_from_trajectory("mtm_sampling", trajectory, h, 0.0)
        return sm.clone()[None, :], ev.clone()[None, :]

    @torch.no_grad()
    def noise_adding_lambda(self, trajectory: Dict[str, torch.Tensor], h: int, lmbda: float):
        ev, sm = self._plan_from_trajectory("noise_adding_lambda", trajectory, h, lmbda)
        return sm.clone()[None, :], ev.clone()

    @torch.no_grad()
    def critic_lambda_guiding(self, trajectory: Dict[str, torch.Tensor], h: int, lmbda: float):
        ev, sm = self._plan_from_trajectory("critic_lambda_guiding", trajectory, h, lmbda)
        return sm.clone()[None, :], ev.clone()

    @torch.no_grad()
    def rtg_guiding(self, trajectory: Dict[str, torch.Tensor], h: int, lmbda: float = 0.6):
        ev, sm = self._plan_from_trajectory("rtg_guiding", trajectory, h, lmbda)
        return sm.clone()[None, :], ev.clone()

    # -- validation loss (the forward half of SURVEY.md section 8(f) rank 4) ----------------------------------
    @torch.no_grad()
    def eval_mtm_loss(self, batch: Dict[str, torch.Tensor], data_shapes, discrete_map, entropy_reg, masks=None, eps=None):
        """``compute_mtm_loss`` (finetune_omtm/learner.py:419-503) for logging: the masked-prediction loss of a validation batch
        with the MTM forward on the B200 engine and NO autograd graph -- what ``finetune.py:346-369`` needs between training
        steps.  Training itself (``mtm_update``: backward + optimiser) stays on the reference's module (INTEGRATION.md 3a).

        Same arguments and the same 5-tuple ``(loss, losses, masked_losses, masked_c_losses, entropy)``.  The reference returns
        from inside its loop over modalities after the first continuous non-action key, so ``loss`` is the ``states`` MSE plus
        the action negative log-likelihood and entropy terms, and the three dicts hold ``states`` (+ ``entropy``, ``nll``) only;
        that behaviour is reproduced, not corrected.  ``masks`` (default: one draw of ``create_random_autoregressize_mask`` with
        ``cfg.mask_ratio`` / ``cfg.p_weights`` from numpy's global generator, like the reference) and ``eps`` (the normal draws of
        the single-sample entropy estimate, shape (1, B, T, 1, act)) can be injected for reproducible comparisons."""
        from . import masks as M
        model = self._planner_model()
        self._engine()
        dev = model.pos_embed.device
        targets = self.tokenizer_manager.encode({k: v.to(dev) for k, v in batch.items()})
        if masks is None:
            masks = M.create_random_autoregressize_mask(data_shapes, self.cfg.mask_ratio, self.cfg.traj_length, dev, self.cfg.p_weights)
        B = next(iter(targets.values())).shape[0]
        step = int(model.config.max_batch)
        parts = [model({k: v[b0:b0 + step] for k, v in targets.items()}, masks) for b0 in range(0, B, step)]
        preds = {k: torch.cat([p[k] for p in parts]) for k in ("states", "rewards", "returns")}
        from .mtm_model import SquashedNormal
        preds["actions"] = SquashedNormal(torch.cat([p["actions"].loc for p in parts]), torch.cat([p["actions"].std for p in parts]))

        key = next(k for k in targets if k != "actions")
        if discrete_map[key]:
            raise NotImplementedError("discrete modalities are not supported by the B200 engine")
        target, pred = targets[key].to(torch.float32), preds[key]
        mask = masks[key].to(dev)
        if mask.dim() == 1:
            mask = mask[:, None].repeat(1, target.shape[2])
        raw = (pred - target) ** 2                                    # (B, T, P, d)
        vis = mask[None, :, :, None].to(raw.dtype)
        losses = {key: raw.mean(dim=(2, 3)).mean()}
        masked_c_losses = {key: ((raw * vis).sum(dim=(1, 2, 3)) / mask.sum()).mean()}
        masked_losses = {key: ((raw * (1 - vis)).sum(dim=(1, 2, 3)) / (1 - mask).sum()).mean()}
        loss = torch.sum(torch.stack(list(losses.values())))
        hidden = ~masks["actions"].to(dev).squeeze().to(torch.bool)
        dist = preds["actions"]
        a = targets["actions"].to(torch.float32).clip(-1 + 1e-6, 1 - 1e-6)
        log_likelihood = dist.log_likelihood(a)[:, hidden, :].mean()
        entropy = dist.entropy(eps=eps)[:, hidden, :].mean()
        losses["entropy"] = entropy
        losses["nll"] = -log_likelihood
        loss = loss - (log_likelihood + entropy_reg * entropy)
        return loss, losses, masked_losses, masked_c_losses, entropy

    # -- window builder (host) ------------------------------------------------------------------------------
    def _window_buffers(self, obs_dim: int, act_dim: int, n_env: int = 1):
        """Two pinned host staging buffers (alternating, each guarded by a CUDA event so a buffer is never rewritten while
        its H2D copy is still queued) and one device buffer, laid out [states | actions | rewards | returns_tok]."""
        T = self.cfg.traj_length
        key = (obs_dim, act_dim, T, n_env)
        rings = self.__dict__.setdefault("_win", {})  # one ring per window geometry: groups of different sizes do not evict each other
        ring = rings.get(key)
        if ring is None:
            n = n_env * T * (obs_dim + act_dim + 2)
            dev = torch.zeros(n, dtype=torch.float32, device=self.mtm.pos_embed.device)
            o = [0, n_env * T * obs_dim, n_env * T * (obs_dim + act_dim), n_env * T * (obs_dim + act_dim + 1), n]
            shp = [(n_env, T, obs_dim), (n_env, T, act_dim), (n_env, T), (n_env, T)]
            if n_env == 1:
                shp = [s_[1:] for s_ in shp]
            slots = []
            for _ in range(2):
                host = torch.zeros(n, dtype=torch.float32).pin_memory()
                hn = host.numpy()
                slots.append(SimpleNamespace(host=host, event=torch.cuda.Event(), used=False,
                                             h_states=hn[o[0]:o[1]].reshape(shp[0]), h_actions=hn[o[1]:o[2]].reshape(shp[1]),
                                             h_rewards=hn[o[2]:o[3]].reshape(shp[2]), h_returns=hn[o[3]:o[4]].reshape(shp[3])))
            ring = SimpleNamespace(key=key, slots=slots, turn=0, dev=dev,
                                   d_states=dev[o[0]:o[1]].view(shp[0]), d_actions=dev[o[1]:o[2]].view(shp[1]),
                                   d_rewards=dev[o[2]:o[3]].view(shp[2]), d_returns=dev[o[3]:o[4]].view(shp[3]))
            rings[key] = ring
        slot = ring.slots[ring.turn]
        ring.turn ^= 1
        if slot.used:
            slot.event.synchronize()
        return ring, slot

    def _upload_window(self, ring, slot) -> None:
        ring.dev.copy_(slot.host, non_blocking=True)
        slot.event.record()
        slot.used = True

    def _fill_window(self, states, actions, rewards, returns, sequence_history, horizon: int, percentage: float, rtg,
                     future_obs: bool = False) -> None:
        """learner.py:346-385 (and zeroshot_omtm/learner.py:75-132 when ``future_obs``), written into pinned memory.
        ``states`` (T,obs), ``actions`` (T,act), ``rewards`` (T,), ``returns`` (T,) are numpy views of the staging buffer."""
        T = self.cfg.traj_length
        end_idx = sequence_history["path_length"]
        hl = T - horizon + 1
        lo, hi = end_idx - hl + 1, end_idx + 1
        obs = sequence_history["observations"]
        states[:hl] = obs[lo:hi]
        states[hl:] = 0
        actions[:hl] = sequence_history["actions"][lo:hi]
        actions[hl:] = 0
        rewards[:hl] = sequence_history["rewards"][lo:hi, 0] if getattr(sequence_history["rewards"], "ndim", 0) == 2 else \
            np.asarray(sequence_history["rewards"][lo:hi]).reshape(-1)
        rewards[hl:] = 0
        if future_obs:
            smart_T = T
            if end_idx + horizon > 1000:
                smart_T = smart_T - (end_idx + horizon - 1000)
            states[:smart_T] = obs[lo:lo + T]
        returns[:] = self._rtg_token(percentage, rtg)

    def _rtg_token(self, percentage: float, rtg) -> np.float32:
        """learner.py:368-385: the token of return-to-go ``rtg`` (None: the ``percentage`` point of the dataset's return range),
        one scalar for the whole window: (rtg * 1.0 - mean) / std in float64, rounded once to fp32."""
        if rtg is not None:
            return_to_go = float(rtg)
        else:
            stats = self.tokenizer_manager.tokenizers["returns"].stats
            return_to_go = float(np.asarray(stats.min + (stats.max - stats.min) * percentage).reshape(-1)[0])
        cache = self.__dict__.setdefault("_rtg_tok", {})
        tok = cache.get(return_to_go)
        if tok is None:
            if len(cache) > 4096:
                cache.clear()
            tok = cache[return_to_go] = self._returns_tok(return_to_go * np.ones(1)).reshape(-1)[0]
        return tok

    def _clamped_horizon(self, sequence_history) -> int:
        """learner.py:342-345: early in an episode the planning horizon grows so the window stays full."""
        horizon = self.cfg.horizon
        if sequence_history["path_length"] + horizon < self.cfg.traj_length:
            horizon = self.cfg.traj_length - sequence_history["path_length"]
        return horizon

    @torch.no_grad()
    def action_sample(self, sequence_history, percentage=1.0, horizon=4, plan=True, eval=False, rtg=None):
        action = self._stage_and_plan([sequence_history], percentage, plan, eval, rtg).clone()
        return action if plan and eval else action[None, :]

    @staticmethod
    def _rtg_of(rtg, e: int):
        """``rtg`` may be a scalar (shared) or one value per environment (list / tuple / ndarray)."""
        if isinstance(rtg, (list, tuple)):
            return rtg[e]
        if isinstance(rtg, np.ndarray) and rtg.ndim > 0:
            return rtg.reshape(-1)[e if rtg.size > 1 else 0]
        return rtg

    def _stage_windows(self, histories, horizons, percentage, rtg, future_obs: bool = False):
        """The E windows of ``histories`` (learner.py:346-385, window e with horizon ``horizons[e]``) in ONE pinned staging
        buffer and one H2D copy; returns the device side of the window buffers."""
        E = len(histories)
        h0 = histories[0]
        wb, slot = self._window_buffers(h0["observations"].shape[-1], h0["actions"].shape[-1], n_env=E)
        for e, hist in enumerate(histories):
            v = (slot.h_states, slot.h_actions, slot.h_rewards, slot.h_returns) if E == 1 else \
                (slot.h_states[e], slot.h_actions[e], slot.h_rewards[e], slot.h_returns[e])
            self._fill_window(*v, hist, horizons[e], percentage, self._rtg_of(rtg, e), future_obs=future_obs)
        self._upload_window(wb, slot)
        return wb

    def _stage_and_plan(self, histories, percentage, plan: bool, eval: bool, rtg):
        """Shared body of ``action_sample`` / ``action_sample_batch`` / ``action_sample_async``: the E windows, each with its
        environment's own clamped horizon, and one ``m3pc_plan`` launch sequence.  Returns the engine-owned (E, A) device tensor
        of the eval actions if ``eval`` else of the sampled actions."""
        if eval == True:  # noqa: E712  (mirrors learner.py:339-340)
            assert rtg is not None
        E = len(histories)
        if E < 1:
            raise ValueError("need at least one history")
        if E > int(getattr(self, "max_envs", 1)):
            raise ValueError(f"{E} environments but the Learner was built with max_envs={getattr(self, 'max_envs', 1)}")
        self._engine()
        horizons = [self._clamped_horizon(hist) for hist in histories]
        wb = self._stage_windows(histories, horizons, percentage, rtg)
        guidance, lmbda = self._guidance(plan)
        ev, sm = self._plan_device(guidance, horizons, lmbda, wb.d_states, wb.d_actions, wb.d_rewards, wb.d_returns)
        return ev if eval else sm

    @torch.no_grad()
    def action_sample_batch(self, histories, percentage=1.0, horizon=4, plan=True, eval=False, rtg=None):
        """``action_sample`` for E lock-step environments in one ``m3pc_plan`` launch sequence (SURVEY.md section 8f rank 1;
        the reference plans one environment per call, learner.py:329-417).  ``histories`` is a sequence of E history dicts, each
        at any ``path_length`` (each window gets its own clamped horizon); ``rtg`` a scalar or one value per environment (list,
        tuple or ndarray).  Returns
        (E, act): row e is what ``action_sample(histories[e], ...)`` returns (``eval_action`` if ``eval`` else
        ``sample_action``).  The E windows are built in one pinned staging buffer and travel in one H2D copy; E * act floats
        come back."""
        return self._stage_and_plan(histories, percentage, plan, eval, rtg).clone().reshape(len(histories), -1)

    @torch.no_grad()
    def action_sample_async(self, histories, percentage=1.0, plan=True, eval=False, rtg=None) -> "PlanTicket":
        """``action_sample_batch`` without the host synchronisation (SURVEY.md section 8f rank 3): the window upload, the plan and
        the device-to-host copy of the E actions are enqueued on the current stream and a ticket is returned at once;
        ``ticket.result()`` waits for that copy only.  The reference's callers block in ``action.cpu()`` every step
        (replay_buffer.py:211-214, learner.py:681-689); with a ticket the caller can step other environments meanwhile
        (``m3pc_b200.rollout``)."""
        return self._ticket(self._stage_and_plan(histories, percentage, plan, eval, rtg), len(histories))


class PlanTicket:
    """Pinned landing buffer + CUDA event of one in-flight ``action_sample_async``; recycled through the Learner's pool."""

    def __init__(self, n_env: int, act_dim: int, pool: list):
        self._host = torch.empty(n_env, act_dim, dtype=torch.float32).pin_memory()
        self._event = torch.cuda.Event()
        self._pool = pool
        self._pending = False

    def _submit(self, actions: torch.Tensor) -> None:
        self._host.copy_(actions.reshape(self._host.shape), non_blocking=True)
        self._event.record()
        self._pending = True

    def done(self) -> bool:
        return self._event.query()

    def result(self) -> np.ndarray:
        """(E, act) float32; blocks until the device-to-host copy of THIS plan has landed (not a device-wide sync)."""
        if not self._pending:
            raise RuntimeError("PlanTicket.result() called twice")
        self._event.synchronize()
        out = self._host.numpy().copy()
        self._pending = False
        self._pool.append(self)
        return out


class Learner(PlannerMixin):
    """Constructor-compatible with finetune_omtm/learner.py:17-101 (the optimiser / IQL-trainer halves are not built)."""

    _envs_times_candidates = True  # engine capacity = max_envs * cfg.action_samples rows

    def __init__(self, cfg, env, data_shapes, model_config, pretrain_model_path, obs_mean, obs_std,
                 tokenizer_manager: TokenizerManager, discrete_map: Dict[str, bool], max_envs: int = 1):
        self.cfg = cfg
        self.env = env
        self.max_envs = int(max_envs)  # largest E ``action_sample_batch`` will be given (1 = the reference's behaviour)
        self.mtm: omtm = model_config.create(data_shapes, cfg.traj_length, discrete_map)
        if pretrain_model_path is not None:
            self.mtm.load_state_dict(torch.load(pretrain_model_path, map_location="cpu")["model"])
        self.mtm.to(cfg.device)
        self.tokenizer_manager = tokenizer_manager
        self.obs_mean = obs_mean
        self.obs_std = obs_std
        self.discrete_map = discrete_map
        if env is not None:
            state_dim, action_dim = env.observation_space.shape[0], env.action_space.shape[0]
        else:
            state_dim, action_dim = data_shapes["states"][1], data_shapes["actions"][1]
        om = torch.as_tensor(obs_mean, dtype=torch.float32) if obs_mean is not None else torch.zeros(state_dim)
        os_ = torch.as_tensor(obs_std, dtype=torch.float32) if obs_std is not None else torch.ones(state_dim)
        q_network = TwinQ(state_dim, action_dim, om.to(cfg.device), os_.to(cfg.device)).to(cfg.device)
        # the planners reach the critic as self.iql.qf (learner.py:250-252)
        self.iql = SimpleNamespace(qf=q_network)
