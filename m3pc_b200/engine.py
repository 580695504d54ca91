"""Thin Python owner of one ``m3pc_handle_t`` (include/m3pc.h): parameter upload, forward, plan.

PyTorch is used here only for device memory and streams; every FLOP of the path runs in ``libm3pc.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Mapping, Optional, Sequence

import numpy as np
import torch

from . import _native as nat

MODALITIES = ("states", "actions", "rewards", "returns")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dev_f32(t: torch.Tensor, what: str) -> torch.Tensor:
    if not t.is_cuda:
        raise NotImplementedError(f"{what} must be a CUDA tensor: m3pc_b200 has no CPU path by design")
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.to(torch.float32).contiguous()
    return t


#: ``precision`` names -> M3PC_PREC_* (include/m3pc.h): "bf16" tensor cores at bf16 operands; "fp32" IEEE fp32 FFMA on CUDA cores, the
#: reference's arithmetic; "tf32x3" fp32 operands on the tensor cores with the 3xTF32 split, fp32-grade accuracy
PRECISIONS = {"bf16": nat.PREC_BF16, "fp32": nat.PREC_FP32, "tf32x3": nat.PREC_TF32X3}

class PlanEngine:
    """One engine per (process, device).  Mirrors ``m3pc_create`` .. ``m3pc_destroy``."""

    #: ``m3pc_set_option`` values applied to every engine right after ``m3pc_create`` (parity tests switch between the
    #: result-equivalent launch sequences with it; empty in production)
    default_options: Dict[str, int] = {}

    def __init__(self, *, n_embd: int, n_head: int, n_enc_layer: int, n_dec_layer: int, traj_length: int, obs_dim: int,
                 act_dim: int, precision: str = "bf16", max_batch: int = 1024, chunk: int = 0, critic_hidden: int = 0,
                 device: Optional[torch.device] = None):
        if precision not in PRECISIONS:
            raise ValueError(f"unknown precision {precision!r}: one of {sorted(PRECISIONS)}")
        if not torch.cuda.is_available():
            raise RuntimeError("m3pc_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = nat.lib()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.T, self.D, self.obs, self.act = traj_length, n_embd, obs_dim, act_dim
        self.dims = {"states": obs_dim, "actions": act_dim, "rewards": 1, "returns": 1}
        self.precision = precision
        self.max_batch = int(max_batch)
        self.critic_hidden = int(critic_hidden)
        cfg = nat.Config(n_embd=n_embd, n_head=n_head, n_enc_layer=n_enc_layer, n_dec_layer=n_dec_layer,
                         traj_length=traj_length, obs_dim=obs_dim, act_dim=act_dim,
                         precision=PRECISIONS[precision],
                         max_batch=self.max_batch, chunk=int(chunk), critic_hidden=self.critic_hidden)
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            nat.check(self.lib.m3pc_create(C.byref(self._h), C.byref(cfg)), "m3pc_create")
        for name, value in type(self).default_options.items():
            self.set_option(name, value)
        self.finalized = False
        self.has_critic = False
        # persistent small outputs
        self._eval = torch.empty(act_dim, device=self.device)
        self._sample = torch.empty(act_dim, device=self.device)
        self._partials = torch.zeros(nat.PARTIAL_FLOATS, device=self.device)
        self._indices = torch.zeros(2, dtype=torch.int32, device=self.device)
        self._env_out = {}  # n_env -> (eval (E,A), sample (E,A), indices (E,2))

    # ------------------------------------------------------------------ parameters
    def set_param(self, name: str, value) -> None:
        a = np.ascontiguousarray(value.detach().cpu().numpy() if isinstance(value, torch.Tensor) else np.asarray(value), dtype=np.float32)
        nat.check(self.lib.m3pc_set_param(self._h, name.encode(), a.ctypes.data_as(C.c_void_p), a.size), f"m3pc_set_param({name})")
        self.finalized = False

    def load_state_dict(self, sd: Mapping[str, object]) -> None:
        """Every key of the reference's ``omtm.state_dict()`` (learner.py:33-35)."""
        for k, v in sd.items():
            self.set_param(k, v)

    def load_tokenizer_stats(self, stats: Mapping[str, Mapping[str, object]]) -> None:
        """mean/std of states, rewards, returns (continuous.py:32-62); actions are not normalised."""
        for k in ("states", "rewards", "returns"):
            self.set_param(f"tokenizer.{k}.mean", stats[k]["mean"])
            self.set_param(f"tokenizer.{k}.std", stats[k]["std"])

    def load_critic(self, qsd: Mapping[str, object], obs_mean, obs_std) -> None:
        """TwinQ parameters (finetune_omtm/model.py:146-160) + its observation normaliser."""
        if self.critic_hidden <= 0:
            raise ValueError("engine was created with critic_hidden=0")
        for k, v in qsd.items():
            self.set_param("critic." + k, v)
        self.set_param("critic.obs_mean", obs_mean)
        self.set_param("critic.obs_std", obs_std)
        self.has_critic = True

    def set_option(self, name: str, value: int) -> None:
        """``m3pc_set_option``: pick between result-equivalent launch sequences (see include/m3pc.h for the names)."""
        nat.check(self.lib.m3pc_set_option(self._h, name.encode(), int(value)), f"m3pc_set_option({name})")

    def finalize(self) -> None:
        with torch.cuda.device(self.device):
            nat.check(self.lib.m3pc_finalize_params(self._h), "m3pc_finalize_params")
        self.finalized = True

    # ------------------------------------------------------------------ omtm.forward
    def forward(self, tokens: Mapping[str, torch.Tensor], masks: Mapping[str, object], want: Sequence[str] = MODALITIES
                ) -> Dict[str, torch.Tensor]:
        """tokens[k]: (B,T,d) fp32 CUDA; masks[k]: (T,) of {0,1}.  Returns raw head outputs (B,T,d), plus act_mu/act_std."""
        if not self.finalized:
            self.finalize()
        T = self.T
        ins = {}
        B = None
        for k in MODALITIES:
            t = _dev_f32(tokens[k], f"tokens[{k}]")
            if t.dim() != 3 or t.shape[1] != T or t.shape[2] != self.dims[k]:
                raise ValueError(f"tokens[{k}] has shape {tuple(t.shape)}, expected (B,{T},{self.dims[k]})")
            B = t.shape[0] if B is None else B
            if t.shape[0] != B:
                raise ValueError("all modalities must share the batch size")
            ins[k] = t
        m = np.zeros(4 * T, dtype=np.uint8)
        for i, k in enumerate(MODALITIES):
            mk = masks[k]
            mk = mk.detach().cpu().numpy() if isinstance(mk, torch.Tensor) else np.asarray(mk)
            if mk.shape != (T,):
                raise ValueError(f"masks[{k}] must have shape ({T},)")
            if not np.all((mk == 0) | (mk == 1)):
                raise ValueError("mask entries must be 0 or 1")
            m[i * T:(i + 1) * T] = (mk == 1)
        out: Dict[str, torch.Tensor] = {}
        for k in ("states", "rewards", "returns"):
            if k in want:
                out[k] = torch.empty(B, T, self.dims[k], device=self.device)
        if "actions" in want:
            out["act_mu"] = torch.empty(B, T, self.act, device=self.device)
            out["act_std"] = torch.empty(B, T, self.act, device=self.device)
        with torch.cuda.device(self.device):
            nat.check(self.lib.m3pc_forward(
                self._h, B, _ptr(ins["states"]), _ptr(ins["actions"]), _ptr(ins["rewards"]), _ptr(ins["returns"]),
                m.ctypes.data_as(C.c_void_p), _ptr(out.get("states")), _ptr(out.get("act_mu")), _ptr(out.get("act_std")),
                _ptr(out.get("rewards")), _ptr(out.get("returns")), _stream()), "m3pc_forward")
        return out

    # ------------------------------------------------------------------ planners
    def plan(self, *, guidance: str, horizon: int, n_cand: int, win_states: torch.Tensor, win_actions: torch.Tensor,
             win_rewards: torch.Tensor, win_returns_tok: torch.Tensor, discount: float, temperature: float, lmbda: float,
             eps: Optional[torch.Tensor] = None, expq: Optional[torch.Tensor] = None, seed: int = 0, cand_offset: int = 0,
             debug: bool = False, want_partials: bool = False, n_env: int = 1, exchange: bool = False,
             env_horizons: Optional[Sequence[int]] = None):
        """One M^3PC plan on one window (learner.py:103-327).  All tensors are CUDA fp32, contiguous.
        Returns (eval_action, sample_action, dbg) -- the action tensors are engine-owned and overwritten by the next call.

        ``n_env = E > 1`` plans E lock-step environments in the same launch sequence: windows carry a leading E axis,
        ``eps`` is (E*n_cand, h, A), ``expq`` (E*n_cand,), and the returned actions are (E, A); row e equals the
        single-window call on window e.

        ``exchange=True`` (after ``exchange_connect``): this call plans ONE SHARD (``n_cand`` candidates starting at global id
        ``cand_offset``); the selection kernel exchanges the shard records with every rank over peer memory and merges them, so
        the returned actions (and ``dbg["indices"]``) are the GLOBAL result on every rank.

        ``env_horizons``: one planning horizon per environment (environments at different points of their episodes,
        learner.py:342-345); ``horizon`` must be the largest.  ``eps`` / ``dbg["candidates"]`` keep the (E*n_cand, horizon, A)
        layout and environment e uses the first ``env_horizons[e]`` steps of its rows.  Row e of the result is what the uniform
        call on the environments of e's horizon returns for e; with all entries equal the call is exactly the one without."""
        if not self.finalized:
            self.finalize()
        E = int(n_env)
        if exchange and E > 1:
            raise ValueError("exchange (candidate sharding) plans one environment per call")
        if E < 1:
            raise ValueError("n_env must be >= 1")
        if E > 1 and (want_partials or cand_offset):
            raise ValueError("n_env > 1 cannot be combined with candidate sharding")
        hz = None
        if env_horizons is not None:
            hz = np.ascontiguousarray(np.asarray(env_horizons, dtype=np.int32).reshape(-1))
            if hz.size != E:
                raise ValueError(f"env_horizons has {hz.size} entries, expected n_env={E}")
        if E > 1:
            for t, d in ((win_states, self.obs), (win_actions, self.act), (win_rewards, 1), (win_returns_tok, 1)):
                if t.numel() != E * self.T * d:
                    raise ValueError(f"window tensor of {t.numel()} elements, expected (E={E}, T={self.T}, {d})")
        ev_out, sm_out = self._eval, self._sample
        if E > 1:
            if E not in self._env_out:  # persistent, so the plan's CUDA graph (keyed on buffer addresses) is reused
                self._env_out[E] = (torch.empty(E, self.act, device=self.device), torch.empty(E, self.act, device=self.device),
                                    torch.zeros(E, 2, dtype=torch.int32, device=self.device))
            ev_out, sm_out, idx_out = self._env_out[E]
        else:
            idx_out = self._indices
        a = nat.PlanArgs()
        a.n_env = E
        a.guidance = nat.GUIDANCE[guidance]
        a.horizon, a.n_cand, a.cand_offset = int(horizon), int(n_cand), int(cand_offset)
        a.discount, a.temperature, a.lmbda = float(discount), float(temperature), float(lmbda)
        keep = [_dev_f32(win_states, "win_states"), _dev_f32(win_actions, "win_actions"), _dev_f32(win_rewards, "win_rewards"),
                _dev_f32(win_returns_tok, "win_returns_tok")]
        a.win_states, a.win_actions, a.win_rewards, a.win_returns_tok = (t.data_ptr() for t in keep)
        if eps is not None:
            eps = _dev_f32(eps, "eps")
            a.eps = eps.data_ptr()
        if expq is not None:
            expq = _dev_f32(expq, "expq")
            a.expq = expq.data_ptr()
        a.seed = int(seed) & (2 ** 64 - 1)
        a.out_eval_action, a.out_sample_action = ev_out.data_ptr(), sm_out.data_ptr()
        a.exchange = 1 if exchange else 0
        if hz is not None:
            a.env_horizons = hz.ctypes.data
        dbg = {}
        if (want_partials or debug) and E == 1 and hz is None:
            a.out_partials = self._partials.data_ptr()
            dbg["partials"] = self._partials
        if debug and guidance != "mtm_sampling":
            dbg["expect_return"] = torch.empty(E * n_cand, device=self.device)
            dbg["candidates"] = torch.empty(E * n_cand, horizon, self.act, device=self.device)
            dbg["indices"] = idx_out
            a.dbg_expect_return, a.dbg_candidates = dbg["expect_return"].data_ptr(), dbg["candidates"].data_ptr()
            a.dbg_indices = idx_out.data_ptr()
        with torch.cuda.device(self.device):
            nat.check(self.lib.m3pc_plan(self._h, C.byref(a), _stream()), "m3pc_plan")
        return ev_out, sm_out, dbg

    def merge_partials(self, gathered: torch.Tensor, temperature: float):
        """Combine per-shard records (n_shards, PARTIAL_FLOATS) -> (eval_action, sample_action, indices)."""
        g = _dev_f32(gathered, "partials")
        n = g.numel() // nat.PARTIAL_FLOATS
        with torch.cuda.device(self.device):
            nat.check(self.lib.m3pc_merge_partials(self._h, g.data_ptr(), n, float(temperature), self._eval.data_ptr(),
                                                   self._sample.data_ptr(), self._indices.data_ptr(), _stream()), "m3pc_merge_partials")
        return self._eval, self._sample, self._indices

    # ------------------------------------------------------------------ peer exchange (candidate sharding over GPUs)
    def exchange_local(self):
        """(CUDA IPC handle bytes, device pointer) of this engine's exchange buffer (``m3pc_exchange_local``)."""
        buf = (C.c_uint8 * nat.IPC_HANDLE_BYTES)()
        ptr = C.c_void_p()
        with torch.cuda.device(self.device):
            nat.check(self.lib.m3pc_exchange_local(self._h, buf, C.byref(ptr)), "m3pc_exchange_local")
        return bytes(buf), int(ptr.value)

    def exchange_connect(self, rank: int, world: int, ipc_handles: Optional[Sequence[bytes]] = None,
                         device_ptrs: Optional[Sequence[int]] = None) -> None:
        """Wire the group (``m3pc_exchange_connect``): ``ipc_handles`` -- one per rank, in rank order, from peers in OTHER
        processes -- or ``device_ptrs`` -- exchange-buffer pointers of engines in THIS process."""
        with torch.cuda.device(self.device):
            if ipc_handles is not None:
                blob = b"".join(ipc_handles)
                if len(blob) != world * nat.IPC_HANDLE_BYTES:
                    raise ValueError("need one IPC handle per rank")
                arr = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
                nat.check(self.lib.m3pc_exchange_connect(self._h, int(rank), int(world), arr, None), "m3pc_exchange_connect")
            else:
                ptrs = (C.c_void_p * world)(*[int(p) for p in device_ptrs])
                nat.check(self.lib.m3pc_exchange_connect(self._h, int(rank), int(world), None, ptrs), "m3pc_exchange_connect")

    def exchange_status(self):
        """(plans exchanged so far, epoch of a wait that timed out or 0)."""
        ep, bad = C.c_uint64(), C.c_uint64()
        with torch.cuda.device(self.device):
            nat.check(self.lib.m3pc_exchange_status(self._h, C.byref(ep), C.byref(bad)), "m3pc_exchange_status")
        return int(ep.value), int(bad.value)

    def backward_plan(self, *, mode: str, horizon: int, win_states: torch.Tensor, win_actions: torch.Tensor, win_rewards: torch.Tensor,
                      win_returns_tok: torch.Tensor, eps: Optional[torch.Tensor] = None, debug: bool = False, n_draws: Optional[int] = None,
                      seed: int = 0, env_horizons: Optional[Sequence[int]] = None):
        """Zero-shot backward planners on E environments (zeroshot_omtm/learner.py:60-261). Windows have a leading E axis.
        ``n_draws = C``: C action draws per environment from one set of forward passes -> sample actions (E, C, A); eps (E, C, A).

        ``env_horizons``: one planning horizon per environment (environments at different points of their episodes); ``horizon``
        must be the largest.  When the entries differ the call is ``m3pc_backward_plan_env``: row e is what the uniform call on the
        environments of e's horizon returns for e (no ``states_filled`` debug output)."""
        if not self.finalized:
            self.finalize()
        ws = _dev_f32(win_states, "win_states")
        E = ws.shape[0]
        wa, wr, wt = _dev_f32(win_actions, "win_actions"), _dev_f32(win_rewards, "win_rewards"), _dev_f32(win_returns_tok, "win_returns_tok")
        if env_horizons is not None:
            hz = np.ascontiguousarray(np.asarray(env_horizons, dtype=np.int32).reshape(-1))
            if hz.size != E:
                raise ValueError(f"env_horizons has {hz.size} entries, expected n_env={E}")
            if int(hz.max()) != int(horizon):
                raise ValueError("with env_horizons, horizon must equal its largest entry")
            if int(hz.min()) != int(hz.max()):
                Cn = 1 if n_draws is None else int(n_draws)
                ev = torch.empty(E, self.act, device=self.device)
                sm = torch.empty((E, self.act) if n_draws is None else (E, Cn, self.act), device=self.device)
                if eps is not None:
                    eps = _dev_f32(eps, "eps")
                    if eps.numel() != E * Cn * self.act:
                        raise ValueError(f"eps has {eps.numel()} elements, expected (E={E}, C={Cn}, A={self.act})")
                with torch.cuda.device(self.device):
                    nat.check(self.lib.m3pc_backward_plan_env(self._h, {"id": 0, "piid": 1}[mode], E, hz.ctypes.data, Cn, ws.data_ptr(), wa.data_ptr(),
                                                              wr.data_ptr(), wt.data_ptr(), _ptr(eps), int(seed) & (2 ** 64 - 1), ev.data_ptr(),
                                                              sm.data_ptr(), _stream()), "m3pc_backward_plan_env")
                return ev, sm, {}
        if n_draws is not None:
            Cn = int(n_draws)
            ev = torch.empty(E, self.act, device=self.device)
            sm = torch.empty(E, Cn, self.act, device=self.device)
            if eps is not None:
                eps = _dev_f32(eps, "eps")
                if eps.numel() != E * Cn * self.act:
                    raise ValueError(f"eps has {eps.numel()} elements, expected (E={E}, C={Cn}, A={self.act})")
            with torch.cuda.device(self.device):
                nat.check(self.lib.m3pc_backward_plan_draws(self._h, {"id": 0, "piid": 1}[mode], E, int(horizon), Cn, ws.data_ptr(), wa.data_ptr(),
                                                            wr.data_ptr(), wt.data_ptr(), _ptr(eps), int(seed) & (2 ** 64 - 1), ev.data_ptr(),
                                                            sm.data_ptr(), _stream()), "m3pc_backward_plan_draws")
            return ev, sm, {}
        ev = torch.empty(E, self.act, device=self.device)
        sm = torch.empty(E, self.act, device=self.device)
        filled = torch.empty(E, self.T, self.obs, device=self.device) if debug else None
        if eps is not None:
            eps = _dev_f32(eps, "eps")
        with torch.cuda.device(self.device):
            nat.check(self.lib.m3pc_backward_plan(self._h, {"id": 0, "piid": 1}[mode], E, int(horizon), ws.data_ptr(), wa.data_ptr(),
                                                  wr.data_ptr(), wt.data_ptr(), _ptr(eps), ev.data_ptr(), sm.data_ptr(), _ptr(filled),
                                                  _stream()), "m3pc_backward_plan")
        return ev, sm, ({"states_filled": filled} if debug else {})

    # ------------------------------------------------------------------ introspection
    def last_device_ms(self) -> float:
        ms = C.c_float()
        nat.check(self.lib.m3pc_last_device_ms(self._h, C.byref(ms)), "m3pc_last_device_ms")
        return float(ms.value)

    def last_launch_count(self) -> int:
        n = C.c_int32()
        nat.check(self.lib.m3pc_last_launch_count(self._h, C.byref(n)), "m3pc_last_launch_count")
        return int(n.value)

    def set_profile(self, on: bool) -> None:
        nat.check(self.lib.m3pc_set_profile(self._h, int(bool(on))), "m3pc_set_profile")

    def get_profile(self):
        """(summed GEMM device ms, algorithmic GEMM FLOPs, GEMM launches) of the most recent call in profiling mode."""
        ms, fl, n = C.c_double(), C.c_double(), C.c_int32()
        nat.check(self.lib.m3pc_get_profile(self._h, C.byref(ms), C.byref(fl), C.byref(n)), "m3pc_get_profile")
        return float(ms.value), float(fl.value), int(n.value)

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.m3pc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def engine_from_synthetic(shape, sd, stats, *, precision="bf16", max_batch=1024, chunk=0, critic_sd=None, obs_norm=None,
                          device=None) -> PlanEngine:
    """Build + load an engine from the numpy dicts of ``m3pc_b200.synthetic``."""
    eng = PlanEngine(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer,
                     traj_length=shape.traj_length, obs_dim=shape.obs_dim, act_dim=shape.act_dim, precision=precision,
                     max_batch=max_batch, chunk=chunk, critic_hidden=256 if critic_sd is not None else 0, device=device)
    eng.load_state_dict(sd)
    eng.load_tokenizer_stats(stats)
    if critic_sd is not None:
        eng.load_critic(critic_sd, obs_norm[0], obs_norm[1])
    eng.finalize()
    return eng
