"""``omtm`` / ``omtmConfig`` -- drop-in for research/omtm/models/mtm_model.py:200-221, 324-716 (inference path).

The module owns parameters under exactly the reference's ``state_dict`` key names (so the authors' checkpoints load
with ``load_state_dict``) but none of its sub-modules is ever *called*: ``forward`` hands the tokens to the CUDA engine
(``m3pc_forward`` in include/m3pc.h).  There is no CPU path -- ``forward`` on CPU tensors raises ``NotImplementedError``.

Not provided (out of the planning path, SURVEY.md section 2): ``forward_loss``, ``mask_git_forward``,
``configure_optimizers``, latent_dim != None, discrete modalities, P != 1 tokens per step, training mode.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn

from .engine import MODALITIES, PlanEngine
from .synthetic import sincos_pos_embed


class SquashedNormal:
    """tanh-Gaussian returned for the ``actions`` modality (reference: mtm_model.py:254-291).

    Same surface the planners use: ``.loc``, ``.std``, ``.mean`` (= tanh(loc)), ``.sample(shape)`` / ``.rsample(shape)``.
    """

    def __init__(self, loc: torch.Tensor, std: torch.Tensor):
        self.loc = loc
        self.std = std
        self.scale = std

    @property
    def mean(self) -> torch.Tensor:
        return torch.tanh(self.loc)

    @property
    def device(self):
        return self.loc.device

    def rsample(self, sample_shape=()) -> torch.Tensor:
        shape = tuple(sample_shape) + tuple(self.loc.shape)
        eps = torch.randn(shape, dtype=self.loc.dtype, device=self.loc.device)
        return torch.tanh(self.loc + self.std * eps)

    def sample(self, sample_shape=()) -> torch.Tensor:
        with torch.no_grad():
            return self.rsample(sample_shape)

    # ---- densities (validation loss, finetune_omtm/learner.py:491-499) ----
    def _log_prob_pre(self, u: torch.Tensor) -> torch.Tensor:
        """log density of tanh(u), u ~ N(loc, std): Normal log-density minus log|d tanh / du| = 2 (log 2 - u - softplus(-2u))
        (TanhTransform.log_abs_det_jacobian, mtm_model.py:247-251)."""
        z = (u - self.loc) / self.std
        normal = -0.5 * z * z - torch.log(self.std) - 0.5 * math.log(2.0 * math.pi)
        return normal - 2.0 * (math.log(2.0) - u - torch.nn.functional.softplus(-2.0 * u))

    def log_prob(self, x: torch.Tensor) -> torch.Tensor:
        return self._log_prob_pre(0.5 * (torch.log1p(x) - torch.log1p(-x)))  # atanh as the reference writes it (mtm_model.py:234-236)

    def log_likelihood(self, x: torch.Tensor) -> torch.Tensor:
        """Summed over axis 2 like the reference (mtm_model.py:286-291): (B, T, 1, A) -> (B, T, A)."""
        return self.log_prob(x).sum(dim=2)

    def entropy(self, N: int = 1, eps: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Single-sample estimate -log p(x), x ~ self (mtm_model.py:277-284).  ``eps`` (N, *loc.shape) injects the normal draws
        (test hook); the pre-tanh value is used directly, as the reference's cached transform does."""
        if eps is None:
            eps = torch.randn((N,) + tuple(self.loc.shape), dtype=self.loc.dtype, device=self.loc.device)
        return -self._log_prob_pre(self.loc + self.std * eps).mean(dim=0).sum(dim=2)


@dataclasses.dataclass
class omtmConfig:
    n_embd: int = 128
    n_head: int = 2
    n_enc_layer: int = 1
    n_dec_layer: int = 1
    dropout: float = 0
    embd_pdrop: float = 0
    resid_pdrop: float = 0
    attn_pdrop: float = 0
    norm: str = "l2"
    loss: str = "total"
    reduce_use_sum: bool = False
    loss_keys: Optional[List[str]] = None
    latent_dim: Optional[int] = None
    use_masked_loss: bool = False
    init_temperature: float = 0.1
    target_entropy: float = -3
    use_entropy: bool = True
    # engine options (not in the reference)
    precision: str = "bf16"   # "bf16": tcgen05 tensor cores; "fp32": reference-grade CUDA-core path;
                              # "tf32x3": fp32-grade, the fp32 path with its GEMMs on the tensor cores (3xTF32 split)
    max_batch: int = 1024     # largest batch (candidates or envs) a forward / plan may carry
    chunk: int = 0            # batch rows per kernel sequence (0 = library default)

    def create(self, data_shape, traj_length, discrete_map):
        return omtm(data_shape, traj_length, discrete_map, self)


def _block_params(d: int) -> nn.Module:
    """Parameter container with nn.TransformerEncoderLayer's key names (never called)."""
    m = nn.Module()
    m.self_attn = nn.Module()
    m.self_attn.in_proj_weight = nn.Parameter(torch.empty(3 * d, d))
    m.self_attn.in_proj_bias = nn.Parameter(torch.zeros(3 * d))
    m.self_attn.out_proj = nn.Linear(d, d)
    m.linear1 = nn.Linear(d, 4 * d)
    m.linear2 = nn.Linear(4 * d, d)
    m.norm1 = nn.LayerNorm(d)
    m.norm2 = nn.LayerNorm(d)
    nn.init.xavier_uniform_(m.self_attn.in_proj_weight)
    return m


def _stack_params(d: int, n_layer: int) -> nn.Module:
    m = nn.Module()
    m.layers = nn.ModuleList([_block_params(d) for _ in range(n_layer)])
    m.norm = nn.LayerNorm(d)
    return m


class omtm(nn.Module):
    def __init__(self, data_shapes: Dict[str, Tuple[int, ...]], traj_length: int, discrete_map: Dict[str, bool], config: omtmConfig):
        super().__init__()
        if config.latent_dim is not None:
            raise NotImplementedError("latent_dim != None is not supported by the B200 engine")
        if any(bool(v) for v in discrete_map.values()):
            raise NotImplementedError("discrete modalities are not supported by the B200 engine")
        if tuple(data_shapes.keys()) != MODALITIES:
            raise NotImplementedError(f"data_shapes keys must be {MODALITIES} in this order, got {tuple(data_shapes.keys())}")
        for k, s in data_shapes.items():
            if s[0] != 1:
                raise NotImplementedError(f"{k}: {s[0]} tokens per time step; only P == 1 is supported")
        if data_shapes["rewards"][1] != 1 or data_shapes["returns"][1] != 1:
            raise NotImplementedError("rewards / returns must be scalar per step")
        if config.n_embd != 128 * config.n_head:
            raise NotImplementedError("the B200 attention kernel needs head_dim == 128 (n_embd == 128 * n_head)")
        self.data_shapes = data_shapes
        self.n_embd = config.n_embd
        self.config = config
        self.max_len = traj_length
        self.norm = config.norm
        self.log_temperature = torch.tensor(np.log(config.init_temperature))
        self.target_entropy = config.target_entropy
        d = self.n_embd
        self.encoder_embed_dict = nn.ModuleDict()
        self.decoder_embed_dict = nn.ModuleDict()
        self.mask_token_dict = nn.ParameterDict()
        self.encoder_per_dim_encoding = nn.ParameterDict()
        self.decoder_per_dim_encoding = nn.ParameterDict()
        for key, shape in data_shapes.items():
            self.encoder_embed_dict[key] = nn.Linear(shape[1], d)
            self.decoder_embed_dict[key] = nn.Linear(d, d)
            self.mask_token_dict[key] = nn.Parameter(torch.zeros(1, 1, d))
            self.encoder_per_dim_encoding[key] = nn.Parameter(torch.zeros(1, 1, shape[0], d))
            self.decoder_per_dim_encoding[key] = nn.Parameter(torch.zeros(1, 1, shape[0], d))
        self.encoder = _stack_params(d, config.n_enc_layer)
        self.decoder = _stack_params(d, config.n_dec_layer)
        self.output_head_dict = nn.ModuleDict()
        for key, shape in data_shapes.items():
            if key == "actions":
                actor = nn.Module()
                actor.mu = nn.Linear(d, shape[-1])
                actor.log_std = nn.Linear(d, shape[-1])
                for lin in (actor.mu, actor.log_std):
                    nn.init.orthogonal_(lin.weight.data)
                    lin.bias.data.fill_(0.0)
                self.output_head_dict[key] = actor
            else:
                self.output_head_dict[key] = nn.Sequential(nn.LayerNorm(d), nn.Linear(d, d), nn.GELU(), nn.Linear(d, shape[-1]))
        self.register_buffer("pos_embed", torch.from_numpy(sincos_pos_embed(d, traj_length)))
        self.__dict__["_engine"] = None
        self.__dict__["_engine_synced"] = False
        self.eval()

    # ---- parameters <-> engine ------------------------------------------------------------------------
    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        res = super().load_state_dict(state_dict, strict=strict, **kw)
        self._engine_synced = False
        return res

    def mark_dirty(self) -> None:
        """Call after mutating parameters in place (e.g. an optimiser step) so the engine re-packs them."""
        self._engine_synced = False

    def engine(self, *, max_batch: Optional[int] = None, critic_hidden: int = 0) -> PlanEngine:
        """The CUDA engine bound to this module's parameters (created on first use, on the parameters' device)."""
        dev = self.pos_embed.device
        if dev.type != "cuda":
            raise NotImplementedError("omtm lives on a CPU device: the B200 engine has no CPU path (move it with .to('cuda'))")
        want_batch = max(int(max_batch or 0), int(self.config.max_batch))
        e = self._engine
        if e is None or e.device != dev or e.max_batch < want_batch or (critic_hidden and e.critic_hidden != critic_hidden):
            if e is not None:
                e.close()
            shapes = self.data_shapes
            e = PlanEngine(n_embd=self.n_embd, n_head=self.config.n_head, n_enc_layer=self.config.n_enc_layer,
                           n_dec_layer=self.config.n_dec_layer, traj_length=self.max_len, obs_dim=shapes["states"][1],
                           act_dim=shapes["actions"][1], precision=self.config.precision, max_batch=want_batch,
                           chunk=self.config.chunk, critic_hidden=critic_hidden, device=dev)
            self._engine = e
            self._engine_synced = False
        return e

    def bind_planner(self, tokenizer_manager=None, critic=None, max_batch: Optional[int] = None) -> None:
        """Attach what the fused planners need besides the MTM weights: tokenizer statistics (normalisation happens
        inside the kernels) and the TwinQ critic.  Stored outside the module tree so ``state_dict()`` keeps the
        reference's keys."""
        self.__dict__["_bound"] = (tokenizer_manager, critic, max_batch)
        self._engine_synced = False

    def sync_engine(self) -> PlanEngine:
        """Upload parameters (and, for the planners, tokenizer statistics and TwinQ weights) if anything changed."""
        tokenizer_manager, critic, max_batch = self.__dict__.get("_bound", (None, None, None))
        critic_hidden = 0
        if critic is not None:  # this package's TwinQ keeps hidden_dim; the reference's (finetune_omtm/model.py:146-160) only its layers
            critic_hidden = int(getattr(critic, "hidden_dim", 0) or critic.q1.net[0].out_features)
        e = self.engine(max_batch=max_batch, critic_hidden=critic_hidden)
        if not self._engine_synced or not e.finalized:
            e.load_state_dict(self.state_dict())
            if tokenizer_manager is not None:
                from .tokenizers import engine_stats
                e.load_tokenizer_stats(engine_stats(tokenizer_manager))
            else:  # omtm.forward alone never normalises; identity statistics keep the handle complete
                dims = {k: s[1] for k, s in self.data_shapes.items()}
                e.load_tokenizer_stats({k: {"mean": np.zeros(dims[k], np.float32), "std": np.ones(dims[k], np.float32)}
                                        for k in ("states", "rewards", "returns")})
            if critic is not None:
                e.load_critic(critic.state_dict(), critic.obs_mean, critic.obs_std)
            e.finalize()
            self._engine_synced = True
        return e

    # ---- omtm.forward (mtm_model.py:593-607) ------------------------------------------------------------
    def process_masks(self, trajectories, masks) -> Dict[str, torch.Tensor]:
        """Shape checks of mtm_model.py:559-591; returns the flattened (T*P,) masks."""
        out = {}
        batch = None
        for k, v in trajectories.items():
            assert v.shape[2] == self.data_shapes[k][0], f"{v.shape}, {self.data_shapes}"
            assert v.shape[3] == self.data_shapes[k][1], f"{v.shape}, {self.data_shapes}"
            mask = masks[k]
            if len(mask.shape) == 1:
                mask = mask[:, None].repeat(1, v.shape[2])
            elif len(mask.shape) == 2:
                pass
            else:
                raise NotImplementedError(f"mask shape = {mask.shape}")
            if batch is None:
                batch = v.shape[0]
            else:
                assert batch == v.shape[0]
            out[k] = mask.reshape(-1)
        return out

    @torch.no_grad()
    def forward(self, trajectories: Dict[str, torch.Tensor], masks: Dict[str, torch.Tensor]):
        """trajectories[k]: (B,T,1,d_k) tokenised; masks[k]: (T,) or (T,1).  Returns Dict[k -> (B,T,1,d_k)] with
        ``actions`` a SquashedNormal, like the reference."""
        if self.training:
            raise NotImplementedError("the B200 engine is inference-only: call .eval()")
        if tuple(trajectories.keys()) != MODALITIES:
            raise NotImplementedError(f"trajectories must have keys {MODALITIES} in this order")
        flat = self.process_masks(trajectories, masks)
        eng = self.sync_engine()
        toks = {k: v.to(torch.float32).squeeze(2) for k, v in trajectories.items()}
        raw = eng.forward(toks, {k: flat[k] for k in MODALITIES})
        out = {}
        for k in ("states", "rewards", "returns"):
            out[k] = raw[k].unsqueeze(2)
        out["actions"] = SquashedNormal(raw["act_mu"].unsqueeze(2), raw["act_std"].unsqueeze(2))
        return {k: out[k] for k in MODALITIES}

    def temperature(self):
        return self.log_temperature.exp()
