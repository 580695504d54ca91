"""ctypes binding of the C-ABI in ``include/m3pc.h`` (``m3pc_b200/libm3pc.so``, built from ``m3pc_b200/csrc``).

The library is the product: there is no Python/torch fallback.  ``lib()`` raises ``NativeLibraryError`` if the
shared object is missing or does not export every symbol the header declares.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libm3pc.so")
CSRC = os.path.join(HERE, "csrc")

OK = 0
PREC_BF16, PREC_FP32, PREC_TF32X3 = 0, 1, 2
GUIDE_RTG, GUIDE_CRITIC, GUIDE_NOISE_CRITIC, GUIDE_SAMPLING = 0, 1, 2, 3
MAX_T, MAX_ACT, MAX_OBS = 16, 32, 128
PARTIAL_FLOATS = 8 + 2 * MAX_ACT
IPC_HANDLE_BYTES = 64

GUIDANCE = {
    "rtg_guiding": GUIDE_RTG,
    "critic_lambda_guiding": GUIDE_CRITIC,
    "noise_adding_lambda": GUIDE_NOISE_CRITIC,
    "mtm_sampling": GUIDE_SAMPLING,
}

#: every symbol include/m3pc.h declares (tests/test_abi.py checks the header against this list and the .so)
SYMBOLS = (
    "m3pc_last_error", "m3pc_version", "m3pc_create", "m3pc_destroy", "m3pc_set_param", "m3pc_finalize_params", "m3pc_set_option",
    "m3pc_forward", "m3pc_plan", "m3pc_merge_partials", "m3pc_exchange_local", "m3pc_exchange_connect", "m3pc_exchange_status", "m3pc_backward_plan", "m3pc_backward_plan_draws",
    "m3pc_backward_plan_env", "m3pc_ring_reset", "m3pc_ring_append_slots", "m3pc_ring_write_obs", "m3pc_ring_windows_slots", "m3pc_gemm_bf16", "m3pc_gemm_bf16_grouped", "m3pc_gemm_ln_bf16",
    "m3pc_gemm_bf16_problems", "m3pc_gemm_ln_bf16_grouped", "m3pc_gemm_fp32", "m3pc_gemm_tf32x3",
    "m3pc_layernorm", "m3pc_attention", "m3pc_attention_gather", "m3pc_embed_gather", "m3pc_decoder_scatter_embed", "m3pc_block_forward", "m3pc_heads", "m3pc_sample_candidates", "m3pc_twinq",
    "m3pc_score_select", "m3pc_last_device_ms", "m3pc_last_launch_count", "m3pc_set_profile", "m3pc_get_profile",
)


class NativeLibraryError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ("n_embd", C.c_int32), ("n_head", C.c_int32), ("n_enc_layer", C.c_int32), ("n_dec_layer", C.c_int32),
        ("traj_length", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("precision", C.c_int32),
        ("max_batch", C.c_int32), ("chunk", C.c_int32), ("critic_hidden", C.c_int32), ("reserved", C.c_int32 * 5),
    ]


class PlanArgs(C.Structure):
    _fields_ = [
        ("guidance", C.c_int32), ("horizon", C.c_int32), ("n_cand", C.c_int32), ("cand_offset", C.c_int32),
        ("discount", C.c_float), ("temperature", C.c_float), ("lmbda", C.c_float), ("n_env", C.c_int32),
        ("win_states", C.c_void_p), ("win_actions", C.c_void_p), ("win_rewards", C.c_void_p), ("win_returns_tok", C.c_void_p),
        ("eps", C.c_void_p), ("expq", C.c_void_p), ("seed", C.c_uint64),
        ("out_eval_action", C.c_void_p), ("out_sample_action", C.c_void_p), ("out_partials", C.c_void_p),
        ("dbg_expect_return", C.c_void_p), ("dbg_candidates", C.c_void_p), ("dbg_indices", C.c_void_p),
        ("exchange", C.c_int32), ("reserved0", C.c_int32), ("env_horizons", C.c_void_p), ("reserved1", C.c_void_p * 2),
    ]


class AttnTok(C.Structure):
    """m3pc_attn_tok_t: one query / key / value token of m3pc_attention_gather."""
    _fields_ = [("ptr", C.c_void_p), ("bstride", C.c_int32), ("bdiv", C.c_int32)]


EPI_GELU, EPI_RESIDUAL, EPI_RELU, EPI_ROWTABLE, EPI_OUT_F32 = 1, 2, 4, 8, 16


class GemmProblem(C.Structure):
    """m3pc_gemm_problem_t: one problem of m3pc_gemm_bf16_problems."""
    _fields_ = [("A", C.c_void_p), ("W", C.c_void_p), ("bias", C.c_void_p), ("table", C.c_void_p), ("C", C.c_void_p),
                ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("rows_per_group", C.c_int32), ("flags", C.c_int32)]


class LnJob(C.Structure):
    """m3pc_ln_job_t: one job of m3pc_gemm_ln_bf16_grouped."""
    _fields_ = [("A", C.c_void_p), ("W", C.c_void_p), ("X", C.c_void_p), ("Y", C.c_void_p), ("table", C.c_void_p), ("R", C.c_void_p),
                ("rows_per_group", C.c_int32), ("M", C.c_int32)]


_lib: Optional[C.CDLL] = None


def build(verbose: bool = False) -> str:
    """Compile the library in-tree with nvcc for sm_100a (``make -C m3pc_b200/csrc``)."""
    res = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0:
        raise NativeLibraryError("building libm3pc.so failed (see output above)")
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} not found: build it with `make -C {CSRC}` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "There is no CPU / PyTorch fallback for this path.")
    L = C.CDLL(LIB_PATH)
    missing = [s for s in SYMBOLS if not hasattr(L, s)]
    if missing:
        raise NativeLibraryError(f"{LIB_PATH} does not export {missing}")
    vp, i32, f32p = C.c_void_p, C.c_int32, C.c_void_p
    L.m3pc_last_error.restype = C.c_char_p
    L.m3pc_version.restype = C.c_char_p
    L.m3pc_create.argtypes = [C.POINTER(vp), C.POINTER(Config)]
    L.m3pc_destroy.argtypes = [vp]
    L.m3pc_set_param.argtypes = [vp, C.c_char_p, vp, C.c_size_t]
    L.m3pc_finalize_params.argtypes = [vp]
    L.m3pc_set_option.argtypes = [vp, C.c_char_p, i32]
    L.m3pc_forward.argtypes = [vp, i32, f32p, f32p, f32p, f32p, vp, f32p, f32p, f32p, f32p, f32p, vp]
    L.m3pc_plan.argtypes = [vp, C.POINTER(PlanArgs), vp]
    L.m3pc_merge_partials.argtypes = [vp, f32p, i32, C.c_float, f32p, f32p, vp, vp]
    L.m3pc_exchange_local.argtypes = [vp, vp, C.POINTER(vp)]
    L.m3pc_exchange_connect.argtypes = [vp, i32, i32, vp, vp]
    L.m3pc_exchange_status.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.m3pc_backward_plan.argtypes = [vp, i32, i32, i32, f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, vp]
    L.m3pc_backward_plan_draws.argtypes = [vp, i32, i32, i32, i32, f32p, f32p, f32p, f32p, f32p, C.c_uint64, f32p, f32p, vp]
    L.m3pc_backward_plan_env.argtypes = [vp, i32, i32, vp, i32, f32p, f32p, f32p, f32p, f32p, C.c_uint64, f32p, f32p, vp]
    L.m3pc_ring_write_obs.argtypes = [f32p, i32, i32, i32, i32, vp, i32, i32, i32, f32p, vp]
    L.m3pc_ring_reset.argtypes = [f32p, i32, i32, i32, i32, vp, i32, vp]
    L.m3pc_ring_append_slots.argtypes = [f32p, i32, i32, i32, i32, vp, vp, i32, f32p, f32p, f32p, vp]
    L.m3pc_ring_windows_slots.argtypes = [f32p, i32, i32, i32, i32, vp, vp, vp, i32, i32, i32, f32p, f32p, f32p, f32p, f32p, vp]
    L.m3pc_gemm_bf16.argtypes = [vp, vp, f32p, vp, i32, i32, i32, i32, vp]
    L.m3pc_gemm_bf16_grouped.argtypes = [i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.m3pc_gemm_ln_bf16.argtypes = [vp, vp, f32p, f32p, vp, f32p, f32p, f32p, i32, i32, i32, vp]
    L.m3pc_gemm_bf16_problems.argtypes = [C.POINTER(GemmProblem), i32, C.POINTER(i32), vp]
    L.m3pc_gemm_ln_bf16_grouped.argtypes = [C.POINTER(LnJob), i32, f32p, f32p, f32p, i32, C.POINTER(i32), vp]
    L.m3pc_gemm_fp32.argtypes = [f32p, f32p, f32p, f32p, i32, i32, i32, i32, vp]
    L.m3pc_gemm_tf32x3.argtypes = [f32p, f32p, f32p, f32p, i32, i32, i32, i32, vp]
    L.m3pc_layernorm.argtypes = [f32p, f32p, f32p, vp, i32, i32, i32, vp]
    L.m3pc_attention.argtypes = [vp, vp, i32, i32, i32, i32, vp]
    L.m3pc_attention_gather.argtypes = [C.POINTER(AttnTok), i32, C.POINTER(AttnTok), C.POINTER(AttnTok), i32, i32, i32, i32, vp, i32,
                                        C.POINTER(i32), vp]
    L.m3pc_embed_gather.argtypes = [vp, i32, f32p, f32p, f32p, f32p, vp, f32p, vp, vp]
    L.m3pc_decoder_scatter_embed.argtypes = [vp, i32, vp, vp, f32p, vp]
    L.m3pc_heads.argtypes = [vp, i32, f32p, f32p, f32p, f32p, f32p, f32p, vp]
    L.m3pc_block_forward.argtypes = [vp, i32, i32, i32, i32, f32p, vp, vp]
    L.m3pc_sample_candidates.argtypes = [f32p, f32p, f32p, C.c_uint64, i32, i32, i32, i32, i32, i32, f32p, vp]
    L.m3pc_twinq.argtypes = [vp, f32p, f32p, i32, i32, f32p, vp]
    L.m3pc_score_select.argtypes = [f32p, f32p, f32p, f32p, f32p, vp, C.c_float, C.c_float, C.c_float, i32, i32, i32, i32, C.c_uint64, i32,
                                    f32p, f32p, f32p, f32p, vp, vp]
    L.m3pc_last_device_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.m3pc_last_launch_count.argtypes = [vp, C.POINTER(C.c_int32)]
    L.m3pc_set_profile.argtypes = [vp, i32]
    L.m3pc_get_profile.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32)]
    for s in SYMBOLS:
        if s not in ("m3pc_last_error", "m3pc_version"):
            getattr(L, s).restype = C.c_int
    _lib = L
    return L


def check(rc: int, what: str = "m3pc call") -> None:
    if rc != OK:
        msg = lib().m3pc_last_error().decode("utf-8", "replace")
        kind = {-1: "invalid argument", -2: "CUDA error", -3: "bad call order", -4: "out of memory"}.get(rc, f"error {rc}")
        if rc == -1:
            raise ValueError(f"{what}: {kind}: {msg}")
        raise RuntimeError(f"{what}: {kind}: {msg}")
