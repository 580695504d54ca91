"""The C-ABI library loads and exports exactly what include/m3pc.h declares (no compute: no GPU needed)."""
import ctypes as C
import os
import re
import subprocess

import pytest

from m3pc_b200 import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(nat.LIB_PATH):
        nat.build()
    return nat.lib()


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "m3pc.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(m3pc_[a-z0-9_]+)\s*\(", src)))


def test_header_binding_and_library_agree(lib):
    hdr = _header_symbols()
    assert sorted(nat.SYMBOLS) == hdr, "m3pc_b200/_native.py SYMBOLS is out of sync with include/m3pc.h"
    out = subprocess.run(["nm", "-D", "--defined-only", nat.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = sorted(set(re.findall(r" T (m3pc_[a-z0-9_]+)", out)))
    assert exported == hdr, f"library exports {exported}, header declares {hdr}"


def test_constants_match_header():
    src = open(os.path.join(ROOT, "include", "m3pc.h")).read()
    defs = dict(re.findall(r"#define\s+(M3PC_[A-Z0-9_]+)\s+\(?(-?\d+)\)?\s", src))
    assert int(defs["M3PC_MAX_T"]) == nat.MAX_T and int(defs["M3PC_MAX_ACT"]) == nat.MAX_ACT and int(defs["M3PC_MAX_OBS"]) == nat.MAX_OBS
    assert int(defs["M3PC_PREC_BF16"]) == nat.PREC_BF16 and int(defs["M3PC_PREC_FP32"]) == nat.PREC_FP32
    for name, val in (("RTG", nat.GUIDE_RTG), ("CRITIC", nat.GUIDE_CRITIC), ("NOISE_CRITIC", nat.GUIDE_NOISE_CRITIC), ("SAMPLING", nat.GUIDE_SAMPLING)):
        assert int(defs[f"M3PC_GUIDE_{name}"]) == val
    assert nat.PARTIAL_FLOATS == 8 + 2 * nat.MAX_ACT
    # struct sizes as the header lays them out (LP64)
    assert C.sizeof(nat.Config) == 16 * 4
    assert C.sizeof(nat.PlanArgs) == 8 * 4 + 6 * 8 + 8 + 6 * 8 + 4 * 8
    assert C.sizeof(nat.AttnTok) == 8 + 2 * 4


def test_version_and_error_strings(lib):
    assert b"sm_100a" in lib.m3pc_version()
    assert isinstance(lib.m3pc_last_error(), bytes)


def test_invalid_arguments_are_rejected_without_a_gpu(lib):
    # argument validation happens before any CUDA call
    assert lib.m3pc_create(None, None) == -1
    assert b"null" in lib.m3pc_last_error()
    h = C.c_void_p()
    bad = nat.Config(n_embd=500, n_head=4, n_enc_layer=2, n_dec_layer=1, traj_length=8, obs_dim=11, act_dim=3, max_batch=4)
    assert lib.m3pc_create(C.byref(h), C.byref(bad)) == -1
    assert b"n_embd" in lib.m3pc_last_error()
    bad = nat.Config(n_embd=512, n_head=4, n_enc_layer=2, n_dec_layer=1, traj_length=99, obs_dim=11, act_dim=3, max_batch=4)
    assert lib.m3pc_create(C.byref(h), C.byref(bad)) == -1
    assert lib.m3pc_forward(None, 1, None, None, None, None, None, None, None, None, None, None, None) == -1
    assert lib.m3pc_plan(None, None, None) == -1
    assert lib.m3pc_attention_gather(None, 1, None, None, 1, 0, 1, 1, None, 1, None, None) == -1
    assert lib.m3pc_destroy(None) == 0


def test_release_library_reads_no_environment_switch(lib):
    """Launch choices go through m3pc_set_option only: the library holds no M3PC_* environment variable name and therefore
    reads none."""
    assert nat.LIB_PATH.endswith("libm3pc.so")
    blob = open(nat.LIB_PATH, "rb").read()
    names = set(re.findall(rb"\x00(M3PC_[A-Z][A-Z0-9_]{3,})\x00", blob))  # a getenv() argument is a string of its own
    assert not names, f"environment switch names in the release library: {sorted(names)}"
    assert lib.m3pc_set_option(None, b"graphs", 0) == -1  # argument validation without a GPU


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    h = C.c_void_p()
    ok = nat.Config(n_embd=512, n_head=4, n_enc_layer=2, n_dec_layer=1, traj_length=8, obs_dim=11, act_dim=3, max_batch=4)
    assert lib.m3pc_create(C.byref(h), C.byref(ok)) == -2  # M3PC_ERR_CUDA: fails loudly, never computes on the host
    from m3pc_b200.engine import PlanEngine
    with pytest.raises(RuntimeError):
        PlanEngine(n_embd=512, n_head=4, n_enc_layer=2, n_dec_layer=1, traj_length=8, obs_dim=11, act_dim=3)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "m3pc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f"{f} imports the oracle"


def test_gemm_entry_structs_match_header():
    assert C.sizeof(nat.GemmProblem) == 5 * 8 + 5 * 4 + 4  # padded to pointer alignment
    assert C.sizeof(nat.LnJob) == 6 * 8 + 2 * 4
    src = open(os.path.join(ROOT, "include", "m3pc.h")).read()
    defs = dict(re.findall(r"#define\s+(M3PC_EPI_[A-Z0-9_]+)\s+(\d+)", src))
    assert {k: int(v) for k, v in defs.items()} == {"M3PC_EPI_GELU": nat.EPI_GELU, "M3PC_EPI_RESIDUAL": nat.EPI_RESIDUAL, "M3PC_EPI_RELU": nat.EPI_RELU,
                                                    "M3PC_EPI_ROWTABLE": nat.EPI_ROWTABLE, "M3PC_EPI_OUT_F32": nat.EPI_OUT_F32}


# Pointer values below are never dereferenced: every rule is checked before the first CUDA call, so these run without a GPU.
A16, W16, C16, T16, B16 = 0x10000, 0x20000, 0x30000, 0x40000, 0x50000


def _gemm_rc(lib, n=1, **kw):
    f = dict(A=A16, W=W16, bias=B16, table=None, C=C16, M=256, N=512, K=512, rows_per_group=1, flags=0)
    f.update(kw)
    arr = (nat.GemmProblem * max(n, 1))(*[nat.GemmProblem(**f)] * max(n, 1))
    return lib.m3pc_gemm_bf16_problems(arr, n, None, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(bias=B16 + 4), b"16-byte aligned"),                              # a bias slice at a 4-byte offset (float4 / float2 loads)
    (dict(bias=B16 + 8), b"16-byte aligned"),
    (dict(table=T16 + 4, flags=nat.EPI_ROWTABLE), b"16-byte aligned"),
    (dict(table=T16), b"EPI_ROWTABLE"),                                     # a table without the flag
    (dict(flags=nat.EPI_ROWTABLE), b"EPI_ROWTABLE"),                        # the flag without a table
    (dict(table=T16, flags=nat.EPI_ROWTABLE, rows_per_group=0), b"rows_per_group"),
    (dict(rows_per_group=-3), b"rows_per_group"),
    (dict(table=T16, flags=nat.EPI_ROWTABLE | nat.EPI_RESIDUAL), b"exclude"),  # two residual sources
    (dict(flags=32), b"unknown flag"),
    (dict(C=C16 + 2), b"16-byte aligned"),
    (dict(K=100), b"multiple of 64"),
    (dict(N=200), b"multiple of 128"),
    (dict(A=None), b"null"),
])
def test_gemm_bf16_problems_rejects_without_a_gpu(lib, kw, msg):
    assert _gemm_rc(lib, **kw) == -1
    assert msg in lib.m3pc_last_error(), lib.m3pc_last_error()


def test_gemm_entries_reject_misaligned_bias_and_table_without_a_gpu(lib):
    assert _gemm_rc(lib, n=0) == -1 and _gemm_rc(lib, n=65) == -1
    assert lib.m3pc_gemm_bf16_problems(None, 1, None, None) == -1
    # the older entries share the dispatcher's checks
    assert lib.m3pc_gemm_bf16(A16, W16, B16 + 4, C16, 256, 512, 512, 0, None) == -1
    assert b"16-byte aligned" in lib.m3pc_last_error()
    bias = (C.c_void_p * 2)(B16, B16 + 4)
    ptrs = lambda v: (C.c_void_p * 2)(v, v)
    i32 = lambda *xs: (C.c_int32 * 2)(*xs)
    assert lib.m3pc_gemm_bf16_grouped(2, ptrs(A16), ptrs(W16), bias, ptrs(C16), i32(256, 256), i32(512, 512), i32(512, 512), i32(0, 0), None) == -1
    assert lib.m3pc_gemm_ln_bf16(A16, W16, B16, C16, C16 + 0x100000, B16, B16, T16 + 4, 8, 256, 512, None) == -1
    assert b"16-byte aligned" in lib.m3pc_last_error()


def _ln_rc(lib, n=1, K=512, gamma=B16, **kw):
    f = dict(A=A16, W=W16, X=C16, Y=C16 + 0x100000, table=None, R=None, rows_per_group=1, M=256)
    f.update(kw)
    arr = (nat.LnJob * max(n, 1))(*[nat.LnJob(**f)] * max(n, 1))
    return lib.m3pc_gemm_ln_bf16_grouped(arr, n, B16, gamma, B16, K, None, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(table=T16 + 4, rows_per_group=8), b"16-byte aligned"),
    (dict(R=T16 + 8), b"16-byte aligned"),
    (dict(table=T16, R=T16 + 0x1000), b"excludes"),
    (dict(table=T16, rows_per_group=0), b"rows_per_group"),
    (dict(rows_per_group=0), b"rows_per_group"),
    (dict(n=0), b"1 .. 4"),
    (dict(n=5), b"1 .. 4"),
    (dict(K=96), b"multiple of 64"),
    (dict(gamma=None), b"null"),
    (dict(Y=C16 + 2), b"16-byte aligned"),
    (dict(M=0), b"empty"),
])
def test_gemm_ln_bf16_grouped_rejects_without_a_gpu(lib, kw, msg):
    assert _ln_rc(lib, **kw) == -1
    assert msg in lib.m3pc_last_error(), lib.m3pc_last_error()
