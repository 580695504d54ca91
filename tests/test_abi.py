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
