"""The tf32x3 precision mode's host-side surface (no GPU): the exported kernel entry, the header constant and the Python names."""
import os
import re
import subprocess

import pytest

from m3pc_b200 import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_the_tf32x3_gemm():
    if not os.path.exists(nat.LIB_PATH):
        nat.build()
    out = subprocess.run(["nm", "-D", "--defined-only", nat.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert re.search(r" T m3pc_gemm_tf32x3$", out, flags=re.M)
    assert "m3pc_gemm_tf32x3" in nat.SYMBOLS


def test_header_constant():
    src = open(os.path.join(ROOT, "include", "m3pc.h")).read()
    assert int(re.search(r"#define\s+M3PC_PREC_TF32X3\s+(\d+)", src).group(1)) == 2 == nat.PREC_TF32X3


def test_precision_names():
    from m3pc_b200.engine import PRECISIONS, PlanEngine
    assert PRECISIONS == {"bf16": nat.PREC_BF16, "fp32": nat.PREC_FP32, "tf32x3": nat.PREC_TF32X3}
    with pytest.raises(ValueError, match="unknown precision"):
        PlanEngine(n_embd=512, n_head=4, n_enc_layer=1, n_dec_layer=1, traj_length=4, obs_dim=3, act_dim=2, precision="fp16")
