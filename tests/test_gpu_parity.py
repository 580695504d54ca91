"""Parity tests proper (need a B200): every call goes through the C-ABI (include/m3pc.h) via ctypes.

Tolerances
  fp32 mode  -- "1e-5 with an fp32 accumulate mode" (BASELINE.json north_star): max |x - ref| <= 2e-5 * max(1, max|ref|).
                Measured ~1e-6 against the float64 oracle.
  bf16 mode  -- "within 1e-2 relative error at bf16": max |x - ref| <= 1e-2 * max(1, max|ref|) for states / rewards / returns /
                action mu / action mean; the action std = exp(-5 + 3.5 (tanh(.) + 1)) amplifies its pre-activation error by up
                to 3.5x, so it gets 3.5e-2.  Measured 3e-3 .. 7e-3 (std up to 1.2e-2).
  indices    -- bit-exact wherever the score gap exceeds twice the measured score error.
"""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from m3pc_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

TOL = {"fp32": 2e-5, "bf16": 1e-2}


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(1.0, float(b.abs().max())))


@pytest.fixture(scope="module")
def nat():
    from m3pc_b200 import _native
    _native.lib()
    return _native


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("M,N,K,flags", [(17, 1536, 512, 0), (200, 512, 2048, 1), (333, 256, 23, 4), (64, 1, 256, 0), (1000, 512, 512, 2),
                                         # the 128 x 128 tiling: ragged rows / columns / K, one slab, every epilogue
                                         (128, 128, 16, 0), (129, 130, 17, 2), (1000, 2048, 512, 1), (4099, 257, 100, 6), (13312, 512, 2048, 2)])
def test_gemm_fp32(nat, M, N, K, flags):
    torch.manual_seed(0)
    A, W, b = torch.randn(M, K, device="cuda"), torch.randn(N, K, device="cuda") / K ** 0.5, torch.randn(N, device="cuda")
    Cm = torch.randn(M, N, device="cuda")
    C0 = Cm.clone()
    nat.check(nat.lib().m3pc_gemm_fp32(A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, flags, None))
    ref = A.double() @ W.double().T + b.double()
    if flags & 1: ref = torch.nn.functional.gelu(ref)
    if flags & 4: ref = torch.relu(ref)
    if flags & 2: ref = ref + C0.double()
    assert rel(Cm, ref) < 1e-5


@pytest.mark.parametrize("M,N,K,flags", [(128, 128, 64, 0), (17, 1536, 512, 0), (8125, 512, 512, 2), (1000, 2048, 512, 1), (333, 512, 2048, 2),
                                         (4096, 1536, 512, 0), (130, 128, 128, 4), (1, 128, 64, 0), (20000, 2048, 512, 1), (32768, 512, 2048, 2),
                                         # CTA-pair kernel: ragged / odd row-tile counts, one k-block, resident-A and streaming variants
                                         (13312, 1536, 512, 0), (300, 256, 64, 4), (129, 256, 256, 0), (257, 512, 512, 2), (7168, 2048, 512, 1),
                                         (385, 256, 1024, 0), (640, 1024, 512, 0), (13312, 512, 2048, 2), (4099, 256, 256, 4)])
def test_gemm_bf16_tcgen05(nat, M, N, K, flags):
    """The tensor-core GEMM against an fp64 product of the same bf16 operands (operand rounding excluded):
    fp32-output epilogues must be fp32-accurate, bf16 outputs within half a bf16 ulp of the largest value."""
    torch.manual_seed(1)
    A = torch.randn(M, K, device="cuda").bfloat16()
    W = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16()
    b = torch.randn(N, device="cuda")
    ref = A.double() @ W.double().T + b.double()
    if flags & 1: ref = torch.nn.functional.gelu(ref)
    if flags & 4: ref = torch.relu(ref)
    if flags & 2:
        Cm = torch.randn(M, N, device="cuda")
        ref = ref + Cm.double()
    else:
        Cm = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    nat.check(nat.lib().m3pc_gemm_bf16(A.data_ptr(), W.data_ptr(), b.data_ptr(), Cm.data_ptr(), M, N, K, flags, None))
    torch.cuda.synchronize()
    assert torch.isfinite(Cm.float()).all()
    assert rel(Cm, ref) < (2e-5 if flags & 2 else 4e-3)


@pytest.mark.parametrize("probs", [
    # decoder-embedding runs (two modalities), K/V + Q, heads (two modalities), twin critics, and a 5-problem list (two launches)
    [(5120, 512, 512, 0), (8192, 512, 512, 0)],
    [(13312, 1024, 512, 0), (1024, 512, 512, 0)],
    [(4096, 512, 512, 1), (3072, 512, 512, 1)],
    [(4096, 256, 64, 4), (4096, 256, 64, 4)],
    [(4099, 256, 256, 4), (37, 512, 512, 0), (300, 256, 64, 4), (257, 512, 1024, 2)],
    [(640, 1024, 512, 0), (129, 256, 256, 0), (1000, 2048, 512, 1), (333, 512, 2048, 2), (2000, 256, 128, 4)],
])
def test_gemm_bf16_grouped(nat, probs):
    """Several independent GEMMs in one launch of the CTA-pair kernel: every problem against its own fp64 product."""
    import ctypes as C
    torch.manual_seed(2)
    n = len(probs)
    As, Ws, bs, Cs, refs = [], [], [], [], []
    for (M, N, K, flags) in probs:
        A = torch.randn(M, K, device="cuda").bfloat16()
        W = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16()
        b = torch.randn(N, device="cuda")
        ref = A.double() @ W.double().T + b.double()
        if flags & 1: ref = torch.nn.functional.gelu(ref)
        if flags & 4: ref = torch.relu(ref)
        if flags & 2:
            Cm = torch.randn(M, N, device="cuda")
            ref = ref + Cm.double()
        else:
            Cm = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
        As.append(A); Ws.append(W); bs.append(b); Cs.append(Cm); refs.append(ref)
    vp = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    i32 = lambda xs: (C.c_int32 * n)(*xs)
    nat.check(nat.lib().m3pc_gemm_bf16_grouped(n, vp(As), vp(Ws), vp(bs), vp(Cs), i32([p[0] for p in probs]), i32([p[1] for p in probs]),
                                               i32([p[2] for p in probs]), i32([p[3] for p in probs]), None))
    torch.cuda.synchronize()
    for (M, N, K, flags), Cm, ref in zip(probs, Cs, refs):
        assert torch.isfinite(Cm.float()).all(), (M, N, K, flags)
        assert rel(Cm, ref) < (2e-5 if flags & 2 else 4e-3), (M, N, K, flags)


@pytest.mark.parametrize("M,K,table_rows", [(256, 512, 0), (300, 512, 0), (13312, 512, 0), (13312, 2048, 0), (4000, 512, 1000), (53248 + 77, 2048, 0)])
def test_gemm_residual_layernorm_fused(nat, M, K, table_rows):
    """m3pc_gemm_ln_bf16: X += A W^T + b (or X = table[row / g] + A W^T + b) and Y = LayerNorm(X) in one tensor-core kernel whose
    CTA pair owns whole 512-wide rows -- against plain PyTorch fp32 on the same bf16-rounded operands."""
    L = nat.lib()
    g = torch.Generator(device="cuda").manual_seed(M + K)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    W = (torch.randn(512, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
    bias = torch.randn(512, device="cuda", generator=g)
    gamma = 1 + 0.2 * torch.randn(512, device="cuda", generator=g)
    beta = 0.2 * torch.randn(512, device="cuda", generator=g)
    X = 2.0 * torch.randn(M, 512, device="cuda", generator=g) + 0.5
    Y = torch.full((M, 512), float("nan"), device="cuda", dtype=torch.bfloat16)
    table, grp = None, 1
    if table_rows:
        grp = table_rows
        table = torch.randn((M + grp - 1) // grp, 512, device="cuda", generator=g)
        resid = table.repeat_interleave(grp, dim=0)[:M]
    else:
        resid = X.clone()
    ref_x = resid + A.float() @ W.float().t() + bias
    ref_y = torch.nn.functional.layer_norm(ref_x, (512,), gamma, beta, 1e-5)
    nat.check(L.m3pc_gemm_ln_bf16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), X.data_ptr(), Y.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                  table.data_ptr() if table is not None else None, grp, M, K, None), "m3pc_gemm_ln_bf16")
    torch.cuda.synchronize()
    assert rel(X, ref_x) < 2e-3
    assert torch.isfinite(Y.float()).all()
    assert rel(Y.float(), ref_y) < 1e-2


def test_gemm_rejects_bad_shapes(nat):
    A = torch.zeros(128, 100, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        nat.check(nat.lib().m3pc_gemm_bf16(A.data_ptr(), A.data_ptr(), None, A.data_ptr(), 128, 128, 100, 0, None))
    with pytest.raises(ValueError):
        nat.check(nat.lib().m3pc_gemm_bf16(A.data_ptr(), A.data_ptr(), None, A.data_ptr(), 128, 100, 64, 0, None))


@pytest.mark.parametrize("D", [512, 1024])
def test_layernorm(nat, D):
    torch.manual_seed(0)
    x, g, b = torch.randn(1000, D, device="cuda") * 3 + 1, torch.rand(D, device="cuda") + 0.5, torch.randn(D, device="cuda")
    ref = torch.nn.functional.layer_norm(x.double(), (D,), g.double(), b.double(), 1e-5)
    y = torch.empty(1000, D, device="cuda")
    nat.check(nat.lib().m3pc_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), y.data_ptr(), 1000, D, 0, None))
    y16 = torch.empty(1000, D, device="cuda", dtype=torch.bfloat16)
    nat.check(nat.lib().m3pc_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), y16.data_ptr(), 1000, D, 1, None))
    assert rel(y, ref) < 1e-5 and rel(y16, ref) < 4e-3


@pytest.mark.parametrize("B,S,H", [(5, 13, 4), (3, 32, 4), (2, 64, 8), (70, 17, 4), (1, 9, 4), (33, 10, 4), (7, 40, 4), (66, 48, 4)])
def test_attention(nat, B, S, H):
    torch.manual_seed(0)
    D = H * 128
    qkv = torch.randn(S * B, 3 * D, device="cuda")

    def ref_of(t):
        q, k, v = [u.reshape(S, B, H, 128).permute(1, 2, 0, 3).double() for u in t.split(D, dim=1)]
        return (torch.softmax(q @ k.transpose(-1, -2) / 128 ** 0.5, -1) @ v).permute(2, 0, 1, 3).reshape(S * B, D)

    out = torch.empty(S * B, D, device="cuda")
    nat.check(nat.lib().m3pc_attention(qkv.data_ptr(), out.data_ptr(), B, S, H, 0, None))
    assert rel(out, ref_of(qkv)) < 1e-5
    qkv16 = qkv.bfloat16()
    out16 = torch.empty(S * B, D, device="cuda", dtype=torch.bfloat16)
    nat.check(nat.lib().m3pc_attention(qkv16.data_ptr(), out16.data_ptr(), B, S, H, 1, None))
    assert rel(out16, ref_of(qkv16)) < 8e-3


# ------------------------------------------------------------------------------------------------ omtm.forward
def _module(shape, precision, max_batch=64, chunk=0):
    from m3pc_b200.mtm_model import omtmConfig
    cfg = omtmConfig(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer, dropout=0.1,
                     norm="none", precision=precision, max_batch=max_batch, chunk=chunk)
    m = cfg.create(shape.data_shapes, shape.traj_length, {k: False for k in shape.data_shapes})
    m.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 0).items()})
    return m.to("cuda")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_forward_matches_reference_golden(golden_dir, precision):
    """omtm.forward through the module API against outputs of the REFERENCE itself (tests/golden/forward_hopper.npz)."""
    from m3pc_b200 import masks as M
    from m3pc_b200.tokenizers import manager_from_stats
    z = np.load(os.path.join(golden_dir, "forward_hopper.npz"))
    meta = json.loads(str(z["meta"]))
    shape = syn.shipped_shape("hopper")
    m = _module(shape, precision)
    tm = manager_from_stats(syn.make_tokenizer_stats(shape, meta["stat_seed"]))
    traj = {k: torch.from_numpy(v).cuda() for k, v in syn.make_trajectories(shape, meta["batch"], meta["traj_seed"]).items()}
    enc = tm.encode(traj)
    fns = {"rcbc": M.create_rcbc_mask, "fd": M.create_fd_mask, "pi": M.create_pi_mask, "fid": M.create_fid_mask, "gid": M.create_gid_mask}
    tol = TOL[precision]
    for case in meta["cases"]:
        tag = case["tag"]
        out = m(enc, fns[case["mask"]](shape.traj_length, "cuda", case["idx"]))
        assert list(out.keys()) == ["states", "actions", "rewards", "returns"]
        for k in ("states", "rewards", "returns"):
            assert out[k].shape == z[f"{tag}/{k}"].shape
            assert rel(out[k], torch.from_numpy(z[f"{tag}/{k}"])) < tol, (tag, k)
        assert rel(out["actions"].loc, torch.from_numpy(z[f"{tag}/act_mu"])) < tol, tag
        assert rel(out["actions"].mean, torch.from_numpy(z[f"{tag}/act_mean"])) < tol, tag
        assert rel(out["actions"].std, torch.from_numpy(z[f"{tag}/act_std"])) < 3.5 * tol, tag


@pytest.mark.parametrize("env,batch", [("walker2d", 1), ("halfcheetah", 131), ("hopper", 300)])
def test_forward_fp32_vs_fp64_oracle_ragged_batches(env, batch):
    from oracle import mtm_oracle as mo, planner_oracle as po
    shape = syn.shipped_shape(env)
    m = _module(shape, "fp32", max_batch=512, chunk=128)  # 131 and 300 rows span several ragged chunks
    sd64 = mo.to_torch(syn.make_state_dict(shape, 0), torch.float64)
    traj = {k: torch.from_numpy(v) for k, v in syn.make_trajectories(shape, batch, 11).items()}
    toks = {k: v.unsqueeze(2) for k, v in traj.items()}  # forward takes tokens: feed the raw values as if tokenised
    mask = po.create_fd_mask(shape.traj_length, 3)
    ref = mo.mtm_forward(sd64, {k: v.double() for k, v in toks.items()}, {k: torch.from_numpy(v) for k, v in mask.items()},
                         shape.n_head, shape.n_enc_layer, shape.n_dec_layer)
    out = m({k: v.cuda() for k, v in toks.items()}, {k: torch.from_numpy(v).cuda() for k, v in mask.items()})
    for k in ("states", "rewards", "returns"):
        assert rel(out[k], ref[k]) < TOL["fp32"], k
    assert rel(out["actions"].loc, ref["actions"]["mu"]) < TOL["fp32"]
    assert rel(out["actions"].std, ref["actions"]["std"]) < 3.5 * TOL["fp32"]


def test_forward_scaled_model_bf16():
    """BASELINE.json config 5 shapes: D=1024, 8 heads, 4+2 layers, T=16 (64 decoder tokens)."""
    from oracle import mtm_oracle as mo, planner_oracle as po
    shape = syn.scaled_shape("hopper")
    m = _module(shape, "bf16", max_batch=16)
    traj = {k: torch.from_numpy(v) for k, v in syn.make_trajectories(shape, 9, 11).items()}
    toks = {k: v.unsqueeze(2) for k, v in traj.items()}
    mask = po.create_fd_mask(shape.traj_length, 8)
    ref = mo.mtm_forward(mo.to_torch(syn.make_state_dict(shape, 0), torch.float64), {k: v.double() for k, v in toks.items()},
                         {k: torch.from_numpy(v) for k, v in mask.items()}, shape.n_head, shape.n_enc_layer, shape.n_dec_layer)
    out = m({k: v.cuda() for k, v in toks.items()}, {k: torch.from_numpy(v).cuda() for k, v in mask.items()})
    for k in ("states", "rewards", "returns"):
        assert rel(out[k], ref[k]) < 2e-2, k  # twice the layers of the shipped model


# ------------------------------------------------------------------------------------------------ planners
def _learner(env, guidance, n_cand, temperature, precision, chunk=0, cls=None, scaled=False, **kw):
    from m3pc_b200.learner import Learner
    from m3pc_b200.mtm_model import omtmConfig
    from m3pc_b200.tokenizers import manager_from_stats
    shape = syn.scaled_shape(env) if scaled else syn.shipped_shape(env)
    cfg = SimpleNamespace(traj_length=shape.traj_length, device="cuda", action_samples=n_cand, discount=0.99, temperature=temperature,
                          horizon=4, plan_guidance=guidance, lmbda=0.6)
    mcfg = omtmConfig(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer, dropout=0.1,
                      norm="none", precision=precision, max_batch=n_cand, chunk=chunk)
    om, os_ = syn.make_obs_norm(shape)
    L = (cls or Learner)(cfg, None, shape.data_shapes, mcfg, None, om, os_, manager_from_stats(syn.make_tokenizer_stats(shape, 1)),
                         {k: False for k in shape.data_shapes}, **kw)
    L.mtm.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 0).items()})
    if hasattr(L, "iql"):
        L.iql.qf.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_critic_state_dict(shape).items()})
    return shape, L


def _inject(L, case, z, shape):
    tag, T, h = case["tag"], shape.traj_length, case["horizon"]
    eps = torch.from_numpy(z[f"{tag}/eps"])
    if not case["plan"]:
        L.injected_noise = (eps[0, T - h, 0, :].contiguous().cuda(), None)
    elif case["guidance"] == "noise_adding_lambda":
        L.injected_noise = (eps.contiguous().cuda(), torch.from_numpy(z[f"{tag}/q"]).cuda())
    else:
        L.injected_noise = (eps[:, 0, T - h:, 0, :].contiguous().cuda(), torch.from_numpy(z[f"{tag}/q"]).cuda())


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_planners_match_reference_golden(golden_dir, precision):
    """Learner.action_sample against actions the REFERENCE produced on the same inputs and the same injected noise."""
    z = np.load(os.path.join(golden_dir, "planner.npz"))
    meta = json.loads(str(z["meta"]))
    atol = 1e-4 if precision == "fp32" else 2e-2
    for case in meta["cases"]:
        shape, L = _learner(case["env"], case["guidance"], case["n_cand"], case["temperature"], precision)
        _inject(L, case, z, shape)
        hist = syn.make_history(shape, seed=case["hist_seed"], path_length=case["path_length"])
        kw = dict(percentage=case["percentage"], plan=case["plan"], rtg=case["rtg"])
        act = L.action_sample(hist, eval=case["eval"], **kw)
        ref = z[f"{case['tag']}/action"]
        assert tuple(act.shape) == ref.shape, (case["tag"], act.shape, ref.shape)
        if case["eval"] or not case["plan"] or precision == "fp32":
            np.testing.assert_allclose(act.cpu().numpy(), ref, rtol=0, atol=atol, err_msg=case["tag"])
        if f"{case['tag']}/action_other" in z.files and (precision == "fp32" or not case["eval"]):
            other = L.action_sample(hist, eval=not case["eval"], **{**kw, "rtg": 3.0 if case["rtg"] is None else case["rtg"]})
            np.testing.assert_allclose(other.cpu().numpy(), z[f"{case['tag']}/action_other"], rtol=0, atol=atol, err_msg=case["tag"] + " other")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("env,guidance,temp,N,pl", [("hopper", "rtg_guiding", 0.01, 200, 50), ("hopper", "rtg_guiding", 0.01, 77, 1),
                                                    ("walker2d", "critic_lambda_guiding", 1.0, 130, 50),
                                                    ("walker2d", "critic_lambda_guiding", 1.0, 512, 50),
                                                    ("halfcheetah", "noise_adding_lambda", 1.0, 96, 3)])
def test_plan_internals_vs_fp64_oracle(precision, env, guidance, temp, N, pl):
    """Candidates, per-candidate scores, selected indices and actions against the float64 oracle."""
    from oracle import planner_oracle as po
    shape, L = _learner(env, guidance, N, temp, precision)
    need_c = guidance != "rtg_guiding"
    P = po.from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), dtype=torch.float64,
                          critic_np=syn.make_critic_state_dict(shape) if need_c else None, obs_norm=syn.make_obs_norm(shape) if need_c else None,
                          action_samples=N, temperature=temp, plan_guidance=guidance)
    hist = syn.make_history(shape, seed=9, path_length=pl)
    T, A = shape.traj_length, shape.act_dim
    h = 4 if pl + 4 >= T else T - pl
    rs = np.random.RandomState(3)
    q = torch.from_numpy(rs.exponential(1.0, N))
    if guidance == "noise_adding_lambda":
        eps = torch.from_numpy(rs.randn(N, h, A))
        L.injected_noise = (eps.float().cuda(), q.float().cuda())
    else:
        eps = torch.from_numpy(rs.randn(N, 1, T, 1, A))
        L.injected_noise = (eps[:, 0, T - h:, 0, :].float().contiguous().cuda(), q.float().cuda())
    L.debug_plans = True
    ev = L.action_sample(hist, plan=True, eval=True, rtg=3.0)
    dbg = L.last_plan_debug
    _, ref = P.action_sample(hist, plan=True, eval=True, rtg=3.0, eps=eps, q=q)
    tol = TOL[precision]
    # candidates = tanh(mu + std * eps): the std error (3.5x amplified, see module docstring) is multiplied by |eps| <= ~4
    assert rel(dbg["candidates"], ref["candidates"]) < 3.5 * tol
    J, Jr = dbg["expect_return"].double().cpu(), ref["expect_return"]
    errJ = float((J - Jr).abs().max())
    assert errJ <= tol * max(1.0, float(Jr.abs().max()))
    assert rel(ev, ref["eval_action"]) < (1e-4 if precision == "fp32" else 2e-2)
    # the device argmax / exponential-race sample are consistent with the device scores ...
    amax, sidx = [int(v) for v in dbg["indices"].tolist()]
    assert amax == int(torch.argmax(J))
    w = torch.exp((J - J.max()) * temp)
    assert sidx == int(torch.argmax(w / q))
    # ... and bit-exact with the oracle wherever the score gap exceeds twice the score error
    top2 = torch.topk(Jr, 2).values
    if float(top2[0] - top2[1]) > 2 * errJ:
        assert amax == int(ref["argmax"])
    key = torch.exp((Jr - Jr.max()) * temp) / q
    k2 = torch.topk(key, 2).values
    if float(torch.log(k2[0]) - torch.log(k2[1])) > 2 * temp * 2 * errJ:
        assert sidx == int(ref["sample_idx"])
        assert rel(L.action_sample(hist, plan=True, eval=False, rtg=3.0)[0], ref["sample_action"][0]) < max(tol, 1e-4)


def test_plan_internals_random_sweep():
    """The same comparison over a seeded random sweep of ragged shapes: candidate counts around the tile / chunk / warp boundaries,
    every horizon the window builder can produce (path_length 0 .. 3 -> h = 8 .. 5), the episode end, all three guidances."""
    rs = np.random.RandomState(20260)
    counts = [2, 3, 31, 33, 63, 65, 127, 129, 255, 257, 300, 511]
    lengths = [0, 1, 2, 3, 4, 7, 50, 998]
    guid = [("hopper", "rtg_guiding", 0.01), ("walker2d", "critic_lambda_guiding", 1.0), ("halfcheetah", "noise_adding_lambda", 1.0),
            ("halfcheetah", "rtg_guiding", 0.01), ("hopper", "critic_lambda_guiding", 0.1)]  # temperatures of the reference's configs:
    # the eval action is a softmax average over scores of magnitude ~1e3 (1000 x return-to-go), so at temperature x |dJ| >~ 1 it
    # amplifies a 1e-3 relative score error beyond any fixed action tolerance (checked separately against the device scores in
    # tests/test_gpu_bench_sizes.py)
    for i in range(14):
        env, g, temp = guid[rs.randint(len(guid))]
        N, pl = counts[rs.randint(len(counts))], lengths[rs.randint(len(lengths))]
        precision = "fp32" if i % 4 == 3 else "bf16"
        try:
            test_plan_internals_vs_fp64_oracle(precision, env, g, temp, N, pl)
        except AssertionError as e:
            raise AssertionError(f"sweep case {i}: {precision} {env} {g} temperature={temp} N={N} path_length={pl}: {e}") from e


def test_plan_with_a_single_candidate():
    """N = 1: the softmax is trivially 1, eval action = sampled action = the only candidate."""
    shape, L = _learner("hopper", "rtg_guiding", 1, 0.01, "bf16")
    L.debug_plans = True
    hist = syn.make_history(shape, seed=2, path_length=30)
    ev = L.action_sample(hist, plan=True, eval=True, rtg=3.0)
    cand = L.last_plan_debug["candidates"]
    assert tuple(ev.shape) == (shape.act_dim,) and torch.equal(ev, cand[0, 0])
    sm = L.action_sample(hist, plan=True, eval=False, rtg=3.0)
    assert tuple(sm.shape) == (1, shape.act_dim) and torch.isfinite(sm).all()


def test_planner_method_signatures_and_shapes():
    """rtg_guiding / critic_lambda_guiding / noise_adding_lambda / mtm_sampling called directly, as the reference allows."""
    shape, L = _learner("walker2d", "critic_lambda_guiding", 64, 1.0, "bf16")
    T, A = shape.traj_length, shape.act_dim
    traj = {"states": torch.randn(1, T, shape.obs_dim, device="cuda"), "actions": torch.rand(1, T, A, device="cuda") * 2 - 1,
            "rewards": torch.randn(1, T, 1, device="cuda"), "returns": torch.full((1, T, 1), 3.0, dtype=torch.float64, device="cuda")}
    for fn, args in ((L.rtg_guiding, (traj, 4)), (L.critic_lambda_guiding, (traj, 4, 0.6)), (L.noise_adding_lambda, (traj, 4, 0.6))):
        s, e = fn(*args)
        assert s.shape == (1, A) and e.shape == (A,) and s.is_cuda and float(e.abs().max()) <= 1.0
    s, e = L.mtm_sampling(traj, 4)
    assert s.shape == (1, A) and e.shape == (1, A)
    L.cfg.plan_guidance = "bogus"
    with pytest.raises(AssertionError):
        L.action_sample(syn.make_history(shape), plan=True, eval=True, rtg=1.0)


# ------------------------------------------------------------------------------------------------ size-independent properties at BASELINE sizes
@pytest.mark.parametrize("env,guidance,temp,N", [("walker2d", "critic_lambda_guiding", 1.0, 1024), ("halfcheetah", "rtg_guiding", 0.01, 16384)])
def test_full_size_properties(env, guidance, temp, N):
    """At BASELINE.json's sizes (configs[1], configs[2]): chunk invariance, candidate-permutation equivariance, shard-count
    invariance of the merged result, and softmax sanity -- properties that do not need the (slow) oracle."""
    from m3pc_b200 import dist as mdist
    shape, L = _learner(env, guidance, N, temp, "bf16", chunk=1024)
    eng = L._engine()
    T, A, h = shape.traj_length, shape.act_dim, 4
    g = torch.Generator(device="cuda").manual_seed(0)
    ws, wa = torch.randn(T, shape.obs_dim, device="cuda", generator=g), torch.rand(T, A, device="cuda", generator=g) * 2 - 1
    wr, wt = torch.randn(T, device="cuda", generator=g), torch.full((T,), 0.7, device="cuda")
    eps, q = torch.randn(N, h, A, device="cuda", generator=g), torch.empty(N, device="cuda").exponential_(1.0, generator=g)
    common = dict(guidance=guidance, horizon=h, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt, discount=0.99,
                  temperature=temp, lmbda=0.6)

    def run(engine, eps_, q_, n, off=0, **kw):
        ev, sm, d = engine.plan(n_cand=n, eps=eps_, expq=q_, cand_offset=off, debug=True, **common, **kw)
        return ev.clone(), sm.clone(), {k: v.clone() for k, v in d.items()}

    ev, sm, d = run(eng, eps, q, N)
    J = d["expect_return"]
    assert torch.isfinite(J).all() and float(d["candidates"].abs().max()) <= 1.0  # tanh saturates to exactly 1 in fp32
    assert int(d["indices"][0]) == int(torch.argmax(J))
    w = torch.exp((J.double() - J.double().max()) * temp)
    np.testing.assert_allclose(ev.cpu().numpy(), ((w[:, None] * d["candidates"][:, 0].double()).sum(0) / w.sum()).cpu().numpy(), atol=2e-5)
    assert torch.equal(sm, d["candidates"][int(d["indices"][1]), 0])
    # permutation equivariance: permuting the noise permutes the scores
    perm = torch.randperm(N, device="cuda", generator=g)
    ev_p, _, d_p = run(eng, eps[perm].contiguous(), q[perm].contiguous(), N)
    assert torch.equal(d_p["expect_return"], J[perm])
    np.testing.assert_allclose(ev_p.cpu().numpy(), ev.cpu().numpy(), atol=2e-5)
    assert int(perm[int(d_p["indices"][0])]) == int(d["indices"][0])
    # shard-count invariance: 4 shards + merge == one call
    recs = []
    for r in range(4):
        lo, hi = mdist.shard_range(N, r, 4)
        _, _, ds = run(eng, eps[lo:hi].contiguous(), q[lo:hi].contiguous(), hi - lo, off=lo)
        assert torch.equal(ds["expect_return"], J[lo:hi])
        recs.append(ds["partials"])
    ev_m, sm_m, idx_m = eng.merge_partials(torch.stack(recs), temp)
    np.testing.assert_allclose(ev_m.cpu().numpy(), ev.cpu().numpy(), atol=2e-5)
    assert torch.equal(sm_m, sm) and idx_m.tolist() == d["indices"].tolist()
    hev, hsm, hamax, hsidx = mdist.merge_partials_host(torch.stack(recs).cpu().numpy(), A, temp)
    np.testing.assert_allclose(hev, ev.cpu().numpy(), atol=2e-5)
    assert [hamax, hsidx] == d["indices"].tolist()
    # chunk invariance: a different L2 blocking gives bit-identical scores
    _, L2 = _learner(env, guidance, N, temp, "bf16", chunk=256)
    _, _, d2 = run(L2._engine(), eps, q, N)
    assert torch.equal(d2["expect_return"], J)


def test_philox_noise_is_shard_invariant_and_seeded():
    shape, L = _learner("hopper", "rtg_guiding", 512, 0.01, "bf16")
    eng = L._engine()
    T, A, h = shape.traj_length, shape.act_dim, 4
    ws, wa, wr, wt = torch.randn(T, shape.obs_dim, device="cuda"), torch.rand(T, A, device="cuda"), torch.randn(T, device="cuda"), torch.ones(T, device="cuda")
    common = dict(guidance="rtg_guiding", horizon=h, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt, discount=0.99,
                  temperature=0.01, lmbda=0.6, debug=True)
    _, _, d = eng.plan(n_cand=512, seed=5, **common)
    c = d["candidates"].clone()
    assert float(c.abs().max()) <= 1.0 and float(c.std()) > 0.01
    _, _, d1 = eng.plan(n_cand=256, seed=5, cand_offset=256, **common)
    assert torch.equal(d1["candidates"], c[256:])          # noise is a function of the GLOBAL candidate id
    _, _, d2 = eng.plan(n_cand=512, seed=6, **common)
    assert not torch.equal(d2["candidates"], c)
    z = torch.atanh(c.double().clamp(-0.999999, 0.999999))   # tanh^-1 recovers mu + std * eps: check eps ~ N(0,1) per (t, a)
    zs = (z - z.mean(0)) / z.std(0)
    assert abs(float(zs.mean())) < 0.05 and abs(float((zs ** 2).mean()) - 1.0) < 0.05 and abs(float((zs ** 3).mean())) < 0.3


# ------------------------------------------------------------------------------------------------ deeper decoders
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_plan_scaled_model_last_decoder_layer_restricted(precision, monkeypatch):
    """BASELINE.json config 5 (D=1024, 8 heads, 4+2 layers, T=16, h=8): with more than one decoder layer only the LAST layer
    is restricted to the consumed rows.  Checked against the float64 oracle (which computes every row of every layer) and
    against the same engine with the restriction switched off (m3pc_set_option "restrict_deep_decoder" 0)."""
    from oracle import planner_oracle as po
    N, temp = 24, 0.01
    shape, L = _learner("hopper", "rtg_guiding", N, temp, precision, scaled=True)
    L.cfg.horizon = 8
    T, A, h = shape.traj_length, shape.act_dim, 8
    hist = syn.make_history(shape, seed=9, path_length=50)
    rs = np.random.RandomState(3)
    eps, q = torch.from_numpy(rs.randn(N, 1, T, 1, A)), torch.from_numpy(rs.exponential(1.0, N))
    noise = (eps[:, 0, T - h:, 0, :].float().contiguous().cuda(), q.float().cuda())
    L.injected_noise, L.debug_plans = noise, True
    ev = L.action_sample(hist, plan=True, eval=True, rtg=3.0).clone()
    J = L.last_plan_debug["expect_return"].double().cpu()
    assert L.mtm.sync_engine().last_launch_count() > 0
    P = po.from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), dtype=torch.float64, action_samples=N,
                          temperature=temp, plan_guidance="rtg_guiding", horizon=8)
    _, ref = P.action_sample(hist, plan=True, eval=True, rtg=3.0, eps=eps, q=q)
    tol = 2 * TOL[precision]  # twice the layers of the shipped model
    assert float((J - ref["expect_return"]).abs().max()) <= tol * max(1.0, float(ref["expect_return"].abs().max()))
    assert rel(ev, ref["eval_action"]) < (2e-4 if precision == "fp32" else 4e-2)
    n_restricted = L.mtm.sync_engine().last_launch_count()
    from m3pc_b200.engine import PlanEngine
    monkeypatch.setitem(PlanEngine.default_options, "restrict_deep_decoder", 0)
    _, Lf = _learner("hopper", "rtg_guiding", N, temp, precision, scaled=True)
    Lf.cfg.horizon = 8
    Lf.injected_noise, Lf.debug_plans = noise, True
    Lf.action_sample(hist, plan=True, eval=True, rtg=3.0)
    Jf = Lf.last_plan_debug["expect_return"].double().cpu()
    assert Lf.mtm.sync_engine().last_launch_count() != n_restricted  # the switch really selects the other path
    assert float((J - Jf).abs().max()) <= (1e-4 if precision == "fp32" else TOL["bf16"]) * max(1.0, float(Jf.abs().max()))


# ------------------------------------------------------------------------------------------------ E lock-step environments per plan
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("env,guidance,temp,N,E,chunk", [("walker2d", "critic_lambda_guiding", 1.0, 96, 5, 0), ("hopper", "rtg_guiding", 0.01, 130, 3, 128),
                                                         ("halfcheetah", "noise_adding_lambda", 1.0, 64, 4, 100)])
def test_env_batched_plan_rows_equal_single_env_plans(precision, env, guidance, temp, N, E, chunk):
    """m3pc_plan with n_env = E (SURVEY.md section 8f rank 1): row e of every output equals the single-window plan on window e
    with the same injected noise.  Pass 2 is row-independent and bit-identical; pass 1 runs at B = E instead of B = 1 (tensor-core
    tiles instead of the fused B = 1 kernel), so the candidates differ by bf16 rounding of mu / std.  chunk values that do not
    divide N make a chunk straddle two environments."""
    shape, L = _learner(env, guidance, N, temp, precision, chunk=chunk, max_envs=E)
    T, A, h = shape.traj_length, shape.act_dim, 4
    hists = [syn.make_history(shape, seed=30 + e, path_length=50 + 3 * e) for e in range(E)]
    g = torch.Generator(device="cuda").manual_seed(1)
    eps = torch.randn(E * N, h, A, device="cuda", generator=g)
    q = torch.empty(E * N, device="cuda").exponential_(1.0, generator=g)
    L.debug_plans = True
    L.injected_noise = (eps, q)
    rtgs = [2.0 + 0.25 * e for e in range(E)]
    ev_b = L.action_sample_batch(hists, plan=True, eval=True, rtg=rtgs).clone()
    db = L.last_plan_debug
    sm_b = L.action_sample_batch(hists, plan=True, eval=False, rtg=rtgs).clone()
    assert ev_b.shape == (E, A) and sm_b.shape == (E, A)
    assert db["expect_return"].shape == (E * N,) and db["candidates"].shape == (E * N, h, A) and db["indices"].shape == (E, 2)
    tol = TOL[precision]
    for e in range(E):
        L.injected_noise = (eps[e * N:(e + 1) * N].contiguous(), q[e * N:(e + 1) * N].contiguous())
        ev = L.action_sample(hists[e], plan=True, eval=True, rtg=rtgs[e])
        d = L.last_plan_debug
        Jb, Js = db["expect_return"][e * N:(e + 1) * N].double(), d["expect_return"].double()
        assert rel(db["candidates"][e * N:(e + 1) * N], d["candidates"]) < 3.5 * tol
        errJ = float((Jb - Js).abs().max())
        assert errJ <= tol * max(1.0, float(Js.abs().max()))
        assert rel(ev_b[e], ev) < (1e-4 if precision == "fp32" else 2e-2)
        # selection inside the batched call is consistent with its own scores, per environment
        amax, sidx = [int(v) for v in db["indices"][e].tolist()]
        assert amax == int(torch.argmax(Jb))
        w = torch.exp((Jb - Jb.max()) * temp)
        assert sidx == int(torch.argmax(w / q[e * N:(e + 1) * N].double()))
        assert torch.equal(sm_b[e], db["candidates"][e * N + sidx, 0])
        top2 = torch.topk(Js, 2).values
        if float(top2[0] - top2[1]) > 2 * errJ:
            assert amax == int(d["indices"][0])
    # mtm_sampling (plan=False) on E windows
    eps_s = torch.randn(E, A, device="cuda", generator=g)
    L.injected_noise = (eps_s, None)
    sm_all = L.action_sample_batch(hists, plan=False, eval=False, rtg=rtgs).clone()
    assert sm_all.shape == (E, A)
    for e in (0, E - 1):
        L.injected_noise = (eps_s[e].contiguous(), None)
        single = L.action_sample(hists[e], plan=False, eval=False, rtg=rtgs[e])
        np.testing.assert_allclose(single[0].cpu().numpy(), sm_all[e].cpu().numpy(), atol=1e-4 if precision == "fp32" else 3e-2)


def test_env_batched_plan_philox_and_graph_replay():
    """Production path of the batched plan: on-device Philox noise, CUDA-graph replay; environments draw different noise,
    identical windows with identical seeds reproduce, and E * n_cand above the engine capacity is rejected."""
    E, N = 4, 256
    shape, L = _learner("walker2d", "critic_lambda_guiding", N, 1.0, "bf16", max_envs=E)
    hist = syn.make_history(shape, seed=5, path_length=60)
    L._engine()  # binds the engine (and resets the plan counter) before the seeds are pinned below
    outs = []
    for _ in range(4):  # eager, capture, replay, replay
        L.__dict__["_plan_counter"] = 7
        outs.append(L.action_sample_batch([hist] * E, plan=True, eval=False, rtg=3.0).clone())
    assert torch.isfinite(outs[0]).all() and float(outs[0].abs().max()) <= 1.0
    for o in outs[1:]:
        assert torch.equal(o, outs[0])            # same seed -> same draw, eager == replayed graph
    assert not torch.equal(outs[0][0], outs[0][1])  # same window, different environment -> different noise stream
    ev = L.action_sample_batch([hist] * E, plan=True, eval=True, rtg=3.0)
    assert float((ev - ev[0:1]).abs().max()) < 0.25  # softmax-weighted means of 256 draws from the same distribution agree loosely
    with pytest.raises(ValueError):
        L.action_sample_batch([hist] * (E + 1), plan=True, eval=True, rtg=3.0)


# ------------------------------------------------------------------------------------------------ checkpoints in the reference's formats
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_plan_from_reference_format_checkpoints(golden_dir, precision):
    """mtm_<step>.pt + iql_<step>.pt + d4rl_statistics_*.pkl written by the reference's classes (tests/golden/ckpt) ->
    m3pc_b200.checkpoint.build_learner -> plan on the GPU == the float64 oracle fed the same tensors.  Also exercises a
    non-shipped geometry (D=128, one head, T=4, obs 3 / act 2)."""
    from m3pc_b200 import checkpoint as ck
    from m3pc_b200.mtm_model import omtmConfig
    from oracle import planner_oracle as po
    d = os.path.join(golden_dir, "ckpt")
    N, T, h = 48, 4, 2
    cfg = SimpleNamespace(traj_length=T, device="cuda", action_samples=N, discount=0.99, temperature=1.0, horizon=h,
                          plan_guidance="critic_lambda_guiding", lmbda=0.6)
    mcfg = omtmConfig(n_embd=128, n_head=1, n_enc_layer=1, n_dec_layer=1, dropout=0.1, norm="none", precision=precision, max_batch=N)
    L = ck.build_learner(cfg, mcfg, os.path.join(d, "mtm_7.pt"), os.path.join(d, "d4rl_statistics_tiny.pkl"), iql_path=os.path.join(d, "iql_7.pt"))
    stats = ck.load_trajectory_statistics(os.path.join(d, "d4rl_statistics_tiny.pkl"))
    tm = ck.tokenizer_manager_from_statistics(stats)
    stats_np = {k: {"mean": tm.tokenizers[k]._data_mean.numpy(), "std": tm.tokenizers[k]._data_std.numpy(), "min": stats[k].min, "max": stats[k].max}
                for k in stats}
    shape = syn.ModelShape(obs_dim=3, act_dim=2, n_embd=128, n_head=1, n_enc_layer=1, n_dec_layer=1, traj_length=T)
    P = po.from_synthetic(shape, {k: v.numpy() for k, v in ck.load_mtm_checkpoint(os.path.join(d, "mtm_7.pt")).items()}, stats_np, dtype=torch.float64,
                          critic_np={k: v.numpy() for k, v in ck.load_iql_checkpoint(os.path.join(d, "iql_7.pt")).items()},
                          obs_norm=(stats["states"].mean, stats["states"].std), action_samples=N, temperature=1.0,
                          plan_guidance="critic_lambda_guiding", horizon=h)
    hist = syn.make_history(shape, seed=3, path_length=20)
    rs = np.random.RandomState(5)
    eps, q = torch.from_numpy(rs.randn(N, 1, T, 1, 2)), torch.from_numpy(rs.exponential(1.0, N))
    L.injected_noise = (eps[:, 0, T - h:, 0, :].float().contiguous().cuda(), q.float().cuda())
    L.debug_plans = True
    ev = L.action_sample(hist, plan=True, eval=True, rtg=1.5)
    _, ref = P.action_sample(hist, plan=True, eval=True, rtg=1.5, eps=eps, q=q)
    tol = TOL[precision]
    J, Jr = L.last_plan_debug["expect_return"].double().cpu(), ref["expect_return"]
    assert float((J - Jr).abs().max()) <= tol * max(1.0, float(Jr.abs().max()))
    assert rel(L.last_plan_debug["candidates"], ref["candidates"]) < 3.5 * tol
    assert rel(ev, ref["eval_action"]) < (1e-4 if precision == "fp32" else 2e-2)


# ------------------------------------------------------------------------------------------------ zero-shot backward planners
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_zeroshot_matches_reference_golden(golden_dir, precision):
    from m3pc_b200.zeroshot_learner import Learner as ZLearner
    z = np.load(os.path.join(golden_dir, "zeroshot_hopper.npz"))
    meta = json.loads(str(z["meta"]))
    shape, L = _learner("hopper", "rtg_guiding", 1, 0.01, precision, cls=ZLearner, max_envs=8)
    atol = 1e-4 if precision == "fp32" else 2e-2
    T = shape.traj_length
    for case in meta["cases"]:
        tag = case["tag"]
        hist = syn.make_history(shape, seed=case["hist_seed"], path_length=case["path_length"])
        h = L._clamped_horizon(hist)
        L.injected_eps = torch.from_numpy(z[f"{tag}/eps"])[0, T - h, 0, :].reshape(1, -1).contiguous().cuda()
        fn = getattr(L, case["fn"])
        np.testing.assert_allclose(fn(hist, eval=True, rtg=case["rtg"]).cpu().numpy(), z[f"{tag}/eval_action"], atol=atol, err_msg=tag)
        np.testing.assert_allclose(fn(hist, eval=False, rtg=case["rtg"]).cpu().numpy(), z[f"{tag}/sample_action"], atol=atol, err_msg=tag)
    L.action_piid_list_sample(syn.make_history(shape, seed=4, path_length=50), eval=True, rtg=2.5)
    np.testing.assert_allclose(L.action_list[0].cpu().numpy(), z["piid_pl50/eval_action"], atol=atol)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_zeroshot_batch_rows_equal_single_env_calls(precision):
    """Config-4 extension: E lock-step environments in one call; row e == the B=1 call on history e.  (Not bit-exact: B=1 runs
    the skinny CUDA-core GEMM, E=37 the tcgen05 tiles -- different fp32 summation orders, re-rounded to bf16 between layers.)"""
    from m3pc_b200.zeroshot_learner import Learner as ZLearner
    shape, L = _learner("hopper", "rtg_guiding", 1, 0.01, precision, cls=ZLearner, max_envs=37)
    hists = [syn.make_history(shape, seed=20 + e, path_length=40 + e) for e in range(37)]
    batch = L.action_piid_sample_batch(hists, eval=True, rtg=2.0).clone()
    assert batch.shape == (37, shape.act_dim)
    for e in (0, 5, 36):
        single = L.action_piid_sample(hists[e], eval=True, rtg=2.0)
        np.testing.assert_allclose(single[0].cpu().numpy(), batch[e].cpu().numpy(), atol=1e-5 if precision == "fp32" else 1e-2)
    ids = L.action_id_sample_batch(hists, eval=True, rtg=2.0)
    assert ids.shape == (37, shape.act_dim) and torch.isfinite(ids).all()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_zeroshot_candidate_draws_per_environment(precision):
    """BASELINE.json config 4 shape (E environments x C candidate actions): every draw is tanh(mu_e + std_e * eps[e, c]) of the
    distribution the single-draw planner samples from; draw c of environment e with injected noise == the reference-shaped
    single call with that noise; Philox draws differ across environments / draws and follow the distribution."""
    from m3pc_b200.zeroshot_learner import Learner as ZLearner
    E, C = 9, 64
    shape, L = _learner("hopper", "rtg_guiding", 1, 0.01, precision, cls=ZLearner, max_envs=E)
    A = shape.act_dim
    hists = [syn.make_history(shape, seed=60 + e, path_length=45 + e) for e in range(E)]
    g = torch.Generator(device="cuda").manual_seed(2)
    eps = torch.randn(E, C, A, device="cuda", generator=g)
    L.injected_eps = eps
    ev, draws = L.action_piid_draws_batch(hists, C, rtg=2.0)
    assert ev.shape == (E, A) and draws.shape == (E, C, A) and float(draws.abs().max()) <= 1.0
    for e, c in ((0, 0), (4, 17), (8, 63)):
        L.injected_eps = eps[:, c, :].contiguous()
        one = L.action_piid_sample_batch(hists, eval=False, rtg=2.0)
        assert torch.equal(one[e], draws[e, c])
    L.injected_eps = eps[:, 0, :].contiguous()
    assert torch.equal(L.action_piid_sample_batch(hists, eval=True, rtg=2.0), ev)
    # on-device noise: atanh(draw) = mu + std * z with z ~ N(0, 1) per (environment, draw)
    L.injected_eps = None
    ev2, d2 = L.action_piid_draws_batch(hists, 4096, rtg=2.0)
    assert torch.equal(ev2, ev)
    z = torch.atanh(d2.double().clamp(-0.9999999, 0.9999999))
    zs = (z - z.mean(1, keepdim=True)) / z.std(1, keepdim=True)
    assert abs(float((zs ** 3).mean())) < 0.1 and abs(float((zs ** 4).mean()) - 3.0) < 0.3
    np.testing.assert_allclose(torch.tanh(z.mean(1)).cpu().numpy(), ev.double().cpu().numpy(), atol=0.05)
    assert not torch.equal(d2[0, 0], d2[0, 1]) and not torch.equal(d2[0, 0], d2[1, 0])
    _, d3 = L.action_piid_draws_batch(hists, 4096, rtg=2.0)
    assert not torch.equal(d3, d2)  # the plan counter advances the Philox key


def test_plan_with_fused_residual_layernorm_forced_at_small_shapes(monkeypatch):
    """The engine uses the fused residual GEMM + LayerNorm kernel from 1024 rows up; option "fused_ln_min_rows" = 129 forces it at
    test sizes so the oracle comparison covers its wiring (out-projection + norm2, linear2 + next norm1 / final encoder norm,
    the table-residual form of the shared-history block, the restricted decoder layer)."""
    from m3pc_b200.engine import PlanEngine
    monkeypatch.setitem(PlanEngine.default_options, "fused_ln_min_rows", 129)
    test_plan_internals_vs_fp64_oracle("bf16", "walker2d", "critic_lambda_guiding", 1.0, 130, 50)
    test_plan_internals_vs_fp64_oracle("bf16", "hopper", "rtg_guiding", 0.01, 200, 50)
    test_env_batched_plan_rows_equal_single_env_plans("bf16", "walker2d", "critic_lambda_guiding", 1.0, 96, 5, 0)


def test_plan_graphs_are_dropped_when_parameters_change(monkeypatch):
    """A captured plan graph has the weight / tokenizer / critic arena addresses and the scalar statistics baked into its
    kernel nodes.  Replaying it after ``load_state_dict`` / ``mark_dirty`` (INTEGRATION.md: after every optimiser step) must
    use the NEW parameters: m3pc_set_param / m3pc_finalize_params drop the graphs.  Checked against an engine that never
    captures (option "graphs" = 0) loaded with the same new parameters."""
    from m3pc_b200.engine import PlanEngine
    from m3pc_b200.tokenizers import manager_from_stats
    shape, L = _learner("walker2d", "critic_lambda_guiding", 256, 1.0, "bf16")
    hist = syn.make_history(shape, seed=4, path_length=80)
    L.seed = 3

    def run(Lx):
        Lx.__dict__["_plan_counter"] = 0  # same Philox key every call
        return Lx.action_sample(hist, plan=True, eval=True, rtg=3.0).double().cpu()

    a = [run(L) for _ in range(4)]  # eager, capture + replay, replay, replay
    np.testing.assert_allclose(a[3].numpy(), a[0].numpy(), atol=1e-6)
    # new weights (a different arena content, same size), new tokenizer statistics, new critic, then an in-place update
    sd2 = {k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 5).items()}
    L.mtm.load_state_dict(sd2)
    L.tokenizer_manager = manager_from_stats(syn.make_tokenizer_stats(shape, 9))
    L.__dict__["_planner_bound"] = None  # re-bind the new tokenizer manager
    with torch.no_grad():
        for p in L.iql.qf.parameters():
            p.mul_(0.5)
    b = [run(L) for _ in range(3)]
    with torch.no_grad():
        L.mtm.encoder.layers[0].linear1.weight.mul_(1.25)
        L.mtm.output_head_dict["rewards"][3].bias.add_(0.3)
    L.mtm.mark_dirty()
    c = [run(L) for _ in range(3)]
    monkeypatch.setitem(PlanEngine.default_options, "graphs", 0)
    _, R = _learner("walker2d", "critic_lambda_guiding", 256, 1.0, "bf16")
    R.seed = 3
    R.mtm.load_state_dict(sd2)
    R.tokenizer_manager = manager_from_stats(syn.make_tokenizer_stats(shape, 9))
    with torch.no_grad():
        for p in R.iql.qf.parameters():
            p.mul_(0.5)
    rb = run(R)
    with torch.no_grad():
        R.mtm.encoder.layers[0].linear1.weight.mul_(1.25)
        R.mtm.output_head_dict["rewards"][3].bias.add_(0.3)
    R.mtm.mark_dirty()
    rc = run(R)
    assert float((a[0] - rb).abs().max()) > 1e-3 and float((rb - rc).abs().max()) > 1e-5  # the updates really change the plan
    for x in b:
        np.testing.assert_allclose(x.numpy(), rb.numpy(), atol=1e-6)
    for x in c:
        np.testing.assert_allclose(x.numpy(), rc.numpy(), atol=1e-6)


def test_select_survives_non_finite_scores():
    """NaN scores must not turn into an out-of-bounds read (which would poison the CUDA context): the plan returns NaN actions
    and candidate index 0, and the next plan on the same handle works."""
    shape, L = _learner("hopper", "rtg_guiding", 128, 0.01, "bf16")
    hist = syn.make_history(shape, seed=4, path_length=80)
    good = L.action_sample(hist, plan=True, eval=True, rtg=3.0).clone()
    bad_hist = dict(hist, observations=hist["observations"].copy())
    bad_hist["observations"][:] = np.nan
    L.debug_plans = True
    ev = L.action_sample(bad_hist, plan=True, eval=True, rtg=3.0)
    sm = L.action_sample(bad_hist, plan=True, eval=False, rtg=3.0)
    torch.cuda.synchronize()
    assert bool(torch.isnan(ev).all()) and bool(torch.isnan(sm).all())
    assert L.last_plan_debug["indices"].tolist() == [0, 0]
    L.debug_plans = False
    again = L.action_sample(hist, plan=True, eval=True, rtg=3.0)
    assert bool(torch.isfinite(again).all()) and again.shape == good.shape


@pytest.mark.parametrize("world", [2, 4])
def test_peer_exchange_in_the_select_kernel_matches_one_call(world, monkeypatch):
    """Candidate sharding with the production transport: `world` engines (one per shard, here in ONE process on one GPU, each on
    its own stream; peers wired by device pointer) plan their shards with exchange = 1 -- selection, all-gather of the records
    over peer memory and the merge happen inside each shard's select kernel.  Every shard must return the result of the
    unsharded call, for several consecutive plans (epoch / slot alternation) and through CUDA-graph replay."""
    from m3pc_b200 import dist as mdist
    from m3pc_b200.engine import PlanEngine
    # Several ranks share ONE GPU here: a rank's select kernel spins until its peers' records arrive, and a peer's COOPERATIVE
    # B = 1 kernel (one CTA on every SM, all co-resident) could not start next to that spinning block.  With one GPU per rank
    # (the real deployment, tools/multigpu_check.sh) this cannot happen; here pass 1 uses the per-op launches instead.
    monkeypatch.setitem(PlanEngine.default_options, "fused_b1", 0)
    N, temp, guidance = 1024, 0.01, "rtg_guiding"
    shape, L0 = _learner("halfcheetah", guidance, N, temp, "bf16")
    full = L0._engine()
    T, A, h = shape.traj_length, shape.act_dim, 4
    shards = []
    for r in range(world):
        _, Lr = _learner("halfcheetah", guidance, N // world + 1, temp, "bf16")
        shards.append(Lr._engine())
    ptrs = [e.exchange_local()[1] for e in shards]
    for r, e in enumerate(shards):
        e.exchange_connect(r, world, device_ptrs=ptrs)
    streams = [torch.cuda.Stream() for _ in range(world)]
    g = torch.Generator(device="cuda").manual_seed(0)
    # persistent window buffers: a plan's CUDA graph is keyed on their addresses
    ws, wa = torch.empty(T, shape.obs_dim, device="cuda"), torch.empty(T, A, device="cuda")
    wr, wt = torch.empty(T, device="cuda"), torch.full((T,), 0.7, device="cuda")
    for it in range(6):
        ws.copy_(torch.randn(T, shape.obs_dim, device="cuda", generator=g))
        wa.copy_(torch.rand(T, A, device="cuda", generator=g) * 2 - 1)
        wr.copy_(torch.randn(T, device="cuda", generator=g))
        common = dict(guidance=guidance, horizon=h, win_states=ws, win_actions=wa, win_rewards=wr, win_returns_tok=wt, discount=0.99,
                      temperature=temp, lmbda=0.6, seed=77 + it)
        inject = it < 2  # eager with injected noise first, then Philox through the graph path
        if inject:
            eps, q = torch.randn(N, h, A, device="cuda", generator=g), torch.empty(N, device="cuda").exponential_(1.0, generator=g)
        ev, sm, d = full.plan(n_cand=N, eps=eps if inject else None, expq=q if inject else None, debug=inject, **common)
        ev, sm = ev.clone(), sm.clone()
        torch.cuda.synchronize()
        outs = []
        for r, e in enumerate(shards):
            lo, hi = mdist.shard_range(N, r, world)
            with torch.cuda.stream(streams[r]):
                e_ev, e_sm, e_d = e.plan(n_cand=hi - lo, cand_offset=lo, eps=eps[lo:hi].contiguous() if inject else None,
                                         expq=q[lo:hi].contiguous() if inject else None, debug=inject, exchange=True, **common)
                outs.append((e_ev.clone(), e_sm.clone(), e_d["indices"].clone() if inject else None))
        torch.cuda.synchronize()
        for r, (e_ev, e_sm, e_idx) in enumerate(outs):
            np.testing.assert_allclose(e_ev.cpu().numpy(), ev.cpu().numpy(), atol=2e-5, err_msg=f"plan {it} rank {r}")
            assert torch.equal(e_sm, sm), (it, r)
            if inject:
                assert e_idx.tolist() == d["indices"].tolist()
    for e in shards:
        assert e.exchange_status() == (6, 0)


@pytest.mark.parametrize("M,K,table_rows", [(26624, 512, 0), (26624, 2048, 0), (4000, 512, 1000), (777, 2048, 0)])
def test_gemm_ln_unit_sizes_are_bit_identical(nat, M, K, table_rows):
    """The fused residual GEMM + LayerNorm kernel picks 128- or 256-row units per launch (from K and the row count); scores must not
    depend on that choice -- candidate shards of different sizes have to reproduce the unsharded plan bit for bit -- so both unit
    sizes are required to give identical X and Y."""
    from m3pc_b200.engine import engine_from_synthetic
    shape = syn.shipped_shape("hopper")
    eng = engine_from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), max_batch=8)  # a handle for m3pc_set_option
    L = nat.lib()
    g = torch.Generator(device="cuda").manual_seed(M + K)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    W = (torch.randn(512, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
    bias, gamma, beta = torch.randn(512, device="cuda", generator=g), 1 + 0.2 * torch.randn(512, device="cuda", generator=g), 0.2 * torch.randn(512, device="cuda", generator=g)
    X0 = 2.0 * torch.randn(M, 512, device="cuda", generator=g) + 0.5
    table, grp = None, 1
    if table_rows:
        grp = table_rows
        table = torch.randn((M + grp - 1) // grp, 512, device="cuda", generator=g)
    outs = {}
    try:
        for rows in (128, 256, 0):
            eng.set_option("gemm_ln_unit_rows", rows)
            X, Y = X0.clone(), torch.full((M, 512), float("nan"), device="cuda", dtype=torch.bfloat16)
            nat.check(L.m3pc_gemm_ln_bf16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), X.data_ptr(), Y.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                          table.data_ptr() if table is not None else None, grp, M, K, None), "m3pc_gemm_ln_bf16")
            torch.cuda.synchronize()
            outs[rows] = (X, Y)
    finally:
        eng.set_option("gemm_ln_unit_rows", 0)
    assert torch.equal(outs[128][0], outs[256][0]) and torch.equal(outs[128][1], outs[256][1])
    assert torch.equal(outs[0][0], outs[256][0]) and torch.equal(outs[0][1], outs[256][1])
