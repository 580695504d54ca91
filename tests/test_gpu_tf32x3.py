"""The fp32-grade tensor-core precision mode (M3PC_PREC_TF32X3, precision="tf32x3"): the 3xTF32 split GEMM on its own
(m3pc_gemm_tf32x3) and the whole engine in that mode, held to the bars of the fp32 mode.

Tolerances
  kernel   -- max |C - C64| <= 1e-5 * max(1, max |C64|) against the float64 product, and no more than twice the error of
              m3pc_gemm_fp32 (IEEE fp32 FFMA) on the same inputs.
  forward  -- 1e-5 against the float64 oracle (3e-5 on the action std, whose pre-activation error exp(3.5 tanh(.)) amplifies).
  planners -- the fp32 mode's: actions to 1e-4, scores to 2e-5 relative, indices exact wherever the score gap exceeds twice the
              measured score error.
"""
import ctypes as C
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from m3pc_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

SMALL_ROWS = 128  # gemm_tf32x3.cu kTf32x3SmallRows: problems of at most this many rows run on the CUDA-core fp32 kernel
ORDER = ("states", "actions", "rewards", "returns")


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(1.0, float(b.abs().max())))


@pytest.fixture(scope="module")
def nat():
    from m3pc_b200 import _native
    _native.lib()
    return _native


def _gemm(nat, fn, A, W, b, C0, flags):
    Cm = C0.clone()
    M, K = A.shape
    N = W.shape[0]
    nat.check(getattr(nat.lib(), fn)(A.data_ptr(), W.data_ptr(), b.data_ptr() if b is not None else None, Cm.data_ptr(), M, N, K, flags, None))
    torch.cuda.synchronize()
    return Cm


def _inputs(M, N, K, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    C0 = torch.randn(M, N, device="cuda", generator=g)
    return A, W, b, C0


def _ref(A, W, b, C0, flags):
    ref = A.double() @ W.double().T
    if b is not None:
        ref += b.double()
    if flags & 1:
        ref = torch.nn.functional.gelu(ref)
    if flags & 4:
        ref = torch.relu(ref)
    if flags & 2:
        ref += C0.double()
    return ref


# ------------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("M,N,K,flags", [
    (1, 512, 512, 0), (17, 1536, 2048, 1), (17, 256, 512, 6),                    # small problems (CUDA-core kernel)
    (129, 2048, 512, 2), (129, 256, 2048, 4), (129, 512, 512, 5),                # one row pair, mostly empty
    (4097, 512, 2048, 2), (4097, 1536, 512, 1), (4097, 256, 512, 3), (4097, 2048, 2048, 6),
    (106496, 1536, 512, 0), (106496, 512, 512, 2), (106496, 2048, 512, 1), (106496, 512, 2048, 2),  # the pass-2 GEMMs of a step
    (106496 - 77, 256, 2048, 4),
])
def test_gemm_tf32x3_vs_fp64(nat, M, N, K, flags):
    A, W, b, C0 = _inputs(M, N, K)
    ref = _ref(A, W, b, C0, flags)
    err = rel(_gemm(nat, "m3pc_gemm_tf32x3", A, W, b, C0, flags), ref)
    err32 = rel(_gemm(nat, "m3pc_gemm_fp32", A, W, b, C0, flags), ref)
    assert err <= 1e-5 and err <= 2 * err32, (err, err32)


def test_gemm_tf32x3_without_bias(nat):
    A, W, _, C0 = _inputs(1000, 512, 512, seed=3)
    ref = _ref(A, W, None, C0, 0)
    assert rel(_gemm(nat, "m3pc_gemm_tf32x3", A, W, None, C0, 0), ref) <= 1e-5


def test_gemm_tf32x3_small_row_threshold(nat):
    """At most SMALL_ROWS rows (and shapes the TMA / CTA-pair tiles cannot take: N not a multiple of 256, K not a multiple of 4)
    run the CUDA-core fp32 kernel, so the result is m3pc_gemm_fp32's bit for bit; one row more runs the tensor-core kernel."""
    for M, N, K in ((SMALL_ROWS, 512, 512), (1, 2048, 2048), (1000, 384, 512), (1000, 512, 23)):
        A, W, b, C0 = _inputs(M, N, K, seed=M + N + K)
        assert torch.equal(_gemm(nat, "m3pc_gemm_tf32x3", A, W, b, C0, 1), _gemm(nat, "m3pc_gemm_fp32", A, W, b, C0, 1)), (M, N, K)
    A, W, b, C0 = _inputs(SMALL_ROWS + 1, 512, 512, seed=5)
    tf, fp = _gemm(nat, "m3pc_gemm_tf32x3", A, W, b, C0, 1), _gemm(nat, "m3pc_gemm_fp32", A, W, b, C0, 1)
    assert not torch.equal(tf, fp)  # a different summation: the tensor-core kernel ran
    ref = _ref(A, W, b, C0, 1)
    assert rel(tf, ref) <= 1e-5 and rel(tf, ref) <= 2 * rel(fp, ref)


def test_gemm_tf32x3_is_deterministic(nat):
    A, W, b, C0 = _inputs(4097, 1536, 512, seed=9)
    assert torch.equal(_gemm(nat, "m3pc_gemm_tf32x3", A, W, b, C0, 2), _gemm(nat, "m3pc_gemm_tf32x3", A, W, b, C0, 2))


def test_gemm_tf32x3_rejects_bad_arguments(nat):
    A, W, b, C0 = _inputs(256, 256, 64)
    with pytest.raises(ValueError):
        nat.check(nat.lib().m3pc_gemm_tf32x3(A.data_ptr(), W.data_ptr(), b.data_ptr(), C0.data_ptr(), 256, 256, 64, 8, None))
    with pytest.raises(ValueError):
        nat.check(nat.lib().m3pc_gemm_tf32x3(A.data_ptr() + 4, W.data_ptr(), b.data_ptr(), C0.data_ptr(), 255, 256, 64, 0, None))


def test_row_table_epilogue_decoder_embed(nat):
    """The row-table epilogue (decoder embedding: per-token table row + GEMM, K4 m3pc_decoder_scatter_embed) against the oracle."""
    from m3pc_b200.engine import engine_from_synthetic
    from oracle import mtm_oracle as mo, planner_oracle as po
    shape = syn.shipped_shape("hopper")
    B = 200
    eng = engine_from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), precision="tf32x3", max_batch=256)
    sd = mo.to_torch(syn.make_state_dict(shape, 0), torch.float64)
    traj = {k: torch.from_numpy(v) for k, v in syn.make_trajectories(shape, B, 11).items()}
    mask = po.create_fd_mask(shape.traj_length, 4)
    out = mo.mtm_forward(sd, {k: traj[k].unsqueeze(2).double() for k in ORDER}, {k: torch.from_numpy(v) for k, v in mask.items()},
                         shape.n_head, shape.n_enc_layer, shape.n_dec_layer, return_stages=True)
    m = np.concatenate([mask[k] for k in ORDER]).astype(np.uint8)
    tm = lambda x: x.permute(1, 0, 2).reshape(-1, x.shape[-1]).contiguous()  # noqa: E731  (B, S, D) -> token-major rows
    enc_out, dec_in = out["_stages"]["enc_out"], out["_stages"]["dec_in"]
    e = tm(enc_out).float().cuda()
    x = torch.full((dec_in.shape[1] * B, dec_in.shape[2]), float("nan"), device="cuda")
    nat.check(nat.lib().m3pc_decoder_scatter_embed(eng._h, B, e.data_ptr(), m.ctypes.data_as(C.c_void_p), x.data_ptr(), None))
    torch.cuda.synchronize()
    assert rel(x, tm(dec_in)) < 1e-5


# ------------------------------------------------------------------------------------------------ omtm.forward
def _module(shape, precision, max_batch, chunk=0):
    from m3pc_b200.mtm_model import omtmConfig
    cfg = omtmConfig(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer, dropout=0.1,
                     norm="none", precision=precision, max_batch=max_batch, chunk=chunk)
    m = cfg.create(shape.data_shapes, shape.traj_length, {k: False for k in shape.data_shapes})
    m.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 0).items()})
    return m.to("cuda")


@pytest.mark.parametrize("scaled,batch,h", [(False, 300, 3), (False, 1, 3), (True, 9, 8)])
def test_forward_vs_fp64_oracle(scaled, batch, h):
    """The hopper model (300 rows: the tensor-core GEMMs; B = 1: the small-problem path) and the scaled one (D = 1024, 4 + 2
    layers, T = 16)."""
    from oracle import mtm_oracle as mo, planner_oracle as po
    shape = syn.scaled_shape("hopper") if scaled else syn.shipped_shape("hopper")
    m = _module(shape, "tf32x3", max_batch=max(16, batch))
    traj = {k: torch.from_numpy(v) for k, v in syn.make_trajectories(shape, batch, 11).items()}
    toks = {k: v.unsqueeze(2) for k, v in traj.items()}
    mask = po.create_fd_mask(shape.traj_length, h)
    ref = mo.mtm_forward(mo.to_torch(syn.make_state_dict(shape, 0), torch.float64), {k: v.double() for k, v in toks.items()},
                         {k: torch.from_numpy(v) for k, v in mask.items()}, shape.n_head, shape.n_enc_layer, shape.n_dec_layer)
    out = m({k: v.cuda() for k, v in toks.items()}, {k: torch.from_numpy(v).cuda() for k, v in mask.items()})
    for k in ("states", "rewards", "returns"):
        assert rel(out[k], ref[k]) < 1e-5, (k, rel(out[k], ref[k]))
    assert rel(out["actions"].loc, ref["actions"]["mu"]) < 1e-5
    assert rel(out["actions"].std, ref["actions"]["std"]) < 3e-5


# ------------------------------------------------------------------------------------------------ planners
def _learner(env, guidance, n_cand, temperature, precision, cls=None, **kw):
    from m3pc_b200.learner import Learner
    from m3pc_b200.mtm_model import omtmConfig
    from m3pc_b200.tokenizers import manager_from_stats
    shape = syn.shipped_shape(env)
    cfg = SimpleNamespace(traj_length=shape.traj_length, device="cuda", action_samples=n_cand, discount=0.99, temperature=temperature,
                          horizon=4, plan_guidance=guidance, lmbda=0.6)
    mcfg = omtmConfig(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer, dropout=0.1,
                      norm="none", precision=precision, max_batch=n_cand)
    om, os_ = syn.make_obs_norm(shape)
    L = (cls or Learner)(cfg, None, shape.data_shapes, mcfg, None, om, os_, manager_from_stats(syn.make_tokenizer_stats(shape, 1)),
                         {k: False for k in shape.data_shapes}, **kw)
    L.mtm.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(shape, 0).items()})
    if hasattr(L, "iql"):
        L.iql.qf.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_critic_state_dict(shape).items()})
    return shape, L


def test_planners_match_reference_golden(golden_dir):
    """The three guidances and mtm_sampling against actions the REFERENCE produced on the same inputs and injected noise."""
    z = np.load(os.path.join(golden_dir, "planner.npz"))
    meta = json.loads(str(z["meta"]))
    for case in meta["cases"]:
        shape, L = _learner(case["env"], case["guidance"], case["n_cand"], case["temperature"], "tf32x3")
        tag, T, h = case["tag"], shape.traj_length, case["horizon"]
        eps = torch.from_numpy(z[f"{tag}/eps"])
        if not case["plan"]:
            L.injected_noise = (eps[0, T - h, 0, :].contiguous().cuda(), None)
        elif case["guidance"] == "noise_adding_lambda":
            L.injected_noise = (eps.contiguous().cuda(), torch.from_numpy(z[f"{tag}/q"]).cuda())
        else:
            L.injected_noise = (eps[:, 0, T - h:, 0, :].contiguous().cuda(), torch.from_numpy(z[f"{tag}/q"]).cuda())
        hist = syn.make_history(shape, seed=case["hist_seed"], path_length=case["path_length"])
        kw = dict(percentage=case["percentage"], plan=case["plan"], rtg=case["rtg"])
        act = L.action_sample(hist, eval=case["eval"], **kw)
        np.testing.assert_allclose(act.cpu().numpy(), z[f"{tag}/action"], rtol=0, atol=1e-4, err_msg=tag)
        if f"{tag}/action_other" in z.files:
            other = L.action_sample(hist, eval=not case["eval"], **{**kw, "rtg": 3.0 if case["rtg"] is None else case["rtg"]})
            np.testing.assert_allclose(other.cpu().numpy(), z[f"{tag}/action_other"], rtol=0, atol=1e-4, err_msg=tag + " other")


@pytest.mark.parametrize("env,guidance,temp,N,path_lengths", [
    ("walker2d", "critic_lambda_guiding", 1.0, 1024, [50 + 3 * e for e in range(8)]),  # the default workload's step: E = 8 x N = 1024
    ("hopper", "rtg_guiding", 0.01, 200, [1, 2, 50, 7, 60]),                          # mixed horizons (env_horizons)
    ("halfcheetah", "noise_adding_lambda", 1.0, 256, [40, 41, 42]),
])
def test_env_batched_plan_matches_fp32_mode(env, guidance, temp, N, path_lengths):
    """A multi-environment plan in tf32x3 against the same plan in the fp32 mode: scores, candidates and actions to the fp32 mode's
    tolerances, and the same argmax / sampled candidate wherever the score gap exceeds twice the score difference.  These cases --
    the default workload's E = 8 x N = 1024 step, a mixed-horizon plan -- have no golden vectors of the reference: they are
    checked against the oracle transitively, through the fp32 mode, which tests/test_gpu_parity.py holds to the fp64 oracle
    (the tf32x3 planners themselves meet the golden vectors in test_planners_match_reference_golden above)."""
    E = len(path_lengths)
    hists = [syn.make_history(syn.shipped_shape(env), seed=30 + e, path_length=p) for e, p in enumerate(path_lengths)]
    rtgs = [2.0 + 0.25 * e for e in range(E)]
    g = torch.Generator(device="cuda").manual_seed(1)
    A = syn.shipped_shape(env).act_dim
    eps = torch.randn(E * N, 4, A, device="cuda", generator=g)
    q = torch.empty(E * N, device="cuda").exponential_(1.0, generator=g)
    res = {}
    for precision in ("fp32", "tf32x3"):
        _, L = _learner(env, guidance, N, temp, precision, max_envs=E)
        hz = [L._clamped_horizon(hist) for hist in hists]  # environment e plans the first hz[e] steps of its candidate rows
        L.debug_plans = True
        L.injected_noise = (eps, q)
        ev = L.action_sample_batch(hists, plan=True, eval=True, rtg=rtgs).clone()
        d = {k: v.clone() for k, v in L.last_plan_debug.items()}
        sm = L.action_sample_batch(hists, plan=True, eval=False, rtg=rtgs).clone()
        res[precision] = (ev, sm, d)
    (ev32, sm32, d32), (ev, sm, d) = res["fp32"], res["tf32x3"]
    J32, J = d32["expect_return"].double(), d["expect_return"].double()
    assert torch.isfinite(J).all()
    assert float((J - J32).abs().max()) <= 2e-5 * max(1.0, float(J32.abs().max()))
    for e in range(E):
        rows = slice(e * N, (e + 1) * N)
        assert rel(d["candidates"][rows, :hz[e]], d32["candidates"][rows, :hz[e]]) < 7e-5, e
    assert rel(ev, ev32) < 1e-4
    for e in range(E):
        Je, J32e = J[e * N:(e + 1) * N], J32[e * N:(e + 1) * N]
        errJ = float((Je - J32e).abs().max())
        top2 = torch.topk(J32e, 2).values
        if float(top2[0] - top2[1]) > 2 * errJ:
            assert int(d["indices"][e][0]) == int(d32["indices"][e][0]), e
        key = torch.exp((J32e - J32e.max()) * temp) / q[e * N:(e + 1) * N].double()
        k2 = torch.topk(key, 2).values
        if float(torch.log(k2[0]) - torch.log(k2[1])) > 2 * temp * 2 * errJ:
            assert int(d["indices"][e][1]) == int(d32["indices"][e][1]), e
            np.testing.assert_allclose(sm[e].cpu().numpy(), sm32[e].cpu().numpy(), atol=1e-4)


def test_zeroshot_matches_reference_golden(golden_dir):
    from m3pc_b200.zeroshot_learner import Learner as ZLearner
    z = np.load(os.path.join(golden_dir, "zeroshot_hopper.npz"))
    meta = json.loads(str(z["meta"]))
    shape, L = _learner("hopper", "rtg_guiding", 1, 0.01, "tf32x3", cls=ZLearner, max_envs=8)
    T = shape.traj_length
    for case in meta["cases"]:
        tag = case["tag"]
        hist = syn.make_history(shape, seed=case["hist_seed"], path_length=case["path_length"])
        h = L._clamped_horizon(hist)
        L.injected_eps = torch.from_numpy(z[f"{tag}/eps"])[0, T - h, 0, :].reshape(1, -1).contiguous().cuda()
        fn = getattr(L, case["fn"])
        np.testing.assert_allclose(fn(hist, eval=True, rtg=case["rtg"]).cpu().numpy(), z[f"{tag}/eval_action"], atol=1e-4, err_msg=tag)
        np.testing.assert_allclose(fn(hist, eval=False, rtg=case["rtg"]).cpu().numpy(), z[f"{tag}/sample_action"], atol=1e-4, err_msg=tag)
    L.action_piid_list_sample(syn.make_history(shape, seed=4, path_length=50), eval=True, rtg=2.5)
    np.testing.assert_allclose(L.action_list[0].cpu().numpy(), z["piid_pl50/eval_action"], atol=1e-4)
    # E = 150 environments: pass rows above the small-problem threshold, row e equal to the B = 1 call to the fp32 tolerance
    Lb = _learner("hopper", "rtg_guiding", 1, 0.01, "tf32x3", cls=ZLearner, max_envs=150)[1]
    hists = [syn.make_history(shape, seed=20 + e, path_length=40 + e % 50) for e in range(150)]
    batch = Lb.action_piid_sample_batch(hists, eval=True, rtg=2.0).clone()
    for e in (0, 77, 149):
        np.testing.assert_allclose(Lb.action_piid_sample(hists[e], eval=True, rtg=2.0)[0].cpu().numpy(), batch[e].cpu().numpy(), atol=1e-5)


# ------------------------------------------------------------------------------------------------ graphs and parameter updates
def test_graph_replay_is_bit_identical_to_eager():
    E, N = 4, 512
    shape, L = _learner("walker2d", "critic_lambda_guiding", N, 1.0, "tf32x3", max_envs=E)
    hists = [syn.make_history(shape, seed=5 + e, path_length=60) for e in range(E)]
    L._engine()
    outs = []
    for _ in range(4):  # eager, capture, replay, replay
        L.__dict__["_plan_counter"] = 7
        outs.append(L.action_sample_batch(hists, plan=True, eval=False, rtg=3.0).clone())
    assert torch.isfinite(outs[0]).all()
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


def test_parameter_updates_reach_the_next_plan(monkeypatch):
    """m3pc_set_param + m3pc_finalize_params (load_state_dict / mark_dirty) after a captured plan: the next plans use the new
    weights, equal to an engine that never captures loaded with them."""
    from m3pc_b200.engine import PlanEngine
    shape, L = _learner("walker2d", "critic_lambda_guiding", 256, 1.0, "tf32x3")
    hist = syn.make_history(shape, seed=4, path_length=80)
    L.seed = 3

    def run(Lx):
        Lx.__dict__["_plan_counter"] = 0
        return Lx.action_sample(hist, plan=True, eval=True, rtg=3.0).double().cpu()

    a = [run(L) for _ in range(3)]  # eager, capture + replay, replay
    np.testing.assert_allclose(a[2].numpy(), a[0].numpy(), atol=1e-6)
    with torch.no_grad():
        L.mtm.encoder.layers[0].linear1.weight.mul_(1.25)
        L.mtm.output_head_dict["rewards"][3].bias.add_(0.3)
    L.mtm.mark_dirty()
    b = [run(L) for _ in range(3)]
    monkeypatch.setitem(PlanEngine.default_options, "graphs", 0)
    _, R = _learner("walker2d", "critic_lambda_guiding", 256, 1.0, "tf32x3")
    R.seed = 3
    with torch.no_grad():
        R.mtm.encoder.layers[0].linear1.weight.mul_(1.25)
        R.mtm.output_head_dict["rewards"][3].bias.add_(0.3)
    R.mtm.mark_dirty()
    rb = run(R)
    assert float((a[0] - rb).abs().max()) > 1e-5
    for x in b:
        np.testing.assert_allclose(x.numpy(), rb.numpy(), atol=1e-6)


@pytest.mark.parametrize("precision", ["bf16", "fp32", "tf32x3"])
@pytest.mark.parametrize("hidden", [64, 200])
def test_twinq_critic_width_not_a_multiple_of_128(nat, precision, hidden):
    """A TwinQ whose width is not a multiple of 128 runs its two hidden layers on the fp32 operands in every mode (bf16 mode keeps
    its tensor-core critic for widths that are), on the mode's fp32 kernel: CUDA cores in bf16 and fp32 mode, the 3xTF32 kernel's
    dispatcher in tf32x3 mode.  K7 m3pc_twinq against the float64 oracle at the fp32 bar."""
    from m3pc_b200.engine import PlanEngine
    from oracle import mtm_oracle as mo
    shape = syn.shipped_shape("walker2d")
    eng = PlanEngine(n_embd=shape.n_embd, n_head=shape.n_head, n_enc_layer=shape.n_enc_layer, n_dec_layer=shape.n_dec_layer,
                     traj_length=shape.traj_length, obs_dim=shape.obs_dim, act_dim=shape.act_dim, precision=precision, max_batch=512,
                     critic_hidden=hidden)
    eng.load_state_dict(syn.make_state_dict(shape, 0))
    eng.load_tokenizer_stats(syn.make_tokenizer_stats(shape, 1))
    qsd_np = syn.make_critic_state_dict(shape, hidden=hidden)
    om, os_ = syn.make_obs_norm(shape)
    eng.load_critic(qsd_np, om, os_)
    eng.finalize()
    T, A, obs, h, N = shape.traj_length, shape.act_dim, shape.obs_dim, 4, 300
    rs = np.random.RandomState(1)
    sp = torch.from_numpy(rs.randn(N, T, obs)).float().cuda()
    cand = torch.from_numpy(rs.rand(N, h, A) * 2 - 1).float().cuda()
    q = torch.empty(N * h, device="cuda")
    nat.check(nat.lib().m3pc_twinq(eng._h, sp.data_ptr(), cand.data_ptr(), N, h, q.data_ptr(), None))
    torch.cuda.synchronize()
    st = mo.stats_to_torch(syn.make_tokenizer_stats(shape, 1), torch.float64)["states"]
    s_hat = sp.double().cpu()[:, T - h:] * st["std"] + st["mean"]
    ref = mo.twinq(mo.to_torch(qsd_np, torch.float64), torch.from_numpy(om).double(), torch.from_numpy(os_).double(),
                   s_hat.reshape(N * h, obs), cand.double().cpu().reshape(N * h, A))
    assert rel(q, ref) < 2e-5
