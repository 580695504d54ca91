"""Kernel-level parity: every fused memory-bound kernel of the path through its own C-ABI entry (SURVEY.md section 8b:
K1 m3pc_embed_gather, K4 m3pc_decoder_scatter_embed, K5 m3pc_heads, K6 m3pc_sample_candidates, K7 m3pc_twinq,
K8 m3pc_score_select) against the stage tensors of the float64 oracle (oracle/mtm_oracle.py ``_stages``,
oracle/planner_oracle.py), in both precision modes.  Layout: the library's token-major rows (row = token * B + b)."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from m3pc_b200 import synthetic as syn

pytestmark = pytest.mark.gpu
TOL = {"fp32": 2e-5, "bf16": 1e-2}
ORDER = ("states", "actions", "rewards", "returns")


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(1.0, float(b.abs().max())))


def tok_major(x):  # oracle (B, S, D) -> library (S*B, D)
    return x.permute(1, 0, 2).reshape(-1, x.shape[-1]).contiguous()


@pytest.fixture(scope="module")
def nat():
    from m3pc_b200 import _native
    _native.lib()
    return _native


def _engine(shape, precision, critic=False, max_batch=256):
    from m3pc_b200.engine import engine_from_synthetic
    return engine_from_synthetic(shape, syn.make_state_dict(shape, 0), syn.make_tokenizer_stats(shape, 1), precision=precision, max_batch=max_batch,
                                 critic_sd=syn.make_critic_state_dict(shape) if critic else None, obs_norm=syn.make_obs_norm(shape) if critic else None)


def _stages(shape, B, mask_fn, idx, seed=11):
    from oracle import mtm_oracle as mo
    sd = mo.to_torch(syn.make_state_dict(shape, 0), torch.float64)
    traj = {k: torch.from_numpy(v) for k, v in syn.make_trajectories(shape, B, seed).items()}
    toks = {k: traj[k].unsqueeze(2).double() for k in ORDER}
    mask = mask_fn(shape.traj_length, idx)
    out = mo.mtm_forward(sd, toks, {k: torch.from_numpy(v) for k, v in mask.items()}, shape.n_head, shape.n_enc_layer, shape.n_dec_layer,
                         return_stages=True)
    m = np.concatenate([mask[k] for k in ORDER]).astype(np.uint8)
    return sd, traj, m, out


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("mask_name,idx,B", [("fd", 4, 37), ("rcbc", 4, 1), ("pi", 3, 130), ("fid", 0, 5)])
def test_k1_embed_gather(nat, precision, mask_name, idx, B):
    from oracle import mtm_oracle as mo, planner_oracle as po
    shape = syn.shipped_shape("walker2d")
    eng = _engine(shape, precision)
    sd, traj, m, out = _stages(shape, B, getattr(po, f"create_{mask_name}_mask"), idx)
    enc_in = out["_stages"]["enc_in"]  # (B, S, D)
    S, D = enc_in.shape[1], enc_in.shape[2]
    dev = {k: traj[k].float().cuda().contiguous() for k in ORDER}
    x = torch.full((S * B, D), float("nan"), device="cuda")
    y = torch.full((S * B, D), float("nan"), device="cuda", dtype=torch.bfloat16 if precision == "bf16" else torch.float32)
    nat.check(nat.lib().m3pc_embed_gather(eng._h, B, dev["states"].data_ptr(), dev["actions"].data_ptr(), dev["rewards"].data_ptr(),
                                          dev["returns"].data_ptr(), m.ctypes.data_as(C.c_void_p), x.data_ptr(), y.data_ptr(), None))
    torch.cuda.synchronize()
    assert rel(x, tok_major(enc_in)) < 2e-5  # the embedding itself is fp32 in both modes
    ln = mo.layer_norm(enc_in, sd["encoder.layers.0.norm1.weight"], sd["encoder.layers.0.norm1.bias"])
    assert rel(y, tok_major(ln)) < (2e-5 if precision == "fp32" else 8e-3)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("stack,B,S", [(0, 150, 13), (0, 3, 17), (1, 40, 32), (0, 1100, 13)])
def test_k2_k3_block_forward(nat, precision, stack, B, S):
    """One transformer block of the handle through its own entry (K2 GEMMs + K3 attention + the fused LayerNorms) against the
    oracle's restatement of nn.TransformerEncoderLayer (oracle/mtm_oracle.py:encoder_layer); 1100 x 13 rows takes the fused
    residual-GEMM + LayerNorm kernels, the small cases the plain tiles."""
    from oracle import mtm_oracle as mo
    shape = syn.shipped_shape("walker2d")
    eng = _engine(shape, precision, max_batch=max(256, B))
    sd = mo.to_torch(syn.make_state_dict(shape, 0), torch.float64)
    D = shape.n_embd
    name = ("encoder", "decoder")[stack]
    n_layer = (shape.n_enc_layer, shape.n_dec_layer)[stack]
    torch.manual_seed(B + S)
    x0 = torch.randn(B, S, D, dtype=torch.float64)
    for layer in range(n_layer):
        ref = mo.encoder_layer(x0, sd, f"{name}.layers.{layer}", shape.n_head)
        nxt = f"{name}.layers.{layer + 1}.norm1" if layer + 1 < n_layer else f"{name}.norm"
        ref_y = mo.layer_norm(ref, sd[nxt + ".weight"], sd[nxt + ".bias"])
        x = tok_major(x0).float().cuda()
        y = torch.full((S * B, D), float("nan"), device="cuda", dtype=torch.bfloat16 if precision == "bf16" else torch.float32)
        nat.check(nat.lib().m3pc_block_forward(eng._h, stack, layer, B, S, x.data_ptr(), y.data_ptr(), None))
        torch.cuda.synchronize()
        tol = TOL[precision]
        assert rel(x, tok_major(ref)) < tol, (layer, rel(x, tok_major(ref)))
        assert rel(y, tok_major(ref_y)) < (2e-5 if precision == "fp32" else 2e-2), layer
        # without the trailing LayerNorm the residual stream is the same
        x2 = tok_major(x0).float().cuda()
        nat.check(nat.lib().m3pc_block_forward(eng._h, stack, layer, B, S, x2.data_ptr(), None, None))
        torch.cuda.synchronize()
        assert rel(x2, x) < (1e-6 if precision == "fp32" else 2e-3)
    with pytest.raises(ValueError):
        nat.check(nat.lib().m3pc_block_forward(eng._h, 2, 0, B, S, x.data_ptr(), None, None))
    with pytest.raises(ValueError):
        nat.check(nat.lib().m3pc_block_forward(eng._h, stack, n_layer, B, S, x.data_ptr(), None, None))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("mask_name,idx,B", [("fd", 4, 200), ("pi", 3, 33), ("rcbc", 0, 2)])
def test_k4_decoder_scatter_embed(nat, precision, mask_name, idx, B):
    from oracle import planner_oracle as po
    shape = syn.shipped_shape("hopper")
    eng = _engine(shape, precision)
    sd, traj, m, out = _stages(shape, B, getattr(po, f"create_{mask_name}_mask"), idx)
    enc_out, dec_in = out["_stages"]["enc_out"], out["_stages"]["dec_in"]
    D, T4 = dec_in.shape[2], dec_in.shape[1]
    e = tok_major(enc_out).cuda()
    e = e.bfloat16() if precision == "bf16" else e.float()
    x = torch.full((T4 * B, D), float("nan"), device="cuda")
    nat.check(nat.lib().m3pc_decoder_scatter_embed(eng._h, B, e.data_ptr(), m.ctypes.data_as(C.c_void_p), x.data_ptr(), None))
    torch.cuda.synchronize()
    assert torch.isfinite(x).all()
    assert rel(x, tok_major(dec_in)) < (2e-5 if precision == "fp32" else 8e-3)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_k5_heads(nat, precision):
    from oracle import planner_oracle as po
    shape = syn.shipped_shape("walker2d")
    B = 45
    eng = _engine(shape, precision)
    sd, traj, m, out = _stages(shape, B, po.create_fd_mask, 4)
    xdec = tok_major(out["_stages"]["decoder_x"]).float().cuda()
    T, A, obs = shape.traj_length, shape.act_dim, shape.obs_dim
    o = {k: torch.full((B, T, d), float("nan"), device="cuda") for k, d in (("states", obs), ("mu", A), ("std", A), ("rewards", 1), ("returns", 1))}
    nat.check(nat.lib().m3pc_heads(eng._h, B, xdec.data_ptr(), o["states"].data_ptr(), o["mu"].data_ptr(), o["std"].data_ptr(),
                                   o["rewards"].data_ptr(), o["returns"].data_ptr(), None))
    torch.cuda.synchronize()
    tol = TOL[precision]
    for k in ("states", "rewards", "returns"):
        assert rel(o[k], out[k].squeeze(2)) < tol, k
    assert rel(o["mu"], out["actions"]["mu"].squeeze(2)) < tol
    assert rel(o["std"], out["actions"]["std"].squeeze(2)) < 3.5 * tol


@pytest.mark.parametrize("noise_mode", [0, 1])
def test_k6_sample_candidates(nat, noise_mode):
    T, A, h, N = 8, 6, 4, 333
    rs = np.random.RandomState(0)
    mu, std = torch.from_numpy(rs.randn(T, A)).float().cuda(), torch.from_numpy(rs.rand(T, A) + 0.1).float().cuda()
    eps = torch.from_numpy(rs.randn(N, h, A)).float().cuda()
    out = torch.empty(N, h, A, device="cuda")
    nat.check(nat.lib().m3pc_sample_candidates(mu.data_ptr(), std.data_ptr(), eps.data_ptr(), 0, N, h, A, T, noise_mode, 0, out.data_ptr(), None))
    if noise_mode == 0:
        ref = torch.tanh(mu.double()[None, T - h:] + std.double()[None, T - h:] * eps.double())
    else:
        ref = torch.clamp(torch.tanh(mu.double())[None, T - h:] + 0.09 * eps.double(), -0.99999, 0.99999)
    assert rel(out, ref) < 1e-6
    # Philox: a function of (seed, GLOBAL candidate id) only
    a, b = torch.empty(N, h, A, device="cuda"), torch.empty(100, h, A, device="cuda")
    nat.check(nat.lib().m3pc_sample_candidates(mu.data_ptr(), std.data_ptr(), None, 9, N, h, A, T, noise_mode, 0, a.data_ptr(), None))
    nat.check(nat.lib().m3pc_sample_candidates(mu.data_ptr(), std.data_ptr(), None, 9, 100, h, A, T, noise_mode, 200, b.data_ptr(), None))
    assert torch.equal(a[200:300], b) and float(a.std()) > 0.01


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_k7_twinq(nat, precision):
    from oracle import mtm_oracle as mo
    shape = syn.shipped_shape("walker2d")
    eng = _engine(shape, precision, critic=True, max_batch=512)
    T, A, obs, h, N = shape.traj_length, shape.act_dim, shape.obs_dim, 4, 300
    rs = np.random.RandomState(1)
    sp = torch.from_numpy(rs.randn(N, T, obs)).float().cuda()
    cand = torch.from_numpy(rs.rand(N, h, A) * 2 - 1).float().cuda()
    q = torch.empty(N * h, device="cuda")
    nat.check(nat.lib().m3pc_twinq(eng._h, sp.data_ptr(), cand.data_ptr(), N, h, q.data_ptr(), None))
    st = mo.stats_to_torch(syn.make_tokenizer_stats(shape, 1), torch.float64)["states"]
    om, os_ = [torch.from_numpy(v).double() for v in syn.make_obs_norm(shape)]
    qsd = mo.to_torch(syn.make_critic_state_dict(shape), torch.float64)
    s_hat = sp.double().cpu()[:, T - h:] * st["std"] + st["mean"]
    ref = mo.twinq(qsd, om, os_, s_hat.reshape(N * h, obs), cand.double().cpu().reshape(N * h, A))
    assert rel(q, ref) < (2e-5 if precision == "fp32" else 1e-2)


@pytest.mark.parametrize("kind,temp", [("rtg", 0.01), ("critic", 1.0)])
@pytest.mark.parametrize("h", [4, 7])
def test_k8_score_select(nat, kind, temp, h):
    """The closed-form TD(lambda) score against the reference's loop (learner.py:301-316, restated in the oracle) and the
    softmax / arg-max / Exp(1)-race selection against float64."""
    T, A, N, disc, lm = 8, 3, 777, 0.99, 0.6
    rs = np.random.RandomState(4)
    rew, ret = torch.from_numpy(rs.randn(N, T)).float(), torch.from_numpy(rs.randn(N, T) * 0.1).float()
    qv = torch.from_numpy(rs.randn(N * h) * 3).float()
    cand = torch.from_numpy(rs.rand(N, h, A) * 2 - 1).float()
    expq = torch.from_numpy(rs.exponential(1.0, N)).float()
    stats = np.array([0.3, 1.7, -0.2, 0.9], dtype=np.float32)
    J = torch.empty(N, device="cuda"); ev = torch.empty(A, device="cuda"); sm = torch.empty(A, device="cuda")
    idx = torch.zeros(2, dtype=torch.int32, device="cuda"); part = torch.zeros(nat.PARTIAL_FLOATS, device="cuda")
    d = lambda t: t.cuda().contiguous()
    rew_d, ret_d, qv_d, cand_d, expq_d = d(rew), d(ret), d(qv), d(cand), d(expq)
    nat.check(nat.lib().m3pc_score_select(rew_d.data_ptr(), ret_d.data_ptr() if kind == "rtg" else None, qv_d.data_ptr() if kind == "critic" else None,
                                          cand_d.data_ptr(), expq_d.data_ptr(), stats.ctypes.data_as(C.c_void_p), disc, lm, temp, N, h, T, A, 0, 0,
                                          J.data_ptr(), ev.data_ptr(), sm.data_ptr(), part.data_ptr(), idx.data_ptr(), None))
    # reference loop in float64 on the de-normalised predictions
    r = rew.double() * float(stats[1]) + float(stats[0])
    g = ret.double() * float(stats[3]) + float(stats[2])
    Jr = torch.zeros(N, dtype=torch.float64)
    for t in range(h):
        vals = torch.zeros(N, t + 1, dtype=torch.float64)
        if t > 0:
            vals[:, :t] = r[:, T - h:T - h + t]
        vals[:, t] = g[:, T - h + t] * 1000 if kind == "rtg" else qv.double().reshape(N, h)[:, t]
        vals = vals * torch.cumprod(disc * torch.ones(t + 1, dtype=torch.float64), 0)[None]
        Jr = Jr + vals.sum(-1) * ((1 - lm) * lm ** t if t < h - 1 else lm ** t)
    assert rel(J, Jr) < 2e-6
    Jd = J.double().cpu()
    w = torch.exp((Jd - Jd.max()) * temp)
    np.testing.assert_allclose(ev.cpu().numpy(), ((w[:, None] * cand[:, 0].double()).sum(0) / w.sum()).numpy(), atol=2e-5)
    assert idx.tolist() == [int(torch.argmax(Jd)), int(torch.argmax(w / expq.double()))]
    assert torch.equal(sm.cpu(), cand[idx[1].item(), 0])
    assert float(part[0]) == float(Jd.max()) and abs(float(part[1]) - float(w.sum())) < 1e-3 * float(w.sum())
