"""Host-side mirror of the reference API: masks, tokenizers, state_dict layout, window builder, error behaviour (CPU only)."""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from m3pc_b200 import masks as M
from m3pc_b200 import synthetic as syn
from m3pc_b200.learner import PlannerMixin
from m3pc_b200.mtm_model import SquashedNormal, omtm, omtmConfig
from m3pc_b200.tokenizers import ContinuousTokenizer, DataStatistics, TokenizerManager, manager_from_stats
from oracle import mtm_oracle as mo
from oracle import planner_oracle as po


def test_mask_creators_bit_exact_vs_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "masks.npz"))
    fns = {"rcbc": M.create_rcbc_mask, "fd": M.create_fd_mask, "pi": M.create_pi_mask, "fid": M.create_fid_mask, "gid": M.create_gid_mask}
    for key in z.files:
        T, name, idx = key.split("/")
        T, idx = int(T[1:]), int(idx)
        m = fns[name](T, "cpu", idx)
        assert list(m.keys()) == ["states", "actions", "rewards", "returns"]
        got = np.stack([m[k].numpy() for k in m])
        assert all(v.dtype == torch.float64 for v in m.values())
        assert np.array_equal(got, z[key]), key
        assert np.array_equal(M.mask_bits(name, T, idx), z[key].astype(np.uint8).reshape(-1))
    with pytest.raises(ValueError):
        M.create_fd_mask(8, "cpu", 8)


def test_random_autoregressive_masks_bit_exact_vs_reference(golden_dir):
    """The validation-loss mask draw (finetune_omtm/masks.py:64-125) consumes numpy's global generator in the reference's order:
    same seed, same masks (fixture written by the reference, tests/golden/gen_valloss_fixture.py)."""
    import json
    z = np.load(os.path.join(golden_dir, "valloss.npz"))
    meta = json.loads(str(z["meta"]))
    shapes = {"states": (1, 17), "actions": (1, 6), "rewards": (1, 1), "returns": (1, 1)}
    n = 0
    for ci, (ratios, pw) in enumerate(meta["mask_configs"]):
        ratios = tuple(ratios) if isinstance(ratios, list) else ratios
        for seed in range(meta["mask_seeds"]):
            for T in (8, 16):
                np.random.seed(seed)
                m = M.create_random_autoregressize_mask(shapes, ratios, T, "cpu", tuple(pw))
                assert list(m.keys()) == list(shapes) and all(v.dtype == torch.float64 and tuple(v.shape) == (T, 1) for v in m.values())
                assert np.array_equal(np.stack([m[k].numpy()[:, 0] for k in m]), z[f"mask/{ci}/{T}/{seed}"]), (ci, T, seed)
                assert not bool(m["actions"].eq(1).all())
                n += 1
    assert n == 360
    rs = np.random.RandomState(5)
    one = M.create_full_random_mask((1, 3), 10, 0.4, "cpu", rs)
    assert tuple(one.shape) == (10, 1) and int(one.sum()) == 4


def test_kept_token_counts():
    # SURVEY.md appendix: rcbc 17 / fd 13 / pi=gid 10 / fid 12 at idx=4; 9 / 9 / 8 / 8 at idx=0
    for idx, want in ((4, (17, 13, 10, 12)), (0, (9, 9, 8, 8))):
        got = tuple(int(M.mask_bits(k, 8, idx).sum()) for k in ("rcbc", "fd", "pi", "fid"))
        assert got == want


def test_tokenizers_match_oracle():
    shape = syn.shipped_shape("walker2d")
    stats = syn.make_tokenizer_stats(shape, 1)
    tm = manager_from_stats(stats)
    traj = {k: torch.from_numpy(v) for k, v in syn.make_trajectories(shape, 4, 3).items()}
    enc = tm.encode(traj)
    ref = mo.encode_all(traj, mo.stats_to_torch(stats))
    for k in traj:
        assert enc[k].shape == (4, 8, 1, traj[k].shape[-1]) and enc[k].dtype == torch.float32
        assert torch.equal(enc[k], ref[k])
    dec = tm.decode({k: enc[k] for k in ("states", "rewards", "returns")})
    for k in dec:
        np.testing.assert_allclose(dec[k].numpy(), traj[k].numpy(), rtol=1e-5, atol=1e-5)
    # float64 returns are normalised in float64 and only then cast (continuous.py:74-79)
    r64 = torch.full((1, 8, 1), 3.0, dtype=torch.float64)
    got = tm.tokenizers["returns"].encode(r64)
    want = ((r64 - torch.from_numpy(stats["returns"]["mean"]).double()) / torch.from_numpy(stats["returns"]["std"]).double()).float().unsqueeze(2)
    assert got.dtype == torch.float32 and torch.equal(got, want)
    with pytest.raises(AssertionError):
        tm.tokenizers["states"].encode(torch.zeros(8, 17))
    es = tm.engine_stats()
    assert np.array_equal(es["actions"]["std"], np.ones(6, np.float32)) and np.array_equal(es["states"]["mean"], stats["states"]["mean"])


def test_small_std_is_not_normalised():
    ds = SimpleNamespace(trajectory_statistics=lambda: {"states": DataStatistics(np.zeros(3), np.array([0.05, 0.5, 2.0]), -np.ones(3), np.ones(3))})
    tok = ContinuousTokenizer.create("states", ds)
    assert np.allclose(tok._data_std.numpy(), [1.0, 0.5, 2.0])


def test_state_dict_layout_matches_reference():
    shape = syn.shipped_shape("hopper")
    sd = syn.make_state_dict(shape, 0)
    m = omtmConfig(n_embd=512, n_head=4, n_enc_layer=2, n_dec_layer=1, dropout=0.1, norm="none").create(
        shape.data_shapes, shape.traj_length, {k: False for k in shape.data_shapes})
    own = m.state_dict()
    assert set(own.keys()) == set(sd.keys())  # the synthetic dict was loaded into the reference with strict=True (gen_golden.py)
    for k, v in sd.items():
        assert tuple(own[k].shape) == v.shape, k
    res = m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert np.array_equal(m.pos_embed.numpy(), sd["pos_embed"])
    assert sum(p.numel() for p in m.parameters()) == 11_326_995  # SURVEY.md: parameter count of the shipped hopper model
    assert not m.training


def test_unsupported_configurations_raise():
    shape = syn.shipped_shape("hopper")
    dm = {k: False for k in shape.data_shapes}
    with pytest.raises(NotImplementedError):
        omtmConfig(n_embd=512, n_head=4, latent_dim=64).create(shape.data_shapes, 8, dm)
    with pytest.raises(NotImplementedError):
        omtmConfig(n_embd=512, n_head=4).create(shape.data_shapes, 8, {**dm, "actions": True})
    with pytest.raises(NotImplementedError):
        omtmConfig(n_embd=512, n_head=2).create(shape.data_shapes, 8, dm)  # head_dim 256
    m = omtmConfig(n_embd=512, n_head=4).create(shape.data_shapes, 8, dm)
    toks = {k: torch.zeros(2, 8, 1, d[1]) for k, d in shape.data_shapes.items()}
    with pytest.raises(NotImplementedError):  # no CPU path
        m(toks, M.create_fd_mask(8, "cpu", 4))
    with pytest.raises(NotImplementedError):  # 3-D masks, as mtm_model.py:579
        m.process_masks(toks, {k: torch.zeros(2, 8, 1) for k in toks})
    with pytest.raises(AssertionError):  # feature-dim check, mtm_model.py:565-570
        m.process_masks({**toks, "states": torch.zeros(2, 8, 1, 5)}, M.create_fd_mask(8, "cpu", 4))


def test_squashed_normal_surface():
    torch.manual_seed(0)
    d = SquashedNormal(torch.randn(1, 8, 1, 3), torch.rand(1, 8, 1, 3))
    assert torch.equal(d.mean, torch.tanh(d.loc))
    s = d.sample((5,))
    assert s.shape == (5, 1, 8, 1, 3) and float(s.abs().max()) <= 1.0
    torch.manual_seed(3)
    a = d.sample((4,))
    torch.manual_seed(3)
    eps = torch.randn(4, 1, 8, 1, 3)
    assert torch.allclose(a, torch.tanh(d.loc + d.std * eps))


class _HostPlanner(PlannerMixin):
    """PlannerMixin with only the host pieces wired (no engine): exercises the window builder on numpy buffers."""

    def __init__(self, shape, stats, horizon=4):
        self.cfg = SimpleNamespace(traj_length=shape.traj_length, horizon=horizon)
        self.tokenizer_manager = manager_from_stats(stats)
        rt = self.tokenizer_manager.tokenizers["returns"]
        self.__dict__["_rt_norm"] = (rt._data_mean.double().numpy(), rt._data_std.double().numpy(), True)


@pytest.mark.parametrize("path_length,future", [(50, False), (0, False), (2, False), (3, False), (50, True), (997, True), (998, True), (1, True)])
def test_window_builder_matches_oracle(path_length, future):
    shape = syn.shipped_shape("hopper")
    stats = syn.make_tokenizer_stats(shape, 1)
    hist = syn.make_history(shape, seed=4, path_length=path_length)
    P = po.from_synthetic(shape, syn.make_state_dict(shape, 0), stats, action_samples=1)
    H = _HostPlanner(shape, stats)
    T = shape.traj_length
    for rtg, pct in ((3.0, 1.0), (None, 0.8)):
        traj, h = P.build_window(hist, percentage=pct, rtg=rtg, future_obs=future)
        assert H._clamped_horizon(hist) == h
        s, a, r, t = np.full((T, shape.obs_dim), 9, np.float32), np.full((T, shape.act_dim), 9, np.float32), np.full(T, 9, np.float32), np.full(T, 9, np.float32)
        H._fill_window(s, a, r, t, hist, h, pct, rtg, future_obs=future)
        assert np.array_equal(s, traj["states"][0].numpy()) and np.array_equal(a, traj["actions"][0].numpy())
        assert np.array_equal(r, traj["rewards"][0, :, 0].numpy())
        tok = mo.encode_all({"returns": traj["returns"]}, mo.stats_to_torch(stats))["returns"][0, :, 0, 0].numpy()
        assert np.array_equal(t, tok)  # float64 normalisation, single rounding


def test_eval_requires_rtg():
    shape = syn.shipped_shape("hopper")
    H = _HostPlanner(shape, syn.make_tokenizer_stats(shape, 1))
    with pytest.raises(AssertionError):
        H.action_sample(syn.make_history(shape), eval=True, rtg=None)


def test_bench_reference_arm_prints_contract_line():
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                          "--workload", "hopper_rtg_625"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "plans_per_sec" and line["unit"] == "plans/s"
    assert line["steps"] == 2  # --steps sets the number of timed plans
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0
