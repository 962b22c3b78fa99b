"""Batched observation stage (first 'next' row, SURVEY.md section 8f): descriptor synthesis on the CPU, percentile
normalisation and the whole observe() call on the GPU."""
import os

import numpy as np
import pytest

from oracle import composer
from util import reference_path


def _state(n_env, n_dot, seed):
    from qdsim import synth
    rng = np.random.default_rng(seed)
    dev = synth.sample_devices(n_env, n_dot, seed=seed)
    mb = synth.model_batch(dev)
    gv = rng.uniform(-2, 4, (n_env, n_dot))
    vgm = -np.eye(n_dot + 1) + rng.normal(0, 0.05, (n_env, n_dot + 1, n_dot + 1))
    origin = rng.normal(0, 0.1, (n_env, n_dot + 1))
    sv = rng.uniform(0.3, 0.7, n_env)
    return dev, mb, gv, vgm, origin, sv


def test_obs_scans_match_the_composer_env_by_env():
    from qdsim import obs
    dev, mb, gv, vgm, origin, sv = _state(5, 4, 1)
    scans = obs.obs_scans(mb, gv, sv, vgm, origin, -1.7, 1.7, 16, peak_width=dev["peak_width"], seeds=np.arange(15))
    assert len(scans) == 15
    for e in range(5):
        for c in range(3):
            rec = scans[e * 3 + c]
            want = composer.do2d_virtual_coupled(5, c + 1, gv[e, c] - 1.7, gv[e, c] + 1.7, 16, c + 2, gv[e, c + 1] - 1.7,
                                                 gv[e, c + 1] + 1.7, 16, np.append(gv[e], sv[e]), vgm[e], origin[e])
            got = composer.affine_grid(rec["v0"][:5], rec["dx"][:5], rec["dy"][:5], 16, 16)
            assert np.allclose(got, want, atol=1e-12)
            assert rec["env_id"] == e and rec["pix_offset"] == (e * 3 + c) * 256
    phys = obs.obs_scans(mb, gv, 0.0, None, None, -1.0, 1.0, 8, virtual=False, seeds=np.arange(15))
    want = composer.do2d(5, 2, gv[3, 1] - 1, gv[3, 1] + 1, 8, 3, gv[3, 2] - 1, gv[3, 2] + 1, 8)
    rec = phys[3 * 3 + 1]
    assert np.allclose(composer.affine_grid(rec["v0"][:5], rec["dx"][:5], rec["dy"][:5], 8, 8), want, atol=1e-12)


def test_obs_scans_radial_and_peak_width_rules():
    from qdsim import obs
    dev, mb, gv, vgm, origin, sv = _state(4, 3, 2)
    gt = gv + np.array([[0.5, 0.2, 0.1], [35.0, 0.0, 0.0], [0.0, 0.0, -50.0], [1.0, 1.0, 1.0]])
    radial = dict(zero_radius=np.full(4, 25.0), ramp_distance=np.full(4, 32.0), full_noise_distance=np.full(4, 33.0),
                  max_amplitude=0.05)
    s = obs.obs_scans(mb, gv, sv, vgm, origin, -1.5, 1.5, 32, gate_ground_truth=gt, radial=radial,
                      peak_width=0.3, peak_width_alpha=0.01, seeds=np.arange(8))
    assert list(s["rad_mode"]) == [1, 1, 2, 1, 1, 2, 1, 1]          # a pair is replaced iff either dot is > 33 V away
    assert np.allclose(s["rad_alpha"], 0.05 / 32.0) and np.allclose(s["rad_x0"][0], gv[0, 0] - 1.5 - gt[0, 0])
    want_pw = np.clip(0.3 - np.abs(0.01 * (abs(gv[0, 0]) + abs(gv[0, 1])) / 2), 0, 1)
    assert np.isclose(s["peak_width"][0], want_pw)


@pytest.mark.gpu
@pytest.mark.parametrize("per_env,n_env", [(3 * 32 * 32, 7), (1000, 3), (7 * 64 * 64, 4), (2, 2)])
def test_percentile_normalisation_is_bit_exact_vs_numpy(engine, per_env, n_env):
    import torch
    rng = np.random.default_rng(per_env)
    z = rng.normal(0.6, 0.3, (n_env, per_env)).astype(np.float32)
    z[0, : per_env // 2] = z[0, 0]                                   # heavy ties
    if n_env > 2:
        z[2] = 0.25                                                  # constant image -> zeros
    z_dev = torch.from_numpy(z).cuda()
    stats = torch.empty((n_env, 2), dtype=torch.float64, device="cuda")
    out = engine.normalise_obs(z_dev.clone(), per_env=per_env, n_env=n_env, stats=stats)
    torch.cuda.synchronize()
    for e in range(n_env):
        img = z[e].astype(np.float64)
        p_low, p_high = np.percentile(img, 0.5), np.percentile(img, 99.5)
        want = np.clip((img - p_low) / (p_high - p_low), 0, 1) if p_high > p_low else np.zeros_like(img)
        assert stats[e, 0].item() == p_low and stats[e, 1].item() == p_high
        assert np.array_equal(out[e].cpu().numpy(), want.astype(np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ties_low_fit", "ties_low_overflow", "ties_high_overflow", "median", "ragged_1500",
                                  "two_values", "negative_and_zero", "sensor_like", "exactly_1024", "k_plus_2_equals_m"])
def test_percentile_kernel_paths_are_bit_exact(engine, case):
    """The extreme-rank path of qd_normalise_reg_kernel (thread minima / maxima -> short lists -> rank by counting) and its
    fallbacks (more than 1024 pixels tied at an extreme, non-extreme percentiles), on inputs built to hit each of them:
    statistics and fp32 images bit for bit against np.percentile + the reference's expression (env.py:471-509)."""
    import torch
    rng = np.random.default_rng(sum(map(ord, case)))
    q_low, q_high, per_env, n_env = 0.5, 99.5, 7 * 64 * 64, 3
    if case == "ragged_1500":
        per_env = 1500
    elif case == "exactly_1024":
        per_env = 1024
    elif case == "k_plus_2_equals_m":
        per_env = 700                                             # q = 0.5 / 99.5 -> k_lo = 3: far inside; then stress q
        q_low, q_high = 40.0, 60.0                                # k_lo + 2 = 281 <= 700 = M: still the extreme-rank path
    z = rng.normal(0.6, 0.3, (n_env, per_env)).astype(np.float32)
    if case == "ties_low_fit":
        z[0, rng.choice(per_env, 600, replace=False)] = z[0].min() - 1.0          # 600 pixels tied at the minimum
        z[1, rng.choice(per_env, 900, replace=False)] = z[1].max() + 1.0          # 900 tied at the maximum
    elif case == "ties_low_overflow":
        z[0, rng.choice(per_env, 5000, replace=False)] = z[0].min() - 1.0         # list overflow -> full radix select
    elif case == "ties_high_overflow":
        z[1, rng.choice(per_env, 9000, replace=False)] = z[1].max() + 0.5
    elif case == "median":
        q_low, q_high = 50.0, 50.0                                                # not extreme: full radix select
    elif case == "two_values":
        z[:] = np.where(rng.random(z.shape) < 0.5, np.float32(0.1), np.float32(0.9))
    elif case == "negative_and_zero":
        z[0] = rng.normal(0.0, 1e-3, per_env).astype(np.float32)
        z[0, ::7] = 0.0
        z[1, ::5] = -0.0
    elif case == "sensor_like":                                                   # plateaus + tiny noise, like a real image
        z = (np.float32(0.0305) + np.float32(1e-4) * rng.standard_normal((n_env, per_env))).astype(np.float32)
        z[:, : per_env // 3] += np.float32(0.4)
    z_dev = torch.from_numpy(np.ascontiguousarray(z)).cuda()
    stats = torch.empty((n_env, 2), dtype=torch.float64, device="cuda")
    out = engine.normalise_obs(z_dev.clone(), per_env=per_env, n_env=n_env, q_low=q_low, q_high=q_high, stats=stats)
    torch.cuda.synchronize()
    for e in range(n_env):
        img = z[e].astype(np.float64)
        p_low, p_high = np.percentile(img, q_low), np.percentile(img, q_high)
        want = np.clip((img - p_low) / (p_high - p_low), 0, 1) if p_high > p_low else np.zeros_like(img)
        assert stats[e, 0].item() == p_low and stats[e, 1].item() == p_high, (case, e)
        assert np.array_equal(out[e].cpu().numpy(), want.astype(np.float32)), (case, e)


@pytest.mark.gpu
def test_observe_batch_end_to_end(engine):
    """obs_scans -> scan kernel -> normalisation, against the oracle + np.percentile env by env."""
    import torch
    from qdsim import FLAG_LATCH, obs
    from util import oracle_batch
    dev, mb, gv, vgm, origin, sv = _state(3, 4, 3)
    engine.set_models(mb)
    scans = obs.obs_scans(mb, gv, sv, vgm, origin, -1.8, 1.8, 32, peak_width=dev["peak_width"], seeds=np.arange(9) + 5)
    z_dev = torch.empty(9 * 32 * 32, dtype=torch.float32, device="cuda")
    img = obs.observe(engine, scans, z_dev, flags=FLAG_LATCH)
    torch.cuda.synchronize()
    assert img.shape == (3, 3, 32, 32)
    z_ref, _, _ = oracle_batch(mb, scans, FLAG_LATCH)
    z_ref = z_ref.reshape(3, 3, 32, 32)
    for e in range(3):
        p_low, p_high = np.percentile(z_ref[e], 0.5), np.percentile(z_ref[e], 99.5)
        want = np.clip((z_ref[e] - p_low) / (p_high - p_low), 0, 1)
        np.testing.assert_allclose(img[e].cpu().numpy(), want, rtol=0, atol=5e-6)
    assert img.min().item() == 0.0 and img.max().item() == 1.0


@pytest.mark.gpu
def test_batched_env_shell_runs_episodes_on_the_gpu(engine):
    import torch
    from qdsim.vector_env import BatchedDeviceEnv, EnvConfig
    env = BatchedDeviceEnv(48, 4, engine=engine, config=EnvConfig(resolution=24, max_steps=3), seed=5)
    obs0, info = env.reset()
    assert obs0["image"].shape == (48, 3, 24, 24) and obs0["image"].is_cuda
    assert float(obs0["image"].min()) >= 0.0 and float(obs0["image"].max()) <= 1.0
    assert np.abs(obs0["obs_gate_voltages"]).max() <= 1.0 + 1e-6
    rng = np.random.default_rng(0)
    for k in range(3):
        o, r, term, trunc, info = env.step(rng.uniform(-1, 1, (48, 4)), rng.uniform(-1, 1, (48, 3)))
        assert o["image"].shape == (48, 3, 24, 24) and torch.isfinite(o["image"]).all()
        assert r["gates"].shape == (48, 4) and r["barriers"].shape == (48, 3)
        assert ((r["gates"] >= 0) & (r["gates"] <= 1)).all()
        assert trunc.all() == (k == 2) and not term.any()
    # steering every env to its ground truth gives full reward and a structured (non-noise) image
    gt_g = (info["gate_ground_truth"] - env.plunger_min) / (env.plunger_max - env.plunger_min) * 2 - 1
    gt_b = (info["barrier_ground_truth"] - env.barrier_min) / (env.barrier_max - env.barrier_min) * 2 - 1
    o, r, *_ = env.step(gt_g, gt_b)
    assert np.allclose(r["gates"], 1.0) and np.allclose(r["barriers"], 1.0, atol=1e-5)
    # far from the ground truth most scans are replaced by white noise (radial rule), near it none are
    assert (env._scans()["rad_mode"] == 1).all()


def test_agent_views_follow_the_reference_channel_and_transpose_rule():
    """Literal per-env transcription of multi_agent_wrapper.py:147-178, 311-347 vs the batched torch views."""
    import torch
    from qdsim import agents
    n_dot, E, H = 5, 3, 6
    rng = np.random.default_rng(0)
    image = rng.random((E, n_dot - 1, H, H)).astype(np.float32)           # [env, pair, iy, ix]
    obs = {"image": torch.from_numpy(image), "obs_gate_voltages": rng.random((E, n_dot)).astype(np.float32),
           "obs_barrier_voltages": rng.random((E, n_dot - 1)).astype(np.float32)}
    views = agents.agent_observations(obs, n_dot)
    assert list(views) == [f"plunger_{i}" for i in range(5)] + [f"barrier_{j}" for j in range(4)]
    for e in range(E):
        global_image = np.transpose(image[e], (1, 2, 0))                    # the reference's (H, W, N-1)
        for i in range(n_dot):
            ch = [0, 0] if i == 0 else [n_dot - 2, n_dot - 2] if i == n_dot - 1 else [i - 1, i]
            img1, img2 = global_image[:, :, ch[0]], global_image[:, :, ch[1]]
            if i == n_dot - 1:
                img1, img2 = img1.T, img2.T
            elif i != 0:
                img2 = img2.T
            want = np.stack([img1, img2], axis=2)                          # (H, W, 2)
            got = views[f"plunger_{i}"]["image"][e].numpy()                # (2, H, W)
            assert np.array_equal(np.transpose(got, (1, 2, 0)), want)
            assert views[f"plunger_{i}"]["voltage"][e, 0] == obs["obs_gate_voltages"][e, i]
        for j in range(n_dot - 1):
            got = views[f"barrier_{j}"]["image"][e].numpy()
            assert np.array_equal(got[0], global_image[:, :, j])
            assert views[f"barrier_{j}"]["voltage"][e, 0] == obs["obs_barrier_voltages"][e, j]
    # views, not copies, for the single-channel agents
    assert views["barrier_2"]["image"].data_ptr() == obs["image"][:, 2:3].data_ptr()


@pytest.mark.skipif(not os.path.exists(reference_path("qadapt", "utils", "vary_peak_width.py")) and
                    not os.path.exists(reference_path("qadapt", "environment", "utils", "vary_peak_width.py")),
                    reason="reference tree not present")
def test_variable_peak_width_matches_reference_class():
    """obs_scans(peak_width_alpha=...) against the reference's own VaryPeakWidth (utils/vary_peak_width.py), imported
    as it is (pure NumPy)."""
    import glob
    import importlib.util
    from qdsim import obs, synth
    path = glob.glob(reference_path("qadapt", "**", "vary_peak_width.py"), recursive=True)[0]
    spec = importlib.util.spec_from_file_location("ref_vpw", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    e, n = 3, 4
    dev = synth.sample_devices(e, n, seed=9)
    mb = synth.model_batch(dev)
    rng = np.random.default_rng(2)
    gate_v = rng.uniform(-40, 40, size=(e, n))
    alpha = rng.uniform(1e-4, 8e-3, size=e)
    pw0 = dev["peak_width"]
    scans = obs.obs_scans(mb, gate_v, 0.0, np.broadcast_to(-np.eye(n + 1), (e, n + 1, n + 1)), np.zeros((e, n + 1)), -1.5,
                          1.5, 16, peak_width=pw0, peak_width_alpha=alpha)
    for env in range(e):
        ref = mod.VaryPeakWidth(pw0[env], alpha[env])
        for ch in range(n - 1):
            want = ref.linearly_vary_peak_width(gate_v[env, ch], gate_v[env, ch + 1])
            assert scans["peak_width"][env * (n - 1) + ch] == want


@pytest.mark.skipif(not os.path.exists(reference_path("qadapt", "environment", "qarray_base_class.py")),
                    reason="reference tree not present")
def test_radial_noise_descriptor_and_oracle_match_the_reference_method(monkeypatch):
    """S7: QarrayBaseClass._apply_radial_noise (qarray_base_class.py:444-493), compiled from the reference's source text and
    run with np.random.randn replaced by known normals, against obs_scans' radial descriptor + the oracle's radial_noise --
    both branches (additive ramp, full replacement)."""
    import ast
    import types
    from oracle import noise
    from qdsim import obs, synth
    path = reference_path("qadapt", "environment", "qarray_base_class.py")
    tree = ast.parse(open(path).read(), filename=path)
    body = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name == "_apply_radial_noise"]
    ns = {"np": np}
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    res, e, n = 16, 2, 3
    dev = synth.sample_devices(e, n, seed=4)
    mb = synth.model_batch(dev)
    rng = np.random.default_rng(8)
    gt = rng.uniform(-5, 5, size=(e, n))
    gate_v = gt + np.array([[3.0, -25.0, 28.0], [45.0, 2.0, -1.0]])          # env 1, pair 0 lies beyond full_noise_distance
    radial = dict(zero_radius=np.array([22.0, 25.0]), ramp_distance=np.array([30.0, 33.0]),
                  full_noise_distance=np.array([35.0, 38.0]), max_amplitude=0.05)
    window = np.array([1.6, 1.9])
    scans = obs.obs_scans(mb, gate_v, 0.0, np.broadcast_to(-np.eye(n + 1), (e, n + 1, n + 1)), np.zeros((e, n + 1)),
                          -window, window, res, gate_ground_truth=gt, radial=radial, seeds=np.arange(e * (n - 1)))
    normals = rng.standard_normal((res, res))
    monkeypatch.setattr(np.random, "randn", lambda *shape: normals.reshape(shape))
    z = rng.uniform(0.2, 1.0, size=(res, res))
    modes = []
    for env in range(e):
        me = types.SimpleNamespace(radial_noise_config={"enabled": True, "max_amplitude": 0.05},
                                   radial_noise_full_noise_distance=radial["full_noise_distance"][env],
                                   radial_noise_zero_radius=radial["zero_radius"][env],
                                   radial_noise_ramp_distance=radial["ramp_distance"][env],
                                   obs_voltage_min=-window[env], obs_voltage_max=window[env], obs_image_size=res)
        for ch in range(n - 1):
            want = ns["_apply_radial_noise"](me, z, gate_v[env, ch], gate_v[env, ch + 1], gt[env, ch], gt[env, ch + 1])
            rec = scans[env * (n - 1) + ch]
            got = noise.radial_noise(z, normals, int(rec["rad_mode"]), rec["rad_x0"], rec["rad_dx"], rec["rad_y0"],
                                     rec["rad_dy"], rec["rad_alpha"], rec["rad_zero_radius"], rec["rad_max_amp"])
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-14)
            modes.append(int(rec["rad_mode"]))
    assert set(modes) == {1, 2}
