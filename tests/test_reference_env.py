"""The REAL reference ``QuantumDeviceEnv`` (src/qadapt/environment/env.py) running reset() / step() UNCHANGED on top of
our drop-in ``qarray`` / ``qarray_latched`` packages (north_star: "src/qadapt's env ... run unchanged on top").
Needs the upstream ``src`` tree (``QADAPT_SRC``); the engine is the CPU oracle here, see tests/ref_harness.py."""
import os

import numpy as np
import pytest
import yaml

import ref_harness

needs_reference = pytest.mark.skipif(not os.path.isdir(ref_harness.REF), reason="reference tree not present")


def _config(tmp_path, num_dots=4, res=10, update_method=None):
    cfg = yaml.safe_load(open(os.path.join(ref_harness.REF, "qadapt/environment/env_config.yaml")))
    cfg["simulator"]["num_dots"] = num_dots
    cfg["simulator"]["resolution"] = res
    cfg["simulator"]["max_steps"] = 3
    cfg["capacitance_model"]["update_method"] = update_method
    path = tmp_path / "env_config.yaml"
    path.write_text(yaml.safe_dump(cfg))
    return str(path)


# update_method "fake" is bit-rotted in the reference itself for barrier models: fake_capacitance_model returns the
# (N, N+1) model.cgd, which QarrayBaseClass._update_virtual_gate_matrix then fails to hstack (qarray_base_class.py:922);
# "kalman" / "direct" need the CNN checkpoint.
@needs_reference
@pytest.mark.parametrize("update_method", [None, "perfect"])
def test_reference_env_reset_and_step_run_unchanged(monkeypatch, tmp_path, update_method):
    base, envmod, eng = ref_harness.install(monkeypatch)
    import qarray_latched
    np.random.seed(3)
    env = envmod.QuantumDeviceEnv(config_path=_config(tmp_path, update_method=update_method))
    assert isinstance(env.array.model, qarray_latched.TunnelCoupledChargeSensed)
    obs, info = env.reset()
    assert obs["image"].shape == (10, 10, 3) and obs["image"].dtype == np.float32
    assert 0.0 <= obs["image"].min() and obs["image"].max() <= 1.0
    launches = eng.launch_count
    for _ in range(3):
        action = {"action_gate_voltages": np.random.uniform(-1, 1, 4), "action_barrier_voltages": np.random.uniform(-1, 1, 3)}
        obs, reward, terminated, truncated, info = env.step(action)
        assert obs["image"].shape == (10, 10, 3) and np.isfinite(obs["image"]).all()
        assert reward["gates"].shape == (4,) and reward["barriers"].shape == (3,)
        assert obs["obs_gate_voltages"].shape == (4,) and np.abs(obs["obs_gate_voltages"]).max() <= 1 + 1e-6
    assert truncated and not terminated
    assert eng.launch_count == launches + 9            # three steps x (N-1) scans through charge_sensor_open(vg_flat, vb)
    state = info["current_device_state"]
    assert state["virtual_gate_matrix"].shape == (5, 5) and len(state["gate_ground_truth"]) == 4


@needs_reference
def test_batched_env_shell_matches_the_reference_env_logic(monkeypatch, tmp_path):
    """BatchedDeviceEnv (qdsim/vector_env.py) against the REAL QuantumDeviceEnv on the same device and ranges:
    ground truth, action rescale, rewards, the scan windows it would launch, the radial-noise amplitude field."""
    base, envmod, eng = ref_harness.install(monkeypatch)
    from oracle import composer, noise
    from qdsim import synth
    from qdsim.vector_env import BatchedDeviceEnv, EnvConfig
    np.random.seed(11)
    env = envmod.QuantumDeviceEnv(config_path=_config(tmp_path, res=8, update_method="perfect"))
    m, arr = env.array.model, env.array
    N, B = 4, 3
    b = BatchedDeviceEnv(1, N, engine=None, config=EnvConfig(resolution=8, max_steps=3, update_method="perfect"))
    noise_p = m.noise_model._kernel_params()
    b.dev = {"Cdd": m.Cdd[None], "Cgd": m.Cgd[None], "Cds": m.Cds[None], "Cgs": m.Cgs[None], "Cbd": m.Cbd[None],
             "Cbg": m.Cbg[None], "Cbs": m.Cbs[None], "tc_base": np.array([arr.barrier_tc_base]),
             "alpha": np.array([arr.barrier_alpha]), "peak_width": np.array([m.coulomb_peak_width]),
             "p_leads": m.latching_model.p_leads[None], "p_inter": m.latching_model.p_inter[None],
             "white_amp": np.array([noise_p["white_amp"]]), "tele_p01": np.array([noise_p["tele_p01"]]),
             "tele_p10": np.array([noise_p["tele_p10"]]), "tele_amp": np.array([noise_p["tele_amp"]])}
    b.mb = synth.tunnel_batch(b.dev)
    assert np.allclose(b.mb.cgd_full[0], m.cgd_full) and np.allclose(b.mb.cdd_inv_full[0], m.cdd_inv_full)
    b.window_delta = np.array([env.window_delta])
    b.radial = dict(zero_radius=np.array([arr.radial_noise_zero_radius]),
                    ramp_distance=np.array([arr.radial_noise_ramp_distance]),
                    full_noise_distance=np.array([arr.radial_noise_full_noise_distance]), max_amplitude=0.05)
    b.vgm = m.gate_voltage_composer.virtual_gate_matrix[None].copy()
    b.origin = m.gate_voltage_composer.virtual_gate_origin[None].copy()
    b.plunger_min, b.plunger_max = env.plunger_min[None], env.plunger_max[None]
    b.barrier_min, b.barrier_max = env.barrier_min[None], env.barrier_max[None]
    b.step_count, b._episode = 0, 1
    # "perfect" virtual gate matrix as the reference sets it
    import qdsim.maxwell as mx
    assert np.allclose(b.vgm[0], -mx.optimal_vgm(m.cdd_inv_full, m.cgd_full[:, :5]))
    # ground truth
    gt_g, gt_b, gt_s = b._ground_truth()
    st = env.device_state
    np.testing.assert_allclose(gt_g[0], st["gate_ground_truth"], rtol=1e-5)
    np.testing.assert_allclose(gt_b[0], st["barrier_ground_truth"], rtol=1e-5)
    np.testing.assert_allclose(gt_s[0], st["sensor_ground_truth"], rtol=1e-9)
    b.gate_gt, b.barrier_gt, b.sensor_gt = gt_g, gt_b, gt_s
    # step: rescale + reward
    rng = np.random.default_rng(0)
    for _ in range(2):
        ga, ba = rng.uniform(-1.2, 1.2, N), rng.uniform(-1.2, 1.2, B)
        _, reward, term, trunc, info = env.step({"action_gate_voltages": ga, "action_barrier_voltages": ba}, skip_obs=True)
        _, r2, t2, tr2, i2 = b.step(ga[None], ba[None], skip_obs=True)
        np.testing.assert_allclose(i2["current_gate_voltages"][0], info["current_device_state"]["current_gate_voltages"], rtol=1e-6)
        np.testing.assert_allclose(i2["current_barrier_voltages"][0], info["current_device_state"]["current_barrier_voltages"], rtol=1e-6)
        np.testing.assert_allclose(r2["gates"][0], reward["gates"], rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(r2["barriers"][0], reward["barriers"], rtol=1e-5, atol=1e-7)
        assert bool(tr2[0]) == trunc and bool(t2[0]) == term
    # the scan windows of the next observation == the grids the facade builds (qarray_base_class.py:143-154)
    scans = b._scans()
    gv = info["current_device_state"]["current_gate_voltages"]
    wd = env.window_delta
    for c in range(3):
        rec = scans[c]
        want = m.gate_voltage_composer.do2d(f"vP{c + 1}", gv[c] - wd, gv[c] + wd, 8, f"vP{c + 2}", gv[c + 1] - wd,
                                            gv[c + 1] + wd, 8, np.append(gv, st["sensor_ground_truth"]), True)
        got = composer.affine_grid(rec["v0"][:5], rec["dx"][:5], rec["dy"][:5], 8, 8)
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6)
        assert np.allclose(rec["v0"][5:8], info["current_device_state"]["current_barrier_voltages"])
        # radial-noise amplitude field == the facade's (np.random.randn forced to ones turns its output into amplitude)
        monkeypatch.setattr(np.random, "randn", lambda *shape: np.ones(shape))
        arr.gate_ground_truth = st["gate_ground_truth"]
        ref_amp = arr._apply_radial_noise(np.zeros((8, 8)), float(gv[c]), float(gv[c + 1]),
                                          float(st["gate_ground_truth"][c]), float(st["gate_ground_truth"][c + 1]))
        monkeypatch.undo() if False else None
        ours = noise.radial_noise(np.zeros((8, 8)), np.ones(64), int(rec["rad_mode"]), float(rec["rad_x0"]),
                                  float(rec["rad_dx"]), float(rec["rad_y0"]), float(rec["rad_dy"]), float(rec["rad_alpha"]),
                                  float(rec["rad_zero_radius"]), float(rec["rad_max_amp"]))
        np.testing.assert_allclose(ours, ref_amp, rtol=1e-5, atol=1e-7)


def test_reward_curves_cover_every_branch():
    from qdsim.vector_env import EnvConfig, barrier_reward, gate_reward
    d = np.array([0.0, 0.5, 1.0, 1.5, 20.0, 40.0, 60.0])
    assert np.allclose(gate_reward(d, EnvConfig()), [1, 1, 1, 0.5 * 38.5 / 39, 0.5 * 20 / 39, 0, 0])
    assert np.allclose(gate_reward(d, EnvConfig(gate_curve_type="linear"))[:3], [1, 0.75, 0.5])
    assert np.allclose(gate_reward(d, EnvConfig(gate_curve_type="polynomial"))[:3], [1, 0.625, 0.5])
    sparse = gate_reward(np.array([1.0, 2.0, 6.0, 10.0, 11.0]), EnvConfig(sparse_reward=True))
    assert np.allclose(sparse, [1, 1, 0.25, 0, 0])
    assert np.allclose(barrier_reward(np.array([0, 3, 6, 9.0]), EnvConfig()), [1, 0.5, 0, 0])
    assert np.allclose(barrier_reward(np.array([0, 2, 2.1]), EnvConfig(sparse_reward=True)), [1, 1, 0])
