"""Several charge sensors, CPU side: the per-sensor random streams and the oracle's multi-sensor scan
(``oracle/multisensor.py``) against the one-sensor oracle and against the closed form of the signal.

* Philox streams with ``sensor=0`` are the one-sensor streams for every purpose; sensors 1..3 draw other numbers.
* A second sensor that no dot and no other gate sees leaves channel 0 equal to the one-sensor oracle, with noise,
  latching and radial noise on.
* Swapping two sensors together with their rows and gates swaps the channels (noise-free).
* ``dPhi^s_k = C_ss (2 (t_s + k) + 1) + 2 sum_j C_sj e_j + 2 sum_{o != s} C_so t_o``, evaluated on its own, gives
  ``charge_sensor_signal`` at 2..4 sensors.
* The occupations do not depend on the sensor count.
"""
import numpy as np
import pytest

from oracle import multisensor as ms
from oracle import noise, philox, sensor
from oracle import scan as oscan
from qdsim import maxwell, synth
from qdsim.engine import ModelBatch


def ms_batch(n_dot, n_sensor, seed=0, n_env=1, algorithm="default", thermal=False):
    dev = synth.sample_devices(n_env, n_dot, seed=500 + seed, n_sensor=n_sensor)
    mb = synth.model_batch(dev, algorithm=algorithm, thermal=thermal, latching=True, noise=True)
    return dev, mb


def model(mb, e=0, pink=0.0, noisy=True):
    p = mb.params[e]
    n = mb.n_dot
    return oscan.Model(
        cdd_inv=mb.cdd_inv_gs[e], cdd=mb.cdd_gs[e], cgd=mb.cgd_full[e, :n], cdd_inv_full=mb.cdd_inv_full[e],
        cgd_full=mb.cgd_full[e], algorithm=mb.algorithm, kT=float(p["kT"]), latching=bool(p["latching"]),
        p_leads=p["p_leads"][:n].copy(), p_inter=p["p_inter"].reshape(8, 8)[:n, :n].copy(),
        white_amp=float(p["white_amp"]) if noisy else 0.0, tele_p01=float(p["tele_p01"]), tele_p10=float(p["tele_p10"]),
        tele_amp=float(p["tele_amp"]) if noisy else 0.0, pink_amp=pink if noisy else 0.0)


def window(mb, res=12, seed=1, rad_mode=1):
    """A 2-d window over the first two plungers (the first plunger alone for one dot) around the ground truth."""
    gt = synth.ground_truth(mb)[0]
    v0 = gt.copy()
    dx = np.zeros_like(gt)
    dy = np.zeros_like(gt)
    v0[0] -= 1.5
    dx[0] = 3.0 / (res - 1)
    j = 1 if mb.n_dot > 1 else mb.n_dot
    v0[j] -= 1.5 if mb.n_dot > 1 else 0.1
    dy[j] = (3.0 if mb.n_dot > 1 else 0.2) / (res - 1)
    return oscan.Scan(v0=v0, dx=dx, dy=dy, nx=res, ny=res, peak_width=0.15, seed=seed, rad_mode=rad_mode,
                      rad=(-1.0, 0.3, -0.5, 0.3, 0.02, 0.5, 0.05))


# ---------------------------------------------------------------------------------------------------------------------
# random streams
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("purpose", [0, 1, 2, 3])
def test_sensor_zero_stream_is_the_one_sensor_stream(purpose):
    idx = np.arange(0, 5000, 7, dtype=np.uint64) + np.uint64(1 << 33)
    for a, b in zip(ms.words(0xDEADBEEF12345, idx, purpose), philox.words(0xDEADBEEF12345, idx, purpose)):
        np.testing.assert_array_equal(a, b)
    others = [np.stack(ms.words(0xDEADBEEF12345, idx, purpose, s)) for s in range(4)]
    for s in range(4):
        for o in range(s):
            assert (others[s] != others[o]).mean() > 0.99


def test_sensor_zero_draws_are_the_one_sensor_draws():
    d0, d = ms.pixel_draws(77, 999), philox.pixel_draws(77, 999)
    for k in d:
        np.testing.assert_array_equal(d0[k], d[k])
    np.testing.assert_array_equal(ms.row_draws(77, 33), philox.row_draws(77, 33))
    for carry in (False, True):
        np.testing.assert_array_equal(ms.pink_noise(77, 5, 40, carry), noise.pink_noise(77, 5, 40, carry))
    for s in (1, 2, 3):
        assert not np.array_equal(ms.pixel_draws(77, 999, s)["z_white"], d["z_white"])
        assert not np.array_equal(ms.row_draws(77, 33, s), philox.row_draws(77, 33))
        assert not np.array_equal(ms.pink_noise(77, 5, 40, sensor=s), noise.pink_noise(77, 5, 40))


# ---------------------------------------------------------------------------------------------------------------------
# the scan
# ---------------------------------------------------------------------------------------------------------------------
def decoupled_pair(n_dot, seed=0):
    """A one-sensor batch and the same device with a second sensor that sees neither the dots nor the other gates."""
    dev = synth.sample_devices(1, n_dot, seed=600 + seed)
    N = n_dot
    cgd2 = np.concatenate([dev["Cgd"], np.zeros((1, N, 1))], axis=-1)
    cds2 = np.concatenate([dev["Cds"], np.zeros((1, 1, N))], axis=1)
    cgs2 = np.zeros((1, 2, N + 2))
    cgs2[:, 0, :N + 1] = dev["Cgs"][:, 0]
    cgs2[:, 1, N + 1] = 0.97
    kw = dict(p_leads=dev["p_leads"], p_inter=dev["p_inter"], white_amp=dev["white_amp"], tele_p01=dev["tele_p01"],
              tele_p10=dev["tele_p10"], tele_amp=dev["tele_amp"])
    one = ModelBatch.from_capacitances(dev["Cdd"], dev["Cgd"], dev["Cds"], dev["Cgs"], **kw)
    two = ModelBatch.from_capacitances(dev["Cdd"], cgd2, cds2, cgs2, **kw)
    return one, two


@pytest.mark.parametrize("n_dot", [1, 2, 4])
@pytest.mark.parametrize("white_on", ["input", "output"])
def test_decoupled_second_sensor_leaves_channel_zero(n_dot, white_on):
    one, two = decoupled_pair(n_dot)
    assert two.n_sensor == 2
    np.testing.assert_allclose(two.cdd_inv_full[0, :n_dot + 1, :n_dot + 1], one.cdd_inv_full[0], rtol=1e-14, atol=0)
    for rad_mode in (1, 2):
        s1 = window(one, rad_mode=rad_mode)
        s2 = oscan.Scan(v0=np.append(s1.v0, 0.3), dx=np.append(s1.dx, 0.0), dy=np.append(s1.dy, 0.0), nx=s1.nx,
                        ny=s1.ny, peak_width=s1.peak_width, seed=s1.seed, rad_mode=rad_mode, rad=s1.rad)
        z1, n1 = oscan.simulate_scan(model(one, pink=0.05), s1, carry_rows=True, white_on=white_on)
        z2, n2 = ms.simulate_scan(model(two, pink=0.05), s2, carry_rows=True, white_on=white_on)
        assert z2.shape == (12, 12, 2)
        np.testing.assert_array_equal(n2, n1)
        np.testing.assert_allclose(z2[..., 0], z1, rtol=0, atol=1e-12)
        # the one-sensor call of the multi-sensor oracle is the one-sensor oracle
        z1m, n1m = ms.simulate_scan(model(one, pink=0.05), s1, carry_rows=True, white_on=white_on)
        np.testing.assert_array_equal(z1m, z1)
        np.testing.assert_array_equal(n1m, n1)


@pytest.mark.parametrize("n_dot", [2, 3])
def test_swapping_sensors_swaps_channels(n_dot):
    dev, mb = ms_batch(n_dot, 2, seed=n_dot)
    N = n_dot
    perm = list(range(N)) + [N + 1, N]
    cgd = dev["Cgd"][..., perm]
    cds = dev["Cds"][:, ::-1]
    cgs = dev["Cgs"][:, ::-1][..., perm]
    mb_sw = ModelBatch.from_capacitances(dev["Cdd"], cgd, cds, cgs, p_leads=dev["p_leads"], p_inter=dev["p_inter"])
    s = window(mb, rad_mode=0)
    s_sw = oscan.Scan(v0=s.v0[perm], dx=s.dx[perm], dy=s.dy[perm], nx=s.nx, ny=s.ny, peak_width=s.peak_width, seed=s.seed)
    z, n = ms.simulate_scan(model(mb, noisy=False), s)
    z_sw, n_sw = ms.simulate_scan(model(mb_sw, noisy=False), s_sw)
    np.testing.assert_array_equal(n_sw, n)
    np.testing.assert_allclose(z_sw[..., ::-1], z, rtol=1e-12, atol=1e-12)
    assert np.abs(z[..., 0] - z[..., 1]).max() > 1e-3          # the two sensors do see different signals


def delta_phi_signal(n, v, cdd_inv_full, cgd_full, gamma, xi, eta):
    """The closed form of the signal of every sensor, (P, N), (P, NV) -> (P, S)."""
    N = n.shape[-1]
    S = cdd_inv_full.shape[0] - N
    u = v @ cgd_full.T
    e = n - u[:, :N]
    t = np.rint(u[:, N:]) + xi - u[:, N:]
    C = cdd_inv_full
    z = np.zeros((n.shape[0], S))
    for s in range(S):
        cross = sum(C[N + s, N + o] * t[:, o] for o in range(S) if o != s)
        base = 2.0 * (e @ C[N + s, :N]) + 2.0 * cross
        for k in range(-5, 5):
            dphi = C[N + s, N + s] * (2.0 * (t[:, s] + k) + 1.0) + base
            z[:, s] += 1.0 / (1.0 + (dphi / gamma) ** 2)
    return z + eta


@pytest.mark.parametrize("n_sensor", [2, 3, 4])
def test_closed_form_matches_charge_sensor_signal(n_sensor):
    dev, mb = ms_batch(3, n_sensor, seed=n_sensor)
    rng = np.random.default_rng(n_sensor)
    gt = synth.ground_truth(mb)[0]
    v = gt + rng.uniform(-2.0, 2.0, size=(400, gt.size))
    n = rng.integers(0, 3, size=(400, 3)).astype(np.float64)
    xi = rng.normal(0.0, 0.05, size=(400, n_sensor))
    eta = rng.normal(0.0, 0.01, size=(400, n_sensor))
    ref = sensor.charge_sensor_signal(n, v, mb.cdd_inv_full[0], mb.cgd_full[0], 0.12, input_noise=xi, output_noise=eta)
    got = delta_phi_signal(n, v, mb.cdd_inv_full[0], mb.cgd_full[0], 0.12, xi, eta)
    assert ref.shape == (400, n_sensor)
    np.testing.assert_allclose(got, ref, rtol=1e-9, atol=1e-9)
    # the cross term matters: dropping it changes the signal
    C = mb.cdd_inv_full[0]
    assert np.abs(C[3:, 3:] - np.diag(np.diag(C[3:, 3:]))).max() > 0


@pytest.mark.parametrize("algorithm", ["default", "brute_force"])
def test_occupations_do_not_depend_on_the_sensor_count(algorithm):
    for n_sensor in (1, 2, 4):
        dev, mb = ms_batch(3, n_sensor, seed=9, algorithm=algorithm)
        m = model(mb)
        m.max_charge_carriers = 4
        s = window(mb, rad_mode=0)
        z, n = ms.simulate_scan(m, s)
        if n_sensor == 1:
            n_ref = n
            assert z.shape == (12, 12)
        else:
            assert z.shape == (12, 12, n_sensor)
            np.testing.assert_array_equal(n, n_ref)


def test_embedding_takes_every_sensor_row():
    dev, mb = ms_batch(3, 3, n_env=2)
    cdd_nm, cgd_nm = maxwell.embed_sensor(dev["Cdd"], dev["Cgd"], dev["Cds"], dev["Cgs"])
    assert cdd_nm.shape == (2, 6, 6) and cgd_nm.shape == (2, 6, 6)
    np.testing.assert_array_equal(cdd_nm[:, 3:, :3], dev["Cds"])
    np.testing.assert_array_equal(cgd_nm[:, 3:], dev["Cgs"])
    assert mb.n_sensor == 3 and mb.cgd_full.shape == (2, 6, 6)
    # the sensor rows of the one-sensor device are unchanged by the extra sensors
    one = synth.sample_devices(2, 3, seed=500)
    np.testing.assert_array_equal(dev["Cds"][:, :1], one["Cds"])
    np.testing.assert_array_equal(dev["Cgs"][:, 0, :4], one["Cgs"][:, 0])


# ---------------------------------------------------------------------------------------------------------------------
# the drop-in classes, host side (no GPU: construction, Maxwell matrices, optimal voltages, refusals)
# ---------------------------------------------------------------------------------------------------------------------
CDD = [[0, .12], [.12, 0]]
CGD = [[1.0, .35, 0, 0], [.3, .97, 0, 0]]
CDS = [[.04, .045], [.05, .02]]
CGS = [[6e-5, 3e-5, .98, .01], [2e-5, 5e-5, .02, .96]]


def test_drop_ins_take_two_sensors():
    import qarray
    from qarray_latched import TunnelCoupledChargeSensed
    for m in (qarray.ChargeSensedDotArray(Cdd=CDD, Cgd=CGD, Cds=CDS, Cgs=CGS, algorithm="default", implementation="jax"),
              TunnelCoupledChargeSensed(Cdd=CDD, Cgd=CGD, Cds=CDS, Cgs=CGS, num_charge_states=32)):
        assert m.n_sensor == 2 and m.cdd_inv_full.shape == (4, 4) and m.cgd_full.shape == (4, 4)
        target = np.array([1.0, 2.0, 0.5, 0.5])
        v = m.optimal_Vg(target)
        np.testing.assert_allclose(m.cgd_full @ v, target, atol=1e-6)   # four gates reach any four occupations
        assert m.compute_optimal_virtual_gate_matrix().shape == (4, 4)


def test_drop_ins_refuse_five_sensors_and_too_many_voltages():
    import qarray
    from qarray_latched import TunnelCoupledChargeSensed
    cds = np.full((5, 2), 0.04)
    cgs = np.hstack([np.full((5, 2), 1e-5), 0.9 * np.eye(5)])
    cgd = np.hstack([np.asarray(CGD)[:, :2], np.zeros((2, 5))])
    with pytest.raises(NotImplementedError, match="1..4 charge sensors"):
        qarray.ChargeSensedDotArray(Cdd=CDD, Cgd=cgd, Cds=cds, Cgs=cgs, algorithm="default", implementation="jax")
    with pytest.raises(NotImplementedError, match="1..4 charge sensors"):
        TunnelCoupledChargeSensed(Cdd=CDD, Cgd=cgd, Cds=cds, Cgs=cgs, num_charge_states=32)
    dev = synth.sample_barrier_devices(1, 8, seed=3, n_sensor=2)          # 10 gates + 7 barriers = 17 voltages
    with pytest.raises(ValueError, match="at most 16"):
        TunnelCoupledChargeSensed(Cdd=dev["Cdd"][0], Cgd=dev["Cgd"][0], Cds=dev["Cds"][0], Cgs=dev["Cgs"][0],
                                  Cbd=dev["Cbd"][0], Cbg=dev["Cbg"][0], Cbs=dev["Cbs"][0], num_charge_states=32)
