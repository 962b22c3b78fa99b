"""Dot arrays read by several charge sensors on the GPU: the QD_MSENSOR instances of the scan kernel behind every scan and
points entry, the two drop-in classes, and the one-sensor path around them, against the NumPy oracle
(``oracle/multisensor.py``).

Bars: hard-argmin charge maps equal to the oracle's off near-ties (best / second-best margin <= 1e-9; with latching, whole
scans with a near-tie are left out, since one flip runs on along the row); thermal <n> within 1e-9; every z channel within
1e-6 of the oracle (plus the 5e-6 of the fp32 Box-Muller draws when noise is on) where the occupations agree; the tunnel
path per channel with ``util.assert_z_given_n``.
"""
import numpy as np
import pytest
import torch

from oracle import composer
from oracle import multisensor as ms
from qdsim import (FLAG_CARRY_ROWS, FLAG_LATCH, FLAG_NOISE, FLAG_PINK, FLAG_RADIAL, FLAG_THERMAL, FLAG_WHITE_ON_OUTPUT,
                   N_F64, N_U8, QdError, synth)
from qdsim.engine import PARAMS_DTYPE, ModelBatch, new_scans
from util import assert_z_given_n, compare_charges, oracle_model, oracle_scan

pytestmark = pytest.mark.gpu

TIE = 1e-9
Z_RTOL, Z_NOISY_ATOL = 1e-6, 5e-6
N_ATOL, GAP_MIN = 1e-6, 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# inputs and the oracle
# ---------------------------------------------------------------------------------------------------------------------
def ms_batch(n_dot, n_sensor, algorithm="default", thermal=False, res=16, seed=0, n_env=2, offset_range=2.5,
             radial=True, max_charge_carriers=3):
    dev = synth.sample_devices(n_env, n_dot, seed=700 + 11 * n_dot + seed, n_sensor=n_sensor)
    mb = synth.model_batch(dev, algorithm=algorithm, thermal=thermal, latching=True, noise=True,
                           max_charge_carriers=max_charge_carriers)
    mb.params["pink_amp"] = 0.02
    if n_dot >= 2:
        scans = synth.env_step_scans(mb, dev, res=res, seed=seed + 3, offset_range=offset_range, radial=radial)
    else:                                         # one dot: its plunger along x, sensor 0's gate along y
        gt = synth.ground_truth(mb)
        scans = new_scans(n_env)
        scans["v0"][:, :mb.n_gate] = gt
        scans["v0"][:, :2] -= 1.5
        scans["dx"][:, 0] = 3.0 / (res - 1)
        scans["dy"][:, 1] = 0.2 / (res - 1)
        scans["peak_width"] = dev["peak_width"]
        scans["seed"] = np.arange(n_env) + 1000 * seed + 1
        scans["pix_offset"] = np.arange(n_env) * res * res
        scans["env_id"] = np.arange(n_env)
        scans["nx"] = scans["ny"] = res
    return dev, mb, scans


def oracle_ms(mb, scans, flags, n_charge=None):
    """The multi-sensor oracle over every scan: z (S, ny, nx, n_sensor), n (S, ny, nx, N), margin (S, ny, nx)."""
    zs, ns, mgs = [], [], []
    for i, rec in enumerate(scans):
        m = oracle_model(mb, int(rec["env_id"]), flags)
        s = oracle_scan(rec, mb.n_volt, flags)
        kw = dict(carry_rows=bool(flags & FLAG_CARRY_ROWS), white_on="output" if flags & FLAG_WHITE_ON_OUTPUT else "input",
                  return_margin=True)
        if n_charge is None:
            z, n, mg = ms.simulate_scan(m, s, **kw)
        else:
            z, n, mg = ms.simulate_scan_closed(m, int(np.broadcast_to(n_charge, (len(scans),))[i]), s, **kw)
        zs.append(z.reshape(z.shape[:2] + (-1,)))
        ns.append(n)
        mgs.append(mg)
    return np.stack(zs), np.stack(ns), np.stack(mgs)


def per_scan(flat, scans, tail):
    """Host output [pixels(, ...)] -> (n_scan, ny, nx, *tail) (equal-size scans)."""
    ny, nx = int(scans["ny"][0]), int(scans["nx"][0])
    flat = np.asarray(flat).reshape((-1,) + tail)
    return np.stack([flat[int(r["pix_offset"]):int(r["pix_offset"]) + ny * nx].reshape((ny, nx) + tail) for r in scans])


def check(mb, scans, flags, z, n, z_ref, n_ref, margin, thermal=False):
    """Charge maps, <n> and every z channel against the oracle; returns the fraction of pixels compared for z."""
    S = mb.n_sensor
    z = per_scan(z, scans, (S,))
    n = per_scan(n, scans, (mb.n_dot,))
    replaced = np.array([bool(flags & FLAG_RADIAL) and r["rad_mode"] == 2 for r in scans])
    keep = ~replaced
    if thermal:
        np.testing.assert_allclose(n[keep], n_ref[keep], rtol=0, atol=1e-9)
        agree = np.ones(n.shape[:3], dtype=bool)
    else:
        use = keep.copy()
        if flags & FLAG_LATCH:                       # a near-tie flip runs on along a latched row: leave such scans out
            use &= (margin > TIE).reshape(len(scans), -1).all(axis=1)
            assert use[keep].mean() >= 0.5, "too few scans without a near-tie"
        if use.any():
            compare_charges(n[use], n_ref[use], margin[use], tie_tol=TIE)
        agree = (np.rint(n) == np.rint(n_ref)).all(axis=-1)
    agree[replaced] = True
    if replaced.any():
        assert (n[replaced] == 0).all()
    noisy = bool(flags & (FLAG_NOISE | FLAG_PINK | FLAG_RADIAL))
    tol = Z_RTOL * np.abs(z_ref) + (Z_NOISY_ATOL if noisy else 1e-7)
    bad = (np.abs(z - z_ref) > tol) & agree[..., None]
    assert not bad.any(), f"{bad.sum()} z values off, worst {np.abs(z - z_ref)[bad].max():.3e}"
    assert agree.mean() > 0.9
    return agree.mean()


# ---------------------------------------------------------------------------------------------------------------------
# Path A, open: affine windows
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("thermal", [False, True])
@pytest.mark.parametrize("algorithm", ["default", "thresholded", "brute_force"])
@pytest.mark.parametrize("n_dot", range(1, 9))
def test_open_scans_match_the_oracle(engine, n_dot, algorithm, thermal):
    n_sensor = 2 + (n_dot + len(algorithm)) % 3
    dev, mb, scans = ms_batch(n_dot, n_sensor, algorithm, thermal, seed=n_dot,
                              max_charge_carriers=3 if n_dot <= 6 else 2)     # (the oracle walks every candidate)
    assert mb.n_sensor == n_sensor
    engine.set_models(mb)
    # thermal: <n> is compared at 1e-9, so no latching (its rounded compare flips at half-integer <n>)
    flags = FLAG_NOISE | FLAG_RADIAL | FLAG_PINK | (FLAG_THERMAL if thermal else FLAG_LATCH)
    scans["rad_mode"][-1] = 2
    z, n = engine.scan_open_host(scans, flags=flags)
    assert z.shape == (len(scans) * 256, n_sensor)
    z_ref, n_ref, margin = oracle_ms(mb, scans, flags)
    check(mb, scans, flags, z, n, z_ref, n_ref, margin, thermal=thermal)


FLAG_GROUPS = {
    "latch": FLAG_LATCH,
    "white_telegraph": FLAG_NOISE,
    "pink": FLAG_PINK,
    "radial": FLAG_RADIAL,
    "carry_rows": FLAG_CARRY_ROWS | FLAG_LATCH | FLAG_NOISE | FLAG_PINK,
    "white_on_output": FLAG_WHITE_ON_OUTPUT | FLAG_NOISE,
}


@pytest.mark.parametrize("group", sorted(FLAG_GROUPS))
@pytest.mark.parametrize("n_sensor", [2, 3, 4])
def test_flag_groups(engine, n_sensor, group):
    flags = FLAG_GROUPS[group]
    dev, mb, scans = ms_batch(4, n_sensor, res=20, seed=20 + n_sensor)
    mb.params["tele_amp"] = 0.03                 # a telegraph term that shows
    mb.params["tele_p01"] = 0.05
    mb.params["tele_p10"] = 0.08
    engine.set_models(mb)
    if flags & FLAG_RADIAL:
        scans["rad_mode"][::3] = 2
        scans["rad_max_amp"] = 0.2
        scans["rad_zero_radius"] = 0.5
    z, n = engine.scan_open_host(scans, n_type=N_U8, flags=flags)
    z_ref, n_ref, margin = oracle_ms(mb, scans, flags)
    check(mb, scans, flags, z, n, z_ref, n_ref, margin)
    if flags & (FLAG_NOISE | FLAG_PINK):         # every sensor draws its own noise
        zz = per_scan(z, scans, (n_sensor,))
        z_free, _, _ = oracle_ms(mb, scans, 0)
        d = zz - z_free
        assert not np.allclose(d[..., 0], d[..., 1])


@pytest.mark.parametrize("algorithm,thermal", [("default", False), ("default", True), ("brute_force", False),
                                               ("brute_force", True), ("thresholded", False)])
@pytest.mark.parametrize("n_dot", [2, 5])
def test_voltage_lists(engine, n_dot, algorithm, thermal):
    dev, mb, scans = ms_batch(n_dot, 3, algorithm, thermal, seed=40)
    engine.set_models(mb)
    flags = FLAG_NOISE | FLAG_RADIAL | (FLAG_THERMAL if thermal else FLAG_LATCH)
    rec = scans[:1].copy()
    rng = np.random.default_rng(n_dot)
    gt = synth.ground_truth(mb)[0]
    v = gt + rng.uniform(-2.0, 2.0, size=(7, 19, mb.n_gate))
    z, n = engine.points_open_host(rec, v, n_type=N_F64, flags=flags)
    assert z.shape == (7, 19, 3) and n.shape == (7, 19, n_dot)
    m = oracle_model(mb, int(rec[0]["env_id"]), flags)
    s = oracle_scan(rec[0], mb.n_volt, flags)
    z_ref, n_ref, margin = ms.simulate_points(m, v, s, white_on="input", return_margin=True)
    fake = new_scans(1)
    fake["nx"], fake["ny"] = 19, 7
    check(mb, fake, flags, z.reshape(-1, 3), n.reshape(-1, n_dot), z_ref[None], n_ref[None], margin[None],
          thermal=thermal)


# ---------------------------------------------------------------------------------------------------------------------
# closed arrays
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("thermal", [False, True])
@pytest.mark.parametrize("algorithm", ["default", "brute_force"])
@pytest.mark.parametrize("n_dot", [2, 4])
def test_closed_scans(engine, n_dot, algorithm, thermal):
    dev, mb, scans = ms_batch(n_dot, 2, algorithm, thermal, seed=60, offset_range=1.5)
    engine.set_models(mb)
    flags = FLAG_NOISE | FLAG_RADIAL | FLAG_PINK | (FLAG_THERMAL if thermal else FLAG_LATCH)
    q = np.arange(len(scans)) % 3 + n_dot - 1
    z, n = engine.scan_closed_host(scans, q, flags=flags)
    z_ref, n_ref, margin = oracle_ms(mb, scans, flags, n_charge=q)
    check(mb, scans, flags, z, n, z_ref, n_ref, margin, thermal=thermal)
    # voltage list
    rec = scans[:1].copy()
    gt = synth.ground_truth(mb)[0]
    v = gt + np.random.default_rng(3).uniform(-1.5, 1.5, size=(3, 11, mb.n_gate))
    zp, np_ = engine.points_closed_host(rec, int(q[0]), v, n_type=N_F64, flags=flags)
    m = oracle_model(mb, int(rec[0]["env_id"]), flags)
    zr, nr, mg = ms.simulate_points_closed(m, int(q[0]), v, oracle_scan(rec[0], mb.n_volt, flags), return_margin=True)
    fake = new_scans(1)
    fake["nx"], fake["ny"] = 11, 3
    check(mb, fake, flags, zp.reshape(-1, 2), np_.reshape(-1, n_dot), zr[None], nr[None], mg[None], thermal=thermal)


# ---------------------------------------------------------------------------------------------------------------------
# the tunnel path
# ---------------------------------------------------------------------------------------------------------------------
def tunnel_ms_batch(n_dot, n_sensor, barriers, seed, n_env=2, res=12):
    dev = synth.sample_barrier_devices(n_env, n_dot, seed=seed, n_sensor=n_sensor)
    if barriers:
        mb = synth.tunnel_batch(dev)
    else:
        from qdsim import maxwell
        cdd_nm, cgd_nm = maxwell.embed_sensor(dev["Cdd"], dev["Cgd"], dev["Cds"], dev["Cgs"])
        _, cdi_f, cgd_f = maxwell.maxwell(cdd_nm, cgd_nm)
        params = np.zeros(n_env, dtype=PARAMS_DTYPE)
        params["tc_base"] = 0.05
        params["white_amp"], params["tele_p01"], params["tele_p10"] = dev["white_amp"], dev["tele_p01"], dev["tele_p10"]
        params["tele_amp"] = dev["tele_amp"]
        params["latching"] = 1
        params["p_leads"][:, :n_dot] = dev["p_leads"]
        pin = np.zeros((n_env, 8, 8))
        pin[:, :n_dot, :n_dot] = dev["p_inter"]
        params["p_inter"] = pin.reshape(n_env, -1)
        mb = ModelBatch(algorithm="tunnel", n_gate=n_dot + n_sensor, cdd_inv_gs=np.ascontiguousarray(cdi_f[:, :n_dot, :n_dot]),
                        cdd_gs=None, cdd_inv_full=cdi_f, cgd_full=cgd_f, params=params)
    scans = synth.env_step_scans(mb, dev, res=res, seed=seed + 1, offset_range=2.0)
    return mb, scans


@pytest.mark.parametrize("n_dot,n_sensor,barriers", [(3, 2, True), (4, 2, True), (5, 2, True), (6, 2, True),
                                                     (3, 2, False), (4, 2, False), (5, 2, False), (6, 2, False),
                                                     (4, 4, False)])
def test_tunnel_path(engine, n_dot, n_sensor, barriers):
    mb, scans = tunnel_ms_batch(n_dot, n_sensor, barriers, seed=80 + n_dot)
    assert mb.n_sensor == n_sensor
    assert mb.n_volt == (2 * n_dot + n_sensor - 1 if barriers else n_dot + n_sensor)
    engine.set_models(mb)
    for flags in (0, FLAG_LATCH | FLAG_NOISE):
        z, n = engine.scan_open_host(scans, flags=flags)
        z_ref, n_ref, gap = oracle_ms(mb, scans, flags)
        z = per_scan(z, scans, (n_sensor,))
        n = per_scan(n, scans, (n_dot,))
        ok = gap > GAP_MIN
        if flags:                                    # latching: the scans whose pixels are all clear of degeneracies
            ok &= ok.reshape(len(scans), -1).all(axis=1)[:, None, None]
        else:
            assert ok.mean() > 0.5
        np.testing.assert_allclose(n[ok], n_ref[ok], rtol=0, atol=N_ATOL)
        for i, rec in enumerate(scans):
            e = int(rec["env_id"])
            for s in range(n_sensor):
                w = float(np.abs(mb.cdd_inv_full[e, n_dot + s, :n_dot]).max())
                assert_z_given_n(z[i, ..., s], z_ref[i, ..., s], n[i], n_ref[i], ok[i], w, float(rec["peak_width"]),
                                 noise_atol=5e-6 if flags else 0.0, what=f"scan {i} sensor {s}:")


# ---------------------------------------------------------------------------------------------------------------------
# a decoupled second sensor against the one-sensor path
# ---------------------------------------------------------------------------------------------------------------------
def decoupled_batches(n_env, n_dot, seed):
    dev = synth.sample_devices(n_env, n_dot, seed=seed)
    N = n_dot
    kw = dict(p_leads=dev["p_leads"], p_inter=dev["p_inter"], white_amp=dev["white_amp"], tele_p01=dev["tele_p01"],
              tele_p10=dev["tele_p10"], tele_amp=dev["tele_amp"])
    one = ModelBatch.from_capacitances(dev["Cdd"], dev["Cgd"], dev["Cds"], dev["Cgs"], **kw)
    cgs2 = np.zeros((n_env, 2, N + 2))
    cgs2[:, 0, :N + 1] = dev["Cgs"][:, 0]
    cgs2[:, 1, N + 1] = 0.97
    two = ModelBatch.from_capacitances(dev["Cdd"], np.concatenate([dev["Cgd"], np.zeros((n_env, N, 1))], axis=-1),
                                       np.concatenate([dev["Cds"], np.zeros((n_env, 1, N))], axis=1), cgs2, **kw)
    return dev, one, two


def test_decoupled_second_sensor_equals_the_one_sensor_path(engine, monkeypatch):
    """A bench-like batch (8 dots, 64 x 64, latching, noise and radial noise, 448 scans): channel 0 of the two-sensor
    run is the one-sensor run (fast kernel, and the generic kernel) within 1e-6, with identical charge maps."""
    dev, one, two = decoupled_batches(64, 8, seed=901)
    scans = synth.env_step_scans(one, dev, res=64, seed=902, offset_range=5.0)
    scans["rad_mode"][::7] = 2
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    engine.set_models(one)
    z_fast, n_fast = engine.scan_open_host(scans, flags=flags)
    monkeypatch.setenv("QDSIM_GENERIC_SCAN", "1")
    z_gen, n_gen = engine.scan_open_host(scans, flags=flags)
    monkeypatch.delenv("QDSIM_GENERIC_SCAN")
    scans2 = scans.copy()
    scans2["v0"][:, one.n_gate] = 0.4                # the decoupled sensor's own gate
    engine.set_models(two)
    z2, n2 = engine.scan_open_host(scans2, flags=flags)
    assert z2.shape == (len(scans) * 4096, 2)
    for z1, n1 in ((z_fast, n_fast), (z_gen, n_gen)):
        np.testing.assert_array_equal(n2, n1)
        np.testing.assert_allclose(z2[:, 0], z1, rtol=0, atol=1e-6)
    assert np.isfinite(z2).all() and np.abs(z2[:, 1]).max() > 0


# ---------------------------------------------------------------------------------------------------------------------
# layout safety
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_sensor", [2, 3, 4])
def test_ragged_scans_with_gaps_and_canaries(engine, n_sensor):
    dev, mb, _ = ms_batch(3, n_sensor, seed=70)
    engine.set_models(mb)
    gt = synth.ground_truth(mb)
    shapes = [(37, 5), (1, 1), (33, 2), (64, 3), (1, 7), (31, 1)]
    scans = new_scans(len(shapes))
    off = 3
    for i, (nx, ny) in enumerate(shapes):
        e = i % mb.n_env
        scans[i]["v0"][:mb.n_gate] = gt[e]
        scans[i]["v0"][0] -= 1.0
        scans[i]["dx"][0] = 2.0 / nx
        scans[i]["dy"][1] = 2.0 / max(ny, 2)
        scans[i]["nx"], scans[i]["ny"], scans[i]["env_id"] = nx, ny, e
        scans[i]["pix_offset"] = off
        scans[i]["peak_width"] = 0.15
        scans[i]["seed"] = 50 + i
        off += nx * ny + 5                         # a gap of 5 pixels after every scan
    total = off + 9
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_PINK
    zd = torch.full((total, n_sensor), float("nan"), dtype=torch.float32, device="cuda")
    nd = torch.full((total, 3), 255, dtype=torch.uint8, device="cuda")
    engine.scan_open(scans, zd, nd, n_type=N_U8, flags=flags)
    torch.cuda.synchronize()
    assert engine.status() == 0
    zd, nd = zd.cpu().numpy(), nd.cpu().numpy()
    covered = np.zeros(total, dtype=bool)
    for r in scans:
        covered[int(r["pix_offset"]):int(r["pix_offset"]) + int(r["nx"]) * int(r["ny"])] = True
    assert np.isnan(zd[~covered]).all() and (nd[~covered] == 255).all(), "a canary was overwritten"
    assert np.isfinite(zd[covered]).all() and (nd[covered] < 255).all()
    zh, nh = engine.scan_open_host(scans, n_type=N_U8, flags=flags)     # (host outputs end at the last scan's end)
    cov = covered[:len(zh)]
    np.testing.assert_array_equal(zh[cov], zd[:len(zh)][cov])
    np.testing.assert_array_equal(nh[cov], nd[:len(zh)][cov])
    for i, r in enumerate(scans):                  # each scan against the oracle
        o, nx, ny = int(r["pix_offset"]), int(r["nx"]), int(r["ny"])
        m = oracle_model(mb, int(r["env_id"]), flags)
        z_ref, n_ref, mg = ms.simulate_scan(m, oracle_scan(r, mb.n_volt, flags), return_margin=True)
        if (mg > TIE).all():
            np.testing.assert_array_equal(nd[o:o + nx * ny], n_ref.reshape(-1, 3))
            np.testing.assert_allclose(zd[o:o + nx * ny], z_ref.reshape(-1, n_sensor), rtol=Z_RTOL, atol=Z_NOISY_ATOL)
    # the uploaded descriptors, launched again into an offset that breaks the vector alignment: refused
    if n_sensor in (2, 4):
        zbig = torch.zeros(total * n_sensor + 1, dtype=torch.float32, device="cuda")
        with pytest.raises(QdError):
            engine.scan_open(scans, zbig[1:].data_ptr(), None, flags=flags)


def test_one_sensor_outputs_unchanged_around_a_multi_sensor_set(engine):
    from torch.profiler import ProfilerActivity, profile
    dev1, mb1, scans1 = ms_batch(4, 1, res=32, seed=90)
    dev2, mb2, scans2 = ms_batch(4, 2, res=32, seed=90)
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    engine.set_models(mb1)
    with profile(activities=[ProfilerActivity.CUDA]) as p1:
        z_a, n_a = engine.scan_open_host(scans1, flags=flags)
        torch.cuda.synchronize()
    engine.set_models(mb2)
    with profile(activities=[ProfilerActivity.CUDA]) as p2:
        engine.scan_open_host(scans2, flags=flags)
        torch.cuda.synchronize()
    engine.set_models(mb1)
    z_b, n_b = engine.scan_open_host(scans1, flags=flags)
    assert z_a.tobytes() == z_b.tobytes() and n_a.tobytes() == n_b.tobytes()
    names1 = {e.name for e in p1.events() if "qd_scan" in e.name}
    names2 = {e.name for e in p2.events() if "qd_scan" in e.name}
    assert any("qd_scan_fast_kernel<4>" in k for k in names1), names1
    assert any("qd_scan_kernel<4, 32, false, false>" in k for k in names2), names2      # QD_ALG_DEFAULT | QD_MSENSOR


# ---------------------------------------------------------------------------------------------------------------------
# rejections
# ---------------------------------------------------------------------------------------------------------------------
def test_rejections(engine):
    dev, mb, scans = ms_batch(3, 2, seed=95)
    for d in (3, 8):                                 # n_sensor 0 and 5
        bad = ModelBatch(algorithm="default", n_gate=mb.n_gate, cdd_inv_gs=mb.cdd_inv_gs, cdd_gs=mb.cdd_gs,
                         cdd_inv_full=np.tile(np.eye(d), (mb.n_env, 1, 1)), cgd_full=np.zeros((mb.n_env, d, mb.n_gate)),
                         params=mb.params)
        with pytest.raises(QdError) as e:
            engine.set_models(bad)
        assert e.value.code == -1
    tdev = synth.sample_barrier_devices(1, 8, seed=96, n_sensor=2)     # 10 gates + 7 barriers = 17 voltages
    with pytest.raises(QdError) as e:
        engine.set_models(synth.tunnel_batch(tdev))
    assert e.value.code == -1
    engine.set_models(mb)
    with pytest.raises(QdError) as e:
        engine.scan_obs_host(scans, flags=FLAG_NOISE)
    assert e.value.code == -5


# ---------------------------------------------------------------------------------------------------------------------
# the drop-in classes
# ---------------------------------------------------------------------------------------------------------------------
CDD = [[0, .12], [.12, 0]]
CGD = [[1.0, .35, 0, 0], [.3, .97, 0, 0]]
CDS = [[.04, .045], [.05, .02]]
CGS = [[6e-5, 3e-5, .98, .01], [2e-5, 5e-5, .02, .96]]


def test_charge_sensed_dot_array_two_sensors():
    import qarray
    from oracle import sensor
    m = qarray.ChargeSensedDotArray(Cdd=CDD, Cgd=CGD, Cds=CDS, Cgs=CGS, coulomb_peak_width=0.15, algorithm="default",
                                    implementation="jax")
    assert m.n_sensor == 2 and m.cdd_inv_full.shape == (4, 4)
    z, n = m.do2d_open(1, -3.0, 1.0, 24, 2, -3.0, 1.0, 20)
    assert z.shape == (20, 24, 2) and n.shape == (20, 24, 2)
    vg = composer.do2d(4, 1, -3.0, 1.0, 24, 2, -3.0, 1.0, 20)
    z_ref = sensor.charge_sensor_signal(n.reshape(-1, 2), vg.reshape(-1, 4), m.cdd_inv_full, m.cgd_full, 0.15)
    np.testing.assert_allclose(z.reshape(-1, 2), z_ref, rtol=1e-6, atol=1e-7)
    n_gs = m.ground_state_open(vg)
    np.testing.assert_array_equal(n_gs, n)
    z1, n1 = m.charge_sensor_open(vg[3])
    assert z1.shape == (24, 2)
    np.testing.assert_allclose(z1, z[3], rtol=1e-6, atol=1e-7)
    zd, nd1 = m.do1d_open(1, -3.0, 1.0, 17)
    assert zd.shape == (17, 2) and nd1.shape == (17, 2)
    zc, nc = m.do2d_closed(1, -3.0, 1.0, 24, 2, -3.0, 1.0, 20, 2)
    assert zc.shape == (20, 24, 2) and (nc.sum(axis=-1) == 2).all()
    zc_ref = sensor.charge_sensor_signal(nc.reshape(-1, 2), vg.reshape(-1, 4), m.cdd_inv_full, m.cgd_full, 0.15)
    np.testing.assert_allclose(zc.reshape(-1, 2), zc_ref, rtol=1e-6, atol=1e-7)
    z1c, n1c = m.charge_sensor_closed(vg[3], 2)
    np.testing.assert_array_equal(n1c, nc[3])
    assert z1c.shape == (24, 2)
    assert m.ground_state_closed(vg, 2).shape == (20, 24, 2)
    zdc, _ = m.do1d_closed(1, -3.0, 1.0, 9, 1)
    assert zdc.shape == (9, 2)
    target = np.array([1.0, 2.0, 0.5, 0.5])
    vopt = m.optimal_Vg(target)
    assert vopt.shape == (4,)
    np.testing.assert_allclose(m.cgd_full @ vopt, target, atol=1e-6)      # four gates reach any four occupations
    assert m.compute_optimal_virtual_gate_matrix().shape == (4, 4)


def test_tunnel_coupled_charge_sensed_two_sensors():
    from qarray_latched import TunnelCoupledChargeSensed
    from oracle import sensor
    m = TunnelCoupledChargeSensed(Cdd=CDD, Cgd=CGD, Cds=CDS, Cgs=CGS, coulomb_peak_width=0.15, num_charge_states=32,
                                  tc=0.05)
    assert m.n_sensor == 2
    vg = composer.do2d(4, 1, -3.0, 1.0, 12, 2, -3.0, 1.0, 10)
    z, n = m.charge_sensor_open(vg)
    assert z.shape == (10, 12, 2) and n.shape == (10, 12, 2)
    z_ref = sensor.charge_sensor_signal(n.reshape(-1, 2), vg.reshape(-1, 4), m.cdd_inv_full, m.cgd_full, 0.15)
    np.testing.assert_allclose(z.reshape(-1, 2), z_ref, rtol=1e-6, atol=1e-7)
    assert m.do2d_open(1, -3.0, 1.0, 12, 2, -3.0, 1.0, 10)[0].shape == (10, 12, 2)
    assert m.do1d_open(1, -3.0, 1.0, 7)[0].shape == (7, 2)
    assert m.optimal_Vg(np.array([1.0, 1.0, 0.5, 0.5])).shape == (4,)
