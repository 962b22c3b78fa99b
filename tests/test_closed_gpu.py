"""Closed arrays (fixed total charge per scan) on the GPU: qd_scan_closed / qd_scan_closed_host / qd_points_closed_host and
the closed methods of ``ChargeSensedDotArray``, against the plain-C restatement (``qd_cport_scans_closed``) and the NumPy
oracle (``oracle.closed.ground_state_closed``).

Covered: 1..8 dots, ``default`` and ``brute_force``, T = 0 and T > 0, affine batches with a different total charge per
scan, explicit voltage lists; windows where the closed relaxation clamps dots and where it clamps none, candidate weights
k = 0 and k = N - 1, Q = 0 and (brute force) Q = 15; latching, carry-rows, noise, 1/f and radial noise; the drop-in class;
the open path of the same engine before and after closed calls.  Every case first asserts that it reaches what it is named
for (host-side predicates on the oracle's closed relaxation).

Bars: hard argmin equal to the C restatement except at near-ties (best / second-best margin <= 1e-9, or a relaxed
occupation within 1e-9 of an integer: the two relaxations may floor it differently), which are counted and bounded;
latched outputs compared on the rows where the unlatched ones agree; sum n = Q exactly at T = 0, to 1e-9 at T > 0; thermal
<n> within 1e-9; z within 1e-6 relative when noise-free, 5e-6 absolute with noise.
"""
import numpy as np
import pytest

from oracle import closed, composer, path_a
from qdsim import (FLAG_CARRY_ROWS, FLAG_LATCH, FLAG_NOISE, FLAG_PINK, FLAG_RADIAL, FLAG_THERMAL, N_F64, N_U8, QdError,
                   synth)
from qdsim.engine import new_scans
from util import oracle_model, oracle_scan

pytestmark = pytest.mark.gpu

TIE = 1e-9
MAX_TIE_FRAC = 0.005
Z_RTOL, Z_NOISY_ATOL = 1e-6, 5e-6


# ---------------------------------------------------------------------------------------------------------------------
# inputs and host-side reach predicates
# ---------------------------------------------------------------------------------------------------------------------
def closed_batch(n_dot, algorithm="default", thermal=False, res=16, seed=0, n_env=2, offset_range=2.0, radial=True):
    dev = synth.sample_devices(n_env, n_dot, seed=300 + 7 * n_dot + seed)
    mb = synth.model_batch(dev, algorithm=algorithm, thermal=thermal, latching=True, noise=True)
    mb.params["pink_amp"] = 0.02
    if n_dot >= 2:
        scans = synth.env_step_scans(mb, dev, res=res, seed=seed + 11, offset_range=offset_range, radial=radial)
    else:                                         # one dot: its plunger along x, the sensor gate along y
        gt = synth.ground_truth(mb)
        scans = new_scans(n_env)
        scans["v0"][:, :2] = gt[:, :2] - 1.5
        scans["dx"][:, 0] = 3.0 / (res - 1)
        scans["dy"][:, 1] = 0.2 / (res - 1)
        scans["peak_width"] = dev["peak_width"]
        scans["seed"] = np.arange(n_env) + 1000 * seed
        scans["pix_offset"] = np.arange(n_env) * res * res
        scans["env_id"] = np.arange(n_env)
        scans["nx"] = scans["ny"] = res
    return mb, scans


def relaxed(mb, scans, q):
    """The oracle's closed relaxation of every pixel, (S, ny, nx, N)."""
    out = []
    for i, rec in enumerate(scans):
        e, nv = int(rec["env_id"]), mb.n_volt
        v = composer.affine_grid(rec["v0"][:nv], rec["dx"][:nv], rec["dy"][:nv], int(rec["nx"]), int(rec["ny"]))
        g = v.reshape(-1, nv) @ mb.cgd_full[e, :mb.n_dot].T
        out.append(closed.continuous_relaxation_closed(g, mb.cdd_gs[e], mb.cdd_inv_gs[e], int(q[i])).reshape(
            int(rec["ny"]), int(rec["nx"]), mb.n_dot))
    return np.stack(out)


def near_integer(nc):
    """Pixels with a relaxed occupation within 1e-9 of an integer (other than an exact 0: a clamped dot is 0 exactly)."""
    frac = np.abs(nc - np.rint(nc))
    return ((frac <= 1e-9) & (nc > 1e-9)).any(axis=-1)


def cport(mb, scans, q, flags):
    from oracle.cport import closed as cp
    z, n, _, margin = cp.run_scans_closed(mb, scans, q, flags, want_margin=True)
    S, ny, nx = len(scans), int(scans["ny"][0]), int(scans["nx"][0])
    return z.reshape(S, ny, nx).astype(np.float64), n.reshape(S, ny, nx, mb.n_dot), margin.reshape(S, ny, nx)


def gpu(engine, mb, scans, q, flags, n_type=None):
    engine.set_models(mb)
    z, n = engine.scan_closed_host(scans, q, n_type=n_type, flags=flags)
    S, ny, nx = len(scans), int(scans["ny"][0]), int(scans["nx"][0])
    return z.reshape(S, ny, nx).astype(np.float64), n.reshape(S, ny, nx, mb.n_dot).astype(np.float64)


def q_per_scan(n_dot, n_scan, algorithm, offset=0):
    """A different total charge per scan around N (brute force: small enough for the C restatement at 8 dots)."""
    base = [n_dot - 1, n_dot, n_dot + 1, n_dot + 2] if algorithm == "default" else [max(n_dot - 1, 0), n_dot, n_dot + 1]
    q = np.array([base[(i + offset) % len(base)] for i in range(n_scan)], dtype=np.int32)
    return np.clip(q, 0, 15 if algorithm == "brute_force" else 251)


def compare_hard(n_g, n_c, margin, near, q):
    """Charges equal except at near-ties; sum n = Q exactly.  Returns the number of differing near-tie pixels."""
    assert (n_g.sum(axis=-1) == q[:, None, None]).all(), "sum n != Q"
    diff = (n_g != np.rint(n_c)).any(axis=-1)
    tie = (margin <= TIE) | near
    assert not (diff & ~tie).any(), f"{(diff & ~tie).sum()} pixels differ away from near-ties, first at {np.argwhere(diff & ~tie)[:5]}"
    assert (diff & tie).mean() <= MAX_TIE_FRAC, f"too many differing near-ties: {(diff & tie).mean():.4f}"
    return int((diff & tie).sum())


# ---------------------------------------------------------------------------------------------------------------------
# affine batches: 1..8 dots, default / brute force, T = 0 / T > 0
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algorithm", ["default", "brute_force"])
@pytest.mark.parametrize("n_dot", range(1, 9))
def test_closed_hard_argmin_matches_cport(engine, n_dot, algorithm):
    res = 16 if (algorithm == "default" or n_dot <= 6) else 10
    mb, scans = closed_batch(n_dot, algorithm, res=res, seed=1)
    q = q_per_scan(n_dot, len(scans), algorithm)
    assert len(set(q.tolist())) > 1 or len(scans) == 1 or n_dot == 1
    near = near_integer(relaxed(mb, scans, q)) if algorithm == "default" else np.zeros((len(scans), res, res), bool)
    # noise-free: z to 1e-6 relative given equal charges
    z_c, n_c, margin = cport(mb, scans, q, 0)
    z_g, n_g = gpu(engine, mb, scans, q, 0)
    compare_hard(n_g, n_c, margin, near, q)
    same = (n_g == n_c).all(axis=-1)
    assert np.allclose(z_g[same], z_c[same], rtol=Z_RTOL, atol=1e-7)
    # latching + noise + radial: equal on the rows whose unlatched charges agree
    fl = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    z_cl, n_cl, _ = cport(mb, scans, q, fl)
    z_gl, n_gl = gpu(engine, mb, scans, q, fl)
    rows = same.all(axis=2)
    assert rows.mean() > 0.9
    assert np.array_equal(n_gl[rows], n_cl[rows])
    assert np.allclose(z_gl[rows], z_cl[rows], rtol=0, atol=Z_NOISY_ATOL)
    assert (n_gl.sum(axis=-1) == q[:, None, None]).all()
    # the latching changed something (the case reaches the latching pass; one dot always holds all Q carriers)
    assert n_dot == 1 or not np.array_equal(n_cl, n_c)


@pytest.mark.parametrize("algorithm", ["default", "brute_force"])
@pytest.mark.parametrize("n_dot", range(1, 9))
def test_closed_thermal_matches_cport(engine, n_dot, algorithm):
    res = 12 if (algorithm == "brute_force" and n_dot == 8) else 16
    mb, scans = closed_batch(n_dot, algorithm, thermal=True, res=res, seed=2)
    q = q_per_scan(n_dot, len(scans), algorithm, offset=1)
    _, n_c, _ = cport(mb, scans, q, FLAG_THERMAL)
    z_g, n_g = gpu(engine, mb, scans, q, FLAG_THERMAL, n_type=N_F64)
    near = near_integer(relaxed(mb, scans, q)) if algorithm == "default" else np.zeros(n_g.shape[:3], bool)
    bad = (np.abs(n_g - n_c) > 1e-9).any(axis=-1)
    assert not (bad & ~near).any(), f"max |<n> - <n>_C| = {np.abs(n_g - n_c)[bad & ~near].max():.3e}"
    assert bad.mean() <= MAX_TIE_FRAC
    assert np.allclose(n_g.sum(axis=-1), q[:, None, None], rtol=0, atol=1e-9)
    assert n_dot == 1 or not np.allclose(n_g, np.rint(n_g), atol=1e-6)       # a real Boltzmann average


# ---------------------------------------------------------------------------------------------------------------------
# branches
# ---------------------------------------------------------------------------------------------------------------------
def test_closed_relaxation_with_and_without_clamped_dots(engine):
    """A small total charge clamps dots to 0 in the relaxation (non-empty active set); a large one clamps none."""
    n_dot = 4
    mb, scans = closed_batch(n_dot, "default", res=24, seed=3, offset_range=1.0)
    for q_val, want_clamped in ((1, True), (3 * n_dot, False)):
        q = np.full(len(scans), q_val, dtype=np.int32)
        nc = relaxed(mb, scans, q)
        clamped = (nc <= 0.0).any(axis=-1)
        assert clamped.mean() > 0.5 if want_clamped else not clamped.any(), (q_val, clamped.mean())
        z_c, n_c, margin = cport(mb, scans, q, 0)
        z_g, n_g = gpu(engine, mb, scans, q, 0)
        compare_hard(n_g, n_c, margin, near_integer(nc), q)


def test_closed_candidate_weights_zero_and_n_minus_one(engine):
    """k = Q - sum floor(n_c) = sum frac(n_c) takes its extreme values 0 and N - 1 in the batch (k = 0 needs integral
    relaxed occupations: the scan of total charge 0)."""
    n_dot = 3
    mb, scans = closed_batch(n_dot, "default", res=32, seed=4, offset_range=2.5)
    q = q_per_scan(n_dot, len(scans), "default")
    q[0] = 0
    nc = relaxed(mb, scans, q)
    k = q[:, None, None] - np.floor(nc).sum(axis=-1)
    assert (k == 0).any() and (k == n_dot - 1).any(), np.unique(k)
    z_c, n_c, margin = cport(mb, scans, q, 0)
    _, n_g = gpu(engine, mb, scans, q, 0)
    compare_hard(n_g, n_c, margin, near_integer(nc), q)


@pytest.mark.parametrize("algorithm,q_val", [("default", 0), ("brute_force", 0), ("brute_force", 15)])
def test_closed_extreme_totals(engine, algorithm, q_val):
    n_dot = 3
    mb, scans = closed_batch(n_dot, algorithm, res=16, seed=5)
    q = np.full(len(scans), q_val, dtype=np.int32)
    z_c, n_c, margin = cport(mb, scans, q, 0)
    _, n_g = gpu(engine, mb, scans, q, 0)
    near = near_integer(relaxed(mb, scans, q)) if algorithm == "default" else np.zeros(n_g.shape[:3], bool)
    compare_hard(n_g, n_c, margin, near, q)
    if q_val == 0:
        assert (n_g == 0).all()
    else:
        assert (n_g.max(axis=-1) >= 6).any()                    # the box {0..15} is used well beyond the open default


# ---------------------------------------------------------------------------------------------------------------------
# flags the C restatement does not carry (1/f) and carry-rows, against the NumPy oracle
# ---------------------------------------------------------------------------------------------------------------------
def oracle_closed(mb, scans, q, flags):
    zs, ns, ms = [], [], []
    for i, rec in enumerate(scans):
        m = oracle_model(mb, int(rec["env_id"]), flags)
        z, n, mg = closed.simulate_scan_closed(m, int(q[i]), oracle_scan(rec, mb.n_volt, flags),
                                               carry_rows=bool(flags & FLAG_CARRY_ROWS), return_margin=True)
        zs.append(z), ns.append(n), ms.append(mg)
    return np.stack(zs), np.stack(ns), np.stack(ms)


@pytest.mark.parametrize("flags", [FLAG_NOISE | FLAG_PINK | FLAG_RADIAL, FLAG_LATCH | FLAG_NOISE | FLAG_CARRY_ROWS])
def test_closed_pink_and_carry_rows_match_oracle(engine, flags):
    n_dot = 3
    mb, scans = closed_batch(n_dot, "default", res=16, seed=6)
    q = q_per_scan(n_dot, len(scans), "default")
    z_o, n_o, margin = oracle_closed(mb, scans, q, flags)
    z_g, n_g = gpu(engine, mb, scans, q, flags)
    nc = relaxed(mb, scans, q)
    tie = (margin <= TIE) | near_integer(nc)
    if flags & FLAG_CARRY_ROWS:
        ok = ~tie.reshape(len(scans), -1).any(axis=1)[:, None, None] & np.ones(tie.shape, bool)
    else:
        ok = ~tie
    assert ok.mean() > 0.5
    assert np.array_equal(n_g[ok], n_o[ok])
    assert np.allclose(z_g[ok], z_o[ok], rtol=0, atol=Z_NOISY_ATOL)
    if flags & FLAG_PINK:
        z_np, _, _ = oracle_closed(mb, scans, q, flags & ~FLAG_PINK)
        assert np.abs(z_np - z_o).max() > 1e-3                  # the 1/f term is on


# ---------------------------------------------------------------------------------------------------------------------
# explicit voltage lists, device outputs, the drop-in class, the open path alongside
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algorithm,thermal", [("default", False), ("default", True), ("brute_force", False),
                                               ("brute_force", True)])
def test_closed_points_match_oracle(engine, algorithm, thermal):
    n_dot = 4
    mb, scans = closed_batch(n_dot, algorithm, thermal=thermal, res=12, seed=7)
    engine.set_models(mb)
    rng = np.random.default_rng(8)
    rec = scans[0]
    nv = mb.n_volt
    v = composer.affine_grid(rec["v0"][:nv], rec["dx"][:nv], rec["dy"][:nv], 12, 12)
    v = v + rng.normal(0.0, 0.05, size=v.shape)                  # not an affine grid
    q = 5
    flags = FLAG_THERMAL if thermal else 0
    z_g, n_g = engine.points_closed_host(rec, q, v, n_type=N_F64, flags=flags)
    m = oracle_model(mb, int(rec["env_id"]), flags)
    z_o, n_o, margin = closed.simulate_points_closed(m, q, v, oracle_scan(rec, nv, flags), return_margin=True)
    if thermal:
        assert np.allclose(n_g, n_o, rtol=0, atol=1e-9)
        assert np.allclose(n_g.sum(axis=-1), q, rtol=0, atol=1e-9)
    else:
        g = v.reshape(-1, nv) @ mb.cgd_full[0, :n_dot].T
        nc = closed.continuous_relaxation_closed(g, mb.cdd_gs[0], mb.cdd_inv_gs[0], q).reshape(12, 12, n_dot)
        near = near_integer(nc) if algorithm == "default" else np.zeros((12, 12), bool)
        ok = ~((margin <= TIE) | near)
        assert ok.mean() > 0.9
        assert np.array_equal(n_g[ok], n_o[ok])
        assert (n_g.sum(axis=-1) == q).all()
        assert np.allclose(z_g[ok], z_o[ok], rtol=Z_RTOL, atol=1e-7)


def test_closed_device_outputs_equal_host_outputs(engine):
    import torch
    n_dot = 4
    mb, scans = closed_batch(n_dot, "default", res=16, seed=9)
    q = q_per_scan(n_dot, len(scans), "default")
    fl = FLAG_LATCH | FLAG_NOISE
    z_h, n_h = gpu(engine, mb, scans, q, fl)
    pixels = len(scans) * 16 * 16
    z_d = torch.empty(pixels, dtype=torch.float32, device="cuda")
    n_d = torch.empty((pixels, n_dot), dtype=torch.uint8, device="cuda")
    engine.scan_closed(scans, q, z_d, n_d, N_U8, fl)
    torch.cuda.synchronize()
    assert engine.status() == 0
    assert np.array_equal(z_d.cpu().numpy().reshape(z_h.shape), z_h.astype(np.float32))
    assert np.array_equal(n_d.cpu().numpy().reshape(n_h.shape), n_h)


def test_open_path_unchanged_around_closed_calls(engine):
    n_dot = 4
    mb, scans = closed_batch(n_dot, "default", res=32, seed=10)
    engine.set_models(mb)
    fl = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    z0, n0 = engine.scan_open_host(scans, n_type=N_U8, flags=fl)
    q = q_per_scan(n_dot, len(scans), "default")
    engine.scan_closed_host(scans, q, flags=fl)
    engine.points_closed_host(scans[0], 4, np.zeros((3, 5, mb.n_volt)))
    z1, n1 = engine.scan_open_host(scans, n_type=N_U8, flags=fl)
    assert np.array_equal(z0, z1) and np.array_equal(n0, n1)
    assert not np.array_equal(n0.reshape(-1, n_dot).sum(axis=-1), np.resize(np.repeat(q, 32 * 32), n0.shape[0]))


def test_closed_rejects_unsupported_and_invalid(engine):
    mb, scans = closed_batch(3, "default", res=8, seed=11)
    engine.set_models(mb)
    for bad in (-1, 252):
        with pytest.raises(QdError) as e:
            engine.scan_closed_host(scans, bad)
        assert e.value.code == -1
    mbt = synth.model_batch(synth.sample_devices(1, 3, seed=1), algorithm="thresholded")
    engine.set_models(mbt)
    with pytest.raises(QdError) as e:
        engine.scan_closed_host(scans[:1], 2)
    assert e.value.code == -5
    bdev = synth.sample_barrier_devices(1, 3, seed=5)
    tmb = synth.tunnel_batch(bdev, latching=False, noise=False)
    engine.set_models(tmb)
    tscans = synth.env_step_scans(tmb, bdev, res=8, seed=6, radial=False)[:1]
    with pytest.raises(QdError) as e:
        engine.scan_closed_host(tscans, 2, n_type=N_F64)
    assert e.value.code == -5
    with pytest.raises(QdError) as e:
        engine.points_closed_host(tscans[0], 2, np.zeros((2, 2, tmb.n_volt)))
    assert e.value.code == -5
    mbb = synth.model_batch(synth.sample_devices(1, 3, seed=1), algorithm="brute_force")
    engine.set_models(mbb)
    with pytest.raises(QdError) as e:
        engine.scan_closed_host(scans[:1], 16)
    assert e.value.code == -1


@pytest.mark.parametrize("algorithm,T", [("default", 0.0), ("default", 100.0), ("brute_force", 0.0)])
def test_dropin_closed_methods(algorithm, T):
    import qarray
    n_dot = 3
    dev = synth.sample_devices(1, n_dot, seed=12)
    kw = {"implementation": "jax", "max_charge_carriers": 2} if algorithm == "brute_force" else {}
    m = qarray.ChargeSensedDotArray(dev["Cdd"][0], dev["Cgd"][0], dev["Cds"][0], dev["Cgs"][0], algorithm=algorithm,
                                    T=T, coulomb_peak_width=0.2, **kw)
    q = 4
    kT = path_a.K_B * T
    vg = np.random.default_rng(13).uniform(-3.0, 0.0, size=(5, 7, n_dot + 1))
    n = m.ground_state_closed(vg, q)
    assert n.shape == (5, 7, n_dot)
    n_o = closed.ground_state_closed(vg.reshape(-1, n_dot + 1), m.cgd, m.cdd_inv, m.cdd, q, algorithm, kT=kT)
    atol = 1e-9 if T > 0 else 0.0
    assert np.allclose(n.reshape(-1, n_dot), n_o, rtol=0, atol=atol)
    z, n2 = m.charge_sensor_closed(vg, q)
    assert z.shape == (5, 7, 1) and np.array_equal(n2, n)
    z1, n1 = m.do1d_closed(1, -3.0, 0.0, 9, q)
    assert z1.shape == (9, 1) and n1.shape == (9, n_dot)
    z2, n2 = m.do2d_closed(1, -3.0, 0.0, 10, 2, -3.0, 0.0, 8, q)
    assert z2.shape == (8, 10, 1) and n2.shape == (8, 10, n_dot)
    v = m.gate_voltage_composer.do2d(1, -3.0, 0.0, 10, 2, -3.0, 0.0, 8)
    zp, np_ = m.charge_sensor_closed(v, q)
    assert np.allclose(n2, np_, rtol=0, atol=atol)
    assert np.allclose(z2, zp, rtol=1e-6, atol=1e-7)
    assert np.allclose(n2.sum(axis=-1), q, rtol=0, atol=1e-9)
    with pytest.raises(ValueError):
        m.do2d_closed(1, -3.0, 0.0, 10, 2, -3.0, 0.0, 8, 2.5)
    t = qarray.ChargeSensedDotArray(dev["Cdd"][0], dev["Cgd"][0], dev["Cds"][0], dev["Cgs"][0], algorithm="thresholded")
    with pytest.raises(NotImplementedError):
        t.do2d_closed(1, -3.0, 0.0, 10, 2, -3.0, 0.0, 8, q)
