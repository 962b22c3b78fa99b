"""Closed arrays (fixed total charge on the dots), CPU side: the NumPy oracle's closed relaxation and ground state, the
plain-C restatement's closed scans, and the argument checks of the closed entry points that run without a GPU.

* ``continuous_relaxation_closed`` satisfies sum n = Q, n >= 0 and the KKT conditions; it is the open relaxation at the
  shifted potentials g + nu* cdd 1 (the route the kernel takes), and sum n(g + nu cdd 1) is non-decreasing in nu -- on
  random devices at 2..8 dots, Q in {0, 1, N, 3N}, in windows where some dots are clamped to 0 and where none is;
* at 2 dots closed ``default`` equals closed ``brute_force`` at every pixel (the feasible set is a line, the energy along it
  convex);
* the C restatement's closed scans equal the oracle (charges where the margin exceeds 1e-9, z to 1e-6) with latching and
  noise on;
* invalid totals and the unsupported algorithms are refused by the oracle, the C restatement and the drop-in class.
"""
import numpy as np
import pytest

from oracle import closed, path_a
from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, synth
from util import oracle_model, oracle_scan

TIE = 1e-9


def devices(n_dot, n_env=4, seed=0):
    dev = synth.sample_devices(n_env, n_dot, seed=100 + n_dot + seed)
    return dev, synth.model_batch(dev, algorithm="default", latching=True, noise=True)


def random_potentials(rng, n_dot, q, p=400):
    """Dot potentials around Q / N carriers per dot, a third of the rows with some dots pushed far below 0."""
    g = rng.uniform(-1.0, 1.0, size=(p, n_dot)) + q / n_dot
    far = rng.random((p, n_dot)) < 0.3
    g[: p // 3] = np.where(far[: p // 3], -rng.uniform(1.0, 4.0, size=(p // 3, n_dot)), g[: p // 3])
    return g


def shifted_root(g, cdd, q):
    """nu* with sum open_relax(g + nu* c) = q, c = cdd 1, by bisection (every row)."""
    c = cdd.sum(axis=1)
    lo = np.full(len(g), (-g / c).min(axis=1) - 1.0)
    hi = np.full(len(g), (-g / c).max(axis=1) + q / c.sum() + 1.0)
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        s = path_a.continuous_relaxation(g + mid[:, None] * c, cdd).sum(axis=1)
        lo, hi = np.where(s < q, mid, lo), np.where(s < q, hi, mid)
    return 0.5 * (lo + hi)


@pytest.mark.parametrize("n_dot", range(2, 9))
def test_closed_relaxation_kkt_shift_and_monotone(n_dot):
    _, mb = devices(n_dot)
    rng = np.random.default_rng(n_dot)
    clamped_rows = free_rows = 0
    for e in range(mb.n_env):
        a, cdd = mb.cdd_inv_gs[e], mb.cdd_gs[e]
        for q in (0, 1, n_dot, 3 * n_dot):
            g = random_potentials(rng, n_dot, q)
            n = closed.continuous_relaxation_closed(g, cdd, a, q)
            assert np.allclose(n.sum(axis=1), q, rtol=0, atol=1e-9)
            assert (n >= 0).all()
            # KKT: grad = 2 A (n - g) = lam 1 + mu, mu >= 0 on the clamped dots, 0 on the free ones
            grad = 2.0 * (n - g) @ a.T
            free = n > 1e-9
            if q > 0:
                lam = np.where(free, grad, 0.0).sum(axis=1) / free.sum(axis=1)
                mu = grad - lam[:, None]
                scale = 1.0 + np.abs(grad).max(axis=1, keepdims=True)
                assert (np.abs(np.where(free, mu, 0.0)) <= 1e-9 * scale).all()
                assert (np.where(free, 0.0, mu) >= -1e-10 * scale).all()
                clamped_rows += int((~free).any(axis=1).sum())
                free_rows += int(free.all(axis=1).sum())
            # the open relaxation at the shifted potentials g + nu* cdd 1
            c = cdd.sum(axis=1)
            if q > 0:
                nu = shifted_root(g, cdd, q)
                n_shift = path_a.continuous_relaxation(g + nu[:, None] * c, cdd)
                assert np.allclose(n, n_shift, rtol=0, atol=1e-7)
            # sum n(g + nu c) is non-decreasing in nu
            nus = np.linspace(-(np.abs(g).max() + q + 2.0), np.abs(g).max() + q + 2.0, 41)
            sums = np.stack([path_a.continuous_relaxation(g + v * c, cdd).sum(axis=1) for v in nus], axis=1)
            assert (np.diff(sums, axis=1) >= -1e-9).all()
    assert clamped_rows > 0 and free_rows > 0, (clamped_rows, free_rows)


def closed_scan_batch(n_dot, q_of_scan, res=12, seed=0, algorithm="default", max_charge_carriers=4):
    dev = synth.sample_devices(2, n_dot, seed=200 + n_dot + seed)
    mb = synth.model_batch(dev, algorithm=algorithm, latching=True, noise=True, max_charge_carriers=max_charge_carriers)
    scans = synth.env_step_scans(mb, dev, res=res, seed=seed + 1, offset_range=2.0)
    q = np.resize(np.asarray(q_of_scan, dtype=np.int32), len(scans))
    return mb, scans, q


def oracle_closed(mb, scans, q, flags):
    zs, ns, ms = [], [], []
    for i, rec in enumerate(scans):
        m = oracle_model(mb, int(rec["env_id"]), flags)
        z, n, mg = closed.simulate_scan_closed(m, int(q[i]), oracle_scan(rec, mb.n_volt, flags), return_margin=True)
        zs.append(z), ns.append(n), ms.append(mg)
    return np.stack(zs), np.stack(ns), np.stack(ms)


def test_two_dots_default_equals_brute_force():
    for q in (0, 1, 2, 5):
        mb, scans, qs = closed_scan_batch(2, [q], res=24)
        mb_b, _, _ = closed_scan_batch(2, [q], res=24, algorithm="brute_force")
        _, n_d, _ = oracle_closed(mb, scans, qs, 0)
        _, n_b, _ = oracle_closed(mb_b, scans, qs, 0)
        assert np.array_equal(n_d, n_b), q
        assert (n_d.sum(axis=-1) == q).all()


@pytest.mark.parametrize("n_dot,algorithm,q_of_scan", [
    (2, "default", [0, 3]), (3, "default", [1, 4]), (4, "default", [4, 6]), (6, "default", [6, 9]),
    (8, "default", [8, 11]), (2, "brute_force", [2, 5]), (3, "brute_force", [3, 5]), (4, "brute_force", [4, 6]),
])
def test_cport_closed_matches_oracle(n_dot, algorithm, q_of_scan):
    from oracle.cport import closed as cport
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    mb, scans, q = closed_scan_batch(n_dot, q_of_scan, algorithm=algorithm)
    z_ref, n_ref, margin = oracle_closed(mb, scans, q, flags)
    zc, nc, _ = cport.run_scans_closed(mb, scans, q, flags)
    S, ny, nx = z_ref.shape
    safe = ~(margin <= TIE).any(axis=2)                     # rows without a near-tie (latching carries choices along x)
    assert safe.mean() > 0.9
    nc = nc.reshape(S, ny, nx, n_dot)
    assert np.array_equal(nc[safe], n_ref[safe])
    assert (nc.sum(axis=-1) == q[:, None, None]).all()
    zc = zc.astype(np.float64).reshape(S, ny, nx)
    assert np.allclose(zc[safe], z_ref[safe], rtol=1e-6, atol=1e-6)


def test_cport_closed_thermal_mean_sums_to_q():
    from oracle.cport import closed as cport
    from qdsim import FLAG_THERMAL
    dev = synth.sample_devices(2, 3, seed=7)
    mb = synth.model_batch(dev, thermal=True, latching=False, noise=False)
    scans = synth.env_step_scans(mb, dev, res=10, seed=3, offset_range=2.0, radial=False)
    q = np.array([2, 4, 3, 5], dtype=np.int32)[: len(scans)]
    _, n_ref, _ = oracle_closed(mb, scans, q, FLAG_THERMAL)
    _, nc, _ = cport.run_scans_closed(mb, scans, q, FLAG_THERMAL)
    assert np.allclose(nc.reshape(n_ref.shape), n_ref, rtol=0, atol=1e-9)
    assert np.allclose(n_ref.sum(axis=-1), q[:, None, None], rtol=0, atol=1e-9)
    assert not np.allclose(n_ref, np.rint(n_ref))             # the average is not a hard argmin


def test_closed_configurations_are_the_filtered_product():
    for n_dot, q in ((1, 3), (2, 4), (3, 3), (4, 2)):
        full = path_a.brute_force_configurations(n_dot, q)
        assert np.array_equal(closed.closed_configurations(n_dot, q), full[full.sum(axis=1) == q])


@pytest.mark.parametrize("algorithm,bad", [("default", -1), ("default", 252), ("brute_force", 16), ("default", 1.5),
                                           ("default", "2"), ("default", True)])
def test_oracle_rejects_invalid_n_charge(algorithm, bad):
    g = np.zeros((1, 2))
    with pytest.raises(ValueError):
        closed.ground_state_closed(g, np.eye(2), np.eye(2), np.eye(2), bad, algorithm)


@pytest.mark.parametrize("algorithm", ["thresholded", "tunnel"])
def test_oracle_rejects_unsupported_algorithms(algorithm):
    with pytest.raises(NotImplementedError):
        closed.ground_state_closed(np.zeros((1, 2)), np.eye(2), np.eye(2), np.eye(2), 1, algorithm)


def test_cport_rejects_invalid_n_charge_and_algorithms():
    from oracle.cport import closed as cport
    mb, scans, _ = closed_scan_batch(2, [1], res=4)
    for q in (-1, 252):
        with pytest.raises(ValueError):
            cport.run_scans_closed(mb, scans, q, 0)
    mb.algorithm = "thresholded"
    with pytest.raises(ValueError):
        cport.run_scans_closed(mb, scans, 1, 0)


def dropin(algorithm="default", **kw):
    import qarray
    dev = synth.sample_devices(1, 2, seed=5)
    return qarray.ChargeSensedDotArray(dev["Cdd"][0], dev["Cgd"][0], dev["Cds"][0], dev["Cgs"][0], algorithm=algorithm,
                                       **kw)


@pytest.mark.parametrize("bad", [-1, 252, 1.5, "3", None, True, np.array([1, 2])])
def test_dropin_rejects_invalid_n_charges(bad):
    m = dropin()
    with pytest.raises(ValueError):
        m.ground_state_closed(np.zeros((3, 3)), bad)
    with pytest.raises(ValueError):
        m.do2d_closed(1, -1.0, 1.0, 4, 2, -1.0, 1.0, 4, bad)
    b = dropin("brute_force", implementation="jax", max_charge_carriers=3)
    with pytest.raises(ValueError):
        b.charge_sensor_closed(np.zeros((3, 3)), 16)


def test_dropin_thresholded_closed_is_not_implemented():
    m = dropin("thresholded")
    for call in (lambda: m.ground_state_closed(np.zeros((2, 3)), 1), lambda: m.charge_sensor_closed(np.zeros((2, 3)), 1),
                 lambda: m.do1d_closed(1, -1.0, 1.0, 4, 1), lambda: m.do2d_closed(1, -1.0, 1.0, 4, 2, -1.0, 1.0, 4, 1)):
        with pytest.raises(NotImplementedError):
            call()
