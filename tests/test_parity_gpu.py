"""GPU parity tests: the CUDA path through the C ABI vs the CPU oracle on the same seeded inputs.

Bars (north_star): integer charge configurations bit-exact; noise-free sensor signal within 1e-6 relative; noisy
outputs draw-for-draw (same Philox stream) within the fp32 evaluation error of the normals (abs 2e-6 on O(1) signals).
"""
import numpy as np
import pytest

from util import compare_charges, oracle_batch

pytestmark = pytest.mark.gpu

Z_RTOL = 1e-6      # noise-free sensor signal, relative (north_star)
Z_NOISY_ATOL = 5e-6


def _setup(engine, n_dot, n_env=3, algorithm="default", res=64, seed=11, **kw):
    from qdsim import synth
    dev = synth.sample_devices(n_env, n_dot, seed=seed)
    mb = synth.model_batch(dev, algorithm=algorithm, **kw)
    engine.set_models(mb)
    scans = synth.env_step_scans(mb, dev, res=res, seed=seed + 1, offset_range=3.0)
    return dev, mb, scans


def _run(engine, scans, n_type, flags):
    z, n = engine.scan_open_host(scans, n_type=n_type, flags=flags)
    res_y, res_x = int(scans["ny"][0]), int(scans["nx"][0])
    z = z.reshape(len(scans), res_y, res_x)
    if n is not None:
        n = n.reshape(len(scans), res_y, res_x, -1)
    return z, n


@pytest.mark.parametrize("n_dot", [2, 3, 4, 5, 6, 7, 8])
def test_default_noise_free_bit_exact(engine, n_dot):
    """BASELINE config 1 generalised: T=0, no noise, no latching -> bit-exact charge map, z within 1e-6."""
    from qdsim import N_U8
    n_env = 2 if n_dot >= 7 else 3
    dev, mb, scans = _setup(engine, n_dot, n_env=n_env, latching=False, noise=False)
    z, n = _run(engine, scans, N_U8, 0)
    z_ref, n_ref, margin = oracle_batch(mb, scans, 0)
    compare_charges(n, n_ref, margin)
    safe = margin > 1e-9
    np.testing.assert_allclose(z[safe], z_ref[safe], rtol=Z_RTOL, atol=0)
    assert n.max() > 0 and (n == 0).any(), "window should straddle the empty / occupied boundary"


@pytest.mark.parametrize("n_dot", [2, 4, 8])
def test_latching_draw_for_draw(engine, n_dot):
    """Latched charge maps are bit-exact because both sides consume the same Philox uniforms."""
    from qdsim import FLAG_LATCH, N_U8
    dev, mb, scans = _setup(engine, n_dot, n_env=2, latching=True, noise=False)
    z, n = _run(engine, scans, N_U8, FLAG_LATCH)
    z_ref, n_ref, margin = oracle_batch(mb, scans, FLAG_LATCH)
    assert (margin > 1e-9).all()
    assert np.array_equal(n.astype(np.int64), np.rint(n_ref).astype(np.int64))
    np.testing.assert_allclose(z, z_ref, rtol=Z_RTOL, atol=0)
    # latching must actually have done something on these devices (p ~ U[0.2, 1])
    _, n_free = _run(engine, scans, N_U8, 0)
    assert (n_free != n).any()


@pytest.mark.parametrize("carry", [False, True])
def test_full_noise_model(engine, carry):
    """White + telegraph + radial noise + latching, rows independent or one flat pass."""
    from qdsim import FLAG_CARRY_ROWS, FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_U8
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL | (FLAG_CARRY_ROWS if carry else 0)
    dev, mb, scans = _setup(engine, 4, n_env=3, latching=True, noise=True)
    mb.params["tele_p01"] = 0.05          # make the telegraph chain flip often enough to be tested
    mb.params["tele_p10"] = 0.1
    mb.params["tele_amp"] = 0.01
    engine.set_models(mb)
    scans["rad_zero_radius"] = 1.0        # put the windows inside the noisy annulus
    scans["rad_alpha"] = 0.02
    scans["rad_mode"][-1] = 2             # last scan: replaced by white noise
    z, n = _run(engine, scans, N_U8, flags)
    z_ref, n_ref, margin = oracle_batch(mb, scans, flags)
    assert np.array_equal(n[:-1].astype(np.int64), np.rint(n_ref[:-1]).astype(np.int64))
    np.testing.assert_allclose(z, z_ref, rtol=0, atol=Z_NOISY_ATOL)
    assert abs(z[-1].std() - 1.0) < 0.05 and abs(z[-1].mean()) < 0.05


def test_thermal_softmin(engine):
    from qdsim import FLAG_THERMAL, N_F64
    dev, mb, scans = _setup(engine, 4, n_env=2, latching=False, noise=False, thermal=True)
    z, n = _run(engine, scans, N_F64, FLAG_THERMAL)
    z_ref, n_ref, _ = oracle_batch(mb, scans, FLAG_THERMAL)
    np.testing.assert_allclose(n, n_ref, rtol=0, atol=1e-9)
    np.testing.assert_allclose(z, z_ref, rtol=Z_RTOL, atol=1e-7)
    assert (np.abs(n - np.rint(n)) > 1e-3).any(), "kT > 0 must give non-integer occupations somewhere"


def test_thresholded(engine):
    from qdsim import N_U8
    dev, mb, scans = _setup(engine, 5, n_env=2, algorithm="thresholded", latching=False, noise=False, threshold=0.6)
    z, n = _run(engine, scans, N_U8, 0)
    z_ref, n_ref, margin = oracle_batch(mb, scans, 0)
    compare_charges(n, n_ref, margin)


@pytest.mark.parametrize("n_dot", [2, 3, 4, 5])
def test_brute_force(engine, n_dot):
    from qdsim import N_U8
    dev, mb, scans = _setup(engine, n_dot, n_env=2, algorithm="brute_force", res=32, latching=False, noise=False)
    z, n = _run(engine, scans, N_U8, 0)
    z_ref, n_ref, margin = oracle_batch(mb, scans, 0)
    compare_charges(n, n_ref, margin)
    np.testing.assert_allclose(z[margin > 1e-9], z_ref[margin > 1e-9], rtol=Z_RTOL, atol=0)


def test_ragged_sizes_and_offsets(engine):
    """nx, ny not multiples of the warp width; scans placed at arbitrary pixel offsets; 1x1 scan."""
    from qdsim import FLAG_LATCH, N_U8
    dev, mb, scans = _setup(engine, 3, n_env=2, latching=True, noise=False)
    shapes = [(1, 1), (33, 5), (7, 70), (64, 64)]
    off = 0
    for rec, (nx, ny) in zip(scans, shapes):
        rec["nx"], rec["ny"], rec["pix_offset"] = nx, ny, off
        off += nx * ny + 3
    z, n = engine.scan_open_host(scans, n_type=N_U8, flags=FLAG_LATCH)
    for i, (nx, ny) in enumerate(shapes):
        z_ref, n_ref, margin = oracle_batch(mb, scans, FLAG_LATCH, which=[i])
        o = int(scans["pix_offset"][i])
        assert np.array_equal(n[o:o + nx * ny].reshape(ny, nx, -1).astype(np.int64), np.rint(n_ref[0]).astype(np.int64))
        np.testing.assert_allclose(z[o:o + nx * ny].reshape(ny, nx), z_ref[0], rtol=Z_RTOL, atol=0)


def test_points_mode_matches_affine(engine):
    """The arbitrary-voltage-list entry point gives the same answer as the affine scan on the same grid."""
    from oracle import composer
    from qdsim import FLAG_LATCH, N_U8
    dev, mb, scans = _setup(engine, 4, n_env=1, latching=True, noise=False)
    rec = scans[1]
    nv = mb.n_volt
    v = composer.affine_grid(rec["v0"][:nv], rec["dx"][:nv], rec["dy"][:nv], 64, 64)
    z_p, n_p = engine.points_open_host(rec, v, n_type=N_U8, flags=FLAG_LATCH)
    z_ref, n_ref, margin = oracle_batch(mb, scans, FLAG_LATCH, which=[1])
    assert np.array_equal(n_p.astype(np.int64), np.rint(n_ref[0]).astype(np.int64))
    np.testing.assert_allclose(z_p, z_ref[0], rtol=Z_RTOL, atol=0)


def test_errors(engine):
    from qdsim import FLAG_THERMAL, N_U8, QdError, synth
    dev, mb, scans = _setup(engine, 2, n_env=1, latching=False, noise=False)
    bad = scans.copy()
    bad["env_id"] = 5
    with pytest.raises(QdError):
        engine.scan_open_host(bad, n_type=N_U8)
    with pytest.raises(QdError):
        engine.scan_open_host(scans, n_type=N_U8, flags=FLAG_THERMAL)
    with pytest.raises(ValueError):
        engine.points_open_host(scans[0], np.zeros((4, 4, 7)))
