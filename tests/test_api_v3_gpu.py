"""ABI 3 additions, on the GPU through the C ABI: compact observation path (qd_scan_obs_host), sticky status word
(uint8 / latching-key range), flag validation (QD_FLAG_LATCH_EXACT, QD_N_U8 on the tunnel path), launch ordering across
streams, host-buffer argument checks, the small-call fast path."""
import numpy as np
import pytest

from util import oracle_batch

pytestmark = pytest.mark.gpu


def _batch(engine, n_env=6, n_dot=4, res=32, seed=11, **kw):
    from qdsim import synth
    dev = synth.sample_devices(n_env, n_dot, seed=seed)
    mb = synth.model_batch(dev, **kw)
    engine.set_models(mb)
    return dev, mb, synth.env_step_scans(mb, dev, res=res, seed=seed + 1, offset_range=3.0)


def _normalise_ref(z, per_env, q_low=0.5, q_high=99.5):
    """QuantumDeviceEnv._normalise_obs (env.py:471-509) per env block, in fp64."""
    z = np.asarray(z, dtype=np.float64).reshape(-1, per_env)
    lo = np.percentile(z, q_low, axis=1, keepdims=True)
    hi = np.percentile(z, q_high, axis=1, keepdims=True)
    with np.errstate(invalid="ignore", divide="ignore"):
        out = np.where(hi > lo, np.clip((z - lo) / (hi - lo), 0.0, 1.0), 0.0)
    return out, np.concatenate([lo, hi], axis=1)


@pytest.mark.parametrize("n_env,res", [(6, 32), (3, 17)])
def test_obs_host_uint8_is_the_normalised_oracle_image_within_one_lsb(engine, n_env, res):
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_NONE, Z_F16, Z_F32, Z_U8
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    dev, mb, scans = _batch(engine, n_env=n_env, res=res)
    per_env = 3 * res * res
    z32, _ = engine.scan_open_host(scans, n_type=N_NONE, flags=flags)
    u8, stats = engine.scan_obs_host(scans, z_type=Z_U8, flags=flags, want_stats=True)
    assert u8.dtype == np.uint8 and u8.shape == (len(scans), res, res)
    # (1) exactly the library's own fp32 image, normalised and quantised
    ref, st_ref = _normalise_ref(z32, per_env)
    np.testing.assert_allclose(stats, st_ref, rtol=0, atol=1e-12)
    np.testing.assert_array_equal(u8, np.rint(255.0 * ref).astype(np.uint8).reshape(u8.shape))
    # (2) the ORACLE's image (fp64, its own noise arithmetic) normalised the reference's way: +-1 LSB
    z_or, _, _ = oracle_batch(mb, scans, flags)
    ref_or, _ = _normalise_ref(z_or, per_env)
    assert np.abs(u8.astype(np.int64) - np.rint(255.0 * ref_or).astype(np.int64).reshape(u8.shape)).max() <= 1
    # half / float variants of the same call
    f16, _ = engine.scan_obs_host(scans, z_type=Z_F16, flags=flags)
    np.testing.assert_array_equal(f16.reshape(-1), ref.reshape(-1).astype(np.float32).astype(np.float16))
    f32, _ = engine.scan_obs_host(scans, z_type=Z_F32, flags=flags)
    np.testing.assert_array_equal(f32.reshape(-1), ref.reshape(-1).astype(np.float32))
    raw16, _ = engine.scan_obs_host(scans, z_type=Z_F16, flags=flags, normalise=False)
    np.testing.assert_array_equal(raw16.reshape(-1), z32.astype(np.float16))
    raw32, _ = engine.scan_obs_host(scans, z_type=Z_F32, flags=flags, normalise=False)
    np.testing.assert_array_equal(raw32.reshape(-1), z32)


def test_obs_host_pipelined_batch_equals_the_unpipelined_one(engine):
    """>= 4096 scans: the call is cut into chunks of envs; every env must come out as in a single-chunk call."""
    from qdsim import FLAG_LATCH, FLAG_NOISE, Z_U8
    flags = FLAG_LATCH | FLAG_NOISE
    dev, mb, scans = _batch(engine, n_env=2100, res=8, seed=21)        # 6300 scans -> 3 chunks
    big, _ = engine.scan_obs_host(scans, z_type=Z_U8, flags=flags)
    pick = np.array([0, 1, 700, 1399, 1400, 2099])
    for e in pick:
        sub = scans[3 * e:3 * e + 3].copy()
        sub["pix_offset"] = np.arange(3) * 64
        one, _ = engine.scan_obs_host(sub, z_type=Z_U8, flags=flags)
        np.testing.assert_array_equal(one, big[3 * e:3 * e + 3])


def test_obs_host_rejects_bad_arguments(engine):
    from qdsim import QdError, Z_U8
    dev, mb, scans = _batch(engine)
    with pytest.raises(QdError):
        engine.scan_obs_host(scans, z_type=Z_U8, normalise=False)              # uint8 needs a normalised image
    with pytest.raises(QdError):
        engine.scan_obs_host(scans[:4], z_type=Z_U8)                           # not a multiple of scans_per_env
    bad = scans.copy()
    bad["pix_offset"][1] += 5
    with pytest.raises(QdError):
        engine.scan_obs_host(bad, z_type=Z_U8)


def test_latch_exact_flag_equals_rounded_on_integers_and_is_refused_on_non_integers(engine):
    from qdsim import FLAG_LATCH, FLAG_LATCH_EXACT, FLAG_THERMAL, N_F64, N_U8, QdError, synth
    dev, mb, scans = _batch(engine)
    z0, n0 = engine.scan_open_host(scans, n_type=N_U8, flags=FLAG_LATCH)
    z1, n1 = engine.scan_open_host(scans, n_type=N_U8, flags=FLAG_LATCH | FLAG_LATCH_EXACT)
    np.testing.assert_array_equal(n0, n1)
    np.testing.assert_array_equal(z0, z1)
    z_ref, n_ref, margin = oracle_batch(mb, scans, FLAG_LATCH | FLAG_LATCH_EXACT)     # the oracle's exact compare agrees
    safe = (margin > 1e-9).all(axis=2)
    assert (n1.reshape(n_ref.shape).astype(np.int64) == np.rint(n_ref).astype(np.int64))[safe].all()
    with pytest.raises(QdError) as ei:
        engine.scan_open_host(scans, n_type=N_F64, flags=FLAG_LATCH | FLAG_LATCH_EXACT | FLAG_THERMAL)
    assert ei.value.code == -5
    bdev = synth.sample_barrier_devices(1, 4, seed=3)
    engine.set_models(synth.tunnel_batch(bdev))
    tscans = synth.env_step_scans(engine.models, bdev, res=8, seed=4)
    with pytest.raises(QdError) as ei:
        engine.scan_open_host(tscans, n_type=N_F64, flags=FLAG_LATCH | FLAG_LATCH_EXACT)
    assert ei.value.code == -5
    with pytest.raises(QdError) as ei:                                            # <n> is not an integer: no uint8 map
        engine.scan_open_host(tscans, n_type=N_U8, flags=0)
    assert ei.value.code == -1


def test_occupation_overflow_is_reported_not_saturated(engine):
    from qdsim import N_U8, STATUS_OCC_OVERFLOW, QdError
    import torch
    dev, mb, scans = _batch(engine, latching=False, noise=False)
    far = scans[:3].copy()
    far["pix_offset"] = np.arange(3) * 32 * 32
    far["v0"][:, 0] -= 400.0                       # ~400 carriers on dot 0 (cgd ~ -1): outside 0..255
    with pytest.raises(QdError) as ei:
        engine.scan_open_host(far, n_type=N_U8, flags=0)
    assert ei.value.code == -1 and "carriers" in str(ei.value)
    assert engine.status() == 0                    # the synchronous call consumed the flag
    # asynchronous entry: the caller polls the sticky word after synchronising
    z = torch.empty(3 * 1024, dtype=torch.float32, device="cuda")
    n = torch.empty((3 * 1024, 4), dtype=torch.uint8, device="cuda")
    engine.scan_open(far, z, n, N_U8, 0)
    torch.cuda.synchronize()
    assert engine.status(clear=False) & STATUS_OCC_OVERFLOW
    assert engine.status() & STATUS_OCC_OVERFLOW and engine.status() == 0
    ok = scans[:3].copy()
    ok["pix_offset"] = np.arange(3) * 32 * 32
    engine.scan_open_host(ok, n_type=N_U8, flags=0)          # and the context keeps working


def test_host_buffers_are_checked_before_the_library_writes_into_them(engine):
    from qdsim import N_U8
    dev, mb, scans = _batch(engine)
    pixels = len(scans) * 32 * 32
    with pytest.raises(AssertionError):
        engine.scan_open_host(scans, n_type=N_U8, n_out=np.empty((pixels, 4), dtype=np.float32))   # wrong dtype
    with pytest.raises(AssertionError):
        engine.scan_open_host(scans, n_type=N_U8, n_out=np.empty((pixels - 1, 4), dtype=np.uint8))  # too small
    with pytest.raises(AssertionError):
        engine.scan_open_host(scans, n_type=N_U8, n_out=np.empty((pixels, 8), dtype=np.uint8)[:, ::2])  # strided


def test_gaps_between_scans_come_back_as_zeros(engine):
    """Scans that do not tile the output range: the copy-back moves whole ranges, the gaps must not be stale memory."""
    from qdsim import N_U8
    dev, mb, scans = _batch(engine, latching=False, noise=False)
    engine.scan_open_host(scans, n_type=N_U8)                        # dirty the context's scratch
    s = scans[:2].copy()
    s["pix_offset"] = [0, 3000]                                      # 1024 pixels, gap, 1024 pixels
    z, n = engine.scan_open_host(s, n_type=N_U8)
    assert z.shape[0] == 4024
    assert (z[1024:3000] == 0).all() and (n[1024:3000] == 0).all()
    for big in (False, True):                                         # the pipelined (large) path as well
        if big:
            s = np.tile(scans[:1], 300).copy()
            s["pix_offset"] = np.arange(300) * 2048                  # every scan followed by a 1024-pixel gap
            z, n = engine.scan_open_host(s, n_type=N_U8)
            assert z.shape[0] == 299 * 2048 + 1024
            zz = np.concatenate([z, np.zeros(1024, dtype=z.dtype)]).reshape(300, 2048)
            assert (zz[:, 1024:] == 0).all() and (zz[:, :1024] == zz[0, :1024]).all()


def test_launches_on_different_streams_do_not_trample_the_descriptor_scratch(engine):
    """qd_scan_open on stream A, then immediately on stream B with other descriptors: B's staging must wait for A's kernel
    (the context's descriptor buffer is shared)."""
    import torch
    from qdsim import FLAG_LATCH, FLAG_NOISE, N_U8
    flags = FLAG_LATCH | FLAG_NOISE
    dev, mb, scans = _batch(engine, n_env=600, res=32, seed=31)
    a, b = scans[: 900].copy(), scans[900:].copy()
    b["pix_offset"] -= b["pix_offset"][0]
    pa, pb = 900 * 1024, len(b) * 1024
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    za, zb = torch.empty(pa, device="cuda"), torch.empty(pb, device="cuda")
    na, nb = torch.empty((pa, 4), dtype=torch.uint8, device="cuda"), torch.empty((pb, 4), dtype=torch.uint8, device="cuda")
    for _ in range(3):
        engine.scan_open(a, za, na, N_U8, flags, sa)
        engine.scan_open(b, zb, nb, N_U8, flags, sb)
    torch.cuda.synchronize()
    za2, na2 = engine.scan_open_host(a, n_type=N_U8, flags=flags)
    zb2, nb2 = engine.scan_open_host(b, n_type=N_U8, flags=flags)
    assert np.array_equal(za.cpu().numpy(), za2) and np.array_equal(na.cpu().numpy(), na2)
    assert np.array_equal(zb.cpu().numpy(), zb2) and np.array_equal(nb.cpu().numpy(), nb2)


def test_batched_env_observations_do_not_alias(engine):
    """obs_t must survive the next step (ADVICE r1): the shell ping-pongs between two image buffers."""
    import torch
    from qdsim.vector_env import BatchedDeviceEnv, EnvConfig
    env = BatchedDeviceEnv(4, 4, engine=engine, seed=5, config=EnvConfig(resolution=16, max_steps=5))
    obs0, _ = env.reset()
    keep = obs0["image"].clone()
    rng = np.random.default_rng(0)
    obs1, *_ = env.step(rng.uniform(-1, 1, (4, 4)), rng.uniform(-1, 1, (4, 3)))
    assert obs1["image"].data_ptr() != obs0["image"].data_ptr()
    assert torch.equal(obs0["image"], keep), "the previous observation was overwritten by the step"
    assert not torch.equal(obs1["image"], keep)


@pytest.mark.parametrize("n_dot,alg", [(8, "default"), (4, "default"), (5, "thresholded"), (2, "default"), (3, "default"),
                                       (6, "default"), (7, "thresholded")])
def test_fast_and_generic_scan_kernels_agree(engine, n_dot, alg, monkeypatch):
    """qd_scan_fast_kernel (the hot instantiation) against qd_scan_kernel on the same batch: identical charge maps, images
    equal to fp32 rounding (the sensor's dot term is summed in a different order)."""
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_F32, N_U8, synth
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    dev = synth.sample_devices(40, n_dot, seed=100 + n_dot)
    mb = synth.model_batch(dev, algorithm=alg, threshold=0.7)
    engine.set_models(mb)
    scans = synth.env_step_scans(mb, dev, res=48, seed=200 + n_dot, offset_range=4.0)
    scans["rad_mode"][::7] = 2                      # some windows replaced by pure noise
    out = {}
    for generic in ("1", "0"):
        monkeypatch.setenv("QDSIM_GENERIC_SCAN", generic)
        for fl in (flags, FLAG_LATCH, 0):
            out[generic, fl] = engine.scan_open_host(scans, n_type=N_U8, flags=fl)
        out[generic, "f32"] = engine.scan_open_host(scans, n_type=N_F32, flags=flags)
    for fl in (flags, FLAG_LATCH, 0, "f32"):
        zg, ng = out["1", fl]
        zf, nf = out["0", fl]
        assert np.array_equal(ng, nf), f"flags {fl}: {(ng != nf).any(axis=-1).sum()} pixels differ"
        np.testing.assert_allclose(zf, zg, rtol=2e-7, atol=1e-7)


def test_fast_kernel_flat_pass_and_wide_search(engine, monkeypatch):
    """Carry-rows (one warp per scan) and a strongly coupled device where dominance decides nothing (the Gray walk runs all
    2^N settings) through both kernels."""
    from qdsim import FLAG_CARRY_ROWS, FLAG_LATCH, FLAG_NOISE, N_U8, synth
    dev = synth.sample_devices(3, 6, seed=77)
    dev["Cdd"] *= 4.0                               # strong inter-dot coupling: wide undecided sets
    mb = synth.model_batch(dev)
    engine.set_models(mb)
    scans = synth.env_step_scans(mb, dev, res=40, seed=78, offset_range=1.0)
    res = {}
    for generic in ("1", "0"):
        monkeypatch.setenv("QDSIM_GENERIC_SCAN", generic)
        res[generic] = [engine.scan_open_host(scans, n_type=N_U8, flags=f)
                        for f in (FLAG_LATCH | FLAG_NOISE | FLAG_CARRY_ROWS, FLAG_LATCH | FLAG_NOISE)]
    for (zg, ng), (zf, nf) in zip(res["1"], res["0"]):
        assert np.array_equal(ng, nf)
        np.testing.assert_allclose(zf, zg, rtol=2e-7, atol=1e-7)
    z_ref, n_ref, margin = oracle_batch(mb, scans, FLAG_LATCH | FLAG_NOISE)
    safe = (margin > 1e-9).all(axis=2)
    nf = res["0"][1][1].reshape(n_ref.shape)
    assert (nf.astype(np.int64) == np.rint(n_ref).astype(np.int64))[safe].all()


@pytest.mark.parametrize("n_dot,res,carry", [(4, 40, False), (3, 33, True), (8, 64, False)])
def test_pink_noise_matches_the_oracle_definition(engine, n_dot, res, carry):
    """QD_FLAG_PINK (north_star's 1/f noise; the reference has none): draw-for-draw against oracle/noise.py::pink_noise."""
    from qdsim import FLAG_CARRY_ROWS, FLAG_LATCH, FLAG_NOISE, FLAG_PINK, N_U8, synth
    dev = synth.sample_devices(3, n_dot, seed=300 + n_dot)
    mb = synth.model_batch(dev)
    mb.params["pink_amp"] = [2e-3, 0.0, 5e-4]
    engine.set_models(mb)
    scans = synth.env_step_scans(mb, dev, res=res, seed=301, offset_range=2.0, radial=False)
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_PINK | (FLAG_CARRY_ROWS if carry else 0)
    z, n = engine.scan_open_host(scans, n_type=N_U8, flags=flags)
    z0, n0 = engine.scan_open_host(scans, n_type=N_U8, flags=flags & ~FLAG_PINK)
    z_ref, n_ref, margin = oracle_batch(mb, scans, flags)
    np.testing.assert_allclose(z.reshape(z_ref.shape), z_ref, rtol=0, atol=5e-6)
    assert np.array_equal(n, n0)                                        # input noise does not touch the charge state
    per_env = (n_dot - 1) * res * res
    assert np.array_equal(z[per_env:2 * per_env], z0[per_env:2 * per_env])    # pink_amp = 0: term off
    assert np.abs(z[:per_env] - z0[:per_env]).max() > 1e-4               # and it is really there for env 0
