"""Percentile normalisation of the observation (csrc/qd_normalise.cuh) against NumPy in fp64, on each of the three
kernels normalise_launch picks from the env's image size, for every output type, and through the two callers that reach
the large-image kernels: qd_scan_obs_host and obs.observe at the env's default resolution.

Bars: the statistics equal np.percentile and the fp32 / half / uint8 images equal the reference's expression stored the
way the kernels store it (fp64 -> fp32 -> half; rint(255 x)), value for value.  NaN and inf are outside the contract:
the sensor does not produce them."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

Q_PAIRS = [(0.5, 99.5), (0.0, 100.0), (0.0, 0.0), (100.0, 100.0), (50.0, 50.0), (12.5, 87.5)]
KERNEL_NAMES = {"reg": "qd_normalise_reg_kernel<", "smem": ", true>", "global": ", false>"}


def _kernel(per_env):
    """The kernel normalise_launch (csrc/qd_api.cu) runs for an env of per_env pixels."""
    if per_env <= 32 * 1024:                  # 1024 threads x 32 values in registers
        return "reg"
    return "smem" if per_env * 4 <= 200 * 1024 else "global"


def _reference(z, per_env, q_low, q_high):
    """QuantumDeviceEnv._normalise_obs (env.py:471-509) per env block, in fp64: stats [n_env, 2] and the image in [0, 1]."""
    img = np.asarray(z, dtype=np.float64).reshape(-1, per_env)
    lo = np.percentile(img, q_low, axis=1, keepdims=True)
    hi = np.percentile(img, q_high, axis=1, keepdims=True)
    with np.errstate(invalid="ignore", divide="ignore"):
        want = np.where(hi > lo, np.clip((img - lo) / (hi - lo), 0.0, 1.0), 0.0)
    return np.concatenate([lo, hi], axis=1), want


def _typed(want, z_type):
    """The kernels' store of a normalised fp64 value: fp32; half via fp32 (two roundings); uint8 = rint(255 v)."""
    from qdsim import Z_F16, Z_F32
    if z_type == Z_F32:
        return want.astype(np.float32)
    if z_type == Z_F16:
        return want.astype(np.float32).astype(np.float16)
    return np.rint(255.0 * want).astype(np.uint8)


def _mismatch(got, want, what):
    """None if got equals want value for value, else how they differ (in units of the type's last bit on [0.5, 1))."""
    got = np.asarray(got).reshape(want.shape)
    if np.array_equal(got, want):
        return None
    bad = got != want
    lsb = 1.0 if want.dtype == np.uint8 else float(np.spacing(want.dtype.type(0.5)))
    err = np.abs(got.astype(np.float64) - want.astype(np.float64)).max() / lsb
    return f"{what}: {bad.sum()} of {bad.size} values differ ({bad.mean():.2%}), by up to {err:.3g} LSB"


def _assert_same(got, want, what):
    msg = _mismatch(got, want, what)
    if msg:
        pytest.fail(msg)


def _assert_stats(got, want, what):
    got = np.asarray(got)
    if not np.array_equal(got, want):                           # -0.0 == +0.0: a tie of signed zeros may pick either
        i = np.argwhere(got != want)[0]
        pytest.fail(f"{what}: stats differ at env {i[0]}: {got[tuple(i)]!r} != {want[tuple(i)]!r}")


def _image(kind, n_env, n, rng):
    """n_env images of n float32 pixels of one kind, each env drawn on its own."""
    z = rng.normal(0.6, 0.3, (n_env, n)).astype(np.float32)
    ties = 1500 if n > 3000 else n // 2                         # > 1024 ties defeat the register kernel's short lists
    for e in range(n_env):
        if kind == "constant":
            z[e] = 0.0
        elif kind == "two_values":
            z[e] = np.where(rng.random(n) < 0.5, np.float32(0.1), np.float32(0.9))
        elif kind == "ties_min":
            z[e, rng.choice(n, ties, replace=False)] = z[e].min() - 1.0
        elif kind == "ties_max":
            z[e, rng.choice(n, ties, replace=False)] = z[e].max() + 0.5
        elif kind == "signed_zeros":
            z[e] = rng.normal(0.0, 1e-3, n).astype(np.float32)
            z[e, ::7] = 0.0
            z[e, 3::5] = -0.0
        elif kind == "binades":                                 # every radix byte decided by a histogram
            z[e] = (rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-30, 30, n)).astype(np.float32)
        elif kind == "sensor_like":                             # plateaus + 1e-4 noise, like a real charge-sensor image
            z[e] = (np.float32(0.0305) + np.float32(1e-4) * rng.standard_normal(n)).astype(np.float32)
            z[e, : n // 3] += np.float32(0.4)
    return z


def _normalise_all(engine, z, per_env, n_env, q_low, q_high, what):
    """Every output type and buffer arrangement of one image against the reference: fp32 into its own buffer with stats,
    fp32 in place (as obs.observe calls it) without, half with stats, uint8 without.  Each output buffer carries a guard
    tail that must come back untouched, and the input must too."""
    import torch
    from qdsim import Z_F16, Z_F32, Z_U8
    n, guard = n_env * per_env, 256
    stats_want, want = _reference(z, per_env, q_low, q_high)
    z_dev = torch.from_numpy(np.ascontiguousarray(z).reshape(-1)).cuda()

    def buffer(dtype, fill):
        b = torch.full((n + guard,), fill, dtype=dtype, device="cuda")
        return b, b[:n]

    results = []
    f32_buf, f32 = buffer(torch.float32, -3.0)
    stats = torch.full((n_env, 2), np.nan, dtype=torch.float64, device="cuda")
    engine.normalise_obs(z_dev, out=f32, per_env=per_env, n_env=n_env, q_low=q_low, q_high=q_high, stats=stats)
    results.append((Z_F32, "fp32", f32_buf, stats))
    inplace_buf, inplace = buffer(torch.float32, -3.0)
    inplace.copy_(z_dev)
    engine.normalise_obs(inplace, per_env=per_env, n_env=n_env, q_low=q_low, q_high=q_high)
    results.append((Z_F32, "fp32 in place", inplace_buf, None))
    f16_buf, f16 = buffer(torch.float16, -3.0)
    stats16 = torch.full((n_env, 2), np.nan, dtype=torch.float64, device="cuda")
    engine.normalise_obs_typed(z_dev, f16, Z_F16, per_env=per_env, n_env=n_env, q_low=q_low, q_high=q_high,
                               stats=stats16)
    results.append((Z_F16, "half", f16_buf, stats16))
    u8_buf, u8 = buffer(torch.uint8, 0xAB)
    engine.normalise_obs_typed(z_dev, u8, Z_U8, per_env=per_env, n_env=n_env, q_low=q_low, q_high=q_high)
    results.append((Z_U8, "uint8", u8_buf, None))
    torch.cuda.synchronize()
    assert np.array_equal(z_dev.cpu().numpy(), np.asarray(z).reshape(-1)), f"{what}: the input was written"
    for z_type, name, buf, st in results:
        host = buf.cpu().numpy()
        assert (host[n:] == host[-1]).all() and host[-1] == (0xAB if z_type == Z_U8 else -3.0), \
            f"{what}, {name}: written past the last env"
        if st is not None:
            _assert_stats(st.cpu().numpy(), stats_want, f"{what}, {name}")
    msgs = [_mismatch(buf.cpu().numpy()[:n], _typed(want, z_type), f"{what}, {name}")
            for z_type, name, buf, _ in results]
    if any(msgs):
        pytest.fail("\n".join(m for m in msgs if m))
    return stats_want


SIZES = [(1, "reg"), (2, "reg"), (1023, "reg"), (1024, "reg"), (1025, "reg"), (32767, "reg"), (32768, "reg"),
         (32769, "smem"), (40000, "smem"), (40001, "smem"), (51200, "smem"),
         (51201, "global"), (70000, "global"), (70001, "global")]
KINDS = ["constant", "two_values", "ties_min", "ties_max", "signed_zeros", "binades", "sensor_like"]


@pytest.mark.parametrize("per_env,kernel", SIZES, ids=[f"{n}-{k}" for n, k in SIZES])
@pytest.mark.parametrize("kind", KINDS)
def test_normalisation_equals_numpy_for_every_kernel_type_and_percentile_pair(engine, per_env, kernel, kind):
    """Boundaries of the three size classes (1 / 2 pixels, 1024 threads, 32 x 1024 registers, 200 KB of shared memory),
    sizes that are not a multiple of 32 (the n_round tail of qd_normalise_kernel), the 5- and 8-dot envs at the default
    resolution 100 (40 000 and 70 000 pixels); extreme, full-range, single-rank and interior percentile pairs."""
    assert _kernel(per_env) == kernel
    n_env = 3
    rng = np.random.default_rng([per_env, KINDS.index(kind)])
    z = _image(kind, n_env, per_env, rng)
    for q_low, q_high in Q_PAIRS:
        _normalise_all(engine, z, per_env, n_env, q_low, q_high, f"{kind}, per_env {per_env}, q ({q_low}, {q_high})")


def test_each_size_class_runs_the_kernel_it_is_named_for(engine):
    """The size classes above, as the launches themselves report them (kernel names in a torch.profiler trace)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from qdsim import Z_U8
    for per_env in [32768, 32769, 51200, 51201]:
        z = torch.rand(2 * per_env, device="cuda")
        out = torch.empty(2 * per_env, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            engine.normalise_obs_typed(z, out, Z_U8, per_env=per_env, n_env=2)
            torch.cuda.synchronize()
        names = [e.key for e in prof.key_averages() if "qd_normalise" in e.key]
        assert len(names) == 1, names
        assert KERNEL_NAMES[_kernel(per_env)] in names[0], (per_env, names)
        assert "unsigned char" in names[0]


@pytest.mark.parametrize("per_env", [7 * 64 * 64, 40000, 70000])
@pytest.mark.parametrize("ratio", [1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6])
def test_normalisation_is_exact_when_the_spread_is_small_next_to_the_level(engine, per_env, ratio):
    """level + sigma N(0, 1) in fp32 with p_low / (p_high - p_low) ~ ratio: the case where an output computed as
    x * (1 / span) - p_low / span in fp32 loses about log2(ratio) bits."""
    level = 3.0
    sigma = level / (2 * 2.5758 * ratio)                         # the 0.5 .. 99.5 % spread of a normal is 5.15 sigma
    rng = np.random.default_rng(int(np.log10(ratio)) + per_env)
    z = (level + sigma * rng.standard_normal((4, per_env))).astype(np.float32)
    stats = _normalise_all(engine, z, per_env, 4, 0.5, 99.5, f"{_kernel(per_env)}, per_env {per_env}, ratio {ratio:g}")
    reached = stats[:, 0] / (stats[:, 1] - stats[:, 0])
    assert (reached > ratio / 3).all() and (reached < ratio * 3).all(), reached


@pytest.mark.parametrize("per_env", [1000, 32769, 51201])
def test_normalisation_of_many_envs_runs_in_several_waves(engine, per_env):
    """600 envs: one CTA of 1024 threads per env and at most one per SM, so the grid runs in several waves.  Each env has
    its own level and spread (p_low / span up to ~1e5), every seventh is constant."""
    n_env = 600
    rng = np.random.default_rng(per_env)
    level = rng.uniform(-5.0, 5.0, (n_env, 1))
    spread = np.abs(level) * 10.0 ** rng.uniform(-6.0, 0.0, (n_env, 1)) + 1e-6
    z = (level + spread * rng.standard_normal((n_env, per_env))).astype(np.float32)
    z[::7] = np.float32(1.25)
    _normalise_all(engine, z, per_env, n_env, 0.5, 99.5, f"{n_env} envs of {per_env}")


def _scans_16(engine, n_scan, seed):
    """n_scan 16 x 16 scans of 5-dot devices (four per device), latching + white / telegraph / radial noise."""
    from qdsim import synth
    dev = synth.sample_devices(n_scan // 4, 5, seed=seed)
    mb = synth.model_batch(dev)
    engine.set_models(mb)
    return synth.env_step_scans(mb, dev, res=16, seed=seed + 1, offset_range=3.0)


@pytest.mark.parametrize("scans_per_env,kernel", [(160, "smem"), (256, "global")])
def test_obs_host_normalises_large_envs_across_chunks(engine, scans_per_env, kernel):
    """qd_scan_obs_host with scans_per_env consecutive scans per env: 40 960 or 65 536 pixels per env, 6400 scans, so the
    call is cut into three chunks of envs (n_scan / 2048, chunk borders on env borders), each normalised with its own
    stats offset.  Every env's stats and image against the reference applied to the same call's raw fp32 image."""
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, Z_F16, Z_F32, Z_U8
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    scans = _scans_16(engine, 6400, seed=31)
    per_env = scans_per_env * 256
    assert _kernel(per_env) == kernel and len(scans) // 2048 == 3
    raw, _ = engine.scan_obs_host(scans, z_type=Z_F32, flags=flags, normalise=False, scans_per_env=scans_per_env)
    assert np.unique(raw).size > 1000
    stats_want, want = _reference(raw, per_env, 0.5, 99.5)
    for z_type, name in [(Z_F32, "fp32"), (Z_F16, "half"), (Z_U8, "uint8")]:
        img, stats = engine.scan_obs_host(scans, z_type=z_type, flags=flags, want_stats=True, scans_per_env=scans_per_env)
        _assert_stats(stats, stats_want, f"{kernel}, {name}")
        _assert_same(img, _typed(want, z_type), f"{kernel}, {name}")


@pytest.mark.parametrize("n_dot,kernel", [(5, "smem"), (8, "global")])
def test_observe_at_the_default_resolution_normalises_in_place_like_numpy(engine, n_dot, kernel):
    """obs.observe as BatchedDeviceEnv.step calls it at EnvConfig.resolution = 100: the 5-dot (40 000 pixels per env) and
    8-dot (70 000) envs normalise in place in the shared-memory and the global-memory kernel."""
    import torch
    from qdsim import obs, synth
    n_env, res = 3, 100
    rng = np.random.default_rng(n_dot)
    dev = synth.sample_devices(n_env, n_dot, seed=n_dot)
    mb = synth.model_batch(dev)
    engine.set_models(mb)
    gv = rng.uniform(-2, 4, (n_env, n_dot))
    vgm = -np.eye(n_dot + 1) + rng.normal(0, 0.05, (n_env, n_dot + 1, n_dot + 1))
    origin = rng.normal(0, 0.1, (n_env, n_dot + 1))
    scans = obs.obs_scans(mb, gv, rng.uniform(0.3, 0.7, n_env), vgm, origin, -1.8, 1.8, res,
                          peak_width=dev["peak_width"], seeds=np.arange(n_env * (n_dot - 1)) + 11)
    per_env = (n_dot - 1) * res * res
    assert _kernel(per_env) == kernel
    raw = torch.empty(n_env * per_env, dtype=torch.float32, device="cuda")
    img = torch.empty_like(raw)
    obs.observe(engine, scans, raw, normalise=False)
    out = obs.observe(engine, scans, img)
    torch.cuda.synchronize()
    assert out.shape == (n_env, n_dot - 1, res, res)
    _, want = _reference(raw.cpu().numpy(), per_env, 0.5, 99.5)
    for e in range(n_env):
        _assert_same(out[e].cpu().numpy(), want[e].astype(np.float32), f"{n_dot} dots, env {e}")
