"""Parity ON THE BENCHED CONFIGURATION (BASELINE config 4 as bench.py times it: 8-dot latched array, 64x64 windows,
offset_range = 5.0, latching + white / telegraph / radial noise) -- not on a smaller cousin of it: thousands of the very
scans of the timed batch are re-run by the plain-C restatement (oracle/cport) and compared bit for bit (charge maps) and at
5e-6 absolute (sensor images).  bench.py prints the same check as ``parity_sample`` on every run.

Path B (what env.step runs): the same for the tunnel-coupled workload of ``bench.py --path B`` against the C restatement
of the reference's formulation (oracle/cport/qd_cport_b.c), on as many pixels as that 4^N-candidate code finishes in
seconds."""
import os

import numpy as np
import pytest

from util import cport_parity

pytestmark = pytest.mark.gpu


def test_benched_path_a_batch_matches_c_restatement(engine):
    import bench
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_U8
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    n_env, n_dot, res = 2048, 8, 64
    dev, mb, sets = bench.build_workload(n_env, n_dot, res, 0, 1, "A")       # the bench's own builder, rank 0, step 0
    scans = sets[0]
    engine.set_models(mb)
    z, n = engine.scan_open_host(scans, n_type=N_U8, flags=flags)
    rng = np.random.default_rng(7)
    pick = np.sort(rng.choice(len(scans), size=2240, replace=False))
    rep = bench.parity_sample(mb, scans, flags, z, n, pick, res)
    assert rep["scans"] == 2240 and rep["pixels"] == 2240 * res * res
    assert rep["n_mismatch"] == 0, rep
    assert rep["z_max_abs"] <= 5e-6, rep
    assert rep["tie_rows"] <= 0.005 * rep["rows"], rep
    # the first 2048 envs of the 16384-env bench batch are exactly this batch (same seeds, env-major sampling)? No --
    # the device generator draws per-array blocks of size n_env, so assert only what is true: same builder, same flags.


def test_benched_path_b_batch_matches_c_restatement(engine):
    import bench
    from oracle import composer, cport
    from qdsim import N_F64
    from util import oracle_model, oracle_scan
    n_env, n_dot, res = 4, 8, 64
    dev, mb, sets = bench.build_workload(n_env, n_dot, res, 0, 1, "B")
    scans = sets[0][:4].copy()                                                # 4 windows of 64 x 64 = 16384 pixels
    scans["pix_offset"] = np.arange(len(scans)) * res * res
    engine.set_models(mb)
    z, n = engine.scan_open_host(scans, n_type=N_F64, flags=0)
    n = n.reshape(len(scans), res * res, n_dot)
    cores = os.cpu_count() or 1
    worst = 0.0
    for i, rec in enumerate(scans):
        m = oracle_model(mb, int(rec["env_id"]), 0)
        s = oracle_scan(rec, mb.n_volt, 0)
        v = composer.affine_grid(s.v0, s.dx, s.dy, s.nx, s.ny).reshape(-1, mb.n_volt)
        n_ref, gap, _ = cport.tunnel_ground_state(m, v, threads=cores)
        ok = gap > 1e-5
        assert ok.mean() > 0.95
        err = np.abs(n[i] - n_ref)[ok].max()
        worst = max(worst, float(err))
        assert err <= 2e-6, f"scan {i}: max |<n> - <n>_ref| = {err:.2e}"
    print(f"benched Path B sample: 16384 pixels, max |d<n>| = {worst:.2e}")


# The two Path A configurations tools/sweep.py times besides the headline.  Its builders are inline in main(), so they are
# restated here; the flags are sweep.py's FLAGS (sweep.py:25), with FLAG_THERMAL added for the thermal variant.
def _sample(scans, z, n, n_dot, res, size, seed):
    """``size`` seeded scans of a batch laid out at pix_offset = i * res^2, re-laid out the same way."""
    pick = np.sort(np.random.default_rng(seed).choice(len(scans), size=size, replace=False))
    sub = scans[pick].copy()
    sub["pix_offset"] = np.arange(size) * res * res
    return sub, z.reshape(len(scans), res * res)[pick], n.reshape(len(scans), res * res, n_dot)[pick]


def test_benched_config3_brute_force_matches_c_restatement(engine):
    """BASELINE config 3 at sweep.py --quick size (sweep.py:177-181): 256 envs, 6 dots, brute_force, max_charge_carriers
    = 4, seeds 4 / 5, 64 x 64, latching + noise.  The whole batch runs; 8 seeded scans are compared with the C port."""
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_U8, synth
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    res, n_dot = 64, 6
    dev = synth.sample_devices(256, n_dot, seed=4)
    mb = synth.model_batch(dev, algorithm="brute_force", max_charge_carriers=4)
    scans = synth.env_step_scans(mb, dev, res=res, seed=5)
    engine.set_models(mb)
    z, n = engine.scan_open_host(scans, n_type=N_U8, flags=flags)
    sub, zs, ns = _sample(scans, z, n, n_dot, res, 8, seed=3)
    rep = cport_parity(mb, sub, flags, zs.reshape(-1), ns.reshape(-1, n_dot), threads=os.cpu_count() or 1)
    assert rep["n_mismatch"] == 0 and rep["z_max_abs"] <= 5e-6, rep
    assert rep["tie_rows"] <= 0.02 * rep["rows"], rep


def test_benched_thermal_variant_matches_c_restatement(engine):
    """The thermal variant of config 4 (sweep.py:139-144): 2048 envs, 8 dots, T ~ U[50, 200] mK, seeds 8 / 9, 64 x 64,
    latching + noise, N_F32 occupations.  The whole batch runs; 64 seeded scans are compared with the C port by the causal
    latching check, and the sample must send warps to the block accumulation of the Boltzmann average."""
    from oracle import cport
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, FLAG_THERMAL, N_F32, synth
    from test_search_gpu import block_warp_share, check_thermal_latched
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL | FLAG_THERMAL
    res, n_dot = 64, 8
    dev = synth.sample_devices(2048, n_dot, seed=8)
    mb = synth.model_batch(dev, thermal=True)
    scans = synth.env_step_scans(mb, dev, res=res, seed=9)
    engine.set_models(mb)
    z, n = engine.scan_open_host(scans, n_type=N_F32, flags=flags)
    sub, zs, ns = _sample(scans, z, n, n_dot, res, 64, seed=5)
    assert block_warp_share(mb, sub) > 0.05
    threads = os.cpu_count() or 1
    zc, nc, _ = cport.run_scans(mb, sub, flags, threads=threads)
    _, nf, _ = cport.run_scans(mb, sub, flags & ~FLAG_LATCH, threads=threads)
    shape = (len(sub), res, res)
    # N_F32: the fp32 rounding of <n> <= 8 is below 1e-6; the latch decisions were made on the fp64 <n>
    check_thermal_latched(zs.reshape(shape), ns.reshape(shape + (n_dot,)), zc.reshape(shape), nc.reshape(shape + (n_dot,)),
                          nf.reshape(shape + (n_dot,)), carry_rows=False, noisy=True, n_atol=1e-6)
