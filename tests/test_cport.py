"""The plain-C restatement (oracle/cport) agrees with the NumPy oracle on seeded inputs.  CPU only."""
import numpy as np
import pytest

from util import oracle_batch


# (n_dot, algorithm, max_charge_carriers, flags, offset_range).  The brute-force and 8-dot thermal cases use windows up
# to 6 V off the set point, so that dots sit below 0 and above max_charge_carriers: the box edges of the search.
@pytest.mark.parametrize("n_dot,alg,maxc,flag_names,offset_range", [
    (2, "default", 4, (), 3.0), (4, "default", 4, ("LATCH", "NOISE", "RADIAL"), 3.0),
    (4, "default", 4, ("LATCH", "NOISE", "CARRY_ROWS"), 3.0), (6, "default", 4, ("LATCH",), 3.0),
    (5, "thresholded", 4, (), 3.0), (3, "brute_force", 4, (), 3.0), (4, "default", 4, ("THERMAL",), 3.0),
    (3, "default", 4, ("NOISE", "WHITE_ON_OUTPUT"), 3.0),
    (3, "brute_force", 15, ("THERMAL",), 6.0), (4, "brute_force", 0, (), 6.0),
    (4, "brute_force", 1, ("THERMAL", "LATCH"), 6.0), (5, "brute_force", 4, ("THERMAL",), 6.0),
    (8, "default", 4, ("THERMAL",), 6.0), (8, "thresholded", 4, ("THERMAL",), 6.0),
    (3, "brute_force", 15, ("LATCH", "NOISE"), 6.0),
])
def test_cport_matches_numpy_oracle(n_dot, alg, maxc, flag_names, offset_range):
    import qdsim
    from oracle import cport
    from qdsim import synth
    flags = 0
    for f in flag_names:
        flags |= getattr(qdsim, "FLAG_" + f)
    dev = synth.sample_devices(2, n_dot, seed=40 + n_dot)
    mb = synth.model_batch(dev, algorithm=alg, thermal="THERMAL" in flag_names, threshold=0.6, max_charge_carriers=maxc)
    mb.params["tele_p01"], mb.params["tele_p10"], mb.params["tele_amp"] = 0.04, 0.07, 0.01
    res = 24 if n_dot < 8 else 12
    scans = synth.env_step_scans(mb, dev, res=res, seed=5, offset_range=offset_range)
    scans["rad_zero_radius"], scans["rad_alpha"] = 1.0, 0.02
    z, n, _ = cport.run_scans(mb, scans, flags, threads=2)
    z_ref, n_ref, _ = oracle_batch(mb, scans, flags)
    np.testing.assert_allclose(n.reshape(n_ref.shape), n_ref, rtol=0, atol=1e-10)
    np.testing.assert_allclose(z.reshape(z_ref.shape), z_ref, rtol=3e-7, atol=1e-7)


@pytest.mark.parametrize("n_dot,vc", [(4, False), (5, False), (6, True), (8, False)])
def test_tunnel_cport_matches_numpy_oracle(n_dot, vc):
    """Path B in plain C (reference formulation: all 4^N candidates, Jacobi eigen-solve) against the NumPy restatement."""
    from oracle import composer, cport, path_b
    from qdsim import synth
    from util import oracle_model, oracle_scan
    dev = synth.sample_barrier_devices(1, n_dot, seed=60 + n_dot)
    mb = synth.tunnel_batch(dev)
    if vc:
        mb.params["vc_alpha"], mb.params["vc_beta"] = 0.07, 0.05
    res = 10 if n_dot <= 6 else 5
    scans = synth.env_step_scans(mb, dev, res=res, seed=61, offset_range=2.5)
    m = oracle_model(mb, 0, 0)
    s = oracle_scan(scans[1], mb.n_volt, 0)
    v = composer.affine_grid(s.v0, s.dx, s.dy, s.nx, s.ny).reshape(-1, mb.n_volt)
    n_ref, gap_ref = path_b.ground_state_open(m, v, return_gap=True)
    n_c, gap_c, _ = cport.tunnel_ground_state(m, v, threads=2)
    ok = gap_ref > 1e-6
    assert ok.mean() > 0.95
    np.testing.assert_allclose(n_c[ok], n_ref[ok], rtol=0, atol=1e-9)
    np.testing.assert_allclose(gap_c[ok], gap_ref[ok], rtol=1e-7, atol=1e-10)


@pytest.mark.parametrize("name", ["ref_4dot_tunnel_identity_vgm", "ref_6dot_tunnel_linear_capacitance",
                                  "ref_4dot_tunnel_strong_coupling", "ref_4dot_constant_tc_no_barriers"])
def test_tunnel_cport_matches_the_reference_itself(name):
    """... and against the fixtures the reference's own code produced (tests/golden/make_reference_golden.py)."""
    import test_reference_golden as t
    from oracle import cport
    from util import oracle_model
    d = t.load(name)
    mb = t.product_model(d)
    m = oracle_model(mb, 0, 0)
    v = t.v_ext(d).reshape(-1, mb.n_volt)
    n_c, gap_c, _ = cport.tunnel_ground_state(m, v, threads=2)
    ok = gap_c > 1e-6
    np.testing.assert_allclose(n_c[ok], d["n"].reshape(-1, n_c.shape[1])[ok], rtol=0, atol=1e-9)
