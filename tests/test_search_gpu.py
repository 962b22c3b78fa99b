"""Path A's exact searches against the references, at the dot counts and branches where they diverge.

Thermal launches and brute-force launches always run the general scan kernel (``qd_scan_kernel``), so the fast/generic
A/B test never sees them.  This file compares them with the NumPy oracle, or with the plain-C restatement
(oracle/cport) where the oracle's dense candidate arrays would be too large:

* brute force (``ground_state_brute``): 2..8 dots, max_charge_carriers from 0 to 15, windows with dots pinned to BOTH faces
  of the box [0, max_charge_carriers], per-item tree orders (one scan alone vs. the same scan inside a big batch), the
  identity tree order of explicit voltage lists, and the thermal second walk (PASS 1);
* the Boltzmann average of ``ground_state_box``: the Gray-code walk (at most six dots left free by the 40 kT dominance
  test in a warp) and the block accumulation (more than six), the non-integral latching carry across 32-pixel chunks,
  and the non-affine (voltage list) instance.

Every case first asserts that it reaches what it is named for, from the host-side helpers ``thermal_wide_warps`` and
``pinned_faces``: a change of the synthetic inputs cannot quietly turn it into a weaker case.

Bars: hard argmin bit-exact wherever best / second-best margin > 1e-9 (rows with such a near-tie are skipped under
latching); thermal <n> within 1e-9 (N_F64), N_F32 equal to float32 of the N_F64 output; thermal + latching by the causal
check of ``util.explain_latched_mismatches``; z noise-free rtol 1e-6 (+ atol 1e-7 for the fp32 C port or thermal
outputs), noisy atol 5e-6.
"""
import os

import numpy as np
import pytest

from util import compare_charges, explain_latched_mismatches, oracle_batch

pytestmark = pytest.mark.gpu

TIE = 1e-9
Z_RTOL, Z_ATOL, Z_NOISY_ATOL = 1e-6, 1e-7, 5e-6
N_ATOL_THERMAL = 1e-9


# ---------------------------------------------------------------------------------------------------------------------
# host-side reach predicates
# ---------------------------------------------------------------------------------------------------------------------
def potentials(mb, scan):
    """g = cgd . v of every pixel of an affine scan record, (ny, nx, N)."""
    from oracle import composer
    nv, n = mb.n_volt, mb.n_dot
    v = composer.affine_grid(scan["v0"][:nv], scan["dx"][:nv], scan["dy"][:nv], int(scan["nx"]), int(scan["ny"]))
    return v @ mb.cgd_full[int(scan["env_id"]), :n, :].T


def thermal_wide_warps(mb, scan, kT):
    """Per 32-pixel warp (ny, ceil(nx / 32)): the largest number of dots the 40 kT dominance test of
    ``ground_state_box`` leaves free, with the thresholded fixes applied.  More than six sends the warp to the block
    accumulation, at most six to the Gray-code walk.  Mirrors the kernel: exact relaxation -> floor -> lin = 2 Cinv (f - g)
    -> a_j = lin_j + Cinv_jj; dot j is fixed when a_j + sneg_j > 40 kT or a_j + spos_j < -40 kT, where spos / sneg sum the
    positive / negative off-diagonal entries of 2 Cinv in row j."""
    from oracle.path_a import continuous_relaxation
    e, n = int(scan["env_id"]), mb.n_dot
    nx, ny = int(scan["nx"]), int(scan["ny"])
    g = potentials(mb, scan).reshape(-1, n)
    cinv = mb.cdd_inv_gs[e]
    nc = continuous_relaxation(g, mb.cdd_gs[e])
    f = np.floor(nc)
    a = 2.0 * (f - g) @ cinv.T + np.diag(cinv)
    off = 2.0 * (cinv - np.diag(np.diag(cinv)))
    spos, sneg = np.where(off > 0, off, 0.0).sum(axis=1), np.where(off < 0, off, 0.0).sum(axis=1)
    cut = 40.0 * kT
    fixed = (a + sneg > cut) | (a + spos < -cut)
    if mb.algorithm == "thresholded":
        fixed |= ~(np.abs(nc - f - 0.5) < 0.5 * float(mb.params["threshold"][e]))
    free = (n - fixed.sum(axis=1)).reshape(ny, nx)
    chunks = -(-nx // 32)
    free = np.pad(free, ((0, 0), (0, chunks * 32 - nx)), mode="edge")       # idle lanes repeat the last pixel
    return free.reshape(ny, chunks, 32).max(axis=2)


def pinned_faces(mb, scan, maxc):
    """(low, high) masks (ny, nx): pixels with some g_j < -0.5 (a dot pinned to 0 carriers) and with some
    g_j > maxc + 0.5 (a dot pinned to max_charge_carriers)."""
    g = potentials(mb, scan)
    return (g < -0.5).any(axis=-1), (g > maxc + 0.5).any(axis=-1)


def block_warp_share(mb, scans):
    w = np.concatenate([thermal_wide_warps(mb, s, float(mb.params["kT"][int(s["env_id"])])).ravel() for s in scans])
    return float((w > 6).mean())


# ---------------------------------------------------------------------------------------------------------------------
# inputs, runs and references
# ---------------------------------------------------------------------------------------------------------------------
def make_case(n_dot, algorithm="brute_force", maxc=4, n_env=2, n_scans=None, res=32, seed=11, offset_range=3.0,
              thermal=False, kT_scale=1.0, latching=False, noise=False, threshold=0.6):
    from qdsim import synth
    dev = synth.sample_devices(n_env, n_dot, seed=seed)
    mb = synth.model_batch(dev, algorithm=algorithm, thermal=thermal, latching=latching, noise=noise,
                           max_charge_carriers=maxc, threshold=threshold)
    mb.params["kT"] *= kT_scale
    if noise:
        mb.params["tele_p01"], mb.params["tele_p10"], mb.params["tele_amp"] = 0.04, 0.09, 0.01
    scans = synth.env_step_scans(mb, dev, res=res, seed=seed + 1, offset_range=offset_range)
    if n_scans is not None:
        scans = scans[:n_scans].copy()
    scans["rad_zero_radius"], scans["rad_alpha"] = 1.0, 0.02
    return mb, scans


def run_gpu(engine, mb, scans, n_type, flags):
    """(z (S, ny, nx), n (S, ny, nx, N)) of scans laid out at pix_offset = i * nx * ny."""
    engine.set_models(mb)
    ny, nx = int(scans["ny"][0]), int(scans["nx"][0])
    assert (scans["pix_offset"] == np.arange(len(scans)) * nx * ny).all()
    z, n = engine.scan_open_host(scans, n_type=n_type, flags=flags)
    return z.reshape(len(scans), ny, nx), n.reshape(len(scans), ny, nx, mb.n_dot)


def reference(mb, scans, flags, use_cport):
    """(z, n, margin) stacked per scan, from the NumPy oracle or (``use_cport``) the C restatement."""
    if not use_cport:
        return oracle_batch(mb, scans, flags)
    from oracle import cport
    sc = np.ascontiguousarray(scans).copy()
    S, ny, nx = len(sc), int(sc["ny"][0]), int(sc["nx"][0])
    sc["pix_offset"] = np.arange(S) * nx * ny
    z, n, _, margin = cport.run_scans(mb, sc, flags, threads=os.cpu_count() or 1, want_margin=True)
    return (z.astype(np.float64).reshape(S, ny, nx), n.reshape(S, ny, nx, mb.n_dot), margin.reshape(S, ny, nx))


def check_hard(z, n, z_ref, n_ref, margin, flags, fp32_ref):
    from qdsim import FLAG_CARRY_ROWS, FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL
    if flags & FLAG_LATCH:
        # a near-tie upstream changes what the latch sees downstream in the same sequence: skip those rows
        tie = (margin <= TIE).any(axis=2)
        if flags & FLAG_CARRY_ROWS:
            tie[:] = tie.any(axis=1, keepdims=True)
        assert tie.mean() <= 0.02, f"too many rows with a near-tie: {tie.mean():.3f}"
        safe = np.repeat(~tie[:, :, None], z.shape[2], axis=2)
        bad = (n.astype(np.int64) != np.rint(n_ref).astype(np.int64)).any(axis=-1) & safe
        assert not bad.any(), f"{bad.sum()} of {safe.sum()} pixels differ, first at {np.argwhere(bad)[:5]}"
    else:
        compare_charges(n, n_ref, margin)
        safe = margin > TIE
    if flags & (FLAG_NOISE | FLAG_RADIAL):
        np.testing.assert_allclose(z[safe], z_ref[safe], rtol=0, atol=Z_NOISY_ATOL)
    else:
        np.testing.assert_allclose(z[safe], z_ref[safe], rtol=Z_RTOL, atol=Z_ATOL if fp32_ref else 0.0)


def check_thermal(z, n, z_ref, n_ref, noisy=False):
    np.testing.assert_allclose(n, n_ref, rtol=0, atol=N_ATOL_THERMAL)
    np.testing.assert_allclose(z, z_ref, rtol=0 if noisy else Z_RTOL, atol=Z_NOISY_ATOL if noisy else Z_ATOL)


def check_thermal_latched(z, n, z_ref, n_ref, n_free_ref, carry_rows, noisy=False, n_atol=N_ATOL_THERMAL):
    """Causal check: every pixel whose latched <n> differs lies downstream, in its latching sequence, of a pixel whose
    unlatched <n> is within 1e-9 of a half-integer (where the rounded latch compare may go either way)."""
    differing = 0
    for i in range(len(z)):
        d, _, _ = explain_latched_mismatches(n[i], n_ref[i], n_free_ref[i], np.full(z[i].shape, np.inf),
                                             carry_rows=carry_rows, n_atol=n_atol, half_tol=1e-9)
        differing += d
    assert differing <= 0.01 * z.size, f"{differing} of {z.size} latched pixels differ"
    ok = np.abs(n - n_ref).max(axis=-1) <= n_atol
    np.testing.assert_allclose(z[ok], z_ref[ok], rtol=0 if noisy else Z_RTOL, atol=Z_NOISY_ATOL if noisy else Z_ATOL)


def assert_fractional(n, what):
    assert (np.abs(n - np.rint(n)) > 1e-3).mean() > 0.001, f"{what}: kT > 0 must give non-integer occupations"


def points_of(mb, rec):
    from oracle import composer
    nv = mb.n_volt
    return composer.affine_grid(rec["v0"][:nv], rec["dx"][:nv], rec["dy"][:nv], int(rec["nx"]), int(rec["ny"]))


# ---------------------------------------------------------------------------------------------------------------------
# brute force, hard argmin
# ---------------------------------------------------------------------------------------------------------------------
# (n_dot, max_charge_carriers, scans, resolution, offset_range).  The C port visits all (maxc + 1)^N candidates, so the
# 8-dot cases stay at <= 512 / 2048 pixels.
BF_FACES = [(2, 15, 6, 32, 18.0), (3, 15, 4, 32, 18.0), (4, 7, 3, 32, 10.0), (5, 4, 4, 32, 6.0), (6, 4, 3, 32, 6.0),
            (7, 3, 2, 32, 6.0), (8, 2, 2, 32, 6.0), (8, 4, 2, 16, 6.0)]


def bf_faces_case(n_dot, maxc, n_scans, res, offset_range):
    """``n_scans`` windows out of a pool of 16 envs: alternately the one with the most pixels pinned to the lower face
    and the one with the most pinned to the upper face."""
    mb, pool = make_case(n_dot, maxc=maxc, n_env=16, res=res, seed=100 + 10 * n_dot + maxc, offset_range=offset_range)
    faces = [pinned_faces(mb, s, maxc) for s in pool]
    lows = np.argsort([-lo.mean() for lo, _ in faces], kind="stable")
    highs = np.argsort([-hi.mean() for _, hi in faces], kind="stable")
    pick = []
    for a, b in zip(lows, highs):
        pick += [int(i) for i in (a, b) if i not in pick]
    scans = np.ascontiguousarray(pool[sorted(pick[:n_scans])])
    scans["pix_offset"] = np.arange(len(scans)) * res * res
    return mb, scans


@pytest.mark.parametrize("n_dot,maxc,n_scans,res,offset_range", BF_FACES)
def test_brute_force_both_faces(engine, n_dot, maxc, n_scans, res, offset_range):
    from qdsim import N_U8
    mb, scans = bf_faces_case(n_dot, maxc, n_scans, res, offset_range)
    low = np.stack([pinned_faces(mb, s, maxc)[0] for s in scans])
    high = np.stack([pinned_faces(mb, s, maxc)[1] for s in scans])
    assert low.mean() > 0.05 and high.mean() > 0.05, (low.mean(), high.mean())
    use_cport = (maxc + 1) ** n_dot > 1000
    z, n = run_gpu(engine, mb, scans, N_U8, 0)
    z_ref, n_ref, margin = reference(mb, scans, 0, use_cport)
    check_hard(z, n, z_ref, n_ref, margin, 0, use_cport)
    assert (n == maxc).any() and (n == 0).any() and ((n > 0) & (n < maxc)).any()


@pytest.mark.parametrize("maxc", [0, 1])
def test_brute_force_degenerate_boxes(engine, maxc):
    """max_charge_carriers = 0 (a single candidate) and 1 (two values per dot)."""
    from qdsim import N_U8
    mb, scans = make_case(4, maxc=maxc, n_env=2, res=32, seed=71, offset_range=4.0)
    low = np.stack([pinned_faces(mb, s, maxc)[0] for s in scans])
    high = np.stack([pinned_faces(mb, s, maxc)[1] for s in scans])
    assert low.any() and high.any()
    z, n = run_gpu(engine, mb, scans, N_U8, 0)
    z_ref, n_ref, margin = reference(mb, scans, 0, False)
    check_hard(z, n, z_ref, n_ref, margin, 0, False)
    if maxc == 0:
        assert (n == 0).all()
    else:
        assert (n == 0).any() and (n == 1).any() and n.max() == 1


@pytest.mark.parametrize("extra", ["", "NOISE|RADIAL"])
def test_brute_force_latched_keys_up_to_15(engine, extra):
    """Integral latching on keys holding up to 15 carriers per dot (max_charge_carriers = 15, 3 dots)."""
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_U8
    flags = FLAG_LATCH | ((FLAG_NOISE | FLAG_RADIAL) if extra else 0)
    mb, scans = make_case(3, maxc=15, n_env=2, res=48, seed=81, offset_range=18.0, latching=True, noise=bool(extra))
    high = np.stack([pinned_faces(mb, s, 15)[1] for s in scans])
    assert high.mean() > 0.05
    z, n = run_gpu(engine, mb, scans, N_U8, flags)
    z_ref, n_ref, margin = reference(mb, scans, flags, True)
    check_hard(z, n, z_ref, n_ref, margin, flags, True)
    _, n_free = run_gpu(engine, mb, scans, N_U8, flags & ~FLAG_LATCH)
    assert (n_free != n).any(), "latching must reject some transitions"
    assert (n >= 10).any(), "keys above 9 must occur"


def test_brute_force_item_geometry(engine):
    """One scan launched alone (items of one 32-pixel chunk, each with its own tree order) and the same scan inside a
    batch of 512 (items of several rows): both equal the reference."""
    from qdsim import N_U8, synth
    n_dot, maxc = 5, 4
    dev = synth.sample_devices(128, n_dot, seed=91)
    mb = synth.model_batch(dev, algorithm="brute_force", latching=False, noise=False, max_charge_carriers=maxc)
    batch = synth.env_step_scans(mb, dev, res=64, seed=92, offset_range=6.0)
    assert len(batch) >= 512
    k = 77
    one = batch[k:k + 1].copy()
    one["pix_offset"] = 0
    low, high = pinned_faces(mb, one[0], maxc)
    assert low.any() and high.any()
    z1, n1 = run_gpu(engine, mb, one, N_U8, 0)
    zb, nb = run_gpu(engine, mb, batch, N_U8, 0)
    z_ref, n_ref, margin = reference(mb, one, 0, True)
    check_hard(z1, n1, z_ref, n_ref, margin, 0, True)
    check_hard(zb[k:k + 1], nb[k:k + 1], z_ref, n_ref, margin, 0, True)


def test_brute_force_points_identity_order(engine):
    """An explicit voltage list keeps the identity tree order; same answer as the reference on the affine grid."""
    from qdsim import N_U8
    maxc = 7
    mb, scans = bf_faces_case(4, maxc, 3, 48, 10.0)
    low = np.stack([pinned_faces(mb, s, maxc)[0] for s in scans])
    high = np.stack([pinned_faces(mb, s, maxc)[1] for s in scans])
    assert low.mean() > 0.05 and high.mean() > 0.05, (low.mean(), high.mean())
    engine.set_models(mb)
    n_all = []
    for i, rec in enumerate(scans):
        z, n = engine.points_open_host(rec, points_of(mb, rec), n_type=N_U8, flags=0)
        z_ref, n_ref, margin = reference(mb, scans[i:i + 1], 0, True)
        check_hard(z[None], n[None], z_ref, n_ref, margin, 0, True)
        n_all.append(n)
    n_all = np.stack(n_all)
    assert (n_all == maxc).any() and (n_all == 0).any() and ((n_all > 0) & (n_all < maxc)).any()


# ---------------------------------------------------------------------------------------------------------------------
# brute force, thermal (the second walk)
# ---------------------------------------------------------------------------------------------------------------------
# n_dot -> (max_charge_carriers, scans, resolution)
BF_THERMAL = {2: (4, 4, 32), 3: (4, 4, 32), 5: (3, 4, 32), 6: (3, 3, 24), 7: (2, 2, 24), 8: (2, 2, 24)}


@pytest.mark.parametrize("kT_scale", [1.0, 3.0])
@pytest.mark.parametrize("n_dot", sorted(BF_THERMAL))
def test_brute_force_thermal(engine, n_dot, kT_scale):
    from qdsim import FLAG_LATCH, FLAG_THERMAL, N_F32, N_F64
    maxc, n_scans, res = BF_THERMAL[n_dot]
    mb, scans = make_case(n_dot, maxc=maxc, n_env=2, n_scans=n_scans, res=res, seed=120 + n_dot, thermal=True,
                          kT_scale=kT_scale, latching=True)
    use_cport = n_dot >= 5
    z, n = run_gpu(engine, mb, scans, N_F64, FLAG_THERMAL)
    z_ref, n_ref, _ = reference(mb, scans, FLAG_THERMAL, use_cport)
    assert_fractional(n_ref, "reference")
    check_thermal(z, n, z_ref, n_ref)
    _, n32 = run_gpu(engine, mb, scans, N_F32, FLAG_THERMAL)
    assert np.array_equal(n32, n.astype(np.float32)), "N_F32 must be float32 of the N_F64 occupations"
    flags = FLAG_THERMAL | FLAG_LATCH
    zl, nl = run_gpu(engine, mb, scans, N_F64, flags)
    zl_ref, nl_ref, _ = reference(mb, scans, flags, use_cport)
    assert (np.abs(nl_ref - n_ref) > 1e-3).any(), "latching must reject some transitions"
    check_thermal_latched(zl, nl, zl_ref, nl_ref, n_ref, carry_rows=False)


@pytest.mark.parametrize("n_dot", [3, 6])
def test_brute_force_thermal_points(engine, n_dot):
    from qdsim import FLAG_THERMAL, N_F64
    maxc, n_scans, res = BF_THERMAL[n_dot]
    mb, scans = make_case(n_dot, maxc=maxc, n_env=1, n_scans=2, res=res, seed=140 + n_dot, thermal=True, kT_scale=3.0)
    engine.set_models(mb)
    for i, rec in enumerate(scans):
        z, n = engine.points_open_host(rec, points_of(mb, rec), n_type=N_F64, flags=FLAG_THERMAL)
        z_ref, n_ref, _ = reference(mb, scans[i:i + 1], FLAG_THERMAL, n_dot >= 5)
        assert_fractional(n_ref, "reference")
        check_thermal(z[None], n[None], z_ref, n_ref)


# ---------------------------------------------------------------------------------------------------------------------
# default / thresholded, thermal: the two ways of accumulating the Boltzmann average
# ---------------------------------------------------------------------------------------------------------------------
# (n_dot, algorithm, kT scale): at 7 dots the sampled temperatures rarely leave more than six dots free, so kT is raised
BLOCK_CASES = [(8, "default", 1.0), (8, "thresholded", 1.0), (7, "default", 2.0), (7, "thresholded", 2.0)]


@pytest.mark.parametrize("n_dot,algorithm,kT_scale", BLOCK_CASES)
def test_thermal_block_accumulation(engine, n_dot, algorithm, kT_scale):
    from qdsim import FLAG_THERMAL, N_F32, N_F64
    mb, scans = make_case(n_dot, algorithm=algorithm, n_env=2, res=64, seed=150 + n_dot, offset_range=2.0,
                          thermal=True, kT_scale=kT_scale, threshold=0.9)
    share = block_warp_share(mb, scans)
    assert 0.05 <= share <= 0.95, f"block-branch warps: {share:.3f} (both branches must be reached)"
    z, n = run_gpu(engine, mb, scans, N_F64, FLAG_THERMAL)
    z_ref, n_ref, _ = reference(mb, scans, FLAG_THERMAL, False)
    assert_fractional(n_ref, "reference")
    check_thermal(z, n, z_ref, n_ref)
    _, n32 = run_gpu(engine, mb, scans, N_F32, FLAG_THERMAL)
    assert np.array_equal(n32, n.astype(np.float32)), "N_F32 must be float32 of the N_F64 occupations"


@pytest.mark.parametrize("n_dot,algorithm", [(4, "default"), (6, "thresholded")])
def test_thermal_gray_walk(engine, n_dot, algorithm):
    from qdsim import FLAG_THERMAL, N_F32, N_F64
    mb, scans = make_case(n_dot, algorithm=algorithm, n_env=2, res=64, seed=160 + n_dot, thermal=True, kT_scale=3.0,
                          threshold=0.9)
    assert block_warp_share(mb, scans) == 0.0
    z, n = run_gpu(engine, mb, scans, N_F64, FLAG_THERMAL)
    z_ref, n_ref, _ = reference(mb, scans, FLAG_THERMAL, False)
    assert_fractional(n_ref, "reference")
    check_thermal(z, n, z_ref, n_ref)
    _, n32 = run_gpu(engine, mb, scans, N_F32, FLAG_THERMAL)
    assert np.array_equal(n32, n.astype(np.float32)), "N_F32 must be float32 of the N_F64 occupations"


@pytest.mark.parametrize("carry", [False, True])
def test_thermal_latched_carry_across_chunks(engine, carry):
    """Non-integral latching on 64-pixel rows: a pixel at the start of a 32-pixel chunk that is rejected takes the
    occupations carried over from the previous chunk (or, in a flat pass, the previous row)."""
    from qdsim import FLAG_CARRY_ROWS, FLAG_LATCH, FLAG_THERMAL, N_F64
    flags = FLAG_THERMAL | FLAG_LATCH | (FLAG_CARRY_ROWS if carry else 0)
    mb, scans = make_case(5, algorithm="default", n_env=2, res=64, seed=171, thermal=True, kT_scale=3.0, latching=True)
    z, n = run_gpu(engine, mb, scans, N_F64, flags)
    z_ref, n_ref, _ = reference(mb, scans, flags, False)
    _, n_free, _ = reference(mb, scans, flags & ~FLAG_LATCH, False)
    # reach: rejected transitions at chunk starts, where the held occupations come from the carry
    rejected = np.abs(n_ref - n_free).max(axis=-1) > 1e-3
    assert rejected[:, :, 32].any() and (np.abs(n_ref[:, :, 32] - np.rint(n_ref[:, :, 32])) > 1e-3).any()
    check_thermal_latched(z, n, z_ref, n_ref, n_free, carry_rows=carry)


def test_thermal_points(engine):
    """The voltage-list instance of the thermal box search (non-affine relaxation)."""
    from qdsim import FLAG_THERMAL, N_F64
    mb, scans = make_case(5, algorithm="default", n_env=1, res=48, seed=181, thermal=True, kT_scale=3.0)
    engine.set_models(mb)
    for i, rec in enumerate(scans):
        z, n = engine.points_open_host(rec, points_of(mb, rec), n_type=N_F64, flags=FLAG_THERMAL)
        z_ref, n_ref, _ = reference(mb, scans[i:i + 1], FLAG_THERMAL, False)
        check_thermal(z[None], n[None], z_ref, n_ref)
    assert_fractional(n_ref, "reference")
