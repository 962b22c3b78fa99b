"""Shared helpers of the parity tests: turn the product-side batch (ModelBatch + qd_scan records) into the oracle's
Model / Scan objects so both sides see the same numbers."""
from __future__ import annotations

import os

import numpy as np

from oracle import scan as oscan

# ``src`` of a checkout of the upstream project (edwindn/rl-agent-for-qubit-array-tuning).  The tests that run its own code
# next to ours skip when ``QADAPT_SRC`` does not point at one.
REFERENCE_SRC = os.environ.get("QADAPT_SRC", "")


def reference_path(*parts: str) -> str:
    """``parts`` under the upstream ``src`` tree, or "" (which exists nowhere) when ``QADAPT_SRC`` is not set."""
    return os.path.join(REFERENCE_SRC, *parts) if REFERENCE_SRC else ""


def oracle_model(mb, e: int, flags: int = 0):
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_PINK, FLAG_THERMAL
    p = mb.params[e]
    n = mb.n_dot
    noise = bool(flags & FLAG_NOISE)
    return oscan.Model(
        cdd_inv=mb.cdd_inv_gs[e], cdd=None if mb.cdd_gs is None else mb.cdd_gs[e],
        cgd=mb.cgd_full[e, :n, :], cdd_inv_full=mb.cdd_inv_full[e], cgd_full=mb.cgd_full[e],
        algorithm=mb.algorithm, threshold=float(p["threshold"]), max_charge_carriers=int(p["max_charge_carriers"]),
        kT=float(p["kT"]) if flags & FLAG_THERMAL else 0.0,
        latching=bool(p["latching"]) and bool(flags & FLAG_LATCH),
        p_leads=p["p_leads"][:n].copy(), p_inter=p["p_inter"].reshape(8, 8)[:n, :n].copy(),
        white_amp=float(p["white_amp"]) if noise else 0.0, tele_p01=float(p["tele_p01"]),
        tele_p10=float(p["tele_p10"]), tele_amp=float(p["tele_amp"]) if noise else 0.0,
        pink_amp=float(p["pink_amp"]) if (flags & FLAG_PINK) and "pink_amp" in (p.dtype.names or ()) else 0.0,
        n_gate=mb.n_gate, cbg=None if mb.cbg is None else mb.cbg[e], tc_base=float(p["tc_base"]),
        alpha=p["alpha"].copy(), num_charge_states=mb.num_charge_states,
        charge_state_batch_size=mb.charge_state_batch_size, vc_alpha=float(p["vc_alpha"]), vc_beta=float(p["vc_beta"]),
        vc_kind=int(p["vc_kind"]), vc_vchar=float(p["vc_vchar"]) if float(p["vc_vchar"]) > 0 else 1.0)


def oracle_scan(rec, n_volt: int, flags: int = 0):
    from qdsim import FLAG_RADIAL
    rad_mode = int(rec["rad_mode"]) if flags & FLAG_RADIAL else 0
    return oscan.Scan(
        v0=rec["v0"][:n_volt].copy(), dx=rec["dx"][:n_volt].copy(), dy=rec["dy"][:n_volt].copy(),
        nx=int(rec["nx"]), ny=int(rec["ny"]), peak_width=float(rec["peak_width"]), seed=int(rec["seed"]),
        rad_mode=rad_mode,
        rad=(float(rec["rad_x0"]), float(rec["rad_dx"]), float(rec["rad_y0"]), float(rec["rad_dy"]),
             float(rec["rad_alpha"]), float(rec["rad_zero_radius"]), float(rec["rad_max_amp"])))


def oracle_batch(mb, scans, flags: int = 0, which=None):
    """Run the oracle over ``scans[which]``; returns (z, n, margin) stacked, each scan (ny, nx[, N])."""
    from qdsim import FLAG_CARRY_ROWS, FLAG_LATCH_EXACT, FLAG_WHITE_ON_OUTPUT
    which = range(len(scans)) if which is None else which
    zs, ns, ms = [], [], []
    for i in which:
        rec = scans[i]
        m = oracle_model(mb, int(rec["env_id"]), flags)
        s = oracle_scan(rec, mb.n_volt, flags)
        z, n, mg = oscan.simulate_scan(
            m, s, latch_compare="exact" if flags & FLAG_LATCH_EXACT else "rounded",
            carry_rows=bool(flags & FLAG_CARRY_ROWS),
            white_on="output" if flags & FLAG_WHITE_ON_OUTPUT else "input", return_margin=True)
        zs.append(z)
        ns.append(n)
        ms.append(mg)
    return np.stack(zs), np.stack(ns), np.stack(ms)


def compare_charges(n_gpu, n_ref, margin, tie_tol=1e-9, max_tie_frac=0.005):
    """Bit-exact on every pixel whose best/second-best energy gap exceeds ``tie_tol`` (an exact tie has no defined
    winner across two summation orders); the near-tie set itself must be tiny."""
    n_gpu = np.asarray(n_gpu).astype(np.int64)
    n_ref = np.rint(np.asarray(n_ref)).astype(np.int64)
    safe = margin > tie_tol
    assert (~safe).mean() <= max_tie_frac, f"too many near-ties: {(~safe).mean():.4f}"
    bad = (n_gpu != n_ref).any(axis=-1) & safe
    assert not bad.any(), f"{bad.sum()} of {bad.size} pixels differ, first at {np.argwhere(bad)[:5]}"
    return int((~safe).sum())


def _params_from_bytes(raw):
    """Fixture bytes -> current PARAMS_DTYPE.  Older fixtures hold older, shorter records: 712 bytes before ABI 2 (no
    vc_alpha / vc_beta), 728 bytes in ABI 2 (8 reserved bytes where pink_amp is now; no vc_vchar / vc_kind)."""
    from qdsim import PARAMS_DTYPE
    raw = np.ascontiguousarray(raw)
    if raw.size % PARAMS_DTYPE.itemsize == 0:
        return raw.view(PARAMS_DTYPE).copy()
    new_tail = ("vc_vchar", "vc_kind", "reserved0")
    abi2 = np.dtype([(n, PARAMS_DTYPE.fields[n][0]) for n in PARAMS_DTYPE.names if n not in new_tail], align=True)
    abi1 = np.dtype([(n, PARAMS_DTYPE.fields[n][0]) for n in PARAMS_DTYPE.names
                     if n not in new_tail + ("vc_alpha", "vc_beta")], align=True)
    assert abi2.itemsize == 728 and abi1.itemsize == 712, (abi2.itemsize, abi1.itemsize)
    legacy = abi2 if raw.size % 728 == 0 else abi1
    assert raw.size % legacy.itemsize == 0, raw.size
    old = raw.view(legacy)
    out = np.zeros(old.shape, dtype=PARAMS_DTYPE)
    for n in legacy.names:
        out[n] = old[n]
    return out


def load_golden(name):
    """tests/golden/<name>.npz -> (ModelBatch, scans, flags, z, n, margin): inputs rebuilt through the product's host code
    from the RAW capacitances stored in the fixture."""
    import os
    from qdsim import PARAMS_DTYPE, SCAN_DTYPE
    from qdsim.engine import ModelBatch
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz")
    d = np.load(path)
    params = _params_from_bytes(d["params"])
    if str(d["algorithm"]) == "tunnel":
        from qdsim.engine import tunnel_model_batch
        mb = tunnel_model_batch(d["Cdd"], d["Cgd"], d["Cds"], d["Cgs"], d["Cbd"], d["Cbg"], d["Cbs"],
                                params["tc_base"], params["alpha"][:, :d["Cbd"].shape[-1]])
    else:
        mb = ModelBatch.from_capacitances(d["Cdd"], d["Cgd"], d["Cds"], d["Cgs"], algorithm=str(d["algorithm"]))
    mb.params = params
    scans = d["scans"].view(SCAN_DTYPE).copy()
    return mb, scans, int(d["flags"]), d["z"], d["n"], d["margin"]


GOLDEN_CASES = ["c1_2dot_64x64_noise_free", "c2_4dot_latched_full_noise", "c2b_4dot_flat_pass", "c3_6dot_brute_force",
                "c4_8dot_latched_full_noise", "t_3dot_thermal", "t_5dot_thresholded"]
GOLDEN_TUNNEL_CASES = ["b_4dot_tunnel_latched_noise", "b_6dot_tunnel_coupled"]


# ---------------------------------------------------------------------------------------------------------------------
# Parity of a whole batch against the C restatement (oracle/cport): what bench.py's `parity_sample` and the
# benched-configuration GPU tests run.
# ---------------------------------------------------------------------------------------------------------------------
def cport_parity(mb, scans, flags, z_gpu, n_gpu, threads: int = 0, tie_tol: float = 1e-9, z_atol: float = 5e-6):
    """Compare the CUDA outputs of ``scans`` (z float32 [pixels], n [pixels, N]; pix_offset = i * nx * ny) with the
    plain-C restatement run on the same descriptors.

    Charge maps are compared bit for bit on every ROW that holds no near-tie (best / second-best candidate gap <=
    ``tie_tol``: an exact tie has no defined winner across two summation orders, and under latching the pixels downstream
    of it in the same row inherit the choice); the sensor image at ``z_atol`` absolute on the same rows.
    Returns dict(scans, pixels, rows, tie_rows, n_mismatch, z_max_abs, cpu_seconds)."""
    from oracle import cport
    from qdsim import FLAG_CARRY_ROWS
    scans = np.ascontiguousarray(scans)
    nx, ny = int(scans["nx"][0]), int(scans["ny"][0])
    assert (scans["nx"] == nx).all() and (scans["ny"] == ny).all()
    n_dot = mb.n_dot
    zc, nc, dt, margin = cport.run_scans(mb, scans, flags, threads=threads, want_margin=True)
    S = len(scans)
    margin = margin.reshape(S, ny, nx)
    if flags & FLAG_CARRY_ROWS:                                   # a flat pass carries state across the row ends
        tie_row = np.repeat((margin <= tie_tol).any(axis=(1, 2))[:, None], ny, axis=1)
    else:
        tie_row = (margin <= tie_tol).any(axis=2)                 # (S, ny)
    ng = np.asarray(n_gpu).reshape(S, ny, nx, n_dot).astype(np.int64)
    nr = np.rint(nc).reshape(S, ny, nx, n_dot).astype(np.int64)
    zg = np.asarray(z_gpu, dtype=np.float64).reshape(S, ny, nx)
    zr = zc.astype(np.float64).reshape(S, ny, nx)
    safe = ~tie_row
    mism = (ng != nr).any(axis=-1) & safe[:, :, None]
    dz = np.abs(zg - zr) * safe[:, :, None]
    return {"scans": S, "pixels": S * nx * ny, "rows": int(safe.size), "tie_rows": int(tie_row.sum()),
            "n_mismatch": int(mism.sum()), "z_max_abs": float(dz.max()), "z_atol": z_atol, "tie_tol": tie_tol,
            "cpu_seconds": float(dt), "ok": bool(mism.sum() == 0 and dz.max() <= z_atol)}


def explain_latched_mismatches(n_gpu, n_ref, n_free_ref, gap, carry_rows: bool = False, n_atol: float = 1e-6,
                               gap_min: float = 1e-5, half_tol: float = 2e-6):
    """Causal check of a latched tunnel-path image (non-integer <n>, rounded latch compare).

    ``n_gpu`` / ``n_ref``: latched occupations (ny, nx, N) of the CUDA path and of the oracle; ``n_free_ref``: the oracle's
    UNLATCHED <n>; ``gap``: spectral gap per pixel.  The CUDA <n> carries up to ``n_atol`` of eigen-solver error, so a latch
    decision (made on round(<n>)) may legitimately differ only where the oracle's free <n> lies within ``half_tol`` of a
    half-integer on some dot, or where the ground vector itself is ill-conditioned (gap <= ``gap_min``).  Everything
    downstream of such a pixel in the same latching sequence (row; whole scan for a flat pass) may then differ.  Asserts
    that EVERY differing pixel is explained that way -- a latching bug elsewhere fails -- and returns
    (n_differing_pixels, n_ambiguous_sequences, n_sequences)."""
    n_gpu, n_ref, n_free_ref = (np.asarray(a, dtype=np.float64) for a in (n_gpu, n_ref, n_free_ref))
    ny, nx, nd = n_ref.shape
    frac = n_free_ref - np.floor(n_free_ref)
    ambiguous = (np.abs(frac - 0.5) <= half_tol).any(axis=-1) | (np.asarray(gap).reshape(ny, nx) <= gap_min)
    differs = np.abs(n_gpu - n_ref).max(axis=-1) > n_atol
    if carry_rows:
        amb, dif = ambiguous.reshape(1, -1), differs.reshape(1, -1)
    else:
        amb, dif = ambiguous, differs
    n_amb_seq = 0
    for r in range(dif.shape[0]):
        first_amb = int(np.argmax(amb[r])) if amb[r].any() else amb.shape[1]
        n_amb_seq += int(amb[r].any())
        if dif[r].any():
            first_dif = int(np.argmax(dif[r]))
            assert first_amb <= first_dif, (
                f"sequence {r}: first differing pixel at {first_dif} (gpu {n_gpu.reshape(-1, nd)[r * dif.shape[1] + first_dif] if not carry_rows else ''}) "
                f"has no ambiguous pixel (half-integer <n> or gap <= {gap_min}) at or before it (first ambiguous: {first_amb})")
    return int(dif.sum()), n_amb_seq, int(dif.shape[0])


Z_RTOL = 1e-6        # north_star: noise-free sensor signals within 1e-6 relative


def assert_z_given_n(z, z_ref, n, n_ref, ok, w_max, gamma, noise_atol: float = 0.0, what: str = ""):
    """Tunnel-path sensor signal at ``Z_RTOL`` = 1e-6 relative GIVEN <n>.

    The kernel evaluates the Lorentzians of the tunnel path in fp64, so the only other error in z is the one <n> carries in
    (the eigen-solver's, <= 1e-6 by its own test): each of the ten Lorentzians 1 / (1 + x^2) has |d/dx| <= 3 sqrt(3) / 8 and
    dx / dn_j = 2 cdd_inv_full[N, j] / gamma, so |dz| <= 10 * 0.65 * 2 max_j|w_j| / gamma * |dn|, with the MEASURED |dn| of
    the same pixel.  Budget per pixel: 1e-6 |z_ref| + that propagated term + 1e-7 (fp32 image) [+ noise_atol when the
    fp32 Box-Muller noise terms are on]."""
    z, z_ref = np.asarray(z, dtype=np.float64), np.asarray(z_ref, dtype=np.float64)
    dn = np.abs(np.asarray(n, dtype=np.float64) - np.asarray(n_ref, dtype=np.float64)).max(axis=-1).reshape(z_ref.shape)
    sens = 10 * 0.6495191 * 2.0 * np.broadcast_to(np.asarray(w_max, dtype=np.float64) / np.asarray(gamma, dtype=np.float64),
                                                    z_ref.shape)
    budget = Z_RTOL * np.abs(z_ref) + sens * dn + 1e-7 + noise_atol
    err = np.abs(z.reshape(z_ref.shape) - z_ref)
    ok = np.asarray(ok).reshape(z_ref.shape)
    assert (err[ok] <= budget[ok]).all(), f"{what} sensor error exceeds the 1e-6 budget by {np.max((err - budget)[ok]):.3e}"
    return float(err[ok].max()) if ok.any() else 0.0


def sensor_w_max(mb, e: int = 0):
    """max_j |cdd_inv_full[N, j]|: the sensor <-> dot coupling that scales dz / d<n>."""
    n = mb.n_dot
    return float(np.abs(mb.cdd_inv_full[e, n, :n]).max())
