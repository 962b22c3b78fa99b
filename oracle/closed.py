"""Closed arrays on Path A: the ground state with a fixed total charge ``Q = n_charge`` on the dots (qarray 1.6.0's
``ChargeSensedDotArray.ground_state_closed`` / ``charge_sensor_closed`` / ``do1d_closed`` / ``do2d_closed``), and the
whole scan built on it.

Test infrastructure (see ``oracle/__init__.py``).  Parity unpinned like the rest of Path A (the wheel is absent); restated
on the open path's decisions (``oracle/path_a.py``, SURVEY.md Appendix B) with these for the closed form:

* matrices as for the open path: dot potentials ``g = cgd v``, ``A = cdd_inv``, ``cdd = A^-1`` (dot-only Maxwell);
* the relaxation is the exact minimiser of ``(n - g)^T A (n - g)`` over ``n >= 0``, ``sum n = Q`` (upstream: BoxOSQP with
  ``A = [1^T; I]``, ``l = [Q, 0...]``, ``u = [Q, inf...]``, then ``clip(., 0, Q)``), solved exactly.  The QP is strictly
  convex, so the minimiser is unique.  ``continuous_relaxation_closed`` finds it the obviously correct way: the
  equality-constrained solution of every free set, the feasible one of lowest energy.  (The kernel uses that
  ``A (cdd 1) = 1``: the closed solution is the open relaxation at ``g + nu* cdd 1``.)
* ``default``: candidates ``floor(n_c) + {0,1}^N`` kept only if their sum is ``Q`` (decided in integers): the ``C(N, k)``
  deltas of weight ``k = Q - sum floor(n_c)``, never none;
* ``brute_force``: every ``n in {0..Q}^N`` with ``sum n = Q`` (``max_charge_carriers`` is not used);
* enumeration order (dot 0 slowest), first minimum wins; ``kT > 0``: Boltzmann average over the same candidates, which
  sums to ``Q``;
* latching, sensor, noise and radial noise after the ground state are the open path's (``oracle/scan.py``);
* ``thresholded`` closed is not supported (it can empty the candidate set), nor the tunnel path's closed methods;
  ``0 <= Q <= 251`` for ``default`` (no dot reaches the 252 carriers of the uint8 charge map), ``Q <= 15`` for
  ``brute_force`` (4 bits per dot in the kernel's codes).
"""
from __future__ import annotations

import numpy as np

from . import latching, noise, path_a, philox, sensor
from .composer import affine_grid


CLOSED_MAX_CHARGE = {"default": 251, "brute_force": 15}


def check_closed(algorithm: str, n_charge) -> int:
    """The total charge as an int, or ValueError / NotImplementedError for what the closed path does not take."""
    algorithm = algorithm.lower()
    if algorithm not in CLOSED_MAX_CHARGE:
        raise NotImplementedError(f"closed arrays: algorithm {algorithm} is not supported (default and brute_force are)")
    if isinstance(n_charge, (bool, np.bool_)) or not isinstance(n_charge, (int, np.integer, float, np.floating)) \
            or not float(n_charge).is_integer():
        raise ValueError(f"n_charge must be an integer, got {n_charge!r}")
    q = int(n_charge)
    if not 0 <= q <= CLOSED_MAX_CHARGE[algorithm]:
        raise ValueError(f"n_charge must be in 0..{CLOSED_MAX_CHARGE[algorithm]} for {algorithm}, got {q}")
    return q


def continuous_relaxation_closed(g: np.ndarray, cdd: np.ndarray, cdd_inv: np.ndarray, n_charge: float) -> np.ndarray:
    """Exact minimiser of ``(n-g)^T cdd_inv (n-g)`` over ``n >= 0``, ``sum n = n_charge`` for every row of ``g`` (P, N).

    For every free set F (the other dots at 0): ``n_F = A_FF^-1 (A_F g + t 1)`` with ``t`` such that ``sum n_F = Q``
    (``A = cdd_inv``); among the primal-feasible ones (``n_F >= 0``) the one of lowest energy.  A single free dot is always
    feasible, so every row has an answer.  ``cdd`` is not needed by this formulation (kept for the kernel's signature)."""
    del cdd
    g = np.asarray(g, dtype=np.float64)
    a = np.asarray(cdd_inv, dtype=np.float64)
    q = float(n_charge)
    p, n_dot = g.shape
    ag = g @ a.T
    best_e = np.full(p, np.inf)
    out = np.zeros((p, n_dot))
    for mask in range(1, 1 << n_dot):
        f = np.array([(mask >> j) & 1 == 1 for j in range(n_dot)])
        aff_inv = np.linalg.inv(a[np.ix_(f, f)])
        u = ag[:, f] @ aff_inv.T                           # A_FF^-1 (A g)_F
        v = aff_inv.sum(axis=1)                            # A_FF^-1 1
        t = (q - u.sum(axis=1)) / v.sum()
        n = np.zeros((p, n_dot))
        n[:, f] = u + t[:, None] * v[None, :]
        r = n - g
        e = np.einsum("pi,ij,pj->p", r, a, r)
        take = (n[:, f] >= -1e-12).all(axis=1) & (e < best_e)
        best_e = np.where(take, e, best_e)
        out[take] = n[take]
    return np.clip(out, 0.0, q)


def closed_configurations(n_dot: int, n_charge: int) -> np.ndarray:
    """Every n in {0..Q}^N with sum n = Q, dot 0 slowest (ascending order of the full product)."""
    out = []

    def rec(prefix, rem, left):
        if left == 1:
            out.append(prefix + [rem])
            return
        for v in range(rem + 1):
            rec(prefix + [v], rem - v, left - 1)
    rec([], n_charge, n_dot)
    return np.array(out, dtype=np.float64)


def ground_state_closed(vg, cgd, cdd_inv, cdd, n_charge, algorithm: str = "default", max_charge_carriers: int = 4,
                        kT: float = 0.0, return_margin: bool = False, chunk: int = 2048):
    """Closed-array ground state for voltages ``vg`` (P, G) -> (P, N) float64, total charge ``n_charge`` on the dots.
    ``max_charge_carriers`` is accepted for qarray's signature and not used (the box is {0..n_charge})."""
    del max_charge_carriers
    q = check_closed(algorithm, n_charge)
    algorithm = algorithm.lower()
    vg = np.asarray(vg, dtype=np.float64)
    cgd = np.asarray(cgd, dtype=np.float64)
    cdd_inv = np.asarray(cdd_inv, dtype=np.float64)
    n_dot = cdd_inv.shape[0]
    if vg.shape[-1] != cgd.shape[1]:
        raise ValueError(f"The shape of vg is in correct it should be of shape (..., n_gate) = (...,{cgd.shape[1]})")
    p_total = vg.shape[0]
    n_out = np.empty((p_total, n_dot))
    margin_out = np.empty(p_total)
    deltas = path_a._binary_deltas(n_dot)
    brute = closed_configurations(n_dot, q) if algorithm == "brute_force" else None
    for s in range(0, p_total, chunk):
        g = vg[s:s + chunk] @ cgd.T
        if algorithm == "brute_force":
            r = brute[None, :, :] - g[:, None, :]
            e = np.einsum("pmi,ij,pmj->pm", r, cdd_inv, r)
            n, margin = path_a._select(e, brute, kT)
        else:
            n_c = continuous_relaxation_closed(g, cdd, cdd_inv, q)
            fl = np.floor(n_c)
            confs = fl[:, None, :] + deltas[None, :, :]
            r = confs - g[:, None, :]
            e = np.einsum("pmi,ij,pmj->pm", r, cdd_inv, r)
            keep = (fl.astype(np.int64).sum(axis=1)[:, None] + deltas.astype(np.int64).sum(axis=1)[None, :]) == q
            e = np.where(keep, e, np.inf)
            n, margin = path_a._select(e, confs, kT)
        n_out[s:s + chunk] = n
        margin_out[s:s + chunk] = margin
    if return_margin:
        return n_out, margin_out
    return n_out


def simulate_points_closed(m, n_charge, v, s, latch_compare: str = "rounded", carry_rows: bool = False,
                           white_on: str = "input", return_margin: bool = False):
    """``oracle.scan.simulate_points`` for a closed array of ``n_charge`` carriers: the closed ground state, then the open
    path's latching, sensor, noise and radial noise.  ``m``: an ``oracle.scan.Model`` (default / brute_force)."""
    v = np.asarray(v, dtype=np.float64)
    ny, nx = v.shape[:2]
    n_dot = m.cdd_inv.shape[0]
    v = v.reshape(ny * nx, -1)
    n, margin = ground_state_closed(v, m.cgd, m.cdd_inv, m.cdd, n_charge, m.algorithm, m.max_charge_carriers, m.kT,
                                    return_margin=True)
    n = n.reshape(ny, nx, n_dot)
    draws = philox.pixel_draws(s.seed, ny * nx)
    u_row = philox.row_draws(s.seed, ny)
    if m.latching:
        n = latching.add_latching(n, draws["u_latch"].reshape(ny, nx), m.p_leads, m.p_inter,
                                  compare=latch_compare, carry_rows=carry_rows)
    noise_in = noise.input_noise(draws, ny, nx, m.white_amp, m.tele_p01, m.tele_p10, m.tele_amp, u_row,
                                 carry_rows=carry_rows, white_on=white_on)
    if m.pink_amp != 0.0:
        noise_in = noise_in + m.pink_amp * noise.pink_noise(s.seed, ny, nx, carry_rows=carry_rows)
    out_noise = None
    if white_on == "output" and m.white_amp != 0.0:
        out_noise = (m.white_amp * draws["z_white"]).reshape(ny * nx, 1)
    z = sensor.charge_sensor_signal(n.reshape(ny * nx, n_dot), v, m.cdd_inv_full, m.cgd_full, s.peak_width,
                                    input_noise=noise_in.reshape(ny * nx, 1), output_noise=out_noise)
    z = noise.radial_noise(z.reshape(ny, nx), draws["z_radial"], s.rad_mode, *s.rad)
    if return_margin:
        return z, n, margin.reshape(ny, nx)
    return z, n


def simulate_scan_closed(m, n_charge, s, latch_compare: str = "rounded", carry_rows: bool = False,
                         white_on: str = "input", return_margin: bool = False):
    """``oracle.scan.simulate_scan`` for a closed array: ``(z (ny, nx), n (ny, nx, N)[, margin (ny, nx)])``."""
    v = affine_grid(s.v0, s.dx, s.dy, s.nx, s.ny)
    return simulate_points_closed(m, n_charge, v, s, latch_compare, carry_rows, white_on, return_margin)
