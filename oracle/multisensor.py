"""Dot arrays read by several charge sensors: the whole scan of ``oracle/scan.py`` with ``S = n_sensor`` sensors.

Test infrastructure (see ``oracle/__init__.py``).  qarray's ``ChargeSensedDotArray`` takes any number of sensors (``Cds``
(S, N), ``Cgs`` (S, G); every sensor method returns ``z`` of shape (..., S)).  The signal is the reference's
``charge_sensor_signal`` (``oracle/sensor.py``, a literal restatement of TunnelCoupledChargeSensed.py:320-380), which
already loops over the sensors.  In closed form, for sensor ``s`` at a pixel, with ``u = cgd_full v`` over all
``D = N + S`` rows, dot residuals ``e_j = n_j - u_j``, ``t_o = rint(u_{N+o}) + xi_o - u_{N+o}`` for every sensor ``o``
(``xi_o``: sensor ``o``'s input noise) and ``C = cdd_inv_full``:

    dPhi^s_k = C_ss (2 (t_s + k) + 1) + 2 sum_j C_{s,j} e_j + 2 sum_{o != s} C_{s,o} t_o,      k = -5 .. 4
    z_s      = sum_k 1 / (1 + (dPhi^s_k / gamma)^2) + eta_s

(sensor indices of ``C`` count from row ``N``): one sensor is perturbed, the others sit at their rounded, noisy
occupations.  With ``S = 1`` the last sum vanishes and this is the one-sensor signal.

The reference's wheel is absent, so the noise of several sensors and its random streams are this project's decisions:

* each sensor has its own independent white, telegraph and 1/f noise with the env's amplitudes and probabilities (qarray's
  ``sample_input_noise(shape)`` draws over the trailing ``n_sensor`` axis);
* Philox counter word ``c3`` = sensor index for every stream purpose: 0 (per pixel), 1 (telegraph row start), 2 and 3
  (1/f).  ``oracle/philox.py`` fixes ``c3 = 0``, so sensor 0 draws exactly the one-sensor numbers and a one-sensor scan
  is unchanged;
* the latching uniform is per pixel, not per sensor: the ``w2`` word of sensor 0's block (the ``w2`` word of the blocks of
  sensors ``s >= 1`` is unused);
* radial noise: mode 1 adds ``z_rad,s * amp(ix, iy)`` to each channel (one amplitude map, each channel's own normal); mode
  2 replaces each channel by its own unit normal (the kernels then also zero the occupations, as for one sensor);
* white noise on the output moves each sensor's white noise to its own ``eta_s``.

Limits: ``1 <= S <= 4`` (``QD_MAX_SENSORS``) and at most 16 voltages; the tunnel path with barriers has ``2N + S - 1`` of
them.  The functions return ``z`` of shape (ny, nx) for one sensor, as ``oracle/scan.py`` does, and (ny, nx, S) otherwise.
"""
from __future__ import annotations

import numpy as np

from . import closed, composer, latching, noise, path_a, philox, sensor

MAX_SENSORS = 4


def words(seed: int, index, purpose: int = 0, sensor: int = 0):
    """``philox.words`` of charge sensor ``sensor``: counter ``(index_lo, index_hi, purpose, sensor)``."""
    index = np.asarray(index, dtype=np.uint64)
    k0, k1 = philox._key(seed)
    lo = (index & philox._MASK32).astype(np.uint32)
    hi = (index >> philox._SHIFT32).astype(np.uint32)
    return philox.philox4x32_10(lo, hi, np.uint32(purpose), np.uint32(sensor), k0, k1)


def pixel_draws(seed: int, n_pixels: int, sensor: int = 0):
    """``philox.pixel_draws`` of charge sensor ``sensor``."""
    w0, w1, w2, w3 = words(seed, np.arange(n_pixels, dtype=np.uint64), 0, sensor)
    u1 = ((w0 >> np.uint32(8)).astype(np.float64) + 1.0) * philox.INV_2_24
    u2 = philox.u24(w1)
    r = np.sqrt(-2.0 * np.log(u1))
    ang = 2.0 * np.pi * u2
    return {"z_white": r * np.cos(ang), "z_radial": r * np.sin(ang), "u_latch": philox.u24(w2), "u_tele": philox.u24(w3)}


def row_draws(seed: int, n_rows: int, sensor: int = 0):
    """``philox.row_draws`` of charge sensor ``sensor``."""
    w0, _, _, _ = words(seed, np.arange(n_rows, dtype=np.uint64), 1, sensor)
    return philox.u24(w0)


def pink_noise(seed: int, ny: int, nx: int, carry_rows: bool = False, sensor: int = 0):
    """``noise.pink_noise`` of charge sensor ``sensor``: the same four chains on that sensor's streams 2 and 3."""
    def four_normals(index, purpose):
        w0, w1, w2, w3 = words(seed, index, purpose, sensor)
        out = []
        for wa, wb in ((w0, w1), (w2, w3)):
            u1 = ((wa >> np.uint32(8)).astype(np.float64) + 1.0) * philox.INV_2_24
            u2 = philox.u24(wb)
            r = np.sqrt(-2.0 * np.log(u1))
            out += [r * np.cos(2.0 * np.pi * u2), r * np.sin(2.0 * np.pi * u2)]
        return np.stack(out, axis=-1)

    xi = four_normals(np.arange(ny * nx, dtype=np.uint64), 2).reshape(ny, nx, 4)
    start = four_normals(np.arange(ny, dtype=np.uint64), 3)
    a = np.exp(-1.0 / np.asarray(noise.PINK_TAUS))
    b = np.sqrt(1.0 - a * a)
    out = np.zeros((ny, nx))
    x = start[0].copy()
    for iy in range(ny):
        if not carry_rows:
            x = start[iy].copy()
        for ix in range(nx):
            x = a * x + b * xi[iy, ix]
            out[iy, ix] = 0.5 * x.sum()
    return out


def n_sensor_of(m) -> int:
    """Sensors of an ``oracle.scan.Model``: the rows of cdd_inv_full after the dots."""
    return m.cdd_inv_full.shape[0] - m.cdd_inv.shape[0]


def sensor_stage(m, n, v, s, carry_rows: bool = False, white_on: str = "input"):
    """Latching, the noise of every sensor, the signal and radial noise after the ground state.

    ``n`` (ny, nx, N) ground-state occupations, ``v`` (ny*nx, n_volt) voltages -> ``(z (ny, nx, S), n (ny, nx, N))``."""
    ny, nx, n_dot = n.shape
    n_s = n_sensor_of(m)
    draws = [pixel_draws(s.seed, ny * nx, k) for k in range(n_s)]
    if m.latching:
        n = latching.add_latching(n, draws[0]["u_latch"].reshape(ny, nx), m.p_leads, m.p_inter, carry_rows=carry_rows)
    noise_in = np.zeros((ny * nx, n_s))
    noise_out = np.zeros((ny * nx, n_s))
    for k in range(n_s):
        u_row = row_draws(s.seed, ny, k)
        nk = noise.input_noise(draws[k], ny, nx, m.white_amp, m.tele_p01, m.tele_p10, m.tele_amp, u_row,
                               carry_rows=carry_rows, white_on=white_on)
        if m.pink_amp != 0.0:
            nk = nk + m.pink_amp * pink_noise(s.seed, ny, nx, carry_rows=carry_rows, sensor=k)
        noise_in[:, k] = nk.reshape(-1)
        if white_on == "output" and m.white_amp != 0.0:
            noise_out[:, k] = m.white_amp * draws[k]["z_white"]
    z = sensor.charge_sensor_signal(n.reshape(ny * nx, n_dot), v, m.cdd_inv_full, m.cgd_full, s.peak_width,
                                    input_noise=noise_in, output_noise=noise_out).reshape(ny, nx, n_s)
    z = np.stack([noise.radial_noise(z[..., k], draws[k]["z_radial"], s.rad_mode, *s.rad) for k in range(n_s)], axis=-1)
    return z, n


def _out(z, n_s):
    return z[..., 0] if n_s == 1 else z


def simulate_points(m, v, s, carry_rows: bool = False, white_on: str = "input", return_margin: bool = False):
    """``oracle.scan.simulate_points`` with ``S`` sensors (rounded latching compare): ``z`` (ny, nx) for one sensor,
    (ny, nx, S) otherwise."""
    v = np.asarray(v, dtype=np.float64)
    ny, nx = v.shape[:2]
    n_dot = m.cdd_inv.shape[0]
    v = v.reshape(ny * nx, -1)
    if m.algorithm == "tunnel":
        from . import path_b
        n, margin = path_b.ground_state_open(m, v, return_gap=True)
    else:
        n, margin = path_a.ground_state_open(v, m.cgd, m.cdd_inv, m.cdd, m.algorithm, m.threshold,
                                             m.max_charge_carriers, m.kT, return_margin=True)
    z, n = sensor_stage(m, n.reshape(ny, nx, n_dot), v, s, carry_rows, white_on)
    z = _out(z, n_sensor_of(m))
    return (z, n, margin.reshape(ny, nx)) if return_margin else (z, n)


def simulate_scan(m, s, carry_rows: bool = False, white_on: str = "input", return_margin: bool = False):
    v = composer.affine_grid(s.v0, s.dx, s.dy, s.nx, s.ny)
    return simulate_points(m, v, s, carry_rows, white_on, return_margin)


def simulate_points_closed(m, n_charge, v, s, carry_rows: bool = False, white_on: str = "input",
                           return_margin: bool = False):
    """``oracle.closed.simulate_points_closed`` with ``S`` sensors."""
    v = np.asarray(v, dtype=np.float64)
    ny, nx = v.shape[:2]
    n_dot = m.cdd_inv.shape[0]
    v = v.reshape(ny * nx, -1)
    n, margin = closed.ground_state_closed(v, m.cgd, m.cdd_inv, m.cdd, n_charge, m.algorithm, m.max_charge_carriers,
                                           m.kT, return_margin=True)
    z, n = sensor_stage(m, n.reshape(ny, nx, n_dot), v, s, carry_rows, white_on)
    z = _out(z, n_sensor_of(m))
    return (z, n, margin.reshape(ny, nx)) if return_margin else (z, n)


def simulate_scan_closed(m, n_charge, s, carry_rows: bool = False, white_on: str = "input", return_margin: bool = False):
    v = composer.affine_grid(s.v0, s.dx, s.dy, s.nx, s.ny)
    return simulate_points_closed(m, n_charge, v, s, carry_rows, white_on, return_margin)
