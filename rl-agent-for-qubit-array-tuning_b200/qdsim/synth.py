"""Seeded synthetic devices and scan windows with the reference's sampling distributions (SURVEY.md section 8d).

Device parameters follow src/qadapt/environment/qarray_config.yaml:10-66 as sampled by
src/qadapt/environment/qarray_base_class.py:254-298 (Cdd / Cgd distance rules, plunger block of Cgd symmetrised),
:376-390 (Cds, Cgs), :392-441 (noise), :495-519 (latching); scan windows follow env_config.yaml:20 (half-width
U[1.5, 2.0] V) around ``ground truth + U[-5, 5] V`` with the virtual-gate matrix ``-I`` (electrons,
qarray_base_class.py:868-877) and the sensor gate at its optimum (qarray_config.yaml:122).
Vectorised over envs: one generator seeded with ``seed`` draws every array with a leading env axis.
"""
from __future__ import annotations

import numpy as np

from . import maxwell
from .engine import ModelBatch, new_scans, tunnel_model_batch


def _by_distance(rng, n_env, n_rows, n_cols, ranges, offset=0.0):
    """Matrix whose (i, j) entry ~ U[ranges[d]] with d = int(|i - (j + offset)|) clipped to the last rule."""
    i = np.arange(n_rows)[:, None]
    j = np.arange(n_cols)[None, :] + offset
    d = np.abs(i - j).astype(int)
    if offset:
        d = np.maximum(1, d)
    d = np.minimum(d, len(ranges) - 1)
    lo = np.array([r[0] for r in ranges])[d]
    hi = np.array([r[1] for r in ranges])[d]
    return rng.uniform(lo, hi, size=(n_env, n_rows, n_cols))


def sample_devices(n_env: int, n_dot: int, seed: int = 1234, n_sensor: int = 1):
    """Raw (non-Maxwell) capacitance matrices + model parameters of ``n_env`` random devices.

    ``n_sensor`` > 1: sensor 0 and every other draw are those of the one-sensor device; sensors 1.. have their own gates
    (gate N + s), couplings to the dots from the same range as sensor 0's and up to 0.02 to the other sensor gates."""
    rng = np.random.default_rng(seed)
    N = n_dot
    cdd = _by_distance(rng, n_env, N, N, [(0.0, 0.0), (0.0, 0.2), (0.0, 0.1), (0.0, 0.0)])
    cdd = np.triu(cdd, 1)
    cdd = cdd + np.swapaxes(cdd, -1, -2)
    cgd_pl = _by_distance(rng, n_env, N, N, [(0.95, 1.0), (0.3, 0.7), (0.01, 0.3), (0.0, 0.01)])
    cgd_pl = 0.5 * (cgd_pl + np.swapaxes(cgd_pl, -1, -2))
    cgd = np.zeros((n_env, N, N + 1))
    cgd[:, :, :N] = cgd_pl
    cds = rng.uniform(0.035, 0.05, size=(n_env, 1, N))
    cgs = np.concatenate([rng.uniform(0.0, 1e-4, size=(n_env, 1, N)), rng.uniform(0.95, 1.0, size=(n_env, 1, 1))], axis=-1)
    p01 = rng.uniform(0.0, 0.01, n_env)
    p_inter = rng.uniform(0.2, 1.0, size=(n_env, N, N))
    p_inter = np.triu(p_inter, 1)
    p_inter = p_inter + np.swapaxes(p_inter, -1, -2)
    if n_sensor > 1:
        S = n_sensor
        rs = np.random.default_rng([seed, 91])
        cgd = np.concatenate([cgd, np.zeros((n_env, N, S - 1))], axis=-1)
        cds = np.concatenate([cds, rs.uniform(0.035, 0.05, size=(n_env, S - 1, N))], axis=1)
        cgs_all = np.zeros((n_env, S, N + S))
        cgs_all[:, 0, :N + 1] = cgs[:, 0]
        cgs_all[:, 1:, :N] = rs.uniform(0.0, 1e-4, size=(n_env, S - 1, N))
        cgs_all[:, :, N:] += rs.uniform(0.0, 0.02, size=(n_env, S, S)) * (1.0 - np.eye(S))
        cgs_all[:, np.arange(1, S), N + np.arange(1, S)] = rs.uniform(0.95, 1.0, size=(n_env, S - 1))
        cgs = cgs_all
    return {
        "Cdd": cdd, "Cgd": cgd, "Cds": cds, "Cgs": cgs,
        "white_amp": rng.uniform(0.0, 1e-4, n_env),
        "tele_p01": p01, "tele_p10": rng.uniform(0.0, 100.0, n_env) * p01, "tele_amp": rng.uniform(0.0, 0.012, n_env),
        "p_leads": rng.uniform(0.2, 1.0, size=(n_env, N)), "p_inter": p_inter,
        "T": rng.uniform(50.0, 200.0, n_env),
        "peak_width": rng.uniform(0.05, 0.4, n_env),      # yaml says U[0, 0.4]; keep gamma away from 0
    }


def model_batch(dev: dict, algorithm: str = "default", thermal: bool = False, latching: bool = True,
                noise: bool = True, max_charge_carriers: int = 4, threshold: float = 1.0) -> ModelBatch:
    return ModelBatch.from_capacitances(
        dev["Cdd"], dev["Cgd"], dev["Cds"], dev["Cgs"], algorithm=algorithm,
        T=dev["T"] if thermal else 0.0, threshold=threshold, max_charge_carriers=max_charge_carriers,
        p_leads=dev["p_leads"] if latching else None, p_inter=dev["p_inter"] if latching else None,
        white_amp=dev["white_amp"] if noise else 0.0, tele_p01=dev["tele_p01"] if noise else 0.0,
        tele_p10=dev["tele_p10"] if noise else 0.0, tele_amp=dev["tele_amp"] if noise else 0.0)


def sample_barrier_devices(n_env: int, n_dot: int, seed: int = 1234, n_sensor: int = 1):
    """``sample_devices`` plus the barrier matrices and the barrier-voltage model of the tunnel-coupled path
    (qarray_config.yaml:72-100; qarray_base_class.py:300-357, 521-534).  ``n_sensor`` as in ``sample_devices``."""
    dev = sample_devices(n_env, n_dot, seed, n_sensor)
    rng = np.random.default_rng([seed, 77])
    N, B, G = n_dot, n_dot - 1, n_dot + 1
    dev["Cbd"] = _by_distance(rng, n_env, N, B, [(0.04, 0.08), (0.04, 0.08), (0.01, 0.03), (0.005, 0.015)], offset=0.5)
    cbg = _by_distance(rng, n_env, G, B, [(0.08, 0.15), (0.08, 0.15), (0.03, 0.18), (0.01, 0.03)], offset=0.5)
    cbg[:, N, :] = rng.uniform(0.03, 0.18, size=(n_env, B))                 # sensor gate: the distance-2 rule
    cbs = rng.uniform(3e-4, 1e-3, size=(n_env, 1, B))
    if n_sensor > 1:                                                        # the other sensor gates: the same rules
        rs = np.random.default_rng([seed, 78])
        cbg = np.concatenate([cbg, rs.uniform(0.03, 0.18, size=(n_env, n_sensor - 1, B))], axis=1)
        cbs = np.concatenate([cbs, rs.uniform(3e-4, 1e-3, size=(n_env, n_sensor - 1, B))], axis=1)
    dev["Cbg"] = np.ascontiguousarray(np.swapaxes(cbg, -1, -2))              # (E, B, G)
    dev["Cbs"] = cbs
    dev["tc_base"] = rng.uniform(0.5, 3.0, n_env)
    dev["alpha"] = rng.uniform(0.8, 2.0, size=(n_env, B))
    return dev


def tunnel_batch(dev: dict, latching: bool = True, noise: bool = True) -> ModelBatch:
    return tunnel_model_batch(
        dev["Cdd"], dev["Cgd"], dev["Cds"], dev["Cgs"], dev["Cbd"], dev["Cbg"], dev["Cbs"], dev["tc_base"], dev["alpha"],
        p_leads=dev["p_leads"] if latching else None, p_inter=dev["p_inter"] if latching else None,
        white_amp=dev["white_amp"] if noise else 0.0, tele_p01=dev["tele_p01"] if noise else 0.0,
        tele_p10=dev["tele_p10"] if noise else 0.0, tele_amp=dev["tele_amp"] if noise else 0.0)


def ground_truth(mb: ModelBatch, dots: float = 1.0, sensor: float = 0.53):
    """Gate voltages (E, G) that put every dot at ``dots`` carriers and every sensor at ``sensor``."""
    n = np.concatenate([np.full(mb.n_dot, dots), np.full(mb.n_sensor, sensor)])
    return maxwell.optimal_vg(mb.cdd_inv_full, mb.cgd_full[:, :, :mb.n_gate], n)


def env_step_scans(mb: ModelBatch, dev: dict, res: int = 64, seed: int = 7, offset_range: float = 5.0,
                   radial: bool = True, step: int = 0):
    """Scan descriptors of one ``env.step`` for every env: N-1 adjacent-pair windows per env, env-major.

    Virtual-gate coordinates with VGM = -I: physical gate voltages ``vg = -Vd``; the swept pair (x = left dot,
    y = right dot) runs over ``centre +- half_width``; the other plungers sit at their centre voltage, the sensor
    gate at its optimum.  Output layout: scan ``e*(N-1) + c`` -> pixels ``[(e*(N-1)+c) * res^2, ...)``.
    """
    rng = np.random.default_rng([seed, step])
    E, N, G = mb.n_env, mb.n_dot, mb.n_gate
    gt_phys = ground_truth(mb)                            # (E, G)
    gt_virtual = -gt_phys                                 # Vd = VGM^-1 vg with VGM = -I
    centre = gt_virtual[:, :N] + rng.uniform(-offset_range, offset_range, size=(E, N))
    half = rng.uniform(1.5, 2.0, size=E)
    n_scan = E * (N - 1)
    scans = new_scans(n_scan)
    env = np.repeat(np.arange(E), N - 1)
    ch = np.tile(np.arange(N - 1), E)
    vd = np.concatenate([centre, gt_virtual[:, N:]], axis=1)[env]       # (n_scan, G) all gates at their set point
    step_v = (2.0 * half / (res - 1))[env]
    rows = np.arange(n_scan)
    v0 = vd.copy()
    v0[rows, ch] = centre[env, ch] - half[env]
    v0[rows, ch + 1] = centre[env, ch + 1] - half[env]
    scans["v0"][:, :G] = -v0
    if mb.n_volt > G:                                     # tunnel path: barrier voltages ride along, constant per scan
        vb = rng.uniform(-1.0, 3.0, size=(E, mb.n_volt - G))
        scans["v0"][:, G:mb.n_volt] = vb[env]
    scans["dx"][rows, ch] = -step_v
    scans["dy"][rows, ch + 1] = -step_v
    scans["peak_width"] = dev["peak_width"][env]
    scans["seed"] = (np.uint64(seed) << np.uint64(40)) + (np.uint64(step) << np.uint64(24)) + rows.astype(np.uint64)
    scans["pix_offset"] = rows.astype(np.int64) * res * res
    scans["env_id"] = env
    scans["nx"] = res
    scans["ny"] = res
    if radial:
        zero_r = rng.uniform(20.0, 30.0, size=E)
        ramp = zero_r + rng.uniform(5.0, 10.0, size=E)
        scans["rad_mode"] = 1
        scans["rad_x0"] = centre[env, ch] - half[env] - gt_virtual[env, ch]
        scans["rad_dx"] = step_v
        scans["rad_y0"] = centre[env, ch + 1] - half[env] - gt_virtual[env, ch + 1]
        scans["rad_dy"] = step_v
        scans["rad_max_amp"] = 0.05
        scans["rad_alpha"] = (0.05 / ramp)[env]
        scans["rad_zero_radius"] = zero_r[env]
    return scans
