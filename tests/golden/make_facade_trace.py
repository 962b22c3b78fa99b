#!/usr/bin/env python
"""Record what the REAL reference facade passes to the drop-in classes, and what comes back (CPU container only).

``QarrayBaseClass._get_obs`` (src/qadapt/environment/qarray_base_class.py:171-229) is imported unchanged
(tests/ref_harness.py) and driven for a few observations in BOTH modes -- barrier mode (``TunnelCoupledChargeSensed``:
``gate_voltage_composer.do2d('vP#', ..., add_full_crosstalk=True)`` -> ``charge_sensor_open(vg_flat, vb)``, :143-163) and
non-barrier mode (``ChargeSensedDotArray.do2d_open``, :128-137) -- with the virtual gate matrix as the env leaves it
(-I for electrons, perfect, updated from a capacitance estimate).  Every call that crosses into the drop-in classes is
logged: constructor kwargs (as the facade sampled them), VGM / origin / peak width at call time, ``do2d`` arguments and
returned grid, ``charge_sensor_open`` / ``do2d_open`` arguments, the scan seed drawn from ``np.random``, and the outputs
the CPU ``OracleEngine`` produced (plus, for the tunnel path, the oracle's unlatched <n> and spectral gap, which the causal
latching check needs).  ``tests/test_facade_trace_gpu.py`` replays the log through the SAME drop-in classes with the CUDA
engine underneath and compares.

    python tests/golden/make_facade_trace.py        ->  tests/golden/facade_trace_{barriers,no_barriers}.npz
"""
import os
import pickle
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "rl-agent-for-qubit-array-tuning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import ref_harness  # noqa: E402


def _noise_kwargs(model):
    return dict(model.noise_model._kernel_params())


def _latch_kwargs(model):
    lm = model.latching_model
    if not getattr(lm, "exists", False):
        return None
    return {"n_dots": model.n_dot, "p_leads": np.asarray(lm.p_leads, dtype=np.float64), "p_inter": np.asarray(lm.p_inter, dtype=np.float64)}


def record(use_barriers: bool, num_dots: int, res: int, seed: int):
    mp = pytest.MonkeyPatch()
    try:
        base_mod, env_mod, eng = ref_harness.install(mp)
        from qdsim import FLAG_LATCH, runtime
        from qdsim.composer import GateVoltageComposer
        np.random.seed(seed)
        facade = base_mod.QarrayBaseClass(num_dots=num_dots, use_barriers=use_barriers, obs_image_size=res,
                                          obs_voltage_min=-1.7, obs_voltage_max=1.7)
        m = facade.model
        ctor = {k: np.asarray(getattr(m, k), dtype=np.float64) for k in ("Cdd", "Cgd", "Cds", "Cgs")}
        ctor.update(coulomb_peak_width=float(m.coulomb_peak_width), T=float(m.T), max_charge_carriers=int(m.max_charge_carriers),
                    noise=_noise_kwargs(m), latching=_latch_kwargs(m), charge_carrier=m.charge_carrier)
        if use_barriers:
            ctor.update({k: np.asarray(getattr(m, k), dtype=np.float64) for k in ("Cbd", "Cbg", "Cbs", "Cbb")})
            ctor.update(tc=float(m.tc), tc_base=float(m.barrier_model.tc_base), alpha=np.asarray(m.barrier_model.alpha, dtype=np.float64),
                        num_charge_states=int(m.num_charge_states), charge_state_batch_size=int(m.charge_state_batch_size),
                        use_sparse=bool(m.use_sparse))
        else:
            ctor.update(algorithm=m.algorithm, implementation=m.implementation)

        calls = []
        seeds = []
        real_seed = runtime.fresh_seed

        def logging_seed():
            s = real_seed()
            seeds.append(s)
            return s

        mod = sys.modules[type(m).__module__]
        mp.setattr(mod, "fresh_seed", logging_seed)
        comp = m.gate_voltage_composer
        real_do2d = GateVoltageComposer.do2d
        last_grid = {}

        def logging_do2d(self, *a, **k):
            vg = real_do2d(self, *a, **k)
            last_grid["args"] = a
            last_grid["vg"] = np.array(vg)
            return vg

        mp.setattr(GateVoltageComposer, "do2d", logging_do2d)
        real_cso, real_d2o = type(m).charge_sensor_open, type(m).do2d_open

        def logging_cso(self, vg, vb=None):
            z, n = real_cso(self, vg, vb) if vb is not None else real_cso(self, vg)
            entry = {"kind": "charge_sensor_open", "vgm": np.array(comp.virtual_gate_matrix), "origin": np.array(comp.virtual_gate_origin),
                     "peak_width": float(self.coulomb_peak_width), "do2d_args": last_grid.get("args"), "vg_grid": last_grid.get("vg"),
                     "vg": np.array(vg), "vb": None if vb is None else np.array(vb), "seed": seeds[-1], "z": np.array(z), "n": np.array(n)}
            # what the causal latching check needs: the oracle's unlatched <n> and the spectral gap of every pixel
            from oracle import scan as oscan
            from util import oracle_model, oracle_scan
            mb = self._model_batch()
            om = oracle_model(mb, 0, 0)
            from qdsim.engine import new_scans
            s = new_scans(1)
            s["peak_width"], s["seed"], s["nx"], s["ny"] = entry["peak_width"], entry["seed"], len(entry["vg"]), 1
            v = np.concatenate([entry["vg"], entry["vb"]], axis=1) if vb is not None else entry["vg"]
            _, n_free, gap = oscan.simulate_points(om, v.reshape(1, -1, v.shape[-1]), oracle_scan(s[0], mb.n_volt, 0),
                                                   return_margin=True)
            entry["n_free"], entry["gap"] = np.array(n_free).reshape(-1, self.n_dot), np.array(gap).reshape(-1)
            calls.append(entry)
            return z, n

        def logging_d2o(self, *a):
            z, n = real_d2o(self, *a)
            calls.append({"kind": "do2d_open", "args": a, "vgm": np.array(comp.virtual_gate_matrix),
                          "origin": np.array(comp.virtual_gate_origin), "peak_width": float(self.coulomb_peak_width),
                          "seed": seeds[-1], "z": np.array(z), "n": np.array(n)})
            return z, n

        if use_barriers:
            mp.setattr(type(m), "charge_sensor_open", logging_cso)
        else:
            mp.setattr(type(m), "do2d_open", logging_d2o)

        rng = np.random.default_rng(seed + 1)
        gt = np.asarray(m.optimal_Vg(facade.optimal_VG_center))                  # physical optimum, (N+1,)
        states = ["identity", "perfect", "updated"]
        for state in states:
            if not use_barriers:
                # non-barrier mode sweeps PHYSICAL gates (do2d_open(gate index, ...), :128-137): the VGM plays no role
                gates = -(gt[:num_dots] + rng.uniform(-1.0, 1.0, num_dots)) if m.charge_carrier == "electrons" \
                    else gt[:num_dots] + rng.uniform(-1.0, 1.0, num_dots)
                facade.gate_ground_truth = None
                obs = facade._get_obs(gates, None, float(gt[num_dots]))
                assert obs["image"].shape == (res, res, num_dots - 1)
                continue
            if state == "identity":
                facade._reset_virtual_gate_matrix_to_identity()
            elif state == "perfect":
                facade._reset_virtual_gate_matrix_to_perfect()
            else:
                est = np.abs(np.asarray(m.cgd)[:, :num_dots]) * (1.0 + 0.05 * rng.standard_normal((num_dots, num_dots)))
                facade._update_virtual_gate_matrix(est)
            vgm = np.asarray(comp.virtual_gate_matrix)
            v_virtual = np.linalg.solve(vgm, gt - np.asarray(comp.virtual_gate_origin))
            gates = v_virtual[:num_dots] + rng.uniform(-1.0, 1.0, num_dots)
            barriers = rng.uniform(0.0, 3.0, num_dots - 1)
            facade.gate_ground_truth = None                                        # radial noise is the facade's own NumPy code
            obs = facade._get_obs(gates, barriers, float(v_virtual[num_dots]))
            assert obs["image"].shape == (res, res, num_dots - 1)
        return {"ctor": ctor, "calls": calls, "use_barriers": use_barriers, "num_dots": num_dots, "res": res,
                "obs_voltage": (-1.7, 1.7)}
    finally:
        mp.undo()


def main():
    out = {"barriers": record(True, 4, 20, 101), "no_barriers": record(False, 4, 24, 202)}
    for name, tr in out.items():
        path = os.path.join(HERE, f"facade_trace_{name}.npz")
        blob = np.frombuffer(pickle.dumps(tr, protocol=4), dtype=np.uint8)
        np.savez_compressed(path, trace=blob)
        print(path, len(tr["calls"]), "calls", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
