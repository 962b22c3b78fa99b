"""Golden vectors made by the REFERENCE ITSELF (needs the upstream project's ``src`` tree; the fixtures are committed,
the reference is not):

    QADAPT_SRC=<upstream checkout>/src python tests/golden/make_reference_golden.py

The reference's tunnel-coupled simulator (Path B, what ``env.step`` executes) is in-tree Python
(src/qarray_latched/DotArrays/*.py).  It is imported unmodified through ``refshim`` (eager NumPy
evaluation of its jax calls, inert shims for the absent ``qarray`` type names), constructed exactly like
``QarrayBaseClass._load_model_with_barriers`` does (src/qadapt/environment/qarray_base_class.py:817-838) and driven
exactly like ``_get_charge_sensor_data`` does (:143-163): ``gate_voltage_composer.do2d('vP#', ..., gate_voltages,
add_full_crosstalk=True)`` -> ``charge_sensor_open(vg_flat, vb)``.  No latching / noise model (those classes live in
the absent wheel), so every number in these files comes from reference code.

Each ``ref_*.npz`` holds the raw inputs (non-Maxwell capacitances, barrier model, virtual gate matrix, window) and the
reference's outputs: ``cdd_inv_full`` / ``cgd_full`` (Maxwell conversion, S1), ``vg`` (scan grid, S2), ``n`` (ground
state occupations, B1-B6), ``z`` (sensor signal, S3/S4).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (HERE, ROOT, os.path.join(ROOT, "rl-agent-for-qubit-array-tuning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

# name: (n_dot, res, seed, pair (1-based left dot), vgm kind, with_cbb, barriers?)
CASES = {
    "ref_4dot_tunnel_identity_vgm": dict(n_dot=4, res=32, seed=11, pair=2, vgm="identity", cbb=False),
    "ref_4dot_tunnel_perfect_vgm_cbb": dict(n_dot=4, res=20, seed=12, pair=1, vgm="perfect", cbb=True),
    "ref_5dot_tunnel_low_occupancy": dict(n_dot=5, res=16, seed=13, pair=3, vgm="identity", cbb=False, offset=-1.2),
    "ref_6dot_tunnel_identity_vgm": dict(n_dot=6, res=16, seed=14, pair=4, vgm="identity", cbb=True),
    "ref_8dot_tunnel_identity_vgm": dict(n_dot=8, res=12, seed=15, pair=5, vgm="identity", cbb=False),
    "ref_4dot_constant_tc_no_barriers": dict(n_dot=4, res=16, seed=16, pair=1, vgm="identity", cbb=False, barriers=False),
    # voltage_capacitance_model.type: linear (qarray_config.yaml:103-105, 132-134; qarray_base_class.py:842-852)
    "ref_4dot_tunnel_linear_capacitance": dict(n_dot=4, res=20, seed=17, pair=2, vgm="identity", cbb=False, vc=(0.08, 0.06)),
    "ref_6dot_tunnel_linear_capacitance": dict(n_dot=6, res=12, seed=18, pair=3, vgm="perfect", cbb=False, vc=(0.05, 0.10)),
    # the reference's other factories (voltage_dependent_capacitance.py:138-168; unreachable from the shipped facade)
    "ref_4dot_tunnel_quadratic_capacitance": dict(n_dot=4, res=16, seed=22, pair=2, vgm="identity", cbb=False, vc=(0.004, 0.05),
                                                  vc_kind="quadratic"),
    "ref_5dot_tunnel_sigmoid_capacitance": dict(n_dot=5, res=14, seed=23, pair=2, vgm="identity", cbb=False, vc=(0.4, 0.03),
                                                vc_kind="sigmoid", vc_vchar=4.0),
    # the env's own regime (env.py:808-858): barriers up to +-15 V from their optimum, i.e. tunnel couplings from 1e-9 to 1e7,
    # and windows tens of volts from the ground truth (occupations of 10-40 carriers on some dots, none on others)
    "ref_4dot_tunnel_strong_coupling": dict(n_dot=4, res=16, seed=19, pair=2, vgm="identity", cbb=False, vb_shift=-8.0),
    "ref_4dot_tunnel_closed_barriers": dict(n_dot=4, res=16, seed=20, pair=1, vgm="identity", cbb=False, vb_shift=+14.0,
                                            offset=2.5),
    "ref_6dot_tunnel_far_window": dict(n_dot=6, res=10, seed=21, pair=3, vgm="identity", cbb=False, offset=22.0, spread=12.0,
                                       vb_shift=14.0),
}


def case_inputs(n_dot, res, seed, pair, vgm, cbb, offset=0.0, barriers=True, vc=None, vb_shift=0.0, spread=2.0,
                vc_kind="linear", vc_vchar=1.0):
    """Raw inputs of one case, drawn with the reference's sampling ranges (qdsim.synth)."""
    from qdsim import synth
    dev = synth.sample_barrier_devices(1, n_dot, seed=seed)
    rng = np.random.default_rng([seed, 5])
    raw = {k: dev[k][0] for k in ("Cdd", "Cgd", "Cds", "Cgs", "Cbd", "Cbg", "Cbs")}
    B = n_dot - 1
    raw["Cbb"] = None
    if cbb:                                              # qarray_config.yaml Cbb ranges are irrelevant: the term is 0
        c = np.triu(rng.uniform(0.01, 0.05, size=(B, B)), 1)
        raw["Cbb"] = c + c.T
    raw.update(tc_base=float(dev["tc_base"][0]), alpha=dev["alpha"][0], peak_width=float(dev["peak_width"][0]),
               T=float(dev["T"][0]), tc=0.7, barriers=barriers)
    raw["barrier_voltages"] = rng.uniform(-1.0, 3.0, size=B) + vb_shift
    raw["half"] = float(rng.uniform(1.5, 2.0))
    raw["centre_offset"] = rng.uniform(-spread, spread, size=n_dot) + offset
    raw.update(res=res, pair=pair, vgm_kind=vgm, vc=np.array(vc if vc is not None else (0.0, 0.0)),
               vc_kind=np.array({"linear": 0, "quadratic": 1, "sigmoid": 2}[vc_kind]), vc_vchar=np.array(float(vc_vchar)))
    return raw


def run_reference(raw):
    """-> dict of the reference's outputs for one case."""
    from refshim import reference_modules
    n_dot = raw["Cdd"].shape[0]
    with reference_modules() as ref:
        kw = {}
        if raw["barriers"]:
            kw = dict(Cbd=raw["Cbd"], Cbg=raw["Cbg"], Cbs=raw["Cbs"], Cbb=raw["Cbb"],
                      barrier_model=ref.BarrierVoltageModel(n_barrier=n_dot - 1, n_dot=n_dot, tc_base=raw["tc_base"],
                                                            alpha=list(raw["alpha"])))
        model = ref.TunnelCoupledChargeSensed(
            Cdd=raw["Cdd"], Cgd=raw["Cgd"], Cds=raw["Cds"], Cgs=raw["Cgs"], coulomb_peak_width=raw["peak_width"],
            T=raw["T"], max_charge_carriers=4, tc=raw["tc"], noise_model=None, latching_model=None,
            voltage_capacitance_model=None, use_sparse=False, num_charge_states=32, charge_state_batch_size=1000,
            charge_carrier="electrons", **kw)
        if raw["vc"].any():                              # qarray_base_class.py:846-852
            vdc = sys.modules["qarray_latched.DotArrays.voltage_dependent_capacitance"]
            import jax.numpy as jnp
            c0, g0 = jnp.array(model.cdd_full), jnp.array(model.cgd_full)
            kind = int(raw.get("vc_kind", 0))
            if kind == 1:
                model.voltage_capacitance_model = vdc.create_quadratic_capacitance_model(
                    cdd_0=c0, cgd_0=g0, gamma=float(raw["vc"][0]), beta=float(raw["vc"][1]))
            elif kind == 2:
                model.voltage_capacitance_model = vdc.create_sigmoid_capacitance_model(
                    cdd_0=c0, cgd_0=g0, v_char=float(raw["vc_vchar"]), delta=float(raw["vc"][0]), beta=float(raw["vc"][1]))
            else:
                model.voltage_capacitance_model = vdc.create_linear_capacitance_model(
                    cdd_0=c0, cgd_0=g0, alpha=float(raw["vc"][0]), beta=float(raw["vc"][1]))
        comp = model.gate_voltage_composer
        perfect_vgm = np.array(comp.virtual_gate_matrix)
        if raw["vgm_kind"] == "identity":                # qarray_base_class.py:868-877 (electrons: -I)
            comp.virtual_gate_matrix = -np.eye(model.n_gate)
        # ground truth in virtual coordinates: solve with the reference's own matrices (no upstream optimal_Vg here)
        n_target = np.concatenate([np.ones(n_dot), [0.53]])
        vg_gt = np.linalg.solve(model.cgd_full[:, :model.n_gate], n_target)     # continuous minimum == n_target
        vd_gt = np.linalg.solve(np.array(comp.virtual_gate_matrix), vg_gt - np.array(comp.virtual_gate_origin))
        gate_voltages = vd_gt.copy()
        gate_voltages[:n_dot] += raw["centre_offset"]
        g1 = raw["pair"]
        v1, v2, half, res = gate_voltages[g1 - 1], gate_voltages[g1], raw["half"], raw["res"]
        vg = comp.do2d(f"vP{g1}", v1 - half, v1 + half, res, f"vP{g1 + 1}", v2 - half, v2 + half, res,
                       gate_voltages, True)
        vg_flat = vg.reshape(-1, vg.shape[-1])
        if raw["barriers"]:
            vb = np.full((vg_flat.shape[0], n_dot - 1), raw["barrier_voltages"])
            z, n = model.charge_sensor_open(vg_flat, vb)
        else:
            z, n = model.charge_sensor_open(vg_flat)
        return dict(cdd_full=np.array(model.cdd_full), cdd_inv_full=np.array(model.cdd_inv_full),
                    cgd_full=np.array(model.cgd_full), perfect_vgm=perfect_vgm,
                    vgm=np.array(comp.virtual_gate_matrix), origin=np.array(comp.virtual_gate_origin),
                    gate_voltages=gate_voltages, window=np.array([v1 - half, v1 + half, v2 - half, v2 + half]),
                    vg=np.array(vg), z=np.array(z, dtype=np.float64).reshape(res, res),
                    n=np.array(n, dtype=np.float64).reshape(res, res, n_dot))


# ---------------------------------------------------------------------------------------------------------------------
# Path A: the constant-interaction ground state lives in the absent qarray wheel, but the reference carries in-tree
# mirrors of its pieces.  These goldens execute THOSE FUNCTIONS (compiled from the reference's own source text, nothing
# copied): free_energy + open_charge_configurations_jax (src/qarray_latched/functions.py:30-47), convert_to_maxwell
# (DotArrays/_helper_functions.py:129-164), GateVoltageComposer.do2d with physical gates (GateVoltageComposer.py:224-255),
# optimal_Vg + compute_optimal_virtual_gate_matrix (src/qarray_latched/optimal_v_calc.py:10-44).  The one piece that
# cannot run is the ADMM solver of the relaxation QP (jaxopt.BoxOSQP, functions.py:66-81): its PROBLEM is taken from
# the reference (P = cdd_inv, q = -cdd_inv cgd vg, n >= 0) and solved exactly with scipy.optimize.nnls.
# ---------------------------------------------------------------------------------------------------------------------
CASES_A = {
    "ref_a_2dot_64x64": dict(n_dot=2, res=64, seed=21, pair=1),
    "ref_a_4dot_32x32": dict(n_dot=4, res=32, seed=22, pair=2),
    "ref_a_6dot_20x20": dict(n_dot=6, res=20, seed=23, pair=3),
    "ref_a_8dot_16x16": dict(n_dot=8, res=16, seed=24, pair=6),
}


def _reference_functions(path, names, namespace):
    """Compile the named top-level functions of a reference source file into ``namespace`` (the file itself cannot be
    imported: it needs jaxopt and plots at import time)."""
    import ast
    tree = ast.parse(open(path).read(), filename=path)
    body = [node for node in ast.walk(tree) if isinstance(node, ast.FunctionDef) and node.name in names]
    assert {b.name for b in body} == set(names), [b.name for b in body]
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), namespace)
    return namespace


def run_reference_path_a(n_dot, res, seed, pair):
    from scipy.optimize import nnls
    import refshim
    from qdsim import synth
    dev = synth.sample_devices(1, n_dot, seed=seed)
    rng = np.random.default_rng([seed, 6])
    Cdd, Cgd, Cds, Cgs = (dev[k][0] for k in ("Cdd", "Cgd", "Cds", "Cgs"))
    with refshim.reference_modules() as ref:
        import jax.numpy as jnp
        helpers = sys.modules["qarray_latched.DotArrays._helper_functions"]
        composer_mod = sys.modules["qarray_latched.DotArrays.GateVoltageComposer"]
        fn = _reference_functions(os.path.join(refshim.ref_src(), "qarray_latched", "functions.py"),
                                  ["free_energy", "open_charge_configurations_jax"], {"jnp": jnp})
        opt = _reference_functions(os.path.join(refshim.ref_src(), "qarray_latched", "optimal_v_calc.py"),
                                   ["optimal_Vg", "compute_optimal_virtual_gate_matrix"],
                                   {"np": np, "CddInv": None, "Cgd_holes": None, "VectorList": None})
        cdd, cdd_inv, cgd = (np.array(a) for a in helpers.convert_to_maxwell(Cdd, Cgd))
        cdd_full, cdd_inv_full, cgd_full = (np.array(a) for a in helpers._convert_to_maxwell_with_sensor(Cdd, Cgd, Cds, Cgs))
        n_target = np.concatenate([np.ones(n_dot), [0.53]])
        vg_opt = opt["optimal_Vg"](cdd_inv_full, cgd_full, n_target, rcond=1e-3)
        vgm_opt = opt["compute_optimal_virtual_gate_matrix"](cdd_inv_full, cgd_full)
        comp = composer_mod.GateVoltageComposer(n_gate=n_dot + 1, n_dot=n_dot, n_sensor=1)
        half = float(rng.uniform(1.5, 2.0))
        centre = vg_opt[:n_dot] + rng.uniform(-2.5, 2.5, size=n_dot)       # holes convention: cgd = -Cgd, vg < 0 fills dots
        x0, y0 = centre[pair - 1], centre[pair]
        grid = comp.do2d(pair, x0 - half, x0 + half, res, pair + 1, y0 - half, y0 + half, res)
        base = np.concatenate([centre, vg_opt[n_dot:]])
        base[pair - 1] = base[pair] = 0.0
        vg = grid + base                                                    # other plungers at their set point
        r = np.linalg.cholesky(cdd_inv).T
        flat = vg.reshape(-1, n_dot + 1)
        n_c = np.empty((flat.shape[0], n_dot))
        n_out = np.empty((flat.shape[0], n_dot))
        margin = np.empty(flat.shape[0])
        for i, v in enumerate(flat):
            n_c[i] = nnls(r, r @ (cgd @ v), maxiter=200)[0]                  # the reference's QP, solved exactly
            basis = fn["open_charge_configurations_jax"](jnp.array(n_c[i]))
            energies = np.asarray(fn["free_energy"](v, cdd_inv, cgd, basis))
            k = int(np.argmin(energies))
            n_out[i] = basis[k]
            e = np.sort(energies)
            margin[i] = e[1] - e[0]
    return dict(Cdd=Cdd, Cgd=Cgd, Cds=Cds, Cgs=Cgs, cdd=cdd, cdd_inv=cdd_inv, cgd=cgd, cdd_inv_full=cdd_inv_full,
                cgd_full=cgd_full, vg_opt=vg_opt, vgm_opt=vgm_opt, n_target=n_target, base=base, pair=pair, res=res,
                window=np.array([x0 - half, x0 + half, y0 - half, y0 + half]), vg=vg,
                n_continuous=n_c.reshape(res, res, n_dot), n=n_out.reshape(res, res, n_dot),
                margin=margin.reshape(res, res))


# ---------------------------------------------------------------------------------------------------------------------
# Virtualisation in the loop (SURVEY 8f rank 2): the reference's Kalman / direct updaters are plain NumPy and import as
# they are; the VGM update is a method of QarrayBaseClass (which cannot be imported: it needs the qarray wheel), so the
# two methods are compiled from the reference's source text and called on a stand-in ``self``.
# ---------------------------------------------------------------------------------------------------------------------
def run_reference_virtualisation(n_env=5, n_dot=6, n_step=8, seed=31):
    import importlib.util
    import types
    import refshim
    from qdsim import synth
    rng = np.random.default_rng(seed)
    base = os.path.join(refshim.ref_src(), "qadapt", "capacitance_model")
    out = {}
    for method, fname, cls in (("kalman", "KalmanUpdater.py", "KalmanCapacitanceUpdater"),
                               ("direct", "DirectUpdater.py", "DirectCapacitanceUpdater")):
        spec = importlib.util.spec_from_file_location("ref_" + method, os.path.join(base, fname))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        for k_out in (3, 2):
            values = rng.normal(0.0, 0.3, size=(n_step, n_env, n_dot - 1, k_out)).astype(np.float32)
            log_vars = rng.uniform(-8.0, 0.0, size=(n_step, n_env, n_dot - 1, k_out)).astype(np.float32)
            means = np.zeros((n_step, n_env, n_dot, n_dot))
            variances = np.zeros_like(means)
            full = np.zeros_like(means)
            for e in range(n_env):
                upd = getattr(mod, cls)(n_dots=n_dot, prior_mean=0.3, prior_variance=0.5, variance_threshold=0.05,
                                        process_noise=0.01 if e % 2 else 0.0, include_nnn=(k_out == 3),
                                        prior_mean_nnn=0.15)
                for t in range(n_step):
                    for i in range(n_dot - 1):       # the caller's loop, env.py:596-618 (values negated there)
                        upd.update_from_scan(left_dot=i, ml_outputs=[
                            (-float(values[t, e, i, k]), float(log_vars[t, e, i, k])) for k in range(k_out)])
                    means[t, e], variances[t, e], full[t, e] = upd.means, upd.variances, upd.get_full_matrix()
            tag = f"{method}_k{k_out}"
            out.update({tag + "_values": values, tag + "_log_vars": log_vars, tag + "_means": means,
                        tag + "_variances": variances, tag + "_full": full})
    # VGM update, barrier mode
    dev = synth.sample_barrier_devices(n_env, n_dot, seed=seed)
    mb = synth.tunnel_batch(dev)
    fn = _reference_functions(os.path.join(refshim.ref_src(), "qadapt", "environment", "qarray_base_class.py"),
                              ["_update_virtual_gate_matrix", "_set_vgm_for_target_effective_coupling"], {"np": np})
    est = rng.uniform(0.0, 0.6, size=(n_env, n_dot, n_dot))
    est = 0.5 * (est + est.transpose(0, 2, 1))
    est[:, np.arange(n_dot), np.arange(n_dot)] = 1.0
    target = np.broadcast_to(np.eye(n_dot), (n_env, n_dot, n_dot)).copy()
    target[:, 0, 1] = target[:, 1, 0] = rng.uniform(-0.4, 0.4, size=n_env)
    vgm_e, vgm_h, vgm_t = [], [], []
    for e in range(n_env):
        for carrier, sink in (("electrons", vgm_e), ("h", vgm_h)):
            composer = types.SimpleNamespace(virtual_gate_matrix=None)
            model = types.SimpleNamespace(cgd_full=mb.cgd_full[e], cdd_inv_full=mb.cdd_inv_full[e], n_gate=n_dot + 1,
                                          charge_carrier=carrier, gate_voltage_composer=composer)
            me = types.SimpleNamespace(use_barriers=True, model=model, num_dots=n_dot, num_barrier_voltages=n_dot - 1)
            fn["_update_virtual_gate_matrix"](me, est[e])
            sink.append(np.array(composer.virtual_gate_matrix))
        fn["_set_vgm_for_target_effective_coupling"](me, target[e])          # 'h' model from the loop above
        vgm_t.append(np.array(composer.virtual_gate_matrix))
    out.update(cdd_inv_full=mb.cdd_inv_full, cgd_full=mb.cgd_full, cgd_estimate=est, vgm_electrons=np.stack(vgm_e),
               vgm_holes=np.stack(vgm_h), target=target, vgm_target_holes=np.stack(vgm_t), n_dot=n_dot)
    return out


def main(only=None):
    if not only or "ref_virtualisation" in only:
        np.savez_compressed(os.path.join(HERE, "ref_virtualisation.npz"), **run_reference_virtualisation())
        print("ref_virtualisation: kalman/direct x {3, 2} outputs, VGM update", flush=True)
    for name, spec in CASES_A.items():
        if only and name not in only:
            continue
        out = run_reference_path_a(**spec)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print(f"{name}: n range [{out['n'].min():.0f}, {out['n'].max():.0f}], relaxed pixels "
              f"{(out['vg'].reshape(-1, out['vg'].shape[-1]) @ out['cgd'].T < 0).any(axis=1).mean():.2f}, "
              f"min margin {out['margin'].min():.2e}", flush=True)
    for name, spec in CASES.items():
        if only and name not in only:
            continue
        raw = case_inputs(**spec)
        out = run_reference(raw)
        save = {k: v for k, v in raw.items() if v is not None}
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **save, **out)
        n = out["n"]
        print(f"{name}: n range [{n.min():.3f}, {n.max():.3f}], z range [{out['z'].min():.4f}, {out['z'].max():.4f}], "
              f"non-integer pixels {(np.abs(n - np.rint(n)).max(axis=-1) > 1e-3).mean():.2f}", flush=True)


if __name__ == "__main__":
    main(sys.argv[1:])
