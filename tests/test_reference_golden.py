"""Parity against the REFERENCE ITSELF (tests/golden/ref_*.npz).

The fixtures were produced by running the reference's unmodified in-tree simulator
(src/qarray_latched/DotArrays: TunnelCoupledChargeSensed.charge_sensor_open -> _ground_state_open ->
build_charge_states / hamiltonian_build / barrier_voltage_model, plus GateVoltageComposer.do2d and the Maxwell
conversion) in this container -- see tests/golden/make_reference_golden.py and tests/golden/refshim.py.  They pin, with
numbers that come from reference code only:

* S1  Maxwell conversion with sensor + barriers           (_helper_functions.py:29-164)
* S2  coupled virtual scan grid                           (GateVoltageComposer.py:170-255)
* A1  optimal virtual gate matrix                         (TunnelCoupledChargeSensed.py:176-183)
* B1-B6 tunnel-coupled ground state <n>                   (ground_state.py:24-166 and callees)
* S3/S4 sensor signal                                     (TunnelCoupledChargeSensed.py:320-380)

CPU: the oracle and the product's host code reproduce them.  GPU: the CUDA path reproduces them through the drop-in
class and through the batched affine-scan entry.  Pixels whose Hamiltonian has a (near-)degenerate ground state have no
unique <n> (any vector of the eigenspace is a valid LAPACK answer); they are excluded by spectral gap and must be rare.
"""
import os

import numpy as np
import pytest

from oracle import scan as oscan
from util import reference_path

HERE = os.path.dirname(os.path.abspath(__file__))
REF_CASES = ["ref_4dot_tunnel_identity_vgm", "ref_4dot_tunnel_perfect_vgm_cbb", "ref_5dot_tunnel_low_occupancy",
             "ref_6dot_tunnel_identity_vgm", "ref_8dot_tunnel_identity_vgm", "ref_4dot_constant_tc_no_barriers",
             "ref_4dot_tunnel_linear_capacitance", "ref_6dot_tunnel_linear_capacitance",
             "ref_4dot_tunnel_quadratic_capacitance", "ref_5dot_tunnel_sigmoid_capacitance",
             "ref_4dot_tunnel_strong_coupling", "ref_4dot_tunnel_closed_barriers", "ref_6dot_tunnel_far_window"]
GAP_TOL = 1e-6            # spectral gap below which <n> is not unique
N_ATOL_CPU = 1e-11        # LAPACK (reference run) vs LAPACK (oracle); measured 5e-14
N_ATOL_GPU = 2e-6         # Householder + Sturm multisection + inverse iteration on the GPU (tests/test_tunnel_gpu.py)
# sensor signal on the GPU: 1e-6 relative GIVEN <n> (util.assert_z_given_n: fp64 Lorentzians on the tunnel path; the only
# other term is the propagated, measured <n> difference of the same pixel)


def load(name):
    d = dict(np.load(os.path.join(HERE, "golden", name + ".npz")))
    d["barriers"] = bool(d["barriers"])
    return d


def product_model(d):
    """ModelBatch built by the product's host code from the fixture's RAW capacitances."""
    from qdsim import PARAMS_DTYPE
    from qdsim.engine import ModelBatch, tunnel_model_batch
    from qdsim import maxwell
    n = d["Cdd"].shape[0]
    if d["barriers"]:
        mb = tunnel_model_batch(d["Cdd"][None], d["Cgd"][None], d["Cds"][None], d["Cgs"][None], d["Cbd"][None],
                                d["Cbg"][None], d["Cbs"][None], float(d["tc_base"]), d["alpha"][None])
        if "vc" in d:
            mb.params["vc_alpha"], mb.params["vc_beta"] = d["vc"]
            mb.params["vc_kind"] = int(d["vc_kind"]) if "vc_kind" in d else 0
            mb.params["vc_vchar"] = float(d["vc_vchar"]) if "vc_vchar" in d else 1.0
        return mb
    cdd_nm, cgd_nm = maxwell.embed_sensor(d["Cdd"][None], d["Cgd"][None], d["Cds"][None], d["Cgs"][None])
    _, cdd_inv_full, cgd_full = maxwell.maxwell(cdd_nm, cgd_nm)
    params = np.zeros(1, dtype=PARAMS_DTYPE)
    params["tc_base"] = float(d["tc"])                     # constant nearest-neighbour coupling (ground_state.py:92-101)
    return ModelBatch(algorithm="tunnel", n_gate=n + 1, cdd_inv_gs=np.ascontiguousarray(cdd_inv_full[:, :n, :n]),
                      cdd_gs=None, cdd_inv_full=cdd_inv_full, cgd_full=cgd_full, params=params, cbg=None)


def v_ext(d):
    res = int(d["res"])
    vg = d["vg"].reshape(res, res, -1)
    if not d["barriers"]:
        return vg
    vb = np.broadcast_to(d["barrier_voltages"], (res, res, d["barrier_voltages"].size))
    return np.concatenate([vg, vb], axis=-1)


def oracle_run(d):
    from util import oracle_model
    mb = product_model(d)
    m = oracle_model(mb, 0, 0)
    s = oscan.Scan(v0=None, dx=None, dy=None, nx=int(d["res"]), ny=int(d["res"]), peak_width=float(d["peak_width"]))
    return oscan.simulate_points(m, v_ext(d), s, return_margin=True)


@pytest.mark.parametrize("name", REF_CASES)
def test_host_code_matches_reference_matrices(name):
    """S1, S2, A1: Maxwell matrices, virtual gate matrix and the scan grid equal the reference's."""
    from qdsim import maxwell
    from qdsim.composer import GateVoltageComposer
    d = load(name)
    mb = product_model(d)
    np.testing.assert_allclose(mb.cdd_inv_full[0], d["cdd_inv_full"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(mb.cgd_full[0], d["cgd_full"], rtol=0, atol=0)
    n_gate = d["Cgd"].shape[1]
    vgm = maxwell.optimal_vgm(mb.cdd_inv_full[0], mb.cgd_full[0][:, :n_gate], electrons=True)
    np.testing.assert_allclose(vgm, d["perfect_vgm"], rtol=1e-10, atol=1e-12)
    comp = GateVoltageComposer(n_gate=n_gate, n_dot=n_gate - 1, n_sensor=1, virtual_gate_matrix=d["vgm"],
                               virtual_gate_origin=d["origin"])
    g1, res, w = int(d["pair"]), int(d["res"]), d["window"]
    args = (f"vP{g1}", w[0], w[1], res, f"vP{g1 + 1}", w[2], w[3], res, d["gate_voltages"], True)
    np.testing.assert_allclose(comp.do2d(*args), d["vg"], rtol=1e-12, atol=1e-12)
    v0, dx, dy = comp.affine2d(*args)
    iy, ix = np.meshgrid(np.arange(res), np.arange(res), indexing="ij")
    grid = v0 + ix[..., None] * dx + iy[..., None] * dy
    np.testing.assert_allclose(grid, d["vg"], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("name", REF_CASES)
def test_oracle_matches_reference(name):
    """B1-B6 + S3: the NumPy restatement equals the reference's own output on the reference's own grid."""
    d = load(name)
    z, n, gap = oracle_run(d)
    ok = gap > GAP_TOL
    assert ok.mean() > 0.98, f"{(~ok).sum()} degenerate pixels"
    np.testing.assert_allclose(n[ok], d["n"][ok], rtol=0, atol=N_ATOL_CPU)
    np.testing.assert_allclose(z[ok], d["z"][ok], rtol=1e-11, atol=1e-13)
    if "closed_barriers" not in name:                             # (that fixture is the t -> 0 limit: integer charges)
        assert np.abs(d["n"] - np.rint(d["n"])).max() > 1e-2      # the fixture exercises real tunnel mixing


@pytest.mark.skipif(not os.path.isdir(reference_path("qarray_latched")), reason="reference tree not present")
def test_reference_regenerates_fixture():
    """The committed fixtures are what the reference produces today (guards against stale or hand-edited files): one of
    each family is regenerated from the upstream ``src`` tree (``QADAPT_SRC``) and compared."""
    import sys
    sys.path.insert(0, os.path.join(HERE, "golden"))
    import make_reference_golden as gen
    for name in ("ref_4dot_tunnel_identity_vgm", "ref_6dot_tunnel_linear_capacitance"):
        out = gen.run_reference(gen.case_inputs(**gen.CASES[name]))
        d = load(name)
        np.testing.assert_allclose(out["n"], d["n"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(out["z"], d["z"], rtol=0, atol=1e-12)
    out = gen.run_reference_path_a(**gen.CASES_A["ref_a_4dot_32x32"])
    d = load_a("ref_a_4dot_32x32")
    assert np.array_equal(out["n"], d["n"])
    np.testing.assert_allclose(out["n_continuous"], d["n_continuous"], rtol=0, atol=1e-12)
    out = gen.run_reference_virtualisation()
    d = dict(np.load(os.path.join(HERE, "golden", "ref_virtualisation.npz")))
    for k in ("kalman_k3_means", "direct_k2_variances", "vgm_electrons", "vgm_target_holes"):
        np.testing.assert_allclose(out[k], d[k], rtol=0, atol=1e-12)
    import qarray                                             # the product's packages are back after the shim context
    assert "rl-agent-for-qubit-array-tuning_b200" in qarray.__file__


def _drop_in(d, device=0):
    from qarray_latched.DotArrays import BarrierVoltageModel, TunnelCoupledChargeSensed
    n = d["Cdd"].shape[0]
    kw = {}
    if d["barriers"]:
        kw = dict(Cbd=d["Cbd"], Cbg=d["Cbg"], Cbs=d["Cbs"], Cbb=d.get("Cbb"),
                  barrier_model=BarrierVoltageModel(n_barrier=n - 1, n_dot=n, tc_base=float(d["tc_base"]),
                                                    alpha=list(d["alpha"])))
    model = TunnelCoupledChargeSensed(
        Cdd=d["Cdd"], Cgd=d["Cgd"], Cds=d["Cds"], Cgs=d["Cgs"], coulomb_peak_width=float(d["peak_width"]),
        T=float(d["T"]), max_charge_carriers=4, tc=float(d["tc"]), noise_model=None, latching_model=None,
        voltage_capacitance_model=None, use_sparse=False, num_charge_states=32, charge_state_batch_size=1000,
        charge_carrier="electrons", device=device, **kw)
    if "vc" in d and d["vc"].any():                      # qarray_base_class.py:846-852
        from qarray_latched.DotArrays import voltage_dependent_capacitance as vdc
        kind = int(d["vc_kind"]) if "vc_kind" in d else 0
        a, b = float(d["vc"][0]), float(d["vc"][1])
        if kind == 1:
            model.voltage_capacitance_model = vdc.create_quadratic_capacitance_model(
                cdd_0=model.cdd_full, cgd_0=model.cgd_full, gamma=a, beta=b)
        elif kind == 2:
            model.voltage_capacitance_model = vdc.create_sigmoid_capacitance_model(
                cdd_0=model.cdd_full, cgd_0=model.cgd_full, v_char=float(d["vc_vchar"]), delta=a, beta=b)
        else:
            model.voltage_capacitance_model = vdc.create_linear_capacitance_model(
                cdd_0=model.cdd_full, cgd_0=model.cgd_full, alpha=a, beta=b)
    return model


@pytest.mark.gpu
@pytest.mark.parametrize("name", REF_CASES)
def test_gpu_drop_in_class_matches_reference(name):
    """The reference's call sequence (qarray_base_class.py:143-163) on the drop-in class, CUDA underneath."""
    d = load(name)
    model = _drop_in(d)
    np.testing.assert_allclose(model.gate_voltage_composer.virtual_gate_matrix, d["perfect_vgm"], rtol=1e-10, atol=1e-12)
    model.gate_voltage_composer.virtual_gate_matrix = d["vgm"]
    g1, res, w = int(d["pair"]), int(d["res"]), d["window"]
    vg = model.gate_voltage_composer.do2d(f"vP{g1}", w[0], w[1], res, f"vP{g1 + 1}", w[2], w[3], res,
                                          d["gate_voltages"], True)
    vg_flat = vg.reshape(-1, vg.shape[-1])
    if d["barriers"]:
        vb = np.full((vg_flat.shape[0], d["barrier_voltages"].size), d["barrier_voltages"])
        z, n = model.charge_sensor_open(vg_flat, vb)
    else:
        z, n = model.charge_sensor_open(vg_flat)
    _, _, gap = oracle_run(d)
    ok = gap > 1e-5
    assert ok.mean() > 0.98
    n, z = n.reshape(res, res, -1), z.reshape(res, res)
    np.testing.assert_allclose(n[ok], d["n"][ok], rtol=0, atol=N_ATOL_GPU)
    from util import assert_z_given_n
    w_max = float(np.abs(model.cdd_inv_full[-1, :-1]).max())
    assert_z_given_n(z, d["z"], n, d["n"], ok, w_max, float(d["peak_width"]), what=name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", REF_CASES)
def test_gpu_affine_scan_matches_reference(engine, name):
    """Same through the batched entry the bench uses: affine descriptor, qd_scan_open_host."""
    from qdsim import N_F64
    from qdsim.composer import GateVoltageComposer
    from qdsim.engine import new_scans
    d = load(name)
    mb = product_model(d)
    engine.set_models(mb)
    n_gate = d["Cgd"].shape[1]
    comp = GateVoltageComposer(n_gate=n_gate, n_dot=n_gate - 1, n_sensor=1, virtual_gate_matrix=d["vgm"],
                               virtual_gate_origin=d["origin"])
    g1, res, w = int(d["pair"]), int(d["res"]), d["window"]
    v0, dx, dy = comp.affine2d(f"vP{g1}", w[0], w[1], res, f"vP{g1 + 1}", w[2], w[3], res, d["gate_voltages"], True)
    s = new_scans(1)
    s["v0"][0, :n_gate], s["dx"][0, :n_gate], s["dy"][0, :n_gate] = v0, dx, dy
    if d["barriers"]:
        s["v0"][0, n_gate:mb.n_volt] = d["barrier_voltages"]
    s["nx"], s["ny"], s["peak_width"] = res, res, float(d["peak_width"])
    z, n = engine.scan_open_host(s, n_type=N_F64, flags=0)
    _, _, gap = oracle_run(d)
    ok = gap > 1e-5
    n, z = n.reshape(res, res, -1), z.reshape(res, res)
    np.testing.assert_allclose(n[ok], d["n"][ok], rtol=0, atol=N_ATOL_GPU)
    from util import assert_z_given_n, sensor_w_max
    assert_z_given_n(z, d["z"], n, d["n"], ok, sensor_w_max(mb), float(d["peak_width"]), what=name)


# ---------------------------------------------------------------------------------------------------------------------
# Path A: fixtures made by executing the reference's in-tree mirrors of the absent qarray functions
# (make_reference_golden.py::run_reference_path_a): free_energy + floor/ceil enumeration (qarray_latched/functions.py:30-47),
# convert_to_maxwell, the physical-gate do2d grid, optimal_Vg / optimal virtual gate matrix (optimal_v_calc.py:10-44),
# with the relaxation QP of functions.py:66-81 solved exactly (NNLS).  Integer charges: bit-exact outside exact ties.
# ---------------------------------------------------------------------------------------------------------------------
REF_A_CASES = ["ref_a_2dot_64x64", "ref_a_4dot_32x32", "ref_a_6dot_20x20", "ref_a_8dot_16x16"]
TIE_TOL = 1e-9


def load_a(name):
    return dict(np.load(os.path.join(HERE, "golden", name + ".npz")))


@pytest.mark.parametrize("name", REF_A_CASES)
def test_path_a_host_code_matches_reference_mirrors(name):
    from qdsim import maxwell
    from qdsim.composer import GateVoltageComposer
    d = load_a(name)
    cdd, cdd_inv, cgd = maxwell.maxwell(d["Cdd"], d["Cgd"])
    np.testing.assert_allclose(cdd, d["cdd"], rtol=0, atol=1e-15)
    np.testing.assert_allclose(cdd_inv, d["cdd_inv"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(cgd, d["cgd"], rtol=0, atol=0)
    cdd_nm, cgd_nm = maxwell.embed_sensor(d["Cdd"], d["Cgd"], d["Cds"], d["Cgs"])
    _, cdd_inv_full, cgd_full = maxwell.maxwell(cdd_nm, cgd_nm)
    np.testing.assert_allclose(cdd_inv_full, d["cdd_inv_full"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(maxwell.optimal_vg(cdd_inv_full, cgd_full, d["n_target"], 1e-3), d["vg_opt"],
                               rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(maxwell.optimal_vgm(cdd_inv_full, cgd_full), d["vgm_opt"], rtol=1e-9, atol=1e-11)
    n_dot, res, pair, w = d["Cdd"].shape[0], int(d["res"]), int(d["pair"]), d["window"]
    comp = GateVoltageComposer(n_gate=n_dot + 1, n_dot=n_dot, n_sensor=1)
    grid = comp.do2d(pair, w[0], w[1], res, pair + 1, w[2], w[3], res) + d["base"]
    np.testing.assert_allclose(grid, d["vg"], rtol=1e-13, atol=1e-13)


@pytest.mark.parametrize("name", REF_A_CASES)
def test_path_a_oracle_matches_reference_mirrors(name):
    from oracle import path_a
    d = load_a(name)
    n_dot = d["Cdd"].shape[0]
    vg = d["vg"].reshape(-1, n_dot + 1)
    n_c = path_a.continuous_relaxation(vg @ d["cgd"].T, d["cdd"])
    np.testing.assert_allclose(n_c, d["n_continuous"].reshape(-1, n_dot), rtol=0, atol=1e-9)     # exact LCP == exact QP
    n, margin = path_a.ground_state_open(vg, d["cgd"], d["cdd_inv"], d["cdd"], "default", return_margin=True)
    safe = d["margin"].reshape(-1) > TIE_TOL
    assert safe.mean() > 0.995
    assert np.array_equal(n[safe], d["n"].reshape(-1, n_dot)[safe])
    np.testing.assert_allclose(margin[safe], d["margin"].reshape(-1)[safe], rtol=1e-6, atol=1e-10)


@pytest.mark.parametrize("name", REF_A_CASES)
def test_path_a_cport_matches_reference_mirrors(name):
    from oracle import cport
    from qdsim import N_U8  # noqa: F401
    from qdsim.engine import ModelBatch, new_scans
    d = load_a(name)
    n_dot, res = d["Cdd"].shape[0], int(d["res"])
    mb = ModelBatch.from_capacitances(d["Cdd"], d["Cgd"], d["Cds"], d["Cgs"], algorithm="default")
    s = _affine_scan_a(d, new_scans)
    _, nc, _ = cport.run_scans(mb, s, 0, threads=2)
    safe = d["margin"] > TIE_TOL
    assert np.array_equal(nc.reshape(res, res, n_dot)[safe], d["n"][safe])


def _affine_scan_a(d, new_scans):
    from qdsim.composer import GateVoltageComposer
    n_dot, res, pair, w = d["Cdd"].shape[0], int(d["res"]), int(d["pair"]), d["window"]
    comp = GateVoltageComposer(n_gate=n_dot + 1, n_dot=n_dot, n_sensor=1)
    v0, dx, dy = comp.affine2d(pair, w[0], w[1], res, pair + 1, w[2], w[3], res)
    s = new_scans(1)
    s["v0"][0, :n_dot + 1], s["dx"][0, :n_dot + 1], s["dy"][0, :n_dot + 1] = v0 + d["base"], dx, dy
    s["nx"], s["ny"] = res, res
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("name", REF_A_CASES)
def test_path_a_gpu_matches_reference_mirrors(engine, name):
    """CUDA path, both entries: the drop-in class on the reference's explicit grid and the batched affine scan."""
    from qarray import ChargeSensedDotArray
    from qdsim import N_U8
    from qdsim.engine import ModelBatch, new_scans
    d = load_a(name)
    n_dot, res = d["Cdd"].shape[0], int(d["res"])
    safe = d["margin"] > TIE_TOL
    model = ChargeSensedDotArray(Cdd=d["Cdd"], Cgd=d["Cgd"], Cds=d["Cds"], Cgs=d["Cgs"], coulomb_peak_width=0.2, T=0.0,
                                 algorithm="default", implementation="jax", max_charge_carriers=4)
    np.testing.assert_allclose(model.optimal_Vg(d["n_target"]), d["vg_opt"], rtol=1e-10, atol=1e-12)
    n = model.ground_state_open(d["vg"])
    assert np.array_equal(np.rint(n).astype(np.int64)[safe], d["n"].astype(np.int64)[safe])
    engine.set_models(ModelBatch.from_capacitances(d["Cdd"], d["Cgd"], d["Cds"], d["Cgs"], algorithm="default"))
    _, n2 = engine.scan_open_host(_affine_scan_a(d, new_scans), n_type=N_U8, flags=0)
    assert np.array_equal(n2.reshape(res, res, n_dot).astype(np.int64)[safe], d["n"].astype(np.int64)[safe])
