"""Import-surface compatibility with the REAL reference facade, when ``QADAPT_SRC`` points at the upstream project's
``src`` tree.  The reference's QarrayBaseClass is imported unchanged with our ``qarray`` /
``qarray_latched`` packages first on sys.path, and constructs its model through our classes.  Nothing here computes."""
import os
import sys
import types

import numpy as np
import pytest

from util import REFERENCE_SRC as REF
pytestmark = pytest.mark.skipif(not os.path.isdir(REF), reason="reference tree not present")


@pytest.fixture()
def reference_facade(monkeypatch):
    # stand-ins for modules the reference imports at module scope but does not need on this path
    if "jax" not in sys.modules:
        jax = types.ModuleType("jax")
        jnp = types.ModuleType("jax.numpy")
        jnp.full = np.full
        jnp.array = np.array
        jnp.ndarray = np.ndarray
        jax.numpy = jnp
        monkeypatch.setitem(sys.modules, "jax", jax)
        monkeypatch.setitem(sys.modules, "jax.numpy", jnp)
    if "matplotlib" not in sys.modules:
        mpl = types.ModuleType("matplotlib")
        mpl.use = lambda *a, **k: None
        plt = types.ModuleType("matplotlib.pyplot")
        mpl.pyplot = plt
        monkeypatch.setitem(sys.modules, "matplotlib", mpl)
        monkeypatch.setitem(sys.modules, "matplotlib.pyplot", plt)
    monkeypatch.syspath_prepend(REF)
    # our drop-ins must win over the reference's vendored qarray_latched
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rl-agent-for-qubit-array-tuning_b200")
    monkeypatch.syspath_prepend(pkg)
    for name in [m for m in sys.modules if m.startswith(("qadapt", "qarray_latched"))]:
        monkeypatch.delitem(sys.modules, name)
    # bind the reference's packages as bare namespaces: their __init__ pulls gymnasium / ray, which this path never uses
    for name, path in (("qadapt", REF + "/qadapt"), ("qadapt.environment", REF + "/qadapt/environment")):
        pkg_mod = types.ModuleType(name)
        pkg_mod.__path__ = [path]
        monkeypatch.setitem(sys.modules, name, pkg_mod)
    import importlib
    mod = importlib.import_module("qadapt.environment.qarray_base_class")
    # the reference re-inserts its own src dir at sys.path[0] on import; make sure our packages were the ones bound
    import qarray
    assert "rl-agent-for-qubit-array-tuning_b200" in qarray.__file__
    return mod


def test_reference_facade_builds_its_model_through_our_classes(reference_facade):
    import qarray
    base = reference_facade.QarrayBaseClass(num_dots=4, use_barriers=False, obs_image_size=32)
    m = base.model
    assert isinstance(m, qarray.ChargeSensedDotArray)
    assert m.n_dot == 4 and m.n_gate == 5 and m.cgd_full.shape == (5, 5) and m.cdd_inv_full.shape == (5, 5)
    # attribute surface the facade and env.py read or assign
    base._reset_virtual_gate_matrix_to_identity()
    assert np.array_equal(m.gate_voltage_composer.virtual_gate_matrix, np.eye(5))
    base._reset_virtual_gate_matrix_to_perfect()
    assert np.allclose(m.cdd_inv_full @ m.cgd_full @ m.gate_voltage_composer.virtual_gate_matrix, -np.eye(5), atol=1e-9)
    base._update_virtual_gate_matrix(np.abs(m.cgd[:, :4]) if False else np.eye(4) + 0.1)
    vg = m.optimal_Vg(base.optimal_VG_center)
    assert vg.shape == (5,)
    assert isinstance(m.latching_model, qarray.LatchingModel) and m.noise_model._kernel_params()["white_amp"] >= 0


def test_reference_facade_builds_the_barrier_model_through_our_classes(reference_facade):
    import qarray_latched
    base = reference_facade.QarrayBaseClass(num_dots=4, use_barriers=True, obs_image_size=32)
    m = base.model
    assert isinstance(m, qarray_latched.TunnelCoupledChargeSensed)
    assert "rl-agent-for-qubit-array-tuning_b200" in qarray_latched.__file__
    assert m.n_barrier == 3 and m.cgd_full.shape == (5, 8) and m.num_charge_states == 32
    assert m.charge_carrier == "electrons"
    assert np.allclose(m.gate_voltage_composer.virtual_gate_matrix,
                       np.linalg.pinv(m.cdd_inv_full @ m.cgd_full[:, :5]), atol=1e-9)
    base._reset_virtual_gate_matrix_to_identity()
    assert np.array_equal(m.gate_voltage_composer.virtual_gate_matrix, -np.eye(5))
    base._update_virtual_gate_matrix(np.eye(4) + 0.05)
    pg, bg, sg = base.calculate_ground_truth(np.zeros(4), np.zeros(3)) if False else (None, None, None)
    mb = m._model_batch()
    assert mb.algorithm == "tunnel" and mb.n_volt == 8 and mb.cbg.shape == (1, 3, 5)
    # the composer call the facade makes every step (qarray_base_class.py:143-154)
    vg = m.gate_voltage_composer.do2d("vP1", -1.0, 1.0, 32, "vP2", -1.0, 1.0, 32, np.zeros(5), True)
    assert vg.shape == (32, 32, 5)


def test_reference_facade_with_linear_voltage_capacitance(reference_facade, tmp_path):
    """``voltage_capacitance_model.type: linear`` (qarray_config.yaml:132-134): the facade builds the linear model on the
    model's own matrices (qarray_base_class.py:842-852) and our class turns it into the two kernel parameters."""
    import yaml
    cfg_path = os.path.join(REF, "qadapt", "environment", "qarray_config.yaml")
    cfg = yaml.safe_load(open(cfg_path))
    cfg["simulator"]["voltage_capacitance_model"]["type"] = "linear"
    p = tmp_path / "qarray_config_linear.yaml"
    p.write_text(yaml.safe_dump(cfg))
    base = reference_facade.QarrayBaseClass(num_dots=4, use_barriers=True, obs_image_size=16, config_path=str(p))
    m = base.model
    assert m.voltage_capacitance_model is not None and m.voltage_capacitance_model.kind == "linear"
    mb = m._model_batch()
    assert 0.05 <= mb.params["vc_alpha"][0] <= 0.10 and 0.05 <= mb.params["vc_beta"][0] <= 0.10
