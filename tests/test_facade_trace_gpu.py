"""The reference facade's own call sequence, replayed on the CUDA engine (north_star: "src/qadapt's env ... run unchanged on
top").  tests/golden/make_facade_trace.py recorded -- in the CPU container, with the REAL ``QarrayBaseClass._get_obs``
(src/qadapt/environment/qarray_base_class.py:171-229) on top of the drop-in classes -- every constructor
kwarg, VGM assignment, ``do2d`` / ``charge_sensor_open`` / ``do2d_open`` argument and scan seed, together with the outputs of
the CPU oracle engine.  Here the SAME drop-in classes are built from the recorded kwargs and driven with the recorded
arguments, with ``libqdsim.so`` underneath; outputs are compared with the recorded ones.  Barrier and non-barrier mode."""
import os
import pickle
import sys

import numpy as np
import pytest

from util import assert_z_given_n, explain_latched_mismatches

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _load(name):
    return pickle.loads(np.load(os.path.join(HERE, "golden", f"facade_trace_{name}.npz"))["trace"].tobytes())


def _noise_and_latching(ctor):
    import qarray
    nz = ctor["noise"]
    noise = qarray.WhiteNoise(amplitude=nz.get("white_amp", 0.0)) + qarray.TelegraphNoise(
        p01=nz.get("tele_p01", 0.0), p10=nz.get("tele_p10", 0.0), amplitude=nz.get("tele_amp", 0.0))
    lt = ctor["latching"]
    latching = qarray.LatchingModel(n_dots=lt["n_dots"], p_leads=lt["p_leads"], p_inter=lt["p_inter"]) if lt else None
    return noise, latching


def _pin_seeds(monkeypatch, module, seeds):
    it = iter(seeds)
    monkeypatch.setattr(module, "fresh_seed", lambda: next(it))


def test_barrier_mode_trace_replays_on_cuda(monkeypatch):
    from qarray_latched.DotArrays.barrier_voltage_model import BarrierVoltageModel
    from qarray_latched.DotArrays.TunnelCoupledChargeSensed import TunnelCoupledChargeSensed
    tr = _load("barriers")
    c = tr["ctor"]
    noise, latching = _noise_and_latching(c)
    n_dot = tr["num_dots"]
    bm = BarrierVoltageModel(n_barrier=n_dot - 1, n_dot=n_dot, tc_base=c["tc_base"], alpha=list(c["alpha"]))
    m = TunnelCoupledChargeSensed(
        Cdd=c["Cdd"], Cgd=c["Cgd"], Cds=c["Cds"], Cgs=c["Cgs"], Cbd=c["Cbd"], Cbg=c["Cbg"], Cbs=c["Cbs"], Cbb=c["Cbb"],
        barrier_model=bm, coulomb_peak_width=c["coulomb_peak_width"], T=c["T"], max_charge_carriers=c["max_charge_carriers"],
        tc=c["tc"], noise_model=noise, latching_model=latching, voltage_capacitance_model=None, use_sparse=c["use_sparse"],
        num_charge_states=c["num_charge_states"], charge_state_batch_size=c["charge_state_batch_size"],
        charge_carrier=c["charge_carrier"])
    _pin_seeds(monkeypatch, sys.modules[TunnelCoupledChargeSensed.__module__], [e["seed"] for e in tr["calls"]])
    res = tr["res"]
    w_max = float(np.abs(m.cdd_inv_full[-1, :-1]).max())
    states = set()
    n_amb = 0
    for e in tr["calls"]:
        comp = m.gate_voltage_composer
        comp.virtual_gate_matrix, comp.virtual_gate_origin = e["vgm"], e["origin"]         # qarray_base_class.py:876-946
        states.add(e["vgm"].tobytes())
        m.coulomb_peak_width = e["peak_width"]
        vg = comp.do2d(*e["do2d_args"])                                                      # :143-154
        np.testing.assert_allclose(vg, e["vg_grid"], rtol=0, atol=1e-12)
        z, n = m.charge_sensor_open(vg.reshape(-1, vg.shape[-1]), e["vb"])                   # :157-163
        assert z.shape == e["z"].shape and n.shape == e["n"].shape
        # the facade's call is ONE latching sequence over the flattened image
        d, a, _ = explain_latched_mismatches(n.reshape(1, -1, n_dot), e["n"].reshape(1, -1, n_dot),
                                             e["n_free"].reshape(1, -1, n_dot), e["gap"].reshape(1, -1), carry_rows=True)
        n_amb += a
        same = (np.abs(n - e["n"]).max(axis=-1) <= 1e-6) & (e["gap"] > 1e-5)
        assert same.mean() > 0.5 or a == 1
        assert_z_given_n(z.reshape(-1), e["z"].reshape(-1), n, e["n"], same, w_max, e["peak_width"], noise_atol=5e-6)
        assert z.reshape(res, res).shape == (res, res)
    assert len(states) == 3                       # -I, perfect and an updated virtual gate matrix were exercised
    assert n_amb <= 2, f"{n_amb} of {len(tr['calls'])} recorded calls hit a half-integer / small-gap pixel"


def test_non_barrier_mode_trace_replays_on_cuda(monkeypatch):
    import qarray
    tr = _load("no_barriers")
    c = tr["ctor"]
    noise, latching = _noise_and_latching(c)
    m = qarray.ChargeSensedDotArray(Cdd=c["Cdd"], Cgd=c["Cgd"], Cds=c["Cds"], Cgs=c["Cgs"],
                                    coulomb_peak_width=c["coulomb_peak_width"], T=c["T"], noise_model=noise,
                                    latching_model=latching, algorithm=c["algorithm"], implementation=c["implementation"],
                                    max_charge_carriers=c["max_charge_carriers"])
    _pin_seeds(monkeypatch, sys.modules[qarray.ChargeSensedDotArray.__module__], [e["seed"] for e in tr["calls"]])
    n_dot = tr["num_dots"]
    for e in tr["calls"]:
        m.coulomb_peak_width = e["peak_width"]
        z, n = m.do2d_open(*e["args"])                                                       # :128-137
        assert z.shape == e["z"].shape and n.shape == e["n"].shape
        # T > 0 (the facade passes T ~ U[50, 200]): occupations are Boltzmann averages; the rounded latch compare may flip
        # where a free <n> sits on a half-integer -- explained the same way, rows are independent here
        from util import oracle_batch  # noqa: F401
        free = e["n"]                                                                       # upper bound of ambiguity: latched n
        gap = np.full(e["z"].shape[:2], np.inf)
        d, a, rows = explain_latched_mismatches(n, e["n"], free, gap, n_atol=1e-8, half_tol=1e-7)
        same = np.abs(n - e["n"]).max(axis=-1) <= 1e-8
        assert same.mean() > 0.99
        np.testing.assert_allclose(z[..., 0][same], e["z"][..., 0][same], rtol=0, atol=5e-6)
