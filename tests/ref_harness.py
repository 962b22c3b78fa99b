"""Test-only harness: import the REAL reference facade / env from the upstream ``src`` tree (``QADAPT_SRC``) on top of
our drop-in ``qarray`` / ``qarray_latched`` packages, on a machine without a GPU.

* modules the reference imports but this path never needs (jax.numpy, matplotlib, gymnasium) get tiny stand-ins;
* the engine behind the drop-in classes is replaced by ``OracleEngine`` -- the CPU oracle answering the same calls.
  This is legitimate ONLY here: the point of these tests is interface compatibility and the host-side env logic, not
  GPU numerics (those are the -m gpu parity tests).  The product never does this.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np

from util import REFERENCE_SRC as REF
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "rl-agent-for-qubit-array-tuning_b200")


class OracleEngine:
    """Duck-types qdsim.Engine's host-buffer calls with the CPU oracle."""

    def __init__(self):
        self.models = None
        self.launch_count = 0

    def set_models(self, mb):
        self.models = mb

    def _run(self, rec, v, flags, affine):
        from qdsim import FLAG_CARRY_ROWS, FLAG_LATCH_EXACT, FLAG_WHITE_ON_OUTPUT
        from oracle import scan as oscan
        from util import oracle_model, oracle_scan
        m = oracle_model(self.models, int(rec["env_id"]), flags)
        s = oracle_scan(rec, self.models.n_volt, flags)
        kw = dict(latch_compare="exact" if flags & FLAG_LATCH_EXACT else "rounded",
                  carry_rows=bool(flags & FLAG_CARRY_ROWS), white_on="output" if flags & FLAG_WHITE_ON_OUTPUT else "input")
        self.launch_count += 1
        return oscan.simulate_scan(m, s, **kw) if affine else oscan.simulate_points(m, v, s, **kw)

    def scan_one_host(self, scan, n_type=3, flags=0):
        return self.scan_open_host(scan, n_type=n_type, flags=flags)

    def scan_open_host(self, scans, n_type=1, flags=0, want_z=True, z_out=None, n_out=None):
        zs, ns = [], []
        for rec in scans:
            z, n = self._run(rec, None, flags, True)
            zs.append(z.reshape(-1))
            ns.append(n.reshape(-1, n.shape[-1]))
        return np.concatenate(zs).astype(np.float32), np.concatenate(ns)

    def points_open_host(self, scan, v, n_type=3, flags=0, want_z=True):
        rec = np.asarray(scan).reshape(-1)[0]
        z, n = self._run(rec, v, flags, False)
        return (z.astype(np.float32) if want_z else None), n


def install(monkeypatch):
    """Returns (qarray_base_class module, env module) of the reference, bound to our drop-ins + the oracle engine."""
    for p in (ROOT, os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    if "jax" not in sys.modules:
        jax = types.ModuleType("jax")
        jnp = types.ModuleType("jax.numpy")
        jnp.full, jnp.array, jnp.ndarray = np.full, np.array, np.ndarray
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
    if "gymnasium" not in sys.modules:
        gym = types.ModuleType("gymnasium")

        class Env:
            def reset(self, seed=None, options=None):
                return None

        class _Space:
            def __init__(self, *a, **k):
                self.args, self.kwargs = a, k

        spaces = types.ModuleType("gymnasium.spaces")
        spaces.Dict = spaces.Box = spaces.Discrete = _Space
        gym.Env, gym.spaces = Env, spaces
        monkeypatch.setitem(sys.modules, "gymnasium", gym)
        monkeypatch.setitem(sys.modules, "gymnasium.spaces", spaces)
    monkeypatch.syspath_prepend(REF)
    monkeypatch.syspath_prepend(PKG)
    for name in [m for m in sys.modules if m.startswith(("qadapt", "qarray_latched"))]:
        monkeypatch.delitem(sys.modules, name)
    for name, path in (("qadapt", REF + "/qadapt"), ("qadapt.environment", REF + "/qadapt/environment"),
                       ("qadapt.capacitance_model", REF + "/qadapt/capacitance_model")):
        mod = types.ModuleType(name)
        mod.__path__ = [path]
        if name == "qadapt.capacitance_model":
            mod.CapacitancePredictionModel = object      # the CNN is only built for update_method kalman / direct
        monkeypatch.setitem(sys.modules, name, mod)
    import importlib
    from qdsim import runtime
    eng = OracleEngine()
    owner = {}

    def engine_for(model, device=None):
        key = (id(model), model._version)
        if owner.get("k") != key:
            eng.set_models(model._model_batch())
            owner["k"] = key
        return eng

    monkeypatch.setattr(runtime, "engine_for", engine_for)
    import qarray.charge_sensed as cs
    importlib.import_module("qarray_latched.DotArrays.TunnelCoupledChargeSensed")
    tc = sys.modules["qarray_latched.DotArrays.TunnelCoupledChargeSensed"]     # the module, not the class it exports
    monkeypatch.setattr(cs, "engine_for", engine_for)
    monkeypatch.setattr(tc, "engine_for", engine_for)
    base = importlib.import_module("qadapt.environment.qarray_base_class")
    env = importlib.import_module("qadapt.environment.env")
    return base, env, eng
