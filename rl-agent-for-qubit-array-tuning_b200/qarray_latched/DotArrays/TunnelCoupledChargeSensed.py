"""``TunnelCoupledChargeSensed`` -- drop-in for the reference's vendored class
(src/qarray_latched/DotArrays/TunnelCoupledChargeSensed.py:28-471) as constructed at
src/qadapt/environment/qarray_base_class.py:817-838 and called at :163 (``charge_sensor_open(vg_flat, vb)``).

Same constructor keywords, attributes, return conventions and errors.  The per-pixel work -- continuous relaxation,
4^N candidate enumeration with stable top-``num_charge_states`` selection, tunnel-coupled Hamiltonian, ground eigenvector,
occupation expectation, latching, sensor and noise (qarray_latched/DotArrays/ground_state.py:24-166) -- runs in the
QD_ALG_TUNNEL kernels of libqdsim.so."""
from __future__ import annotations

import numpy as np

from qarray.latching_models import LatchingBaseModel
from qarray.noise_models import BaseNoiseModel
from qdsim import FLAG_LATCH, FLAG_NOISE, N_F64, PARAMS_DTYPE, QD_MAX_DOTS, QD_MAX_SENSORS, QD_MAX_VOLT, maxwell
from qdsim.composer import GateVoltageComposer
from qdsim.engine import K_B, ModelBatch, new_scans
from qdsim.runtime import engine_for, fresh_seed

from .barrier_voltage_model import BarrierVoltageModel

_RECORD_FIELDS = {"T", "tc", "noise_model", "latching_model", "barrier_model", "num_charge_states",
                  "charge_state_batch_size", "voltage_capacitance_model"}


def _positive(a, name):
    if a is None:
        return None
    a = np.array(a, dtype=np.float64)
    if (a < 0).any():
        raise ValueError(f"{name} must be positive valued")
    return a


class TunnelCoupledChargeSensed:
    def __init__(self, Cdd, Cgd, Cds, Cgs, algorithm: str | None = "brute-force", implementation: str | None = "jax",
                 use_sparse: bool | None = False, num_charge_states: int | None = None,
                 charge_state_batch_size: int | None = None, tunneling_convention: str = "fermionic_negative",
                 threshold: float | str = 1.0, max_charge_carriers: int | None = None, polish: bool = True,
                 batch_size: int | None = None, charge_carrier: str = "h", T: float = 0.0, n_peak: int = 5,
                 coulomb_peak_width: float = 0.1, noise_model: BaseNoiseModel | None = None,
                 latching_model: LatchingBaseModel | None = None, tc: float = 0,
                 voltage_capacitance_model=None, constant_charge_shift: int | None = None,
                 Cbd=None, Cbg=None, Cbs=None, Cbb=None, barrier_model: BarrierVoltageModel | None = None,
                 device: int | None = None):
        object.__setattr__(self, "_version", 0)
        self.algorithm, self.implementation = algorithm, implementation
        self.use_sparse = use_sparse
        self.num_charge_states = num_charge_states
        self.charge_state_batch_size = charge_state_batch_size
        self.tunneling_convention = tunneling_convention
        self.threshold, self.max_charge_carriers, self.polish, self.batch_size = threshold, max_charge_carriers, polish, batch_size
        self.charge_carrier = charge_carrier
        self.T = float(T)
        self.n_peak = n_peak
        self.coulomb_peak_width = coulomb_peak_width
        self.noise_model = noise_model if noise_model is not None else BaseNoiseModel()
        self.latching_model = latching_model if latching_model is not None else LatchingBaseModel()
        self.tc = tc
        self.voltage_capacitance_model = voltage_capacitance_model
        self.constant_charge_shift = constant_charge_shift
        self.barrier_model = barrier_model
        self.device = device
        if n_peak != 5:
            raise NotImplementedError("the sensor kernel evaluates n_peak = 5 (the reference's value)")
        if constant_charge_shift is not None:
            raise NotImplementedError("constant_charge_shift is None at every reference call site")
        self.update_capacitance_matrices(Cdd, Cgd, Cds, Cgs, Cbd, Cbg, Cbs, Cbb)

        self.gate_voltage_composer = GateVoltageComposer(n_gate=self.n_gate, n_dot=self.n_dot, n_sensor=self.n_sensor)
        self.gate_voltage_composer.virtual_gate_matrix = maxwell.optimal_vgm(
            self.cdd_inv_full, self.cgd_full[:, :self.n_gate], electrons=(charge_carrier == "electrons"))
        self.gate_voltage_composer.virtual_gate_origin = np.zeros(self.n_gate)
        if self.barrier_model is not None:
            self.barrier_model.validate_dimensions(self.n_gate, self.n_dot, self.n_sensor)

    def __setattr__(self, name, value):
        if name in _RECORD_FIELDS and "_version" in self.__dict__:
            object.__setattr__(self, "_version", self._version + 1)
        object.__setattr__(self, name, value)

    def update_capacitance_matrices(self, Cdd, Cgd, Cds, Cgs, Cbd=None, Cbg=None, Cbs=None, Cbb=None):
        self.Cdd, self.Cgd = _positive(Cdd, "Cdd"), _positive(Cgd, "Cgd")
        self.Cds, self.Cgs = _positive(Cds, "Cds"), _positive(Cgs, "Cgs")
        self.Cbd, self.Cbg = _positive(Cbd, "Cbd"), _positive(Cbg, "Cbg")
        self.Cbs, self.Cbb = _positive(Cbs, "Cbs"), _positive(Cbb, "Cbb")
        self.n_dot = self.Cdd.shape[0]
        self.n_sensor = self.Cds.shape[0]
        self.n_gate = self.Cgd.shape[1]
        self.n_barrier = self.Cbd.shape[1] if self.Cbd is not None else 0
        self._assert_shape()
        if not 1 <= self.n_sensor <= QD_MAX_SENSORS:
            raise NotImplementedError(f"libqdsim simulates 1..{QD_MAX_SENSORS} charge sensors, got {self.n_sensor}")
        if self.n_gate + self.n_barrier > QD_MAX_VOLT:
            raise ValueError(f"libqdsim takes at most {QD_MAX_VOLT} gate and barrier voltages, got n_gate + n_barrier = "
                             f"{self.n_gate} + {self.n_barrier}")
        cdd_nm, cgd_nm = maxwell.embed_sensor(self.Cdd, self.Cgd, self.Cds, self.Cgs, self.Cbd, self.Cbs)
        self.cdd_full, self.cdd_inv_full, self.cgd_full = maxwell.maxwell(cdd_nm, cgd_nm)
        self.cdd, self.cdd_inv, self.cgd = maxwell.maxwell(self.Cdd, self.Cgd)
        self.cbd = self.cbg = self.cbs = self.cbb = None
        self.cgs, self.cds = self.Cgs, self.Cds
        object.__setattr__(self, "_version", self._version + 1)

    # ---- device constants ----------------------------------------------------------------------------------
    def _model_batch(self) -> ModelBatch:
        vcm = self.voltage_capacitance_model
        if vcm is not None:
            # the linear model of create_linear_capacitance_model as the facade builds it (qarray_base_class.py:846-851:
            # cdd_0 = model.cdd_full, cgd_0 = model.cgd_full): two scalars per env, applied per pixel in the kernel
            if getattr(vcm, "kind", None) not in ("linear", "quadratic", "sigmoid"):
                raise NotImplementedError("voltage-dependent capacitance models: linear, quadratic and sigmoid (the "
                                          "reference's factories) are wired into the kernel; build one with "
                                          "qarray_latched.DotArrays.voltage_dependent_capacitance.create_*_capacitance_model")
            if not (np.allclose(vcm.cdd_0, self.cdd_full, rtol=1e-12, atol=0) and
                    np.allclose(vcm.cgd_0, self.cgd_full, rtol=1e-12, atol=0)):
                raise NotImplementedError("the capacitance model must be built on the model's own cdd_full / "
                                          "cgd_full (as qarray_base_class.py:846-851 does)")
        if not isinstance(self.num_charge_states, int):
            raise NotImplementedError("num_charge_states=None builds a dense 5^N x 5^N Hamiltonian per pixel in the "
                                      "reference (infeasible beyond N~3, SURVEY.md section 8a); pass an int (32)")
        if self.use_sparse:
            raise NotImplementedError("use_sparse is False in the shipped configuration (qarray_config.yaml:128)")
        n, d = self.n_dot, self.n_dot + self.n_sensor
        params = np.zeros(1, dtype=PARAMS_DTYPE)
        params["kT"] = K_B * self.T                       # read but unused by the reference's tunnel path (ground_state.py:48)
        for k, v in self.noise_model._kernel_params().items():
            params[k] = v
        lm = self.latching_model
        if getattr(lm, "exists", False):
            params["latching"] = 1
            params["p_leads"][0, :n] = lm.p_leads
            pin = np.zeros((QD_MAX_DOTS, QD_MAX_DOTS))
            pin[:n, :n] = lm.p_inter
            params["p_inter"][0] = pin.reshape(-1)
        use_barriers = self.barrier_model is not None and self.n_barrier > 0
        if use_barriers:
            params["tc_base"] = self.barrier_model.tc_base
            params["alpha"][0, :self.n_barrier] = np.asarray(self.barrier_model.alpha, dtype=np.float64)
        else:
            params["tc_base"] = self.tc                   # constant nearest-neighbour coupling (ground_state.py:92-101)
        if vcm is not None:
            params["vc_alpha"], params["vc_beta"] = vcm.alpha, vcm.beta
            params["vc_kind"] = {"linear": 0, "quadratic": 1, "sigmoid": 2}[vcm.kind]
            params["vc_vchar"] = getattr(vcm, "v_char", 1.0)
        cbg = None
        if use_barriers:
            cbg = np.zeros((1, self.n_barrier, self.n_gate)) if self.Cbg is None else self.Cbg[None]
        return ModelBatch(algorithm="tunnel", n_gate=self.n_gate, cdd_inv_gs=self.cdd_inv_full[None, :n, :n].copy(),
                          cdd_gs=None, cdd_inv_full=self.cdd_inv_full[None], cgd_full=self.cgd_full[None],
                          params=params, cbg=cbg, num_charge_states=self.num_charge_states,
                          charge_state_batch_size=self.charge_state_batch_size or 0)

    def _flags(self, sensor: bool) -> int:
        f = FLAG_LATCH if getattr(self.latching_model, "exists", False) else 0
        if sensor and self.noise_model._kernel_params():
            f |= FLAG_NOISE
        return f

    def _points(self, vg, vb, sensor: bool):
        vg = np.asarray(vg, dtype=np.float64)
        if vg.shape[-1] != self.n_gate:
            raise ValueError(f"The shape of vg is in correct it should be of shape (..., n_gate) = (...,{self.n_gate})")
        if self.n_barrier > 0:
            if vb is None or self.barrier_model is None:
                raise ValueError("barrier voltages vb and a barrier_model are required for a model built with Cbd/Cbg/Cbs")
            vb = np.asarray(vb, dtype=np.float64).reshape(*vg.shape[:-1], -1)
            v = np.concatenate([vg, vb], axis=-1)
        else:
            v = vg
        lead = v.shape[:-1]
        nx = lead[-1] if lead else 1
        ny = int(np.prod(lead[:-1])) if len(lead) > 1 else 1
        s = new_scans(1)
        s["peak_width"] = float(self.coulomb_peak_width)
        s["seed"] = fresh_seed()
        z, n = engine_for(self, self.device).points_open_host(
            s, v.reshape(ny, nx, v.shape[-1]), n_type=N_F64, flags=self._flags(sensor), want_z=sensor)
        n = n.reshape(*lead, self.n_dot)
        if sensor:
            return z.astype(np.float64).reshape(*lead, self.n_sensor), n
        return n

    # ---- reference API -------------------------------------------------------------------------------------
    def ground_state_open(self, vg, vb=None):
        return self._points(vg, vb, sensor=False)

    def charge_sensor_open(self, vg, vb=None):
        return self._points(vg, vb, sensor=True)

    def do1d_open(self, gate, min, max, points):  # noqa: A002
        return self.charge_sensor_open(self.gate_voltage_composer.do1d(gate, min, max, points))

    def do2d_open(self, x_gate, x_min, x_max, x_points, y_gate, y_min, y_max, y_points):
        return self.charge_sensor_open(
            self.gate_voltage_composer.do2d(x_gate, x_min, x_max, x_points, y_gate, y_min, y_max, y_points))

    def optimal_Vg(self, n_charges, rcond: float = 1e-3):
        n_charges = np.asarray(n_charges, dtype=np.float64)
        assert n_charges.shape == (self.n_dot + self.n_sensor,), "The n_charge vector must be of shape (n_dot + n_sensor)"
        return maxwell.optimal_vg(self.cdd_inv_full, self.cgd_full[:, :self.n_gate], n_charges, rcond)

    def compute_optimal_virtual_gate_matrix(self):
        vgm = maxwell.optimal_vgm(self.cdd_inv_full, self.cgd_full[:, :self.n_gate],
                                  electrons=(self.charge_carrier == "electrons"))
        self.gate_voltage_composer.virtual_gate_matrix = vgm
        return vgm

    def ground_state_closed(self, vg, n_charge):
        raise NotImplementedError("closed arrays are dead code in the reference's fork (undefined _ground_state_closed)")

    charge_sensor_closed = do1d_closed = do2d_closed = ground_state_closed

    def _assert_shape(self):
        assert self.Cgd.shape[0] == self.n_dot, f"Cgd must be of shape (n_dot, n_gate) = ({self.n_dot}, {self.n_gate})"
        assert self.Cds.shape == (self.n_sensor, self.n_dot), "Cds must be of shape (n_sensor, n_dot)"
        assert self.Cgs.shape == (self.n_sensor, self.n_gate), "Cgs must be of shape (n_sensor, n_gate)"
