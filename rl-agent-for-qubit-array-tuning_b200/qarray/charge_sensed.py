"""``ChargeSensedDotArray`` -- drop-in for qarray==1.6.0's class of the same name as the reference constructs and calls it
(src/qadapt/environment/qarray_base_class.py:744-756 constructor kwargs; :128-137 ``do2d_open``; :1247, 1272
``optimal_Vg``; attribute reads listed in SURVEY.md section 8b).  Same names, argument meaning, return conventions and
error behaviour; the arithmetic runs in the sm_100a kernels of libqdsim.so (no CPU path)."""
from __future__ import annotations

import numpy as np

from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_THERMAL, N_F64, N_U8, QD_MAX_SENSORS, QD_MAX_VOLT, maxwell
from qdsim._lib import CLOSED_MAX_CHARGE
from qdsim.composer import GateVoltageComposer
from qdsim.engine import ModelBatch, new_scans
from qdsim.runtime import engine_for, fresh_seed

from .latching_models import LatchingBaseModel
from .noise_models import BaseNoiseModel

# algorithm x implementation table of the reference (src/qarray_latched/DotArrays/_helper_functions.py:202-210).
# Every implementation name maps onto the CUDA kernels.
_COMBINATIONS = {"default": ["rust", "python", "jax"], "thresholded": ["rust", "python"], "brute_force": ["jax", "python"]}
_RECORD_FIELDS = {"T", "threshold", "max_charge_carriers", "algorithm", "noise_model", "latching_model"}


def _positive_matrix(a, name):
    a = np.array(a, dtype=np.float64)
    if a.ndim != 2:
        raise ValueError(f"{name} must be a matrix")
    if (a < 0).any():
        raise ValueError(f"{name} must be positive valued")
    return a


class ChargeSensedDotArray:
    def __init__(self, Cdd, Cgd, Cds, Cgs, algorithm: str = "default", implementation: str = "rust",
                 threshold: float | str = 1.0, max_charge_carriers: int | None = None, polish: bool = True,
                 batch_size: int | None = None, charge_carrier: str = "h", T: float = 0.0, n_peak: int = 5,
                 coulomb_peak_width: float = 0.1, noise_model: BaseNoiseModel | None = None,
                 latching_model: LatchingBaseModel | None = None, device: int | None = None):
        object.__setattr__(self, "_version", 0)
        self.Cdd = _positive_matrix(Cdd, "Cdd")
        self.Cgd = _positive_matrix(Cgd, "Cgd")
        self.Cds = _positive_matrix(Cds, "Cds")
        self.Cgs = _positive_matrix(Cgs, "Cgs")
        self.n_dot = self.Cdd.shape[0]
        self.n_sensor = self.Cds.shape[0]
        self.n_gate = self.Cgd.shape[1]
        self._assert_shape()

        algorithm = algorithm.lower()
        assert algorithm in _COMBINATIONS, f"Algorithm {algorithm} not supported"
        assert implementation.lower() in _COMBINATIONS[algorithm], \
            f"Implementation {implementation} not supported for algorithm {algorithm}"
        if algorithm == "brute_force":
            assert max_charge_carriers is not None, "The maximum number of charge carriers must be specified"
        if n_peak != 5:
            raise NotImplementedError("the sensor kernel evaluates n_peak = 5 (the reference's value)")
        if not 1 <= self.n_sensor <= QD_MAX_SENSORS:
            raise NotImplementedError(f"libqdsim simulates 1..{QD_MAX_SENSORS} charge sensors, got {self.n_sensor}")
        if self.n_gate > QD_MAX_VOLT:
            raise ValueError(f"libqdsim takes at most {QD_MAX_VOLT} gate voltages, got n_gate = {self.n_gate}")
        self.algorithm = algorithm
        self.implementation = implementation
        self.threshold = 1.0 if threshold == "auto" else float(threshold)
        self.max_charge_carriers = max_charge_carriers
        self.polish = polish
        self.batch_size = batch_size
        self.charge_carrier = charge_carrier
        self.T = float(T)
        self.n_peak = n_peak
        self.coulomb_peak_width = coulomb_peak_width
        self.noise_model = noise_model if noise_model is not None else BaseNoiseModel()
        self.latching_model = latching_model if latching_model is not None else LatchingBaseModel()
        self.device = device

        # Maxwell matrices: dot-only set for the ground state, full [dots, sensor] set for the sensor
        self.cdd, self.cdd_inv, self.cgd = maxwell.maxwell(self.Cdd, self.Cgd)
        cdd_nm, cgd_nm = maxwell.embed_sensor(self.Cdd, self.Cgd, self.Cds, self.Cgs)
        self.cdd_full, self.cdd_inv_full, self.cgd_full = maxwell.maxwell(cdd_nm, cgd_nm)
        self.cgs, self.cds = self.Cgs, self.Cds

        self.gate_voltage_composer = GateVoltageComposer(n_gate=self.n_gate, n_dot=self.n_dot, n_sensor=self.n_sensor)
        self.gate_voltage_composer.virtual_gate_matrix = maxwell.optimal_vgm(
            self.cdd_inv_full, self.cgd_full, electrons=(charge_carrier == "electrons"))
        self.gate_voltage_composer.virtual_gate_origin = np.zeros(self.n_gate)

    def __setattr__(self, name, value):
        if name in _RECORD_FIELDS and "_version" in self.__dict__:
            object.__setattr__(self, "_version", self._version + 1)     # device-resident constants are stale
        object.__setattr__(self, name, value)

    # ---- device constants ----------------------------------------------------------------------------------
    def _model_batch(self) -> ModelBatch:
        noise = self.noise_model._kernel_params()
        lm = self.latching_model
        latch = getattr(lm, "exists", False)
        return ModelBatch.from_capacitances(
            self.Cdd, self.Cgd, self.Cds, self.Cgs, algorithm=self.algorithm, T=self.T, threshold=self.threshold,
            max_charge_carriers=self.max_charge_carriers if self.max_charge_carriers is not None else 0,
            p_leads=lm.p_leads if latch else None, p_inter=lm.p_inter if latch else None, **noise)

    def _flags(self, sensor: bool) -> int:
        f = 0
        if getattr(self.latching_model, "exists", False):
            f |= FLAG_LATCH
        if self.T > 0:
            f |= FLAG_THERMAL
        if sensor and self.noise_model._kernel_params():
            f |= FLAG_NOISE
        return f

    def _scan_record(self):
        s = new_scans(1)
        s["peak_width"] = float(self.coulomb_peak_width)
        s["seed"] = fresh_seed()
        return s

    # ---- reference API -------------------------------------------------------------------------------------
    def do2d_open(self, x_gate, x_min, x_max, x_points, y_gate, y_min, y_max, y_points):
        """2-d sweep, open array.  Returns ``(z (y, x, n_sensor), n (y, x, n_dot))``."""
        # One persistent descriptor per model object; a sweep of PHYSICAL gates (what the facade's non-barrier mode calls,
        # qarray_base_class.py:128-137) does not depend on the virtual gate matrix, so its affine form is cached by
        # arguments -- this call is latency-bound (BASELINE config 1), every microsecond of host work shows.
        d = self.__dict__
        s = d.get("_scan1")
        if s is None:
            s = d["_scan1"] = new_scans(1)
            d["_scan1_views"] = (s["v0"][0], s["dx"][0], s["dy"][0])
            d["_affine_cache"] = {}
        key = (x_gate, x_min, x_max, x_points, y_gate, y_min, y_max, y_points)
        aff = d["_affine_cache"].get(key)
        if aff is None:
            aff = self.gate_voltage_composer.affine2d(x_gate, x_min, x_max, x_points, y_gate, y_min, y_max, y_points)
            physical = all(isinstance(g, (int, np.integer)) or (isinstance(g, str) and not g.startswith("v"))
                           for g in (x_gate, y_gate))
            if physical:
                if len(d["_affine_cache"]) > 64:
                    d["_affine_cache"].clear()
                d["_affine_cache"][key] = aff
        if d.get("_scan1_aff") is not aff:          # (a cached sweep of physical gates: the descriptor already holds it)
            ng = self.n_gate
            v0v, dxv, dyv = d["_scan1_views"]
            v0v[:ng], dxv[:ng], dyv[:ng] = aff
            d["_scan1_aff"] = aff
        fl = d.get("_flags_cache")
        if fl is None or fl[0] != self._version:
            fl = d["_flags_cache"] = (self._version, self._flags(True))
        flags = fl[1]
        pw = float(self.coulomb_peak_width)
        last = d.get("_scan1_last")
        if last != (pw, x_points, y_points):
            s["peak_width"] = pw
            s["nx"], s["ny"] = x_points, y_points
            d["_scan1_last"] = (pw, x_points, y_points)
        if flags:                                   # the seed only feeds latching / noise draws
            s["seed"] = fresh_seed()
        # hard argmin (T = 0): the occupations are small integers -- fetch them as one byte per dot (an eighth of the bytes
        # the kernel has to push over PCIe) and widen here; thermal averages come back as float64
        z, n = engine_for(self, self.device).scan_one_host(s, N_F64 if flags & FLAG_THERMAL else N_U8, flags,
                                                           x_points * y_points)
        return (z.astype(np.float64).reshape(y_points, x_points, self.n_sensor),
                n.astype(np.float64).reshape(y_points, x_points, self.n_dot))

    def do1d_open(self, gate, min, max, points):  # noqa: A002
        """1-d sweep, open array.  Returns ``(z (points, n_sensor), n (points, n_dot))``."""
        return self.charge_sensor_open(self.gate_voltage_composer.do1d(gate, min, max, points))

    def _points(self, vg, sensor: bool):
        vg = np.asarray(vg, dtype=np.float64)
        if vg.shape[-1] != self.n_gate:
            raise ValueError(f"The shape of vg is in correct it should be of shape (..., n_gate) = (...,{self.n_gate})")
        lead = vg.shape[:-1]
        nx = lead[-1] if lead else 1
        ny = int(np.prod(lead[:-1])) if len(lead) > 1 else 1
        z, n = engine_for(self, self.device).points_open_host(
            self._scan_record(), vg.reshape(ny, nx, self.n_gate), n_type=N_F64, flags=self._flags(sensor), want_z=sensor)
        n = n.reshape(*lead, self.n_dot)
        if sensor:
            return z.astype(np.float64).reshape(*lead, self.n_sensor), n
        return n

    def ground_state_open(self, vg):
        """Ground-state occupations, (..., n_gate) -> (..., n_dot)."""
        return self._points(vg, sensor=False)

    def charge_sensor_open(self, vg):
        """Sensor signal and occupations, (..., n_gate) -> ((..., n_sensor), (..., n_dot))."""
        return self._points(vg, sensor=True)

    def optimal_Vg(self, n_charges, rcond: float = 1e-3):
        n_charges = np.asarray(n_charges, dtype=np.float64)
        assert n_charges.shape == (self.n_dot + self.n_sensor,), "The n_charge vector must be of shape (n_dot + n_sensor)"
        return maxwell.optimal_vg(self.cdd_inv_full, self.cgd_full, n_charges, rcond)

    def compute_optimal_virtual_gate_matrix(self):
        vgm = maxwell.optimal_vgm(self.cdd_inv_full, self.cgd_full, electrons=(self.charge_carrier == "electrons"))
        self.gate_voltage_composer.virtual_gate_matrix = vgm
        return vgm

    # ---- closed arrays: n_charges carriers in total on the dots ----------------------------------------------
    def _n_charge(self, n_charges) -> int:
        """The total charge as an int; NotImplementedError for ``thresholded``, ValueError for a non-integer or an
        out-of-range value (0..251 for ``default``, 0..15 for ``brute_force``)."""
        if self.algorithm not in CLOSED_MAX_CHARGE:
            raise NotImplementedError(f"closed arrays: the {self.algorithm} algorithm is not supported (its candidate set "
                                      "can be empty under the sum constraint); use default or brute_force")
        if isinstance(n_charges, (bool, np.bool_)) or not isinstance(n_charges, (int, np.integer, float, np.floating)) \
                or not float(n_charges).is_integer():
            raise ValueError(f"n_charges must be an integer, got {n_charges!r}")
        q = int(n_charges)
        if not 0 <= q <= CLOSED_MAX_CHARGE[self.algorithm]:
            raise ValueError(f"n_charges must be in 0..{CLOSED_MAX_CHARGE[self.algorithm]} for {self.algorithm}, got {q}")
        return q

    def _points_closed(self, vg, n_charges, sensor: bool):
        q = self._n_charge(n_charges)
        vg = np.asarray(vg, dtype=np.float64)
        if vg.shape[-1] != self.n_gate:
            raise ValueError(f"The shape of vg is in correct it should be of shape (..., n_gate) = (...,{self.n_gate})")
        lead = vg.shape[:-1]
        nx = lead[-1] if lead else 1
        ny = int(np.prod(lead[:-1])) if len(lead) > 1 else 1
        z, n = engine_for(self, self.device).points_closed_host(
            self._scan_record(), q, vg.reshape(ny, nx, self.n_gate), n_type=N_F64, flags=self._flags(sensor),
            want_z=sensor)
        n = n.reshape(*lead, self.n_dot)
        if sensor:
            return z.astype(np.float64).reshape(*lead, self.n_sensor), n
        return n

    def ground_state_closed(self, vg, n_charges):
        """Ground-state occupations of the closed array, (..., n_gate) -> (..., n_dot), summing to ``n_charges``."""
        return self._points_closed(vg, n_charges, sensor=False)

    def charge_sensor_closed(self, vg, n_charges):
        """Sensor signal and occupations of the closed array, (..., n_gate) -> ((..., n_sensor), (..., n_dot))."""
        return self._points_closed(vg, n_charges, sensor=True)

    def do1d_closed(self, gate, min, max, points, n_charges):  # noqa: A002
        """1-d sweep, closed array.  Returns ``(z (points, n_sensor), n (points, n_dot))``."""
        q = self._n_charge(n_charges)
        return self.charge_sensor_closed(self.gate_voltage_composer.do1d(gate, min, max, points), q)

    def do2d_closed(self, x_gate, x_min, x_max, x_points, y_gate, y_min, y_max, y_points, n_charges):
        """2-d sweep, closed array.  Returns ``(z (y, x, n_sensor), n (y, x, n_dot))``."""
        q = self._n_charge(n_charges)
        s = self._scan_record()
        v0, dx, dy = self.gate_voltage_composer.affine2d(x_gate, x_min, x_max, x_points, y_gate, y_min, y_max, y_points)
        s["v0"][0, :self.n_gate], s["dx"][0, :self.n_gate], s["dy"][0, :self.n_gate] = v0, dx, dy
        s["nx"], s["ny"] = x_points, y_points
        flags = self._flags(True)
        z, n = engine_for(self, self.device).scan_closed_host(s, q, N_F64 if flags & FLAG_THERMAL else N_U8, flags)
        return (z.astype(np.float64).reshape(y_points, x_points, self.n_sensor),
                n.astype(np.float64).reshape(y_points, x_points, self.n_dot))

    def _assert_shape(self):
        assert self.Cdd.shape == (self.n_dot, self.n_dot), "Cdd must be square"
        assert self.Cgd.shape[0] == self.n_dot, f"Cgd must be of shape (n_dot, n_gate) = ({self.n_dot}, {self.n_gate})"
        assert self.Cds.shape == (self.n_sensor, self.n_dot), "Cds must be of shape (n_sensor, n_dot)"
        assert self.Cgs.shape == (self.n_sensor, self.n_gate), "Cgs must be of shape (n_sensor, n_gate)"
