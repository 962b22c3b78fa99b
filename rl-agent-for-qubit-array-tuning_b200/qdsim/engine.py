"""Host engine: one ``Engine`` per (process, GPU) wrapping a ``qd_ctx`` of libqdsim.so.

This is the batched entry point (thousands of independent env.step calls per launch).  The reference-compatible
single-device classes (``qarray.ChargeSensedDotArray`` ...) sit on top of it.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib, maxwell
from ._lib import (ALGORITHMS, FLAG_CARRY_ROWS, FLAG_LATCH, FLAG_LATCH_EXACT, FLAG_NOISE, FLAG_PINK, FLAG_RADIAL,  # noqa: F401
                   FLAG_THERMAL, FLAG_WHITE_ON_OUTPUT, N_DTYPES, N_F32, N_F64, N_NONE, N_U8, PARAMS_DTYPE,
                   QD_MAX_DOTS, QD_MAX_SENSORS, QD_MAX_VOLT, SCAN_DTYPE, Z_DTYPES, Z_F16, Z_F32, Z_U8, QdError)

K_B = 8.617333262145e-5  # eV/K (src/qarray_latched/DotArrays/_helper_functions.py:213-214)


@dataclass
class ModelBatch:
    """Per-env constants of ``n_env`` devices in Maxwell form (fp64), as uploaded by ``qd_set_models``."""
    algorithm: str
    n_gate: int
    cdd_inv_gs: np.ndarray            # (E, N, N)
    cdd_gs: np.ndarray | None         # (E, N, N)
    cdd_inv_full: np.ndarray          # (E, D, D)
    cgd_full: np.ndarray              # (E, D, NV)
    params: np.ndarray                # (E,) PARAMS_DTYPE
    cbg: np.ndarray | None = None     # (E, B, G)
    num_charge_states: int = 32
    charge_state_batch_size: int = 1000

    @property
    def n_env(self) -> int:
        return self.cdd_inv_gs.shape[0]

    @property
    def n_dot(self) -> int:
        return self.cdd_inv_gs.shape[-1]

    @property
    def n_volt(self) -> int:
        return self.cgd_full.shape[-1]

    @property
    def n_sensor(self) -> int:
        return self.cdd_inv_full.shape[-1] - self.n_dot

    @classmethod
    def from_capacitances(cls, Cdd, Cgd, Cds, Cgs, algorithm: str = "default", T=0.0, threshold=1.0,
                          max_charge_carriers: int = 4, p_leads=None, p_inter=None, white_amp=0.0, tele_p01=0.0,
                          tele_p10=0.0, tele_amp=0.0) -> "ModelBatch":
        """Path A (``ChargeSensedDotArray``) batch from non-Maxwell matrices with a leading env axis.

        The dots' ground state uses the dot-only Maxwell matrices, the sensors the full [dots, sensors] system
        (SURVEY.md Appendix B.1; TunnelCoupledChargeSensed.py:117-130 keeps both sets).  ``Cds`` (S, N) and ``Cgs`` (S, G)
        hold one row per charge sensor, 1 <= S <= ``QD_MAX_SENSORS``.
        """
        Cdd = np.asarray(Cdd, dtype=np.float64)
        Cgd = np.asarray(Cgd, dtype=np.float64)
        Cds = np.asarray(Cds, dtype=np.float64)
        Cgs = np.asarray(Cgs, dtype=np.float64)
        if Cdd.ndim == 2:
            Cdd, Cgd, Cds, Cgs = Cdd[None], Cgd[None], Cds[None], Cgs[None]
        n_env, n_dot = Cdd.shape[0], Cdd.shape[-1]
        cdd, cdd_inv, _ = maxwell.maxwell(Cdd, Cgd)
        cdd_full_nm, cgd_full_nm = maxwell.embed_sensor(Cdd, Cgd, Cds, Cgs)
        _, cdd_inv_full, cgd_full = maxwell.maxwell(cdd_full_nm, cgd_full_nm)
        params = np.zeros(n_env, dtype=PARAMS_DTYPE)
        params["kT"] = K_B * np.broadcast_to(np.asarray(T, dtype=np.float64), (n_env,))
        params["threshold"] = threshold
        params["max_charge_carriers"] = max_charge_carriers
        params["white_amp"] = white_amp
        params["tele_p01"] = tele_p01
        params["tele_p10"] = tele_p10
        params["tele_amp"] = tele_amp
        if p_leads is not None:
            pl = np.broadcast_to(np.asarray(p_leads, dtype=np.float64), (n_env, n_dot))
            pi = np.broadcast_to(np.asarray(p_inter, dtype=np.float64), (n_env, n_dot, n_dot))
            params["latching"] = 1
            params["p_leads"][:, :n_dot] = pl
            pin = np.zeros((n_env, QD_MAX_DOTS, QD_MAX_DOTS))
            pin[:, :n_dot, :n_dot] = pi
            params["p_inter"] = pin.reshape(n_env, -1)
        return cls(algorithm=algorithm, n_gate=Cgd.shape[-1], cdd_inv_gs=cdd_inv, cdd_gs=cdd,
                   cdd_inv_full=cdd_inv_full, cgd_full=cgd_full, params=params)


def tunnel_model_batch(Cdd, Cgd, Cds, Cgs, Cbd, Cbg, Cbs, tc_base, alpha, p_leads=None, p_inter=None, white_amp=0.0,
                       tele_p01=0.0, tele_p10=0.0, tele_amp=0.0, num_charge_states: int = 32,
                       charge_state_batch_size: int = 1000) -> ModelBatch:
    """Path B (``TunnelCoupledChargeSensed`` with barriers) batch from non-Maxwell matrices with a leading env axis.
    ``Cds`` / ``Cgs`` / ``Cbs`` hold one row per charge sensor.  Barriers are voltage sources: extra columns of cgd (src/qarray_latched/DotArrays/_helper_functions.py:60-126); the
    ground state uses the dot block of the FULL inverse (ground_state.py:60-65)."""
    Cdd, Cgd, Cds, Cgs, Cbd, Cbg, Cbs = (np.asarray(a, dtype=np.float64) for a in (Cdd, Cgd, Cds, Cgs, Cbd, Cbg, Cbs))
    n_env, n_dot, n_barrier = Cdd.shape[0], Cdd.shape[-1], Cbd.shape[-1]
    cdd_nm, cgd_nm = maxwell.embed_sensor(Cdd, Cgd, Cds, Cgs, Cbd, Cbs)
    _, cdd_inv_full, cgd_full = maxwell.maxwell(cdd_nm, cgd_nm)
    params = np.zeros(n_env, dtype=PARAMS_DTYPE)
    params["white_amp"], params["tele_p01"], params["tele_p10"], params["tele_amp"] = white_amp, tele_p01, tele_p10, tele_amp
    params["tc_base"] = tc_base
    params["alpha"][:, :n_barrier] = np.broadcast_to(np.asarray(alpha, dtype=np.float64), (n_env, n_barrier))
    if p_leads is not None:
        params["latching"] = 1
        params["p_leads"][:, :n_dot] = np.broadcast_to(np.asarray(p_leads, dtype=np.float64), (n_env, n_dot))
        pin = np.zeros((n_env, QD_MAX_DOTS, QD_MAX_DOTS))
        pin[:, :n_dot, :n_dot] = np.broadcast_to(np.asarray(p_inter, dtype=np.float64), (n_env, n_dot, n_dot))
        params["p_inter"] = pin.reshape(n_env, -1)
    return ModelBatch(algorithm="tunnel", n_gate=Cgd.shape[-1], cdd_inv_gs=np.ascontiguousarray(cdd_inv_full[:, :n_dot, :n_dot]),
                      cdd_gs=None, cdd_inv_full=cdd_inv_full, cgd_full=cgd_full, params=params, cbg=Cbg,
                      num_charge_states=num_charge_states, charge_state_batch_size=charge_state_batch_size)


def new_scans(n: int) -> np.ndarray:
    """Zero-initialised array of ``n`` scan descriptors (``qd_scan``)."""
    s = np.zeros(n, dtype=SCAN_DTYPE)
    s["peak_width"] = 1.0
    return s


def _ptr(a) -> int | None:
    """Device / host pointer of a torch tensor, numpy array, int or None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()


class Engine:
    """One ``qd_ctx``: owns the device-resident model records of its env shard.  Not thread-safe."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        rc = self._lib.qd_create(int(device), C.byref(self._ctx))
        if rc != 0:
            raise QdError(rc, self._lib.qd_last_error(None).decode())
        self.device = int(device)
        self.models: ModelBatch | None = None
        self.n_sensor = 1                   # charge sensors of the uploaded model set: z is [pixels, n_sensor]
        self._one_bufs: dict = {}           # staging buffers of scan_one_host, by (pixels, n_type)

    # -- lifecycle -------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.qd_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise QdError(rc, self._lib.qd_last_error(self._ctx).decode())

    # -- models ----------------------------------------------------------------------------------------------
    def set_models(self, mb: ModelBatch):
        alg = ALGORITHMS.get(mb.algorithm.lower())
        if alg is None:
            raise AssertionError(f"Algorithm {mb.algorithm} not supported")
        d = mb.cdd_inv_full.shape[-1]
        desc = _lib.ModelDesc(mb.n_env, mb.n_dot, d - mb.n_dot, mb.n_volt, mb.n_gate, alg, mb.num_charge_states,
                              mb.charge_state_batch_size or 0)
        arrs = [np.ascontiguousarray(a, dtype=np.float64) if a is not None else None
                for a in (mb.cdd_inv_gs, mb.cdd_gs, mb.cdd_inv_full, mb.cgd_full, mb.cbg)]
        params = np.ascontiguousarray(mb.params, dtype=PARAMS_DTYPE)
        self._check(self._lib.qd_set_models(self._ctx, C.byref(desc), *[_ptr(a) for a in arrs], _ptr(params)))
        self.models = mb
        self.n_sensor = d - mb.n_dot

    def _z(self, pixels: int, z_out, want_z: bool, shape=None):
        """The host sensor buffer of a call: ``shape`` (default ``(pixels,)``) for one sensor, ``shape + (S,)`` otherwise."""
        if not want_z:
            return None
        s = self.n_sensor
        if z_out is None:
            shape = (pixels,) if shape is None else shape
            return np.empty(shape if s == 1 else shape + (s,), dtype=np.float32)
        assert z_out.dtype == np.float32 and z_out.size >= pixels * s and z_out.flags.c_contiguous, \
            "z_out must be a C-contiguous float32 array with at least pixels * n_sensor elements"
        return z_out

    # -- launches --------------------------------------------------------------------------------------------
    def scan_open(self, scans: np.ndarray, z_out, n_out=None, n_type: int = N_NONE, flags: int = 0, stream=None):
        """Asynchronous batched launch into DEVICE buffers (torch tensors or raw pointers).  ``z_out``: float32
        [pixels, n_sensor] (aligned to 4 n_sensor bytes for two or four sensors), ``n_out``: [pixels, N]."""
        assert scans.dtype == SCAN_DTYPE and scans.flags.c_contiguous
        self._check(self._lib.qd_scan_open(self._ctx, len(scans), _ptr(scans), _ptr(z_out), _ptr(n_out), n_type,
                                           flags, self._stream(stream)))

    @staticmethod
    def _stream(stream):
        return None if stream is None else (stream if isinstance(stream, int) else stream.cuda_stream)

    def scan_upload(self, scans: np.ndarray, stream=None):
        """Copy descriptors to the device once; ``scan_launch`` then re-runs them without any host traffic."""
        assert scans.dtype == SCAN_DTYPE and scans.flags.c_contiguous
        self._check(self._lib.qd_scan_upload(self._ctx, len(scans), _ptr(scans), self._stream(stream)))

    def scan_launch(self, z_out, n_out=None, n_type: int = N_NONE, flags: int = 0, stream=None):
        """One launch over the uploaded descriptors into DEVICE buffers laid out as in ``scan_open``."""
        self._check(self._lib.qd_scan_launch(self._ctx, _ptr(z_out), _ptr(n_out), n_type, flags, self._stream(stream)))

    def scan_open_host(self, scans: np.ndarray, n_type: int | None = None, flags: int = 0, want_z: bool = True,
                       z_out: np.ndarray | None = None, n_out: np.ndarray | None = None):
        """Synchronous launch returning host arrays ``(z float32 [pixels] (one sensor) or [pixels, S], n [pixels, N] or
        None)``.

        ``n_type`` defaults to what the model produces: uint8 for a hard argmin, float64 for non-integer occupations
        (tunnel-coupled models, ``FLAG_THERMAL``) -- the library refuses a uint8 charge map there instead of truncating.

        Large batches are pipelined inside the library (compute of one chunk overlaps the PCIe copy of the previous
        one); pass pinned ``z_out`` / ``n_out`` (e.g. ``torch.empty(..., pin_memory=True).numpy()``) for full copy speed.
        """
        assert scans.dtype == SCAN_DTYPE and scans.flags.c_contiguous
        if n_type is None:
            n_type = N_F64 if (self.models.algorithm.lower() == "tunnel" or flags & FLAG_THERMAL) else N_U8
        pixels = int((scans["pix_offset"] + scans["nx"].astype(np.int64) * scans["ny"]).max())
        z = self._z(pixels, z_out, want_z)
        n = None
        if n_type != N_NONE:
            n = n_out if n_out is not None else np.empty((pixels, self.models.n_dot), dtype=N_DTYPES[n_type])
        # the library copies pixels * N elements of n_type into n: a short, mistyped or strided buffer would be overrun
        assert n is None or (n.dtype == N_DTYPES[n_type] and n.size >= pixels * self.models.n_dot and n.flags.c_contiguous), \
            "n_out must be a C-contiguous array of the n_type's dtype with at least pixels * n_dot elements"
        self._check(self._lib.qd_scan_open_host(self._ctx, len(scans), _ptr(scans), _ptr(z), _ptr(n), n_type, flags))
        return z, n

    def scan_one_host(self, scan: np.ndarray, n_type: int = N_F64, flags: int = 0, pixels: int | None = None):
        """One scan window (a single ``do2d_open``), minimal host overhead: ``scan`` is a 1-element ``SCAN_DTYPE`` array with
        ``pix_offset == 0``; returns ``(z float32 [ny * nx] (one sensor) or [ny * nx, S], n [ny * nx, N])`` -- views of per-engine staging buffers that the
        NEXT call overwrites (the drop-in class widens them to fresh float64 arrays).  ``pixels`` = ny * nx if the caller has
        it at hand (reading it back from the record costs a microsecond).  The library takes its single-scan path:
        descriptor in the kernel parameters, outputs written straight into mapped pinned memory, one sync."""
        if pixels is None:
            pixels = int(scan["nx"][0]) * int(scan["ny"][0])
        key = (pixels, n_type)
        buf = self._one_bufs.get(key)
        if buf is None:
            if len(self._one_bufs) > 16:
                self._one_bufs.clear()
            z = self._z(pixels, None, True)
            n = np.empty((pixels, self.models.n_dot), dtype=N_DTYPES[n_type])
            buf = self._one_bufs[key] = (z, n, z.ctypes.data, n.ctypes.data, (self.models.n_dot, self.n_sensor))
        if buf[4] != (self.models.n_dot, self.n_sensor):
            self._one_bufs.clear()
            return self.scan_one_host(scan, n_type, flags, pixels)
        rc = self._lib.qd_scan_open_host(self._ctx, 1, scan.ctypes.data, buf[2], buf[3], n_type, flags)
        if rc != 0:
            self._check(rc)
        return buf[0], buf[1]

    def scan_obs_host(self, scans: np.ndarray, z_type: int = Z_U8, flags: int = 0, normalise: bool = True,
                      q_low: float = 0.5, q_high: float = 99.5, out: np.ndarray | None = None, want_stats: bool = False,
                      scans_per_env: int | None = None):
        """The observation of one batched env.step in HOST memory, compact element type (``Z_F32`` / ``Z_F16`` /
        ``Z_U8`` = rint(255 x)): scans -> per-env percentile normalisation on the device (env.py:471-509) -> typed
        copy-back, pipelined over chunks of envs.  ``scans``: env-major, ``scans_per_env`` (default N-1) equal-size
        descriptors per env.  One-sensor model sets only (the env's observation is one sensor's image).  Returns ``(image [n_scan, ny, nx] of the z_type's dtype, stats [n_env, 2] or None)``."""
        assert scans.dtype == SCAN_DTYPE and scans.flags.c_contiguous
        spe = scans_per_env or (self.models.n_dot - 1)
        ny, nx = int(scans["ny"][0]), int(scans["nx"][0])
        pixels = len(scans) * ny * nx
        if out is None:
            out = np.empty(pixels, dtype=Z_DTYPES[z_type])
        assert out.dtype == Z_DTYPES[z_type] and out.size >= pixels and out.flags.c_contiguous
        stats = np.empty((len(scans) // spe, 2), dtype=np.float64) if (want_stats and normalise) else None
        self._check(self._lib.qd_scan_obs_host(self._ctx, len(scans), _ptr(scans), spe, _ptr(out), z_type,
                                               1 if normalise else 0, q_low, q_high, _ptr(stats), flags))
        return out.reshape(-1)[:pixels].reshape(len(scans), ny, nx), stats

    def points_open_host(self, scan: np.ndarray, v: np.ndarray, n_type: int = N_F64, flags: int = 0,
                         want_z: bool = True):
        """Arbitrary voltage list ``v`` (ny, nx, n_volt) -> ``(z (ny, nx) (one sensor) or (ny, nx, S) float32,
        n (ny, nx, N))``."""
        v = np.ascontiguousarray(v, dtype=np.float64)
        ny, nx, nv = v.shape
        if nv != self.models.n_volt:
            raise ValueError(f"The shape of vg is in correct it should be of shape (..., n_gate) = (...,{self.models.n_volt})")
        scan = np.ascontiguousarray(scan, dtype=SCAN_DTYPE).reshape(1)
        z = self._z(ny * nx, None, want_z, (ny, nx))
        n = np.empty((ny, nx, self.models.n_dot), dtype=N_DTYPES[n_type]) if n_type != N_NONE else None
        self._check(self._lib.qd_points_open_host(self._ctx, _ptr(scan), ny, nx, _ptr(v), _ptr(z), _ptr(n), n_type,
                                                  flags))
        return z, n

    # -- closed arrays (fixed total charge per scan) -----------------------------------------------------------
    @staticmethod
    def _n_charge(n_charge, n_scan: int) -> np.ndarray:
        """Total charges as a contiguous int32 array of one entry per scan (a scalar applies to every scan)."""
        q = np.asarray(n_charge)
        if q.dtype.kind not in "iu" and not (q.dtype.kind == "f" and np.array_equal(q, np.round(q))):
            raise ValueError(f"n_charge must be integer-valued, got {n_charge!r}")
        return np.ascontiguousarray(np.broadcast_to(q.astype(np.int32), (n_scan,)))

    def scan_closed(self, scans: np.ndarray, n_charge, z_out, n_out=None, n_type: int = N_NONE, flags: int = 0,
                    stream=None):
        """``scan_open`` for closed arrays: scan i holds ``n_charge[i]`` carriers in total (a scalar: every scan)."""
        assert scans.dtype == SCAN_DTYPE and scans.flags.c_contiguous
        q = self._n_charge(n_charge, len(scans))
        self._check(self._lib.qd_scan_closed(self._ctx, len(scans), _ptr(scans), _ptr(q), _ptr(z_out), _ptr(n_out), n_type,
                                             flags, self._stream(stream)))

    def scan_closed_host(self, scans: np.ndarray, n_charge, n_type: int | None = None, flags: int = 0,
                         want_z: bool = True, z_out: np.ndarray | None = None, n_out: np.ndarray | None = None):
        """``scan_open_host`` for closed arrays: scan i holds ``n_charge[i]`` carriers in total (a scalar: every scan)."""
        assert scans.dtype == SCAN_DTYPE and scans.flags.c_contiguous
        q = self._n_charge(n_charge, len(scans))
        if n_type is None:
            n_type = N_F64 if flags & FLAG_THERMAL else N_U8
        pixels = int((scans["pix_offset"] + scans["nx"].astype(np.int64) * scans["ny"]).max())
        z = self._z(pixels, z_out, want_z)
        n = None
        if n_type != N_NONE:
            n = n_out if n_out is not None else np.empty((pixels, self.models.n_dot), dtype=N_DTYPES[n_type])
        assert n is None or (n.dtype == N_DTYPES[n_type] and n.size >= pixels * self.models.n_dot and n.flags.c_contiguous), \
            "n_out must be a C-contiguous array of the n_type's dtype with at least pixels * n_dot elements"
        self._check(self._lib.qd_scan_closed_host(self._ctx, len(scans), _ptr(scans), _ptr(q), _ptr(z), _ptr(n), n_type,
                                                  flags))
        return z, n

    def points_closed_host(self, scan: np.ndarray, n_charge, v: np.ndarray, n_type: int = N_F64, flags: int = 0,
                           want_z: bool = True):
        """``points_open_host`` for a closed array of ``n_charge`` carriers in total."""
        q = int(self._n_charge(n_charge, 1)[0])
        v = np.ascontiguousarray(v, dtype=np.float64)
        ny, nx, nv = v.shape
        if nv != self.models.n_volt:
            raise ValueError(f"The shape of vg is in correct it should be of shape (..., n_gate) = (...,{self.models.n_volt})")
        scan = np.ascontiguousarray(scan, dtype=SCAN_DTYPE).reshape(1)
        z = self._z(ny * nx, None, want_z, (ny, nx))
        n = np.empty((ny, nx, self.models.n_dot), dtype=N_DTYPES[n_type]) if n_type != N_NONE else None
        self._check(self._lib.qd_points_closed_host(self._ctx, _ptr(scan), q, ny, nx, _ptr(v), _ptr(z), _ptr(n), n_type,
                                                    flags))
        return z, n

    def normalise_obs(self, z, out=None, per_env: int | None = None, n_env: int | None = None, q_low: float = 0.5,
                      q_high: float = 99.5, stats=None, stream=None):
        """Per-env percentile normalisation of DEVICE images (``QuantumDeviceEnv._normalise_obs``, env.py:471-509):
        ``z`` holds ``n_env`` consecutive blocks of ``per_env`` float32 (all channels of one env); in place by default."""
        out = z if out is None else out
        n_env = self.models.n_env if n_env is None else n_env
        per_env = z.numel() // n_env if per_env is None else per_env
        self._check(self._lib.qd_normalise_obs(self._ctx, _ptr(z), _ptr(out), per_env, n_env, q_low, q_high, _ptr(stats),
                                               self._stream(stream)))
        return out

    def normalise_obs_typed(self, z, out, z_type: int, per_env: int | None = None, n_env: int | None = None,
                            q_low: float = 0.5, q_high: float = 99.5, stats=None, stream=None):
        """``normalise_obs`` into a DEVICE buffer of a compact element type (``Z_F16`` / ``Z_U8``)."""
        n_env = self.models.n_env if n_env is None else n_env
        per_env = z.numel() // n_env if per_env is None else per_env
        self._check(self._lib.qd_normalise_obs_typed(self._ctx, _ptr(z), _ptr(out), z_type, per_env, n_env, q_low, q_high,
                                                     _ptr(stats), self._stream(stream)))
        return out

    # -- introspection ---------------------------------------------------------------------------------------
    def status(self, clear: bool = True) -> int:
        """Sticky ``QD_STATUS_*`` bits raised by this context's kernels (check after synchronising an async launch)."""
        return int(self._lib.qd_status(self._ctx, 1 if clear else 0))

    @property
    def launch_count(self) -> int:
        return int(self._lib.qd_launch_count(self._ctx))

    def fp64_peak_tflops(self, iters: int = 4096) -> float:
        out = C.c_double()
        self._check(self._lib.qd_measure_fp64_peak(self._ctx, iters, C.byref(out)))
        return out.value

    def fp32_peak_tflops(self, iters: int = 4096) -> float:
        out = C.c_double()
        self._check(self._lib.qd_measure_fp32_peak(self._ctx, iters, C.byref(out)))
        return out.value
