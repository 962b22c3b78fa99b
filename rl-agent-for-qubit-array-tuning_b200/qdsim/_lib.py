"""ctypes binding of libqdsim.so (include/qdsim.h).  There is NO fallback: if the CUDA library is missing or does
not load, importing the engine raises -- the product path never computes on the CPU."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

QD_MAX_DOTS = 8
QD_MAX_VOLT = 16
QD_MAX_SENSORS = 4

# enum qd_algorithm
ALG_DEFAULT, ALG_THRESHOLDED, ALG_BRUTE_FORCE, ALG_TUNNEL = 0, 1, 2, 3
ALGORITHMS = {"default": ALG_DEFAULT, "thresholded": ALG_THRESHOLDED, "brute_force": ALG_BRUTE_FORCE,
              "tunnel": ALG_TUNNEL}
# enum qd_ntype
N_NONE, N_U8, N_F32, N_F64 = 0, 1, 2, 3
N_DTYPES = {N_U8: np.uint8, N_F32: np.float32, N_F64: np.float64}
# enum qd_ztype (compact observation images)
Z_F32, Z_F16, Z_U8 = 0, 1, 2
Z_DTYPES = {Z_F32: np.float32, Z_F16: np.float16, Z_U8: np.uint8}
STATUS_OCC_OVERFLOW = 0x1
# closed entry points (qd_scan_closed ...): largest total charge per algorithm (QD_ERR_INVALID above it)
CLOSED_MAX_CHARGE = {"default": 251, "brute_force": 15}
# flags
FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, FLAG_THERMAL = 0x01, 0x02, 0x04, 0x08
FLAG_CARRY_ROWS, FLAG_LATCH_EXACT, FLAG_WHITE_ON_OUTPUT, FLAG_PINK = 0x10, 0x20, 0x40, 0x80

SCAN_DTYPE = np.dtype([
    ("v0", "f8", (QD_MAX_VOLT,)), ("dx", "f8", (QD_MAX_VOLT,)), ("dy", "f8", (QD_MAX_VOLT,)),
    ("peak_width", "f8"),
    ("rad_x0", "f8"), ("rad_dx", "f8"), ("rad_y0", "f8"), ("rad_dy", "f8"),
    ("rad_alpha", "f8"), ("rad_zero_radius", "f8"), ("rad_max_amp", "f8"),
    ("seed", "u8"), ("pix_offset", "i8"),
    ("env_id", "i4"), ("nx", "i4"), ("ny", "i4"), ("rad_mode", "i4"),
], align=True)
assert SCAN_DTYPE.itemsize == 480, SCAN_DTYPE.itemsize

PARAMS_DTYPE = np.dtype([
    ("kT", "f8"), ("threshold", "f8"), ("white_amp", "f8"),
    ("tele_p01", "f8"), ("tele_p10", "f8"), ("tele_amp", "f8"),
    ("p_leads", "f8", (QD_MAX_DOTS,)), ("p_inter", "f8", (QD_MAX_DOTS * QD_MAX_DOTS,)),
    ("tc_base", "f8"), ("alpha", "f8", (QD_MAX_DOTS,)), ("vc_alpha", "f8"), ("vc_beta", "f8"),
    ("max_charge_carriers", "i4"), ("latching", "i4"), ("pink_amp", "f8"),
    ("vc_vchar", "f8"), ("vc_kind", "i4"), ("reserved0", "i4"),
], align=True)
assert PARAMS_DTYPE.itemsize == 744, PARAMS_DTYPE.itemsize
VC_LINEAR, VC_QUADRATIC, VC_SIGMOID = 0, 1, 2


class ModelDesc(C.Structure):
    _fields_ = [("n_env", C.c_int32), ("n_dot", C.c_int32), ("n_sensor", C.c_int32), ("n_volt", C.c_int32),
                ("n_gate", C.c_int32), ("algorithm", C.c_int32), ("num_charge_states", C.c_int32),
                ("charge_state_batch_size", C.c_int32)]


class QdError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libqdsim error {code}: {message}")
        self.code = code


def lib_path() -> str:
    here = os.path.dirname(os.path.abspath(__file__))
    return os.environ.get("QDSIM_LIB", os.path.join(here, "..", "csrc", "libqdsim.so"))


EXPORTS = ("qd_abi_version", "qd_create", "qd_destroy", "qd_last_error", "qd_set_models", "qd_scan_open",
           "qd_scan_upload", "qd_scan_launch", "qd_scan_open_host", "qd_normalise_obs", "qd_normalise_obs_typed",
           "qd_scan_obs_host", "qd_status", "qd_points_open_host", "qd_launch_count", "qd_measure_fp64_peak",
           "qd_measure_fp32_peak", "qd_scan_closed", "qd_scan_closed_host", "qd_points_closed_host")
ABI_VERSION = 3

_lib = None


def load() -> C.CDLL:
    """Load libqdsim.so and declare the prototypes.  Raises OSError when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise OSError(f"{path} not found: build it with `python __graft_entry__.py build` "
                      f"(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    vp, dp = C.c_void_p, C.POINTER(C.c_double)
    lib.qd_abi_version.restype = C.c_int
    lib.qd_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.qd_create.restype = C.c_int
    lib.qd_destroy.argtypes = [vp]
    lib.qd_destroy.restype = None
    lib.qd_last_error.argtypes = [vp]
    lib.qd_last_error.restype = C.c_char_p
    lib.qd_set_models.argtypes = [vp, C.POINTER(ModelDesc), vp, vp, vp, vp, vp, vp]
    lib.qd_set_models.restype = C.c_int
    lib.qd_scan_open.argtypes = [vp, C.c_int, vp, vp, vp, C.c_int, C.c_uint, vp]
    lib.qd_scan_open.restype = C.c_int
    lib.qd_scan_upload.argtypes = [vp, C.c_int, vp, vp]
    lib.qd_scan_upload.restype = C.c_int
    lib.qd_scan_launch.argtypes = [vp, vp, vp, C.c_int, C.c_uint, vp]
    lib.qd_scan_launch.restype = C.c_int
    lib.qd_scan_open_host.argtypes = [vp, C.c_int, vp, vp, vp, C.c_int, C.c_uint]
    lib.qd_scan_open_host.restype = C.c_int
    lib.qd_points_open_host.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, vp, C.c_int, C.c_uint]
    lib.qd_points_open_host.restype = C.c_int
    lib.qd_scan_closed.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_uint, vp]
    lib.qd_scan_closed.restype = C.c_int
    lib.qd_scan_closed_host.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_uint]
    lib.qd_scan_closed_host.restype = C.c_int
    lib.qd_points_closed_host.argtypes = [vp, vp, C.c_int32, C.c_int, C.c_int, vp, vp, vp, C.c_int, C.c_uint]
    lib.qd_points_closed_host.restype = C.c_int
    lib.qd_normalise_obs.argtypes = [vp, vp, vp, C.c_int64, C.c_int, C.c_double, C.c_double, vp, vp]
    lib.qd_normalise_obs.restype = C.c_int
    lib.qd_normalise_obs_typed.argtypes = [vp, vp, vp, C.c_int, C.c_int64, C.c_int, C.c_double, C.c_double, vp, vp]
    lib.qd_normalise_obs_typed.restype = C.c_int
    lib.qd_scan_obs_host.argtypes = [vp, C.c_int, vp, C.c_int, vp, C.c_int, C.c_int, C.c_double, C.c_double, vp, C.c_uint]
    lib.qd_scan_obs_host.restype = C.c_int
    lib.qd_status.argtypes = [vp, C.c_int]
    lib.qd_status.restype = C.c_int
    lib.qd_launch_count.argtypes = [vp]
    lib.qd_launch_count.restype = C.c_int64
    lib.qd_measure_fp64_peak.argtypes = [vp, C.c_int, dp]
    lib.qd_measure_fp64_peak.restype = C.c_int
    lib.qd_measure_fp32_peak.argtypes = [vp, C.c_int, dp]
    lib.qd_measure_fp32_peak.restype = C.c_int
    if lib.qd_abi_version() != ABI_VERSION:
        raise OSError(f"{path}: ABI version {lib.qd_abi_version()} != {ABI_VERSION}")
    _lib = lib
    return lib
