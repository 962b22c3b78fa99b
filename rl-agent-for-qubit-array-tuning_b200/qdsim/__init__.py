"""qdsim -- host side of the B200-native charge-stability simulator (libqdsim.so).

``Engine`` is the batched entry point; ``qarray`` / ``qarray_latched`` (sibling packages) are the drop-in classes with
the reference's names and signatures.  Importing this package does not touch CUDA; creating an ``Engine`` does and
raises if the library or a GPU is missing (there is no CPU fallback).
"""
from ._lib import (QD_MAX_DOTS, QD_MAX_SENSORS, QD_MAX_VOLT, ALG_BRUTE_FORCE, ALG_DEFAULT, ALG_THRESHOLDED, ALG_TUNNEL, FLAG_CARRY_ROWS, FLAG_LATCH,  # noqa: F401
                   FLAG_LATCH_EXACT, FLAG_NOISE, FLAG_PINK, FLAG_RADIAL, FLAG_THERMAL, FLAG_WHITE_ON_OUTPUT, N_F32, N_F64, N_NONE,
                   N_U8, PARAMS_DTYPE, SCAN_DTYPE, STATUS_OCC_OVERFLOW, Z_DTYPES, Z_F16, Z_F32, Z_U8, QdError)
from .engine import K_B, Engine, ModelBatch, new_scans  # noqa: F401
