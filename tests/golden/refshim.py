"""Test infrastructure: run the REFERENCE's own tunnel-coupled simulator (``src/qarray_latched`` of the upstream project,
unmodified, imported where it lies) in a container that has neither ``jax`` nor ``qarray``.

Two stand-ins are installed into ``sys.modules`` before the reference is imported:

* ``jax`` / ``jax.numpy`` / ``jax.lax`` -- an EAGER NumPy evaluation of exactly the API subset the reference's
  Path B files touch (``jit`` = identity, ``vmap`` = Python loop over the mapped axis, ``lax.scan`` / ``fori_loop`` /
  ``cond`` = their definitional Python loops, ``.at[idx].set`` = copy-and-assign, ``argsort`` = stable like JAX's,
  ``linalg.eigh`` = LAPACK).  Everything is float64, i.e. JAX with ``jax_enable_x64`` (SURVEY.md section 8a B1).  No
  arithmetic of the reference is restated here: the shim only supplies the array primitives the reference's code calls.
* ``qarray`` -- INERT type shims for the names ``qarray_latched`` imports at module level from the absent
  ``qarray==1.6.0`` wheel (matrix type wrappers, ``LatchingBaseModel`` / ``BaseNoiseModel`` = the no-op base classes,
  ``_validate_vg`` = the check the fork itself carries at ``_helper_functions.py:217-223``).  Upstream-only arithmetic
  (``optimal_Vg``, ``compute_threshold``, latching, noise) is NOT provided: goldens made through this shim pin the
  in-tree reference code only -- Maxwell conversion, grid composer, relaxation, candidate selection, Hamiltonian,
  ground state, occupation expectation, sensor.

Used by ``tests/golden/make_reference_golden.py`` (fixture generator) and, when ``QADAPT_SRC`` points at the upstream
``src`` tree, by ``tests/test_reference_golden.py::test_reference_regenerates`` .  Never imported by the product.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np


def ref_src() -> str:
    """``src`` of a checkout of the upstream project, from ``QADAPT_SRC``.  Raises when it is not set or not a directory:
    without it the product's own drop-in ``qarray_latched`` would be the one imported."""
    src = os.environ.get("QADAPT_SRC", "")
    if not src or not os.path.isdir(src):
        raise RuntimeError(f"QADAPT_SRC={src!r}: set it to the src directory of a checkout of the upstream project")
    return os.path.abspath(src)


# ---------------------------------------------------------------------------------------------------------------------
# jax stand-in
# ---------------------------------------------------------------------------------------------------------------------
class _At:
    def __init__(self, arr):
        self._arr = arr

    def __getitem__(self, idx):
        return _AtIdx(self._arr, idx)


class _AtIdx:
    def __init__(self, arr, idx):
        self._arr, self._idx = arr, idx

    def set(self, value):
        out = self._arr.copy()
        out[self._idx] = value
        return out

    def add(self, value):
        out = self._arr.copy()
        np.add.at(out, self._idx, value)
        return out


class JArr(np.ndarray):
    """ndarray with jax's functional-update accessor."""

    @property
    def at(self):
        return _At(self)

    def block_until_ready(self):
        return self


def _j(a):
    return np.asarray(a).view(JArr)


def _wrap(fn):
    def inner(*args, **kwargs):
        out = fn(*args, **kwargs)
        if isinstance(out, np.ndarray):
            return out.view(JArr)
        if isinstance(out, (tuple, list)) and out and all(isinstance(o, np.ndarray) for o in out):
            return type(out)(o.view(JArr) for o in out) if not hasattr(out, "_fields") else out
        return out
    inner.__name__ = getattr(fn, "__name__", "wrapped")
    return inner


def _argsort(a, axis=-1, **kw):
    kw.pop("stable", None)
    return np.argsort(a, axis=axis, kind="stable").view(JArr)          # jnp.argsort is stable by default


def _jit(fn=None, **_kw):
    if fn is None:
        return lambda f: f
    return fn


def _tree_map_axis(x, axis, i):
    if axis is None:
        return x
    return np.take(np.asarray(x), i, axis=axis)


def _vmap(fn, in_axes=0, out_axes=0, **_kw):
    def mapped(*args):
        axes = in_axes if isinstance(in_axes, (tuple, list)) else (in_axes,) * len(args)
        n = next(np.asarray(a).shape[ax] for a, ax in zip(args, axes) if ax is not None)
        outs = [fn(*[_tree_map_axis(a, ax, i) for a, ax in zip(args, axes)]) for i in range(n)]
        if isinstance(outs[0], tuple):
            oax = out_axes if isinstance(out_axes, (tuple, list)) else (out_axes,) * len(outs[0])
            return tuple(np.stack([o[k] for o in outs], axis=oax[k]).view(JArr) for k in range(len(outs[0])))
        return np.stack(outs, axis=out_axes if not isinstance(out_axes, (tuple, list)) else out_axes[0]).view(JArr)
    return mapped


def _scan(f, init, xs, length=None):
    carry = init
    ys = []
    n = len(xs) if xs is not None else length
    for i in range(n):
        carry, y = f(carry, xs[i] if xs is not None else None)
        ys.append(y)
    ys = None if all(y is None for y in ys) else np.stack(ys)
    return carry, ys


def _fori_loop(lo, hi, body, val):
    for i in range(int(lo), int(hi)):
        val = body(i, val)
    return val


def _cond(pred, true_fn, false_fn, *operands):
    return true_fn(*operands) if bool(pred) else false_fn(*operands)


def make_jax():
    jax = types.ModuleType("jax")
    jnp = types.ModuleType("jax.numpy")
    lax = types.ModuleType("jax.lax")
    exp = types.ModuleType("jax.experimental")
    sparse = types.ModuleType("jax.experimental.sparse")
    for name in ("zeros", "ones", "array", "asarray", "full", "arange", "eye", "einsum", "where", "concatenate", "clip",
                 "floor", "expand_dims", "diag", "conj", "tile", "stack", "meshgrid", "exp", "abs", "sqrt", "sum",
                 "mean", "zeros_like", "ones_like", "linspace", "dot", "matmul", "outer", "maximum", "minimum", "round",
                 "argmin", "argmax", "min", "max", "log", "repeat", "reshape", "transpose", "squeeze", "take",
                 "cumsum", "prod", "sign", "isfinite", "isnan", "logical_and", "logical_or", "logical_not"):
        setattr(jnp, name, _wrap(getattr(np, name)))
    jnp.all, jnp.any = np.all, np.any
    jnp.argsort = _argsort
    jnp.ix_ = np.ix_
    jnp.inf, jnp.pi, jnp.nan, jnp.newaxis = np.inf, np.pi, np.nan, None
    jnp.ndarray = np.ndarray
    jnp.int32, jnp.int64, jnp.float32, jnp.float64 = np.int32, np.int64, np.float32, np.float64
    jnp.complex64, jnp.complex128, jnp.bool_ = np.complex64, np.complex128, np.bool_
    linalg = types.ModuleType("jax.numpy.linalg")
    for name in ("eigh", "inv", "pinv", "norm", "cholesky", "solve", "eigvalsh"):
        setattr(linalg, name, getattr(np.linalg, name))
    jnp.linalg = linalg
    lax.scan, lax.fori_loop, lax.cond = _scan, _fori_loop, _cond
    jax.numpy, jax.lax, jax.experimental = jnp, lax, exp
    exp.sparse = sparse
    sparse.BCOO = type("BCOO", (), {})                  # annotation target only (use_sparse is False)
    jax.jit, jax.vmap = _jit, _vmap
    jax.config = types.SimpleNamespace(update=lambda *a, **k: None)
    jax.nn = types.SimpleNamespace(sigmoid=lambda x: 1.0 / (1.0 + np.exp(-np.asarray(x, dtype=np.float64))))   # definition
    jax.devices = lambda *a, **k: []
    return {"jax": jax, "jax.numpy": jnp, "jax.numpy.linalg": linalg, "jax.lax": lax, "jax.experimental": exp,
            "jax.experimental.sparse": sparse}


# ---------------------------------------------------------------------------------------------------------------------
# qarray stand-in: inert types only
# ---------------------------------------------------------------------------------------------------------------------
def make_qarray():
    def mod(name):
        return types.ModuleType(name)

    class _Matrix(np.ndarray):                              # type name only: no validation, no arithmetic
        def __new__(cls, a):
            return np.array(a, dtype=np.float64).view(cls)

    q = mod("qarray")
    functions = mod("qarray.functions")

    def _absent(name):
        def f(*a, **k):
            raise NotImplementedError(f"qarray.{name} lives in the absent qarray==1.6.0 wheel")
        return f
    functions.compute_optimal_virtual_gate_matrix = _absent("functions.compute_optimal_virtual_gate_matrix")
    functions.optimal_Vg = _absent("functions.optimal_Vg")
    functions.compute_threshold = lambda cdd: 1.0          # only feeds a printed warning (_helper_functions.py:180-199)

    qtypes = mod("qarray.qarray_types")
    for name in ("CddInv", "Cdd", "VectorList", "CddNonMaxwell", "CgdNonMaxwell", "NegativeValuedMatrix",
                 "CdsNonMaxwell", "CgsNonMaxwell", "Vector", "PositiveValuedMatrix"):
        setattr(qtypes, name, type(name, (_Matrix,), {}))

    latching = mod("qarray.latching_models")

    class LatchingBaseModel:                                # the no-op base model
        def add_latching(self, n, measurement_shape=None):
            return n
    latching.LatchingBaseModel = LatchingBaseModel

    noise = mod("qarray.noise_models")

    class BaseNoiseModel:                                   # the no-noise base model
        def sample_input_noise(self, shape):
            return np.zeros(shape)

        def sample_output_noise(self, shape):
            return np.zeros(shape)
    noise.BaseNoiseModel = BaseNoiseModel

    pyimpl = mod("qarray.python_implementations")
    helper = mod("qarray.python_implementations.helper_functions")
    helper.free_energy = _absent("python_implementations.helper_functions.free_energy")   # closed arrays only
    dot_arrays = mod("qarray.DotArrays")
    dhelper = mod("qarray.DotArrays._helper_functions")

    def _validate_vg(vg, n_gate):                           # same check as the fork's own _helper_functions.py:217-223
        if vg.shape[-1] != n_gate:
            raise ValueError(f"The shape of vg is in correct it should be of shape (..., n_gate) = (...,{n_gate})")
    dhelper._validate_vg = _validate_vg
    q.functions, q.qarray_types, q.latching_models, q.noise_models = functions, qtypes, latching, noise
    q.python_implementations, q.DotArrays = pyimpl, dot_arrays
    pyimpl.helper_functions = helper
    dot_arrays._helper_functions = dhelper
    q.LatchingBaseModel, q.BaseNoiseModel = LatchingBaseModel, BaseNoiseModel
    return {"qarray": q, "qarray.functions": functions, "qarray.qarray_types": qtypes,
            "qarray.latching_models": latching, "qarray.noise_models": noise,
            "qarray.python_implementations": pyimpl, "qarray.python_implementations.helper_functions": helper,
            "qarray.DotArrays": dot_arrays, "qarray.DotArrays._helper_functions": dhelper}


class reference_modules:
    """Context manager: the reference's ``qarray_latched`` importable on the stand-ins; ``sys.modules`` / ``sys.path``
    restored on exit, so the product's own ``qarray`` / ``qarray_latched`` packages are untouched."""

    _PREFIXES = ("jax", "qarray", "qarray_latched")

    def __enter__(self):
        self._saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] in self._PREFIXES}
        for k in self._saved:
            del sys.modules[k]
        sys.modules.update(make_jax())
        sys.modules.update(make_qarray())
        src = ref_src()
        self._path = list(sys.path)
        sys.path.insert(0, src)
        import importlib
        tccs = importlib.import_module("qarray_latched.DotArrays.TunnelCoupledChargeSensed")
        tccs = sys.modules["qarray_latched.DotArrays.TunnelCoupledChargeSensed"]
        bvm = sys.modules["qarray_latched.DotArrays.barrier_voltage_model"]
        assert os.path.abspath(tccs.__file__).startswith(src + os.sep), tccs.__file__
        return types.SimpleNamespace(TunnelCoupledChargeSensed=tccs.TunnelCoupledChargeSensed,
                                     BarrierVoltageModel=bvm.BarrierVoltageModel, tccs=tccs)

    def __exit__(self, *exc):
        for k in [k for k in sys.modules if k.split(".")[0] in self._PREFIXES]:
            del sys.modules[k]
        sys.modules.update(self._saved)
        sys.path[:] = self._path
        return False
