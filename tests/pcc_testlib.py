"""Shared test helpers: ctypes views of the C-ABI PODs, loaders for the
oracle (oracle/liboracle.so) and the compiled reference
(oracle/_ref/libtmc13_ref.so), the recorded outputs of that reference
(tests/golden/reference_tape.npz), and the synthetic point-cloud generators
of SURVEY.md 8(d).  TEST INFRASTRUCTURE ONLY."""
import atexit
import ctypes as C
import functools
import hashlib
import inspect
import json
import os
import subprocess

import numpy as np
from numpy.lib.recfunctions import structured_to_unstructured

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")

MAX_QP_LAYERS = 32
MAX_AC_QP_LAYERS = 32


class RahtParams(C.Structure):
    _fields_ = [
        ("prediction_enabled", C.c_int32),
        ("integer_haar", C.c_int32),
        ("prediction_threshold0", C.c_int32),
        ("prediction_threshold1", C.c_int32),
        ("subnode_prediction_enabled", C.c_int32),
        ("prediction_search_range", C.c_int32),
        ("pred_weight_parent", C.c_int32 * 19),
        ("pred_weight_child", C.c_int32 * 12),
        ("raht_extension", C.c_int32),
    ]


class QpSet(C.Structure):
    _fields_ = [
        ("num_layers", C.c_int32),
        ("layers", (C.c_int32 * 2) * MAX_QP_LAYERS),
        ("max_qp", C.c_int32),
        ("fixed_point_qp_offset", C.c_int32),
        ("num_ac_coeff_qp_layers", C.c_int32),
        ("ac_coeff_qps", ((C.c_int32 * 2) * 7) * MAX_AC_QP_LAYERS),
    ]


class Predictor(C.Structure):
    _fields_ = [
        ("neighbor_count", C.c_uint32),
        ("predictor_index", C.c_uint32 * 3),
        ("weight", C.c_uint32 * 3),
    ]


DEFAULT_PARENT_W = [4, 2, 2, 2, 1, 1, 1, 1, 1, 2, 1, 2, 2, 1, 1, 1, 1, 1, 1]


def set_prediction_weights(p, w):
    """RahtPredictionParams::setPredictionWeights (tmc3/hls.h:456-465)."""
    child = [w[4], w[4], w[3], w[4], w[3], w[3], w[4], w[4], w[4], w[4], w[4], w[4]]
    parent = [w[0], w[1], w[1], w[1], w[2], w[2], w[2], w[2], w[2], w[1], w[2],
              w[1], w[1], w[2], w[2], w[2], w[2], w[2], w[2]]
    for i in range(19):
        p.pred_weight_parent[i] = parent[i]
    for i in range(12):
        p.pred_weight_child[i] = child[i]


def make_params(prediction=1, haar=0, thr0=2, thr1=6, subnode=1,
                search_range=50000, weights=(9, 3, 1, 5, 2), ext=1):
    p = RahtParams()
    p.prediction_enabled = prediction
    p.integer_haar = haar
    p.prediction_threshold0 = thr0
    p.prediction_threshold1 = thr1
    p.subnode_prediction_enabled = subnode
    p.prediction_search_range = search_range
    p.raht_extension = ext
    for i in range(19):
        p.pred_weight_parent[i] = DEFAULT_PARENT_W[i]
    if subnode:
        # TMC3.cpp:1894-1906: weights are only derived when sub-node
        # prediction is on; otherwise the constructor defaults stay.
        set_prediction_weights(p, list(weights))
    return p


def make_qpset(qp=34, chroma_offset=-2, bitdepth=8, layers=None,
               fixed_point_qp_offset=0, ac_qps=None):
    q = QpSet()
    if layers is None:
        layers = [(qp, chroma_offset)]
    q.num_layers = len(layers)
    for i, (a, b) in enumerate(layers):
        q.layers[i][0] = a
        q.layers[i][1] = b
    q.max_qp = 51 + 6 * (bitdepth - 8)
    q.fixed_point_qp_offset = fixed_point_qp_offset
    q.num_ac_coeff_qp_layers = 0
    if ac_qps is not None:
        q.num_ac_coeff_qp_layers = len(ac_qps)
        for l, layer in enumerate(ac_qps):
            for c in range(7):
                q.ac_coeff_qps[l][c][0] = layer[c][0]
                q.ac_coeff_qps[l][c][1] = layer[c][1]
    return q


# --------------------------------------------------------------------------
# library loaders

def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


_oracle = None
_ref = None


def build_oracle():
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "oracle"])


def load_oracle():
    global _oracle
    if _oracle is None:
        path = os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(path) or any(
            os.path.getmtime(os.path.join(ORACLE_DIR, f)) > os.path.getmtime(path)
            for f in os.listdir(ORACLE_DIR) if f.endswith((".c", ".h"))):
            build_oracle()
        lib = C.CDLL(path)
        lib.oracle_raht.restype = C.c_int
        lib.oracle_isqrt.restype = C.c_uint32
        lib.oracle_isqrt.argtypes = [C.c_uint64]
        lib.oracle_irsqrt.restype = C.c_uint64
        lib.oracle_irsqrt.argtypes = [C.c_uint64]
        lib.oracle_morton_addr.restype = C.c_int64
        lib.oracle_morton_addr.argtypes = [C.c_int32] * 3
        lib.oracle_morton3d_add.restype = C.c_uint64
        lib.oracle_morton3d_add.argtypes = [C.c_uint64] * 2
        lib.oracle_quantize.restype = C.c_int64
        lib.oracle_quantize.argtypes = [C.c_int, C.c_int64]
        lib.oracle_scale.restype = C.c_int64
        lib.oracle_scale.argtypes = [C.c_int, C.c_int64]
        lib.oracle_fixed_mul.restype = C.c_int64
        lib.oracle_fixed_mul.argtypes = [C.c_int64] * 2
        lib.oracle_div_approx.restype = C.c_int64
        lib.oracle_div_approx.argtypes = [C.c_int64, C.c_uint64, C.c_int32]
        _oracle = lib
    return _oracle


def ref_available():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libtmc13_ref.so"))


def load_ref():
    """The compiled, unmodified reference (built by `make -C oracle ref`)."""
    global _ref
    if _ref is None:
        lib = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "libtmc13_ref.so"))
        for name in ("tmc13ref_raht", "tmc13ref_morton_sort", "tmc13ref_attr_raht",
                     "tmc13ref_quant_weights", "tmc13ref_lift"):
            getattr(lib, name).restype = C.c_double
        lib.tmc13ref_isqrt.restype = C.c_uint32
        lib.tmc13ref_isqrt.argtypes = [C.c_uint64]
        lib.tmc13ref_irsqrt.restype = C.c_uint64
        lib.tmc13ref_irsqrt.argtypes = [C.c_uint64]
        lib.tmc13ref_morton_addr.restype = C.c_int64
        lib.tmc13ref_morton_addr.argtypes = [C.c_int32] * 3
        lib.tmc13ref_morton3d_add.restype = C.c_uint64
        lib.tmc13ref_morton3d_add.argtypes = [C.c_uint64] * 2
        lib.tmc13ref_quantize.restype = C.c_int64
        lib.tmc13ref_quantize.argtypes = [C.c_int, C.c_int64]
        lib.tmc13ref_scale.restype = C.c_int64
        lib.tmc13ref_scale.argtypes = [C.c_int, C.c_int64]
        lib.tmc13ref_fixed_mul.restype = C.c_int64
        lib.tmc13ref_fixed_mul.argtypes = [C.c_int64] * 2
        lib.tmc13ref_div_approx.restype = C.c_int64
        lib.tmc13ref_div_approx.argtypes = [C.c_int64, C.c_uint64, C.c_int32]
        _ref = lib
    return _ref


# --------------------------------------------------------------------------
# recorded outputs of the compiled reference
#
# The reference is only available where its sources are, so every ref_*
# function below replays what it returned when it was recorded
# (tests/golden/make_golden.py runs the suite with PCCB200_RECORD_REFERENCE=1
# and the compiled reference present).  Entries are keyed by the function and
# a digest of its arguments, so a test whose inputs drift fails instead of
# comparing against another case.  Large arrays are kept as digests
# (`Recorded`, compared with `same`), small ones and scalars by value.  Inputs
# that were never recorded go to the compiled reference when it is present.

TAPE_PATH = os.path.join(ROOT, "tests", "golden", "reference_tape.npz")
RECORDING = os.environ.get("PCCB200_RECORD_REFERENCE") == "1"
_BY_VALUE_BYTES = 256
_tape = None


class Recorded:
    """an array the reference returned, known by its digest (see `digest`)"""

    def __init__(self, sha256, shape):
        self.sha256, self.shape = sha256, tuple(shape)

    def __repr__(self):
        return f"Recorded(shape={self.shape}, sha256={self.sha256[:12]}...)"


def digest(x):
    """sha256 (first 128 bits) of an integer array's shape and values (the
    dtype does not count: equal digests <=> np.array_equal); bytes count as a
    uint8 array"""
    if isinstance(x, Recorded):
        return x.sha256
    if isinstance(x, (bytes, bytearray)):
        x = np.frombuffer(x, dtype=np.uint8)
    x = np.asarray(x)
    if x.dtype.names:  # predictors: one column per field element
        x = structured_to_unstructured(x)
    if x.dtype.kind not in "iub":
        raise TypeError(f"digest of a {x.dtype} array")
    v = x.astype(np.uint64).view(np.int64) if x.dtype == np.uint64 else x.astype(np.int64)
    h = hashlib.sha256(repr(x.shape).encode())
    h.update(np.ascontiguousarray(v).tobytes())
    return h.hexdigest()[:32]


def same(*xs):
    """all arguments (arrays, bytes, Recorded) hold the same values"""
    return len({digest(x) for x in xs}) == 1


def _token(a):
    if a is None or isinstance(a, (bool, str)):
        return repr(a)
    if isinstance(a, (int, np.integer)):
        return repr(int(a))
    if isinstance(a, (float, np.floating)):
        return repr(float(a))
    if isinstance(a, C.Structure):
        return "pod:" + bytes(a).hex()
    if isinstance(a, (tuple, list)):
        return "(" + ",".join(_token(x) for x in a) + ")"
    return "array:" + digest(a)


def _encode(out, name, arrays, by_value):
    if isinstance(out, tuple):
        return {"tuple": [_encode(x, f"{name}/{i}", arrays, by_value) for i, x in enumerate(out)]}
    if isinstance(out, (bytes, bytearray)):
        return {"sha256": digest(out), "shape": [len(out)]}
    if isinstance(out, np.ndarray):
        if out.nbytes <= _BY_VALUE_BYTES and not out.dtype.names:
            return {"list": out.tolist(), "dtype": out.dtype.str}
        if by_value:  # stored in the narrowest integer type that holds it
            arrays[name] = out.astype(np.result_type(np.min_scalar_type(out.min()), np.min_scalar_type(out.max())))
            return {"array": name, "dtype": out.dtype.str}
        return {"sha256": digest(out), "shape": list(out.shape)}
    if isinstance(out, list):
        return {"value": [int(x) for x in out]}
    return {"value": out.item() if isinstance(out, np.generic) else out}


def _decode(e, arrays):
    if "tuple" in e:
        return tuple(_decode(x, arrays) for x in e["tuple"])
    if "array" in e:
        return arrays[e["array"]].astype(e["dtype"])
    if "list" in e:
        return np.array(e["list"], dtype=e["dtype"])
    if "sha256" in e:
        return Recorded(e["sha256"], e["shape"])
    return e["value"]


def _read_tape():
    if not os.path.exists(TAPE_PATH):
        return {}, {}
    with np.load(TAPE_PATH) as z:
        return json.loads(z["index"].tobytes()), {k: z[k] for k in z.files if k != "index"}


def _save_tape():
    """merge this process's recordings into the tape (the fuzz tools record
    from subprocesses of the test run)"""
    index, arrays = _read_tape()
    index.update(_tape[0])
    arrays.update(_tape[1])
    text = json.dumps(index, sort_keys=True, separators=(",", ":")).encode()
    np.savez_compressed(TAPE_PATH, index=np.frombuffer(text, dtype=np.uint8), **arrays)


def _load_tape():
    global _tape
    if _tape is None:
        if RECORDING:
            _tape = ({}, {})
            atexit.register(_save_tape)
        else:
            _tape = _read_tape()
    return _tape


def taped(by_value=False):
    """replay (or, when recording, record) the outputs of a ref_* function;
    by_value keeps whole arrays, for tests that measure how far the oracle
    is from the reference rather than asserting equality"""

    def wrap(fn):
        sig = inspect.signature(fn)

        @functools.wraps(fn)
        def call(*args, **kw):
            bound = sig.bind(*args, **kw)
            bound.apply_defaults()
            key = hashlib.sha256((fn.__name__ + _token(tuple(bound.arguments.values()))).encode()).hexdigest()[:32]
            index, arrays = _load_tape()
            if not RECORDING and key in index:
                return _decode(index[key], arrays)
            if any(isinstance(a, Recorded) for a in bound.arguments.values()):
                raise LookupError(f"{fn.__name__}: no recorded output for these inputs")
            try:
                out = fn(*bound.args, **bound.kwargs)
            except OSError as e:
                raise LookupError(
                    f"{fn.__name__}: no recorded output for these inputs and no compiled reference in "
                    "oracle/_ref; re-record with tests/golden/make_golden.py") from e
            if RECORDING:
                index[key] = _encode(out, key, arrays, by_value)
            return out

        return call

    return wrap


def _run_raht(fn, forward, params, qpset, morton, attrs, coeffs, qpoffs):
    n, a = attrs.shape
    attrs = np.ascontiguousarray(attrs, dtype=np.int32).copy()
    morton = np.ascontiguousarray(morton, dtype=np.int64)
    if forward:
        coeffs = np.zeros((a, n), dtype=np.int32)
    else:
        coeffs = np.ascontiguousarray(coeffs, dtype=np.int32).copy()
    if qpoffs is not None:
        qpoffs = np.ascontiguousarray(qpoffs, dtype=np.int32)
    r = fn(C.c_int(1 if forward else 0), C.byref(params), C.byref(qpset),
           _ptr(qpoffs, C.c_int32), _ptr(morton, C.c_int64),
           _ptr(attrs, C.c_int32), C.c_int(a), C.c_int(n),
           _ptr(coeffs, C.c_int32))
    return attrs, coeffs, r


def oracle_raht(forward, params, qpset, morton, attrs, coeffs=None, qpoffs=None):
    """-> (attrs_out [N,A], coeffs [A,N])"""
    a, c, r = _run_raht(load_oracle().oracle_raht, forward, params, qpset,
                        morton, attrs, coeffs, qpoffs)
    assert r == 0
    return a, c


@taped()
def ref_raht(forward, params, qpset, morton, attrs, coeffs=None, qpoffs=None,
             want_time=False):
    a, c, t = _run_raht(load_ref().tmc13ref_raht, forward, params, qpset,
                        morton, attrs, coeffs, qpoffs)
    return (a, c, t) if want_time else (a, c)


def oracle_morton_sort(xyz):
    xyz = np.ascontiguousarray(xyz, dtype=np.int32)
    n = xyz.shape[0]
    keys = np.zeros(n, dtype=np.int64)
    order = np.zeros(n, dtype=np.int32)
    load_oracle().oracle_morton_sort(_ptr(xyz, C.c_int32), C.c_int(n),
                                     _ptr(keys, C.c_int64), _ptr(order, C.c_int32))
    return keys, order


@taped()
def ref_morton_sort(xyz):
    xyz = np.ascontiguousarray(xyz, dtype=np.int32)
    n = xyz.shape[0]
    keys = np.zeros(n, dtype=np.int64)
    order = np.zeros(n, dtype=np.int32)
    load_ref().tmc13ref_morton_sort(_ptr(xyz, C.c_int32), C.c_int(n),
                                    _ptr(keys, C.c_int64), _ptr(order, C.c_int32))
    return keys, order


@taped()
def ref_elementwise(name, dtype, *columns):
    """the reference's scalar helper tmc13ref_<name> applied to every row of
    the argument columns -> array of `dtype`"""
    lib = load_ref() if name != "iatan2" else _load_liftref()
    f = getattr(lib, "tmc13ref_" + name)
    return np.array([f(*map(int, row)) for row in zip(*columns)], dtype=dtype)


import sys as _sys

_sys.path.insert(0, os.path.join(ROOT, "mpeg-pcc-tmc13_b200"))
from pcc_attr_b200.synth import (cloud_cube, cloud_lidar, cloud_random, cloud_shell,  # noqa: E402,F401
                                 np_morton, sort_cloud)


# --------------------------------------------------------------------------
# host emulation of the product's kernel bodies (tests/emu) — CPU tests only

_emu = None


def load_emu():
    global _emu
    if _emu is None:
        emu_dir = os.path.join(ROOT, "tests", "emu")
        subprocess.check_call(["make", "-s", "-C", emu_dir])
        lib = C.CDLL(os.path.join(emu_dir, "libemu.so"))
        lib.emu_raht.restype = C.c_int
        for nm, res, args in (
            ("isqrt", C.c_uint32, [C.c_uint64]),
            ("irsqrt", C.c_uint64, [C.c_uint64]),
            ("morton_addr", C.c_int64, [C.c_int32] * 3),
            ("morton3d_add", C.c_uint64, [C.c_uint64] * 2),
            ("quantize", C.c_int64, [C.c_int, C.c_int64]),
            ("scale", C.c_int64, [C.c_int, C.c_int64]),
            ("fixed_mul", C.c_int64, [C.c_int64] * 2),
            ("div_approx", C.c_int64, [C.c_int64, C.c_uint64, C.c_int32]),
        ):
            f = getattr(lib, "emu_" + nm)
            f.restype = res
            f.argtypes = args
        _emu = lib
    return _emu


def emu_raht(forward, params, qpset, morton, attrs, coeffs=None, qpoffs=None):
    a, c, r = _run_raht(load_emu().emu_raht, forward, params, qpset, morton,
                        attrs, coeffs, qpoffs)
    assert r == 0, r
    return a, c


# --------------------------------------------------------------------------
# lifting helpers

PREDICTOR_DTYPE = np.dtype([("neighbor_count", "<u4"), ("predictor_index", "<u4", 3),
                            ("weight", "<u4", 3)])


def synth_predictors(n, lod_count, seed, k=3):
    """Synthetic LoD structure: cumulative LoD sizes (coarse -> fine, roughly
    x4 per level) and predictors whose neighbours lie in strictly coarser
    LoDs with 8-bit weights summing to 256, like AttributeLods::generate
    produces for the lifting transform."""
    rng = np.random.default_rng(seed)
    sizes = np.maximum(1, (n * (0.25 ** np.arange(lod_count - 1, -1, -1))).astype(np.int64))
    sizes[-1] = max(1, n - int(sizes[:-1].sum()))
    npl = np.cumsum(sizes).astype(np.uint32)
    npl[-1] = n
    preds = np.zeros(n, dtype=PREDICTOR_DTYPE)
    start = int(npl[0])
    for l in range(1, lod_count):
        s, e = int(npl[l - 1]), int(npl[l])
        m = e - s
        if m <= 0:
            continue
        cnt = rng.integers(1, k + 1, size=m)
        cnt = np.minimum(cnt, s)
        idx = rng.integers(0, s, size=(m, 3))
        w = rng.integers(1, 200, size=(m, 3)).astype(np.int64)
        for c in (1, 2, 3):
            sel = cnt == c
            ww = w[sel, :c]
            ww = np.maximum(1, (ww * 256) // ww.sum(axis=1, keepdims=True))
            ww[:, 0] += 256 - ww.sum(axis=1)
            w[sel, :c] = ww
            w[sel, c:] = 0
            idx[sel, c:] = 0
        preds["neighbor_count"][s:e] = cnt
        preds["predictor_index"][s:e] = idx
        preds["weight"][s:e] = w
    return preds, npl


def _pp(preds):
    return C.cast(preds.ctypes.data, C.POINTER(Predictor))


def oracle_quant_weights(preds):
    lib = load_oracle()
    qw = np.zeros(preds.shape[0], dtype=np.uint64)
    lib.oracle_quant_weights(_pp(preds), C.c_int(preds.shape[0]), _ptr(qw, C.c_uint64))
    return qw


def oracle_lift(forward, preds, qw, npl, attrs):
    lib = load_oracle()
    a = np.ascontiguousarray(attrs, dtype=np.int64).copy()
    if a.ndim == 1:
        a = a[:, None]
    lib.oracle_lift(C.c_int(1 if forward else 0), _pp(preds), _ptr(qw, C.c_uint64),
                    C.c_int(a.shape[0]), _ptr(npl, C.c_uint32), C.c_int(len(npl)),
                    _ptr(a, C.c_int64), C.c_int(a.shape[1]))
    return a


@taped()
def ref_quant_weights(preds):
    qw = np.zeros(preds.shape[0], dtype=np.uint64)
    load_ref().tmc13ref_quant_weights(_pp(preds), C.c_int(preds.shape[0]), _ptr(qw, C.c_uint64))
    return qw


@taped()
def ref_lift(forward, preds, qw, npl, attrs):
    a = np.ascontiguousarray(attrs, dtype=np.int64).copy()
    if a.ndim == 1:
        a = a[:, None]
    load_ref().tmc13ref_lift(C.c_int(1 if forward else 0), _pp(preds), _ptr(qw, C.c_uint64),
                             C.c_int(a.shape[0]), _ptr(npl, C.c_uint32), C.c_int(len(npl)),
                             _ptr(a, C.c_int64), C.c_int(a.shape[1]))
    return a


# --------------------------------------------------------------------------
# LoD build helpers

MAX_LODS = 32


class LodParams(C.Structure):
    _fields_ = [
        ("num_detail_levels", C.c_int32),
        ("lod_decimation_type", C.c_int32),
        ("lod_sampling_period", C.c_int32 * MAX_LODS),
        ("dist2", C.c_int32),
        ("num_pred_nearest_neighbours", C.c_int32),
        ("inter_lod_search_range", C.c_int32),
        ("intra_lod_search_range", C.c_int32),
        ("intra_lod_prediction_skip_layers", C.c_int32),
        ("prediction_with_distribution", C.c_int32),
        ("lod_neigh_bias", C.c_int32 * 3),
        ("pred_weight_blending", C.c_int32),
    ]


def make_lod_params(levels=12, decimation=0, period=4, dist2=0, k=3, inter_range=1100000,
                    intra_range=0, skip_layers=None, distribution=1, bias=(1, 1, 1), blending=0):
    p = LodParams()
    p.num_detail_levels = levels
    p.lod_decimation_type = decimation
    for i in range(MAX_LODS):
        p.lod_sampling_period[i] = period
    p.dist2 = dist2
    p.num_pred_nearest_neighbours = k
    p.inter_lod_search_range = inter_range
    p.intra_lod_search_range = intra_range
    # lifting forces "skip all layers" (tmc3/encoder.cpp:777-780)
    p.intra_lod_prediction_skip_layers = levels + 1 if skip_layers is None else skip_layers
    p.prediction_with_distribution = distribution
    for i in range(3):
        p.lod_neigh_bias[i] = bias[i]
    p.pred_weight_blending = blending
    return p


def _run_lod(fn, params, xyz):
    xyz = np.ascontiguousarray(xyz, dtype=np.int32)
    n = xyz.shape[0]
    preds = np.zeros(n, dtype=PREDICTOR_DTYPE)
    indexes = np.zeros(n, dtype=np.uint32)
    npl = np.zeros(MAX_LODS, dtype=np.uint32)
    cnt = C.c_int32(0)
    r = fn(C.byref(params), _ptr(xyz, C.c_int32), C.c_int(n), _pp(preds), _ptr(indexes, C.c_uint32),
           _ptr(npl, C.c_uint32), C.byref(cnt))
    return preds, indexes, npl[:cnt.value].copy(), r


@taped()
def ref_lod_build(params, xyz):
    load_ref().tmc13ref_lod_build.restype = C.c_double
    p, i, n, t = _run_lod(load_ref().tmc13ref_lod_build, params, xyz)
    return p, i, n


def oracle_lod_build(params, xyz):
    lib = load_oracle()
    lib.oracle_lod_build.restype = C.c_int
    p, i, n, r = _run_lod(lib.oracle_lod_build, params, xyz)
    assert r == 0
    return p, i, n


def emu_lod_build(params, xyz):
    lib = load_emu()
    lib.emu_lod_build.restype = C.c_int
    p, i, n, r = _run_lod(lib.emu_lod_build, params, xyz)
    assert r == 0, r
    return p, i, n


# --------------------------------------------------------------------------
# lifting quantisation / whole lifting encoder

_liftref = None


def liftref_available():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libtmc13_lift.so"))


@taped()
def ref_lift_encode(lod_params, qpset, lcp_enabled, xyz, attrs, bitdepth=8):
    """The reference's own lifting encoder (LoD build, weights, forward lifting,
    quantisation (+LCP), reconstruction): -> (values [N,A] predictor order,
    recon [N,A] input order, lcp coefficients)."""
    _load_liftref()
    xyz = np.ascontiguousarray(xyz, dtype=np.int32)
    attrs = np.ascontiguousarray(attrs, dtype=np.int32)
    n, a = attrs.shape
    values = np.zeros((n, a), dtype=np.int32)
    recon = np.zeros((n, a), dtype=np.int32)
    lcp = np.zeros(MAX_LODS, dtype=np.int8)
    _liftref.tmc13ref_lift_encode(
        C.byref(lod_params), C.byref(qpset), C.c_int(lcp_enabled), _ptr(xyz, C.c_int32),
        _ptr(attrs, C.c_int32), C.c_int(n), C.c_int(a), C.c_int(bitdepth),
        _ptr(values, C.c_int32), _ptr(recon, C.c_int32), _ptr(lcp, C.c_int8))
    return values, recon, lcp[:lod_params.num_detail_levels].copy()


def oracle_lcp_coeffs(coeffs, npl, num_detail_levels):
    lib = load_oracle()
    coeffs = np.ascontiguousarray(coeffs, dtype=np.int64)
    out = np.zeros(num_detail_levels, dtype=np.int8)
    lib.oracle_lcp_coeffs(_ptr(coeffs, C.c_int64), C.c_int(coeffs.shape[0]), _ptr(npl, C.c_uint32),
                          C.c_int(len(npl)), C.c_int(num_detail_levels), _ptr(out, C.c_int8))
    return out


def oracle_lift_quant(forward, qpset, qw, npl, attrs, lcp=None, values=None, qpo=None):
    lib = load_oracle()
    a = np.ascontiguousarray(attrs, dtype=np.int64).copy()
    n, A = a.shape
    v = np.zeros((n, A), dtype=np.int32) if values is None else np.ascontiguousarray(values, dtype=np.int32).copy()
    lib.oracle_lift_quant(C.c_int(1 if forward else 0), C.byref(qpset), _ptr(qpo, C.c_int32),
                          _ptr(qw, C.c_uint64), C.c_int(n), _ptr(npl, C.c_uint32), C.c_int(len(npl)),
                          _ptr(a, C.c_int64), C.c_int(A), _ptr(lcp, C.c_int8), _ptr(v, C.c_int32))
    return a, v


def finish_lift_recon(inv, bitdepth):
    """divExp2RoundHalfInf(x, 8) then clip (tmc3/AttributeEncoder.cpp:1484-1493)"""
    r = np.where(inv >= 0, (inv + 128) >> 8, -((128 - inv) >> 8))
    return np.clip(r, 0, (1 << bitdepth) - 1).astype(np.int32)


def oracle_lift_encode(lod_params, qpset, lcp_enabled, xyz, attrs, bitdepth=8):
    """The oracle chain equivalent to the reference's lifting encoder."""
    preds, indexes, npl = oracle_lod_build(lod_params, xyz)
    qw = oracle_quant_weights(preds)
    a = attrs[indexes].astype(np.int64) << 8
    fwd = oracle_lift(1, preds, qw, npl, a)
    lcp = None
    if lcp_enabled and attrs.shape[1] == 3:
        lcp = oracle_lcp_coeffs(fwd, npl, lod_params.num_detail_levels)
    rec_coef, values = oracle_lift_quant(1, qpset, qw, npl, fwd, lcp=lcp)
    inv = oracle_lift(0, preds, qw, npl, rec_coef)
    out = np.zeros_like(attrs)
    out[indexes] = finish_lift_recon(inv, bitdepth)
    return values, out, (lcp if lcp is not None else np.zeros(lod_params.num_detail_levels, dtype=np.int8))


def _attr_lift(fn, forward, lod_params, qpset, lcp_enabled, xyz, attrs, values, lcp, bitdepth, qpo=None):
    xyz = np.ascontiguousarray(xyz, dtype=np.int32)
    attrs = np.ascontiguousarray(attrs, dtype=np.int32).copy()
    n, a = attrs.shape
    if forward:
        values = np.zeros((n, a), dtype=np.int32)
        lcp = np.zeros(MAX_LODS, dtype=np.int8)
    else:
        values = np.ascontiguousarray(values, dtype=np.int32)
        l2 = np.zeros(MAX_LODS, dtype=np.int8)
        l2[:len(lcp)] = lcp
        lcp = l2
    r = fn(C.c_int(1 if forward else 0), C.byref(lod_params), C.byref(qpset), C.c_int(lcp_enabled),
           _ptr(qpo, C.c_int32), _ptr(xyz, C.c_int32), _ptr(attrs, C.c_int32), C.c_int(a), C.c_int(n),
           C.c_int(bitdepth), _ptr(values, C.c_int32), _ptr(lcp, C.c_int8))
    assert r == 0, r
    return values, attrs, lcp[:lod_params.num_detail_levels].copy()


def emu_attr_lift(forward, lod_params, qpset, lcp_enabled, xyz, attrs, values=None, lcp=None, bitdepth=8):
    lib = load_emu()
    lib.emu_attr_lift.restype = C.c_int
    return _attr_lift(lib.emu_attr_lift, forward, lod_params, qpset, lcp_enabled, xyz, attrs, values,
                      lcp, bitdepth)


# --------------------------------------------------------------------------
# spherical coordinates (row N2)

def _load_liftref():
    global _liftref
    if _liftref is None:
        _liftref = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "libtmc13_lift.so"))
        _liftref.tmc13ref_lift_encode.restype = C.c_double
    return _liftref


def _i3(v):
    return (C.c_int32 * 3)(*[int(x) for x in v])


def _run_rpl(fn, origin, theta, xyz, weight=None, min_pos=None, emu=False):
    xyz = np.ascontiguousarray(xyz, dtype=np.int32)
    theta = np.ascontiguousarray(theta, dtype=np.int32)
    out = np.zeros_like(xyz)
    bbox = np.zeros(6, dtype=np.int32)
    if emu:
        fn(_i3(origin), _ptr(theta, C.c_int32), C.c_int(theta.size),
           None if weight is None else _i3(weight), None if min_pos is None else _i3(min_pos),
           _ptr(xyz, C.c_int32), C.c_int64(xyz.shape[0]), _ptr(out, C.c_int32),
           _ptr(bbox, C.c_int32))
    else:
        fn(_i3(origin), _ptr(theta, C.c_int32), C.c_int(theta.size), _ptr(xyz, C.c_int32),
           C.c_int64(xyz.shape[0]), _ptr(out, C.c_int32), _ptr(bbox, C.c_int32))
    return out, bbox


@taped()
def ref_xyz_to_rpl(origin, theta, xyz):
    return _run_rpl(_load_liftref().tmc13ref_xyz_to_rpl, origin, theta, xyz)


def oracle_xyz_to_rpl(origin, theta, xyz):
    return _run_rpl(load_oracle().oracle_xyz_to_rpl, origin, theta, xyz)


def emu_xyz_to_rpl(origin, theta, xyz, weight=None, min_pos=None):
    return _run_rpl(load_emu().emu_xyz_to_rpl, origin, theta, xyz, weight, min_pos, emu=True)


def _run_offset_scale(fn, min_pos, weight, pos):
    pos = np.ascontiguousarray(pos, dtype=np.int32).copy()
    fn(_i3(min_pos), _i3(weight), _ptr(pos, C.c_int32), C.c_int64(pos.shape[0]))
    return pos


@taped()
def ref_offset_and_scale(min_pos, weight, pos):
    return _run_offset_scale(_load_liftref().tmc13ref_offset_and_scale, min_pos, weight, pos)


def oracle_offset_and_scale(min_pos, weight, pos):
    return _run_offset_scale(load_oracle().oracle_offset_and_scale, min_pos, weight, pos)


@taped()
def ref_normalised_axes_weights(box_max, forced_max_log2=0):
    out = (C.c_int32 * 3)()
    _load_liftref().tmc13ref_normalised_axes_weights(_i3(box_max), C.c_int(forced_max_log2), out)
    return [int(v) for v in out]


def lidar_lasers(num=64, lo=-0.43, hi=0.04):
    """elevation tangents of a spinning LiDAR in the reference's fixed point
    (gps.angularTheta: tan(theta) * 2^18), ascending"""
    return np.rint(np.tan(np.linspace(lo, hi, num)) * (1 << 18)).astype(np.int32)


# --------------------------------------------------------------------------
# symbol preparation for the entropy coder (row N1)

def _run_symbols(fn, coeffs):
    coeffs = np.ascontiguousarray(coeffs, dtype=np.int32)
    a, n = coeffs.shape
    runs = np.zeros(n, dtype=np.int32)
    values = np.zeros((n, a), dtype=np.int32)
    ctx = np.zeros(n, dtype=np.uint8)
    tail = C.c_int32(0)
    fn.restype = C.c_int
    cnt = fn(_ptr(coeffs, C.c_int32), C.c_int(a), C.c_int(n), _ptr(runs, C.c_int32),
             _ptr(values, C.c_int32), _ptr(ctx, C.c_uint8), C.byref(tail))
    return runs[:cnt].copy(), values[:cnt].copy(), (ctx[:cnt].copy() if a == 3 else None), tail.value


def oracle_coeff_symbols(coeffs):
    return _run_symbols(load_oracle().oracle_coeff_symbols, coeffs)


def emu_coeff_symbols(coeffs):
    return _run_symbols(load_emu().emu_coeff_symbols, coeffs)


@taped()
def ref_raht_encode_payload(params, qpset, xyz, attrs, bitdepth=8):
    """the reference's own RAHT attribute encoder (sort, transform, coefficient
    walk, arithmetic coding) -> (payload bytes, reconstruction [N, A])"""
    lib = _load_liftref()
    xyz = np.ascontiguousarray(xyz, dtype=np.int32)
    attrs = np.ascontiguousarray(attrs, dtype=np.int32)
    n, a = attrs.shape
    cap = 64 + n * a * 8
    buf = np.zeros(cap, dtype=np.uint8)
    recon = np.zeros((n, a), dtype=np.int32)
    lib.tmc13ref_raht_encode_payload.restype = C.c_int
    ln = lib.tmc13ref_raht_encode_payload(
        C.byref(params), C.byref(qpset), _ptr(xyz, C.c_int32), _ptr(attrs, C.c_int32), C.c_int(n),
        C.c_int(a), C.c_int(bitdepth), _ptr(buf, C.c_uint8), C.c_int(cap), _ptr(recon, C.c_int32))
    assert ln >= 0
    return bytes(buf[:ln]), recon


@taped()
def ref_symbols_payload(mode, runs, values, ctx, tail, n):
    """a symbol stream through the reference's PCCResidualsEncoder -> payload bytes
    (mode 0: its encode() members; mode 1: encodeSymbol with the given selectors)"""
    lib = _load_liftref()
    runs = np.ascontiguousarray(runs, dtype=np.int32)
    values = np.ascontiguousarray(values, dtype=np.int32)
    a = values.shape[1]
    c8 = np.ascontiguousarray(ctx if ctx is not None else np.zeros(len(runs)), dtype=np.uint8)
    cap = 64 + n * a * 8
    buf = np.zeros(cap, dtype=np.uint8)
    lib.tmc13ref_symbols_payload.restype = C.c_int
    ln = lib.tmc13ref_symbols_payload(
        C.c_int(mode), _ptr(runs, C.c_int32), _ptr(values, C.c_int32), _ptr(c8, C.c_uint8),
        C.c_int(len(runs)), C.c_int(tail), C.c_int(a), C.c_int(n), _ptr(buf, C.c_uint8), C.c_int(cap))
    assert ln >= 0
    return bytes(buf[:ln])


@taped()
def ref_decode_symbol_stream(payload, n, a):
    """the symbol stream as the reference's RAHT decoder reads it"""
    lib = _load_liftref()
    buf = np.frombuffer(payload, dtype=np.uint8).copy()
    runs = np.zeros(n, dtype=np.int32)
    values = np.zeros((n, a), dtype=np.int32)
    tail = C.c_int32(0)
    lib.tmc13ref_decode_symbol_stream.restype = C.c_int
    cnt = lib.tmc13ref_decode_symbol_stream(
        _ptr(buf, C.c_uint8), C.c_int(len(buf)), C.c_int(n), C.c_int(a), _ptr(runs, C.c_int32),
        _ptr(values, C.c_int32), C.byref(tail))
    return runs[:cnt].copy(), values[:cnt].copy(), tail.value


# --------------------------------------------------------------------------
# estimateDist2 (row N3, first half)

def _run_dist2(fn, xyz, period, rng_, pct):
    xyz = np.ascontiguousarray(xyz, dtype=np.int32)
    fn.restype = C.c_int
    return fn(_ptr(xyz, C.c_int32), C.c_int(xyz.shape[0]), C.c_int(period), C.c_int(rng_),
              C.c_float(pct))


@taped()
def ref_estimate_dist2(xyz, period=100, search_range=128, pct=0.85):
    return _run_dist2(_load_liftref().tmc13ref_estimate_dist2, xyz, period, search_range, pct)


def oracle_estimate_dist2(xyz, period=100, search_range=128, pct=0.85):
    return _run_dist2(load_oracle().oracle_estimate_dist2, xyz, period, search_range, pct)


def emu_estimate_dist2(xyz, period=100, search_range=128, pct=0.85):
    return _run_dist2(load_emu().emu_estimate_dist2, xyz, period, search_range, pct)


# --------------------------------------------------------------------------
# the other two quantisation-weight derivations (row L5)

@taped()
def ref_quant_weights_fixed(preds, neigh_weight):
    qw = np.zeros(preds.shape[0], dtype=np.uint64)
    load_ref().tmc13ref_quant_weights_fixed(_pp(preds), C.c_int(preds.shape[0]), _i3(neigh_weight),
                                            _ptr(qw, C.c_uint64))
    return qw


def oracle_quant_weights_fixed(preds, neigh_weight):
    qw = np.zeros(preds.shape[0], dtype=np.uint64)
    load_oracle().oracle_quant_weights_fixed(_pp(preds), C.c_int(preds.shape[0]),
                                             _i3(neigh_weight), _ptr(qw, C.c_uint64))
    return qw


def emu_quant_weights_fixed(preds, npl, neigh_weight):
    npl = np.ascontiguousarray(npl, dtype=np.uint32)
    qw = np.zeros(preds.shape[0], dtype=np.uint64)
    lib = load_emu()
    lib.emu_quant_weights_fixed.restype = C.c_int
    rc = lib.emu_quant_weights_fixed(_pp(preds), C.c_int(preds.shape[0]), _ptr(npl, C.c_uint32),
                                     C.c_int(npl.size), _i3(neigh_weight), _ptr(qw, C.c_uint64))
    assert rc == 0
    return qw


@taped()
def ref_quant_weights_scalable(preds, npl, num_points, min_log2):
    npl = np.ascontiguousarray(npl, dtype=np.uint32)
    qw = np.zeros(preds.shape[0], dtype=np.uint64)
    load_ref().tmc13ref_quant_weights_scalable(
        _pp(preds), C.c_int(preds.shape[0]), _ptr(npl, C.c_uint32), C.c_int(npl.size),
        C.c_uint64(num_points), C.c_int(min_log2), _ptr(qw, C.c_uint64))
    return qw


def oracle_quant_weights_scalable(npl, num_points, min_log2):
    npl = np.ascontiguousarray(npl, dtype=np.uint32)
    qw = np.zeros(int(npl[-1]), dtype=np.uint64)
    load_oracle().oracle_quant_weights_scalable(_ptr(npl, C.c_uint32), C.c_int(npl.size),
                                                C.c_uint64(num_points), C.c_int(min_log2),
                                                _ptr(qw, C.c_uint64))
    return qw


def emu_quant_weights_scalable(npl, num_points, min_log2):
    npl = np.ascontiguousarray(npl, dtype=np.uint32)
    n = int(npl[-1])
    qw = np.zeros(n, dtype=np.uint64)
    lib = load_emu()
    lib.emu_quant_weights_scalable.restype = C.c_int
    rc = lib.emu_quant_weights_scalable(_ptr(npl, C.c_uint32), C.c_int(npl.size),
                                        C.c_uint64(num_points), C.c_int(min_log2), C.c_int(n),
                                        _ptr(qw, C.c_uint64))
    assert rc == 0
    return qw



# ---- recolouring (attribute transfer) ---------------------------------------

class RecolourParams(C.Structure):
    _fields_ = [("dist_offset_fwd", C.c_double), ("dist_offset_bwd", C.c_double),
                ("max_geometry_dist2_fwd", C.c_double), ("max_geometry_dist2_bwd", C.c_double),
                ("max_attribute_dist2_fwd", C.c_double), ("max_attribute_dist2_bwd", C.c_double),
                ("search_range", C.c_int32), ("num_neighbours_fwd", C.c_int32),
                ("num_neighbours_bwd", C.c_int32), ("use_dist_weighted_avg_fwd", C.c_int32),
                ("use_dist_weighted_avg_bwd", C.c_int32),
                ("skip_avg_if_identical_source_point_present_fwd", C.c_int32),
                ("skip_avg_if_identical_source_point_present_bwd", C.c_int32),
                ("reserved", C.c_int32)]


def make_recolour_params(**kw):
    """defaults = tmc3/TMC3.cpp:1500-1551"""
    p = RecolourParams(4., 4., 1000., 1000., 1000., 1000., 1, 8, 1, 1, 1, 1, 0, 0)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _run_recolour(fn, params, sxyz, sattr, scale, off, txyz, bitdepth):
    sxyz = np.ascontiguousarray(sxyz, dtype=np.int32)
    sattr = np.ascontiguousarray(sattr, dtype=np.int32)
    txyz = np.ascontiguousarray(txyz, dtype=np.int32)
    if sattr.ndim == 1:
        sattr = sattr[:, None]
    a = sattr.shape[1]
    out = np.zeros((txyz.shape[0], a), dtype=np.int32)
    o = np.ascontiguousarray(off, dtype=np.int32)
    rc = fn(C.byref(params), _ptr(sxyz, C.c_int32), _ptr(sattr, C.c_int32), C.c_int(a),
            C.c_int(sxyz.shape[0]), C.c_double(scale), _ptr(o, C.c_int32), _ptr(txyz, C.c_int32),
            C.c_int(txyz.shape[0]), C.c_int(bitdepth), _ptr(out, C.c_int32))
    assert rc == 0, rc
    return out


def oracle_recolour(params, sxyz, sattr, scale, off, txyz, bitdepth=8):
    return _run_recolour(load_oracle().oracle_recolour, params, sxyz, sattr, scale, off, txyz, bitdepth)


def emu_recolour(params, sxyz, sattr, scale, off, txyz, bitdepth=8):
    return _run_recolour(load_emu().emu_recolour, params, sxyz, sattr, scale, off, txyz, bitdepth)


_recolourref = None


def recolourref_available():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libtmc13_recolour.so"))


@taped(by_value=True)
def ref_recolour(params, sxyz, sattr, scale, off, txyz, bitdepth=8):
    global _recolourref
    if _recolourref is None:
        _recolourref = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "libtmc13_recolour.so"))
    return _run_recolour(_recolourref.ref_recolour, params, sxyz, sattr, scale, off, txyz, bitdepth)


def coded_geometry(xyz, scale):
    """the geometry an encoder with lossy, duplicate-merging geometry coding would
    code: positions scaled, rounded, made unique (encoder.cpp quantizePositionsUniq)"""
    q = np.rint(xyz.astype(np.float64) * scale).astype(np.int32)
    return np.ascontiguousarray(np.unique(q, axis=0))
