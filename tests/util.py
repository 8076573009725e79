"""Test helpers: ctypes access to the oracle (tests only!), ULP metrics, fixtures."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ORACLE_SO = ROOT / "oracle" / "liboracle.so"
REF_SO = ROOT / "oracle" / "_ref" / "libmagickref.so"
SHIM_DIR = ROOT / "oracle" / "_ref" / "shim"      # MagickCore shim harnesses (imagemagick_b200/shim/Makefile)

_fp = C.POINTER(C.c_float)
_sz, _d, _i, _l = C.c_size_t, C.c_double, C.c_int, C.c_long


def P(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_fp)


class OrcKernel(C.Structure):
    _fields_ = [("width", _sz), ("height", _sz), ("x", _l), ("y", _l), ("values", C.POINTER(_d)),
                ("minimum", _d), ("maximum", _d), ("negative_range", _d), ("positive_range", _d), ("type", _i)]

    def array(self):
        n = self.width * self.height
        return np.array([self.values[i] for i in range(n)]).reshape(self.height, self.width)


# oracle kernel type ids (oracle.h)
ORC_K = dict(blur=0, gaussian=1, disk=2, square=3, diamond=4, octagon=5, plus=6, cross=7, rectangle=8)

_oracle = None
_ref = None


def oracle() -> C.CDLL:
    global _oracle
    if _oracle is None:
        o = C.CDLL(str(ORACLE_SO))
        for f in (o.orc_blur, o.orc_gaussian_blur):
            f.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        o.orc_unsharp.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d, _d, _d]
        o.orc_sharpen.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        o.orc_motion_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d, _d]
        o.orc_bilateral_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _sz, _sz, _d, _d]
        o.orc_rotational_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _d]
        o.orc_statistic.argtypes = [_fp, _fp, _sz, _sz, _i, _i, _sz, _sz]
        o.orc_edge.argtypes = [_fp, _fp, _sz, _sz, _i, _d]
        o.orc_emboss.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        o.orc_emboss_kernel.argtypes = [_d, _d, C.POINTER(OrcKernel)]
        o.orc_equalize.argtypes = [_fp, _sz, _sz, _i, _i]
        o.orc_resize.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz, _i]
        o.orc_resize_ex.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz, _i, C.c_void_p]
        o.orc_filter_weight_ex.argtypes = [_i, C.c_void_p, _d]
        o.orc_filter_weight_ex.restype = _d
        o.orc_filter_support_ex.argtypes = [_i, C.c_void_p]
        o.orc_filter_support_ex.restype = _d
        o.orc_colorspace.argtypes = [_fp, _sz, _sz, _i, _i, _i]
        o.orc_colorspace_ex.argtypes = [_fp, _sz, _sz, _i, _i, _i, C.c_void_p]
        o.orc_log_table.argtypes = [_i, C.c_void_p, _fp]
        o.orc_log_table.restype = None
        o.orc_ycc_table.argtypes = [_fp]
        o.orc_ycc_table.restype = None
        o.orc_sample.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz]
        o.orc_scale.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz]
        o.orc_selective_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d, _d]
        o.orc_adaptive_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        o.orc_adaptive_sharpen.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        o.orc_thumbnail.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz]
        o.orc_kernel_builtin.argtypes = [_i, _d, _d, _d, _d, C.POINTER(OrcKernel)]
        o.orc_kernel_user.argtypes = [_sz, _sz, _l, _l, C.POINTER(_d), C.POINTER(OrcKernel)]
        o.orc_kernel_free.argtypes = [C.POINTER(OrcKernel)]
        o.orc_morphology_apply.argtypes = [_fp, _fp, _sz, _sz, _i, _i, _l, C.POINTER(OrcKernel), _i, _d]
        o.orc_morphology_primitive.argtypes = [_fp, _fp, _sz, _sz, _i, _i, C.POINTER(OrcKernel), _d]
        o.orc_morphology_primitive.restype = _l
        o.orc_filter_weight.argtypes = [_i, _d]
        o.orc_filter_weight.restype = _d
        o.orc_filter_support.argtypes = [_i]
        o.orc_filter_support.restype = _d
        o.orc_optimal_kernel_width_1d.argtypes = [_d, _d]
        o.orc_optimal_kernel_width_1d.restype = _sz
        o.orc_optimal_kernel_width_2d.argtypes = [_d, _d]
        o.orc_optimal_kernel_width_2d.restype = _sz
        o.orc_threshold.argtypes = [_fp, _sz, _sz, _i, _i, C.POINTER(_d)]
        o.orc_set_threads.argtypes = [_i]
        _oracle = o
    return _oracle


def ref() -> C.CDLL:
    """The real reference (ImageMagick compiled from source); only exists where
    oracle/_ref has been built (this container / shipped prebuilt to the GPU box)."""
    global _ref
    if _ref is None:
        r = C.CDLL(str(REF_SO))
        for f in (r.ref_blur, r.ref_gaussian_blur):
            f.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        r.ref_unsharp.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d, _d, _d]
        r.ref_sharpen.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        r.ref_motion_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d, _d]
        r.ref_bilateral_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _sz, _sz, _d, _d]
        r.ref_rotational_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _d]
        r.ref_statistic.argtypes = [_fp, _fp, _sz, _sz, _i, _i, _sz, _sz]
        r.ref_edge.argtypes = [_fp, _fp, _sz, _sz, _i, _d]
        r.ref_emboss.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        r.ref_equalize.argtypes = [_fp, _sz, _sz, _i, _i]
        r.ref_convolve.argtypes = [_fp, _fp, _sz, _sz, _i, C.c_char_p]
        r.ref_morphology.argtypes = [_fp, _fp, _sz, _sz, _i, _i, _l, C.c_char_p]
        r.ref_resize.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz, _i]
        r.ref_resize_defines.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz, _i, C.c_char_p]
        r.ref_colorspace.argtypes = [_fp, _sz, _sz, _i, _i, _i]
        r.ref_colorspace_defines.argtypes = [_fp, _sz, _sz, _i, _i, _i, C.c_char_p]
        r.ref_sample.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz]
        r.ref_scale.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz]
        r.ref_selective_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d, _d]
        r.ref_adaptive_blur.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        r.ref_adaptive_sharpen.argtypes = [_fp, _fp, _sz, _sz, _i, _d, _d]
        r.ref_thumbnail.argtypes = [_fp, _sz, _sz, _i, _fp, _sz, _sz]
        r.ref_kernel.argtypes = [C.c_char_p, _i, C.POINTER(_d), _sz, C.POINTER(_sz), C.POINTER(_sz),
                                 C.POINTER(_l), C.POINTER(_l)]
        r.ref_threshold.argtypes = [_fp, _sz, _sz, _i, _i, _d, C.c_char_p]
        r.ref_version.restype = C.c_char_p
        r.ref_set_threads.argtypes = [_i]
        _ref = r
    return _ref


def ref_kernel(string: str, idx: int = 0):
    vals = (_d * 65536)()
    kw, kh, kx, ky = _sz(), _sz(), _l(), _l()
    rc = ref().ref_kernel(string.encode(), idx, vals, 65536, C.byref(kw), C.byref(kh), C.byref(kx), C.byref(ky))
    if rc:
        return None
    return np.array(vals[: kw.value * kh.value]).reshape(kh.value, kw.value), kx.value, ky.value


# ---- the reference's outputs, stored ----------------------------------------------------------------------------------
# Tests that compare with the reference read what it computed from REF_GOLDEN, so they run without the reference tree.
# A call is identified by the function name, its arguments (input pixels by content) and how it is compared; what is
# stored is a 64-bit digest of the return code and of the output with every float32 mapped to its sign-magnitude
# integer (the relation max_ulp(a, b) == 0 is equality of those integers) or, for exact_bits, to its bit pattern; for
# ref_output() and stored_ref_kernel(), the arrays themselves.
# MB200_RECORD_REF_OUTPUTS=1 runs the real library (oracle/_ref) instead and checks against it;
# tests/golden/make_ref_outputs.py then writes what it returned (save_recording()).
REF_GOLDEN = ROOT / "tests" / "golden" / "ref_outputs.npz"
RECORD = os.environ.get("MB200_RECORD_REF_OUTPUTS") == "1"
REGENERATE = ("tests/golden/make_ref_outputs.py (needs oracle/_ref/libmagickref.so; it also runs this comparison against "
              "the live library, element by element)")
OUT = object()              # argument placeholder: the output buffer


class InOut:
    """Argument placeholder: an output buffer that starts as a copy of `a` (operators that work in place)."""

    def __init__(self, a: np.ndarray):
        self.a = a


_store = None


def save_recording():
    """Writes what the recording run returned to REF_GOLDEN.  Digests go into two uint64 columns (call, output), sorted
    by call; arrays are stored under their own names."""
    assert RECORD and _store
    digests = sorted((int(k[2:], 16), int(v, 16)) for k, v in _store.items() if k.startswith("d:"))
    arrays = {k: v for k, v in _store.items() if not k.startswith("d:")}
    np.savez_compressed(REF_GOLDEN, digests=np.array(digests, np.uint64).reshape(-1, 2), **arrays)


def _golden():
    global _store
    if _store is None:
        if RECORD:
            _store = {}
        else:
            with np.load(REF_GOLDEN) as z:
                _store = {k: z[k] for k in z.files if k != "digests"}
                _store.update((f"d:{int(k):016x}", f"{int(v):016x}") for k, v in z["digests"])
    return _store


def _hash(*parts) -> str:
    h = hashlib.blake2b(digest_size=8)
    for p in parts:
        if isinstance(p, InOut):
            p = ("inout", p.a)
        if isinstance(p, tuple):
            h.update(_hash(*p).encode())
        elif isinstance(p, np.ndarray):
            h.update(repr((p.dtype.str, p.shape)).encode())
            h.update(np.ascontiguousarray(p).tobytes())
        else:
            if isinstance(p, (np.integer, np.floating)):
                p = p.item()
            h.update(repr("out" if p is OUT else p).encode())
    return h.hexdigest()


def _live_call(fn, args, out_shape):
    out = None
    call = []
    for a in args:
        if a is OUT:
            out = np.empty(out_shape, np.float32)
            a = out
        elif isinstance(a, InOut):
            out = a = a.a.copy()
        call.append(P(a) if isinstance(a, np.ndarray) else a)
    return getattr(ref(), fn)(*call), out


def _comparable(a: np.ndarray, mode: str) -> np.ndarray:
    """The integers whose equality is the comparison: "bits" the float32 bit patterns; "ulp" the sign-magnitude order
    (max_ulp == 0); "nan" the same with every NaN mapped to one value."""
    i = np.ascontiguousarray(a, np.float32).view(np.int32).astype(np.int64)
    if mode == "bits":
        return i
    k = np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.where(np.isnan(a), np.int64(1) << 40, k) if mode == "nan" else k


def expect_ref(got, fn: str, *args, rc: int = 0, nan_equal: bool = False, exact_bits: bool = False,
               threads: int = 0) -> None:
    """Asserts that the reference's `fn(*args)` returned `rc` and wrote `got`: max_ulp == 0; with nan_equal, NaN wherever
    the reference has NaN, in any encoding; with exact_bits, the same float32 bit patterns.  `got` None: only the
    return code is compared.  `threads`: the reference's thread count for the call."""
    mode = "rc" if got is None else "bits" if exact_bits else "nan" if nan_equal else "ulp"
    key = "d:" + _hash(fn, threads, mode, *args)
    if RECORD:
        if threads:
            ref().ref_set_threads(threads)
        want_rc, want = _live_call(fn, args, None if got is None else got.shape)
        _golden()[key] = _output_digest(want_rc, want, mode)
        assert want_rc == rc, (fn, want_rc)
        if got is not None:
            d = _comparable(got, mode) != _comparable(want, mode)
            assert not d.any(), (fn, f"{int(d.sum())} elements differ, first at {np.argwhere(d)[0].tolist()}",
                                 f"max ULP {max_ulp(got, want)}")
        return
    stored = _golden().get(key)
    assert stored is not None, f"{fn}: no stored reference output for this call; regenerate with {REGENERATE}"
    assert stored == _output_digest(rc, got, mode), \
        f"{fn}: differs from the reference's output; where and by how much: {REGENERATE}"


def _output_digest(rc: int, out, mode: str) -> str:
    return _hash(rc, None if mode == "rc" else _comparable(out, mode))


def ref_output(fn: str, *args, shape) -> np.ndarray:
    """The array the reference's `fn(*args)` wrote into its OUT argument of the given shape (asserting it returned 0)."""
    key = "a:" + _hash(fn, shape, *args)
    if RECORD:
        rc, out = _live_call(fn, args, shape)
        assert rc == 0, (fn, rc)
        _golden()[key] = out
    out = _golden().get(key)
    assert out is not None, f"{fn}: no stored reference output for this call; regenerate with {REGENERATE}"
    return out


def stored_ref_kernel(string: str, idx: int = 0):
    """ref_kernel() as stored: the reference's kernel list element `idx` for a kernel string as (values, x, y), None
    past the end of the list."""
    key = "k:" + _hash(string, idx)
    if RECORD:
        k = ref_kernel(string, idx)
        _golden()[key] = np.zeros(0) if k is None else np.concatenate([[k[1], k[2], k[0].shape[1]], k[0].ravel()])
    flat = _golden().get(key)
    assert flat is not None, f"{string}: no stored reference kernel; regenerate with {REGENERATE}"
    if flat.size == 0:
        return None
    x, y, w = (int(v) for v in flat[:3])
    return flat[3:].reshape(-1, w), x, y


def orc_kernel(kind: str, rho=0.0, sigma=0.0, xi=0.0, psi=0.0) -> OrcKernel:
    k = OrcKernel()
    rc = oracle().orc_kernel_builtin(ORC_K[kind], rho, sigma, xi, psi, C.byref(k))
    assert rc == 0, (kind, rho, sigma, xi, psi)
    return k


def orc_kernel_from_array(values: np.ndarray, x: int, y: int) -> OrcKernel:
    v = np.ascontiguousarray(values, dtype=np.float64)
    k = OrcKernel()
    rc = oracle().orc_kernel_user(v.shape[1], v.shape[0], x, y, v.ctypes.data_as(C.POINTER(_d)), C.byref(k))
    assert rc == 0
    return k


def orc_morphology(src: np.ndarray, method: int, iterations: int, kernels, bias=0.0) -> np.ndarray:
    h, w, ch = src.shape
    arr = (OrcKernel * len(kernels))(*kernels)
    dst = np.empty_like(src)
    rc = oracle().orc_morphology_apply(P(src), P(dst), w, h, ch, method, iterations, arr, len(kernels), bias)
    assert rc == 0
    return dst


def ulp_distance(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Per-element distance in float32 ULPs (sign-magnitude ordered integers)."""
    assert a.shape == b.shape and a.dtype == np.float32 and b.dtype == np.float32
    ai = a.view(np.int32).astype(np.int64)
    bi = b.view(np.int32).astype(np.int64)
    ai = np.where(ai < 0, -(ai & 0x7FFFFFFF), ai)
    bi = np.where(bi < 0, -(bi & 0x7FFFFFFF), bi)
    return np.abs(ai - bi)


def max_ulp(a, b) -> int:
    return int(ulp_distance(np.ascontiguousarray(a), np.ascontiguousarray(b)).max())


class FilterOptions(C.Structure):
    """mb200_filter_options == orc_filter_options: the "filter:*" expert settings as values."""
    _fields_ = [("set", C.c_uint), ("window", C.c_int), ("keep_filter", C.c_int), ("lobes", C.c_long), ("sigma", C.c_double),
                ("kaiser_beta", C.c_double), ("blur", C.c_double), ("support", C.c_double), ("win_support", C.c_double),
                ("b", C.c_double), ("c", C.c_double)]

    BITS = {"window": 1, "sigma": 2, "kaiser_beta": 4, "lobes": 8, "blur": 16, "support": 32, "win_support": 64, "b": 128, "c": 256}

    @classmethod
    def of(cls, **kw):
        o = cls()
        for k, v in kw.items():
            if k == "keep_filter":
                o.keep_filter = int(v)
                continue
            setattr(o, k, v)
            o.set |= cls.BITS[k]
        return o


class ColorspaceOptions(C.Structure):
    """mb200_colorspace_options == orc_colorspace_options: the image settings TransformImageColorspace reads, as values."""
    _fields_ = [("set", C.c_uint), ("illuminant", C.c_int), ("white_luminance", C.c_double),
                ("film_gamma", C.c_double), ("reference_black", C.c_double), ("reference_white", C.c_double)]

    BITS = {"illuminant": 1, "white_luminance": 2, "film_gamma": 4, "reference_black": 8, "reference_white": 16}
    ILLUMINANTS = {"A": 0, "B": 1, "C": 2, "D50": 3, "D55": 4, "D65": 5, "D75": 6, "E": 7, "F2": 8, "F7": 9, "F11": 10}

    @classmethod
    def of(cls, **kw):
        o = cls()
        for k, v in kw.items():
            setattr(o, k, cls.ILLUMINANTS[v] if k == "illuminant" else v)
            o.set |= cls.BITS[k]
        return o


def ulp_or_noise(a, b, tiny=1.0e-6) -> np.ndarray:
    """ULP distance, except where BOTH values are rounding noise around zero (|v| < tiny Quantum units = 1.5e-11 of full
    scale): a component the reference computes as the difference of two equal numbers -- e.g. the red channel of an
    Adobe98 blue taken to sRGB, whose primaries coincide -- has no significant bits to compare; 0 is returned there."""
    d = ulp_distance(np.ascontiguousarray(a), np.ascontiguousarray(b))
    noise = (np.abs(a) < tiny) & (np.abs(b) < tiny)
    return np.where(noise, 0, d)


def frac_exact(a, b) -> float:
    return float((ulp_distance(np.ascontiguousarray(a), np.ascontiguousarray(b)) == 0).mean())


def make_image(w: int, h: int, ch: int, seed: int = 42, kind: str = "noise") -> np.ndarray:
    """Seeded synthetic pixel cache (raw Quantum floats 0..65535).
    kind: noise | alpha_blocks (fully transparent / opaque regions, exercises
    PerceptibleReciprocal) | gradient | hdr (values outside 0..QuantumRange, negatives)."""
    rng = np.random.default_rng(seed)
    a = (rng.random((h, w, ch), dtype=np.float32) * np.float32(65535.0)).astype(np.float32)
    if kind == "alpha_blocks" and ch in (2, 4):
        a[: h // 2, : w // 2, ch - 1] = 0.0
        a[h // 2:, w // 2:, ch - 1] = 65535.0
        a[h // 3: h // 3 + 2, :, ch - 1] = 1.0
    elif kind == "gradient":
        yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
        for c in range(ch):
            a[..., c] = ((xx * (c + 1) + yy * 3) % 256) * 257.0
    elif kind == "hdr":
        a = (a - 20000.0) * 1.7
    elif kind == "binary":
        a = np.where(a > 40000.0, np.float32(65535.0), np.float32(0.0)).astype(np.float32)
    return np.ascontiguousarray(a)


def parse_thresholds(spec: str):
    """The ParseGeometry step of Black/WhiteThresholdImage (threshold.c:955-985) for the
    'v[,v[,v[,v]]][%]' forms: returns [red, green, blue, alpha] in Quantum units."""
    pct = "%" in spec
    vals = [float(t) for t in spec.replace("%", "").split(",") if t.strip()]
    rho = vals[0]
    thr = [rho, vals[1] if len(vals) > 1 else rho, vals[2] if len(vals) > 2 else rho,
           vals[3] if len(vals) > 3 else 100.0]
    if pct:
        thr = [t * (65535.0 / 100.0) for t in thr]
    return thr


def orc_threshold(src: np.ndarray, op: int, thr) -> np.ndarray:
    h, w, ch = src.shape
    out = src.copy()
    arr = (_d * 4)(*([float(t) for t in thr] + [0.0] * (4 - len(thr))))
    assert oracle().orc_threshold(P(out), w, h, ch, op, arr) == 0
    return out


# ---- run-time switches of the product library (mb200_set_option): restored after every test by conftest.py
_touched_options = {}


def get_option(name: str) -> int:
    from imagemagick_b200 import _lib
    v = C.c_int(0)
    _lib.check(_lib.load().mb200_get_option(name.encode(), C.byref(v)))
    return int(v.value)


def set_option(name: str, value: int) -> None:
    from imagemagick_b200 import _lib
    if name not in _touched_options:
        _touched_options[name] = get_option(name)       # the process default (environment), restored after the test
    _lib.check(_lib.load().mb200_set_option(name.encode(), int(value)))


def reset_options() -> None:
    if not _touched_options:
        return
    from imagemagick_b200 import _lib
    for name, value in list(_touched_options.items()):
        _lib.load().mb200_set_option(name.encode(), value)
    _touched_options.clear()
