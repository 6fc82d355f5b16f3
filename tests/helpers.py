"""Checker-side helpers: drive the compiled reference (oracle/_ref) and the oracle restatement.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline legs import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from jpeg2png_b200 import abi
from jpeg2png_b200.synth import CoefImage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, 'oracle')
REF_SIMD = os.path.join(ORACLE_DIR, '_ref', 'libref_compute.so')
REF_C = os.path.join(ORACLE_DIR, '_ref', 'libref_compute_c.so')
ORACLE_LIB = os.path.join(ORACLE_DIR, 'liboracle.so')
REFERENCE_SRC = '/root/reference'

_cache = {}


def build_oracle_libs() -> None:
    """Compile the checker libraries (never the product)."""
    subprocess.run(['make', '-C', ORACLE_DIR, 'all'], check=True, capture_output=True)


def have_ref() -> bool:
    return os.path.exists(REF_SIMD)


def _load(path):
    if path not in _cache:
        if not os.path.exists(path):
            build_oracle_libs()
        _cache[path] = C.CDLL(path, mode=C.RTLD_LOCAL)
    return _cache[path]


def load_ref(simd: bool = True) -> C.CDLL:
    lib = _load(REF_SIMD if simd else REF_C)
    lib.compute.restype = None
    lib.compute.argtypes = [C.c_uint, C.POINTER(abi.Coef), C.POINTER(abi.Logger),
                            C.POINTER(abi.ProgressBar), C.c_float, C.POINTER(C.c_float), C.c_uint]
    lib.idct8x8s.argtypes = [C.c_void_p]
    lib.dct8x8s.argtypes = [C.c_void_p]
    lib.ref_glue_max_threads.restype = C.c_int
    lib.ref_glue_set_threads.argtypes = [C.c_int]
    return lib


def load_oracle() -> C.CDLL:
    lib = _load(ORACLE_LIB)
    lib.oracle_compute.restype = None
    lib.oracle_compute.argtypes = [C.c_uint, C.POINTER(abi.Coef), C.c_float, C.POINTER(C.c_float),
                                   C.c_uint, C.POINTER(C.c_double)]
    lib.oracle_idct8x8.argtypes = [C.c_void_p]
    lib.oracle_dct8x8.argtypes = [C.c_void_p]
    lib.oracle_decode_coefficients.argtypes = [C.POINTER(abi.Coef)]
    lib.oracle_ycc_to_rgb.argtypes = [C.c_uint, C.c_uint, C.c_uint, C.c_void_p, C.c_uint, C.c_void_p,
                                      C.c_uint, C.c_void_p, C.c_uint, C.c_void_p]
    return lib


def decode_planes(img: CoefImage, channels=(0, 1, 2)):
    """Conventional decode (jpeg.c:83-92 + jpeg2png.c:131-139) with the oracle: list of (h,w) float32."""
    lib = load_oracle()
    ca = abi.CoefArray(img, list(channels))
    out = []
    for k in range(ca.n):
        lib.oracle_decode_coefficients(C.byref(ca.arr[k]))
        out.append(ca.result(k).copy())
    ca.release()
    return out


def _pw(pweight, n):
    arr = (C.c_float * n)(*[float(x) for x in pweight[:n]])
    return arr


def run_compute(kind: str, img: CoefImage, channels, weight, pweight, iterations, fdata=None,
                want_log=False, timer=None):
    """Run one `compute()`-shaped solve on planes `channels` of img.

    kind: 'ref' (SIMD reference build), 'ref_c' (scalar reference build), 'oracle', 'product'.
    pweight: one value per entry of `channels`.  Returns list of (H,W) float32 planes
    (and the objective log for kind == 'oracle' when want_log).
    """
    channels = list(channels)
    if fdata is None:
        fdata = decode_planes(img, channels)
    ca = abi.CoefArray(img, channels, fdata)
    n = len(channels)
    pw = _pw(list(pweight), n)
    log = None
    import time as _time
    t0 = _time.perf_counter()
    if kind in ('ref', 'ref_c'):
        lib = load_ref(simd=(kind == 'ref'))
        lg = abi.Logger(None, b'', 0, 0)
        lib.compute(n, ca.arr, C.byref(lg), None, C.c_float(weight), pw, iterations)
    elif kind == 'oracle':
        lib = load_oracle()
        logbuf = (C.c_double * (4 * max(iterations, 1)))() if want_log else None
        lib.oracle_compute(n, ca.arr, C.c_float(weight), pw, iterations, logbuf)
        if want_log:
            log = np.array(logbuf[:4 * iterations], dtype=np.float64).reshape(iterations, 4)
    elif kind == 'product':
        lib = abi.load_product()
        lg = abi.Logger(None, b'', 0, 0)
        lib.compute(n, ca.arr, C.byref(lg), None, C.c_float(weight), pw, iterations)
    else:
        raise ValueError(kind)
    if timer is not None:
        timer['seconds'] = _time.perf_counter() - t0      # the compute() call only
    out = [ca.result(k).copy() for k in range(n)]
    ca.release()
    return (out, log) if want_log else out


def transform8x8(fn, block) -> np.ndarray:
    """Apply an in-place 8x8 transform (dct8x8s / idct8x8s and their restatements) to a copy of block."""
    p = abi.alloc_floats(64)
    try:
        C.memmove(p, np.ascontiguousarray(block, np.float32).ctypes.data, 256)
        fn(p)
        out = np.empty(64, np.float32)
        C.memmove(out.ctypes.data, p, 256)
    finally:
        abi.free_ptr(p)
    return out


def bits(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_bit_identical(a, b, what=''):
    for k, (p, q) in enumerate(zip(a, b)):
        assert p.shape == q.shape, f'{what} plane {k}: shape {p.shape} vs {q.shape}'
        diff = bits(p) != bits(q)
        if diff.any():
            idx = np.argwhere(diff)[0]
            raise AssertionError(
                f'{what} plane {k}: {int(diff.sum())} of {diff.size} samples differ in bits; first at '
                f'{tuple(idx)}: {p[tuple(idx)]!r} vs {q[tuple(idx)]!r}; max abs diff '
                f'{float(np.max(np.abs(p.astype(np.float64) - q.astype(np.float64))))}')
