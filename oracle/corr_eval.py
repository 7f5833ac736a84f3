"""ctypes binding of oracle/libvwcorreval.so: the CorrEval oracle (vw_corr_eval_oracle.h).
Test infrastructure only.  Images are (rows, cols, 2) float32 {value, valid} or 2-D float32 (all valid); the
disparity is (rows, cols, 3) float32 {dx, dy, valid}; the result is (rows, cols, 2) float32 {value, valid}."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SRC = ("vw_corr_eval_oracle.c",)
# the flags of oracle/Makefile (reference optimisation level, no FMA contraction)
_CFLAGS = ["-O3", "-std=c11", "-msse4.1", "-ffp-contract=off", "-fopenmp", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-parameter"]

METRICS = {"ncc": 0, "stddev": 1, "parabola_curvature": 2, "cramer_rao": 3}


def build(force=False):
    so = os.path.join(_HERE, "libvwcorreval.so")
    deps = [os.path.join(_HERE, f) for f in _SRC + ("vw_corr_eval_oracle.h", "corr_eval.py")]
    if force or not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        tmp = so + f".{os.getpid()}.tmp"
        subprocess.check_call(["gcc"] + _CFLAGS + ["-shared", "-o", tmp] + [os.path.join(_HERE, f) for f in _SRC] + ["-lm"])
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        P, I, F, Z = C.c_void_p, C.c_int, C.c_float, C.c_ssize_t
        L.vwce_corr_eval.argtypes = [P, I, I, Z, P, I, I, Z, P, Z, I, I, I, I, I, F, I, I, I, I, P, Z]
        L.vwce_right_origin.argtypes = [I, I, P, Z, I, I, I, I, I, F, I, I, I, I, C.POINTER(I), C.POINTER(I)]
        _LIB = L
    return _LIB


def masked(img):
    """(rows, cols, 2) float32 {value, valid}; a 2-D image is all valid."""
    a = np.asarray(img, dtype=np.float32)
    if a.ndim == 2:
        a = np.stack([a, np.ones_like(a)], axis=-1)
    return np.ascontiguousarray(a)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _metric(metric):
    if metric not in METRICS:
        raise ValueError(f"corr_eval: invalid metric {metric!r}")
    return METRICS[metric]


def _args(left, disparity, kernel_size, sample_rate, bbox):
    l = masked(left)
    d = np.ascontiguousarray(disparity, dtype=np.float32)
    rows, cols = l.shape[:2]
    if d.shape != (rows, cols, 3):
        raise ValueError("corr_eval: left image and disparity must have the same dimensions")
    if bbox is None:
        bbox = (0, 0, cols, rows)
    return l, d, tuple(int(v) for v in bbox)


def corr_eval(left, right, disparity, kernel_size, metric, sample_rate=1, round_to_int=False, prefilter_kernel_width=0.0,
              bbox=None):
    """CorrEval(...).prerasterize(bbox) as a (y1-y0, x1-x0, 2) array; bbox = (x0, y0, x1, y1), default the whole image."""
    l, d, b = _args(left, disparity, kernel_size, sample_rate, bbox)
    r = masked(right)
    out = np.zeros((max(b[3] - b[1], 0), max(b[2] - b[0], 0), 2), np.float32)
    rc = lib().vwce_corr_eval(_p(l), l.shape[1], l.shape[0], l.shape[1], _p(r), r.shape[1], r.shape[0], r.shape[1],
                              _p(d), d.shape[1], int(kernel_size[0]), int(kernel_size[1]), _metric(metric), int(sample_rate),
                              int(bool(round_to_int)), float(prefilter_kernel_width), b[0], b[1], b[2], b[3],
                              _p(out), max(out.shape[1], 1))
    if rc:
        raise ValueError(f"corr_eval: rc={rc}")
    return out


def right_origin(left_shape, disparity, kernel_size, metric, sample_rate=1, round_to_int=False, prefilter_kernel_width=0.0,
                 bbox=None):
    """right_box.min() of prerasterize(bbox), or None when no sampled disparity of the bbox is valid."""
    d = np.ascontiguousarray(disparity, dtype=np.float32)
    rows, cols = left_shape[:2]
    b = (0, 0, cols, rows) if bbox is None else tuple(int(v) for v in bbox)
    ox, oy = C.c_int(), C.c_int()
    rc = lib().vwce_right_origin(cols, rows, _p(d), d.shape[1], int(kernel_size[0]), int(kernel_size[1]), _metric(metric),
                                 int(sample_rate), int(bool(round_to_int)), float(prefilter_kernel_width), b[0], b[1], b[2], b[3],
                                 C.byref(ox), C.byref(oy))
    if rc < 0:
        raise ValueError(f"right_origin: rc={rc}")
    return (ox.value, oy.value) if rc else None
