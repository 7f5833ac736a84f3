"""ctypes binding of oracle/libvwsubpixel.so: the sub-pixel refinement oracle (vw_subpixel_oracle.h).
Test infrastructure only.  Disparities are (rows, cols, 3) float32 {dx, dy, valid}."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SRC = ("vw_oracle.c", "vw_sgm_oracle.c", "vw_subpixel_oracle.c")
# the flags of oracle/Makefile (reference optimisation level, no FMA contraction)
_CFLAGS = ["-O3", "-std=c11", "-msse4.1", "-ffp-contract=off", "-fopenmp", "-fPIC", "-Wall", "-Wextra", "-Wno-unused-parameter"]

SUBPIXEL_LUCAS_KANADE, SUBPIXEL_FAST_AFFINE, SUBPIXEL_BAYES_EM, SUBPIXEL_PHASE = 0, 1, 2, 3


def build(force=False):
    so = os.path.join(_HERE, "libvwsubpixel.so")
    deps = [os.path.join(_HERE, f) for f in _SRC + ("vw_oracle.h", "vw_subpixel_oracle.h", "subpixel.py")]
    if force or not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        tmp = so + f".{os.getpid()}.tmp"
        subprocess.check_call(["gcc"] + _CFLAGS + ["-shared", "-o", tmp] + [os.path.join(_HERE, f) for f in _SRC] + ["-lm"])
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        P, I, F = C.c_void_p, C.c_int, C.c_float
        L.vwso_expf.argtypes, L.vwso_expf.restype = [F], F
        L.vwso_expf_array.argtypes = [P, I, P]
        L.vwso_spatial_weight.argtypes = [I, I, F, P]
        L.vwso_posv.argtypes = [I, P, P]
        L.vwso_derivative.argtypes = [P, I, I, I, P]
        L.vwso_bilinear.argtypes, L.vwso_bilinear.restype = [P, I, I, F, F], F
        L.vwso_disparity_subsample.argtypes = [P, I, I, P]
        L.vwso_disparity_upsample.argtypes = [P, I, I, P, I, I]
        L.vwso_subpixel_level.argtypes = [I, P, P, I, I, P, I, I, I, I, I, I, I, I, I, I]
        L.vwso_pyramid_subpixel.argtypes = [P, I, I, P, I, P, I, I, I, I, I, I, F, I, I, I, I, I, I, P]
        _LIB = L
    return _LIB


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _rc(rc, what):
    if rc == -2:
        raise NotImplementedError(f"{what}: algorithm not implemented")
    if rc:
        raise ValueError(f"{what}: rc={rc}")


def expf(x):
    x = _f32(x)
    out = np.empty_like(x)
    lib().vwso_expf_array(_p(x), x.size, _p(out))
    return out


def spatial_weight(kx, ky, two_sigma_sqr):
    out = np.empty((ky, kx), np.float32)
    lib().vwso_spatial_weight(kx, ky, float(two_sigma_sqr), _p(out))
    return out


def posv(A, b):
    """Returns (info, solution-or-unchanged b)."""
    A = _f32(A).copy()
    b = _f32(b).copy()
    info = lib().vwso_posv(b.size, _p(A), _p(b))
    return info, b


def derivative(img, dx):
    a = _f32(img)
    out = np.empty_like(a)
    lib().vwso_derivative(_p(a), a.shape[1], a.shape[0], 1 if dx else 0, _p(out))
    return out


def disparity_subsample(disp):
    d = _f32(disp)
    h, w = d.shape[:2]
    out = np.empty((1 + (h - 1) // 2, 1 + (w - 1) // 2, 3), np.float32)
    lib().vwso_disparity_subsample(_p(d), w, h, _p(out))
    return out


def disparity_upsample(disp, shape):
    d = _f32(disp)
    h, w = d.shape[:2]
    out = np.empty((shape[0], shape[1], 3), np.float32)
    lib().vwso_disparity_upsample(_p(d), w, h, _p(out), shape[1], shape[0])
    return out


def subpixel_level(algorithm, disp, left, right, kernel, roi=None, do_h=True, do_v=True):
    """One of subpixel_optimized_LK_2d / _affine_2d / _affine_2d_EM; returns the refined copy.
    roi = (x0, y0, x1, y1), default the whole image."""
    d = _f32(disp).copy()
    l, r = _f32(left), _f32(right)
    h, w = l.shape
    assert d.shape == (h, w, 3)
    if roi is None:
        roi = (0, 0, w, h)
    _rc(lib().vwso_subpixel_level(algorithm, _p(d), _p(l), w, h, _p(r), r.shape[1], r.shape[0], kernel[0], kernel[1],
                                  roi[0], roi[1], roi[2], roi[3], int(bool(do_h)), int(bool(do_v))), "subpixel_level")
    return d


def pyramid_subpixel(disp, left, right, kernel, prefilter_mode=0, prefilter_width=0.0, max_pyramid_levels=2,
                     algorithm=SUBPIXEL_BAYES_EM, bbox=None):
    d = _f32(disp)
    l, r = _f32(left), _f32(right)
    rows, cols = l.shape
    assert d.shape == (rows, cols, 3)
    if bbox is None:
        bbox = (0, 0, cols, rows)
    out = np.empty((bbox[3] - bbox[1], bbox[2] - bbox[0], 3), np.float32)
    _rc(lib().vwso_pyramid_subpixel(_p(d), cols, rows, _p(l), cols, _p(r), r.shape[1], r.shape[0], r.shape[1],
                                    kernel[0], kernel[1], prefilter_mode, float(prefilter_width),
                                    bbox[0], bbox[1], bbox[2], bbox[3], max_pyramid_levels, algorithm, _p(out)),
        "pyramid_subpixel")
    return out
