"""Python host-side mirror of the reference operator interface, over the C ABI (include/vwb200.h).

Names, argument order and error behaviour follow Vision Workbench:
  * calc_disparity            -- src/vw/Stereo/Correlation.h:50-57
  * PyramidCorrelationView    -- src/vw/Stereo/CorrelationView.h:35-193 (cols/rows/planes,
                                 prerasterize(bbox), rasterize(dest, bbox), operator() throws NoImplErr)
  * pyramid_correlate         -- src/vw/Stereo/CorrelationView.h:195-230
  * cross_corr_consistency_check, rm_outliers_using_thresh, disparity_cleanup_using_thresh,
    disparity_mask            -- src/vw/Stereo/Correlate.h:52-58, DisparityMap.h:318-442,97-253

There is no CPU path: every call goes to libvwb200.so (hand-written sm_100a kernels) and raises if
the library or a CUDA device is missing.  Inputs may be numpy arrays (staged through HBM by the
library) or torch CUDA tensors (used in place, results returned as torch CUDA tensors).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libvwb200.so")
_LIB = None

# vw::stereo::CostFunctionType (Stereo/CostFunctions.h:143-149)
ABSOLUTE_DIFFERENCE, SQUARED_DIFFERENCE, CROSS_CORRELATION, CENSUS_TRANSFORM, TERNARY_CENSUS_TRANSFORM = 0, 1, 2, 3, 4
# vw::stereo::PrefilterModeType (Stereo/PrefilterEnum.h:24-28)
PREFILTER_NONE, PREFILTER_LOG, PREFILTER_MEANSUB = 0, 1, 2
# vw::stereo::CorrelationAlgorithm (Stereo/CorrelationAlgorithms.h:29-35)
VW_CORRELATION_BM, VW_CORRELATION_SGM, VW_CORRELATION_MGM, VW_CORRELATION_FINAL_MGM = 0, 1, 2, 3
# SemiGlobalMatcher::SgmSubpixelMode (Stereo/SGM.h:93-99)
SUBPIXEL_NONE, SUBPIXEL_PARABOLA, SUBPIXEL_LINEAR, SUBPIXEL_POLY4, SUBPIXEL_COSINE, SUBPIXEL_LC_BLEND = 0, 1, 2, 3, 4, 5
# PyramidSubpixelView_Algorithm (Stereo/SubpixelView.h:35-40)
SUBPIXEL_LUCAS_KANADE, SUBPIXEL_FAST_AFFINE, SUBPIXEL_BAYES_EM, SUBPIXEL_PHASE = 0, 1, 2, 3
# CorrEval metrics (Stereo/CorrEval.h:88-90), VWB200_CORR_EVAL_*
CORR_EVAL_METRICS = {"ncc": 0, "stddev": 1, "parabola_curvature": 2, "cramer_rao": 3}


class VwError(RuntimeError):
    """Base of the vw::Exception mirror (Core/Exception.h:201-253)."""


class ArgumentErr(VwError):
    pass


class MathErr(VwError):
    pass


class LogicErr(VwError):
    pass


class NoImplErr(VwError):
    pass


class CudaErr(VwError):
    pass


class NoDeviceErr(VwError):
    pass


_ERR = {-1: ArgumentErr, -2: MathErr, -3: LogicErr, -4: NoImplErr, -5: CudaErr, -6: NoDeviceErr, -7: MemoryError}


class CorrParams(C.Structure):
    _fields_ = [("search_x0", C.c_int32), ("search_y0", C.c_int32), ("search_x1", C.c_int32), ("search_y1", C.c_int32),
                ("kernel_x", C.c_int32), ("kernel_y", C.c_int32), ("cost_type", C.c_int32),
                ("prefilter_mode", C.c_int32), ("prefilter_width", C.c_float),
                ("consistency_threshold", C.c_float), ("min_consistency_level", C.c_int32),
                ("filter_half_kernel", C.c_int32), ("max_pyramid_levels", C.c_int32), ("collar_size", C.c_int32),
                ("corr_timeout", C.c_int32), ("seconds_per_op", C.c_double),
                ("algorithm", C.c_int32), ("blob_filter_area", C.c_int32),
                ("sgm_subpixel_mode", C.c_int32), ("sgm_search_buffer_x", C.c_int32), ("sgm_search_buffer_y", C.c_int32),
                ("region_ul_x", C.c_int32), ("region_ul_y", C.c_int32), ("write_debug_images", C.c_int32),
                ("sgm_threads", C.c_int32), ("memory_limit_mb", C.c_double)]


class SgmParams(C.Structure):
    _fields_ = [("search_x", C.c_int32), ("search_y", C.c_int32), ("kernel_size", C.c_int32), ("cost_type", C.c_int32),
                ("ternary_threshold", C.c_int32), ("p1", C.c_int32), ("p2", C.c_int32), ("use_mgm", C.c_int32),
                ("subpixel_mode", C.c_int32), ("search_buffer_x", C.c_int32), ("search_buffer_y", C.c_int32),
                ("conserve_level", C.c_int32), ("memory_limit_mb", C.c_double), ("assumed_threads", C.c_int32),
                ("reserved", C.c_int32)]


class K1Stats(C.Structure):
    _fields_ = [("path", C.c_int32), ("launches", C.c_int32), ("kernel_ms", C.c_float), ("reserved", C.c_int32)]


def lib():
    """Load libvwb200.so.  Fails loudly if it has not been built (python -m visionworkbench_b200.build)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(_SO):
            raise ImportError(f"{_SO} is missing: build it with `python visionworkbench_b200/build.py` "
                              "(the engine has no CPU or PyTorch fallback)")
        L = C.CDLL(_SO)
        L.vwb200_last_error.restype = C.c_char_p
        L.vwb200_version.restype = C.c_char_p
        L.vwb200_kernel_launches.restype = C.c_longlong
        P, I, Z, F, D = C.c_void_p, C.c_int, C.c_ssize_t, C.c_float, C.c_double
        L.vwb200_calc_disparity.argtypes = [I, P, I, I, Z, P, I, I, Z, I, I, I, I, P, Z, I, P]
        L.vwb200_pyramid_down.argtypes = [P, I, I, Z, P, Z, I, P]
        L.vwb200_subsample_mask_by_two.argtypes = [P, I, I, Z, P, Z, I, P]
        L.vwb200_prefilter.argtypes = [P, I, I, Z, I, F, P, Z, I, P]
        L.vwb200_sgm_calc_disparity.argtypes = [P, I, I, Z, P, I, I, Z, I, I, I, I, I, P, Z, C.POINTER(I), C.POINTER(I), I, P]
        L.vwb200_sgm_calc_disparity_subpixel.argtypes = [P, I, I, Z, P, I, I, Z, I, I, I, I, I, I, P, Z, P, Z, C.POINTER(I), C.POINTER(I), I, P]
        L.vwb200_sgm_calc_disparity_ex.argtypes = [C.POINTER(SgmParams), P, I, I, Z, P, I, I, Z, P, Z, P, I, I, Z, P, I, I, Z, P, P, Z, P, Z, P,
                                                   C.POINTER(I), C.POINTER(I), I, P]
        L.vwb200_sgm_disp_bounds.argtypes = [C.POINTER(SgmParams), P, I, I, Z, P, Z, P, I, I, Z, I, I, P, I, P]
        L.vwb200_parabola_subpixel.argtypes = [P, I, I, P, Z, P, I, I, Z, I, I, I, F, I, I, I, I, P, Z, I, P]
        L.vwb200_pyramid_subpixel.argtypes = [P, I, I, P, Z, P, I, I, Z, I, I, I, F, I, I, I, I, P, Z, I, P, I, I]
        L.vwb200_subpixel_refine.argtypes = [I, P, I, I, Z, P, Z, P, I, I, Z, I, I, I, I, I, I, I, I, I, P]
        L.vwb200_last_subpixel_stats.argtypes = [C.POINTER(SubpixelStats)]
        L.vwb200_corr_eval.argtypes = [P, I, I, Z, P, I, I, Z, P, Z, I, I, I, I, I, F, I, I, I, I, P, Z, I, P]
        L.vwb200_cross_corr_consistency_check.argtypes = [P, I, I, Z, P, I, I, Z, F, I, P]
        L.vwb200_rm_outliers_using_thresh.argtypes = [P, I, I, I, I, D, D, P, I, P]
        L.vwb200_disparity_cleanup_using_thresh.argtypes = [P, I, I, I, I, D, D, P, I, P]
        L.vwb200_disparity_mask.argtypes = [P, I, I, P, P, I, I, P, I, P]
        L.vwb200_corr_create.argtypes = [C.POINTER(CorrParams), C.POINTER(P)]
        L.vwb200_corr_set_inputs.argtypes = [P, P, I, I, Z, P, I, I, Z, P, Z, P, Z, I]
        L.vwb200_corr_rasterize.argtypes = [P, I, I, I, I, P, Z, I, P]
        L.vwb200_corr_prerasterize.argtypes = [P, I, I, I, I, P, Z, I, P]
        L.vwb200_corr_set_lr_disp_diff.argtypes = [P, P, I, I, Z, I]
        L.vwb200_corr_num_levels.argtypes = [P, I, I]
        L.vwb200_corr_cols.argtypes = [P]
        L.vwb200_corr_rows.argtypes = [P]
        L.vwb200_corr_destroy.argtypes = [P]
        L.vwb200_corr_destroy.restype = None
        L.vwb200_last_k1_stats.argtypes = [C.POINTER(K1Stats)]
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        msg = lib().vwb200_last_error().decode("utf-8", "replace")
        raise _ERR.get(rc, VwError)(msg)


def device_count():
    return lib().vwb200_device_count()


def kernel_launches():
    return lib().vwb200_kernel_launches()


def last_k1_stats():
    s = K1Stats()
    lib().vwb200_last_k1_stats(C.byref(s))
    return {"path": "exact-int" if s.path == 0 else "general-fp64", "launches": s.launches, "kernel_ms": s.kernel_ms}


class SubpixelStats(C.Structure):
    _fields_ = [("levels", C.c_longlong), ("fixpoint_rounds", C.c_longlong), ("pixels", C.c_longlong),
                ("pixels_reevaluated", C.c_longlong), ("window_evaluations", C.c_longlong), ("lane_slots", C.c_longlong)]


def last_subpixel_stats():
    """Counters of this thread's last sub-pixel refinement call (vwb200_last_subpixel_stats)."""
    s = SubpixelStats()
    _check(lib().vwb200_last_subpixel_stats(C.byref(s)))
    d = {k: getattr(s, k) for k, _ in SubpixelStats._fields_}
    d["simt_efficiency"] = s.window_evaluations / s.lane_slots if s.lane_slots else 0.0
    return d


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def calc_disparity(cost_type, left_in, right_in, search_volume, kernel_size):
    """vw::stereo::calc_disparity (Stereo/Correlation.h:50-57) on already-cropped rasters.

    left_in : (H+ky-1, W+kx-1) float32;  right_in: at least (H+ky-1+sy-1, W+kx-1+sx-1).
    search_volume = (sx, sy), kernel_size = (kx, ky).
    Returns int32 (H, W, 3) {dx, dy, valid} -- PixelMask<Vector2i>.
    """
    sx, sy = search_volume
    kx, ky = kernel_size
    if _is_torch(left_in):
        import torch
        l = left_in.contiguous().float()
        r = right_in.contiguous().float()
        H, W = l.shape[0] - ky + 1, l.shape[1] - kx + 1
        if H <= 0 or W <= 0:
            raise ArgumentErr("calc_disparity: Kernel size too large of active region.")
        out = torch.empty((H, W, 3), dtype=torch.int32, device=l.device)
        _check(lib().vwb200_calc_disparity(cost_type, l.data_ptr(), l.shape[1], l.shape[0], l.stride(0),
                                           r.data_ptr(), r.shape[1], r.shape[0], r.stride(0),
                                           sx, sy, kx, ky, out.data_ptr(), W, 1, _stream_ptr()))
        return out
    l, r = _np(left_in, np.float32), _np(right_in, np.float32)
    H, W = l.shape[0] - ky + 1, l.shape[1] - kx + 1
    if H <= 0 or W <= 0:
        raise ArgumentErr("calc_disparity: Kernel size too large of active region.")
    out = np.empty((H, W, 3), np.int32)
    _check(lib().vwb200_calc_disparity(cost_type, l.ctypes.data, l.shape[1], l.shape[0], l.shape[1],
                                       r.ctypes.data, r.shape[1], r.shape[0], r.shape[1],
                                       sx, sy, kx, ky, out.ctypes.data, W, 0, None))
    return out


def calc_disparity_sgm(left_in, right_in, search_volume, kernel_size, p1=0, p2=0):
    """vw::stereo::calc_disparity_sgm (Stereo/SGM.cc:167-230) for CENSUS_TRANSFORM / SGM on the cropped left_region and
    right_region rasters: the search box is [0, search_volume] (inclusive) for every pixel.  kernel_size 3, 5, 7 or 9.
    Returns int32 (out_h, out_w, 3) {dx, dy, valid} (the raster of SGM.cc:2397-2420: the borders the kernel and the search
    cannot cover are cropped)."""
    sx, sy = search_volume
    ow, oh = C.c_int(0), C.c_int(0)
    if _is_torch(left_in):
        import torch
        l = left_in.contiguous().float()
        r = right_in.contiguous().float()
        _check(lib().vwb200_sgm_calc_disparity(l.data_ptr(), l.shape[1], l.shape[0], l.stride(0), r.data_ptr(), r.shape[1], r.shape[0], r.stride(0),
                                               sx, sy, kernel_size, p1, p2, None, 0, C.byref(ow), C.byref(oh), 1, None))
        out = torch.empty((max(oh.value, 0), max(ow.value, 0), 3), dtype=torch.int32, device=l.device)
        _check(lib().vwb200_sgm_calc_disparity(l.data_ptr(), l.shape[1], l.shape[0], l.stride(0), r.data_ptr(), r.shape[1], r.shape[0], r.stride(0),
                                               sx, sy, kernel_size, p1, p2, out.data_ptr(), ow.value, C.byref(ow), C.byref(oh), 1, _stream_ptr()))
        return out
    l, r = _np(left_in, np.float32), _np(right_in, np.float32)
    args = (l.ctypes.data, l.shape[1], l.shape[0], l.shape[1], r.ctypes.data, r.shape[1], r.shape[0], r.shape[1], sx, sy, kernel_size, p1, p2)
    _check(lib().vwb200_sgm_calc_disparity(*args, None, 0, C.byref(ow), C.byref(oh), 0, None))
    out = np.empty((max(oh.value, 0), max(ow.value, 0), 3), np.int32)
    if out.size:
        _check(lib().vwb200_sgm_calc_disparity(*args, out.ctypes.data, ow.value, C.byref(ow), C.byref(oh), 0, None))
    return out


def calc_disparity_sgm_subpixel(left_in, right_in, search_volume, kernel_size, subpixel_mode=5, p1=0, p2=0):
    """calc_disparity_sgm followed by SemiGlobalMatcher::create_disparity_view_subpixel (Stereo/SGM.cc:1497-1614).
    subpixel_mode: SgmSubpixelMode (SGM.h:93-99), default SUBPIXEL_LC_BLEND.  Returns (int32 (h, w, 3), float32 (h, w, 3))."""
    sx, sy = search_volume
    ow, oh = C.c_int(0), C.c_int(0)
    l, r = _np(left_in, np.float32), _np(right_in, np.float32)
    args = (l.ctypes.data, l.shape[1], l.shape[0], l.shape[1], r.ctypes.data, r.shape[1], r.shape[0], r.shape[1], sx, sy, kernel_size, p1, p2,
            subpixel_mode)
    _check(lib().vwb200_sgm_calc_disparity_subpixel(*args, None, 0, None, 0, C.byref(ow), C.byref(oh), 0, None))
    out = np.empty((max(oh.value, 0), max(ow.value, 0), 3), np.int32)
    sub = np.empty((max(oh.value, 0), max(ow.value, 0), 3), np.float32)
    if out.size:
        _check(lib().vwb200_sgm_calc_disparity_subpixel(*args, out.ctypes.data, ow.value, sub.ctypes.data, ow.value, C.byref(ow), C.byref(oh), 0, None))
    return out, sub


def _sgm_params(search_volume, kernel_size, cost_type=CENSUS_TRANSFORM, use_mgm=False, subpixel_mode=SUBPIXEL_NONE, search_buffer=(2, 2),
                memory_limit_mb=6000, p1=0, p2=0, ternary_threshold=5, conserve_level=-1, assumed_threads=4):
    return SgmParams(int(search_volume[0]), int(search_volume[1]), int(kernel_size), int(cost_type), int(ternary_threshold), int(p1), int(p2),
                     int(bool(use_mgm)), int(subpixel_mode), int(search_buffer[0]), int(search_buffer[1]), int(conserve_level),
                     float(memory_limit_mb), int(assumed_threads), 0)


def calc_disparity_sgm_ex(cost_type, left_in, right_in, search_volume, kernel_size, use_mgm=False, subpixel_mode=SUBPIXEL_NONE,
                          search_buffer=(2, 2), memory_limit_mb=6000, left_mask=None, right_mask=None, prev_disparity=None,
                          bounds=None, p1=0, p2=0, ternary_threshold=5, conserve_level=-1, assumed_threads=4, return_bounds=False):
    """vw::stereo::calc_disparity_sgm with all its arguments (Stereo/SGM.h:361-376, SGM.cc:167-230): cost type
    (CENSUS_TRANSFORM / TERNARY_CENSUS_TRANSFORM), SGM or MGM, sub-pixel mode, search buffer, memory limit, masks and the
    previous pyramid level's disparity (which give every pixel its own search box).  `bounds` (h, w, 4) overrides the boxes.
    Returns (int32 (h, w, 3), float32 (h, w, 3) sub-pixel disparity[, int32 (h, w, 4) boxes])."""
    sp = _sgm_params(search_volume, kernel_size, cost_type, use_mgm, subpixel_mode, search_buffer, memory_limit_mb, p1, p2, ternary_threshold,
                     conserve_level, assumed_threads)
    l, r = _np(left_in, np.float32), _np(right_in, np.float32)
    ow, oh = C.c_int(0), C.c_int(0)
    head = (C.byref(sp), l.ctypes.data, l.shape[1], l.shape[0], l.shape[1], r.ctypes.data, r.shape[1], r.shape[0], r.shape[1])
    _check(lib().vwb200_sgm_calc_disparity_ex(*head, None, 0, None, 0, 0, 0, None, 0, 0, 0, None, None, 0, None, 0, None, C.byref(ow), C.byref(oh), 0, None))
    h, w = max(oh.value, 0), max(ow.value, 0)
    out = np.zeros((h, w, 3), np.int32)
    sub = np.zeros((h, w, 3), np.float32)
    bo = np.zeros((h, w, 4), np.int32)
    if out.size:
        lm = _np(left_mask, np.uint8) if left_mask is not None else None
        rm = _np(right_mask, np.uint8) if right_mask is not None else None
        pv = _np(prev_disparity, np.int32) if prev_disparity is not None else None
        bd = _np(bounds, np.int32) if bounds is not None else None
        if lm is not None and lm.shape != (h, w):
            raise LogicErr("Left mask size does not match the output size.")
        if bd is not None and bd.shape != (h, w, 4):
            raise ArgumentErr("sgm: bounds must be (out_h, out_w, 4)")
        _check(lib().vwb200_sgm_calc_disparity_ex(
            *head, lm.ctypes.data if lm is not None else None, w, rm.ctypes.data if rm is not None else None,
            rm.shape[1] if rm is not None else 0, rm.shape[0] if rm is not None else 0, rm.shape[1] if rm is not None else 0,
            pv.ctypes.data if pv is not None else None, pv.shape[1] if pv is not None else 0, pv.shape[0] if pv is not None else 0,
            pv.shape[1] if pv is not None else 0, bd.ctypes.data if bd is not None else None,
            out.ctypes.data, w, sub.ctypes.data, w, bo.ctypes.data if return_bounds else None, C.byref(ow), C.byref(oh), 0, None))
    return (out, sub, bo) if return_bounds else (out, sub)


def sgm_disp_bounds(shape, search_volume, search_buffer=(2, 2), prev_disparity=None, left_mask=None, right_mask=None, conserve_level=0,
                    use_mgm=False, memory_limit_mb=6000, assumed_threads=4):
    """SemiGlobalMatcher::populate_disp_bound_image + constrain_disp_bound_image (Stereo/SGM.cc:241-668): the search box
    {min_x, min_y, max_x, max_y} of every pixel of an (h, w) output."""
    h, w = int(shape[0]), int(shape[1])
    sp = _sgm_params(search_volume, 5, CENSUS_TRANSFORM, use_mgm, 0, search_buffer, memory_limit_mb, conserve_level=conserve_level,
                     assumed_threads=assumed_threads)
    lm = _np(left_mask, np.uint8) if left_mask is not None else None
    rm = _np(right_mask, np.uint8) if right_mask is not None else None
    pv = _np(prev_disparity, np.int32) if prev_disparity is not None else None
    if lm is not None and lm.shape != (h, w):
        raise LogicErr("Left mask size does not match the output size.")
    out = np.zeros((h, w, 4), np.int32)
    _check(lib().vwb200_sgm_disp_bounds(
        C.byref(sp), pv.ctypes.data if pv is not None else None, pv.shape[1] if pv is not None else 0, pv.shape[0] if pv is not None else 0,
        pv.shape[1] if pv is not None else 0, lm.ctypes.data if lm is not None else None, w, rm.ctypes.data if rm is not None else None,
        rm.shape[1] if rm is not None else 0, rm.shape[0] if rm is not None else 0, rm.shape[1] if rm is not None else 0, w, h, out.ctypes.data, 0, None))
    return out


def pyramid_down(img):
    """subsample(separable_convolution_filter(img, k, k), 2) with k = [1,4,6,4,1]/16
    (Stereo/CorrelationView.cc:210-214)."""
    a = _np(img, np.float32)
    h, w = a.shape
    out = np.empty((1 + (h - 1) // 2, 1 + (w - 1) // 2), np.float32)
    _check(lib().vwb200_pyramid_down(a.ctypes.data, w, h, w, out.ctypes.data, out.shape[1], 0, None))
    return out


def prefilter_image(image, prefilter_mode, prefilter_width):
    """vw::stereo::prefilter_image (Stereo/PreFilter.h:75-95)."""
    a = _np(image, np.float32)
    h, w = a.shape
    out = np.empty_like(a)
    _check(lib().vwb200_prefilter(a.ctypes.data, w, h, w, int(prefilter_mode), float(prefilter_width), out.ctypes.data, w, 0, None))
    return out


def subsample_mask_by_two(mask):
    a = _np(mask, np.uint8)
    h, w = a.shape
    out = np.empty((1 + (h - 1) // 2, 1 + (w - 1) // 2), np.uint8)
    _check(lib().vwb200_subsample_mask_by_two(a.ctypes.data, w, h, w, out.ctypes.data, out.shape[1], 0, None))
    return out


def cross_corr_consistency_check(l2r, r2l, cross_corr_threshold):
    """Stereo/Correlate.h:52-58; returns the checked copy of l2r."""
    a = _np(l2r, np.int32).copy()
    b = _np(r2l, np.int32)
    _check(lib().vwb200_cross_corr_consistency_check(a.ctypes.data, a.shape[1], a.shape[0], a.shape[1],
                                                     b.ctypes.data, b.shape[1], b.shape[0], b.shape[1],
                                                     float(cross_corr_threshold), 0, None))
    return a


def rm_outliers_using_thresh(disparity_map, half_h_kernel, half_v_kernel, pixel_threshold, rejection_threshold):
    a = _np(disparity_map, np.int32)
    out = np.empty_like(a)
    _check(lib().vwb200_rm_outliers_using_thresh(a.ctypes.data, a.shape[1], a.shape[0], half_h_kernel, half_v_kernel,
                                                 pixel_threshold, rejection_threshold, out.ctypes.data, 0, None))
    return out


def disparity_cleanup_using_thresh(disparity_map, h_half_kernel, v_half_kernel, pixel_threshold, rejection_threshold):
    a = _np(disparity_map, np.int32)
    out = np.empty_like(a)
    _check(lib().vwb200_disparity_cleanup_using_thresh(a.ctypes.data, a.shape[1], a.shape[0], h_half_kernel, v_half_kernel,
                                                       pixel_threshold, rejection_threshold, out.ctypes.data, 0, None))
    return out


def disparity_mask(disparity_map, left_mask, right_mask):
    a = _np(disparity_map, np.int32)
    lm, rm = _np(left_mask, np.uint8), _np(right_mask, np.uint8)
    if lm.shape != a.shape[:2]:
        raise ArgumentErr("disparity_mask: input and left mask are not same dimensions.")
    out = np.empty_like(a)
    _check(lib().vwb200_disparity_mask(a.ctypes.data, a.shape[1], a.shape[0], lm.ctypes.data, rm.ctypes.data,
                                       rm.shape[1], rm.shape[0], out.ctypes.data, 0, None))
    return out


class ParabolaSubpixelView:
    """vw::stereo::ParabolaSubpixelView (Stereo/ParabolaSubpixelView.h:27-117): lazy view refining an integer
    disparity (PixelMask<Vector2f> triples, same size as the left image) by a 2-D parabola fit."""

    def __init__(self, disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size):
        self._d = _np(disparity, np.float32)
        self._l, self._r = _np(left_image, np.float32), _np(right_image, np.float32)
        if self._d.shape[:2] != self._l.shape:
            raise ArgumentErr("SubpixelView: Disparity image must match left image.")
        self._mode, self._width, self._k = int(prefilter_mode), float(prefilter_width), (int(kernel_size[0]), int(kernel_size[1]))

    def cols(self):
        return self._l.shape[1]

    def rows(self):
        return self._l.shape[0]

    def planes(self):
        return 1

    def __call__(self, i, j, p=0):
        raise NoImplErr("SubpixelView:operator() has not been implemented.")

    def rasterize(self, dest=None, bbox=None):
        b = _bbox(bbox) if bbox is not None else (0, 0, self.cols(), self.rows())
        w, h = b[2] - b[0], b[3] - b[1]
        if dest is None:
            dest = np.empty((h, w, 3), np.float32)
        _check(lib().vwb200_parabola_subpixel(self._d.ctypes.data, self.cols(), self.rows(), self._l.ctypes.data, self._l.shape[1],
                                              self._r.ctypes.data, self._r.shape[1], self._r.shape[0], self._r.shape[1],
                                              self._k[0], self._k[1], self._mode, self._width, b[0], b[1], b[2], b[3],
                                              dest.ctypes.data, dest.strides[0] // 12, 0, None))
        return dest

    prerasterize = rasterize


def parabola_subpixel(disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size):
    """vw::stereo::parabola_subpixel (Stereo/ParabolaSubpixelView.h:111-117)."""
    return ParabolaSubpixelView(disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size)


class PyramidSubpixelView:
    """vw::stereo::PyramidSubpixelView (Stereo/SubpixelView.h:42-150, .cc:33-224): lazy view refining a
    PixelMask<Vector2f> disparity (float32 (rows, cols, 3) triples, same size as the left image) by iterative
    Lucas-Kanade, affine or Bayes-EM affine sub-pixel correlation over an image pyramid."""

    def __init__(self, disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size,
                 max_pyramid_levels, algorithm, phase_subpixel_accuracy=20):
        self._d = _np(disparity, np.float32)
        self._l, self._r = _np(left_image, np.float32), _np(right_image, np.float32)
        if self._d.shape[:2] != self._l.shape or self._d.ndim != 3 or self._d.shape[2] != 3:
            raise ArgumentErr("SubpixelView: Disparity image must match left image.")
        self._mode, self._width, self._k = int(prefilter_mode), float(prefilter_width), (int(kernel_size[0]), int(kernel_size[1]))
        self._levels, self._alg = int(max_pyramid_levels), int(algorithm)
        self._phase_accuracy = int(phase_subpixel_accuracy)

    def cols(self):
        return self._l.shape[1]

    def rows(self):
        return self._l.shape[0]

    def planes(self):
        return 1

    def __call__(self, i, j, p=0):
        raise NoImplErr("PyramidSubpixelView::operator() is not implemented.")

    def rasterize(self, dest=None, bbox=None):
        b = _bbox(bbox) if bbox is not None else (0, 0, self.cols(), self.rows())
        w, h = b[2] - b[0], b[3] - b[1]
        if dest is None:
            dest = np.empty((h, w, 3), np.float32)
        _check(lib().vwb200_pyramid_subpixel(self._d.ctypes.data, self.cols(), self.rows(), self._l.ctypes.data, self._l.shape[1],
                                             self._r.ctypes.data, self._r.shape[1], self._r.shape[0], self._r.shape[1],
                                             self._k[0], self._k[1], self._mode, self._width, b[0], b[1], b[2], b[3],
                                             dest.ctypes.data, dest.strides[0] // 12, 0, None, self._levels, self._alg))
        return dest

    prerasterize = rasterize


def lk_subpixel(disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size, max_pyramid_levels=2):
    """vw::stereo::lk_subpixel (Stereo/SubpixelView.h:117-125)."""
    return PyramidSubpixelView(disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size,
                               max_pyramid_levels, SUBPIXEL_LUCAS_KANADE)


def affine_subpixel(disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size, max_pyramid_levels=2):
    """vw::stereo::affine_subpixel (Stereo/SubpixelView.h:127-135)."""
    return PyramidSubpixelView(disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size,
                               max_pyramid_levels, SUBPIXEL_FAST_AFFINE)


def bayes_em_subpixel(disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size, max_pyramid_levels=2):
    """vw::stereo::bayes_em_subpixel (Stereo/SubpixelView.h:137-145)."""
    return PyramidSubpixelView(disparity, left_image, right_image, prefilter_mode, prefilter_width, kernel_size,
                               max_pyramid_levels, SUBPIXEL_BAYES_EM)


def _subpixel_refine(algorithm, disparity_map, left_image, right_image, kern_width, kern_height, region_of_interest,
                     do_horizontal_subpixel, do_vertical_subpixel):
    roi = _bbox(region_of_interest)
    if _is_torch(disparity_map):
        import torch
        d = disparity_map.detach().clone().float().contiguous()
        l, r = left_image.contiguous().float(), right_image.contiguous().float()
        if tuple(d.shape) != (l.shape[0], l.shape[1], 3):
            raise ArgumentErr("subpixel_correlation: left image and disparity map do not have the same dimensions.")
        _check(lib().vwb200_subpixel_refine(algorithm, d.data_ptr(), l.shape[1], l.shape[0], l.shape[1], l.data_ptr(), l.stride(0),
                                            r.data_ptr(), r.shape[1], r.shape[0], r.stride(0), kern_width, kern_height,
                                            roi[0], roi[1], roi[2], roi[3], int(bool(do_horizontal_subpixel)),
                                            int(bool(do_vertical_subpixel)), 1, _stream_ptr()))
        return d
    d = np.array(disparity_map, dtype=np.float32, order="C", copy=True)
    l, r = _np(left_image, np.float32), _np(right_image, np.float32)
    if d.shape != (l.shape[0], l.shape[1], 3):
        raise ArgumentErr("subpixel_correlation: left image and disparity map do not have the same dimensions.")
    _check(lib().vwb200_subpixel_refine(algorithm, d.ctypes.data, l.shape[1], l.shape[0], l.shape[1], l.ctypes.data, l.shape[1],
                                        r.ctypes.data, r.shape[1], r.shape[0], r.shape[1], kern_width, kern_height,
                                        roi[0], roi[1], roi[2], roi[3], int(bool(do_horizontal_subpixel)),
                                        int(bool(do_vertical_subpixel)), 0, None))
    return d


def subpixel_optimized_LK_2d(disparity_map, left_image, right_image, kern_width, kern_height, region_of_interest,
                             do_horizontal_subpixel=True, do_vertical_subpixel=True):
    """vw::stereo::subpixel_optimized_LK_2d (Stereo/Correlate.h:95-104).  The reference refines disparity_map in
    place; this returns the refined copy (numpy in, numpy out; torch CUDA in, torch CUDA out)."""
    return _subpixel_refine(SUBPIXEL_LUCAS_KANADE, disparity_map, left_image, right_image, kern_width, kern_height,
                            region_of_interest, do_horizontal_subpixel, do_vertical_subpixel)


def subpixel_optimized_affine_2d(disparity_map, left_image, right_image, kern_width, kern_height, region_of_interest,
                                 do_horizontal_subpixel=True, do_vertical_subpixel=True, verbose=False):
    """vw::stereo::subpixel_optimized_affine_2d (Stereo/Correlate.h:74-83); returns the refined copy."""
    return _subpixel_refine(SUBPIXEL_FAST_AFFINE, disparity_map, left_image, right_image, kern_width, kern_height,
                            region_of_interest, do_horizontal_subpixel, do_vertical_subpixel)


def subpixel_optimized_affine_2d_EM(disparity_map, left_image, right_image, kern_width, kern_height, region_of_interest,
                                    do_horizontal_subpixel=True, do_vertical_subpixel=True, verbose=False):
    """vw::stereo::subpixel_optimized_affine_2d_EM (Stereo/Correlate.h:63-72); returns the refined copy."""
    return _subpixel_refine(SUBPIXEL_BAYES_EM, disparity_map, left_image, right_image, kern_width, kern_height,
                            region_of_interest, do_horizontal_subpixel, do_vertical_subpixel)


def _masked(img):
    """PixelMask<float> raster: (rows, cols, 2) float32 {value, valid}; a 2-D image is all valid."""
    if _is_torch(img):
        import torch
        t = img.detach().float()
        if t.dim() == 2:
            t = torch.stack([t, torch.ones_like(t)], dim=-1)
        return t.contiguous()
    a = np.asarray(img, dtype=np.float32)
    if a.ndim == 2:
        a = np.stack([a, np.ones_like(a)], axis=-1)
    return np.ascontiguousarray(a)


class CorrEval:
    """vw::stereo::CorrEval (Stereo/CorrEval.h:56-129, CorrEval.cc:139-317): lazy view of the quality of a float disparity
    at every pixel -- "ncc", "stddev", "parabola_curvature" or "cramer_rao" over kernel_size windows, at the pixels whose
    coordinates in the rasterised bbox are multiples of sample_rate.  Images are float32 (rows, cols, 2) {value, valid}
    or 2-D float32 (all valid); the disparity is (rows, cols, 3) {dx, dy, valid} of the left image's size.  rasterize()
    returns (rows, cols, 2) {value, valid}: numpy for numpy inputs, torch CUDA tensors (on the current stream) for
    torch CUDA inputs.  prefilter_mode is accepted and unused, as in the reference; prefilter_kernel_width sets the crop
    padding, which moves the right crop's origin and hence the float rounding of the bilinear weights."""

    def __init__(self, left, right, disp, kernel_size, metric, sample_rate, round_to_int, prefilter_mode=0,
                 prefilter_kernel_width=0.0):
        self._torch = _is_torch(disp)
        if any(_is_torch(x) != self._torch or (self._torch and not x.is_cuda) for x in (left, right, disp)):
            raise ArgumentErr("CorrEval: the images and the disparity must all be numpy arrays or all torch CUDA tensors.")
        self._l, self._r = _masked(left), _masked(right)
        if self._torch:
            self._d = disp.detach().float().contiguous()
        else:
            self._d = _np(disp, np.float32)
        if tuple(self._d.shape[:2]) != tuple(self._l.shape[:2]) or self._d.ndim != 3 or self._d.shape[2] != 3:
            raise ArgumentErr("CorrEval: Left image and disparity must have the same dimensions.")
        self._k = (int(kernel_size[0]), int(kernel_size[1]))
        if not all(k > 0 and k % 2 == 1 for k in self._k):
            raise ArgumentErr("CorrEval: The kernel dimensions must be positive and odd.")
        if metric not in CORR_EVAL_METRICS:
            raise ArgumentErr(f"CorrEval: Invalid metric: {metric}.")
        self._metric = CORR_EVAL_METRICS[metric]
        self._sample_rate, self._round = int(sample_rate), int(bool(round_to_int))
        self._prefilter_mode, self._pkw = int(prefilter_mode), float(prefilter_kernel_width)

    def cols(self):
        return self._l.shape[1]

    def rows(self):
        return self._l.shape[0]

    def planes(self):
        return 1

    def __call__(self, i, j, p=0):
        raise NoImplErr("CorrEval::operator() is not implemented.")

    def rasterize(self, dest=None, bbox=None):
        b = _bbox(bbox) if bbox is not None else (0, 0, self.cols(), self.rows())
        w, h = b[2] - b[0], b[3] - b[1]
        l, r, d = self._l, self._r, self._d
        shape = (max(h, 0), max(w, 0), 2)
        if self._torch:
            import torch
            if dest is None:
                dest = torch.empty(shape, dtype=torch.float32, device=d.device)
            elif not (_is_torch(dest) and dest.is_cuda and dest.device == d.device and dest.dtype == torch.float32
                      and tuple(dest.shape) == shape and dest.stride(2) == 1 and dest.stride(1) == 2 and dest.stride(0) % 2 == 0):
                raise ArgumentErr(f"CorrEval: dest must be a float32 CUDA tensor of shape {shape} on {d.device} "
                                  "with contiguous pixels")
            ptr = lambda t: t.data_ptr()
            pitch, on_device, stream = dest.stride(0) // 2, 1, _stream_ptr()
        else:
            if dest is None:
                dest = np.empty(shape, np.float32)
            elif not (isinstance(dest, np.ndarray) and dest.dtype == np.float32 and dest.shape == shape and dest.flags.writeable
                      and dest.strides[2] == 4 and dest.strides[1] == 8 and dest.strides[0] % 8 == 0):
                raise ArgumentErr(f"CorrEval: dest must be a writable float32 numpy array of shape {shape} with contiguous pixels")
            ptr = lambda a: a.ctypes.data
            pitch, on_device, stream = dest.strides[0] // 8, 0, None
        _check(lib().vwb200_corr_eval(ptr(l), l.shape[1], l.shape[0], l.shape[1], ptr(r), r.shape[1], r.shape[0], r.shape[1],
                                      ptr(d), d.shape[1], self._k[0], self._k[1], self._metric, self._sample_rate, self._round,
                                      self._pkw, b[0], b[1], b[2], b[3], ptr(dest), pitch, on_device, stream))
        return dest

    prerasterize = rasterize


def corr_eval(left, right, disp, kernel_size, metric, sample_rate, round_to_int, prefilter_mode=0, prefilter_kernel_width=0.0):
    """vw::stereo::corr_eval (Stereo/CorrEval.h:117-128)."""
    return CorrEval(left, right, disp, kernel_size, metric, sample_rate, round_to_int, prefilter_mode, prefilter_kernel_width)


class BBox2i:
    """vw::BBox2i: half-open [min, max).  BBox2i(x, y, w, h) like Math/BBox.tcc:55-59."""

    def __init__(self, x=0, y=0, w=0, h=0):
        self.x0, self.y0, self.x1, self.y1 = x, y, x + w, y + h

    @classmethod
    def from_corners(cls, x0, y0, x1, y1):
        return cls(x0, y0, x1 - x0, y1 - y0)

    def width(self):
        return max(self.x1 - self.x0, 0)

    def height(self):
        return max(self.y1 - self.y0, 0)

    def __repr__(self):
        return f"BBox2i(({self.x0},{self.y0})-({self.x1},{self.y1}))"


class PyramidCorrelationView:
    """vw::stereo::PyramidCorrelationView (Stereo/CorrelationView.h:35-193) rasterised on a B200.

    Lazy like the reference: construction only records parameters and places the inputs in HBM;
    work happens in rasterize()/prerasterize(), one call per tile bbox, from any number of threads.
    """

    def __init__(self, left, right, left_mask, right_mask, prefilter_mode, prefilter_width,
                 search_region, kernel_size, cost_type, corr_timeout, seconds_per_op,
                 consistency_threshold, min_consistency_level, filter_half_kernel, max_pyramid_levels,
                 algorithm=VW_CORRELATION_BM, collar_size=0, sgm_subpixel_mode=SUBPIXEL_LC_BLEND, sgm_search_buffer=(2, 2),
                 memory_limit_mb=6000, blob_filter_area=0, lr_disp_diff=None, region_ul=(0, 0),
                 write_debug_images=False, sgm_threads=4, streamed=False):
        """Argument order = the reference constructor (Stereo/CorrelationView.h:48-69); sgm_threads stands for
        vw_settings().default_num_threads(), which SGM's memory estimate reads (SGM.cc:715-716).
        lr_disp_diff: float32 (rows, cols, 2) PixelMask<float> array whose pixel (0, 0) is image pixel region_ul; updated in place."""
        if isinstance(search_region, BBox2i):
            s = (search_region.x0, search_region.y0, search_region.x1, search_region.y1)
        else:
            s = tuple(int(v) for v in search_region)
        self._p = CorrParams(s[0], s[1], s[2], s[3], int(kernel_size[0]), int(kernel_size[1]), int(cost_type),
                             int(prefilter_mode), float(prefilter_width), float(consistency_threshold),
                             int(min_consistency_level), int(filter_half_kernel), int(max_pyramid_levels),
                             int(collar_size), int(corr_timeout), float(seconds_per_op), int(algorithm),
                             int(blob_filter_area), int(sgm_subpixel_mode), int(sgm_search_buffer[0]), int(sgm_search_buffer[1]),
                             int(region_ul[0]), int(region_ul[1]), int(bool(write_debug_images)), int(sgm_threads), float(memory_limit_mb))
        self._h = C.c_void_p()
        _check(lib().vwb200_corr_create(C.byref(self._p), C.byref(self._h)))
        self._diff = None
        if lr_disp_diff is not None:
            if _is_torch(lr_disp_diff):
                d = lr_disp_diff
                assert d.dtype.is_floating_point and d.element_size() == 4 and d.dim() == 3 and d.shape[2] == 2 and d.stride(2) == 1 and d.stride(1) == 2
                _check(lib().vwb200_corr_set_lr_disp_diff(self._h, d.data_ptr(), d.shape[1], d.shape[0], d.stride(0) // 2, 1))
            else:
                d = lr_disp_diff
                if not (isinstance(d, np.ndarray) and d.dtype == np.float32 and d.ndim == 3 and d.shape[2] == 2 and d.strides[2] == 4 and d.strides[1] == 8):
                    raise ArgumentErr("lr_disp_diff must be a float32 (rows, cols, 2) array")
                _check(lib().vwb200_corr_set_lr_disp_diff(self._h, d.ctypes.data, d.shape[1], d.shape[0], d.strides[0] // 8, 0))
            self._diff = d
        self._keep = None
        self._device = _is_torch(left)
        if self._device:
            import torch
            l, r = left.contiguous().float(), right.contiguous().float()
            if tuple(left_mask.shape) != tuple(l.shape) or tuple(right_mask.shape) != tuple(r.shape):
                raise ArgumentErr("masks must have the size of their images")
            lm = (left_mask != 0).to(torch.uint8).contiguous() if left_mask.dtype != torch.uint8 else left_mask.contiguous()
            rm = (right_mask != 0).to(torch.uint8).contiguous() if right_mask.dtype != torch.uint8 else right_mask.contiguous()
            self._keep = (l, r, lm, rm)
            _check(lib().vwb200_corr_set_inputs(self._h, l.data_ptr(), l.shape[1], l.shape[0], l.stride(0),
                                                r.data_ptr(), r.shape[1], r.shape[0], r.stride(0),
                                                lm.data_ptr(), lm.stride(0), rm.data_ptr(), rm.stride(0), 1))
        else:
            l, r = _np(left, np.float32), _np(right, np.float32)
            lm, rm = _np(left_mask, np.uint8), _np(right_mask, np.uint8)
            if lm.shape != l.shape or rm.shape != r.shape:
                raise ArgumentErr("masks must have the size of their images")
            if streamed:          # the rasters stay on the host; each rasterize() uploads its tile's region of interest
                self._keep = (l, r, lm, rm)
            _check(lib().vwb200_corr_set_inputs(self._h, l.ctypes.data, l.shape[1], l.shape[0], l.shape[1],
                                                r.ctypes.data, r.shape[1], r.shape[0], r.shape[1],
                                                lm.ctypes.data, lm.shape[1], rm.ctypes.data, rm.shape[1], 2 if streamed else 0))

    def __del__(self):
        try:
            if self._h:
                lib().vwb200_corr_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # --- standard ImageView interface (CorrelationView.h:109-117) ---
    def cols(self):
        return lib().vwb200_corr_cols(self._h)

    def rows(self):
        return lib().vwb200_corr_rows(self._h)

    def planes(self):
        return 1

    def __call__(self, i, j, p=0):
        raise NoImplErr("NewCorrelationView::operator() is not implemented.")

    def num_levels(self, bbox):
        b = _bbox(bbox)
        return lib().vwb200_corr_num_levels(self._h, b[2] - b[0], b[3] - b[1])

    def rasterize(self, dest=None, bbox=None):
        """rasterize(dest, bbox) (CorrelationView.h:123-133).  dest: float32 (h, w, 3) numpy array (or torch
        CUDA tensor) already sized to bbox, or None to allocate.  Pixels are {dx, dy, valid}."""
        return self._run(lib().vwb200_corr_rasterize, dest, bbox)

    def _run(self, fn, dest, bbox):
        b = _bbox(bbox) if bbox is not None else (0, 0, self.cols(), self.rows())
        w, h = b[2] - b[0], b[3] - b[1]
        if dest is not None and _is_torch(dest) or (dest is None and self._device):
            import torch
            if dest is None:
                dest = torch.empty((h, w, 3), dtype=torch.float32, device=self._keep[0].device)
            assert dest.shape == (h, w, 3) and dest.dtype == torch.float32 and dest.stride(2) == 1 and dest.stride(1) == 3
            _check(fn(self._h, b[0], b[1], b[2], b[3], dest.data_ptr(), dest.stride(0) // 3, 1, _stream_ptr()))
            return dest
        if dest is None:
            dest = np.empty((h, w, 3), np.float32)
        assert dest.shape == (h, w, 3) and dest.dtype == np.float32 and dest.strides[2] == 4 and dest.strides[1] == 12
        _check(fn(self._h, b[0], b[1], b[2], b[3], dest.ctypes.data, dest.strides[0] // 12, 0, None))
        return dest

    def prerasterize(self, bbox):
        """prerasterize(bbox): an owning buffer of bbox size (CorrelationView.cc:880-884); processes exactly bbox --
        unlike rasterize() no collar is added (CorrelationView.h:123-133)."""
        return self._run(lib().vwb200_corr_prerasterize, None, bbox)


def _bbox(b):
    if isinstance(b, BBox2i):
        return (b.x0, b.y0, b.x1, b.y1)
    return tuple(int(v) for v in b)


def pyramid_correlate(left, right, left_mask, right_mask, prefilter_mode, prefilter_width, search_region, kernel_size,
                      cost_type, corr_timeout, seconds_per_op, consistency_threshold, min_consistency_level,
                      filter_half_kernel, max_pyramid_levels, algorithm=VW_CORRELATION_BM, collar_size=0,
                      sgm_subpixel_mode=SUBPIXEL_LC_BLEND, sgm_search_buffer=(2, 2), memory_limit_mb=6000, blob_filter_area=0,
                      lr_disp_diff=None, region_ul=(0, 0), write_debug_images=False, **kw):
    """vw::stereo::pyramid_correlate (Stereo/CorrelationView.h:195-230), same positional order."""
    return PyramidCorrelationView(left, right, left_mask, right_mask, prefilter_mode, prefilter_width, search_region,
                                  kernel_size, cost_type, corr_timeout, seconds_per_op, consistency_threshold,
                                  min_consistency_level, filter_half_kernel, max_pyramid_levels, algorithm,
                                  collar_size, sgm_subpixel_mode, sgm_search_buffer, memory_limit_mb, blob_filter_area,
                                  lr_disp_diff, region_ul, write_debug_images, **kw)
