"""CPU tests of the sub-pixel refinement oracle (oracle/vw_subpixel_oracle.c): the reference's Bayes-EM known-answer
tests, the two named substitutions (exp, posv) and the details of the in-place scan."""
import ctypes
import ctypes.util

import numpy as np
import pytest

from subpixel_fixtures import chain_case, check_error, kat_case, smooth_pair


@pytest.fixture(scope="module")
def sp():
    from oracle import subpixel
    subpixel.build()
    return subpixel


# TestSubPixel.cxx:343-404: LOG 1.4, 7x7, default two pyramid levels, the reference's thresholds
@pytest.mark.parametrize("istretch,max_err,max_invalid", [(95, 0.35, 12), (90, 0.36, 12), (80, 0.52, 22), (70, 0.9, 48)])
def test_bayes_em_reference_kat(sp, istretch, max_err, max_invalid):
    left, right, disp, stretch, translation = kat_case(istretch)
    out = sp.pyramid_subpixel(disp, left, right, (7, 7), 1, 1.4, 2, sp.SUBPIXEL_BAYES_EM)
    err, invalid = check_error(out, stretch, translation)
    assert err < max_err and invalid <= max_invalid, (err, invalid)


def _ulp_dist(a, b):
    ia = a.view(np.int32).astype(np.int64)
    ib = b.view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


def test_expf_within_one_ulp_of_libm(sp):
    x = np.linspace(-75.0, 0.0, 2_000_001, dtype=np.float64).astype(np.float32)
    # arguments of the weight templates: -(r^2) / two_sigma_sqr for the kernel sizes in use
    extra = []
    for k in (3, 5, 7, 9, 11, 15, 21, 35):
        tss = np.float32(2.0 * (float(np.float32(k)) / 5.0) ** 2)
        r2 = np.arange(0, 2 * (k // 2) ** 2 + 1, dtype=np.float32)
        extra.append((-r2) / tss)
    x = np.concatenate([x] + extra).astype(np.float32)
    got = sp.expf(x)
    as_double = np.exp(x.astype(np.float64)).astype(np.float32)     # (float)exp((double)x)
    assert _ulp_dist(got, as_double).max() <= 1
    libm = ctypes.CDLL(ctypes.util.find_library("m"))
    libm.expf.argtypes, libm.expf.restype = [ctypes.c_float], ctypes.c_float
    sub = x[::10]
    as_float = np.array([libm.expf(float(v)) for v in sub], np.float32)    # expf
    assert _ulp_dist(got[::10], as_float).max() <= 1
    assert (got == as_double).mean() > 0.999
    assert sp.expf(np.array([-200.0, 0.0], np.float32)).tolist() == [0.0, 1.0]


def test_posv_failure_leaves_rhs_unsolved(sp):
    A = np.array([[4.0, 2.0], [2.0, 1.0]], np.float32)        # singular: the second pivot is 0
    info, b = sp.posv(A, np.array([1.5, -2.0], np.float32))
    assert info == 2 and b.tolist() == [1.5, -2.0]
    info, b = sp.posv(np.full((6, 6), np.nan, np.float32), np.arange(6, dtype=np.float32))
    assert info == 1 and b.tolist() == list(range(6))
    M = np.array([[4.0, 1.0], [1.0, 3.0]], np.float32)
    info, b = sp.posv(M, np.array([1.0, 2.0], np.float32))
    assert info == 0 and np.allclose(M @ b, [1.0, 2.0], atol=1e-6)


def test_disparity_subsample_and_upsample(sp):
    d = np.zeros((5, 4, 3), np.float32)
    d[..., 0] = np.arange(20, dtype=np.float32).reshape(5, 4)
    d[..., 1] = -0.5 * np.arange(20, dtype=np.float32).reshape(5, 4)
    d[..., 2] = 1.0
    d[1, 1, 2] = 0.0
    d[0, 0, 2] = 0.0
    s = sp.disparity_subsample(d)
    assert s.shape == (3, 2, 3)

    def ref(i, j):     # DisparityMap.h:1268-1304 with the constant edge extension
        acc, cnt = np.zeros(2), 0
        for dx, dy, wt in ((0, 0, 10), (1, 0, 5), (0, 1, 5), (-1, 0, 5), (0, -1, 5), (1, 1, 2), (-1, -1, 2), (-1, 1, 2), (1, -1, 2)):
            p = d[min(max(2 * j + dy, 0), 4), min(max(2 * i + dx, 0), 3)]
            if p[2]:
                acc += wt * p[:2].astype(np.float64)
                cnt += wt
        return (acc / (cnt * 2)).astype(np.float32), cnt > 0

    for j in range(3):
        for i in range(2):
            v, ok = ref(i, j)
            assert s[j, i, 2] == (1.0 if ok else 0.0)
            assert np.array_equal(s[j, i, :2], v)
    u = sp.disparity_upsample(s, (5, 4))
    assert np.array_equal(u[..., :2], 2 * s[np.arange(5)[:, None] // 2, np.arange(4)[None, :] // 2, :2])
    assert np.array_equal(u[..., 2], s[np.arange(5)[:, None] // 2, np.arange(4)[None, :] // 2, 2])


def _input_counts(disp, k=3):
    v = np.pad(disp[:, :, 2] != 0, k // 2).astype(int)
    h, w = disp.shape[:2]
    return sum(v[j:j + h, i:i + w] for j in range(k) for i in range(k))


def test_in_place_order_changes_a_later_pixel(sp):
    left, right, disp = chain_case()
    counts = _input_counts(disp)
    # against the input validity, every row-10 pixel from x = 11 on has enough good pixels (>= 9 // 2) ...
    assert (counts[10, 11:29] >= 4).all() and counts[10, 10] < 4
    seq = sp.subpixel_level(sp.SUBPIXEL_BAYES_EM, disp, left, right, (3, 3))
    # ... but the scan updates the map in place: (10, 10) is invalidated first, which starves (11, 10), and so on
    assert (seq[10, 10:30, 2] == 0).all()


def test_zero_levels_equals_one_level_function_call(sp):
    """max_pyramid_levels = 0 is one level-function call on the translated, kernel-padded patch (SubpixelView.cc:39-95,
    :190-223), and a negative level count is clamped to 0."""
    left, right, disp = smooth_pair(48, 56, seed=4)
    k, (h, w) = 5, left.shape
    out = sp.pyramid_subpixel(disp, left, right, (k, k), 0, 0.0, 0, sp.SUBPIXEL_FAST_AFFINE, bbox=(0, 0, w, h))
    # the disparity range of the crop (every pixel, valid or not), truncated
    sx0, sy0 = int(disp[..., 0].min()), int(disp[..., 1].min())
    sx1, sy1 = int(disp[..., 0].max()), int(disp[..., 1].max())
    pw, ph = w + (sx1 - sx0) + 2 * k, h + (sy1 - sy0) + 2 * k

    def crop_const(img, x0, y0):
        ys = np.clip(np.arange(y0, y0 + ph), 0, img.shape[0] - 1)
        xs = np.clip(np.arange(x0, x0 + pw), 0, img.shape[1] - 1)
        return np.ascontiguousarray(img[ys[:, None], xs[None, :]])

    L = crop_const(left, -k, -k)
    R = crop_const(right, sx0 - k, sy0 - k)
    D = np.zeros((ph, pw, 3), np.float32)
    D[k:k + h, k:k + w] = disp
    D[..., 0] -= np.float32(sx0)
    D[..., 1] -= np.float32(sy0)
    D = sp.subpixel_level(sp.SUBPIXEL_FAST_AFFINE, D, L, R, (k, k), roi=(k, k, k + w, k + h))
    ref = D[k:k + h, k:k + w].copy()
    ref[..., 0] += np.float32(sx0)
    ref[..., 1] += np.float32(sy0)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    out2 = sp.pyramid_subpixel(disp, left, right, (k, k), 0, 0.0, -3, sp.SUBPIXEL_FAST_AFFINE, bbox=(0, 0, w, h))
    assert np.array_equal(out.view(np.uint32), out2.view(np.uint32))


def test_phase_and_unknown_algorithms_are_not_implemented(sp):
    left, right, disp = smooth_pair(24, 24)
    for alg in (sp.SUBPIXEL_PHASE, 7, -1):
        with pytest.raises(NotImplementedError):
            sp.pyramid_subpixel(disp, left, right, (5, 5), 0, 0.0, 1, alg)


@pytest.mark.parametrize("alg", [0, 1, 2])
def test_refinement_recovers_a_subpixel_shift(sp, alg):
    left, right, disp = smooth_pair(64, 64, shift=(1.3, -0.6), seed=8)
    out = sp.pyramid_subpixel(disp, left, right, (9, 9), 0, 0.0, 1, alg, bbox=(16, 16, 48, 48))
    ok = out[..., 2] != 0
    assert ok.mean() > 0.8
    assert abs(float(np.median(out[ok, 0])) - 1.3) < 0.1 and abs(float(np.median(out[ok, 1])) + 0.6) < 0.1
