"""CPU tests of the CorrEval oracle (oracle/vw_corr_eval_oracle.c).  The reference ships no CorrEval test, so the oracle
is pinned against a second, vectorised numpy restatement of CorrEval.cc (float32 bilinear path, float64 sums in the
reference's order), against closed-form cases, and on each detail of the reference that changes output bits."""
import numpy as np
import pytest

from corr_eval_fixtures import METRICS, masked, scene, smooth_disparity, texture, tiny_case


@pytest.fixture(scope="module")
def ce():
    from oracle import corr_eval
    corr_eval.build()
    return corr_eval


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ---- the numpy restatement ----------------------------------------------------------------------------------------

def _round_half_away(v):
    a = np.floor(np.abs(v.astype(np.float64)) + 0.5)
    return (np.sign(v) * a).astype(np.float32)


def _gather(img, X, Y):
    """img {value, valid} at integer positions, an invalid 0 outside."""
    h, w = img.shape[:2]
    inside = (X >= 0) & (Y >= 0) & (X < w) & (Y < h)
    Xc, Yc = np.clip(X, 0, w - 1), np.clip(Y, 0, h - 1)
    v = np.where(inside, img[Yc, Xc, 0], np.float32(0)).astype(np.float32)
    ok = inside & (img[Yc, Xc, 1] != 0)
    return v, ok


def _bilinear(img, i, j, ox, oy):
    """BilinearInterpolation of PixelMask<float> at crop-relative double coordinates (i, j); crop origin (ox, oy)."""
    x, y = np.floor(i).astype(np.int64), np.floor(j).astype(np.int64)
    at_int = (x == i) & (y == j)
    nx = (i.astype(np.float32) - x.astype(np.float32)).astype(np.float32)
    ny = (j.astype(np.float32) - y.astype(np.float32)).astype(np.float32)
    one = np.float32(1)
    n1x, n1y = one - nx, one - ny
    X, Y = x + ox, y + oy
    p00, v00 = _gather(img, X, Y)
    p10, v10 = _gather(img, X + 1, Y)
    p01, v01 = _gather(img, X, Y + 1)
    p11, v11 = _gather(img, X + 1, Y + 1)
    r = p00 * n1x
    r = r + p10 * nx
    r = r * n1y
    row = p01 * n1x
    row = row + p11 * nx
    r = r + row * ny
    return np.where(at_int, p00, r), np.where(at_int, v00, v00 & v10 & v01 & v11)


def np_corr_eval(left, right, disp, kernel, metric, sample_rate=1, round_to_int=False, pkw=0.0, bbox=None):
    L, R = masked(left) if left.ndim == 2 else left, masked(right) if right.ndim == 2 else right
    h, w = L.shape[:2]
    x0, y0, x1, y1 = bbox or (0, 0, w, h)
    d = disp[y0:y1, x0:x1].astype(np.float32).copy()
    if round_to_int:
        d[..., :2] = _round_half_away(d[..., :2])
    rows, cols = np.mgrid[0:y1 - y0, 0:x1 - x0]
    sel = (d[..., 2] != 0) & (rows % sample_rate == 0) & (cols % sample_rate == 0)
    out = np.zeros((y1 - y0, x1 - x0, 2), np.float32)
    if not sel.any():
        return out
    col, row, dx, dy = cols[sel], rows[sel], d[..., 0][sel], d[..., 1][sel]
    hx, hy = kernel[0] // 2, kernel[1] // 2
    curv = metric in ("parabola_curvature", "cramer_rao")
    e = 1 + 2 + int(np.ceil(np.float32(pkw))) + 5 + (1 if curv else 0)
    ox = int(np.floor((x0 + col).astype(np.float64) + dx.astype(np.float64)).min()) - hx - e
    oy = int(np.floor((y0 + row).astype(np.float64) + dy.astype(np.float64)).min()) - hy - e

    def patches(sx, sy):
        for c in range(kernel[0]):
            for r in range(kernel[1]):
                lx, ly = x0 + col + c - hx, y0 + row + r - hy
                a = _gather(L, lx, ly)
                i = lx.astype(np.float64) + sx.astype(np.float64) - ox
                j = ly.astype(np.float64) + sy.astype(np.float64) - oy
                if round_to_int:
                    b = _gather(R, i.astype(np.int64) + ox, j.astype(np.int64) + oy)
                else:
                    b = _bilinear(R, i, j, ox, oy)
                yield a, b

    def ncc(sx, sy):
        num = np.zeros(col.shape)
        den1, den2 = num.copy(), num.copy()
        for (a, _), (b, _) in patches(sx, sy):
            a, b = a.astype(np.float64), b.astype(np.float64)
            num = num + a * b
            den1 = den1 + a * a
            den2 = den2 + b * b
        with np.errstate(all="ignore"):
            return np.where((den1 > 0) & (den2 > 0), num / np.sqrt(den1 * den2), -1.0)

    def stddev(which):
        n = np.zeros(col.shape, np.int64)
        m = np.zeros(col.shape)
        for pair in patches(dx, dy):
            v, ok = pair[which]
            n = n + ok
            m = np.where(ok, m + v.astype(np.float64), m)
        with np.errstate(all="ignore"):
            m = m / n
            s = np.zeros(col.shape)
            for pair in patches(dx, dy):
                v, ok = pair[which]
                t = v.astype(np.float64) - m
                s = np.where(ok, s + t * t, s)
            return np.where(n > 0, np.sqrt(s / n), -1.0)

    with np.errstate(all="ignore"):
        if metric == "ncc":
            val = ncc(dx, dy)
            ok = val >= 0
        elif metric == "stddev":
            ls, rs = stddev(0), stddev(1)
            ok = (ls >= 0) & (rs >= 0)
            val = (ls + rs) / 2.0
        else:
            one = np.float32(1)
            C = ncc(dx, dy)
            nb = [ncc(dx + one, dy), ncc(dx - one, dy), ncc(dx, dy + one), ncc(dx, dy - one)]
            ok = (C >= 0) & ~((nb[0] < 0) | (nb[1] < 0) | (nb[2] < 0) | (nb[3] < 0))
            kx = 2.0 * C - nb[0] - nb[1]
            ky = 2.0 * C - nb[2] - nb[3]
            ok &= (kx > 0) & (ky > 0)
            val = np.sqrt(1.0 / kx + 1.0 / ky)
            if metric == "cramer_rao":
                val = val * np.sqrt(np.maximum(1.0 - C, 0.0))
    out[row[ok], col[ok], 0] = val[ok].astype(np.float32)
    out[row[ok], col[ok], 1] = 1.0
    return out


# ---- the oracle against the restatement ---------------------------------------------------------------------------

@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("round_to_int", [False, True])
@pytest.mark.parametrize("sample_rate", [1, 2])
def test_oracle_matches_numpy_restatement(ce, metric, round_to_int, sample_rate):
    left, right, disp = scene(34, 40, seed=5, right_shape=(30, 44))
    disp[3, 4, 0] = 30.0                                  # one disparity pointing outside the right image
    left[5, 6, 0] = np.nan                                # a NaN child in a valid pixel
    for kernel, bbox, pkw in (((5, 3), None, 0.0), ((3, 7), (3, 2, 31, 27), 2.7)):
        got = ce.corr_eval(left, right, disp, kernel, metric, sample_rate, round_to_int, pkw, bbox=bbox)
        ref = np_corr_eval(left, right, disp, kernel, metric, sample_rate, round_to_int, pkw, bbox=bbox)
        assert np.array_equal(_bits(got), _bits(ref)), (kernel, bbox)
        assert got[..., 1].any()


@pytest.mark.parametrize("metric", METRICS)
def test_tiny_disparity_components(ce, metric):
    """A component far below the ulp of the position is lost in double(left_pix) + double(d): a tiny negative one samples
    at the integer position and does not lower the crop origin."""
    left, right, disp, bbox = tiny_case()
    o = ce.right_origin(left.shape, disp, (9, 7), metric, 1, False, 1.4, bbox=bbox)
    e = 1 + 2 + 7 + (1 if metric in ("parabola_curvature", "cramer_rao") else 0)
    assert o[1] == bbox[1] - 3 - e                        # floor(fl(y0 - 1e-20)) == y0
    got = ce.corr_eval(left, right, disp, (9, 7), metric, 1, False, 1.4, bbox=bbox)
    ref = np_corr_eval(left, right, disp, (9, 7), metric, 1, False, 1.4, bbox=bbox)
    assert np.array_equal(_bits(got), _bits(ref)) and got[..., 1].any()


def test_right_origin_is_the_reduced_bbox_minimum(ce):
    left, right, disp = scene(20, 24, seed=8)
    b = (2, 3, 20, 18)
    d = disp[b[1]:b[3], b[0]:b[2]]
    sel = d[..., 2] != 0
    rows, cols = np.mgrid[0:b[3] - b[1], 0:b[2] - b[0]]
    mx = int(np.floor(b[0] + cols[sel] + d[..., 0][sel].astype(np.float64)).min())
    my = int(np.floor(b[1] + rows[sel] + d[..., 1][sel].astype(np.float64)).min())
    # expand(half_kernel), expand(pixel_buffer = 1), expand(2), expand(ceil(w) + 5), and 1 more for the curvature metrics
    assert ce.right_origin(left.shape, disp, (5, 7), "ncc", 1, False, 1.5, bbox=b) == (mx - 2 - 1 - 2 - 7, my - 3 - 1 - 2 - 7)
    assert ce.right_origin(left.shape, disp, (5, 7), "cramer_rao", 1, False, 1.5, bbox=b) == (mx - 13, my - 14)


# ---- closed-form cases ----------------------------------------------------------------------------------------------

def test_ncc_is_exactly_one_for_identical_patches(ce):
    img = texture(24, 30, seed=1)
    disp = np.zeros((24, 30, 3), np.float32)
    disp[..., 2] = 1
    out = ce.corr_eval(img, img, disp, (5, 5), "ncc")
    assert out[..., 1].all()
    assert np.all(out[..., 0] == 1.0)                     # sqrt(fl(a * a)) == a, so num / sqrt(den * den) == 1


def test_integer_shift_is_recovered_at_ncc_one(ce):
    big = texture(60, 70, seed=2)
    left, right = big[10:50, 10:60], big[12:52, 7:57]     # left(x, y) = right(x + 3, y - 2)
    disp = np.zeros((40, 50, 3), np.float32)
    disp[..., 0], disp[..., 1], disp[..., 2] = 3, -2, 1
    out = ce.corr_eval(left, right, disp, (7, 5), "ncc")
    inner = out[4:-4, 3:-6]                               # windows inside both images
    assert inner[..., 1].all() and np.all(inner[..., 0] == 1.0)


def test_stddev_is_the_mean_of_the_valid_patch_stddevs(ce):
    left, right, disp = scene(30, 30, seed=3, invalid_fraction=0.2)
    disp[..., :2] = np.array([2.0, -1.0], np.float32)     # integer: the right patch is a crop
    disp[..., 2] = 1
    out = ce.corr_eval(left, right, disp, (7, 5), "stddev")
    for y, x in ((10, 10), (15, 12), (20, 18)):
        lp = left[y - 2:y + 3, x - 3:x + 4]
        rp = right[y - 3:y + 2, x - 1:x + 6]
        want = (np.std(lp[..., 0][lp[..., 1] != 0].astype(np.float64)) + np.std(rp[..., 0][rp[..., 1] != 0].astype(np.float64))) / 2
        assert out[y, x, 1] == 1 and out[y, x, 0] == pytest.approx(want, rel=1e-6)


def test_cramer_rao_sigma_shrinks_as_the_contrast_grows(ce):
    rng = np.random.default_rng(4)
    t = texture(50, 60, seed=4)
    n1, n2 = rng.normal(0, 0.3, t.shape), rng.normal(0, 0.3, t.shape)
    disp = np.zeros((50, 60, 3), np.float32)
    disp[..., 2] = 1
    med = []
    for contrast in (0.5, 2.0, 8.0):
        left, right = (contrast * t + n1).astype(np.float32), (contrast * t + n2).astype(np.float32)
        out = ce.corr_eval(left, right, disp, (9, 9), "cramer_rao")[8:-8, 8:-8]
        med.append(np.median(out[..., 0][out[..., 1] != 0]))
    assert med[0] > med[1] > med[2] > 0


def test_negative_ncc_gives_an_invalid_pixel(ce):
    # Laplacian-of-Gaussian-like data is zero mean, so an inverted right image correlates negatively
    left = texture(30, 30, seed=6)
    disp = np.zeros((30, 30, 3), np.float32)
    disp[..., 2] = 1
    for metric in ("ncc", "parabola_curvature", "cramer_rao"):
        out = ce.corr_eval(left, -left, disp, (5, 5), metric)
        assert not out[..., 1].any() and not out[..., 0].any(), metric


# ---- the details of the reference that change output bits ---------------------------------------------------------

def test_invalid_left_value_changes_ncc_but_not_stddev(ce):
    left, right, disp = scene(24, 24, seed=7, invalid_fraction=0.0)
    left[12, 12, 1] = 0.0                                 # invalid, keeps its child value
    other = left.copy()
    other[12, 12, 0] += 5.0                               # ... a different child value behind the same invalid mask
    for metric, changes in (("ncc", True), ("stddev", False)):
        a = ce.corr_eval(left, right, disp, (5, 5), metric)
        b = ce.corr_eval(other, right, disp, (5, 5), metric)
        assert (not np.array_equal(_bits(a), _bits(b))) == changes, metric


def test_prefilter_kernel_width_moves_the_origin_and_changes_bits(ce):
    left, right, disp = scene(30, 36, seed=9)
    disp[..., 0] += np.float32(0.123456789)               # fractions down to the last float bits
    o0 = ce.right_origin(left.shape, disp, (5, 5), "ncc", 1, False, 0.0)
    o1 = ce.right_origin(left.shape, disp, (5, 5), "ncc", 1, False, 200.0)
    assert o1 == (o0[0] - 200, o0[1] - 200)
    a = ce.corr_eval(left, right, disp, (5, 5), "ncc", 1, False, 0.0)
    b = ce.corr_eval(left, right, disp, (5, 5), "ncc", 1, False, 200.0)
    assert np.array_equal(a[..., 1], b[..., 1])
    assert not np.array_equal(_bits(a), _bits(b))        # the relative coordinates crossed into larger binades
    assert np.array_equal(_bits(b), _bits(np_corr_eval(left, right, disp, (5, 5), "ncc", 1, False, 200.0)))


def test_sampling_follows_the_bbox_origin(ce):
    left, right, disp = scene(20, 20, seed=10, invalid_fraction=0.0)
    a = ce.corr_eval(left, right, disp, (3, 3), "ncc", 2, bbox=(0, 0, 12, 12))
    b = ce.corr_eval(left, right, disp, (3, 3), "ncc", 2, bbox=(1, 1, 13, 13))
    assert a[0::2, 0::2, 1].all() and not a[1::2, :, 1].any() and not a[:, 1::2, 1].any()
    assert b[0::2, 0::2, 1].all() and not b[1::2, :, 1].any()
    # image pixel (1, 1) is sampled in the second bbox only
    assert a[1, 1, 1] == 0 and b[0, 0, 1] == 1


def test_round_to_int_rounds_half_away_from_zero(ce):
    left, right, _ = scene(20, 24, seed=11)
    for half, whole in ((2.5, 3.0), (-2.5, -3.0), (1.5, 2.0), (-0.5, -1.0)):
        dh, dw = smooth_disparity(20, 24, 1, invalid_fraction=0.0), smooth_disparity(20, 24, 1, invalid_fraction=0.0)
        dh[..., 0], dw[..., 0] = half, whole
        dh[..., 1], dw[..., 1] = -half, -whole
        a = ce.corr_eval(left, right, dh, (5, 5), "ncc", 1, True)
        b = ce.corr_eval(left, right, dw, (5, 5), "ncc", 1, True)
        assert np.array_equal(_bits(a), _bits(b)), half
        assert not np.array_equal(_bits(a), _bits(ce.corr_eval(left, right, dh, (5, 5), "ncc", 1, False))), half


def test_invalid_and_unsampled_disparities_are_not_checked(ce):
    left, right, disp = scene(12, 12, seed=12)
    disp[0, 0, 2] = 0
    disp[0, 0, 0] = np.nan                                # invalid
    disp[1, 1, :] = (np.inf, 0, 1)                        # valid, not sampled at rate 2
    out = ce.corr_eval(left, right, disp, (3, 3), "ncc", 2)
    assert out[0, 0, 1] == 0


# ---- argument errors -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", ["even_kernel", "zero_kernel", "metric", "size", "sample_rate", "bbox", "nan_disp", "inf_disp",
                                  "big_disp", "nan_width", "negative_padding"])
def test_argument_errors(ce, case):
    left, right, disp = scene(12, 14, seed=13)
    kw = dict(kernel_size=(3, 3), metric="ncc", sample_rate=1, round_to_int=False, prefilter_kernel_width=0.0, bbox=None)
    if case == "even_kernel":
        kw["kernel_size"] = (4, 3)
    elif case == "zero_kernel":
        kw["kernel_size"] = (3, 0)
    elif case == "metric":
        kw["metric"] = "phase"
    elif case == "size":
        disp = disp[:, :-1]
    elif case == "sample_rate":
        kw["sample_rate"] = 0
    elif case == "bbox":
        kw["bbox"] = (0, 0, 15, 12)
    elif case == "nan_disp":
        disp[2, 2, :] = (np.nan, 0, 1)
    elif case == "inf_disp":
        disp[4, 2, :] = (0, -np.inf, 1)
    elif case == "big_disp":
        disp[2, 6, :] = (16777216.0, 0, 1)
    elif case == "nan_width":
        kw["prefilter_kernel_width"] = float("nan")
    elif case == "negative_padding":
        kw["prefilter_kernel_width"] = -6.5
    with pytest.raises(ValueError):
        ce.corr_eval(left, right, disp, **kw)
