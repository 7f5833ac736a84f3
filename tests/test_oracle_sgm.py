"""SemiGlobalMatcher core of the oracle (oracle/vw_sgm_oracle.c; SURVEY section 8 row a10): pinned by the reference's own
known-answer test (Stereo/tests/TestSGM.cxx:27-75: constant offset (2,1), search [-4,4]^2, census 3x3, > 99 % correct)
-- on a stored crop of the reference's fixture images, and on a synthetic equivalent."""
import os

import numpy as np
import pytest

SGM_FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sgm_fixture.npz")


def _constant_offset_pair(seed, W=180, H=150, off=(2, 1), smin=(-4, -4), ssize=(9, 9)):
    """left ROI and the right ROI calc_disparity_sgm is given in TestSGM.cxx:47-52 (right = left ROI + search min,
    grown by the search size), for a right image that is the left one shifted by `off`."""
    rng = np.random.default_rng(seed)
    base = np.floor(rng.random((H + 60, W + 60)) * 256)
    # a little spatial correlation, like a real image
    base = np.floor((base + np.roll(base, 1, 0) + np.roll(base, 1, 1) + np.roll(base, (1, 1), (0, 1))) / 4).astype(np.float32)
    x0 = y0 = 30
    left = base[y0:y0 + H, x0:x0 + W]
    ox, oy = x0 + smin[0] - off[0], y0 + smin[1] - off[1]
    right = base[oy:oy + H + ssize[1], ox:ox + W + ssize[0]]
    return np.ascontiguousarray(left), np.ascontiguousarray(right)


@pytest.mark.parametrize("kernel", [3, 5, 7, 9])
def test_sgm_constant_offset_synthetic(oracle, kernel):
    left, right = _constant_offset_pair(7 + kernel)
    d = oracle.sgm_calc_disparity(left, right, (8, 8), kernel)      # search volume (9, 9) -> inclusive maxima (8, 8)
    hk = (kernel - 1) // 2
    assert d.shape == (left.shape[0] - 2 * hk, left.shape[1] - 2 * hk, 3)   # SGM.cc:2404-2420
    dd = d[..., :2] + np.array([-4, -4])
    correct = ((dd[..., 0] == 2) & (dd[..., 1] == 1)).mean()
    assert correct > 0.99, correct
    assert (d[..., 2] == 1).all()


def test_sgm_textureless_image_is_deterministic(oracle):
    """All costs tie: select_best_disparity's smoothing iterations (SGM.cc:1196-1288) must terminate and be repeatable."""
    left = np.full((40, 50), 100.0, np.float32)
    right = np.full((48, 58), 100.0, np.float32)
    a = oracle.sgm_calc_disparity(left, right, (8, 8), 3)
    b = oracle.sgm_calc_disparity(left, right, (8, 8), 3)
    assert np.array_equal(a, b) and a.shape[2] == 3


def test_sgm_rejects_unsupported_kernel(oracle):
    left, right = _constant_offset_pair(1, 60, 50)
    with pytest.raises(ValueError):
        oracle.sgm_calc_disparity(left, right, (8, 8), 11)      # NoImplErr in the reference (SGM.cc:1885-1888)


def test_sgm_reference_fixture_kat(oracle):
    # TestSGM.cxx uses leftRoi (0,0,400,400), whose right ROI starts at (-4,-4); the stored interior ROI of its images
    # (tests/golden/make_sgm_fixture.py) avoids reading outside the file
    g = np.load(SGM_FIXTURE)
    left, right = g["left"].astype(np.float32), g["right"].astype(np.float32)
    d = oracle.sgm_calc_disparity(left, right, (8, 8), 3)
    dd = d[..., :2] + g["search_min"]
    assert ((dd[..., 0] == g["offset"][0]) & (dd[..., 1] == g["offset"][1])).mean() > 0.99


def test_sgm_per_pixel_boxes_reduce_to_the_constant_case(oracle):
    """The per-pixel-box entry (what round 2's device kernels consume) with the full box everywhere must equal the
    constant-box pipeline bit for bit, integer and sub-pixel."""
    left, right = _constant_offset_pair(21, 90, 70)
    oh, ow = oracle.sgm_output_shape(left, right, (8, 8), 5)
    full = np.tile(np.array([0, 0, 8, 8], np.int32), (oh, ow, 1))
    bi, bf = oracle.sgm_calc_disparity_bounds(left, right, (8, 8), 5, full, subpixel_mode=5)
    ci, cf = oracle.sgm_calc_disparity_subpixel(left, right, (8, 8), 5, 5)
    assert np.array_equal(bi, ci) and np.array_equal(bf, cf)


def test_sgm_per_pixel_boxes_ragged(oracle):
    """Random sub-boxes around the truth, empty boxes (-> invalid pixels) and single-disparity boxes."""
    rng = np.random.default_rng(5)
    left, right = _constant_offset_pair(22, 100, 80)
    oh, ow = oracle.sgm_output_shape(left, right, (8, 8), 3)
    b = np.empty((oh, ow, 4), np.int32)
    b[..., 0] = rng.integers(0, 7, (oh, ow)); b[..., 1] = rng.integers(0, 6, (oh, ow))          # truth is (6, 5) in box coordinates
    b[..., 2] = np.minimum(8, np.maximum(b[..., 0], 6) + rng.integers(0, 3, (oh, ow)))
    b[..., 3] = np.minimum(8, np.maximum(b[..., 1], 5) + rng.integers(0, 4, (oh, ow)))
    empty = rng.random((oh, ow)) < 0.05
    b[empty] = (0, 0, -1, -1)
    single = (rng.random((oh, ow)) < 0.05) & ~empty
    b[single] = (6, 5, 6, 5)
    di, df = oracle.sgm_calc_disparity_bounds(left, right, (8, 8), 3, b, subpixel_mode=5)
    assert (di[empty] == 0).all() and (df[empty] == 0).all()
    ok = ~empty
    assert (di[ok][:, 2] == 1).all()
    inside = (di[..., 0] >= b[..., 0]) & (di[..., 0] <= b[..., 2]) & (di[..., 1] >= b[..., 1]) & (di[..., 1] <= b[..., 3])
    assert inside[ok].all()
    assert ((di[..., 0] == 6) & (di[..., 1] == 5))[ok].mean() > 0.97
    assert np.abs(df[ok][:, :2] - di[ok][:, :2]).max() <= 1.0      # sub-pixel offsets stay inside one pixel


def test_sgm_disp_bounds_from_previous_level(oracle):
    """populate_disp_bound_image / constrain_disp_bound_image (SGM.cc:241-668): trusted prior -> 2 * d +- buffer clipped to
    the search box; priors on the edge of a >= 10 wide search are not trusted; untrusted pixels take the hull of the
    trusted boxes within 10 pixels, grown by 2 (or the full box when there is none); masks zero the box."""
    oh, ow, search, buf = 40, 50, (19, 11), (2, 3)
    ok, b = oracle.sgm_disp_bounds((oh, ow), search, buf)                       # no prior: the constant box (:231-239)
    assert ok and (b == np.array([0, 0, 19, 11])).all()
    prev = np.zeros((20, 25, 3), np.int32)
    prev[..., 0] = 4; prev[..., 1] = 3; prev[..., 2] = 1                         # -> (8, 6) at this level
    prev[:, :5, 2] = 0                                                           # invalid prior on the left
    prev[10:, 20:, 0] = 0                                                        # dx = 0 is on the edge of a 20-wide search: not trusted
    ok, b = oracle.sgm_disp_bounds((oh, ow), search, buf, prev=prev)
    assert ok
    assert (b[5, 20] == np.array([6, 3, 10, 9])).all()
    # untrusted pixel within 10 px of trusted ones: hull (6,3)-(10,9) expanded by 2, cropped to the search box
    assert (b[5, 5] == np.array([4, 1, 12, 11])).all()
    # untrusted pixel farther than 10 px from any trusted one keeps the full box at conservation level 0 ...
    prev2 = prev.copy(); prev2[:, :, 2] = 0; prev2[0, 24, 2] = 1
    ok, b2 = oracle.sgm_disp_bounds((oh, ow), search, buf, prev=prev2)
    assert (b2[30, 5] == np.array([0, 0, 19, 11])).all()
    # ... and loses its search area at level 1 (:633-640)
    ok, b3 = oracle.sgm_disp_bounds((oh, ow), search, buf, prev=prev2, conserve_level=1)
    assert (b3[39, 0] == np.array([0, 0, -1, -1])).all()
    # left mask
    lm = np.full((oh, ow), 255, np.uint8); lm[:4] = 0
    ok, b4 = oracle.sgm_disp_bounds((oh, ow), search, buf, prev=prev, lmask=lm)
    assert (b4[:4] == np.array([0, 0, -1, -1])).all() and (b4[5, 20] == b[5, 20]).all()
    # the boxes feed the ragged core
    left, right = _constant_offset_pair(23, 60, 50, off=(2, 1), smin=(0, 0), ssize=(20, 12))
    shape = oracle.sgm_output_shape(left, right, search, 3)
    prev = np.zeros(((shape[0] + 1) // 2, (shape[1] + 1) // 2, 3), np.int32); prev[..., 0] = 1; prev[..., 1] = 1; prev[..., 2] = 1
    ok, bb = oracle.sgm_disp_bounds(shape, search, buf, prev=prev)
    di, _ = oracle.sgm_calc_disparity_bounds(left, right, search, 3, bb)
    assert ((di[..., 0] == 2) & (di[..., 1] == 1)).mean() > 0.99


def test_mgm_accumulation(oracle):
    """MGM (accum_mgm_multithread, SGM.cc:2619-2700): same KAT shape as TestSGM.cxx with use_mgm = true -- the constant
    offset is recovered; the accumulated costs differ from plain SGM (two predecessors averaged), so the sub-pixel part does too."""
    left, right = _constant_offset_pair(31, 120, 90)
    oh, ow = oracle.sgm_output_shape(left, right, (8, 8), 3)
    full = np.tile(np.array([0, 0, 8, 8], np.int32), (oh, ow, 1))
    mi, mf = oracle.sgm_calc_disparity_bounds(left, right, (8, 8), 3, full, subpixel_mode=5, use_mgm=True)
    si, sf = oracle.sgm_calc_disparity_bounds(left, right, (8, 8), 3, full, subpixel_mode=5)
    dd = mi[..., :2] + np.array([-4, -4])
    assert ((dd[..., 0] == 2) & (dd[..., 1] == 1)).mean() > 0.99
    assert not np.array_equal(mf, sf)
    mi2, mf2 = oracle.sgm_calc_disparity_bounds(left, right, (8, 8), 3, full, subpixel_mode=5, use_mgm=True)
    assert np.array_equal(mi, mi2) and np.array_equal(mf, mf2)
    # ragged boxes and empty pixels go through the MGM sweeps as well
    b = full.copy(); b[10:20, 10:30] = (0, 0, -1, -1); b[40:50, :, 0] = 4; b[40:50, :, 1] = 3
    ri, _ = oracle.sgm_calc_disparity_bounds(left, right, (8, 8), 3, b, use_mgm=True)
    assert (ri[10:20, 10:30] == 0).all() and (ri[45, :, 0] >= 4).all()


# ---- the reference's own known-answer vectors for the pieces the SGM branch of the view adds ---------------------------------
_CENSUS_SRC = np.array([[1, 2, 7, 2, 2, 8, 5, 2], [1, 4, 2, 9, 8, 8, 2, 6], [5, 2, 7, 2, 2, 2, 4, 6], [1, 2, 2, 2, 1, 4, 5, 2],
                        [6, 6, 3, 7, 2, 2, 5, 5], [1, 2, 9, 2, 2, 2, 2, 2], [7, 9, 2, 8, 5, 2, 3, 2], [1, 2, 2, 2, 2, 2, 2, 1]], np.uint8)


def test_census_reference_kat(oracle):
    """Image/tests/TestCensusTransform.cxx:25-46 (src(col,row) listed row by row)."""
    cv = lambda c, r, k: oracle.census_value(_CENSUS_SRC, c, r, k)
    assert cv(2, 2, 3) == 0x20 and cv(4, 5, 3) == 0x86 and cv(6, 1, 3) == 0xDB
    assert cv(4, 4, 5) == 0x0088F60D and cv(2, 3, 5) == 0x005D03C4
    assert cv(3, 4, 7) == 0x00001C0000041400


def test_ternary_census_semantics(oracle):
    """Image/CensusTransform.h:167-220: per neighbour 00 / 01 / 11 in reverse raster order, centre skipped; the band is
    [centre - t, centre + t].  Checked against a direct evaluation of the definition; 5x5 keeps 32 of its 48 bits (SGM.cc:1789-1803)."""
    img = _CENSUS_SRC
    def direct(c, r, k, t):
        hk = k // 2
        out, shift = 0, 0
        for rr in range(r + hk, r - hk - 1, -1):
            for cc in range(c + hk, c - hk - 1, -1):
                if rr == r and cc == c:
                    continue
                v, ce = int(img[rr, cc]), int(img[r, c])
                if v >= ce - t:
                    out |= (3 if v > ce + t else 1) << shift
                shift += 2
        return out
    for (c, r) in [(2, 2), (4, 5), (3, 3)]:
        assert oracle.census_value(img, c, r, 3, True, 2) == direct(c, r, 3, 2)
        assert oracle.census_value(img, c, r, 5, True, 1) == direct(c, r, 5, 1) & 0xFFFFFFFF
    assert direct(3, 3, 5, 1) > 0xFFFFFFFF          # the truncation does drop bits here


def test_blob_filter_reference_kat(oracle):
    """Image/tests/TestBlobIndex.cxx:42-59 (three 8-connected blobs) and :101-124 (blob sizes 7, 2, 3) through
    disparity_blob_filter's rule: blobs of at most `area` pixels are eroded (BlobIndex.h:444-453, CorrelationView.cc:242-271)."""
    m = np.zeros((5, 7), np.int32)
    m[1, 1:4] = 1; m[3, 2:4] = 1; m[1:4, 5] = 1; m[2, 6] = 1          # sizes 3, 2, 4 (the last joined through the (6,2) pixel)
    d = np.zeros((5, 7, 3), np.int32); d[..., 0] = 9; d[..., 1] = 7; d[..., 2] = m
    assert (oracle.disparity_blob_filter(d, 1)[..., 2] == m).all()
    assert oracle.disparity_blob_filter(d, 2)[..., 2].sum() == 7 and oracle.disparity_blob_filter(d, 2)[3, 2:4, 2].sum() == 0
    assert oracle.disparity_blob_filter(d, 3)[..., 2].sum() == 4
    e = oracle.disparity_blob_filter(d, 4)
    assert e[..., 2].sum() == 0 and (e[m == 1] == 0).all() and (e[m == 0][:, 0] == 9).all()   # eroded pixels become result_type()
    img = np.array([[0, 0, 0, 1, 8, 0], [0, 1, 0, 0, 0, 0], [0, 1, 0, 0, 1, 1], [1, 1, 0, 0, 0, 1], [1, 0, 1, 0, 0, 0], [0, 1, 0, 0, 0, 0]])
    d = np.zeros((6, 6, 3), np.int32); d[..., 2] = img != 0
    assert oracle.disparity_blob_filter(d, 2)[..., 2].sum() == 10          # the 2-blob goes
    assert oracle.disparity_blob_filter(d, 3)[..., 2].sum() == 7           # ... and the 3-blob
    assert oracle.disparity_blob_filter(d, 6)[..., 2].sum() == 7 and oracle.disparity_blob_filter(d, 7)[..., 2].sum() == 0


def test_parabola_subpixel_mode_and_full_entry(oracle):
    """vwo_calc_disparity_sgm == the older entry points where they overlap; SUBPIXEL_PARABOLA offsets stay inside the
    half-pixel circle (ParabolaFit2d::find_peak, SGMAssist.h:99-134) and the integer part is untouched."""
    left, right = _constant_offset_pair(3, 90, 70)
    a = oracle.sgm_calc_disparity(left, right, (8, 8), 5)
    bi, bf, bb = oracle.calc_disparity_sgm(left, right, (8, 8), 5, subpixel_mode=1)
    assert np.array_equal(a, bi) and (bb == np.array([0, 0, 8, 8])).all()
    off = bf[..., :2] - bi[..., :2]
    assert np.hypot(off[..., 0], off[..., 1]).max() <= 0.5 + 1e-6 and np.abs(off).max() > 0.01
    ci, cf = oracle.sgm_calc_disparity_subpixel(left, right, (8, 8), 5, 5)
    di, df_, _ = oracle.calc_disparity_sgm(left, right, (8, 8), 5, subpixel_mode=5)
    assert np.array_equal(ci, di) and np.array_equal(cf, df_)
    ti, _, _ = oracle.calc_disparity_sgm(left, right, (8, 8), 5, cost_type=4)            # ternary census recovers the offset too
    assert ((ti[..., 0] == 6) & (ti[..., 1] == 5)).mean() > 0.99
    with pytest.raises(ValueError):
        oracle.calc_disparity_sgm(left, right, (8, 8), 5, cost_type=0)                    # NoImplErr (SGM.cc:1888-1892)


@pytest.mark.parametrize("algorithm", [1, 2, 3])
def test_view_sgm_branch_recovers_a_constant_offset(oracle, algorithm):
    """PyramidCorrelationView with algorithm SGM / MGM / FINAL_MGM (CorrelationView.cc:392-595): the statistical bar of
    Stereo/tests/TestPyramidCorrelationView.cxx (>= 0.9 correct, >= 0.99 valid) on a constant shift, with the R->L check,
    the filters and the sub-pixel stage on."""
    rng = np.random.default_rng(5)
    W, H, off = 200, 160, (3, -2)
    base = np.floor(rng.random((H + 40, W + 40)) * 256)
    base = np.floor((base + np.roll(base, 1, 0) + np.roll(base, 1, 1) + np.roll(base, (1, 1), (0, 1))) / 4).astype(np.float32)
    left = np.ascontiguousarray(base[20:20 + H, 20:20 + W]); right = np.ascontiguousarray(base[20 - off[1]:20 - off[1] + H, 20 - off[0]:20 - off[0] + W])
    p = oracle.make_params((-8, -8, 9, 9), (5, 5), cost=3, consistency_threshold=2.0, min_consistency_level=0, filter_half_kernel=3,
                           max_pyramid_levels=2, algorithm=algorithm, sgm_subpixel_mode=5)
    d = oracle.pyramid_correlate(p, left, right, bbox=(20, 20, 180, 140))
    ok = (np.abs(d[..., 0] - off[0]) < 0.5) & (np.abs(d[..., 1] - off[1]) < 0.5) & (d[..., 2] == 1)
    # the R->L pass loses the rows whose partner lies above the left tile: populate_disp_bound_image takes the column extent
    # of the right mask from the row of the LEFT pixel (SGM.cc:343-359), which is empty there -- reference behaviour
    assert ok.mean() > 0.88 and (ok | (d[..., 2] == 0)).all(), (ok.mean(), (d[..., 2] == 1).mean())
    assert (d[20:, :, 2] == 1).mean() > 0.99
    assert (d[..., 0] != np.rint(d[..., 0])).mean() > 0.3          # sub-pixel offsets were applied
