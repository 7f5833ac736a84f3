"""GPU tests of PyramidSubpixelView and the three level functions: bit-identical to the sequential CPU oracle
(values, validity and the values kept by invalidated pixels)."""
import threading

import numpy as np
import pytest

from subpixel_fixtures import chain_case, check_error, kat_case, smooth_pair

pytestmark = pytest.mark.gpu

ALGS = [0, 1, 2]


@pytest.fixture(scope="module")
def vwb():
    import visionworkbench_b200 as v
    assert v.device_count() > 0
    return v


@pytest.fixture(scope="module")
def sp():
    from oracle import subpixel
    subpixel.build()
    return subpixel


def _same(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("alg", ALGS)
@pytest.mark.parametrize("levels", [0, 1, 2, 3])
def test_pyramid_parity_levels(vwb, sp, alg, levels):
    left, right, disp = smooth_pair(96, 112, seed=20 + levels)
    bbox = (20, 16, 84, 72)
    got = vwb.PyramidSubpixelView(disp, left, right, 0, 0.0, (7, 7), levels, alg).rasterize(None, bbox)
    ref = sp.pyramid_subpixel(disp, left, right, (7, 7), 0, 0.0, levels, alg, bbox=bbox)
    assert _same(got, ref)


@pytest.mark.parametrize("alg", ALGS)
@pytest.mark.parametrize("mode,width", [(0, 0.0), (1, 1.4), (2, 2.0)])
def test_pyramid_parity_prefilters(vwb, sp, alg, mode, width):
    left, right, disp = smooth_pair(80, 80, seed=31)
    got = vwb.PyramidSubpixelView(disp, left, right, mode, width, (5, 5), 2, alg).rasterize(None, (10, 10, 70, 70))
    ref = sp.pyramid_subpixel(disp, left, right, (5, 5), mode, width, 2, alg, bbox=(10, 10, 70, 70))
    assert _same(got, ref)


@pytest.mark.parametrize("bbox", [(0, 0, 40, 30), (40, 0, 72, 30), (0, 30, 40, 64), (40, 30, 72, 64), (0, 0, 72, 64)])
def test_pyramid_parity_borders(vwb, sp, bbox):
    left, right, disp = smooth_pair(64, 72, seed=40)
    got = vwb.bayes_em_subpixel(disp, left, right, 1, 1.4, (7, 7)).rasterize(None, bbox)
    ref = sp.pyramid_subpixel(disp, left, right, (7, 7), 1, 1.4, 2, 2, bbox=bbox)
    assert _same(got, ref)


@pytest.mark.parametrize("alg", ALGS)
def test_level_functions_with_roi(vwb, sp, alg):
    left, right, disp = smooth_pair(60, 70, seed=50)
    fn = [vwb.subpixel_optimized_LK_2d, vwb.subpixel_optimized_affine_2d, vwb.subpixel_optimized_affine_2d_EM][alg]
    for roi, k in (((10, 8, 40, 30), (7, 7)), ((0, 0, 70, 60), (9, 5)), ((50, 40, 70, 60), (3, 3))):
        got = fn(disp, left, right, k[0], k[1], roi)
        ref = sp.subpixel_level(alg, disp, left, right, k, roi=roi)
        assert _same(got, ref), (roi, k)


def test_unnormalised_input_takes_the_failed_solve_path(vwb, sp):
    # 12-bit-like values: Bayes-EM likelihoods underflow, gamma = 0/0 = NaN, posv fails for most pixels
    left, right, disp = smooth_pair(64, 64, seed=60, scale=4095.0)
    for alg in ALGS:
        got = vwb.PyramidSubpixelView(disp, left, right, 0, 0.0, (7, 7), 2, alg).rasterize()
        ref = sp.pyramid_subpixel(disp, left, right, (7, 7), 0, 0.0, 2, alg)
        assert _same(got, ref)
    got = vwb.bayes_em_subpixel(disp, left, right, 0, 0.0, (7, 7)).rasterize()
    assert (got[..., 2] == 0).mean() > 0.5


def test_invalidation_chain_fixpoint(vwb, sp):
    left, right, disp = chain_case()
    got = vwb.subpixel_optimized_affine_2d_EM(disp, left, right, 3, 3, (0, 0, 40, 24))
    stats = vwb.last_subpixel_stats()
    ref = sp.subpixel_level(2, disp, left, right, (3, 3))
    assert stats["fixpoint_rounds"] >= 3
    assert _same(got, ref)
    assert (got[10, 10:30, 2] == 0).all()


def test_reference_kat_thresholds_on_gpu(vwb, sp):
    for istretch, max_err, max_invalid in ((95, 0.35, 12), (90, 0.36, 12), (80, 0.52, 22), (70, 0.9, 48)):
        left, right, disp, stretch, translation = kat_case(istretch)
        got = vwb.bayes_em_subpixel(disp, left, right, vwb.PREFILTER_LOG, 1.4, (7, 7)).rasterize()
        assert _same(got, sp.pyramid_subpixel(disp, left, right, (7, 7), 1, 1.4, 2, 2))
        err, invalid = check_error(got, stretch, translation)
        assert err < max_err and invalid <= max_invalid


def test_device_pointers_on_a_caller_stream(vwb, sp):
    import torch
    left, right, disp = smooth_pair(72, 72, seed=70)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        tl, tr, td = (torch.from_numpy(a).cuda() for a in (left, right, disp))
        out = vwb.subpixel_optimized_affine_2d(td, tl, tr, 7, 7, (0, 0, 72, 72))
    s.synchronize()
    assert _same(out.cpu().numpy(), sp.subpixel_level(1, disp, left, right, (7, 7)))


def test_calls_from_several_threads(vwb, sp):
    cases = [smooth_pair(64, 64, seed=80 + i) for i in range(6)]
    res = [None] * len(cases)

    def run(i):
        l, r, d = cases[i]
        res[i] = vwb.PyramidSubpixelView(d, l, r, 1, 1.4, (7, 7), 2, i % 3).rasterize()

    th = [threading.Thread(target=run, args=(i,)) for i in range(len(cases))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for i, (l, r, d) in enumerate(cases):
        assert _same(res[i], sp.pyramid_subpixel(d, l, r, (7, 7), 1, 1.4, 2, i % 3))


def test_errors(vwb):
    left, right, disp = smooth_pair(32, 32)
    with pytest.raises(vwb.NoImplErr):
        vwb.PyramidSubpixelView(disp, left, right, 0, 0.0, (5, 5), 2, vwb.SUBPIXEL_PHASE).rasterize()
    with pytest.raises(vwb.ArgumentErr):
        vwb.PyramidSubpixelView(disp, left, right, 0, 0.0, (4, 5), 2, 0).rasterize()
    with pytest.raises(vwb.ArgumentErr):
        vwb.PyramidSubpixelView(disp, left, right, 0, 0.0, (5, 5), 2, 0).rasterize(None, (0, 0, 40, 10))
    with pytest.raises(vwb.NoImplErr):
        vwb.PyramidSubpixelView(disp, left, right, 0, 0.0, (5, 5), 2, 0)(0, 0)
