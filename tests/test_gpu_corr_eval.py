"""GPU tests of CorrEval: bit-identical to the sequential CPU oracle (values and validity, compared as uint32)."""
import threading

import numpy as np
import pytest

from corr_eval_fixtures import METRICS, scene, tiny_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vwb():
    import visionworkbench_b200 as v
    assert v.device_count() > 0
    return v


@pytest.fixture(scope="module")
def ce():
    from oracle import corr_eval
    corr_eval.build()
    return corr_eval


def _same(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _check(vwb, ce, left, right, disp, kernel, metric, sample_rate=1, round_to_int=False, pkw=0.0, bbox=None):
    got = vwb.CorrEval(left, right, disp, kernel, metric, sample_rate, round_to_int, 0, pkw).rasterize(None, bbox)
    ref = ce.corr_eval(left, right, disp, kernel, metric, sample_rate, round_to_int, pkw, bbox=bbox)
    assert _same(got, ref), f"{metric} {kernel} round={round_to_int} rate={sample_rate} bbox={bbox}: " \
                            f"{int((got.view(np.uint32) != ref.view(np.uint32)).any(-1).sum())} mismatches"
    return got


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("kernel", [(3, 3), (5, 7), (21, 21), (35, 35)])
@pytest.mark.parametrize("round_to_int", [False, True])
@pytest.mark.parametrize("sample_rate", [1, 3])
def test_parity(vwb, ce, metric, kernel, round_to_int, sample_rate):
    left, right, disp = scene(72, 80, seed=31)
    got = _check(vwb, ce, left, right, disp, kernel, metric, sample_rate, round_to_int, 1.4, bbox=(6, 5, 70, 61))
    assert got[..., 1].any()


@pytest.mark.parametrize("metric", METRICS)
def test_bboxes_touching_each_border(vwb, ce, metric):
    left, right, disp = scene(50, 66, seed=32)
    for bbox in ((0, 7, 30, 40), (20, 0, 50, 30), (40, 10, 66, 45), (5, 25, 45, 50), (0, 0, 66, 50)):
        _check(vwb, ce, left, right, disp, (7, 5), metric, 1, False, 0.0, bbox)


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("round_to_int", [False, True])
def test_right_size_outside_masks_and_non_finite_children(vwb, ce, metric, round_to_int):
    left, right, disp = scene(48, 56, seed=33, right_shape=(37, 71), invalid_fraction=0.15)
    disp[10:20, 30:40, 0] += 60.0                         # points outside the right image
    disp[30:34, 5:9, 1] -= 45.0
    left[8, 9, 0], left[20, 21, 0] = np.nan, np.inf       # non-finite children, valid and invalid
    left[20, 21, 1] = 0
    right[15, 17, 0], right[25, 30, 0] = -np.inf, np.nan
    right[25, 30, 1] = 0
    _check(vwb, ce, left, right, disp, (9, 7), metric, 1, round_to_int, 3.2)
    _check(vwb, ce, left, right, disp, (9, 7), metric, 2, round_to_int, 3.2, bbox=(3, 4, 50, 41))


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("round_to_int", [False, True])
def test_tiny_disparity_components(vwb, ce, metric, round_to_int):
    # components of 1e-30 .. 3e-9 of both signs, one of them at the crop's minimum: the coordinate must be rounded in
    # the reference's order, double(left_pix) + double(d) and then - right_box.min()
    left, right, disp, bbox = tiny_case()
    got = _check(vwb, ce, left, right, disp, (9, 7), metric, 1, round_to_int, 1.4, bbox)
    assert got[..., 1].any()


def test_large_kernel_reads_the_left_image_unstaged(vwb, ce):
    left, right, disp = scene(40, 44, seed=34)
    for metric in METRICS:
        _check(vwb, ce, left, right, disp, (63, 61), metric, 2, False, 0.0, bbox=(4, 3, 40, 37))


def test_bbox_without_valid_disparity(vwb, ce):
    left, right, disp = scene(30, 30, seed=35)
    disp[5:15, 5:15, 2] = 0
    disp[5:15, 5:15, 0] = np.nan                          # invalid values are never looked at
    for metric in METRICS:
        got = _check(vwb, ce, left, right, disp, (5, 5), metric, 1, False, 0.0, bbox=(5, 5, 15, 15))
        assert not got.any()


def test_two_dimensional_images_are_all_valid(vwb, ce):
    left, right, disp = scene(30, 34, seed=36)
    got = vwb.CorrEval(left[..., 0], right[..., 0], disp, (5, 5), "ncc", 1, False).rasterize()
    ref = ce.corr_eval(left[..., 0], right[..., 0], disp, (5, 5), "ncc")
    assert _same(got, ref)


def test_device_tensors_on_a_caller_stream(vwb, ce):
    import torch
    left, right, disp = scene(64, 72, seed=37)
    ref = ce.corr_eval(left, right, disp, (11, 9), "cramer_rao", 1, False, 2.0, bbox=(4, 6, 60, 58))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        tl, tr, td = (torch.from_numpy(a).cuda() for a in (left, right, disp))
        got = vwb.CorrEval(tl, tr, td, (11, 9), "cramer_rao", 1, False, 0, 2.0).rasterize(None, (4, 6, 60, 58))
        assert got.is_cuda
        host = got.cpu()
    s.synchronize()
    assert _same(host.numpy(), ref)
    # a 2-D device image is all valid
    got2 = vwb.CorrEval(torch.from_numpy(left[..., 0]).cuda(), torch.from_numpy(right[..., 0]).cuda(), torch.from_numpy(disp).cuda(),
                        (5, 5), "ncc", 1, False).rasterize()
    assert _same(got2.cpu().numpy(), ce.corr_eval(left[..., 0], right[..., 0], disp, (5, 5), "ncc"))


def test_concurrent_calls_from_threads(vwb, ce):
    left, right, disp = scene(80, 96, seed=38)
    tiles = [(x, y, x + 32, y + 40) for y in (0, 40) for x in (0, 32, 64)]
    refs = {(m, t): ce.corr_eval(left, right, disp, (7, 7), m, 1, m == "stddev", 0.0, bbox=t) for m in METRICS for t in tiles}
    views = {m: vwb.CorrEval(left, right, disp, (7, 7), m, 1, m == "stddev") for m in METRICS}
    got, errors = {}, []

    def run(m, t):
        try:
            got[(m, t)] = views[m].rasterize(None, t)
        except Exception as e:  # noqa: BLE001 -- reported below
            errors.append(e)

    th = [threading.Thread(target=run, args=(m, t)) for m in METRICS for t in tiles]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors
    assert all(_same(got[k], refs[k]) for k in refs)


def test_caller_dest(vwb, ce):
    import torch
    left, right, disp = scene(40, 48, seed=40)
    bbox = (4, 4, 36, 30)
    ref = ce.corr_eval(left, right, disp, (5, 5), "ncc", 1, False, bbox=bbox)
    view = vwb.CorrEval(left, right, disp, (5, 5), "ncc", 1, False)
    big = np.full((40, 48, 2), 7.0, np.float32)
    view.rasterize(big[4:30, 4:36], bbox)                 # a strided view of a larger buffer
    assert _same(big[4:30, 4:36], ref) and np.all(big[:4] == 7.0)
    tview = vwb.CorrEval(*(torch.from_numpy(a).cuda() for a in (left, right, disp)), (5, 5), "ncc", 1, False)
    tbig = torch.full((40, 48, 2), 7.0, device="cuda")
    tview.rasterize(tbig[4:30, 4:36], bbox)
    assert _same(tbig[4:30, 4:36].cpu().numpy(), ref)
    for bad in (np.empty((26, 31, 2), np.float32), np.empty((26, 32, 2), np.float64), np.empty((26, 32, 2), np.float32)[:, ::-1],
                np.empty((2, 26, 32), np.float32).transpose(1, 2, 0)):
        with pytest.raises(vwb.ArgumentErr):
            view.rasterize(bad, bbox)
    for bad in (np.empty((26, 32, 2), np.float32), torch.empty((26, 32, 2), device="cuda", dtype=torch.float64),
                torch.empty((26, 32, 2)), torch.empty((26, 33, 2), device="cuda")):
        with pytest.raises(vwb.ArgumentErr):
            tview.rasterize(bad, bbox)


@pytest.mark.parametrize("case", ["even_kernel", "metric", "size", "sample_rate", "bbox", "nan_disp", "big_disp", "nan_width",
                                  "negative_padding", "mixed_inputs"])
def test_argument_errors(vwb, case):
    left, right, disp = scene(12, 14, seed=39)
    args = dict(kernel_size=(3, 3), metric="ncc", sample_rate=1, round_to_int=False, prefilter_kernel_width=0.0)
    bbox = None
    if case == "even_kernel":
        args["kernel_size"] = (3, 2)
    elif case == "metric":
        args["metric"] = "phase"
    elif case == "size":
        disp = disp[:-1]
    elif case == "sample_rate":
        args["sample_rate"] = 0
    elif case == "bbox":
        bbox = (-1, 0, 5, 5)
    elif case == "nan_disp":
        disp[4, 4, :] = (np.nan, 0, 1)
    elif case == "big_disp":
        disp[2, 2, :] = (0, -16777216.0, 1)
    elif case == "nan_width":
        args["prefilter_kernel_width"] = float("nan")
    elif case == "negative_padding":
        args["prefilter_kernel_width"] = -7.0
    elif case == "mixed_inputs":
        import torch
        left = torch.from_numpy(left).cuda()
    dest = np.full((12, 14, 2), 7.0, np.float32) if bbox is None else None
    with pytest.raises(vwb.ArgumentErr):
        vwb.CorrEval(left, right, disp, **args).rasterize(dest, bbox)
    if dest is not None:
        assert np.all(dest == 7.0)                        # nothing is written on a rejected call
