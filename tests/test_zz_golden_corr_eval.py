"""Pins the CorrEval oracle, and the engine on a GPU, to tests/golden/corr_eval.npz
(tests/golden/make_corr_eval_golden.py)."""
import os

import numpy as np
import pytest

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "corr_eval.npz")
METRICS = ("ncc", "stddev", "parabola_curvature", "cramer_rao")
KERNEL, SAMPLE_RATE, PREFILTER_KERNEL_WIDTH = (9, 7), 2, 1.4


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_oracle_corr_eval_golden():
    from oracle import corr_eval
    g = np.load(G)
    for metric in METRICS:
        for rnd in (0, 1):
            got = corr_eval.corr_eval(g["left"], g["right"], g["disparity"], KERNEL, metric, SAMPLE_RATE, bool(rnd),
                                      PREFILTER_KERNEL_WIDTH, bbox=tuple(g["bbox"]))
            assert np.array_equal(_bits(got), _bits(g[f"{metric}_{rnd}"])), (metric, rnd)
            assert g[f"{metric}_{rnd}"][..., 1].any()


@pytest.mark.gpu
def test_gpu_corr_eval_golden():
    import visionworkbench_b200 as v
    g = np.load(G)
    for metric in METRICS:
        for rnd in (0, 1):
            got = v.CorrEval(g["left"], g["right"], g["disparity"], KERNEL, metric, SAMPLE_RATE, bool(rnd), 0,
                             PREFILTER_KERNEL_WIDTH).rasterize(None, tuple(g["bbox"]))
            assert np.array_equal(_bits(got), _bits(g[f"{metric}_{rnd}"])), (metric, rnd)
