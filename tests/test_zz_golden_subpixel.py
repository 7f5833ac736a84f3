"""Pins the sub-pixel refinement oracle, and the engine on a GPU, to tests/golden/subpixel.npz
(tests/golden/make_subpixel_golden.py)."""
import os

import numpy as np
import pytest

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "subpixel.npz")
ALGS = ((0, "lk"), (1, "affine"), (2, "bayes_em"))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_oracle_subpixel_golden():
    from oracle import subpixel
    g = np.load(G)
    for alg, name in ALGS:
        got = subpixel.pyramid_subpixel(g["disparity"], g["left"], g["right"], (7, 7), 1, 1.4, 2, alg, bbox=tuple(g["bbox"]))
        assert np.array_equal(_bits(got), _bits(g[name])), name


@pytest.mark.gpu
def test_gpu_subpixel_golden():
    import visionworkbench_b200 as v
    g = np.load(G)
    for alg, name in ALGS:
        got = v.PyramidSubpixelView(g["disparity"], g["left"], g["right"], 1, 1.4, (7, 7), 2, alg).rasterize(None, tuple(g["bbox"]))
        assert np.array_equal(_bits(got), _bits(g[name])), name
