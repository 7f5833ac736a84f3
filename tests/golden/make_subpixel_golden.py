"""Writes tests/golden/subpixel.npz: PyramidSubpixelView outputs of the CPU oracle (oracle/vw_subpixel_oracle.c) for the
three algorithms on one small [0,1] pair, so that later changes to the oracle or the engine are caught bit for bit.
Run from the repository root:  python tests/golden/make_subpixel_golden.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import subpixel  # noqa: E402
from subpixel_fixtures import smooth_pair  # noqa: E402

BBOX = (6, 5, 58, 50)


def main():
    left, right, disp = smooth_pair(56, 64, seed=123)
    out = {"left": left, "right": right, "disparity": disp, "bbox": np.array(BBOX, np.int32)}
    for alg, name in ((0, "lk"), (1, "affine"), (2, "bayes_em")):
        out[name] = subpixel.pyramid_subpixel(disp, left, right, (7, 7), 1, 1.4, 2, alg, bbox=BBOX)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "subpixel.npz"), **out)


if __name__ == "__main__":
    main()
