"""Writes tests/golden/corr_eval.npz: CorrEval outputs of the CPU oracle (oracle/vw_corr_eval_oracle.c) for the four
metrics, with and without round_to_int, on one small masked pair, so that later changes to the oracle or the engine are
caught bit for bit.  Run from the repository root:  python tests/golden/make_corr_eval_golden.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import corr_eval  # noqa: E402
from corr_eval_fixtures import METRICS, scene  # noqa: E402

BBOX = (5, 4, 55, 44)
KERNEL = (9, 7)
SAMPLE_RATE = 2
PREFILTER_KERNEL_WIDTH = 1.4


def main():
    left, right, disp = scene(48, 60, seed=77, right_shape=(44, 66))
    out = {"left": left, "right": right, "disparity": disp, "bbox": np.array(BBOX, np.int32)}
    for metric in METRICS:
        for rnd in (0, 1):
            out[f"{metric}_{rnd}"] = corr_eval.corr_eval(left, right, disp, KERNEL, metric, SAMPLE_RATE, bool(rnd),
                                                         PREFILTER_KERNEL_WIDTH, bbox=BBOX)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "corr_eval.npz"), **out)


if __name__ == "__main__":
    main()
