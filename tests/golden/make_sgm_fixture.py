"""Store the SemiGlobalMatcher known-answer images (Vision Workbench's src/vw/Stereo/tests/left.tif and
left_const_offset.tif, used by TestSGM.cxx:27-75) as tests/golden/sgm_fixture.npz, which tests/test_oracle_sgm.py reads.

  python tests/golden/make_sgm_fixture.py <Vision Workbench source tree>/src/vw/Stereo/tests

The right file is the left one shifted by (2, 1).  Only a 256 x 256 interior ROI of the left image and the right ROI that
calc_disparity_sgm sees for it (search [-4, 4]^2) are kept, as the files' own 8-bit values."""
import os
import sys

import numpy as np
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))
X0, Y0, SIZE, SMIN, SRANGE = 8, 8, 256, -4, 9


def main(src):
    left = np.array(Image.open(os.path.join(src, "left.tif")))
    right = np.array(Image.open(os.path.join(src, "left_const_offset.tif")))
    assert left.dtype == right.dtype == np.uint8
    rx, ry = X0 + SMIN, Y0 + SMIN
    np.savez_compressed(os.path.join(HERE, "sgm_fixture.npz"),
                        left=left[Y0:Y0 + SIZE, X0:X0 + SIZE], right=right[ry:ry + SIZE + SRANGE, rx:rx + SIZE + SRANGE],
                        search_min=np.array((SMIN, SMIN)), offset=np.array((2, 1)))


if __name__ == "__main__":
    main(sys.argv[1])
