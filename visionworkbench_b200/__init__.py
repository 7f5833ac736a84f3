"""visionworkbench_b200 -- B200-native rasteriser for Vision Workbench's dense stereo correlation
hot path (vw::stereo::PyramidCorrelationView / calc_disparity / best_of_search_convolution and the
SeparableConvolutionView pyramid feeder), the sub-pixel views and CorrEval.  Product code: hand-written sm_100a kernels in csrc/,
reached through the C ABI of include/vwb200.h.  No CPU path, no oracle imports.
"""
from .api import *  # noqa: F401,F403
from .api import lib, device_count, kernel_launches, last_k1_stats, last_subpixel_stats  # noqa: F401
