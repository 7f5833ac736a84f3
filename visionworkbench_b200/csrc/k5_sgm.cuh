// k5_sgm.cuh -- declarations shared by the SemiGlobalMatcher kernels (SURVEY section 8, row a10).
//
// Data in HBM (all ragged buffers follow the reference's m_buffer_starts order: raster order over the output pixels,
// dy-major / dx-minor inside a pixel's search box, Stereo/SGM.cc:677-731):
//   SgmMeta meta[ow*oh]   16 B / pixel : the pixel's search box (inclusive, int16), the offset of its first entry in the
//                                        ragged buffers, its left grey value (u8) and its number of disparities
//   uint8   cost[total]    1 B / entry : Hamming cost of the census signatures (get_hamming_distance_costs, SGM.cc:39-73)
//   uint16  accum[total]   2 B / entry : sum of the path costs of the eight directions (m_accum_buffer)
#pragma once
#include "common.cuh"

namespace vwb200 {

typedef uint8_t sgm_cost_t;     // SemiGlobalMatcher::CostType      (SGM.h:81)
typedef uint16_t sgm_accum_t;   // SemiGlobalMatcher::AccumCostType (SGM.h:82)

struct SgmGeom {
  int sx, sy;                  // max disparity (inclusive); min disparity is 0 (calc_disparity_sgm, SGM.cc:167-230)
  int ndx, ndy, nd;            // sx + 1, sy + 1, their product
  int p1, p2;
  int ow, oh, min_col, min_row;
  int lw, clw, crw, hk;        // left width, census widths, half kernel
};

// one 16-byte record per output pixel; loaded as a uint4
struct __align__(16) SgmMeta {
  short b0, b1, b2, b3;        // search box min_x, min_y, max_x, max_y (inclusive); (0,0,-1,-1) = no search area
  unsigned start;              // first entry of this pixel in cost[] / accum[]
  unsigned val_n;              // bits 0..7: left grey value; bits 8..31: number of disparities
};

struct SgmBox { int b0, b1, b2, b3; };
__host__ __device__ inline int sgm_box_n(int b0, int b1, int b2, int b3) {      // get_num_disparities (SGM.h:244-251)
  return (b2 < b0 || b3 < b1) ? 0 : (b2 - b0 + 1) * (b3 - b1 + 1);
}

// everything one calc_disparity_sgm call needs (device pointers)
struct SgmArgs {
  ImgF left, right;            // the cropped left_region / right_region rasters
  int sx = 0, sy = 0, k = 5;
  int ternary = 0, ternary_threshold = 5;
  int p1 = 0, p2 = 0;
  int use_mgm = 0, subpixel_mode = 0;
  int buf_x = 2, buf_y = 2;
  int conserve_level = -1;     // -1: the reference's retry loop over the levels 0..3 (SGM.cc:476-497)
  double memory_limit_mb = 6000.0;
  int assumed_threads = 4;     // vw_settings().default_num_threads() in calc_main_buf_size (SGM.cc:715-716)
  ImgB lmask{nullptr, 0, 0, 0}, rmask{nullptr, 0, 0, 0};
  const vwb200_dispi* prev = nullptr; int pw = 0, ph = 0; ptrdiff_t ppitch = 0;
  const int* bounds_in = nullptr;      // ow * oh * 4 ints: use these boxes instead of deriving them
  int* bounds_out = nullptr;           // ow * oh * 4 ints (optional)
  vwb200_dispi* out = nullptr; ptrdiff_t opitch = 0;
  float* out_sub = nullptr; ptrdiff_t sub_pitch = 0;   // floats per row
  int bounds_only = 0;
};

int sgm_output_size(int lw, int lh, int rw, int rh, int sx, int sy, int k, int* ow, int* oh);
int sgm_run(const SgmArgs& a, Arena& ar, cudaStream_t st);
// search boxes only (populate_disp_bound_image + constrain_disp_bound_image, SGM.cc:241-668) for an ow x oh output
int sgm_bounds_run(const SgmArgs& a, int ow, int oh, int* d_bounds, Arena& ar, cudaStream_t st);

// k5_sgm_paths.cu
int sgm_paths_launch(const SgmMeta* meta, const sgm_cost_t* cost, sgm_accum_t* const* accum, const SgmGeom& g, unsigned max_n,
                     unsigned max_w, unsigned max_h, Arena& ar, cudaStream_t st);
int mgm_paths_launch(const SgmMeta* meta, const sgm_cost_t* cost, sgm_accum_t* accum, const uint8_t* left8, const SgmGeom& g,
                     size_t total, Arena& ar, cudaStream_t st);

}  // namespace vwb200
