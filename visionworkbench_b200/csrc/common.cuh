// common.cuh -- shared declarations for the vwb200 engine (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string>
#include <atomic>
#include <vector>
#include <algorithm>
#include "../../include/vwb200.h"

namespace vwb200 {

// ---- error plumbing ---------------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

#define VWB_CUDA(expr)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      ::vwb200::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return VWB200_ECUDA;                                                                  \
    }                                                                                       \
  } while (0)

#define VWB_TRY(expr)                        \
  do {                                       \
    int _rc = (expr);                        \
    if (_rc != VWB200_OK) return _rc;        \
  } while (0)

#define VWB_LAUNCH_CHECK()                                                                  \
  do {                                                                                      \
    ::vwb200::g_launches.fetch_add(1, std::memory_order_relaxed);                           \
    cudaError_t _e = cudaGetLastError();                                                    \
    if (_e != cudaSuccess) {                                                                \
      ::vwb200::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return VWB200_ECUDA;                                                                  \
    }                                                                                       \
  } while (0)

int ensure_device();   // VWB200_ENODEVICE when there is no CUDA device

// stream-ordered device buffers owned by one call
struct Arena {
  cudaStream_t st;
  std::vector<void*> ptrs;
  explicit Arena(cudaStream_t s) : st(s) {}
  ~Arena() { for (void* p : ptrs) cudaFreeAsync(p, st); }
  template <class T> int alloc(T** out, size_t n) {
    void* p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, std::max<size_t>(n, 1) * sizeof(T), st);
    if (e != cudaSuccess) { set_error("cudaMallocAsync(%zu bytes) failed: %s", n * sizeof(T), cudaGetErrorString(e)); return VWB200_ENOMEM; }
    ptrs.push_back(p);
    *out = static_cast<T*>(p);
    return VWB200_OK;
  }
};

// ---- image descriptors (device pointers) ------------------------------------------------------
struct ImgF { const float* p; int w, h; ptrdiff_t pitch; };
struct ImgB { const uint8_t* p; int w, h; ptrdiff_t pitch; };

// A zone of the level loop (Stereo/CorrelationView.cc:607-648) or a whole calc_disparity call.
struct Zone {
  long long obase;   // element offset of the zone's output (0,0) in the output buffer
  int opitch;        // output row pitch (elements)
  int w, h;          // output size
  int lx, ly;        // left_region.min  (kernel-padded) in left image coordinates
  int rx, ry;        // right_region.min in right image coordinates
  int sx, sy;        // search volume
  int addx, addy;    // constant added to the children by the K1 epilogue (R->L pass: -search size)
  int nchunks;       // > 1: the disparity range is split over several CTAs (K1G_DCHUNK disparities each)
  int pad0;
  long long sbase;   // element offset of this zone's partial results in the scratch planes [chunk][h][w]
};
// One unit of work of the generic kernel: a TW x TH tile of a zone (x one chunk of its disparity range).
struct Tile { int zone; int tx, ty; int chunk; };

// ---- K1 generic (fp64, any float input, zones) --------------------------------------------
// cost: VWB200_* cost type.  inv_l / inv_r: for NCC, 1/boxsum(v^2) maps whose (0,0) sits at window
// origin (l_ox,l_oy) / (r_ox,r_oy) in image coordinates, pitch in elements.
struct NccMaps { const double* inv_l; int l_ox, l_oy, l_w, l_h; const double* inv_r; int r_ox, r_oy, r_w, r_h; };
// optional event pair recorded around the dominant kernel (kernel-only timing for the roofline)
struct KEvents { cudaEvent_t e0 = nullptr, e1 = nullptr; };
int k1_generic_launch(int cost, ImgF left, ImgF right, const Zone* d_zones, const Tile* d_tiles, int ntiles,
                      int kx, int ky, NccMaps ncc, vwb200_dispi* out, double* scratch_cost, int* scratch_idx, bool clamp_reads,
                      int stage_r_floats, cudaStream_t st, const KEvents* ev = nullptr,    // stage_r_floats: 0 = read through L1
                      const int* zone_gate = nullptr);                                     // != nullptr: only tiles of zones with gate[zone] != 0
bool k1_generic_can_stage(int kx, int ky, int sx, int sy, int nchunks);
long long k1_generic_stage_floats(int kx, int ky, int sx, int sy, int nchunks);
static constexpr int K1G_DCHUNK = 256;
// merge the per-chunk partial results of split zones (zone indices in d_split)
int k1_generic_merge_launch(int cost, const Zone* d_zones, const int* d_split, int nsplit, const double* scratch_cost,
                            const int* scratch_idx, vwb200_dispi* out, cudaStream_t st);
int k1_generic_tile_w(int kx);
int k1_generic_tile_h(int ky);
// ---- K1 zone-int (k1_zone_int.cu): the zone kernel in exact int32 for integer-valued imagery (level 0 of 8-bit rasters) ----
// range = vmax - vmin of both rasters; *ib_out = log2 of the disparities one warp covers (larger zones are split in chunks)
bool k1_zone_int_supported(int cost, int kx, int ky, long long range, int* ib_out);
int k1_zone_int_tile_w(int k);
int k1_zone_int_tile_h();
long long k1_zone_int_stage_u16(int k, int sx, int sy, int nchunks, int ib);
long long k1_zone_int_stage_max();
// zone_flag[zone] is set when a tile of the zone met a non-integer pixel (mean-filled masked pixels): the caller re-runs those
// zones through the fp64 zone kernel
int k1_zone_int_launch(int cost, ImgF left, ImgF right, const Zone* d_zones, const Tile* d_tiles, int ntiles, int k, float vmin, float vmax,
                       int warp_u16, vwb200_dispi* out, double* scratch_cost, int* scratch_idx, int* zone_flag, cudaStream_t st,
                       const KEvents* ev = nullptr);
// integer-valued rasters of a zone batch: enables the zone-int kernel in run_k1_zones.  checked: some pixels were replaced by
// a (non-integer) mean, zones that touch them fall back to the fp64 kernel
struct ZoneIntMode { bool on; float vmin, vmax; bool checked; };
// 1/boxsum(v*v) over window origins [ox0,ox0+ow) x [oy0,oy0+oh) with clamped (constant edge) reads.
int box_sq_inv_launch(ImgF img, int kx, int ky, int ox0, int oy0, int ow, int oh, double* out, cudaStream_t st);
// boxsum(v) (centred == 0) or boxsum((v - c)^2) (centred == 1) as int32 over the same window-origin domain (integer imagery)
int box_sum_i32_launch(ImgF img, int kx, int ky, int ox0, int oy0, int ow, int oh, int* out, cudaStream_t st, int centred = 0,
                       float c = 0.0f);
// left/right are whole images; the logical rasters start at (lox,loy) / (rox,roy) (constant edge extension outside),
// (addx,addy) is added to every output disparity (R->L pass of the level loop)
struct FastOrigin { int lox, loy, rox, roy, addx, addy; };
// NCC / wide-range SquaredCost on the exact-integer path with fp32 screening (k1_screen.cu)
int k1_screen_supported(int cost, int kx, int ky, int sx, int sy, float vmin, float vmax, bool integer_valued);
size_t k1_screen_workspace_bytes(int cost, int W, int H, int sx, int sy, int kx, int ky);
int k1_screen_launch(int cost, ImgF left, ImgF right, int W, int H, int sx, int sy, int kx, int ky, float vmin, float vmax,
                     vwb200_dispi* out, ptrdiff_t opitch, void* workspace, cudaStream_t st, const KEvents* ev = nullptr,
                     const FastOrigin* org = nullptr);
// ---- SemiGlobalMatcher (k5_sgm.cu, k5_sgm_paths.cu; declarations in k5_sgm.cuh) ---------------
// exact sequential re-evaluation of pixels flagged NaN by k1 (NCC zero-energy windows)
int k1_nan_fixup_launch(int cost, ImgF left, ImgF right, const Zone* d_zones, int nzones, int kx, int ky,
                        NccMaps ncc, vwb200_dispi* out, cudaStream_t st, int gridx = 8);

// left/right are whole images; the logical rasters start at (lox,loy) / (rox,roy) (constant edge extension outside),
// (addx,addy) is added to every output disparity (R->L pass of the level loop)
// ---- K1 fast (exact-integer path, single big zone) -------------------------------------------
// Returns VWB200_ENOIMPL if the configuration is outside what the fast path handles.
int k1_fast_supported(int cost, int kx, int ky, int sx, int sy, float vmin, float vmax, bool integer_valued);
int k1_fast_launch(int cost, ImgF left, ImgF right, int W, int H, int sx, int sy, int kx, int ky, float vmin,
                   vwb200_dispi* out, ptrdiff_t opitch, void* workspace, size_t workspace_bytes, cudaStream_t st,
                   const KEvents* ev = nullptr, const struct FastOrigin* org = nullptr);
size_t k1_fast_workspace_bytes(int W, int H, int sx, int sy, int kx, int ky);
// min / max / integer-valuedness of an image (device reduction); result[0]=min,[1]=max,[2]=all-integers(1/0)
int image_stats_launch(ImgF img, float* d_result3, cudaStream_t st);

// ---- K2 pyramid ---------------------------------------------------------------------------------
int crop_extend_f32_launch(ImgF src, int x0, int y0, int w, int h, float* dst, ptrdiff_t dpitch, cudaStream_t st);
int crop_extend_u8_launch(ImgB src, int x0, int y0, int w, int h, int zero_outside, uint8_t* dst, ptrdiff_t dpitch, cudaStream_t st);
// masked mean over every 2nd pixel (CorrelationView.cc:133-136): d_acc = {double sum, double count}
int masked_mean_launch(ImgF img, ImgB mask, double* d_acc2, cudaStream_t st);
int mean_fill_launch(float* img, int w, int h, ptrdiff_t pitch, ImgB mask, const double* d_acc2, cudaStream_t st);
int mask_any_zero_launch(ImgB mask, int* d_flag, cudaStream_t st);      // *d_flag = 1 if the mask holds a zero (caller zeroes it)
int pyramid_down_launch(ImgF in, float* out, ptrdiff_t opitch, cudaStream_t st);
int subsample_mask_launch(ImgB in, uint8_t* out, ptrdiff_t opitch, cudaStream_t st);
// gaussian (separable, constant edge) into out via work; then Laplacian (mode 1) or img - g (mode 2)
int sepconv_launch(ImgF in, const float* d_taps, int n, float* work, float* out, cudaStream_t st);
int prefilter_final_launch(ImgF img, const float* g, int mode, float* out, cudaStream_t st);

// ---- K3 / K4 -------------------------------------------------------------------------------------
int consistency_launch(vwb200_dispi* l2r, int lw, int lh, ptrdiff_t lpitch, const vwb200_dispi* r2l, int rw, int rh,
                       ptrdiff_t rpitch, float thr, cudaStream_t st, int qax = 0, int qay = 0, float* diff = nullptr, ptrdiff_t dpitch = 0,
                       int dox = 0, int doy = 0);
int diff_invalidate_launch(const vwb200_dispi* disp, int w, int h, float* diff, ptrdiff_t dpitch, int dox, int doy, cudaStream_t st);
int sgm_finalize_launch(const float* sub, const vwb200_dispi* disp, int w, int ax, int ay, float* out, ptrdiff_t opitch_px, int ox, int oy,
                        int ow, int oh, cudaStream_t st);
// disparity_blob_filter; work: 2 * w * h ints
int blob_filter_launch(vwb200_dispi* d, int w, int h, int area, int* work, cudaStream_t st);
// pass 1 of the outlier filter evaluated over [x0,x0+ow) x [y0,y0+oh) of the constant-edge-extended input
int rm_outliers_launch(const vwb200_dispi* in, int w, int h, int hx, int hy, double pt, double rt,
                       int x0, int y0, int ow, int oh, vwb200_dispi* out, cudaStream_t st);
// pass 2 (1,1,3.0,0.20) reading the padded pass-1 buffer (w+2)x(h+2)
int cleanup_pass2_launch(const vwb200_dispi* p1, int w, int h, vwb200_dispi* out, cudaStream_t st);
int disparity_mask_launch(const vwb200_dispi* in, int w, int h, ImgB lmask, ImgB rmask, vwb200_dispi* out, cudaStream_t st);
// out[i] = {dx+ax, dy+ay, valid} as float triples (CorrelationView.cc:880-884)
int finalize_launch(const vwb200_dispi* in, int w, int h, int ax, int ay, float* out, ptrdiff_t opitch_px,
                    int ox, int oy, int ow, int oh, cudaStream_t st);

// ---- a11 ParabolaSubpixelView -------------------------------------------------------------------------
int disp_range_launch(const float* disp, int cols, int bx0, int by0, int bw, int bh, int* d_r5, cudaStream_t st);
int meansub_region_launch(const float* e, const float* g, int ew, int m, int w, int h, float* out, cudaStream_t st);
int log_region_launch(const float* g, int gw, int gx0, int gy0, int iw, int ih, int rx0, int ry0, int w, int h, float* out, cudaStream_t st);
int parabola_launch(const float* disp, int cols, int bx0, int by0, int bw, int bh, const float* L, int lw, const float* R, int rw,
                    int srx0, int sry0, int kx, int ky, float* out, cudaStream_t st);

// ---- K6 PyramidSubpixelView (k6_subpixel.cu) ------------------------------------------------------------
int k6_range_launch(const float* disp, int cols, int bx0, int by0, int bw, int bh, int* d_r5, cudaStream_t st);
int k6_disp_crop_launch(const float* disp, int cols, int rows, int x0, int y0, int w, int h, float tx, float ty, float* out, cudaStream_t st);
int k6_disp_out_launch(const float* patch, int pw, int ox, int oy, float tx, float ty, int w, int h, float* out, ptrdiff_t opitch, cudaStream_t st);
int k6_level_run(int alg, float* disp, const float* L, int w, int h, const float* R, int rw, int rh, int kx, int ky,
                 int rx0, int ry0, int rx1, int ry1, Arena& ar, cudaStream_t st, vwb200_subpixel_stats* stats);
int k6_pyramid_run(int alg, float* D, const float* L, const float* R, int pw, int ph, int kx, int ky, int bw, int bh, int levels,
                   Arena& ar, cudaStream_t st, vwb200_subpixel_stats* stats);

// ---- K7 CorrEval (k7_corr_eval.cu) ------------------------------------------------------------------------
// d_org3 = {min over the sampled valid pixels of col + floor(dx), of row + floor(dy), bad-disparity flag}
int k7_origin_launch(const float* D, ptrdiff_t dpitch, int x0, int y0, int bw, int bh, int sample_rate, int round_to_int, int* d_org3,
                     cudaStream_t st);
// writes nothing when d_org3[2] is set
int k7_corr_eval_launch(const float* L, int lw, int lh, ptrdiff_t lpitch, const float* R, int rw, int rh, ptrdiff_t rpitch,
                        const float* D, ptrdiff_t dpitch, int x0, int y0, int bw, int bh, int kx, int ky, int metric, int sample_rate,
                        int round_to_int, int margin, const int* d_org3, float* out, ptrdiff_t opitch, cudaStream_t st);

// ---- host-side restatement-free logic -----------------------------------------------------------
struct Box { int x0, y0, x1, y1; };
struct HostZone { Box img; Box disp; };
// quad-tree search-range refinement (behaviour of Stereo/Correlation.cc:139-328), host side.
void subdivide_regions_host(const vwb200_dispi* disp, int w, int h, int kx, int ky, std::vector<HostZone>& out);

}  // namespace vwb200
