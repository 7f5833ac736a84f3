/*
 * vwb200.h -- C ABI of the B200-native stereo-correlation engine.
 *
 * This is the drop-in boundary for Vision Workbench's dense block-matching path.  VW has no
 * FFI: its "operator API" is the compile-time ImageViewBase<> concept
 * (src/vw/Image/ImageViewBase.h:57-122).  The C++ shim include/vwb200/PyramidCorrelationView.h
 * keeps that concept (prerasterize()/rasterize()) and calls the functions below; no C++ or
 * torch types cross this boundary -- plain pointers, sizes and POD structs only.
 *
 * Conventions
 *  - images are row-major, one plane, pitch in ELEMENTS (vw::ImageView, Image/ImageView.h:226-227)
 *  - boxes are half-open [x0,x1) x [y0,y1) (vw::BBox2i, Math/BBox.tcc)
 *  - integer disparity pixel = {int32 dx, int32 dy, int32 valid(0/1)}   (PixelMask<Vector2i>)
 *  - float   disparity pixel = {float dx, float dy, float valid(0/1)}   (PixelMask<Vector2f>,
 *    Image/PixelMask.h:52-54: 12 bytes)
 *  - every function returns 0 on success or a negative VWB200_E* code; vwb200_last_error()
 *    gives the message of the calling thread's last failure.  The shim maps codes to
 *    vw::ArgumentErr / MathErr / LogicErr (Core/Exception.h:225-253).
 *  - "on_device" != 0 means the pointers are CUDA device pointers on the current device;
 *    otherwise they are host pointers and the call stages them through HBM itself.
 *  - `stream` is a cudaStream_t (or NULL for the library's own per-call stream).  All calls
 *    block until their result is complete unless stated otherwise.
 *  - all entry points are thread-safe (VW calls prerasterize() concurrently from its tile
 *    thread pool, Image/ImageIO.h:228-235).
 *  - there is NO CPU fallback: without a CUDA device every compute call fails with
 *    VWB200_ENODEVICE.
 */
#ifndef VWB200_H
#define VWB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VWB200_OK          0
#define VWB200_EARG       -1   /* -> vw::ArgumentErr */
#define VWB200_EMATH      -2   /* -> vw::MathErr     */
#define VWB200_ELOGIC     -3   /* -> vw::LogicErr    */
#define VWB200_ENOIMPL    -4   /* -> vw::NoImplErr   */
#define VWB200_ECUDA      -5   /* CUDA runtime failure */
#define VWB200_ENODEVICE  -6   /* no CUDA device: the engine has no CPU path */
#define VWB200_ENOMEM     -7

/* vw::stereo::CostFunctionType, src/vw/Stereo/CostFunctions.h:143-149 */
enum { VWB200_ABSOLUTE_DIFFERENCE = 0, VWB200_SQUARED_DIFFERENCE = 1, VWB200_CROSS_CORRELATION = 2,
       VWB200_CENSUS_TRANSFORM = 3, VWB200_TERNARY_CENSUS_TRANSFORM = 4 };
/* vw::stereo::CorrelationAlgorithm, src/vw/Stereo/CorrelationAlgorithms.h:29-35 */
enum { VWB200_CORRELATION_BM = 0, VWB200_CORRELATION_SGM = 1, VWB200_CORRELATION_MGM = 2, VWB200_CORRELATION_FINAL_MGM = 3 };
/* vw::stereo::SemiGlobalMatcher::SgmSubpixelMode, src/vw/Stereo/SGM.h:93-99 */
enum { VWB200_SUBPIXEL_NONE = 0, VWB200_SUBPIXEL_PARABOLA = 1, VWB200_SUBPIXEL_LINEAR = 2, VWB200_SUBPIXEL_POLY4 = 3,
       VWB200_SUBPIXEL_COSINE = 4, VWB200_SUBPIXEL_LC_BLEND = 5 };
/* vw::stereo::PrefilterModeType, src/vw/Stereo/PrefilterEnum.h:24-28 */
enum { VWB200_PREFILTER_NONE = 0, VWB200_PREFILTER_LOG = 1, VWB200_PREFILTER_MEANSUB = 2 };

typedef struct { int32_t dx, dy, valid; } vwb200_dispi;

const char* vwb200_last_error(void);
int vwb200_device_count(void);          /* number of visible CUDA devices (0 if none) */
const char* vwb200_version(void);

/* ---------------------------------------------------------------------------------------------
 * K1: vw::stereo::calc_disparity (src/vw/Stereo/Correlation.h:50-57, Correlation.cc:330-375)
 * -> best_of_search_convolution (Correlation.cc:33-137).
 * left  : (W+kx-1) x (H+ky-1) float; right: at least (W+kx-1+sx-1) x (H+ky-1+sy-1) float.
 * out   : W x H vwb200_dispi, disparities in [0,sx) x [0,sy), first-in-raster-order wins ties,
 *         pixel invalid iff every disparity gave the same cost (Correlation.cc:121-133).
 * ------------------------------------------------------------------------------------------- */
int vwb200_calc_disparity(int cost_type,
                          const float* left,  int lw, int lh, ptrdiff_t lpitch,
                          const float* right, int rw, int rh, ptrdiff_t rpitch,
                          int sx, int sy, int kx, int ky,
                          vwb200_dispi* out, ptrdiff_t opitch,
                          int on_device, void* stream);

/* Statistics of the last vwb200_calc_disparity on this thread: which kernel path ran
 * (0 = exact-integer fast path, 1 = general fp64 path), kernel launches issued, and the device time of
 * the dominant (fused cost-volume + arg-best) kernel measured with CUDA events on its stream. */
typedef struct { int32_t path; int32_t launches; float kernel_ms; int32_t reserved; } vwb200_k1_stats;
int vwb200_last_k1_stats(vwb200_k1_stats* out);

/* ---------------------------------------------------------------------------------------------
 * K2: one Gaussian-pyramid level = subsample(separable_convolution_filter(in,{1,4,6,4,1}/16),2)
 * (src/vw/Stereo/CorrelationView.cc:210-214; Image/Convolution.h:275-328; Image/Filter.h:89-99;
 *  Image/Manipulation.h:238-251).  out is (1+(w-1)/2) x (1+(h-1)/2).  Bit-exact in float.
 * ------------------------------------------------------------------------------------------- */
int vwb200_pyramid_down(const float* in, int w, int h, ptrdiff_t pitch,
                        float* out, ptrdiff_t opitch, int on_device, void* stream);
/* vw::stereo::prefilter_image (src/vw/Stereo/PreFilter.h:75-95): NONE / LaplacianOfGaussian(width) /
 * SubtractedMean(width); gaussian_filter + laplacian_filter of src/vw/Image/Filter.h:204-237,318-335. */
int vwb200_prefilter(const float* in, int w, int h, ptrdiff_t pitch, int mode, float width,
                     float* out, ptrdiff_t opitch, int on_device, void* stream);
/* SubsampleMaskByTwoFunc, src/vw/Stereo/CorrelationView.cc:38-63 */
int vwb200_subsample_mask_by_two(const uint8_t* in, int w, int h, ptrdiff_t pitch,
                                 uint8_t* out, ptrdiff_t opitch, int on_device, void* stream);

/* K3: vw::stereo::cross_corr_consistency_check (src/vw/Stereo/Correlate.cc:1441-1502), in place */
int vwb200_cross_corr_consistency_check(vwb200_dispi* l2r, int lw, int lh, ptrdiff_t lpitch,
                                        const vwb200_dispi* r2l, int rw, int rh, ptrdiff_t rpitch,
                                        float threshold, int on_device, void* stream);

/* K4: rm_outliers_using_thresh / disparity_cleanup_using_thresh / disparity_mask
 * (src/vw/Stereo/DisparityMap.h:318-442, :97-253).  in/out are w x h, dense pitch. */
int vwb200_rm_outliers_using_thresh(const vwb200_dispi* in, int w, int h, int half_h, int half_v,
                                    double pixel_threshold, double rejection_threshold,
                                    vwb200_dispi* out, int on_device, void* stream);
int vwb200_disparity_cleanup_using_thresh(const vwb200_dispi* in, int w, int h, int half_h, int half_v,
                                          double pixel_threshold, double rejection_threshold,
                                          vwb200_dispi* out, int on_device, void* stream);
int vwb200_disparity_mask(const vwb200_dispi* in, int w, int h,
                          const uint8_t* left_mask, const uint8_t* right_mask, int rmw, int rmh,
                          vwb200_dispi* out, int on_device, void* stream);

/* ---------------------------------------------------------------------------------------------
 * vw::stereo::ParabolaSubpixelView::rasterize(dest, bbox) (src/vw/Stereo/ParabolaSubpixelView.h:27-117,
 * .cc:31-330): 3x3 AbsoluteCost patch around the integer disparity, 6x9 pseudo-inverse parabola fit,
 * offset kept when its norm is below 5.  disparity: cols x rows PixelMask<Vector2f> triples (same size as
 * the left image); dest: (x1-x0) x (y1-y0) triples.  Floats agree with the reference within 1e-5.
 * ------------------------------------------------------------------------------------------- */
int vwb200_parabola_subpixel(const float* disparity, int cols, int rows, const float* left, ptrdiff_t lpitch,
                             const float* right, int rcols, int rrows, ptrdiff_t rpitch, int kx, int ky,
                             int prefilter_mode, float prefilter_width, int x0, int y0, int x1, int y1,
                             float* dest, ptrdiff_t dest_pitch, int on_device, void* stream);

/* ---------------------------------------------------------------------------------------------
 * vw::stereo::PyramidSubpixelView::rasterize(dest, bbox) (src/vw/Stereo/SubpixelView.h:42-150,
 * .cc:33-224): iterative sub-pixel refinement of a PixelMask<Vector2f> disparity over an image pyramid
 * of max_pyramid_levels levels (< 0 is clamped to 0).  Arguments as vwb200_parabola_subpixel, plus the
 * algorithm (PyramidSubpixelView_Algorithm).  dest: (x1-x0) x (y1-y0) triples, pitch in pixels.
 * Results are bit-identical to the sequential reference order (DESIGN.md section K6).
 * Odd kernel >= 3 and a bbox inside the image, else VWB200_EARG; SUBPIXEL_PHASE or an unknown
 * algorithm -> VWB200_ENOIMPL.  A disparity value in the bbox that is NaN, infinite or of magnitude >= 2^24 -> VWB200_EARG.
 * The call synchronises the stream (the disparity range is read back, and one flag per validity-fixpoint round).
 * ------------------------------------------------------------------------------------------- */
#define VWB200_SUBPIXEL_LUCAS_KANADE 0
#define VWB200_SUBPIXEL_FAST_AFFINE  1
#define VWB200_SUBPIXEL_BAYES_EM     2
#define VWB200_SUBPIXEL_PHASE        3
int vwb200_pyramid_subpixel(const float* disparity, int cols, int rows, const float* left, ptrdiff_t lpitch,
                            const float* right, int rcols, int rrows, ptrdiff_t rpitch, int kx, int ky,
                            int prefilter_mode, float prefilter_width, int x0, int y0, int x1, int y1,
                            float* dest, ptrdiff_t dest_pitch, int on_device, void* stream,
                            int max_pyramid_levels, int algorithm);
/* One level function, in place: subpixel_optimized_LK_2d / subpixel_optimized_affine_2d /
 * subpixel_optimized_affine_2d_EM (Stereo/Correlate.cc:500-1391, Correlate.h:63-104).  disparity: cols x rows
 * triples (pitch in pixels), left: cols x rows, right: rcols x rrows.  roi = [x0,x1) x [y0,y1); the scan
 * covers the roi grown by one pixel, clipped to the kernel's reach of the image. */
int vwb200_subpixel_refine(int algorithm, float* disparity, int cols, int rows, ptrdiff_t dpitch,
                           const float* left, ptrdiff_t lpitch, const float* right, int rcols, int rrows, ptrdiff_t rpitch,
                           int kx, int ky, int x0, int y0, int x1, int y1, int do_h, int do_v, int on_device, void* stream);
/* Counters of the calling thread's last vwb200_pyramid_subpixel / vwb200_subpixel_refine call.
 * SIMT efficiency = window_evaluations / lane_slots. */
typedef struct {
  long long levels;               /* level-function runs */
  long long fixpoint_rounds;      /* validity-fixpoint rounds summed over the levels */
  long long pixels;               /* pixels in the scan regions */
  long long pixels_reevaluated;   /* evaluations after round 0 */
  long long window_evaluations;   /* window-pixel evaluations (passes x kx x ky) */
  long long lane_slots;           /* sum over warps of 32 x the largest per-lane evaluation count */
} vwb200_subpixel_stats;
int vwb200_last_subpixel_stats(vwb200_subpixel_stats* out);

/* ---------------------------------------------------------------------------------------------
 * vw::stereo::CorrEval::prerasterize(bbox) (src/vw/Stereo/CorrEval.h:56-129, CorrEval.cc:139-317): the quality of a
 * float disparity at every sampled pixel of bbox = [x0,x1) x [y0,y1), as the NCC of the kx x ky patches around the
 * left pixel and the right position pixel + disparity (bilinear unless round_to_int), the mean of the two patch
 * standard deviations, or a localisation sigma from the curvature of the NCC peak.
 * left: lw x lh, right: rw x rh PixelMask<float> = {value, valid} float pairs (pitch in pixels); disparity: lw x lh
 * PixelMask<Vector2f> triples (dpitch in pixels); dest: (x1-x0) x (y1-y0) pairs (dest_pitch in pixels).  Pixels that
 * are not sampled, whose disparity is invalid or whose metric fails are {0, invalid}.
 * VWB200_EARG: a kernel that is not positive and odd, an unknown metric, sample_rate < 1, a bbox outside the left
 * image, a prefilter_kernel_width whose padding ceil(w) + 5 is NaN, negative or above 2^20, or a sampled valid
 * disparity in the bbox that is NaN, infinite or of magnitude >= 2^24 (dest is then left untouched).
 * Bit-identical to the sequential reference order (DESIGN.md section K7).  The call synchronises the stream.
 * ------------------------------------------------------------------------------------------- */
#define VWB200_CORR_EVAL_NCC                0
#define VWB200_CORR_EVAL_STDDEV             1
#define VWB200_CORR_EVAL_PARABOLA_CURVATURE 2
#define VWB200_CORR_EVAL_CRAMER_RAO         3
int vwb200_corr_eval(const float* left, int lw, int lh, ptrdiff_t lpitch, const float* right, int rw, int rh, ptrdiff_t rpitch,
                     const float* disparity, ptrdiff_t dpitch, int kx, int ky, int metric, int sample_rate, int round_to_int,
                     float prefilter_kernel_width, int x0, int y0, int x1, int y1, float* dest, ptrdiff_t dest_pitch,
                     int on_device, void* stream);

/* ---------------------------------------------------------------------------------------------
 * vw::stereo::calc_disparity_sgm (src/vw/Stereo/SGM.cc:167-230, SGM.h:361-376) ->
 * SemiGlobalMatcher::semi_global_matching_func (:2387-2448): u8_convert, (ternary) census costs for kernel 3/5/7/9,
 * per-pixel search boxes, SGM or MGM accumulation along 8 directions, integer winner with the reference's tie
 * smoothing, optional sub-pixel stage.  left / right are the cropped left_region / right_region rasters (any float
 * range).  Disparities lie in [0, search_x] x [0, search_y] (inclusive = search_volume of the reference).
 * out receives out_w x out_h pixels (row pitch opitch elements; the size is (:2397-2420) and can be queried first
 * with all outputs NULL).
 * ------------------------------------------------------------------------------------------- */
/* the simple form: the same search box for every pixel (populate_constant_disp_bound_image, :231-239), plain
 * census costs, no masks, no previous disparity; p1 / p2 <= 0 select the reference's defaults (:108-157) */
int vwb200_sgm_calc_disparity(const float* left, int lw, int lh, ptrdiff_t lpitch,
                              const float* right, int rw, int rh, ptrdiff_t rpitch,
                              int search_x, int search_y, int kernel_size, int p1, int p2,
                              vwb200_dispi* out, ptrdiff_t opitch, int* out_w, int* out_h, int on_device, void* stream);
/* ... followed by SemiGlobalMatcher::create_disparity_view_subpixel (SGM.cc:1497-1614) on the integer result:
 * subpixel_mode = SgmSubpixelMode.  out (may be NULL) gets the integer disparity, out_sub the float
 * {dx, dy, valid} pixels (sub_pitch in pixels).  Floats agree with the reference's double arithmetic within 1e-5. */
int vwb200_sgm_calc_disparity_subpixel(const float* left, int lw, int lh, ptrdiff_t lpitch,
                                       const float* right, int rw, int rh, ptrdiff_t rpitch,
                                       int search_x, int search_y, int kernel_size, int p1, int p2, int subpixel_mode,
                                       vwb200_dispi* out, ptrdiff_t opitch, float* out_sub, ptrdiff_t sub_pitch,
                                       int* out_w, int* out_h, int on_device, void* stream);

/* the full form.  vwb200_sgm_params mirrors the SemiGlobalMatcher constructor (SGM.h:104-121). */
typedef struct {
  int32_t search_x, search_y;            /* max disparity, inclusive (min is 0) */
  int32_t kernel_size;                   /* 3, 5, 7 or 9 */
  int32_t cost_type;                     /* VWB200_CENSUS_TRANSFORM or VWB200_TERNARY_CENSUS_TRANSFORM; anything else:
                                            VWB200_ENOIMPL like SGM.cc:1888-1892 */
  int32_t ternary_threshold;             /* ternary_census_threshold (default 5) */
  int32_t p1, p2;                        /* <= 0: the reference's defaults for the cost type and kernel */
  int32_t use_mgm;
  int32_t subpixel_mode;
  int32_t search_buffer_x, search_buffer_y;   /* sgm_search_buffer, applied around the doubled previous disparity */
  int32_t conserve_level;                /* -1: the reference's retry loop (SGM.cc:476-497): levels 0..3 until the buffers
                                            fit memory_limit_mb; 0..3: exactly that level of constrain_disp_bound_image */
  double  memory_limit_mb;               /* <= 0: 6000 (CorrelationView.h:65) */
  int32_t assumed_threads;               /* vw_settings().default_num_threads() of the size estimate (:715-716); <= 0: 4 */
  int32_t reserved;
} vwb200_sgm_params;
/* lmask (out_w x out_h, the size of the output, :250-256) / rmask (at least output + search, :262-268) / prev (the
 * half-resolution integer disparity of the previous pyramid level) may each be NULL.  bounds != NULL: use these
 * out_w * out_h boxes {min_x, min_y, max_x, max_y} (inclusive; max < min = no search area) instead of deriving them.
 * bounds_out (may be NULL) receives the boxes that were used. */
int vwb200_sgm_calc_disparity_ex(const vwb200_sgm_params* params,
                                 const float* left, int lw, int lh, ptrdiff_t lpitch,
                                 const float* right, int rw, int rh, ptrdiff_t rpitch,
                                 const uint8_t* lmask, ptrdiff_t lmpitch,
                                 const uint8_t* rmask, int rmw, int rmh, ptrdiff_t rmpitch,
                                 const vwb200_dispi* prev, int pw, int ph, ptrdiff_t ppitch,
                                 const int32_t* bounds,
                                 vwb200_dispi* out, ptrdiff_t opitch, float* out_sub, ptrdiff_t sub_pitch,
                                 int32_t* bounds_out, int* out_w, int* out_h, int on_device, void* stream);
/* only SemiGlobalMatcher::populate_disp_bound_image + constrain_disp_bound_image (SGM.cc:241-668) for an
 * ow x oh output: bounds receives ow * oh boxes */
int vwb200_sgm_disp_bounds(const vwb200_sgm_params* params, const vwb200_dispi* prev, int pw, int ph, ptrdiff_t ppitch,
                           const uint8_t* lmask, ptrdiff_t lmpitch, const uint8_t* rmask, int rmw, int rmh, ptrdiff_t rmpitch,
                           int ow, int oh, int32_t* bounds, int on_device, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The lazy view: vw::stereo::PyramidCorrelationView (src/vw/Stereo/CorrelationView.h:35-193,
 * CorrelationView.cc:273-886) behind a handle.  vwb200_corr_params mirrors the constructor
 * arguments (CorrelationView.h:48-69) that the block-matching algorithm uses.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t search_x0, search_y0, search_x1, search_y1;   /* BBox2i search_region */
  int32_t kernel_x, kernel_y;                           /* Vector2i kernel_size (odd) */
  int32_t cost_type;                                    /* CostFunctionType */
  int32_t prefilter_mode; float prefilter_width;
  float   consistency_threshold;                        /* < 0: no L/R check */
  int32_t min_consistency_level;
  int32_t filter_half_kernel;
  int32_t max_pyramid_levels;
  int32_t collar_size;
  int32_t corr_timeout; double seconds_per_op;          /* accepted; timeouts never trigger on the GPU */
  int32_t algorithm;                                    /* CorrelationAlgorithm: BM, SGM, MGM, FINAL_MGM */
  int32_t blob_filter_area;                             /* > 0: disparity_blob_filter (CorrelationView.cc:242-271) */
  /* the remaining constructor arguments (CorrelationView.h:61-69) */
  int32_t sgm_subpixel_mode;                            /* SgmSubpixelMode, default SUBPIXEL_LC_BLEND = 5 */
  int32_t sgm_search_buffer_x, sgm_search_buffer_y;     /* default (2, 2) */
  int32_t region_ul_x, region_ul_y;                     /* image position of lr_disp_diff's pixel (0, 0) */
  int32_t write_debug_images;                           /* accepted, ignored: the engine writes no files */
  int32_t sgm_threads;                                  /* vw_settings().default_num_threads() of SGM's memory estimate; <= 0: 4 */
  double  memory_limit_mb;                              /* <= 0: 6000 */
} vwb200_corr_params;

typedef struct vwb200_corr vwb200_corr;

int  vwb200_corr_create(const vwb200_corr_params* p, vwb200_corr** out);
/* on_device == 0: host rasters, copied to HBM once.  on_device == 1: device rasters, referenced in place.
 * on_device == VWB200_INPUTS_STREAMED: host rasters that STAY on the host -- every rasterize() uploads just its tile's
 * region of interest (left box + kernel padding, right box + search window; CorrelationView.cc:89-97), so rasters larger
 * than HBM work and nothing is resident between calls (the tile feeder; caller pattern Image/ImageIO.h:150-314).
 * Referenced rasters must outlive the handle.  Masks are uint8, nonzero = valid, same size as their image. */
#define VWB200_INPUTS_STREAMED 2
int  vwb200_corr_set_inputs(vwb200_corr* h,
                            const float* left,  int lcols, int lrows, ptrdiff_t lpitch,
                            const float* right, int rcols, int rrows, ptrdiff_t rpitch,
                            const uint8_t* lmask, ptrdiff_t lmpitch,
                            const uint8_t* rmask, ptrdiff_t rmpitch, int on_device);
/* the optional lr_disp_diff output (CorrelationView.h:67-68, .cc:276-283,848-857): a caller-owned cols x rows image of
 * PixelMask<float> = {value, valid} float pairs (row pitch in pixels) whose pixel (0, 0) sits at params.region_ul.
 * rasterize() writes max(|dx_lr + dx_rl|, |dy_lr + dy_rl|) where the L/R check passes (level 0) and invalidates where the
 * final disparity is invalid; other pixels keep their content.  A processed box outside the image -> VWB200_EARG.
 * diff == NULL switches the output off. */
int  vwb200_corr_set_lr_disp_diff(vwb200_corr* h, float* diff, int cols, int rows, ptrdiff_t pitch, int on_device);
int  vwb200_corr_cols(const vwb200_corr* h);
int  vwb200_corr_rows(const vwb200_corr* h);
/* rasterize(dest, bbox): dest receives (x1-x0) x (y1-y0) float disparity pixels (3 floats each),
 * row pitch dest_pitch in PIXELS.  Collar handling as in CorrelationView.h:123-133. */
int  vwb200_corr_rasterize(vwb200_corr* h, int x0, int y0, int x1, int y1,
                           float* dest, ptrdiff_t dest_pitch, int dest_on_device, void* stream);
/* prerasterize(bbox) (CorrelationView.cc:273-886): like rasterize() but processes exactly bbox, without the collar */
int  vwb200_corr_prerasterize(vwb200_corr* h, int x0, int y0, int x1, int y1,
                              float* dest, ptrdiff_t dest_pitch, int dest_on_device, void* stream);
/* levels prerasterize() would use for a bbox of this size (CorrelationView.cc:301-310) */
int  vwb200_corr_num_levels(const vwb200_corr* h, int bw, int bh);
void vwb200_corr_destroy(vwb200_corr* h);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU sharding (SURVEY.md section 8e; the reference has no distributed code): the unit of the path is the output
 * tile (tools/correlate.cc:266, Image/ImageIO.h:289-311), tiles are independent, so a raster shards into contiguous
 * output-row bands, one rank per GPU, with no reduction.  When the INPUT rasters are row-sharded the same way, rank r
 * needs from rank r + 1 the rows its last kernel windows and search rows reach into (ky - 1 rows of the left raster,
 * ky - 1 + sy - 1 of the right one): vwb200_shard_exchange_halos moves them with ncclSend / ncclRecv in one NCCL group.
 * NCCL is bound at run time (libnccl.so.2); without it vwb200_shard_create(world > 1) returns VWB200_ENOIMPL.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t rank, world;
  int32_t y0, y1;                 /* output rows [y0, y1) of this rank */
  int32_t left_rows, right_rows;  /* rows of the left / right raster this rank's launch reads */
  int32_t own_left, own_right;    /* rows resident on this rank before the exchange */
  int32_t recv_left, recv_right;  /* halo rows received from rank + 1 */
  int32_t send_left, send_right;  /* rows sent to rank - 1 (its halo) */
} vwb200_band_plan;
typedef struct vwb200_shard vwb200_shard;
/* band arithmetic for out_rows output rows (left_total_rows / right_total_rows <= 0: out_rows + ky - 1 [+ sy - 1]) */
int  vwb200_shard_plan(int rank, int world, int out_rows, int ky, int sy, int left_total_rows, int right_total_rows,
                       vwb200_band_plan* plan);
/* rank 0 calls this and hands the 128 bytes to every rank (MPI_Bcast, a file, torch.distributed, ...) */
int  vwb200_shard_unique_id(void* id128);
/* collective: every rank calls it with the same id on its own (current) device */
int  vwb200_shard_create(const void* id128, int rank, int world, vwb200_shard** out);
/* asynchronous on `stream` (NULL = the legacy default stream) */
int  vwb200_shard_exchange_halos(vwb200_shard* s, const vwb200_band_plan* plan, float* left_band, int lcols, ptrdiff_t lpitch,
                                 float* right_band, int rcols, ptrdiff_t rpitch, void* stream);
void vwb200_shard_destroy(vwb200_shard* s);

/* Scratch memory is stream-ordered and stays cached in the device's default memory pool between calls (returning it at
 * every synchronisation costs ~100 ms per 8K x 8K call).  vwb200_trim() hands the cached memory back to the driver. */
int vwb200_trim(void);

/* total number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
long long vwb200_kernel_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* VWB200_H */
