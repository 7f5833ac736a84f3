/*
 * vw_corr_eval_oracle.h -- CPU restatement of Vision Workbench's CorrEval (Stereo/CorrEval.h:56-129,
 * CorrEval.cc:15-317): the NCC, stddev, parabola_curvature or cramer_rao quality of a float disparity.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT CODE (see vw_oracle.h).  Built into its own library, libvwcorreval.so.
 *
 * Images are PixelMask<float> as interleaved {value, valid} float pairs; the disparity is PixelMask<Vector2f>
 * as {dx, dy, valid} triples of the left image's size; pitches are in pixels.  A valid channel != 0 is valid.
 * dest receives (x1-x0) x (y1-y0) pairs.  Besides the reference's own argument checks, a sample_rate < 1, a
 * prefilter_kernel_width whose padding ceil(w) + 5 is NaN, negative or above 2^20, and a sampled valid disparity in
 * the bbox that is NaN, infinite or of magnitude >= 2^24 are argument errors (VWCE_EARG).
 */
#ifndef VW_CORR_EVAL_ORACLE_H
#define VW_CORR_EVAL_ORACLE_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { VWCE_NCC = 0, VWCE_STDDEV = 1, VWCE_PARABOLA_CURVATURE = 2, VWCE_CRAMER_RAO = 3 };
enum { VWCE_OK = 0, VWCE_EARG = -1, VWCE_ENOMEM = -3 };

/* CorrEval::prerasterize(bbox) over [x0,x1) x [y0,y1) */
int vwce_corr_eval(const float* left, int lw, int lh, ptrdiff_t lpitch,
                   const float* right, int rw, int rh, ptrdiff_t rpitch,
                   const float* disparity, ptrdiff_t dpitch, int kx, int ky, int metric, int sample_rate,
                   int round_to_int, float prefilter_kernel_width, int x0, int y0, int x1, int y1,
                   float* dest, ptrdiff_t dest_pitch);
/* the right crop's origin right_box.min() that prerasterize(bbox) uses (CorrEval.cc:189-214); returns 1, or 0 when no
 * sampled pixel of the bbox is valid (the box is empty and nothing is evaluated), or VWCE_EARG */
int vwce_right_origin(int lw, int lh, const float* disparity, ptrdiff_t dpitch, int kx, int ky, int metric,
                      int sample_rate, int round_to_int, float prefilter_kernel_width, int x0, int y0, int x1, int y1,
                      int* ox, int* oy);

#ifdef __cplusplus
}
#endif
#endif
