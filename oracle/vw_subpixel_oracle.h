/*
 * vw_subpixel_oracle.h -- CPU restatement of Vision Workbench's iterative sub-pixel refinement:
 * PyramidSubpixelView (Stereo/SubpixelView.cc:33-224) and its three per-level functions
 * subpixel_optimized_LK_2d / subpixel_optimized_affine_2d / subpixel_optimized_affine_2d_EM
 * (Stereo/Correlate.cc:500-844, 848-1199, 1203-1391).
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT CODE (see vw_oracle.h).  Built into its own library,
 * libvwsubpixel.so, together with vw_oracle.c (for the prefilters).
 *
 * Disparity pixels are PixelMask<Vector2f> as {dx, dy, valid} float triples (valid 0 / 1).
 *
 * Two operations are substituted because the reference does not pin them; the CUDA kernels use
 * the same operation sequence (DESIGN.md section K6):
 *   exp(float)   -> vwso_expf: float exp evaluated in double with IEEE basic operations only
 *   posv('L')    -> unblocked Cholesky in LAPACK spotf2 column order (scaling by the reciprocal of the
 *                   pivot) and two triangular solves, all in float; a pivot <= 0 or NaN leaves the
 *                   right-hand side unsolved (info > 0), as LAPACK does.
 */
#ifndef VW_SUBPIXEL_ORACLE_H
#define VW_SUBPIXEL_ORACLE_H

#ifdef __cplusplus
extern "C" {
#endif

/* PyramidSubpixelView_Algorithm (Stereo/SubpixelView.h:35-40) */
enum { VWSO_LUCAS_KANADE = 0, VWSO_FAST_AFFINE = 1, VWSO_BAYES_EM = 2, VWSO_PHASE = 3 };
enum { VWSO_OK = 0, VWSO_EARG = -1, VWSO_ENOIMPL = -2, VWSO_ENOMEM = -3 };

float vwso_expf(float x);
void vwso_expf_array(const float* x, int n, float* out);
/* compute_spatial_weight_image (Correlate.cc:36-55), out: kh x kw */
void vwso_spatial_weight(int kw, int kh, float two_sigma_sqr, float* out);
/* the posv substitution: A n x n row-major symmetric (overwritten), b solved in place unless info > 0 */
int vwso_posv(int n, float* A, float* b);
/* derivative_filter(img, 1, 0) / (0, 1) with ConstantEdgeExtension (Image/Filter.h:275-307) */
void vwso_derivative(const float* img, int w, int h, int dx, float* out);
/* BilinearInterpolation over ZeroEdgeExtension (Image/Interpolation.h:76-110) */
float vwso_bilinear(const float* img, int w, int h, float x, float y);
/* disparity_subsample (DisparityMap.h:1253-1314): out (1+(w-1)/2) x (1+(h-1)/2) */
void vwso_disparity_subsample(const float* in, int w, int h, float* out);
/* crop(disparity_upsample(edge_extend(in)), BBox2i(0,0,ow,oh)) (DisparityMap.h:1316-1358) */
void vwso_disparity_upsample(const float* in, int w, int h, float* out, int ow, int oh);
/* one level function, in place on disp (w x h, same size as left); right is rw x rh */
int vwso_subpixel_level(int algorithm, float* disp, const float* left, int w, int h, const float* right, int rw, int rh,
                        int kx, int ky, int rx0, int ry0, int rx1, int ry1, int do_h, int do_v);
/* PyramidSubpixelView::prerasterize + rasterize over bbox [x0,x1) x [y0,y1); out is bbox-sized */
int vwso_pyramid_subpixel(const float* disp, int cols, int rows, const float* left, int lpitch,
                          const float* right, int rcols, int rrows, int rpitch, int kx, int ky,
                          int prefilter_mode, float prefilter_width, int x0, int y0, int x1, int y1,
                          int max_pyramid_levels, int algorithm, float* out);

#ifdef __cplusplus
}
#endif
#endif
