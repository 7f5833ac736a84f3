/*
 * vw_subpixel_oracle.c -- loop-for-loop restatement of PyramidSubpixelView and the three
 * per-level sub-pixel refinement functions.  See vw_subpixel_oracle.h.  References are to the
 * reference's src/vw/.
 */
#define _GNU_SOURCE
#include "vw_subpixel_oracle.h"
#include "vw_oracle.h"
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <limits.h>

static int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
static int imax(int a, int b) { return a > b ? a : b; }
static int imin(int a, int b) { return a < b ? a : b; }

/* ------------------------------------------------------------------ exp substitution */
/* exp(x) for float x, evaluated in double with +, -, *, / only and rounded once to float:
 * k = round(x / ln 2) by the 1.5 * 2^52 shift, r = x - k ln2 (Cody-Waite split), degree-13 Taylor
 * polynomial of e^r in Horner form, scaled by the exact power of two 2^k. */
static double pow2i(int k) {                       /* 2^k, -1022 <= k <= 1023 */
  union { double d; uint64_t u; } v;
  v.u = (uint64_t)(k + 1023) << 52;
  return v.d;
}
float vwso_expf(float xf) {
  const double x = (double)xf;
  if (x != x) return xf;
  if (x < -104.0) return 0.0f;
  if (x > 89.0) return (float)INFINITY;
  const double shift = 6755399441055744.0;         /* 1.5 * 2^52 */
  const double inv_ln2 = 1.4426950408889634;
  const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10;
  double kd = x * inv_ln2 + shift;
  kd = kd - shift;
  const double r = (x - kd * ln2_hi) - kd * ln2_lo;
  static const double c[14] = { 1.0, 1.0, 1.0 / 2, 1.0 / 6, 1.0 / 24, 1.0 / 120, 1.0 / 720, 1.0 / 5040, 1.0 / 40320,
                                1.0 / 362880, 1.0 / 3628800, 1.0 / 39916800, 1.0 / 479001600, 1.0 / 6227020800.0 };
  double p = c[13];
  for (int i = 12; i >= 0; --i) p = p * r + c[i];
  return (float)(p * pow2i((int)kd));
}
void vwso_expf_array(const float* x, int n, float* out) { for (int i = 0; i < n; ++i) out[i] = vwso_expf(x[i]); }

/* ------------------------------------------------------------------ helpers */
void vwso_spatial_weight(int kw, int kh, float two_sigma_sqr, float* out) {       /* Correlate.cc:36-55 */
  const int cx = kw / 2, cy = kh / 2;
  float sum = 0.0f;
  for (int j = 0; j < kh; ++j)
    for (int i = 0; i < kw; ++i) {
      const int r2 = (i - cx) * (i - cx) + (j - cy) * (j - cy);
      out[j * kw + i] = vwso_expf((float)(-1 * r2) / two_sigma_sqr);
      sum += out[j * kw + i];
    }
  for (int k = 0; k < kw * kh; ++k) out[k] = out[k] / sum;
}

/* the posv('L') substitution (LAPACK spotf2 + spotrs order, unblocked); A row-major symmetric */
int vwso_posv(int n, float* A, float* b) {
  for (int j = 0; j < n; ++j) {
    float dot = 0.0f;
    for (int k = 0; k < j; ++k) dot = dot + A[j * n + k] * A[j * n + k];
    float ajj = A[j * n + j] - dot;
    if (ajj <= 0.0f || ajj != ajj) { A[j * n + j] = ajj; return j + 1; }
    ajj = sqrtf(ajj);
    A[j * n + j] = ajj;
    for (int k = 0; k < j; ++k) {
      const float t = -A[j * n + k];
      for (int i = j + 1; i < n; ++i) A[i * n + j] = A[i * n + j] + t * A[i * n + k];
    }
    const float rcp = 1.0f / ajj;
    for (int i = j + 1; i < n; ++i) A[i * n + j] = A[i * n + j] * rcp;
  }
  for (int i = 0; i < n; ++i) {                   /* L y = b */
    float t = b[i];
    for (int k = 0; k < i; ++k) t = t - A[i * n + k] * b[k];
    b[i] = t / A[i * n + i];
  }
  for (int i = n - 1; i >= 0; --i) {              /* L^T x = y */
    float t = b[i];
    for (int k = i + 1; k < n; ++k) t = t - A[k * n + i] * b[k];
    b[i] = t / A[i * n + i];
  }
  return 0;
}

/* derivative_filter: kernel {0.5, 0, -0.5} applied reversed as a correlation, result = 0 + sum in tap
 * order, ConstantEdgeExtension on this image (Filter.h:275-307, Filter.tcc:107-111, Convolution.h:53-66) */
void vwso_derivative(const float* img, int w, int h, int dx, float* out) {
  const float rk[3] = { -0.5f, 0.0f, 0.5f };
  for (int y = 0; y < h; ++y)
    for (int x = 0; x < w; ++x) {
      float r = 0.0f;
      for (int k = 0; k < 3; ++k) {
        const int sx = dx ? clampi(x - 1 + k, 0, w - 1) : x, sy = dx ? y : clampi(y - 1 + k, 0, h - 1);
        r += rk[k] * img[(size_t)sy * w + sx];
      }
      out[(size_t)y * w + x] = r;
    }
}

/* math::impl::_floor (Math/Functions.h:74-84) with the x86 conversion of out-of-range values (INT_MIN) */
static int32_t cvt_i32(double v) { return (v >= -2147483648.0 && v < 2147483648.0) ? (int32_t)v : INT32_MIN; }
static int32_t floor_i32(double v) {
  const int32_t iv = cvt_i32(v);
  if (v < 0) return ((double)iv == v) ? iv : (int32_t)((uint32_t)iv - 1u);
  return iv;
}
static float at_zero(const float* img, int w, int h, int64_t x, int64_t y) {
  return (x < 0 || y < 0 || x >= w || y >= h) ? 0.0f : img[(size_t)y * w + (size_t)x];
}
float vwso_bilinear(const float* img, int w, int h, float xf, float yf) {          /* Interpolation.h:76-110 */
  const double i = (double)xf, j = (double)yf;
  const int32_t x = floor_i32(i), y = floor_i32(j);
  if ((double)x == i && (double)y == j) return at_zero(img, w, h, x, y);
  const float nx = xf - (float)x, ny = yf - (float)y, n1x = 1.0f - nx, n1y = 1.0f - ny;
  float r = at_zero(img, w, h, x, y) * n1x;
  r += at_zero(img, w, h, (int64_t)x + 1, y) * nx;
  r *= n1y;
  float row = at_zero(img, w, h, x, (int64_t)y + 1) * n1x;
  row += at_zero(img, w, h, (int64_t)x + 1, (int64_t)y + 1) * nx;
  r += row * ny;
  return r;
}

/* DisparitySubsampleView::operator() over ConstantEdgeExtension; double accumulation, the last six
 * neighbours are multiplied in float before the promotion (DisparityMap.h:1268-1304) */
void vwso_disparity_subsample(const float* in, int w, int h, float* out) {
  const int ow = 1 + (w - 1) / 2, oh = 1 + (h - 1) / 2;
  static const int nb[9][3] = { { 0, 0, 10 }, { 1, 0, 5 }, { 0, 1, 5 }, { -1, 0, 5 }, { 0, -1, 5 },
                                { 1, 1, 2 }, { -1, -1, 2 }, { -1, 1, 2 }, { 1, -1, 2 } };
  for (int j = 0; j < oh; ++j)
    for (int i = 0; i < ow; ++i) {
      double bx = 0.0, by = 0.0, cnt = 0.0;
      for (int k = 0; k < 9; ++k) {
        const float* p = in + ((size_t)clampi(2 * j + nb[k][1], 0, h - 1) * w + clampi(2 * i + nb[k][0], 0, w - 1)) * 3;
        if (p[2] == 0.0f) continue;
        cnt += nb[k][2];
        if (k < 3) { bx += (double)nb[k][2] * (double)p[0]; by += (double)nb[k][2] * (double)p[1]; }
        else { bx += (double)((float)nb[k][2] * p[0]); by += (double)((float)nb[k][2] * p[1]); }
      }
      float* o = out + ((size_t)j * ow + i) * 3;
      if (cnt > 0) { o[0] = (float)(bx / (cnt * 2)); o[1] = (float)(by / (cnt * 2)); o[2] = 1.0f; }
      else { o[0] = 0.0f; o[1] = 0.0f; o[2] = 0.0f; }
    }
}

void vwso_disparity_upsample(const float* in, int w, int h, float* out, int ow, int oh) {   /* DisparityMap.h:1331-1334 */
  for (int j = 0; j < oh; ++j)
    for (int i = 0; i < ow; ++i) {
      const float* p = in + ((size_t)clampi(j >> 1, 0, h - 1) * w + clampi(i >> 1, 0, w - 1)) * 3;
      float* o = out + ((size_t)j * ow + i) * 3;
      o[0] = p[0] * 2; o[1] = p[1] * 2; o[2] = p[2];
    }
}

/* norm_2 of a float vector: float squares summed in double, cast to float, sqrt in double (Math/Vector.h:1593-1604) */
static double norm2v(const float* v, int n) {
  double r = 0.0;
  for (int i = 0; i < n; ++i) r += (double)(v[i] * v[i]);
  return sqrt((double)(float)r);
}
static double norm2xy(float a, float b) { const float v[2] = { a, b }; return norm2v(v, 2); }

/* the 6x6 normal matrix of the affine models from its 18 accumulated entries (rhsData indices of
 * Correlate.cc:624-645 plus the symmetric fill of :694-705) */
static void fill_rhs6(const float* R, float* M) {
  static const int idx[36] = { 0, 1, 2, 3, 4, 5,   1, 7, 8, 4, 10, 11,   2, 8, 14, 5, 11, 17,
                               3, 4, 5, 21, 22, 23, 4, 10, 11, 22, 28, 29, 5, 11, 17, 23, 29, 35 };
  for (int k = 0; k < 36; ++k) M[k] = R[idx[k]];
}
static void acc_rhs6(float* R, int ii, int jj, float Ixs, float Ixy, float Iys) {
  const float m0 = (float)(ii * ii), m1 = (float)(ii * jj), m2 = (float)(jj * jj);
  R[0] += m0 * Ixs; R[1] += m1 * Ixs; R[2] += ii * Ixs; R[7] += m2 * Ixs; R[8] += jj * Ixs; R[14] += Ixs;
  R[3] += m0 * Ixy; R[4] += m1 * Ixy; R[5] += ii * Ixy; R[10] += m2 * Ixy; R[11] += jj * Ixy; R[17] += Ixy;
  R[21] += m0 * Iys; R[22] += m1 * Iys; R[23] += ii * Iys; R[28] += m2 * Iys; R[29] += jj * Iys; R[35] += Iys;
}

/* ------------------------------------------------------------------ the level functions */
int vwso_subpixel_level(int alg, float* disp, const float* left, int w, int h, const float* right, int rw, int rh,
                        int kx, int ky, int rx0, int ry0, int rx1, int ry1, int do_h, int do_v) {
  if (alg < 0 || alg > VWSO_BAYES_EM) return VWSO_ENOIMPL;
  if (!do_h && !do_v) return VWSO_OK;
  const float two_sigma_sqr = (float)(2.0 * pow((double)(float)kx / 5.0, 2.0));
  const float max_t = (float)(kx / 2);
  const int khh = ky / 2, khw = kx / 2, kp = kx * ky, thr = kp / 2;
  float* xd = (float*)malloc((size_t)w * h * sizeof(float));
  float* yd = (float*)malloc((size_t)w * h * sizeof(float));
  float* tmpl = (float*)malloc((size_t)kp * sizeof(float));
  if (!xd || !yd || !tmpl) { free(xd); free(yd); free(tmpl); return VWSO_ENOMEM; }
  vwso_derivative(left, w, h, 1, xd);
  vwso_derivative(left, w, h, 0, yd);
  vwso_spatial_weight(kx, ky, two_sigma_sqr, tmpl);

  for (int y = imax(ry0 - 1, khh); y < imin(h - khh, ry1 + 1); ++y)
    for (int x = imax(rx0 - 1, khw); x < imin(w - khw, rx1 + 1); ++x) {
      float* dp = disp + ((size_t)y * w + x) * 3;
      if (dp[2] == 0.0f) continue;
      /* adjust_weight_image (Correlate.cc:1393-1435) reads the current validity of the window; the level
       * loops only ever read w(0,0) (w_ptr is not advanced, :596-599, :947-950, :1306-1309) */
      float sum = 0.0f, w00 = 0.0f;
      int good = 0;
      for (int j = 0; j < ky; ++j)
        for (int i = 0; i < kx; ++i) {
          const int valid = disp[((size_t)(y - khh + j) * w + (x - khw + i)) * 3 + 2] != 0.0f;
          const float wv = valid ? tmpl[j * kx + i] : 0.0f;
          if (valid) { sum += wv; ++good; }
          if (i == 0 && j == 0) w00 = wv;
        }
      w00 = w00 / sum;
      if (good < thr) { dp[2] = 0.0f; continue; }
      const float x_base0 = (float)x + dp[0], y_base0 = (float)y + dp[1];
#define WIN(img, ii, jj) (img)[(size_t)(y + (jj)) * w + (x + (ii))]

      if (alg == VWSO_LUCAS_KANADE) {                                              /* Correlate.cc:1203-1391 */
        float d[2] = { 0.0f, 0.0f };
        for (int iter = 0; iter < 10; ++iter) {
          if (norm2v(d, 2) > max_t) break;
          const float x_base = x_base0, y_base = y_base0;
          float r0 = 0, r1 = 0, r3 = 0, lhs[2] = { 0, 0 };
          for (int jj = -khh; jj <= khh; ++jj) {
            const float xx_partial = x_base + d[0];
            const float yy = y_base + jj + d[1];
            for (int ii = -khw; ii <= khw; ++ii) {
              const float xx = ii + xx_partial;
              const float ip = vwso_bilinear(right, rw, rh, xx, yy);
              const float Ie = ip - WIN(left, ii, jj);
              const float weight = 1.0f * w00;
              const float Ix = WIN(xd, ii, jj), Iy = WIN(yd, ii, jj);
              const float Ixv = weight * Ix, Iyv = weight * Iy, Ixs = Ixv * Ix, Iys = Iyv * Iy, Ixy = Ixv * Iy;
              lhs[0] -= Ixv * Ie;
              lhs[1] -= Iyv * Ie;
              r0 += Ixs; r1 += Ixy; r3 += Iys;
            }
          }
          float M[4] = { r0, r1, r1, r3 };
          vwso_posv(2, M, lhs);
          d[0] += lhs[0]; d[1] += lhs[1];
          if (norm2v(lhs, 2) < 0.05) break;
        }
        if (norm2v(d, 2) > max_t || isnan(d[0]) || isnan(d[1])) dp[2] = 0.0f;
        else { dp[0] += d[0]; dp[1] += d[1]; }
        continue;
      }

      float d[6] = { 1.0f, 0.0f, 0.0f, 0.0f, 1.0f, 0.0f };
      if (alg == VWSO_FAST_AFFINE) {                                                /* Correlate.cc:848-1199 */
        for (int iter = 0; iter < 10; ++iter) {
          if (norm2xy(d[2], d[5]) > max_t) break;
          const float x_base = x_base0, y_base = y_base0;
          float R[36] = { 0 }, lhs[6] = { 0 };
          for (int jj = -khh; jj <= khh; ++jj) {
            const float xx_partial = x_base + d[1] * jj + d[2];
            const float yy_partial = y_base + d[4] * jj + d[5];
            for (int ii = -khw; ii <= khw; ++ii) {
              const float xx = d[0] * ii + xx_partial, yy = d[3] * ii + yy_partial;
              const float ip = vwso_bilinear(right, rw, rh, xx, yy);
              const float Ie = ip - WIN(left, ii, jj);
              const float weight = 1.0f * w00;
              const float Ix = WIN(xd, ii, jj), Iy = WIN(yd, ii, jj);
              const float Ixv = weight * Ix, Iyv = weight * Iy, Ixs = Ixv * Ix, Iys = Iyv * Iy, Ixy = Ixv * Iy;
              const float IxIe = Ixv * Ie, IyIe = Iyv * Ie;
              lhs[0] -= ii * IxIe; lhs[1] -= jj * IxIe; lhs[2] -= IxIe;
              lhs[3] -= ii * IyIe; lhs[4] -= jj * IyIe; lhs[5] -= IyIe;
              acc_rhs6(R, ii, jj, Ixs, Ixy, Iys);
            }
          }
          float M[36];
          fill_rhs6(R, M);
          vwso_posv(6, M, lhs);
          for (int k = 0; k < 6; ++k) d[k] += lhs[k];
          float wl[6];
          memcpy(wl, lhs, sizeof(wl));
          const int kqh = khh / 2, kqw = khw / 2;
          wl[0] *= kqw; wl[1] *= kqh; wl[3] *= kqw; wl[4] *= kqh;
          if (norm2v(wl, 6) < 0.05) break;
        }
      } else {                                                                       /* Correlate.cc:500-844 */
        float curr_sum = 0.0f, prev_sum = 0.0f;
        for (int iter = 0; iter < 10; ++iter) {
          if (norm2xy(d[2], d[5]) > max_t) break;
          const float x_base = x_base0, y_base = y_base0;
          float R[36], lhs[6], prev_lhs[6] = { 0 };
          float var2_plane = 1e-3f, mean_noise = 0.0f, var2_noise = 1e-2f, w_plane = 0.8f, w_noise = 0.2f;
          float in_curr = 0.0f, d_em[6];
          memcpy(d_em, d, sizeof(d_em));
          for (int em = 0; em < 2; ++em) {
            const float noise_norm = (float)(1.0 / sqrt(2 * M_PI * var2_noise));
            const float plane_norm = (float)(1.0 / sqrt(2 * M_PI * var2_plane));
            memset(lhs, 0, sizeof(lhs));
            memset(R, 0, sizeof(R));
            in_curr = 0.0f;
            float mean_noise_tmp = 0.0f, sum_gn = 0.0f, sum_gp = 0.0f;
            int skip = 0;
            for (int jj = -khh; jj <= khh; ++jj) {
              const float xx_partial = x_base + d[1] * jj + d[2];
              const float yy_partial = y_base + d[4] * jj + d[5];
              const float dx_partial = d_em[1] * jj + d_em[2];
              const float dy_partial = d_em[4] * jj + d_em[5];
              for (int ii = -khw; ii <= khw; ++ii) {
                const float xx = d[0] * ii + xx_partial, yy = d[3] * ii + yy_partial;
                const float delta_x = d_em[0] * ii + dx_partial, delta_y = d_em[3] * ii + dy_partial;
                const float ip = vwso_bilinear(right, rw, rh, xx, yy);
                const float Ie = ip - WIN(left, ii, jj);
                in_curr += Ie;
                const float Ix = WIN(xd, ii, jj), Iy = WIN(yd, ii, jj);
                const float tp = Ie - delta_x * Ix - delta_y * Iy;
                const float tn = ip - mean_noise;
                const float ppe = -1 * (tp * tp) / (2 * var2_plane);
                const float pp = (ppe < -75) ? 0.0f : plane_norm * vwso_expf(ppe);
                const float npe = -1 * (tn * tn) / (2 * var2_noise);
                const float np = (npe < -75) ? 0.0f : noise_norm * vwso_expf(npe);
                const float s = pp * w_plane + np * w_noise;
                const float gp = pp * w_plane / s, gn = np * w_noise / s;
                mean_noise_tmp += ip * gn;
                sum_gp += gp;
                sum_gn += gn;
                const float weight = gp * w00;
                if (weight < 1e-26) { skip++; continue; }
                const float Ixv = weight * Ix, Iyv = weight * Iy, Ixs = Ixv * Ix, Iys = Iyv * Iy, Ixy = Ixv * Iy;
                lhs[0] -= ii * Ixv * Ie; lhs[1] -= jj * Ixv * Ie; lhs[2] -= Ixv * Ie;
                lhs[3] -= ii * Iyv * Ie; lhs[4] -= jj * Iyv * Ie; lhs[5] -= Iyv * Ie;
                acc_rhs6(R, ii, jj, Ixs, Ixy, Iys);
              }
            }
            if (skip == kp) break;
            float M[36];
            fill_rhs6(R, M);
            vwso_posv(6, M, lhs);
            mean_noise = mean_noise_tmp / sum_gn;
            w_plane = sum_gp / (float)kp;
            w_noise = sum_gn / (float)kp;
            float diff[6];
            for (int k = 0; k < 6; ++k) diff[k] = prev_lhs[k] - lhs[k];
            const float conv_error = (float)norm2v(diff, 6);
            for (int k = 0; k < 6; ++k) d_em[k] = d[k] + lhs[k];
            if (in_curr < 0) in_curr = -in_curr;
            curr_sum = in_curr;
            memcpy(prev_lhs, lhs, sizeof(lhs));
            if (conv_error < 1E-3 && em > 0) break;
          }
          for (int k = 0; k < 6; ++k) d[k] += lhs[k];
          if (curr_sum < 0) curr_sum = -curr_sum;
          if (prev_sum < curr_sum && iter > 0) break;
          prev_sum = curr_sum;
        }
      }
      if (norm2xy(d[2], d[5]) > max_t || isnan(d[2]) || isnan(d[5])) dp[2] = 0.0f;
      else { dp[0] += d[2]; dp[1] += d[5]; }
#undef WIN
    }
  free(xd); free(yd); free(tmpl);
  return VWSO_OK;
}

/* ------------------------------------------------------------------ PyramidSubpixelView */
typedef struct { float* d; int w, h; } img_t;

static img_t crop_const(const float* src, int sw, int sh, int sp, int x0, int y0, int w, int h) {
  img_t o = { (float*)malloc((size_t)(w > 0 ? w : 1) * (h > 0 ? h : 1) * sizeof(float)), w, h };
  for (int y = 0; y < h; ++y)
    for (int x = 0; x < w; ++x) o.d[(size_t)y * w + x] = src[(size_t)clampi(y0 + y, 0, sh - 1) * sp + clampi(x0 + x, 0, sw - 1)];
  return o;
}
/* crop(prefilter.filter(img), region) over the lazily edge-extended view (PreFilter.h:45-70) */
static img_t filtered_region(const float* img, int w, int h, int pitch, int mode, float width, int x0, int y0, int x1, int y1) {
  img_t o = crop_const(img, w, h, pitch, x0, y0, x1 - x0, y1 - y0);
  if (mode == VWO_PREFILTER_NONE) return o;
  float k[512];
  const int n = vwo_gaussian_kernel((double)width, k, 512);
  if (mode == VWO_PREFILTER_MEANSUB) {
    if (n <= 0) { for (size_t i = 0; i < (size_t)o.w * o.h; ++i) o.d[i] = o.d[i] - o.d[i]; return o; }
    img_t e = crop_const(img, w, h, pitch, x0 - n, y0 - n, o.w + 2 * n, o.h + 2 * n);
    float* g = (float*)malloc((size_t)e.w * e.h * sizeof(float));
    vwo_separable_convolve(e.d, e.w, e.h, e.w, k, n, k, n, 0, g);
    for (int y = 0; y < o.h; ++y)
      for (int x = 0; x < o.w; ++x) o.d[(size_t)y * o.w + x] = o.d[(size_t)y * o.w + x] - g[(size_t)(y + n) * e.w + (x + n)];
    free(g); free(e.d);
    return o;
  }
  const int nx0 = clampi(x0 - 1, 0, w - 1), ny0 = clampi(y0 - 1, 0, h - 1), nx1 = clampi(x1, 0, w - 1) + 1, ny1 = clampi(y1, 0, h - 1) + 1;
  const int m = n > 0 ? n : 0, bx0 = nx0 - m, by0 = ny0 - m;
  img_t e = crop_const(img, w, h, pitch, bx0, by0, nx1 + m - bx0, ny1 + m - by0);
  float* g = (float*)malloc((size_t)e.w * e.h * sizeof(float));
  if (n > 0) vwo_separable_convolve(e.d, e.w, e.h, e.w, k, n, k, n, 0, g);
  else memcpy(g, e.d, (size_t)e.w * e.h * sizeof(float));
#define GAT(X, Y) g[(size_t)(clampi((Y), 0, h - 1) - by0) * e.w + (clampi((X), 0, w - 1) - bx0)]
  for (int y = 0; y < o.h; ++y)
    for (int x = 0; x < o.w; ++x) {
      const int gx = x0 + x, gy = y0 + y;
      float r = 0.0f;
      r = r + 1.0f * GAT(gx, gy - 1);
      r = r + 1.0f * GAT(gx - 1, gy);
      r = r + -4.0f * GAT(gx, gy);
      r = r + 1.0f * GAT(gx + 1, gy);
      r = r + 1.0f * GAT(gx, gy + 1);
      o.d[(size_t)y * o.w + x] = r;
    }
#undef GAT
  free(g); free(e.d);
  return o;
}

int vwso_pyramid_subpixel(const float* disp, int cols, int rows, const float* left, int lpitch,
                          const float* right, int rcols, int rrows, int rpitch, int kx, int ky,
                          int prefilter_mode, float prefilter_width, int x0, int y0, int x1, int y1,
                          int max_pyramid_levels, int algorithm, float* out) {
  if (algorithm < 0 || algorithm > VWSO_BAYES_EM) return VWSO_ENOIMPL;          /* SubpixelView.cc:158-159 */
  if (x1 <= x0 || y1 <= y0 || x0 < 0 || y0 < 0 || x1 > cols || y1 > rows || kx < 3 || ky < 3 || kx % 2 != 1 || ky % 2 != 1)
    return VWSO_EARG;
  const int levels = max_pyramid_levels < 0 ? 0 : max_pyramid_levels;
  const int bw = x1 - x0, bh = y1 - y0;
  /* get_disparity_range over every pixel of the crop, valid or not; BBox2f -> BBox2i truncates (DisparityMap.h:52-66).
   * A crop holding a NaN, an infinity or a magnitude >= 2^24 is rejected, as the engine does. */
  float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
  for (int y = y0; y < y1; ++y)
    for (int x = x0; x < x1; ++x) {
      const float* p = disp + ((size_t)y * cols + x) * 3;
      if (!(fabsf(p[0]) < 16777216.0f) || !(fabsf(p[1]) < 16777216.0f)) return VWSO_EARG;
      mnx = fminf(mnx, p[0]); mny = fminf(mny, p[1]); mxx = fmaxf(mxx, p[0]); mxy = fmaxf(mxy, p[1]);
    }
  const int sx0 = (int)mnx, sy0 = (int)mny, sx1 = (int)mxx, sy1 = (int)mxy;
  /* SubpixelView.cc:45-61 */
  const int rx0 = x0 + sx0 - kx, ry0 = y0 + sy0 - ky, rx1 = x1 + sx1 + kx, ry1 = y1 + sy1 + ky;
  const int pw = rx1 - rx0, ph = ry1 - ry0;
  const int lx0 = x0 - kx, ly0 = y0 - ky;
  img_t L = filtered_region(left, cols, rows, lpitch, prefilter_mode, prefilter_width, lx0, ly0, lx0 + pw, ly0 + ph);
  img_t R = filtered_region(right, rcols, rrows, rpitch, prefilter_mode, prefilter_width, rx0, ry0, rx1, ry1);
  /* crop(edge_extend(disp, Zero), left_crop_bbox) - search_range.min() */
  float* D = (float*)malloc((size_t)pw * ph * 3 * sizeof(float));
  for (int y = 0; y < ph; ++y)
    for (int x = 0; x < pw; ++x) {
      const int gx = lx0 + x, gy = ly0 + y;
      float* o = D + ((size_t)y * pw + x) * 3;
      if (gx < 0 || gy < 0 || gx >= cols || gy >= rows) { o[0] = 0.0f; o[1] = 0.0f; o[2] = 0.0f; }
      else memcpy(o, disp + ((size_t)gy * cols + gx) * 3, 3 * sizeof(float));
      o[0] = o[0] - (float)sx0; o[1] = o[1] - (float)sy0;
    }
  /* the pyramid (SubpixelView.cc:109-128) */
  img_t* lp = (img_t*)calloc((size_t)levels + 1, sizeof(img_t));
  img_t* rp = (img_t*)calloc((size_t)levels + 1, sizeof(img_t));
  int(*roi)[4] = (int(*)[4])calloc((size_t)levels + 1, sizeof(*roi));
  lp[0] = L; rp[0] = R;
  roi[0][0] = kx; roi[0][1] = ky; roi[0][2] = kx + bw; roi[0][3] = ky + bh;
  img_t dsub = { D, pw, ph };
  for (int i = 1; i <= levels; ++i) {
    lp[i].w = 1 + (lp[i - 1].w - 1) / 2; lp[i].h = 1 + (lp[i - 1].h - 1) / 2;
    lp[i].d = (float*)malloc((size_t)lp[i].w * lp[i].h * sizeof(float));
    vwo_subsample2_f32(lp[i - 1].d, lp[i - 1].w, lp[i - 1].h, lp[i - 1].w, lp[i].d);
    rp[i].w = 1 + (rp[i - 1].w - 1) / 2; rp[i].h = 1 + (rp[i - 1].h - 1) / 2;
    rp[i].d = (float*)malloc((size_t)rp[i].w * rp[i].h * sizeof(float));
    vwo_subsample2_f32(rp[i - 1].d, rp[i - 1].w, rp[i - 1].h, rp[i - 1].w, rp[i].d);
    img_t ns = { (float*)malloc((size_t)lp[i].w * lp[i].h * 3 * sizeof(float)), lp[i].w, lp[i].h };
    vwso_disparity_subsample(dsub.d, dsub.w, dsub.h, ns.d);
    if (dsub.d != D) free(dsub.d);
    dsub = ns;
    /* BBox2i / 2 leaves an empty box unchanged (Math/BBox.tcc:270-277) */
    const int empty = roi[i - 1][0] >= roi[i - 1][2] || roi[i - 1][1] >= roi[i - 1][3];
    for (int k = 0; k < 4; ++k) roi[i][k] = empty ? roi[i - 1][k] : roi[i - 1][k] / 2;
  }
  /* coarse to fine (SubpixelView.cc:133-188), then the native-resolution pass (:190-214) */
  for (int i = levels; i >= 0; --i) {
    vwso_subpixel_level(algorithm, dsub.d, lp[i].d, lp[i].w, lp[i].h, rp[i].d, rp[i].w, rp[i].h, kx, ky,
                        roi[i][0], roi[i][1], roi[i][2], roi[i][3], 1, 1);
    if (i == 0) break;
    img_t up = { (float*)malloc((size_t)lp[i - 1].w * lp[i - 1].h * 3 * sizeof(float)), lp[i - 1].w, lp[i - 1].h };
    vwso_disparity_upsample(dsub.d, dsub.w, dsub.h, up.d, up.w, up.h);
    if (dsub.d != D) free(dsub.d);
    dsub = up;
  }
  /* += search_range.min(), then the crop of :220-223 */
  for (int y = 0; y < bh; ++y)
    for (int x = 0; x < bw; ++x) {
      const float* p = dsub.d + ((size_t)(ky + y) * dsub.w + (kx + x)) * 3;
      float* o = out + ((size_t)y * bw + x) * 3;
      o[0] = p[0] + (float)sx0; o[1] = p[1] + (float)sy0; o[2] = p[2];
    }
  if (dsub.d != D) free(dsub.d);
  free(D);
  for (int i = 0; i <= levels; ++i) { free(lp[i].d); free(rp[i].d); }
  free(lp); free(rp); free(roi);
  return VWSO_OK;
}
