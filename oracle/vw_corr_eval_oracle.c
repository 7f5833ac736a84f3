/*
 * vw_corr_eval_oracle.c -- CorrEval (Stereo/CorrEval.cc:15-317) restated loop for loop in C.
 * TEST INFRASTRUCTURE, NOT PRODUCT CODE.  See vw_corr_eval_oracle.h.
 *
 * PixelMask<float> arithmetic (Image/PixelMask.h:359-490): the child is always computed, the validity of a result is
 * the AND of its operands' validities (a scalar operand is valid).  The crops are edge-extended with an invalid pixel
 * whose child is 0 (ValueEdgeExtension, CorrEval.cc:216-223); reads outside a crop see that pixel too (:26-33).
 */
#include "vw_corr_eval_oracle.h"

#include <limits.h>
#include <math.h>
#include <stdlib.h>

typedef struct { float v; int ok; } px;   /* PixelMask<float>: child, is_valid() */
typedef struct { int x0, y0, x1, y1; } box; /* BBox2i, half-open */

static px px_mul(px a, float s) { px r = {a.v * s, a.ok}; return r; }
static px px_add(px a, px b) { px r = {a.v + b.v, a.ok && b.ok}; return r; }

/* crop(edge_extend(img, nodata), b) read at (i, j) of the crop, itself extended with nodata beyond b */
typedef struct { const float* p; int w, h; ptrdiff_t pitch; box b; } crop;
static px crop_at(const crop* c, long long i, long long j) {
  const px nodata = {0.0f, 0};
  if (i < 0 || j < 0 || i >= (long long)c->b.x1 - c->b.x0 || j >= (long long)c->b.y1 - c->b.y0) return nodata;
  const long long x = c->b.x0 + i, y = c->b.y0 + j;
  if (x < 0 || y < 0 || x >= c->w || y >= c->h) return nodata;
  const float* q = c->p + ((size_t)y * c->pitch + (size_t)x) * 2;
  px r = {q[0], q[1] != 0.0f};
  return r;
}

/* BilinearInterpolationImpl (Image/Interpolation.h:76-110) over the crop, PixelMask<float>: real_type float */
static px bilinear(const crop* c, double i, double j) {
  const int x = (int)floor(i), y = (int)floor(j);
  if (x == i && y == j) return crop_at(c, x, y);
  const float normx = (float)i - (float)x, normy = (float)j - (float)y, norm1mx = 1 - normx, norm1my = 1 - normy;
  px result = px_mul(crop_at(c, x, y), norm1mx);
  result = px_add(result, px_mul(crop_at(c, (long long)x + 1, y), normx));
  result = px_mul(result, norm1my);
  px row = px_mul(crop_at(c, x, (long long)y + 1), norm1mx);
  row = px_add(row, px_mul(crop_at(c, (long long)x + 1, (long long)y + 1), normx));
  return px_add(result, px_mul(row, normy));
}

typedef struct {
  int kx, ky, round_to_int;
  box bbox, left_box, right_box;
  crop left, right;
} ctx;

/* calc_patches (CorrEval.cc:15-69); the patches are kx x ky, stored column-major like the (c, r) loops */
static int calc_patches(const ctx* k, float dx, float dy, int col, int row, px* left_patch, px* right_patch) {
  const int hx = k->kx / 2, hy = k->ky / 2;
  for (int c = 0; c < k->kx; c++) {
    for (int r = 0; r < k->ky; r++) {
      int lx = col + k->bbox.x0 + c - hx, ly = row + k->bbox.y0 + r - hy;
      double rx = (double)lx + (double)dx, ry = (double)ly + (double)dy;
      lx -= k->left_box.x0; ly -= k->left_box.y0;
      rx -= k->right_box.x0; ry -= k->right_box.y0;
      if (lx < 0 || ly < 0 || lx >= k->left_box.x1 - k->left_box.x0 || ly >= k->left_box.y1 - k->left_box.y0) return VWCE_EARG;
      left_patch[c * k->ky + r] = crop_at(&k->left, lx, ly);
      if (!k->round_to_int)
        right_patch[c * k->ky + r] = bilinear(&k->right, rx, ry);
      else
        right_patch[c * k->ky + r] = crop_at(&k->right, (int)rx, (int)ry);
    }
  }
  return VWCE_OK;
}

/* calc_ncc (:71-96): is_valid(bool) is always true, so every patch pixel enters the sums */
static double calc_ncc(const px* lp, const px* rp, int n) {
  double num = 0.0, den1 = 0.0, den2 = 0.0;
  for (int k = 0; k < n; k++) {
    double a = lp[k].v;
    double b = rp[k].v;
    num += a * b;
    den1 += a * a;
    den2 += b * b;
  }
  if (den1 > 0.0 && den2 > 0.0) return num / sqrt(den1 * den2);
  return -1.0;
}

/* calc_stddev (:98-137) */
static double calc_stddev(const px* p, int n) {
  int num = 0;
  double mean = 0.0;
  for (int k = 0; k < n; k++) {
    if (!p[k].ok) continue;
    num += 1;
    mean += p[k].v;
  }
  if (num == 0) return -1.0;
  mean /= num;
  double sum = 0.0;
  num = 0;
  for (int k = 0; k < n; k++) {
    if (!p[k].ok) continue;
    num += 1;
    sum += (p[k].v - mean) * (p[k].v - mean);
  }
  if (num == 0) return -1.0;
  return sqrt(sum / num);
}

static int check_args(int lw, int lh, int kx, int ky, int metric, int sample_rate, float pkw, int x0, int y0, int x1, int y1,
                      int* extra_padding) {
  if (lw <= 0 || lh <= 0) return VWCE_EARG;
  if (!(kx > 0 && kx % 2 == 1 && ky > 0 && ky % 2 == 1)) return VWCE_EARG;
  if (metric < VWCE_NCC || metric > VWCE_CRAMER_RAO) return VWCE_EARG;
  if (sample_rate < 1) return VWCE_EARG;
  if (x1 <= x0 || y1 <= y0 || x0 < 0 || y0 < 0 || x1 > lw || y1 > lh) return VWCE_EARG;
  const float pad = ceilf(pkw) + 5.0f;
  if (!(pad >= 0.0f && pad <= 1048576.0f)) return VWCE_EARG;
  *extra_padding = (int)pad;
  return VWCE_OK;
}

/* the rounded disparity of the bbox (:141-151) and right_box (:189-214).  Returns 1 if the box grew, 0 if it is empty. */
static int disp_and_right_box(int kx, int ky, int metric, int sample_rate, int round_to_int, int extra_padding, const float* disparity,
                              ptrdiff_t dpitch, box bbox, float* disp, box* right_box) {
  const int bw = bbox.x1 - bbox.x0, bh = bbox.y1 - bbox.y0;
  for (int col = 0; col < bw; col++)
    for (int row = 0; row < bh; row++) {
      const float* q = disparity + ((size_t)(bbox.y0 + row) * dpitch + (size_t)(bbox.x0 + col)) * 3;
      float* d = disp + ((size_t)row * bw + col) * 3;
      d[0] = q[0]; d[1] = q[1]; d[2] = q[2] != 0.0f;
      /* the engine's rule: sampled valid disparities must keep the double coordinates exact */
      if (d[2] != 0.0f && col % sample_rate == 0 && row % sample_rate == 0 &&
          !(fabsf(d[0]) < 16777216.0f && fabsf(d[1]) < 16777216.0f))
        return VWCE_EARG;
      if (round_to_int) { d[0] = roundf(d[0]); d[1] = roundf(d[1]); }
    }
  const int big = INT_MAX - 1;                        /* BBox() (Math/BBox.tcc:37-44) */
  box rb = {big, big, -big, -big};
  int grown = 0;
  for (int col = 0; col < bw; col++)
    for (int row = 0; row < bh; row++) {
      const float* d = disp + ((size_t)row * bw + col) * 3;
      if (d[2] == 0.0f) continue;
      if (col % sample_rate != 0 || row % sample_rate != 0) continue;
      const double lx = (double)bbox.x0 + (double)col, ly = (double)bbox.y0 + (double)row;
      const double rx = lx + (double)d[0], ry = ly + (double)d[1];
      const double pts[2][2] = {{floor(rx), floor(ry)}, {ceil(rx), ceil(ry)}};
      for (int p = 0; p < 2; p++) {                   /* BBox::grow (Math/BBox.tcc:80-96) */
        if (pts[p][0] > rb.x1) rb.x1 = (int)pts[p][0];
        if (pts[p][0] < rb.x0) rb.x0 = (int)pts[p][0];
        if (pts[p][1] > rb.y1) rb.y1 = (int)pts[p][1];
        if (pts[p][1] < rb.y0) rb.y0 = (int)pts[p][1];
      }
      grown = 1;
    }
  if (grown) {
    int e = 1 + 2 + extra_padding;                    /* BilinearInterpolation::pixel_buffer, 2, m_extra_padding */
    if (metric == VWCE_PARABOLA_CURVATURE || metric == VWCE_CRAMER_RAO) e += 1;
    rb.x0 -= kx / 2 + e; rb.y0 -= ky / 2 + e;
    rb.x1 += kx / 2 + e; rb.y1 += ky / 2 + e;
  }
  *right_box = rb;
  return grown;
}

int vwce_right_origin(int lw, int lh, const float* disparity, ptrdiff_t dpitch, int kx, int ky, int metric,
                      int sample_rate, int round_to_int, float prefilter_kernel_width, int x0, int y0, int x1, int y1,
                      int* ox, int* oy) {
  int pad;
  if (check_args(lw, lh, kx, ky, metric, sample_rate, prefilter_kernel_width, x0, y0, x1, y1, &pad)) return VWCE_EARG;
  const box bbox = {x0, y0, x1, y1};
  float* disp = (float*)malloc((size_t)(x1 - x0) * (y1 - y0) * 3 * sizeof(float));
  if (!disp) return VWCE_ENOMEM;
  box rb;
  const int rc = disp_and_right_box(kx, ky, metric, sample_rate, round_to_int, pad, disparity, dpitch, bbox, disp, &rb);
  free(disp);
  *ox = rb.x0; *oy = rb.y0;
  return rc;
}

int vwce_corr_eval(const float* left, int lw, int lh, ptrdiff_t lpitch,
                   const float* right, int rw, int rh, ptrdiff_t rpitch,
                   const float* disparity, ptrdiff_t dpitch, int kx, int ky, int metric, int sample_rate,
                   int round_to_int, float prefilter_kernel_width, int x0, int y0, int x1, int y1,
                   float* dest, ptrdiff_t dest_pitch) {
  int pad;
  if (check_args(lw, lh, kx, ky, metric, sample_rate, prefilter_kernel_width, x0, y0, x1, y1, &pad)) return VWCE_EARG;
  if (rw < 0 || rh < 0) return VWCE_EARG;
  const int bw = x1 - x0, bh = y1 - y0;
  ctx k;
  k.kx = kx; k.ky = ky; k.round_to_int = round_to_int;
  k.bbox = (box){x0, y0, x1, y1};
  float* disp = (float*)malloc((size_t)bw * bh * 3 * sizeof(float));
  if (!disp) return VWCE_ENOMEM;
  const int grown = disp_and_right_box(kx, ky, metric, sample_rate, round_to_int, pad, disparity, dpitch, k.bbox, disp, &k.right_box);
  if (grown < 0) { free(disp); return grown; }
  k.left_box = (box){x0 - (kx / 2 + pad), y0 - (ky / 2 + pad), x1 + kx / 2 + pad, y1 + ky / 2 + pad};
  k.left = (crop){left, lw, lh, lpitch, k.left_box};
  k.right = (crop){right, rw, rh, rpitch, k.right_box};
  const int n = kx * ky;
  const int curvature = metric == VWCE_PARABOLA_CURVATURE || metric == VWCE_CRAMER_RAO;
  int err = VWCE_OK;

#pragma omp parallel for schedule(dynamic, 1)
  for (int col = 0; col < bw; col++) {
    px* lp = (px*)malloc(sizeof(px) * (size_t)n * 4);
    if (!lp) { err = VWCE_ENOMEM; continue; }
    px *rp = lp + n, *nlp = lp + 2 * n, *nrp = lp + 3 * n;
    for (int row = 0; row < bh; row++) {
      float* o = dest + ((size_t)row * dest_pitch + col) * 2;
      o[0] = 0.0f; o[1] = 0.0f;                       /* the tile starts invalid (:239-241) */
      const float* d = disp + ((size_t)row * bw + col) * 3;
      if (d[2] == 0.0f) continue;
      if (col % sample_rate != 0 || row % sample_rate != 0) continue;
      if (calc_patches(&k, d[0], d[1], col, row, lp, rp)) { err = VWCE_EARG; continue; }
      if (metric == VWCE_NCC) {
        const double ncc = calc_ncc(lp, rp, n);
        if (ncc >= 0) { o[0] = (float)ncc; o[1] = 1.0f; }
      } else if (metric == VWCE_STDDEV) {
        const double ls = calc_stddev(lp, n), rs = calc_stddev(rp, n);
        if (ls >= 0.0 && rs >= 0.0) { o[0] = (float)((ls + rs) / 2.0); o[1] = 1.0f; }
      } else if (curvature) {
        const double C = calc_ncc(lp, rp, n);
        if (C >= 0) {
          const float shifts[4][2] = {{1, 0}, {-1, 0}, {0, 1}, {0, -1}};
          double nbr[4];
          int ok = 1;
          for (int s = 0; s < 4 && ok; s++) {
            const float sx = d[0] + shifts[s][0], sy = d[1] + shifts[s][1];   /* ds.child() += shifts[s], in float */
            if (calc_patches(&k, sx, sy, col, row, nlp, nrp)) { err = VWCE_EARG; ok = 0; break; }
            nbr[s] = calc_ncc(nlp, nrp, n);
            if (nbr[s] < 0) ok = 0;
          }
          if (ok) {
            const double kxx = 2.0 * C - nbr[0] - nbr[1];
            const double kyy = 2.0 * C - nbr[2] - nbr[3];
            if (kxx > 0 && kyy > 0) {
              double sigma = sqrt(1.0 / kxx + 1.0 / kyy);
              if (metric == VWCE_CRAMER_RAO) {
                double resid = 1.0 - C;
                if (resid < 0) resid = 0;
                sigma *= sqrt(resid);
              }
              o[0] = (float)sigma; o[1] = 1.0f;
            }
          }
        }
      }
    }
    free(lp);
  }
  free(disp);
  return err;
}
