// k6_subpixel.cu -- K6: iterative sub-pixel refinement, PyramidSubpixelView (Stereo/SubpixelView.cc:33-224) and its
// per-level functions subpixel_optimized_LK_2d / _affine_2d / _affine_2d_EM (Stereo/Correlate.cc:500-1391).
//
// One thread per pixel walks its window in the reference's jj / ii order with explicitly rounded fp32 operations (no FMA
// contraction) and fp64 where the reference uses double, so results are bit-identical to the sequential CPU order.
// The reference updates the disparity map in place while it scans it: a pixel's weight window sees the CURRENT validity
// of the pixels before it in raster order.  The level is therefore evaluated as a fixpoint: round 0 evaluates every pixel
// against the input validity; round r re-evaluates a pixel only if the validity of an earlier pixel of its window changed
// in round r-1.  Raster order is a DAG, so each round settles at least the first unsettled pixel, and the fixpoint is the
// sequential result.
#include "common.cuh"
#include <climits>

namespace vwb200 {

#define FA __fadd_rn
#define FS __fsub_rn
#define FM __fmul_rn
#define FD __fdiv_rn
#define DA __dadd_rn
#define DS __dsub_rn
#define DM __dmul_rn

// exp(x) for float x, evaluated in double with IEEE basic operations and rounded once to float (the same operation
// sequence as the oracle's vwso_expf): k = round(x / ln 2) by the 1.5 * 2^52 shift, Cody-Waite reduction, degree-13
// Taylor polynomial in Horner form, exact scaling by 2^k.
__device__ __forceinline__ float k6_expf(float xf) {
  const double x = (double)xf;
  if (x != x) return xf;
  if (x < -104.0) return 0.0f;
  if (x > 89.0) return __int_as_float(0x7f800000);
  const double shift = 6755399441055744.0;
  double kd = DA(DM(x, 1.4426950408889634), shift);
  kd = DS(kd, shift);
  const double r = DS(DS(x, DM(kd, 6.93147180369123816490e-01)), DM(kd, 1.90821492927058770002e-10));
  const double c[14] = {1.0, 1.0, 1.0 / 2, 1.0 / 6, 1.0 / 24, 1.0 / 120, 1.0 / 720, 1.0 / 5040, 1.0 / 40320,
                        1.0 / 362880, 1.0 / 3628800, 1.0 / 39916800, 1.0 / 479001600, 1.0 / 6227020800.0};
  double p = c[13];
#pragma unroll
  for (int i = 12; i >= 0; --i) p = DA(DM(p, r), c[i]);
  const double s = __longlong_as_double((long long)((int)kd + 1023) << 52);
  return __double2float_rn(DM(p, s));
}

// math::impl::_floor with the x86 conversion of out-of-range values (INT_MIN), as the oracle states it
__device__ __forceinline__ int k6_floor(double v) {
  const int iv = (v >= -2147483648.0 && v < 2147483648.0) ? (int)v : INT_MIN;
  if (v < 0) return ((double)iv == v) ? iv : (int)((unsigned)iv - 1u);
  return iv;
}
__device__ __forceinline__ float k6_at(const float* __restrict__ img, int w, int h, long long x, long long y) {
  return (x < 0 || y < 0 || x >= w || y >= h) ? 0.0f : __ldg(img + (size_t)y * w + (size_t)x);
}
// BilinearInterpolation over ZeroEdgeExtension (Image/Interpolation.h:76-110): float arithmetic, double coordinates
__device__ __forceinline__ float k6_bilinear(const float* __restrict__ img, int w, int h, float xf, float yf) {
  const double i = (double)xf, j = (double)yf;
  const int x = k6_floor(i), y = k6_floor(j);
  if ((double)x == i && (double)y == j) return k6_at(img, w, h, x, y);
  const float nx = FS(xf, (float)x), ny = FS(yf, (float)y), n1x = FS(1.0f, nx), n1y = FS(1.0f, ny);
  float r = FM(k6_at(img, w, h, x, y), n1x);
  r = FA(r, FM(k6_at(img, w, h, (long long)x + 1, y), nx));
  r = FM(r, n1y);
  float row = FM(k6_at(img, w, h, x, (long long)y + 1), n1x);
  row = FA(row, FM(k6_at(img, w, h, (long long)x + 1, (long long)y + 1), nx));
  return FA(r, FM(row, ny));
}

// norm_2 of a float vector (Math/Vector.h:1593-1604)
template <int N>
__device__ __forceinline__ double k6_norm2(const float* v) {
  double r = 0.0;
#pragma unroll
  for (int i = 0; i < N; ++i) r = DA(r, (double)FM(v[i], v[i]));
  return sqrt((double)__double2float_rn(r));
}

// posv('L') substitution: unblocked Cholesky in spotf2 column order + two triangular solves, float; b left unsolved when
// a pivot is <= 0 or NaN
template <int N>
__device__ __forceinline__ void k6_posv(float (&A)[N][N], float (&b)[N]) {
#pragma unroll
  for (int j = 0; j < N; ++j) {
    float dot = 0.0f;
#pragma unroll
    for (int k = 0; k < j; ++k) dot = FA(dot, FM(A[j][k], A[j][k]));
    float ajj = FS(A[j][j], dot);
    if (!(ajj > 0.0f)) return;
    ajj = __fsqrt_rn(ajj);
    A[j][j] = ajj;
#pragma unroll
    for (int k = 0; k < j; ++k) {
      const float t = -A[j][k];
#pragma unroll
      for (int i = j + 1; i < N; ++i) A[i][j] = FA(A[i][j], FM(t, A[i][k]));
    }
    const float rcp = FD(1.0f, ajj);
#pragma unroll
    for (int i = j + 1; i < N; ++i) A[i][j] = FM(A[i][j], rcp);
  }
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float t = b[i];
#pragma unroll
    for (int k = 0; k < i; ++k) t = FS(t, FM(A[i][k], b[k]));
    b[i] = FD(t, A[i][i]);
  }
#pragma unroll
  for (int i = N - 1; i >= 0; --i) {
    float t = b[i];
#pragma unroll
    for (int k = i + 1; k < N; ++k) t = FS(t, FM(A[k][i], b[k]));
    b[i] = FD(t, A[i][i]);
  }
}

__device__ __forceinline__ void k6_acc_rhs(float* R, int ii, int jj, float Ixs, float Ixy, float Iys) {
  const float m0 = (float)(ii * ii), m1 = (float)(ii * jj), m2 = (float)(jj * jj), fi = (float)ii, fj = (float)jj;
  R[0] = FA(R[0], FM(m0, Ixs)); R[1] = FA(R[1], FM(m1, Ixs)); R[2] = FA(R[2], FM(fi, Ixs));
  R[3] = FA(R[3], FM(m2, Ixs)); R[4] = FA(R[4], FM(fj, Ixs)); R[5] = FA(R[5], Ixs);
  R[6] = FA(R[6], FM(m0, Ixy)); R[7] = FA(R[7], FM(m1, Ixy)); R[8] = FA(R[8], FM(fi, Ixy));
  R[9] = FA(R[9], FM(m2, Ixy)); R[10] = FA(R[10], FM(fj, Ixy)); R[11] = FA(R[11], Ixy);
  R[12] = FA(R[12], FM(m0, Iys)); R[13] = FA(R[13], FM(m1, Iys)); R[14] = FA(R[14], FM(fi, Iys));
  R[15] = FA(R[15], FM(m2, Iys)); R[16] = FA(R[16], FM(fj, Iys)); R[17] = FA(R[17], Iys);
}
// R[0..5]: UL (0,0)(0,1)(0,2)(1,1)(1,2)(2,2); R[6..11]: UR (0,3)(0,4)(0,5)(1,4)(1,5)(2,5); R[12..17]: LR, like UL.
// The symmetric fill of Correlate.cc:694-705 sets (1,3)=(0,4), (2,3)=(0,5), (2,4)=(1,5).
__device__ __forceinline__ void k6_fill(const float* R, float (&M)[6][6]) {
  const float UL[3][3] = {{R[0], R[1], R[2]}, {R[1], R[3], R[4]}, {R[2], R[4], R[5]}};
  const float UR[3][3] = {{R[6], R[7], R[8]}, {R[7], R[9], R[10]}, {R[8], R[10], R[11]}};
  const float LR[3][3] = {{R[12], R[13], R[14]}, {R[13], R[15], R[16]}, {R[14], R[16], R[17]}};
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) { M[i][j] = UL[i][j]; M[i][j + 3] = UR[i][j]; M[j + 3][i] = UR[i][j]; M[i + 3][j + 3] = LR[i][j]; }
}

struct K6Level {
  const float* L; const float* Ix; const float* Iy; int w, h;
  const float* R; int rw, rh;
  int kx, ky;
  int sx0, sy0, sx1, sy1;                 // scan region [sx0,sx1) x [sy0,sy1)
  const float* din;                       // input disparity (values + validity), w x h x 3
  float* dout;                            // refined disparity, starts as a copy of din
  const uint8_t* vin;                     // input validity
  const uint8_t* vprev; uint8_t* vnext;   // validity after round r-1 / r
  const uint8_t* cprev; uint8_t* cnext;   // changed in round r-1 / r
  const float* tmpl;                      // spatial weight template, ky x kx
  int round;
  int* flag;
  unsigned long long* stats;              // [0] re-evaluated pixels, [1] window-pixel evaluations, [2] sum over warps of 32 x max lane
};

// One round of the validity fixpoint.  Returns through dout / vnext / cnext.
template <int ALG>
__global__ void __launch_bounds__(128) k6_level_kernel(K6Level a) {
  extern __shared__ float s_tmpl[];
  const int kp = a.kx * a.ky;
  for (int k = threadIdx.x + threadIdx.y * blockDim.x; k < kp; k += blockDim.x * blockDim.y) s_tmpl[k] = a.tmpl[k];
  __syncthreads();
  const int x = a.sx0 + blockIdx.x * blockDim.x + threadIdx.x, y = a.sy0 + blockIdx.y * blockDim.y + threadIdx.y;
  unsigned evals = 0;
  bool reeval = false;
  if (x < a.sx1 && y < a.sy1) {
    const size_t q = (size_t)y * a.w + x;
    const int khh = a.ky / 2, khw = a.kx / 2;
    bool eval = a.vin[q] != 0;
    if (eval && a.round > 0) {
      // re-evaluate only if an earlier pixel of the window changed validity in the previous round
      bool any = false;
      for (int j = -khh; j <= 0 && !any; ++j)
        for (int i = -khw; i <= khw; ++i) {
          if (j == 0 && i >= 0) break;
          if (a.cprev[(size_t)(y + j) * a.w + (x + i)]) { any = true; break; }
        }
      eval = any;
      reeval = any;
    }
    if (!eval) {
      a.vnext[q] = a.vprev[q];
      a.cnext[q] = 0;
    } else {
      // adjust_weight_image (Correlate.cc:1393-1435): earlier pixels at their current validity, later ones at input
      float sum = 0.0f, w00 = 0.0f;
      int good = 0;
      for (int j = 0; j < a.ky; ++j)
        for (int i = 0; i < a.kx; ++i) {
          const int px = x - khw + i, py = y - khh + j;
          const size_t p = (size_t)py * a.w + px;
          const bool earlier = (py < y) || (py == y && px < x);
          const bool valid = (earlier ? a.vprev[p] : a.vin[p]) != 0;
          const float wv = valid ? s_tmpl[j * a.kx + i] : 0.0f;
          if (valid) { sum = FA(sum, wv); ++good; }
          if (i == 0 && j == 0) w00 = wv;
        }
      w00 = FD(w00, sum);
      const float* dq = a.din + q * 3;
      float* oq = a.dout + q * 3;
      bool valid_out;
      float ox = 0.0f, oy = 0.0f;
      if (good < kp / 2) {
        valid_out = false;
      } else {
        const float max_t = (float)(a.kx / 2);
        const float x_base = FA((float)x, dq[0]), y_base = FA((float)y, dq[1]);
        const float weight0 = FM(1.0f, w00);
#define LP(img, ii, jj) __ldg((img) + (size_t)(y + (jj)) * a.w + (x + (ii)))
        if (ALG == VWB200_SUBPIXEL_LUCAS_KANADE) {
          float d[2] = {0.0f, 0.0f};
          for (int iter = 0; iter < 10; ++iter) {
            if (k6_norm2<2>(d) > (double)max_t) break;
            float r0 = 0.0f, r1 = 0.0f, r3 = 0.0f, lhs[2] = {0.0f, 0.0f};
            for (int jj = -khh; jj <= khh; ++jj) {
              const float xx_partial = FA(x_base, d[0]);
              const float yy = FA(FA(y_base, (float)jj), d[1]);
              for (int ii = -khw; ii <= khw; ++ii) {
                const float xx = FA((float)ii, xx_partial);
                const float ip = k6_bilinear(a.R, a.rw, a.rh, xx, yy);
                const float Ie = FS(ip, LP(a.L, ii, jj));
                const float Ix = LP(a.Ix, ii, jj), Iy = LP(a.Iy, ii, jj);
                const float Ixv = FM(weight0, Ix), Iyv = FM(weight0, Iy);
                lhs[0] = FS(lhs[0], FM(Ixv, Ie));
                lhs[1] = FS(lhs[1], FM(Iyv, Ie));
                r0 = FA(r0, FM(Ixv, Ix)); r1 = FA(r1, FM(Ixv, Iy)); r3 = FA(r3, FM(Iyv, Iy));
              }
            }
            evals += kp;
            float M[2][2] = {{r0, r1}, {r1, r3}};
            k6_posv<2>(M, lhs);
            d[0] = FA(d[0], lhs[0]); d[1] = FA(d[1], lhs[1]);
            if (k6_norm2<2>(lhs) < 0.05) break;
          }
          valid_out = !(k6_norm2<2>(d) > (double)max_t || isnan(d[0]) || isnan(d[1]));
          ox = d[0]; oy = d[1];
        } else {
          float d[6] = {1.0f, 0.0f, 0.0f, 0.0f, 1.0f, 0.0f};
          if (ALG == VWB200_SUBPIXEL_FAST_AFFINE) {
            const int kqh = khh / 2, kqw = khw / 2;
            for (int iter = 0; iter < 10; ++iter) {
              { const float t[2] = {d[2], d[5]}; if (k6_norm2<2>(t) > (double)max_t) break; }
              float R[18], lhs[6];
#pragma unroll
              for (int k = 0; k < 18; ++k) R[k] = 0.0f;
#pragma unroll
              for (int k = 0; k < 6; ++k) lhs[k] = 0.0f;
              for (int jj = -khh; jj <= khh; ++jj) {
                const float xx_partial = FA(FA(x_base, FM(d[1], (float)jj)), d[2]);
                const float yy_partial = FA(FA(y_base, FM(d[4], (float)jj)), d[5]);
                for (int ii = -khw; ii <= khw; ++ii) {
                  const float xx = FA(FM(d[0], (float)ii), xx_partial), yy = FA(FM(d[3], (float)ii), yy_partial);
                  const float ip = k6_bilinear(a.R, a.rw, a.rh, xx, yy);
                  const float Ie = FS(ip, LP(a.L, ii, jj));
                  const float Ix = LP(a.Ix, ii, jj), Iy = LP(a.Iy, ii, jj);
                  const float Ixv = FM(weight0, Ix), Iyv = FM(weight0, Iy);
                  const float IxIe = FM(Ixv, Ie), IyIe = FM(Iyv, Ie);
                  lhs[0] = FS(lhs[0], FM((float)ii, IxIe)); lhs[1] = FS(lhs[1], FM((float)jj, IxIe)); lhs[2] = FS(lhs[2], IxIe);
                  lhs[3] = FS(lhs[3], FM((float)ii, IyIe)); lhs[4] = FS(lhs[4], FM((float)jj, IyIe)); lhs[5] = FS(lhs[5], IyIe);
                  k6_acc_rhs(R, ii, jj, FM(Ixv, Ix), FM(Ixv, Iy), FM(Iyv, Iy));
                }
              }
              evals += kp;
              float M[6][6];
              k6_fill(R, M);
              k6_posv<6>(M, lhs);
#pragma unroll
              for (int k = 0; k < 6; ++k) d[k] = FA(d[k], lhs[k]);
              float wl[6] = {FM(lhs[0], (float)kqw), FM(lhs[1], (float)kqh), lhs[2], FM(lhs[3], (float)kqw), FM(lhs[4], (float)kqh), lhs[5]};
              if (k6_norm2<6>(wl) < 0.05) break;
            }
          } else {
            const int kp_ = kp;
            float curr_sum = 0.0f, prev_sum = 0.0f;
            for (int iter = 0; iter < 10; ++iter) {
              { const float t[2] = {d[2], d[5]}; if (k6_norm2<2>(t) > (double)max_t) break; }
              float R[18], lhs[6], prev_lhs[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f}, d_em[6];
              float mean_noise = 0.0f, w_plane = 0.8f, w_noise = 0.2f;
              const float var2_plane = 1e-3f, var2_noise = 1e-2f;
#pragma unroll
              for (int k = 0; k < 6; ++k) d_em[k] = d[k];
              for (int em = 0; em < 2; ++em) {
                const float noise_norm = __double2float_rn(1.0 / sqrt(2 * M_PI * (double)var2_noise));
                const float plane_norm = __double2float_rn(1.0 / sqrt(2 * M_PI * (double)var2_plane));
#pragma unroll
                for (int k = 0; k < 18; ++k) R[k] = 0.0f;
#pragma unroll
                for (int k = 0; k < 6; ++k) lhs[k] = 0.0f;
                float in_curr = 0.0f, mnt = 0.0f, sgn = 0.0f, sgp = 0.0f;
                int skip = 0;
                for (int jj = -khh; jj <= khh; ++jj) {
                  const float xx_partial = FA(FA(x_base, FM(d[1], (float)jj)), d[2]);
                  const float yy_partial = FA(FA(y_base, FM(d[4], (float)jj)), d[5]);
                  const float dx_partial = FA(FM(d_em[1], (float)jj), d_em[2]);
                  const float dy_partial = FA(FM(d_em[4], (float)jj), d_em[5]);
                  for (int ii = -khw; ii <= khw; ++ii) {
                    const float xx = FA(FM(d[0], (float)ii), xx_partial), yy = FA(FM(d[3], (float)ii), yy_partial);
                    const float delta_x = FA(FM(d_em[0], (float)ii), dx_partial), delta_y = FA(FM(d_em[3], (float)ii), dy_partial);
                    const float ip = k6_bilinear(a.R, a.rw, a.rh, xx, yy);
                    const float Ie = FS(ip, LP(a.L, ii, jj));
                    in_curr = FA(in_curr, Ie);
                    const float Ix = LP(a.Ix, ii, jj), Iy = LP(a.Iy, ii, jj);
                    const float tp = FS(FS(Ie, FM(delta_x, Ix)), FM(delta_y, Iy));
                    const float tn = FS(ip, mean_noise);
                    const float ppe = FD(FM(-1.0f, FM(tp, tp)), FM(2.0f, var2_plane));
                    const float pp = (ppe < -75.0f) ? 0.0f : FM(plane_norm, k6_expf(ppe));
                    const float npe = FD(FM(-1.0f, FM(tn, tn)), FM(2.0f, var2_noise));
                    const float np = (npe < -75.0f) ? 0.0f : FM(noise_norm, k6_expf(npe));
                    const float s = FA(FM(pp, w_plane), FM(np, w_noise));
                    const float gp = FD(FM(pp, w_plane), s), gn = FD(FM(np, w_noise), s);
                    mnt = FA(mnt, FM(ip, gn));
                    sgp = FA(sgp, gp);
                    sgn = FA(sgn, gn);
                    const float weight = FM(gp, w00);
                    if ((double)weight < 1e-26) { skip++; continue; }
                    const float Ixv = FM(weight, Ix), Iyv = FM(weight, Iy);
                    const float fi = (float)ii, fj = (float)jj;
                    lhs[0] = FS(lhs[0], FM(FM(fi, Ixv), Ie)); lhs[1] = FS(lhs[1], FM(FM(fj, Ixv), Ie)); lhs[2] = FS(lhs[2], FM(Ixv, Ie));
                    lhs[3] = FS(lhs[3], FM(FM(fi, Iyv), Ie)); lhs[4] = FS(lhs[4], FM(FM(fj, Iyv), Ie)); lhs[5] = FS(lhs[5], FM(Iyv, Ie));
                    k6_acc_rhs(R, ii, jj, FM(Ixv, Ix), FM(Ixv, Iy), FM(Iyv, Iy));
                  }
                }
                evals += kp;
                if (skip == kp_) break;
                float M[6][6];
                k6_fill(R, M);
                k6_posv<6>(M, lhs);
                mean_noise = FD(mnt, sgn);
                w_plane = FD(sgp, (float)kp_);
                w_noise = FD(sgn, (float)kp_);
                float diff[6];
#pragma unroll
                for (int k = 0; k < 6; ++k) diff[k] = FS(prev_lhs[k], lhs[k]);
                const float conv_error = __double2float_rn(k6_norm2<6>(diff));
#pragma unroll
                for (int k = 0; k < 6; ++k) { d_em[k] = FA(d[k], lhs[k]); prev_lhs[k] = lhs[k]; }
                if (in_curr < 0) in_curr = -in_curr;
                curr_sum = in_curr;
                if ((double)conv_error < 1E-3 && em > 0) break;
              }
#pragma unroll
              for (int k = 0; k < 6; ++k) d[k] = FA(d[k], lhs[k]);
              if (curr_sum < 0) curr_sum = -curr_sum;
              if (prev_sum < curr_sum && iter > 0) break;
              prev_sum = curr_sum;
            }
          }
          { const float t[2] = {d[2], d[5]}; valid_out = !(k6_norm2<2>(t) > (double)max_t || isnan(d[2]) || isnan(d[5])); }
          ox = d[2]; oy = d[5];
        }
#undef LP
      }
      if (valid_out) { oq[0] = FA(dq[0], ox); oq[1] = FA(dq[1], oy); oq[2] = 1.0f; }
      else { oq[0] = dq[0]; oq[1] = dq[1]; oq[2] = 0.0f; }
      const uint8_t nv = valid_out ? 1 : 0;
      a.vnext[q] = nv;
      a.cnext[q] = nv != a.vprev[q];
      if (nv != a.vprev[q]) atomicExch(a.flag, 1);
    }
  }
  // statistics: pixels re-evaluated, window evaluations, warp-lockstep cost
  const unsigned lane_max = __reduce_max_sync(0xffffffffu, evals);
  const unsigned lane_sum = __reduce_add_sync(0xffffffffu, evals);
  const unsigned re = __reduce_add_sync(0xffffffffu, reeval ? 1u : 0u);
  if (((threadIdx.y * blockDim.x + threadIdx.x) & 31) == 0 && (lane_sum || re)) {
    atomicAdd(a.stats + 0, (unsigned long long)re);
    atomicAdd(a.stats + 1, (unsigned long long)lane_sum);
    atomicAdd(a.stats + 2, 32ull * lane_max);
  }
}

// compute_spatial_weight_image (Correlate.cc:36-55), single thread: a serial float sum
__global__ void k6_weight_kernel(int kx, int ky, float two_sigma_sqr, float* out) {
  if (threadIdx.x || blockIdx.x) return;
  const int cx = kx / 2, cy = ky / 2;
  float sum = 0.0f;
  for (int j = 0; j < ky; ++j)
    for (int i = 0; i < kx; ++i) {
      const int r2 = (i - cx) * (i - cx) + (j - cy) * (j - cy);
      out[j * kx + i] = k6_expf(FD((float)(-1 * r2), two_sigma_sqr));
      sum = FA(sum, out[j * kx + i]);
    }
  for (int k = 0; k < kx * ky; ++k) out[k] = FD(out[k], sum);
}

// derivative_filter(img,1,0) / (0,1): taps {-0.5, 0, 0.5} in order from 0, ConstantEdgeExtension on this image
__global__ void k6_deriv_kernel(const float* __restrict__ img, int w, int h, float* __restrict__ ix, float* __restrict__ iy) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const float tap[3] = {-0.5f, 0.0f, 0.5f};
  float rx = 0.0f, ry = 0.0f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    rx = FA(rx, FM(tap[k], img[(size_t)y * w + min(max(x - 1 + k, 0), w - 1)]));
    ry = FA(ry, FM(tap[k], img[(size_t)min(max(y - 1 + k, 0), h - 1) * w + x]));
  }
  ix[(size_t)y * w + x] = rx;
  iy[(size_t)y * w + x] = ry;
}

__global__ void k6_subsample_kernel(const float* __restrict__ in, int w, float* __restrict__ out, int ow, int oh) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= ow || y >= oh) return;
  out[(size_t)y * ow + x] = in[(size_t)(2 * y) * w + 2 * x];
}

// disparity_subsample (DisparityMap.h:1253-1314) over ConstantEdgeExtension
__global__ void k6_disp_subsample_kernel(const float* __restrict__ in, int w, int h, float* __restrict__ out, int ow, int oh) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= ow || j >= oh) return;
  const int nb[9][3] = {{0, 0, 10}, {1, 0, 5}, {0, 1, 5}, {-1, 0, 5}, {0, -1, 5}, {1, 1, 2}, {-1, -1, 2}, {-1, 1, 2}, {1, -1, 2}};
  double bx = 0.0, by = 0.0, cnt = 0.0;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const float* p = in + ((size_t)min(max(2 * j + nb[k][1], 0), h - 1) * w + min(max(2 * i + nb[k][0], 0), w - 1)) * 3;
    if (p[2] == 0.0f) continue;
    cnt = DA(cnt, (double)nb[k][2]);
    if (k < 3) { bx = DA(bx, DM((double)nb[k][2], (double)p[0])); by = DA(by, DM((double)nb[k][2], (double)p[1])); }
    else { bx = DA(bx, (double)FM((float)nb[k][2], p[0])); by = DA(by, (double)FM((float)nb[k][2], p[1])); }
  }
  float* o = out + ((size_t)j * ow + i) * 3;
  if (cnt > 0) { o[0] = __double2float_rn(__ddiv_rn(bx, DM(cnt, 2.0))); o[1] = __double2float_rn(__ddiv_rn(by, DM(cnt, 2.0))); o[2] = 1.0f; }
  else { o[0] = 0.0f; o[1] = 0.0f; o[2] = 0.0f; }
}

// crop(disparity_upsample(edge_extend(in)), BBox2i(0,0,ow,oh))
__global__ void k6_disp_upsample_kernel(const float* __restrict__ in, int w, int h, float* __restrict__ out, int ow, int oh) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= ow || j >= oh) return;
  const float* p = in + ((size_t)min(j >> 1, h - 1) * w + min(i >> 1, w - 1)) * 3;
  float* o = out + ((size_t)j * ow + i) * 3;
  o[0] = FM(p[0], 2.0f); o[1] = FM(p[1], 2.0f); o[2] = p[2];
}

__global__ void k6_validity_kernel(const float* __restrict__ d, size_t n, uint8_t* __restrict__ v) {
  for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x) v[k] = d[k * 3 + 2] != 0.0f;
}

// min / max over EVERY pixel of a bbox crop, truncated to int (get_disparity_range, DisparityMap.h:52-66, then the
// BBox2f -> BBox2i conversion; truncation is monotonic, so min of the truncations == truncation of the min).
// r[4] is set when a value is NaN, infinite or of magnitude >= 2^24: such a crop is rejected (VWB200_EARG).
__global__ void k6_range_kernel(const float* __restrict__ disp, int cols, int bx0, int by0, int bw, int bh, int* __restrict__ r) {
  int mnx = INT_MAX, mny = INT_MAX, mxx = INT_MIN, mxy = INT_MIN, bad = 0;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < (long long)bw * bh; k += (long long)gridDim.x * blockDim.x) {
    const float* p = disp + ((ptrdiff_t)(by0 + (int)(k / bw)) * cols + bx0 + (int)(k % bw)) * 3;
    if (!(fabsf(p[0]) < 16777216.0f) || !(fabsf(p[1]) < 16777216.0f)) { bad = 1; continue; }
    mnx = min(mnx, (int)p[0]); mxx = max(mxx, (int)p[0]);
    mny = min(mny, (int)p[1]); mxy = max(mxy, (int)p[1]);
  }
  mnx = __reduce_min_sync(0xffffffffu, mnx); mny = __reduce_min_sync(0xffffffffu, mny);
  mxx = __reduce_max_sync(0xffffffffu, mxx); mxy = __reduce_max_sync(0xffffffffu, mxy);
  bad = __reduce_or_sync(0xffffffffu, (unsigned)bad);
  if ((threadIdx.x & 31) == 0) {
    atomicMin(r + 0, mnx); atomicMin(r + 1, mny); atomicMax(r + 2, mxx); atomicMax(r + 3, mxy);
    if (bad) atomicExch(r + 4, 1);
  }
}

// crop(edge_extend(disp, Zero), box) - (tx, ty)
__global__ void k6_disp_crop_kernel(const float* __restrict__ disp, int cols, int rows, int x0, int y0, int w, int h, float tx, float ty,
                                    float* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const int gx = x0 + x, gy = y0 + y;
  float v[3] = {0.0f, 0.0f, 0.0f};
  if (gx >= 0 && gy >= 0 && gx < cols && gy < rows) {
    const float* p = disp + ((size_t)gy * cols + gx) * 3;
    v[0] = p[0]; v[1] = p[1]; v[2] = p[2];
  }
  float* o = out + ((size_t)y * w + x) * 3;
  o[0] = FS(v[0], tx); o[1] = FS(v[1], ty); o[2] = v[2];
}

// out(i,j) = patch(ox + i, oy + j) + (tx, ty)
__global__ void k6_disp_out_kernel(const float* __restrict__ patch, int pw, int ox, int oy, float tx, float ty, int w, int h,
                                   float* __restrict__ out, ptrdiff_t opitch) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const float* p = patch + ((size_t)(oy + y) * pw + (ox + x)) * 3;
  float* o = out + ((size_t)y * opitch + x) * 3;
  o[0] = FA(p[0], tx); o[1] = FA(p[1], ty); o[2] = p[2];
}

static dim3 grid2(int w, int h, dim3 b) { return dim3((unsigned)((w + b.x - 1) / b.x), (unsigned)((h + b.y - 1) / b.y)); }

int k6_range_launch(const float* disp, int cols, int bx0, int by0, int bw, int bh, int* d_r5, cudaStream_t st) {
  const int init[5] = {INT_MAX, INT_MAX, INT_MIN, INT_MIN, 0};
  VWB_CUDA(cudaMemcpyAsync(d_r5, init, sizeof(init), cudaMemcpyHostToDevice, st));
  VWB_CUDA(cudaStreamSynchronize(st));
  k6_range_kernel<<<148, 256, 0, st>>>(disp, cols, bx0, by0, bw, bh, d_r5);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}
int k6_disp_crop_launch(const float* disp, int cols, int rows, int x0, int y0, int w, int h, float tx, float ty, float* out, cudaStream_t st) {
  dim3 b(32, 8);
  k6_disp_crop_kernel<<<grid2(w, h, b), b, 0, st>>>(disp, cols, rows, x0, y0, w, h, tx, ty, out);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}
int k6_disp_out_launch(const float* patch, int pw, int ox, int oy, float tx, float ty, int w, int h, float* out, ptrdiff_t opitch, cudaStream_t st) {
  dim3 b(32, 8);
  k6_disp_out_kernel<<<grid2(w, h, b), b, 0, st>>>(patch, pw, ox, oy, tx, ty, w, h, out, opitch);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

// One level function on device buffers, in place on disp (w x h x 3, dense).  L (w x h) and R (rw x rh) dense.
int k6_level_run(int alg, float* disp, const float* L, int w, int h, const float* R, int rw, int rh, int kx, int ky,
                 int rx0, int ry0, int rx1, int ry1, Arena& ar, cudaStream_t st, vwb200_subpixel_stats* stats) {
  const int khh = ky / 2, khw = kx / 2;
  const int sx0 = std::max(rx0 - 1, khw), sx1 = std::min(w - khw, rx1 + 1), sy0 = std::max(ry0 - 1, khh), sy1 = std::min(h - khh, ry1 + 1);
  if (sx0 >= sx1 || sy0 >= sy1) return VWB200_OK;
  const size_t n = (size_t)w * h;
  float *tmpl, *ix, *iy, *din;
  uint8_t *vin, *v0, *v1, *c0, *c1;
  int* flag;
  unsigned long long* dstats;
  VWB_TRY(ar.alloc(&tmpl, (size_t)kx * ky)); VWB_TRY(ar.alloc(&ix, n)); VWB_TRY(ar.alloc(&iy, n)); VWB_TRY(ar.alloc(&din, n * 3));
  VWB_TRY(ar.alloc(&vin, n)); VWB_TRY(ar.alloc(&v0, n)); VWB_TRY(ar.alloc(&v1, n)); VWB_TRY(ar.alloc(&c0, n)); VWB_TRY(ar.alloc(&c1, n));
  VWB_TRY(ar.alloc(&flag, 1)); VWB_TRY(ar.alloc(&dstats, 3));
  const float two_sigma_sqr = (float)(2.0 * std::pow((double)(float)kx / 5.0, 2.0));
  k6_weight_kernel<<<1, 32, 0, st>>>(kx, ky, two_sigma_sqr, tmpl);
  VWB_LAUNCH_CHECK();
  dim3 b2(32, 8);
  k6_deriv_kernel<<<grid2(w, h, b2), b2, 0, st>>>(L, w, h, ix, iy);
  VWB_LAUNCH_CHECK();
  VWB_CUDA(cudaMemcpyAsync(din, disp, n * 3 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  k6_validity_kernel<<<148, 256, 0, st>>>(disp, n, vin);
  VWB_LAUNCH_CHECK();
  VWB_CUDA(cudaMemcpyAsync(v0, vin, n, cudaMemcpyDeviceToDevice, st));
  VWB_CUDA(cudaMemcpyAsync(v1, vin, n, cudaMemcpyDeviceToDevice, st));
  VWB_CUDA(cudaMemsetAsync(c0, 0, n, st));
  VWB_CUDA(cudaMemsetAsync(c1, 0, n, st));
  VWB_CUDA(cudaMemsetAsync(dstats, 0, 3 * sizeof(unsigned long long), st));
  K6Level a{L, ix, iy, w, h, R, rw, rh, kx, ky, sx0, sy0, sx1, sy1, din, disp, vin, v0, v1, c0, c1, tmpl, 0, flag, dstats};
  dim3 b(32, 4), g((unsigned)((sx1 - sx0 + 31) / 32), (unsigned)((sy1 - sy0 + 3) / 4));
  const size_t smem = (size_t)kx * ky * sizeof(float);
  const long long max_rounds = (long long)(sx1 - sx0) * (sy1 - sy0) + 1;
  int rounds = 0;
  for (;;) {
    int h_flag = 0;
    VWB_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    a.round = rounds;
    if (alg == VWB200_SUBPIXEL_LUCAS_KANADE) k6_level_kernel<VWB200_SUBPIXEL_LUCAS_KANADE><<<g, b, smem, st>>>(a);
    else if (alg == VWB200_SUBPIXEL_FAST_AFFINE) k6_level_kernel<VWB200_SUBPIXEL_FAST_AFFINE><<<g, b, smem, st>>>(a);
    else k6_level_kernel<VWB200_SUBPIXEL_BAYES_EM><<<g, b, smem, st>>>(a);
    VWB_LAUNCH_CHECK();
    VWB_CUDA(cudaMemcpyAsync(&h_flag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
    ++rounds;
    if (!h_flag) break;
    if (rounds > max_rounds) { set_error("subpixel: validity fixpoint did not converge"); return VWB200_ELOGIC; }
    { uint8_t* v = a.vnext; a.vnext = const_cast<uint8_t*>(a.vprev); a.vprev = v; }
    { uint8_t* c = a.cnext; a.cnext = const_cast<uint8_t*>(a.cprev); a.cprev = c; }
    // vprev now holds round r's validity; vnext (round r-1) is fully rewritten inside the scan region by the next round
    // and equal to the input outside it
  }
  unsigned long long hs[3];
  VWB_CUDA(cudaMemcpyAsync(hs, dstats, sizeof(hs), cudaMemcpyDeviceToHost, st));
  VWB_CUDA(cudaStreamSynchronize(st));
  if (stats) {
    stats->levels += 1;
    stats->fixpoint_rounds += rounds;
    stats->pixels_reevaluated += (long long)hs[0];
    stats->window_evaluations += (long long)hs[1];
    stats->lane_slots += (long long)hs[2];
    stats->pixels += (long long)(sx1 - sx0) * (sy1 - sy0);
  }
  return VWB200_OK;
}

// PyramidSubpixelView::prerasterize after the crops (SubpixelView.cc:98-214): D (pw x ph x 3) is the translated disparity
// patch, L / R the filtered patches (both pw x ph).  Refines D in place.
int k6_pyramid_run(int alg, float* D, const float* L, const float* R, int pw, int ph, int kx, int ky, int bw, int bh, int levels,
                   Arena& ar, cudaStream_t st, vwb200_subpixel_stats* stats) {
  struct Lv { const float* l; const float* r; int w, h; int roi[4]; };
  std::vector<Lv> lv(levels + 1);
  lv[0] = Lv{L, R, pw, ph, {kx, ky, kx + bw, ky + bh}};
  std::vector<float*> dl(levels + 1);
  dl[0] = D;
  dim3 b(32, 8);
  for (int i = 1; i <= levels; ++i) {
    const int w = 1 + (lv[i - 1].w - 1) / 2, h = 1 + (lv[i - 1].h - 1) / 2;
    float *l, *r, *d;
    VWB_TRY(ar.alloc(&l, (size_t)w * h)); VWB_TRY(ar.alloc(&r, (size_t)w * h)); VWB_TRY(ar.alloc(&d, (size_t)w * h * 3));
    k6_subsample_kernel<<<grid2(w, h, b), b, 0, st>>>(lv[i - 1].l, lv[i - 1].w, l, w, h);
    VWB_LAUNCH_CHECK();
    k6_subsample_kernel<<<grid2(w, h, b), b, 0, st>>>(lv[i - 1].r, lv[i - 1].w, r, w, h);
    VWB_LAUNCH_CHECK();
    k6_disp_subsample_kernel<<<grid2(w, h, b), b, 0, st>>>(dl[i - 1], lv[i - 1].w, lv[i - 1].h, d, w, h);
    VWB_LAUNCH_CHECK();
    Lv n{l, r, w, h, {0, 0, 0, 0}};
    const int* pr = lv[i - 1].roi;
    const bool empty = pr[0] >= pr[2] || pr[1] >= pr[3];     // BBox2i / 2 leaves an empty box unchanged
    for (int k = 0; k < 4; ++k) n.roi[k] = empty ? pr[k] : pr[k] / 2;
    lv[i] = n;
    dl[i] = d;
  }
  float* cur = dl[levels];
  for (int i = levels; i >= 0; --i) {
    VWB_TRY(k6_level_run(alg, cur, lv[i].l, lv[i].w, lv[i].h, lv[i].r, lv[i].w, lv[i].h, kx, ky,
                         lv[i].roi[0], lv[i].roi[1], lv[i].roi[2], lv[i].roi[3], ar, st, stats));
    if (i == 0) break;
    float* up = dl[i - 1];     // the finer level's subsample input is no longer needed: reuse its buffer
    k6_disp_upsample_kernel<<<grid2(lv[i - 1].w, lv[i - 1].h, b), b, 0, st>>>(cur, lv[i].w, lv[i].h, up, lv[i - 1].w, lv[i - 1].h);
    VWB_LAUNCH_CHECK();
    cur = up;
  }
  return VWB200_OK;
}

}  // namespace vwb200
