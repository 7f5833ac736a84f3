// k7_corr_eval.cu -- K7: CorrEval (Stereo/CorrEval.h:56-129, CorrEval.cc:15-317), the per-pixel NCC, stddev,
// parabola_curvature or cramer_rao quality of a float PixelMask<Vector2f> disparity.
//
// One thread per output pixel walks its window in the reference's column-major (c outer, r inner) order with fp64
// sums built from __dmul_rn / __dadd_rn (no FMA contraction) and the float bilinear sequence of
// Image/Interpolation.h:76-110, so results are bit-identical to the sequential CPU order (DESIGN.md section K7).
// The right image is sampled relative to the crop origin right_box.min() (CorrEval.cc:46,52): float(coordinate)
// rounds differently at different magnitudes, so k7_origin_kernel reduces that origin on the device first.
#include "common.cuh"
#include <climits>

namespace vwb200 {

#define FA __fadd_rn
#define FM __fmul_rn
#define DA __dadd_rn
#define DS __dsub_rn
#define DM __dmul_rn
#define DD __ddiv_rn

static constexpr int K7_BX = 32, K7_BY = 8;
static constexpr size_t K7_STAGE_MAX = 48 * 1024;

struct K7Args {
  const float2* L; int lw, lh; ptrdiff_t lpitch;   // PixelMask<float> {value, valid}, pitch in pixels
  const float2* R; int rw, rh; ptrdiff_t rpitch;
  const float* D; ptrdiff_t dpitch;                // PixelMask<Vector2f> {dx, dy, valid}, pitch in pixels
  int x0, y0, bw, bh;                              // bbox
  int kx, ky, sample_rate;
  int margin;                                      // right_box expansion beyond the half kernel: 1 + 2 + extra_padding (+ 1)
  const int* org;                                  // {min over sampled valid pixels of floor(double(x0 + col) + dx), ... y, bad}
  float2* out; ptrdiff_t opitch;
  int staged;                                      // the left tile + halo is in shared memory
};

__device__ __forceinline__ bool k7_sampled(int col, int row, int sr) { return col % sr == 0 && row % sr == 0; }

// The minimum of right_box (CorrEval.cc:189-203) before its expansion, and the engine's rule on sampled valid disparities.
// The coordinate is rounded as the reference rounds it: double(left_pix) + double(d), then floor (ceil >= floor).
template <bool ROUND>
__global__ void k7_origin_kernel(const float* __restrict__ D, ptrdiff_t dpitch, int x0, int y0, int bw, int bh, int sr, int* __restrict__ org) {
  int mnx = INT_MAX, mny = INT_MAX, bad = 0;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < (long long)bw * bh; k += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(k % bw), row = (int)(k / bw);
    const float* p = D + ((size_t)(y0 + row) * dpitch + (size_t)(x0 + col)) * 3;
    if (p[2] == 0.0f || !k7_sampled(col, row, sr)) continue;
    float dx = p[0], dy = p[1];
    if (!(fabsf(dx) < 16777216.0f) || !(fabsf(dy) < 16777216.0f)) { bad = 1; continue; }
    if (ROUND) { dx = roundf(dx); dy = roundf(dy); }
    mnx = min(mnx, __double2int_rd(DA((double)(x0 + col), (double)dx)));
    mny = min(mny, __double2int_rd(DA((double)(y0 + row), (double)dy)));
  }
  mnx = __reduce_min_sync(0xffffffffu, mnx);
  mny = __reduce_min_sync(0xffffffffu, mny);
  bad = __reduce_or_sync(0xffffffffu, (unsigned)bad);
  if ((threadIdx.x & 31) == 0) {
    if (mnx != INT_MAX) { atomicMin(org + 0, mnx); atomicMin(org + 1, mny); }
    if (bad) atomicExch(org + 2, 1);
  }
}

__device__ __forceinline__ float2 k7_right(const K7Args& a, int X, int Y) {
  return (X < 0 || Y < 0 || X >= a.rw || Y >= a.rh) ? make_float2(0.0f, 0.0f) : __ldg(a.R + (size_t)Y * a.rpitch + X);
}

// One axis of a bilinear sample of left pixel l at disparity d: the crop-relative coordinate is rounded twice, as in
// CorrEval.cc:46,52 (right_pix = double(left_pix) + double(d), then right_pix -= right_box.min()); neither step is exact
// in general (a tiny d is lost against l).  Then floor, the integer test and the float weights
// normx = float(q) - float(floor(q)), 1 - normx (Interpolation.h:83-93).
struct K7Axis { int p; bool at_int; float n, n1; };
__device__ __forceinline__ K7Axis k7_axis(int l, float d, int o) {
  const double q = DS(DA((double)l, (double)d), (double)o);
  K7Axis ax;
  ax.p = __double2int_rd(q);
  ax.at_int = (double)ax.p == q;
  ax.n = __fsub_rn(__double2float_rn(q), __int2float_rn(ax.p));
  ax.n1 = __fsub_rn(1.0f, ax.n);
  return ax;
}

// BilinearInterpolation of PixelMask<float> over the invalid edge: the child of every operation is computed, the
// validity is the AND of the four pixels; at an integer position the pixel itself.  (ox, oy): right_box.min().
__device__ __forceinline__ float2 k7_bilinear(const K7Args& a, const K7Axis& ax, const K7Axis& ay, int ox, int oy) {
  const int X = ax.p + ox, Y = ay.p + oy;
  if (ax.at_int && ay.at_int) return k7_right(a, X, Y);
  const float2 p00 = k7_right(a, X, Y), p10 = k7_right(a, X + 1, Y), p01 = k7_right(a, X, Y + 1), p11 = k7_right(a, X + 1, Y + 1);
  float r = FM(p00.x, ax.n1);
  r = FA(r, FM(p10.x, ax.n));
  r = FM(r, ay.n1);
  float row = FM(p01.x, ax.n1);
  row = FA(row, FM(p11.x, ax.n));
  r = FA(r, FM(row, ay.n));
  const bool ok = p00.y != 0.0f && p10.y != 0.0f && p01.y != 0.0f && p11.y != 0.0f;
  return make_float2(r, ok ? 1.0f : 0.0f);
}

// right sample at the axes' crop-relative positions; (ox, oy) = right_box.min()
template <bool ROUND>
__device__ __forceinline__ float2 k7_sample(const K7Args& a, const K7Axis& ax, const K7Axis& ay, int ox, int oy) {
  if (ROUND) return k7_right(a, ax.p + ox, ay.p + oy);   // integer positions: right(x, y) without interpolation
  return k7_bilinear(a, ax, ay, ox, oy);
}

__device__ __forceinline__ void k7_ncc_acc(double a, float bv, double& num, double& den2) {
  const double b = (double)bv;
  num = DA(num, DM(a, b));
  den2 = DA(den2, DM(b, b));
}
__device__ __forceinline__ double k7_ncc(double num, double den1, double den2) {
  if (den1 > 0.0 && den2 > 0.0) return DD(num, __dsqrt_rn(DM(den1, den2)));
  return -1.0;
}

template <int METRIC, bool ROUND>
__global__ void __launch_bounds__(K7_BX * K7_BY) k7_corr_eval_kernel(K7Args a) {
  extern __shared__ float2 s_left[];
  if (__ldg(a.org + 2)) return;                              // the call is rejected: write nothing
  const int hx = a.kx / 2, hy = a.ky / 2;
  const int tw = K7_BX + a.kx - 1, th = K7_BY + a.ky - 1;
  const int cx0 = blockIdx.x * K7_BX, cy0 = blockIdx.y * K7_BY;
  const int lx0 = a.x0 + cx0 - hx, ly0 = a.y0 + cy0 - hy;    // left image position of tile (0, 0)
  if (a.staged) {
    // left crop with the invalid edge applied at staging (CorrEval.cc:216-222)
    for (int k = threadIdx.y * K7_BX + threadIdx.x; k < tw * th; k += K7_BX * K7_BY) {
      const int X = lx0 + k % tw, Y = ly0 + k / tw;
      float2 v = make_float2(0.0f, 0.0f);
      if (X >= 0 && Y >= 0 && X < a.lw && Y < a.lh) {
        v = __ldg(a.L + (size_t)Y * a.lpitch + X);
        v.y = v.y != 0.0f ? 1.0f : 0.0f;
      }
      s_left[k] = v;
    }
    __syncthreads();
  }
  const int col = cx0 + threadIdx.x, row = cy0 + threadIdx.y;
  if (col >= a.bw || row >= a.bh) return;
  float2* o = a.out + (size_t)row * a.opitch + col;
  const float* dp = a.D + ((size_t)(a.y0 + row) * a.dpitch + (size_t)(a.x0 + col)) * 3;
  const float dvalid = dp[2];
  if (dvalid == 0.0f || !k7_sampled(col, row, a.sample_rate)) { *o = make_float2(0.0f, 0.0f); return; }
  float dx = dp[0], dy = dp[1];
  if (ROUND) { dx = roundf(dx); dy = roundf(dy); }
  // right_box.min() = the reduced minimum - half_kernel - margin; left pixel of window column c: x0 + col + c - hx
  const int ox = __ldg(a.org + 0) - hx - a.margin, oy = __ldg(a.org + 1) - hy - a.margin;
  const int kx0 = a.x0 + col - hx, ky0 = a.y0 + row - hy;
  auto left_at = [&](int c, int r) -> float2 {
    if (a.staged) return s_left[(threadIdx.y + r) * tw + threadIdx.x + c];
    const int X = lx0 + threadIdx.x + c, Y = ly0 + threadIdx.y + r;
    if (X < 0 || Y < 0 || X >= a.lw || Y >= a.lh) return make_float2(0.0f, 0.0f);
    const float2 v = __ldg(a.L + (size_t)Y * a.lpitch + X);
    return make_float2(v.x, v.y != 0.0f ? 1.0f : 0.0f);
  };
  float2 res = make_float2(0.0f, 0.0f);

  if (METRIC == VWB200_CORR_EVAL_NCC) {
    double num = 0.0, den1 = 0.0, den2 = 0.0;
    for (int c = 0; c < a.kx; ++c) {
      const K7Axis ax = k7_axis(kx0 + c, dx, ox);
      for (int r = 0; r < a.ky; ++r) {
        const K7Axis ay = k7_axis(ky0 + r, dy, oy);
        const double lv = (double)left_at(c, r).x;
        den1 = DA(den1, DM(lv, lv));
        k7_ncc_acc(lv, k7_sample<ROUND>(a, ax, ay, ox, oy).x, num, den2);
      }
    }
    const double ncc = k7_ncc(num, den1, den2);
    if (ncc >= 0) res = make_float2(__double2float_rn(ncc), 1.0f);
  } else if (METRIC == VWB200_CORR_EVAL_STDDEV) {
    // calc_stddev of each patch: mean over the valid pixels, then the mean squared deviation
    int nl = 0, nr = 0;
    double ml = 0.0, mr = 0.0;
    for (int c = 0; c < a.kx; ++c) {
      const K7Axis ax = k7_axis(kx0 + c, dx, ox);
      for (int r = 0; r < a.ky; ++r) {
        const K7Axis ay = k7_axis(ky0 + r, dy, oy);
        const float2 lv = left_at(c, r), rv = k7_sample<ROUND>(a, ax, ay, ox, oy);
        if (lv.y != 0.0f) { ++nl; ml = DA(ml, (double)lv.x); }
        if (rv.y != 0.0f) { ++nr; mr = DA(mr, (double)rv.x); }
      }
    }
    if (nl > 0 && nr > 0) {
      ml = DD(ml, (double)nl);
      mr = DD(mr, (double)nr);
      double sl = 0.0, sr = 0.0;
      for (int c = 0; c < a.kx; ++c) {
        const K7Axis ax = k7_axis(kx0 + c, dx, ox);
        for (int r = 0; r < a.ky; ++r) {
          const K7Axis ay = k7_axis(ky0 + r, dy, oy);
          const float2 lv = left_at(c, r), rv = k7_sample<ROUND>(a, ax, ay, ox, oy);
          if (lv.y != 0.0f) { const double t = DS((double)lv.x, ml); sl = DA(sl, DM(t, t)); }
          if (rv.y != 0.0f) { const double t = DS((double)rv.x, mr); sr = DA(sr, DM(t, t)); }
        }
      }
      const double ls = __dsqrt_rn(DD(sl, (double)nl)), rs = __dsqrt_rn(DD(sr, (double)nr));
      if (ls >= 0.0 && rs >= 0.0) res = make_float2(__double2float_rn(DD(DA(ls, rs), 2.0)), 1.0f);
    }
  } else {
    // parabola_curvature / cramer_rao: the NCC at d and at the four float-shifted disparities d + (+-1, 0), (0, +-1)
    // (CorrEval.cc:281-291), five accumulator triples in one pass; each keeps its own order.  The left patch and hence
    // den1 are the same for all five.
    const float dxp = FA(dx, 1.0f), dxm = FA(dx, -1.0f), dyp = FA(dy, 1.0f), dym = FA(dy, -1.0f);
    double den1 = 0.0, num[5] = {0.0, 0.0, 0.0, 0.0, 0.0}, den2[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int c = 0; c < a.kx; ++c) {
      const K7Axis ax = k7_axis(kx0 + c, dx, ox), axp = k7_axis(kx0 + c, dxp, ox), axm = k7_axis(kx0 + c, dxm, ox);
      for (int r = 0; r < a.ky; ++r) {
        const K7Axis ay = k7_axis(ky0 + r, dy, oy), ayp = k7_axis(ky0 + r, dyp, oy), aym = k7_axis(ky0 + r, dym, oy);
        const double lv = (double)left_at(c, r).x;
        den1 = DA(den1, DM(lv, lv));
        k7_ncc_acc(lv, k7_sample<ROUND>(a, ax, ay, ox, oy).x, num[0], den2[0]);
        k7_ncc_acc(lv, k7_sample<ROUND>(a, axp, ay, ox, oy).x, num[1], den2[1]);
        k7_ncc_acc(lv, k7_sample<ROUND>(a, axm, ay, ox, oy).x, num[2], den2[2]);
        k7_ncc_acc(lv, k7_sample<ROUND>(a, ax, ayp, ox, oy).x, num[3], den2[3]);
        k7_ncc_acc(lv, k7_sample<ROUND>(a, ax, aym, ox, oy).x, num[4], den2[4]);
      }
    }
    const double C = k7_ncc(num[0], den1, den2[0]);
    double nbr[4];
    bool ok = C >= 0;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      nbr[s] = k7_ncc(num[s + 1], den1, den2[s + 1]);
      if (nbr[s] < 0) ok = false;
    }
    if (ok) {
      const double kxx = DS(DS(DM(2.0, C), nbr[0]), nbr[1]);
      const double kyy = DS(DS(DM(2.0, C), nbr[2]), nbr[3]);
      if (kxx > 0 && kyy > 0) {
        double sigma = __dsqrt_rn(DA(DD(1.0, kxx), DD(1.0, kyy)));
        if (METRIC == VWB200_CORR_EVAL_CRAMER_RAO) {
          double resid = DS(1.0, C);
          if (resid < 0) resid = 0;
          sigma = DM(sigma, __dsqrt_rn(resid));
        }
        res = make_float2(__double2float_rn(sigma), 1.0f);
      }
    }
  }
  *o = res;
}

int k7_origin_launch(const float* D, ptrdiff_t dpitch, int x0, int y0, int bw, int bh, int sample_rate, int round_to_int, int* d_org3,
                     cudaStream_t st) {
  VWB_CUDA(cudaMemsetAsync(d_org3, 0x7f, 2 * sizeof(int), st));   // INT_MAX-like sentinel: no sampled valid pixel
  VWB_CUDA(cudaMemsetAsync(d_org3 + 2, 0, sizeof(int), st));
  const long long n = (long long)bw * bh;
  const int blocks = (int)std::min<long long>((n + 255) / 256, 148 * 8);
  if (round_to_int) k7_origin_kernel<true><<<blocks, 256, 0, st>>>(D, dpitch, x0, y0, bw, bh, sample_rate, d_org3);
  else k7_origin_kernel<false><<<blocks, 256, 0, st>>>(D, dpitch, x0, y0, bw, bh, sample_rate, d_org3);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

template <int METRIC>
static void k7_launch_metric(const K7Args& a, bool round, dim3 g, dim3 b, size_t smem, cudaStream_t st) {
  if (round) k7_corr_eval_kernel<METRIC, true><<<g, b, smem, st>>>(a);
  else k7_corr_eval_kernel<METRIC, false><<<g, b, smem, st>>>(a);
}

int k7_corr_eval_launch(const float* L, int lw, int lh, ptrdiff_t lpitch, const float* R, int rw, int rh, ptrdiff_t rpitch,
                        const float* D, ptrdiff_t dpitch, int x0, int y0, int bw, int bh, int kx, int ky, int metric, int sample_rate,
                        int round_to_int, int margin, const int* d_org3, float* out, ptrdiff_t opitch, cudaStream_t st) {
  K7Args a;
  a.L = reinterpret_cast<const float2*>(L); a.lw = lw; a.lh = lh; a.lpitch = lpitch;
  a.R = reinterpret_cast<const float2*>(R); a.rw = rw; a.rh = rh; a.rpitch = rpitch;
  a.D = D; a.dpitch = dpitch;
  a.x0 = x0; a.y0 = y0; a.bw = bw; a.bh = bh;
  a.kx = kx; a.ky = ky; a.sample_rate = sample_rate; a.margin = margin;
  a.org = d_org3;
  a.out = reinterpret_cast<float2*>(out); a.opitch = opitch;
  const size_t stage = (size_t)(K7_BX + kx - 1) * (size_t)(K7_BY + ky - 1) * sizeof(float2);
  a.staged = stage <= K7_STAGE_MAX;
  const size_t smem = a.staged ? stage : 0;
  const dim3 b(K7_BX, K7_BY), g((unsigned)((bw + K7_BX - 1) / K7_BX), (unsigned)((bh + K7_BY - 1) / K7_BY));
  const bool round = round_to_int != 0;
  switch (metric) {
    case VWB200_CORR_EVAL_NCC: k7_launch_metric<VWB200_CORR_EVAL_NCC>(a, round, g, b, smem, st); break;
    case VWB200_CORR_EVAL_STDDEV: k7_launch_metric<VWB200_CORR_EVAL_STDDEV>(a, round, g, b, smem, st); break;
    case VWB200_CORR_EVAL_PARABOLA_CURVATURE: k7_launch_metric<VWB200_CORR_EVAL_PARABOLA_CURVATURE>(a, round, g, b, smem, st); break;
    case VWB200_CORR_EVAL_CRAMER_RAO: k7_launch_metric<VWB200_CORR_EVAL_CRAMER_RAO>(a, round, g, b, smem, st); break;
    default: set_error("corr_eval: invalid metric %d", metric); return VWB200_EARG;
  }
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

}  // namespace vwb200
