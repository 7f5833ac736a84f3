// k1_screen.cu -- exact-integer fast path with fp32 screening: NCC (CROSS_CORRELATION) and wide-range SquaredCost.
//
// Reference (Stereo/CostFunctions.h:178-236, Stereo/Correlation.cc:79-133), per disparity d:
//     NCC : cost(d) = double(box(l*r)) * sqrt(lp * rp[d]),  lp = 1/box(l^2), rp = 1/box(r^2)    (double, IEEE), arg-MAX, strict '>'
//     SQ  : cost(d) = box((l-r)^2)                                                                 arg-MIN, strict '<'
// both in dy-major / dx-minor order (the first disparity wins ties).  For integer imagery of <= 12 bits the data-dependent
// part of either cost is S' = box((l-c)(r-c)), c = mid-range, which fits int32:
//     NCC : box(l*r)     = S' + c*(Sl + Sr[d]) - N*c^2                Sl, Sr   = box sums of l, r
//     SQ  : box((l-r)^2) = SL2 + SR2[d] - 2*S'                        SL2, SR2 = box sums of (l-c)^2, (r-c)^2
// The hot loop is the one of k1_fast.cu (TMA-staged tiles, 8 columns x 8 dx per lane, sliding IMAD column sums, shuffle
// window sums; work unit = one dx octet x one row half of a band, drawn by the 8 warps from a shared counter) and carries S'
// EXACTLY.  What it does not do is evaluate the cost:
//   * per pixel a float threshold T is kept that is a proven LOWER bound of the best cost seen so far (NCC: in units of
//     cost/sqrt(lp); SQ: of M0 - cost).  Per (pixel, d) 3-4 fp32 operations with directed rounding decide whether the cost
//     CAN reach T ("candidate": float(S') >= T*Qi[d] - B - A[d], resp. float(S') >= T/2 + B + A[d]); everything else
//     (99.9 % of the evaluations) is provably worse than an already-seen disparity and is dropped.
//   * T starts from the exact cost at a PREDICTED disparity (half-resolution AbsoluteCost search on k1_fast, doubled): any
//     searched disparity gives a valid lower bound, a good prediction makes candidates rare (2 per pixel).
//   * a candidate raises T (a float lower bound of its own cost, a handful of flops) and appends (pixel, d, S', upper bound)
//     to a per-CTA list in global memory.
//   * at the end of a band (or when the list is half full) the CTA walks the list with all threads: entries whose upper
//     bound is below the final T are dropped, the survivors (typically 1-3 per pixel) are evaluated with the reference's
//     exact arithmetic (int64 numerator, double multiply / sqrt), and an atomicMax on the cost key followed by an atomicMin
//     on the raster index reproduces "first best wins".
// A disparity whose exact cost ties or beats the final best can never be screened out, so the result is bit-identical to
// the reference.  NaN costs (zero-energy windows), list overflow (flat regions: every disparity ties) and the all-equal
// rule are settled by replay / fix-up kernels on the few pixels concerned.
#include "k1_fast_common.cuh"
#include <algorithm>
#include <cmath>

namespace vwb200 {

enum { M_NCC = 0, M_SQ = 1 };
static constexpr int SD_MAX = 3;                 // dy rows per synchronisation period (ring depth): fewer, cheaper barriers
static inline __host__ __device__ int nq_slots(int sd) { return F_TH + 2 * sd - 1; }
static constexpr float QI_ZERO = 1.0e-30f;      // Qi of a zero-energy right window (its cost is NaN)
static constexpr float NCC_E = 64.0f;           // half ulp of float(S'), |S'| < 2^31
static constexpr float NCC_SLACK = 4096.0f;     // > all roundings of f + A - nB (magnitudes < 2^33) + conversion + E
static constexpr float SQ_SLACK = 8192.0f;

static size_t screen_smem_bytes(const FastGeom& g, int mode) {
  return (size_t)F_TH * F_COLS * 4                                                   // T
         + (size_t)g.ltile_rows * F_COLS * 2 + (size_t)g.ring_slots * g.rw * 2      // left tile, right ring (int16)
         + (mode == M_NCC ? 2 : 1) * (size_t)nq_slots(g.sd) * g.rw * 4 + 128;       // A ring (+ Qi ring)
}
// ring of right rows: a period of sd dy rows needs ltile_rows + sd - 1 rows resident while the next period's sd rows
// arrive; the deepest ring that fits in shared memory is used
static bool screen_geom(FastGeom& g, int mode) {
  const int rrows0 = g.rrows;
  for (int sd = SD_MAX; sd >= 1; --sd) {
    g.sd = sd; g.ring_slots = g.ltile_rows + 2 * sd - 1; g.rrows = rrows0 + SD_MAX;
    if (screen_smem_bytes(g, mode) <= 227 * 1024) return true;
  }
  return false;
}

static bool screen_params(int mode, int kx, int ky, float vmin, float vmax, int* c_out, double* maxc_out) {
  if (mode == M_NCC && (!(vmin >= 0.0f) || !(vmax <= 4095.0f))) return false;      // l*r < 2^24: exact in the reference's float
  if (mode == M_SQ && !((double)vmax - (double)vmin <= 4095.0)) return false;        // (l-r)^2 < 2^24 likewise
  if (!(fabsf(vmin) < 1.0e6f) || !(fabsf(vmax) < 1.0e6f)) return false;
  const int c = (int)floor(((double)vmin + (double)vmax) * 0.5 + 0.5);
  const double maxc = std::max((double)vmax - c, (double)c - vmin);
  if (maxc > 32767.0 || maxc * maxc * kx * ky >= 2147483647.0) return false;
  *c_out = c; *maxc_out = maxc;
  return true;
}

int k1_screen_supported(int cost, int kx, int ky, int sx, int sy, float vmin, float vmax, bool integer_valued) {
  if (cost != VWB200_CROSS_CORRELATION && cost != VWB200_SQUARED_DIFFERENCE) return VWB200_ENOIMPL;
  if (!integer_valued) return VWB200_ENOIMPL;
  const int mode = cost == VWB200_CROSS_CORRELATION ? M_NCC : M_SQ;
  int c; double maxc;
  if (!screen_params(mode, kx, ky, vmin, vmax, &c, &maxc)) return VWB200_ENOIMPL;
  if (kx < 3 || kx > 31 || ky < 1 || ky > 41) return VWB200_ENOIMPL;
  if (sx < F_B || sx > 512 || sy < 1 || (long long)sx * sy < 64 || (long long)sx * sy > 65536) return VWB200_ENOIMPL;
  FastGeom g = make_geom(256, 32, sx, sy, kx, ky);
  if (!screen_geom(g, mode)) return VWB200_ENOIMPL;
  return VWB200_OK;
}

// ---- workspace carving ---------------------------------------------------------------------------------------
struct ScreenWs {
  int16_t *L16, *R16; float *Qp, *Ap, *Bp;
  double *lp, *rp; int *Sl, *Sr;
  unsigned long long* bk; int* bi;   // per-CTA best key / best raster index [148][32][256]
  uint4* list; int cap;              // per-CTA candidate lists [148][cap]
  unsigned long long* pk; int* pi;   // per-dy-chunk partials (J > 1)
  unsigned char* nanflag;            // W x H: replay this pixel (NaN cost seen, or its candidates overflowed the list)
  Zone* zone;
  // seeding stage: half-resolution AbsoluteCost search -> predicted disparity -> exact cost there -> initial threshold
  float *L2, *R2, *T0; vwb200_dispi* d2; unsigned char* ws2; size_t ws2_bytes;
  int W2, H2, kx2, ky2, sx2, sy2;
  size_t total;
};
static inline size_t al(size_t x) { return (x + 255) & ~(size_t)255; }
static ScreenWs carve(const FastGeom& g, int mode, void* base) {
  ScreenWs w;
  unsigned char* p = static_cast<unsigned char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) { unsigned char* q = p ? p + off : nullptr; off += al(bytes); return q; };
  const size_t ow = (size_t)g.W + g.sx - 1, oh = (size_t)g.H + g.sy - 1;
  const size_t qrows = (size_t)g.NB * F_TH + g.sy + SD_MAX;
  w.L16 = (int16_t*)take((size_t)g.NS * g.lrows * F_COLS * 2);
  w.R16 = (int16_t*)take((size_t)g.NS * g.rrows * g.rw * 2);
  w.Qp = (float*)take(mode == M_NCC ? (size_t)g.NS * qrows * g.rw * 4 : 16);
  w.Ap = (float*)take((size_t)g.NS * qrows * g.rw * 4);
  w.Bp = (float*)take((size_t)g.NS * g.NB * F_TH * F_COLS * 4);
  w.lp = (double*)take(mode == M_NCC ? (size_t)g.W * g.H * 8 : 16);
  w.rp = (double*)take(mode == M_NCC ? ow * oh * 8 : 16);
  w.Sl = (int*)take((size_t)g.W * g.H * 4);
  w.Sr = (int*)take(ow * oh * 4);
  const size_t ncta = (size_t)std::min(148, g.NS * g.NB * g.J);          // persistent CTAs actually launched
  w.bk = (unsigned long long*)take(ncta * F_TH * F_COLS * 8);
  w.bi = (int*)take(ncta * F_TH * F_COLS * 4);
  // list capacity: a flush is forced when a list is half full at a dy boundary; 24 entries per pixel of a band is ~25x the
  // typical total per pixel.  Entries that do not fit mark their pixel for replay (correct, slow).
  w.cap = F_TH * (F_COLS - (g.kx - 1)) * 24;
  w.list = (uint4*)take(ncta * w.cap * 16);
  w.pk = (unsigned long long*)take(g.J > 1 ? (size_t)g.J * g.W * g.H * 8 : 16);
  w.pi = (int*)take(g.J > 1 ? (size_t)g.J * g.W * g.H * 4 : 16);
  w.nanflag = take((size_t)g.W * g.H);
  w.zone = (Zone*)take(sizeof(Zone));
  w.W2 = (g.W + 1) / 2; w.H2 = (g.H + 1) / 2;
  w.kx2 = std::max(3, (g.kx / 2) | 1); w.ky2 = std::max(1, (g.ky / 2) | 1);
  w.sx2 = (((g.sx + 1) / 2 + 7) / 8) * 8; w.sy2 = (g.sy + 1) / 2;
  w.L2 = (float*)take((size_t)(w.W2 + w.kx2 - 1) * (w.H2 + w.ky2 - 1) * 4);
  w.R2 = (float*)take((size_t)(w.W2 + w.kx2 - 1 + w.sx2 - 1) * (w.H2 + w.ky2 - 1 + w.sy2 - 1) * 4);
  w.d2 = (vwb200_dispi*)take((size_t)w.W2 * w.H2 * sizeof(vwb200_dispi));
  w.T0 = (float*)take((size_t)g.W * g.H * 4);
  w.ws2_bytes = k1_fast_workspace_bytes(w.W2, w.H2, w.sx2, w.sy2, w.kx2, w.ky2);
  w.ws2 = take(w.ws2_bytes);
  w.total = off;
  return w;
}
size_t k1_screen_workspace_bytes(int cost, int W, int H, int sx, int sy, int kx, int ky) {
  FastGeom g = make_geom(W, H, sx, sy, kx, ky);
  screen_geom(g, cost == VWB200_CROSS_CORRELATION ? M_NCC : M_SQ);
  return carve(g, cost == VWB200_CROSS_CORRELATION ? M_NCC : M_SQ, nullptr).total + 256;
}

__global__ void screen_set_zone_kernel(Zone* dst, Zone z) { *dst = z; }
// constant edge extension (Image/EdgeExtension.tcc:47-59): zones of the level loop may reach outside the rasters
__device__ __forceinline__ float ld_edge(const ImgF& im, int x, int y) {
  x = max(0, min(x, im.w - 1)); y = max(0, min(y, im.h - 1));
  return __ldg(im.p + (ptrdiff_t)y * im.pitch + x);
}

// ---- pack kernels ---------------------------------------------------------------------------------------------
__global__ void screen_pack_img_kernel(ImgF img, int c, FastGeom g, int right, int16_t* __restrict__ out) {
  const int row = blockIdx.x, strip = blockIdx.y;
  const int s0 = strip * g.out_cols;
  const int rowlen = right ? g.rw : F_COLS, nrows = right ? g.rrows : g.lrows;
  const int lw = g.W + g.kx - 1 + (right ? g.sx - 1 : 0), lh = g.H + g.ky - 1 + (right ? g.sy - 1 : 0);
  int16_t* o = out + ((size_t)strip * nrows + row) * rowlen;
  for (int col = threadIdx.x; col < rowlen; col += blockDim.x) {
    const int gx = s0 + col;
    int16_t v = 0;
    if (row < lh && gx < lw) v = (int16_t)((int)ld_edge(img, (right ? g.rox : g.lox) + gx, (right ? g.roy : g.loy) + row) - c);
    o[col] = v;
  }
}
// per right window origin.  NCC: Qi <= 1/sqrt(rp) (QI_ZERO for a zero-energy window), A >= c*Sr.  SQ: A <= SR2/2.
template <int MODE>
__global__ void screen_pack_qa_kernel(const double* __restrict__ rp, const int* __restrict__ Sr, int c, FastGeom g, int qrows,
                                      float* __restrict__ Qp, float* __restrict__ Ap) {
  const int row = blockIdx.x, strip = blockIdx.y;
  const int s0 = strip * g.out_cols;
  const int ow = g.W + g.sx - 1, oh = g.H + g.sy - 1;
  for (int col = threadIdx.x; col < g.rw; col += blockDim.x) {
    const int gx = s0 + col;
    const bool in = row < oh && gx < ow;
    const size_t k = ((size_t)strip * qrows + row) * g.rw + col;
    if (MODE == M_NCC) {
      float qi = 1.0f, av = 0.0f;
      if (in) {
        const double r = rp[(size_t)row * ow + gx];
        if (isinf(r)) qi = QI_ZERO;
        else qi = __fmul_rd(__double2float_rd(1.0 / sqrt(r)), 0.9999997f);
        av = __double2float_ru((double)c * (double)Sr[(size_t)row * ow + gx]);
      }
      Qp[k] = qi; Ap[k] = av;
    } else {
      Ap[k] = in ? __double2float_rd(0.5 * (double)Sr[(size_t)row * ow + gx]) : 0.0f;
    }
  }
}
// per left pixel.  NCC: nB <= -(c*Sl - N c^2) - E, +inf for a zero-energy left window.  SQ: nB <= (SL2 - M0)/2 - E.
template <int MODE>
__global__ void screen_pack_b_kernel(const int* __restrict__ Sl, int c, double K, FastGeom g, float* __restrict__ Bp) {
  const int row = blockIdx.x, strip = blockIdx.y;
  const int s0 = strip * g.out_cols;
  float* b = Bp + ((size_t)strip * g.NB * F_TH + row) * F_COLS;
  for (int col = threadIdx.x; col < F_COLS; col += blockDim.x) {
    const int gx = s0 + col;
    float v = 0.0f;
    if (row < g.H && gx < g.W && col < g.out_cols) {
      const int s = Sl[(size_t)row * g.W + gx];
      if (MODE == M_NCC) v = s == 0 ? INFINITY : __double2float_rd(-((double)c * (double)s - K) - (double)NCC_E);      // K = N c^2
      else v = __double2float_rd(0.5 * ((double)s - K) - (double)NCC_E);                                                // K = M0
    }
    b[col] = v;
  }
}

// ---- seeding stage ---------------------------------------------------------------------------------------------
// every second pixel of every second row (clamped at the edges): integer imagery stays integer
__global__ void screen_subsample2_kernel(ImgF in, int ox, int oy, int ow, int oh, float* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= ow || y >= oh) return;
  out[(size_t)y * ow + x] = ld_edge(in, ox + 2 * x, oy + 2 * y);
}
// T0(pixel) = float lower bound of the exact cost key at d0 = 2 * (half-resolution arg-best): any searched disparity gives
// a valid lower bound of the best cost, a good prediction makes it a tight one (the hot loop then drops everything
// outside the immediate neighbourhood of the peak without creating candidates).
template <int MODE>
__global__ void screen_seed_kernel(ImgF L, ImgF R, const vwb200_dispi* __restrict__ d2, int W2, FastGeom g, int c, long long K,
                                   const int* __restrict__ Sl, const int* __restrict__ Sr, const double* __restrict__ rp,
                                   float* __restrict__ T0) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= g.W || y >= g.H) return;
  const vwb200_dispi q = d2[(size_t)(y >> 1) * W2 + (x >> 1)];
  const int dx = min(2 * q.dx, g.sx - 1), dy = min(2 * q.dy, g.sy - 1);
  int s = 0;
  for (int j = 0; j < g.ky; ++j)
    for (int i = 0; i < g.kx; ++i)
      s += ((int)ld_edge(L, g.lox + x + i, g.loy + y + j) - c) * ((int)ld_edge(R, g.rox + x + i + dx, g.roy + y + j + dy) - c);
  const int ow = g.W + g.sx - 1;
  const size_t kl = (size_t)y * g.W + x, kr = (size_t)(y + dy) * ow + (x + dx);
  float t = 0.0f;
  if (MODE == M_NCC) {
    const double r = rp[kr];
    if (!isinf(r)) {
      const long long slr = (long long)s + (long long)c * ((long long)Sl[kl] + (long long)Sr[kr]) - K;
      t = __double2float_rd((double)slr * sqrt(r) * (1.0 - 1.0e-6));
    }
  } else {
    const long long cost = (long long)Sl[kl] + (long long)Sr[kr] - 2ll * (long long)s;
    t = __double2float_rd((double)(K - cost) * (1.0 - 1.0e-6) - 1.0);
  }
  T0[kl] = t > 0.0f ? t : 0.0f;
}

// ---- device helpers -----------------------------------------------------------------------------------------
// prmt with sign replication (selector nibble 8|k = msb of byte k in all 8 bits); __byte_perm() only honours 3 selector bits
__device__ __forceinline__ int prmt_s(uint32_t a, uint32_t sel) {
  int d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(0u), "r"(sel));
  return d;
}
__device__ __forceinline__ void unpack8s(const uint4 v, int (&o)[8]) {      // int16 pairs -> sign-extended int32 (1 PRMT each)
  o[0] = prmt_s(v.x, 0x9910u); o[1] = prmt_s(v.x, 0xBB32u);
  o[2] = prmt_s(v.y, 0x9910u); o[3] = prmt_s(v.y, 0xBB32u);
  o[4] = prmt_s(v.z, 0x9910u); o[5] = prmt_s(v.z, 0xBB32u);
  o[6] = prmt_s(v.w, 0x9910u); o[7] = prmt_s(v.w, 0xBB32u);
}
__device__ __forceinline__ void load_row_s(const int16_t* lrow, const int16_t* rrow, int (&Lv)[8], int (&Rv)[16]) {
  unpack8s(*reinterpret_cast<const uint4*>(lrow), Lv);
  int t[8];
  unpack8s(*reinterpret_cast<const uint4*>(rrow), t);
#pragma unroll
  for (int i = 0; i < 8; ++i) Rv[i] = t[i];
  unpack8s(*reinterpret_cast<const uint4*>(rrow + 8), t);
#pragma unroll
  for (int i = 0; i < 8; ++i) Rv[8 + i] = t[i];
}

struct ScreenCtx {           // what the exact evaluation needs
  const double* lp; const double* rp;       // NCC
  const int* Sl; const int* Sr;             // NCC: box(l), box(r);  SQ: box((l-c)^2), box((r-c)^2)
  unsigned char* nanflag;
  int W, H, ow, c;
  long long K;                              // NCC: N c^2;  SQ: M0 = 4 N maxc^2 (>= any cost)
  const float* T0;                          // initial thresholds (lower bound of the cost at a predicted disparity) or null
};

// shared-memory accesses by 32-bit shared-window address (no generic-pointer arithmetic on the rare path)
__device__ __forceinline__ float lds_volatile_f32(uint32_t a) {
  float v;
  asm volatile("ld.volatile.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void atoms_max_s32(uint32_t a, int v) {
  asm volatile("red.shared.max.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ int atoms_add_s32(uint32_t a, int v) {
  int old;
  asm volatile("atom.shared.add.s32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
  return old;
}
// per-item constants of the rare path, kept in shared memory so that a call only marshals what changes
struct CandCtx { uint4* list; unsigned char* nan_band; int cap; int W; int cnt; int next[2]; int pad; };

// One candidate (lane-divergent, ~0.1 % of the evaluations): raise the pixel's threshold to a float lower bound of this
// disparity's cost and append it to the CTA's list.  key = pix | didx << 13 (pix = y*256 + x inside the band, didx = raster
// index inside the chunk); t_sa = shared address of the pixel's threshold, c_sa = shared address of the CandCtx.
template <int MODE>
__device__ __noinline__ void screen_candidate(uint32_t t_sa, uint32_t c_sa, uint32_t key, int sprime, float f, float A, float nB, float Qi) {
  const float T = lds_volatile_f32(t_sa);
  if (!(T < INFINITY)) return;                          // pixel closed (outside the raster, or marked for replay)
  const CandCtx* cc = reinterpret_cast<const CandCtx*>(__cvta_shared_to_generic(c_sa));
  const int pix = key & 8191;
  float U, L;
  if (MODE == M_NCC) {
    if (Qi <= QI_ZERO) {                                // zero-energy right window: this cost is NaN, the pixel is replayed
      cc->nan_band[(size_t)(pix >> 8) * cc->W + (pix & 255)] = 1;
      atoms_max_s32(t_sa, 0x7f800000);
      return;
    }
    const float t = (f + A) - nB;                       // ~ box(l*r) + E, within NCC_SLACK
    const float q_up = __frcp_ru(Qi), q_lo = __frcp_rd(__fmul_ru(Qi, 1.000001f));
    const float t_up = t + NCC_SLACK, t_lo = t - NCC_SLACK;
    U = t_up > 0.0f ? __fmul_ru(t_up, q_up) : 0.0f;
    L = t_lo > 0.0f ? __fmul_rd(t_lo, q_lo) : 0.0f;
  } else {
    const float k = 2.0f * ((f - A) - (nB + NCC_E));    // ~ M0 - cost, within SQ_SLACK
    U = k + SQ_SLACK;
    L = fmaxf(k - SQ_SLACK, 0.0f);
  }
  atoms_max_s32(t_sa, __float_as_int(L));
  const int slot = atoms_add_s32(c_sa + (uint32_t)offsetof(CandCtx, cnt), 1);
  if (slot < cc->cap) cc->list[slot] = make_uint4(key, (uint32_t)sprime, __float_as_uint(U), 0u);
  else {                                                // list full: replay the pixel instead
    cc->nan_band[(size_t)(pix >> 8) * cc->W + (pix & 255)] = 1;
    atoms_max_s32(t_sa, 0x7f800000);
  }
}

template <int KX, bool FULL, int MODE>
__device__ __forceinline__ void screen_pass(const int16_t* __restrict__ ltile, const int16_t* __restrict__ rring,
                                            const float* __restrict__ qring, const float* __restrict__ aring,
                                            float* __restrict__ thr, const float* __restrict__ b_band, uint32_t c_sa,
                                            int lane, int g, int ky, int ring_slots, int nq, int rw, int ring_base, int qbase,
                                            int row0, int nb, int sx, int dy_rel) {
  int V[8][F_B];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < F_B; ++b) V[a][b] = 0;
  const int16_t* lp = ltile + row0 * F_COLS + 8 * lane;
  const int16_t* rp = rring + 8 * (lane + g);
  int slot_new = ring_base;
  for (int t = 0; t < ky; ++t) {
    int Lv[8], Rv[16];
    load_row_s(lp + t * F_COLS, rp + slot_new * rw, Lv, Rv);
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = 0; b < F_B; ++b) V[a][b] += Lv[a] * Rv[a + b];
    if (++slot_new == ring_slots) slot_new = 0;
  }
  int slot_old = ring_base;
  int qslot = qbase;                       // ring slot of the right window-origin row (dy + row0 + y)
  for (int y = 0; y < F_RH; ++y) {
    if (y > 0) {
      {
        int Lv[8], Rv[16];
        load_row_s(lp + (y + ky - 1) * F_COLS, rp + slot_new * rw, Lv, Rv);
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < F_B; ++b) V[a][b] += Lv[a] * Rv[a + b];
      }
      {
        int Lo[8], Ro[16];
        load_row_s(lp + (y - 1) * F_COLS, rp + slot_old * rw, Lo, Ro);
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < F_B; ++b) V[a][b] -= Lo[a] * Ro[a + b];
      }
      if (++slot_new == ring_slots) slot_new = 0;
      if (++slot_old == ring_slots) slot_old = 0;
    }
    // per-row operands of the screening test
    float Qv[16], Av[16], Bv[8], Tv[8];
    float* trow = thr + (row0 + y) * F_COLS + lane;
    {
      const float4* ap = reinterpret_cast<const float4*>(aring + qslot * rw + 8 * (lane + g));
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 a = ap[i];
        Av[4 * i] = a.x; Av[4 * i + 1] = a.y; Av[4 * i + 2] = a.z; Av[4 * i + 3] = a.w;
      }
      if (MODE == M_NCC) {
        const float4* qp = reinterpret_cast<const float4*>(qring + qslot * rw + 8 * (lane + g));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 q = qp[i];
          Qv[4 * i] = q.x; Qv[4 * i + 1] = q.y; Qv[4 * i + 2] = q.z; Qv[4 * i + 3] = q.w;
        }
      }
      const float4* bp = reinterpret_cast<const float4*>(b_band + (row0 + y) * F_COLS + 8 * lane);
      const float4 b0 = __ldg(bp), b1 = __ldg(bp + 1);
      Bv[0] = b0.x; Bv[1] = b0.y; Bv[2] = b0.z; Bv[3] = b0.w; Bv[4] = b1.x; Bv[5] = b1.y; Bv[6] = b1.z; Bv[7] = b1.w;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float t = trow[r * 32];
        Tv[r] = MODE == M_NCC ? t : __fmaf_rd(0.5f, t, Bv[r]);            // SQ: T/2 + nB
      }
    }
    // hot part: branch-free over the 8 dx of the octet; bit b of `hit` = some pixel of this lane is a candidate at dx b
    uint32_t hit = 0;
#pragma unroll
    for (int b = 0; b < F_B; ++b) {
      if (!FULL && b >= nb) break;
      int p[8], o[8];
      p[0] = V[0][b];
#pragma unroll
      for (int a = 1; a < 8; ++a) p[a] = p[a - 1] + V[a][b];
      window_sums<KX>(p, o);
      bool any = false;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float f = __int2float_rn(o[r]);
        const float rhs = MODE == M_NCC ? __fadd_rd(__fmaf_rd(Tv[r], Qv[r + b], Bv[r]), -Av[r + b])      // T*Qi - B - E - A
                                        : __fadd_rd(Tv[r], Av[r + b]);                                     // T/2 + nB + A
        any |= !(f < rhs);
      }
      if (any) hit |= 1u << b;
    }
    // rare part (warp-uniform branches): recompute the window sums of the flagged dx (V is unchanged) and hand the
    // candidates over.  ~4 % of the (row, dx) pairs get here.
    if (__any_sync(0xffffffffu, hit != 0)) {
      const uint32_t t_sa = smem_u32(trow);
#pragma unroll
      for (int b = 0; b < F_B; ++b) {
        if (!FULL && b >= nb) break;
        if (!__any_sync(0xffffffffu, (hit >> b) & 1u)) continue;
        int p[8], o[8];
        p[0] = V[0][b];
#pragma unroll
        for (int a = 1; a < 8; ++a) p[a] = p[a - 1] + V[a][b];
        window_sums<KX>(p, o);
        if ((hit >> b) & 1u) {
          const uint32_t key0 = (uint32_t)((row0 + y) * F_COLS + 8 * lane) | ((uint32_t)(dy_rel * sx + F_B * g + b) << 13);
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const float f = __int2float_rn(o[r]);
            const float t = lds_volatile_f32(t_sa + 128u * r);
            const float rhs = MODE == M_NCC ? __fadd_rd(__fmaf_rd(t, Qv[r + b], Bv[r]), -Av[r + b])
                                            : __fadd_rd(__fmaf_rd(0.5f, t, Bv[r]), Av[r + b]);
            if (!(f < rhs)) screen_candidate<MODE>(t_sa + 128u * r, c_sa, key0 + r, o[r], f, Av[r + b], Bv[r], MODE == M_NCC ? Qv[r + b] : 1.0f);
          }
        }
      }
    }
    if (++qslot == nq) qslot = 0;
  }
}

// The reference's cost as an order-preserving 64-bit key (larger = better).  NCC: the bits of the (non-negative) double;
// SQ: M0 - cost.  ok = false: the cost is NaN.
template <int MODE>
__device__ __forceinline__ unsigned long long screen_exact_key(const ScreenCtx& cx, int sprime, int gx, int gy, int dx, int dy, bool* ok) {
  const size_t kl = (size_t)gy * cx.W + gx, kr = (size_t)(gy + dy) * cx.ow + (gx + dx);
  *ok = true;
  if (MODE == M_NCC) {
    const long long slr = (long long)sprime + (long long)cx.c * ((long long)cx.Sl[kl] + (long long)cx.Sr[kr]) - cx.K;
    const double s = __dmul_rn((double)slr, sqrt(__dmul_rn(cx.lp[kl], cx.rp[kr])));     // Correlation.cc:82, CostFunctions.h:227-231
    if (s != s) { *ok = false; return 0ull; }
    return (unsigned long long)__double_as_longlong(s);
  }
  const long long cost = (long long)cx.Sl[kl] + (long long)cx.Sr[kr] - 2ll * (long long)sprime;
  return (unsigned long long)(cx.K - cost);
}

// Walk the CTA's candidate list: exact evaluation of the entries that can still be the best, atomicMax on the key, then
// atomicMin on the raster index among the entries that hold the maximum.
template <int MODE>
__device__ __forceinline__ void screen_flush(const ScreenCtx& cx, const float* __restrict__ thr, uint4* __restrict__ list, int n,
                                             unsigned long long* __restrict__ bk, int* __restrict__ bi, int s0, int y0, int dy0,
                                             int sx, int tid) {
  for (int e = tid; e < n; e += F_THREADS) {
    uint4 v = list[e];
    const int pix = v.x & 8191, didx = v.x >> 13;
    const int y = pix >> 8, x = pix & 255;
    const int toff = y * F_COLS + (x & 7) * 32 + (x >> 3);
    const float T = thr[toff];
    bool alive = T < INFINITY && !(__uint_as_float(v.z) < T);
    if (alive) {
      bool ok;
      const unsigned long long key = screen_exact_key<MODE>(cx, (int)v.y, s0 + x, y0 + y, didx % sx, dy0 + didx / sx, &ok);
      if (!ok) { cx.nanflag[(size_t)(y0 + y) * cx.W + s0 + x] = 1; alive = false; }
      else {
        const unsigned long long old = atomicMax(bk + pix, key);
        if (key > old) bi[pix] = 0x7fffffff;
        v.z = (uint32_t)key; v.w = (uint32_t)(key >> 32);
      }
    }
    if (!alive) v.x = 0xffffffffu;
    list[e] = v;
  }
  __syncthreads();
  for (int e = tid; e < n; e += F_THREADS) {
    const uint4 v = list[e];
    if (v.x == 0xffffffffu) continue;
    const int pix = v.x & 8191;
    const unsigned long long key = (unsigned long long)v.z | ((unsigned long long)v.w << 32);
    if (key == bk[pix]) atomicMin(bi + pix, (int)(v.x >> 13));
  }
  __syncthreads();
}

template <int KX, int MODE>
__global__ void __launch_bounds__(F_THREADS, 1)
k1_screen_kernel(const int16_t* __restrict__ L16, const int16_t* __restrict__ R16, const float* __restrict__ Qp,
                 const float* __restrict__ Ap, const float* __restrict__ Bp, FastGeom G, int qrows, ScreenCtx cx,
                 unsigned long long* __restrict__ bk_all, int* __restrict__ bi_all, uint4* __restrict__ list_all, int cap,
                 vwb200_dispi* __restrict__ out, ptrdiff_t opitch, unsigned long long* __restrict__ part_key, int* __restrict__ part_idx) {
  extern __shared__ __align__(128) unsigned char smem[];
  float* thr = reinterpret_cast<float*>(smem);                                              // [32][8][32]
  int16_t* ltile = reinterpret_cast<int16_t*>(smem + (size_t)F_TH * F_COLS * 4);
  int16_t* rring = ltile + (size_t)G.ltile_rows * F_COLS;
  float* aring = reinterpret_cast<float*>(rring + (size_t)G.ring_slots * G.rw);
  const int SD = G.sd, NQ_SLOTS = nq_slots(G.sd);
  float* qring = aring + (size_t)NQ_SLOTS * G.rw;                                           // NCC only
  uint64_t* bars = reinterpret_cast<uint64_t*>(aring + (size_t)(MODE == M_NCC ? 2 : 1) * NQ_SLOTS * G.rw);
  CandCtx* cc = reinterpret_cast<CandCtx*>(bars + 2);
  const uint32_t c_sa = smem_u32(cc);
  const int tid = threadIdx.x, lane = tid & 31;
  const int ngroups = (G.sx + F_B - 1) / F_B, nunits = ngroups * F_HALVES;
  unsigned long long* bk = bk_all + (size_t)blockIdx.x * F_TH * F_COLS;
  int* bi = bi_all + (size_t)blockIdx.x * F_TH * F_COLS;
  uint4* list = list_all + (size_t)blockIdx.x * cap;
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  __syncthreads();
  uint32_t ph0 = 0, ph1 = 0;
  constexpr uint32_t NRINGS = MODE == M_NCC ? 2u : 1u;
  const uint32_t lbytes = (uint32_t)G.ltile_rows * F_COLS * 2, rrow_bytes = (uint32_t)G.rw * 2, qrow_bytes = (uint32_t)G.rw * 4;
  for (int item = blockIdx.x; item < G.NS * G.NB * G.J; item += gridDim.x) {
    const int chunk = item % G.J, rest = item / G.J;
    const int strip = rest % G.NS, band = rest / G.NS;
    const int y0 = band * F_TH, s0 = strip * G.out_cols;
    const int dy0 = chunk * G.dy_per, ndy = min(G.sy, dy0 + G.dy_per) - dy0;
    const int16_t* lsrc = L16 + ((size_t)strip * G.lrows + y0) * F_COLS;
    const int16_t* rsrc = R16 + ((size_t)strip * G.rrows + y0 + dy0) * G.rw;
    const float* qsrc = Qp + ((size_t)strip * qrows + y0 + dy0) * G.rw;
    const float* asrc = Ap + ((size_t)strip * qrows + y0 + dy0) * G.rw;
    const float* b_band = Bp + ((size_t)strip * G.NB * F_TH + y0) * F_COLS;
    unsigned char* nan_band = cx.nanflag + (size_t)y0 * G.W + s0;
    if (tid == 0) {
      fence_proxy_async();
      // first period: right rows 0 .. ltile_rows + SD - 2 and window-origin rows 0 .. F_TH + SD - 2 (slot = row)
      mbar_expect_tx(&bars[0], lbytes + (uint32_t)(G.ltile_rows + SD - 1) * rrow_bytes + NRINGS * (F_TH + SD - 1) * qrow_bytes);
      tma_load_1d(ltile, lsrc, lbytes, &bars[0]);
      tma_load_1d(rring, rsrc, (uint32_t)(G.ltile_rows + SD - 1) * rrow_bytes, &bars[0]);
      tma_load_1d(aring, asrc, (uint32_t)(F_TH + SD - 1) * qrow_bytes, &bars[0]);
      if (MODE == M_NCC) tma_load_1d(qring, qsrc, (uint32_t)(F_TH + SD - 1) * qrow_bytes, &bars[0]);
      cc->list = list; cc->nan_band = nan_band; cc->cap = cap; cc->W = G.W; cc->cnt = 0; cc->next[0] = 0; cc->next[1] = 0;
    }
    // thresholds: 0 for live pixels (every cost key is >= 0), +inf for closed ones (outside the raster / strip; NCC:
    // zero-energy left window = every cost NaN -> replay)
    for (int k = tid; k < F_TH * F_COLS; k += F_THREADS) {
      const int y = k / F_COLS, r = (k % F_COLS) / 32, l = k % 32;
      const int x = 8 * l + r;
      float t = INFINITY;
      if (x < G.out_cols && s0 + x < G.W && y0 + y < G.H) {
        t = cx.T0 ? cx.T0[(size_t)(y0 + y) * G.W + s0 + x] : 0.0f;
        if (MODE == M_NCC && b_band[y * F_COLS + x] == INFINITY) { t = INFINITY; nan_band[(size_t)y * G.W + x] = 1; }
      }
      thr[k] = t;
      bk[k] = 0ull; bi[k] = 0x7fffffff;
    }
    __syncthreads();
    mbar_wait(&bars[0], ph0); ph0 ^= 1;
    for (int dyp = 0, per = 0; dyp < ndy; dyp += SD, ++per) {
      const int dcur = min(SD, ndy - dyp);                 // dy rows of this period
      const int nnext = min(SD, ndy - dyp - dcur);         // dy rows of the next one: their last rows are fetched now
      if (tid == 0) {
        cc->next[(per + 1) & 1] = 0;
        if (nnext > 0) {
          fence_proxy_async();
          mbar_expect_tx(&bars[1], (uint32_t)nnext * (rrow_bytes + NRINGS * qrow_bytes));
          for (int j = 0; j < nnext; ++j) {
            const int rr = dyp + SD - 1 + G.ltile_rows + j, qr = dyp + SD - 1 + F_TH + j;
            tma_load_1d(rring + (size_t)(rr % G.ring_slots) * G.rw, rsrc + (size_t)rr * G.rw, rrow_bytes, &bars[1]);
            tma_load_1d(aring + (size_t)(qr % NQ_SLOTS) * G.rw, asrc + (size_t)qr * G.rw, qrow_bytes, &bars[1]);
            if (MODE == M_NCC) tma_load_1d(qring + (size_t)(qr % NQ_SLOTS) * G.rw, qsrc + (size_t)qr * G.rw, qrow_bytes, &bars[1]);
          }
        }
      }
      // work units of this period = (dy, dx octet, row half); warps draw them from a shared counter: unit durations
      // differ (candidate handling around the cost peak), a static split leaves warps waiting at the barrier
      for (;;) {
        int u = 0;
        if (lane == 0) u = atoms_add_s32(c_sa + (uint32_t)offsetof(CandCtx, next) + 4u * (per & 1), 1);
        u = __shfl_sync(0xffffffffu, u, 0);
        if (u >= nunits * dcur) break;
        const int dy = dyp + u / nunits, uu2 = u % nunits;
        const int g = uu2 % ngroups, row0 = (uu2 / ngroups) * F_RH;
        const int ring_base = (dy + row0) % G.ring_slots;
        const int qbase = (dy + row0) % NQ_SLOTS;
        if (G.sx - F_B * g >= F_B)
          screen_pass<KX, true, MODE>(ltile, rring, qring, aring, thr, b_band, c_sa, lane, g, G.ky, G.ring_slots, NQ_SLOTS, G.rw, ring_base, qbase, row0,
                                      F_B, G.sx, dy);
        else
          screen_pass<KX, false, MODE>(ltile, rring, qring, aring, thr, b_band, c_sa, lane, g, G.ky, G.ring_slots, NQ_SLOTS, G.rw, ring_base, qbase, row0,
                                       G.sx - F_B * g, G.sx, dy);
      }
      if (nnext > 0) { mbar_wait(&bars[1], ph1); ph1 ^= 1; }
      __syncthreads();
      const int n = min(*reinterpret_cast<volatile int*>(&cc->cnt), cap);
      if (n > cap / 2 || (dyp + dcur == ndy && n > 0)) {        // uniform across the CTA
        __syncthreads();
        if (tid == 0) cc->cnt = 0;
        screen_flush<MODE>(cx, thr, list, n, bk, bi, s0, y0, dy0, G.sx, tid);
      }
    }
    // ---- results of this band (x chunk) ----
    for (int pix = tid; pix < F_TH * G.out_cols; pix += F_THREADS) {
      const int x = pix % G.out_cols, y = pix / G.out_cols;
      const int gx = s0 + x, gy = y0 + y;
      if (gx >= G.W || gy >= G.H) continue;
      const int k = y * F_COLS + x;
      const unsigned long long key = bk[k];
      int bidx = bi[k];
      if (G.J > 1) {
        const size_t pk = ((size_t)chunk * G.H + gy) * G.W + gx;
        part_key[pk] = key; part_idx[pk] = bidx == 0x7fffffff ? 0x7fffffff : bidx + dy0 * G.sx;
        continue;
      }
      if (bidx == 0x7fffffff) bidx = 0;
      vwb200_dispi o;
      o.dx = bidx % G.sx + G.addx; o.dy = bidx / G.sx + G.addy;
      o.valid = cx.nanflag[(size_t)gy * G.W + gx] ? 2 : 1;
      out[(ptrdiff_t)gy * opitch + gx] = o;
    }
    __syncthreads();
  }
}

__global__ void k1_screen_merge_kernel(FastGeom G, const unsigned long long* __restrict__ pk, const int* __restrict__ pi,
                                       const unsigned char* __restrict__ nanflag, vwb200_dispi* __restrict__ out, ptrdiff_t opitch) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= G.W || y >= G.H) return;
  const size_t plane = (size_t)G.W * G.H, k = (size_t)y * G.W + x;
  unsigned long long best = pk[k];
  int bidx = pi[k];
  for (int c = 1; c < G.J; ++c) {
    const unsigned long long cc = pk[c * plane + k];
    const int ci = pi[c * plane + k];
    if (ci != 0x7fffffff && (bidx == 0x7fffffff || cc > best || (cc == best && ci < bidx))) { best = cc; bidx = ci; }
  }
  if (bidx == 0x7fffffff) bidx = 0;
  vwb200_dispi o;
  o.dx = bidx % G.sx + G.addx; o.dy = bidx / G.sx + G.addy;
  o.valid = nanflag[k] ? 2 : 1;
  out[(ptrdiff_t)y * opitch + x] = o;
}

// "every disparity gave the same cost" for pixels whose arg-best is (0,0): exact costs by direct summation, early exit
template <int MODE>
__global__ void k1_screen_allequal_fixup(ImgF L, ImgF R, FastGeom g, const double* __restrict__ lp, const double* __restrict__ rp,
                                         vwb200_dispi* __restrict__ out, ptrdiff_t opitch) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= g.W || y >= g.H) return;
  vwb200_dispi* o = out + (ptrdiff_t)y * opitch + x;
  if (o->valid != 1 || o->dx != g.addx || o->dy != g.addy) return;
  const int ow = g.W + g.sx - 1;
  auto cost = [&](int dx, int dy) -> unsigned long long {
    long long s = 0;
    for (int j = 0; j < g.ky; ++j)
      for (int i = 0; i < g.kx; ++i) {
        const long long a = (long long)ld_edge(L, g.lox + x + i, g.loy + y + j), b = (long long)ld_edge(R, g.rox + x + i + dx, g.roy + y + j + dy);
        s += MODE == M_NCC ? a * b : (a - b) * (a - b);
      }
    if (MODE == M_NCC)
      return (unsigned long long)__double_as_longlong(__dmul_rn((double)s, sqrt(__dmul_rn(lp[(size_t)y * g.W + x], rp[(size_t)(y + dy) * ow + (x + dx)]))));
    return (unsigned long long)s;
  };
  const unsigned long long c0 = cost(0, 0);
  for (int dy = 0; dy < g.sy; ++dy)
    for (int dx = 0; dx < g.sx; ++dx) {
      if (dx == 0 && dy == 0) continue;
      if (cost(dx, dy) != c0) return;
    }
  o->valid = 0;
}

template <int MODE>
static int screen_launch_t(ImgF left, ImgF right, int W, int H, int sx, int sy, int kx, int ky, float vmin, float vmax,
                           vwb200_dispi* out, ptrdiff_t opitch, void* workspace, cudaStream_t st, const KEvents* ev, const FastOrigin* org) {
  FastGeom g = make_geom(W, H, sx, sy, kx, ky);
  if (!screen_geom(g, MODE)) { set_error("k1_screen: search width %d does not fit in shared memory", sx); return VWB200_ENOIMPL; }
  g.scale = 1;
  if (org) { g.lox = org->lox; g.loy = org->loy; g.rox = org->rox; g.roy = org->roy; g.addx = org->addx; g.addy = org->addy; }
  int c; double maxc;
  if (!screen_params(MODE, kx, ky, vmin, vmax, &c, &maxc)) { set_error("k1_screen: unsupported value range"); return VWB200_ENOIMPL; }
  const ScreenWs ws = carve(g, MODE, workspace);
  const int N = kx * ky;
  const int ow = W + sx - 1, oh = H + sy - 1;
  const int qrows = g.NB * F_TH + sy + SD_MAX;
  const long long K = MODE == M_NCC ? (long long)N * c * c : 4ll * N * (long long)maxc * (long long)maxc;
  // exact maps (reference definitions), then the packed hot-loop operands
  if (MODE == M_NCC) {
    VWB_TRY(box_sq_inv_launch(left, kx, ky, g.lox, g.loy, W, H, ws.lp, st));
    VWB_TRY(box_sq_inv_launch(right, kx, ky, g.rox, g.roy, ow, oh, ws.rp, st));
    VWB_TRY(box_sum_i32_launch(left, kx, ky, g.lox, g.loy, W, H, ws.Sl, st));
    VWB_TRY(box_sum_i32_launch(right, kx, ky, g.rox, g.roy, ow, oh, ws.Sr, st));
  } else {
    VWB_TRY(box_sum_i32_launch(left, kx, ky, g.lox, g.loy, W, H, ws.Sl, st, 1, (float)c));
    VWB_TRY(box_sum_i32_launch(right, kx, ky, g.rox, g.roy, ow, oh, ws.Sr, st, 1, (float)c));
  }
  VWB_CUDA(cudaMemsetAsync(ws.nanflag, 0, (size_t)W * H, st));
  {
    dim3 gl(g.lrows, g.NS), gr(g.rrows, g.NS), gq(qrows, g.NS), gb(g.NB * F_TH, g.NS);
    screen_pack_img_kernel<<<gl, 256, 0, st>>>(left, c, g, 0, ws.L16);
    VWB_LAUNCH_CHECK();
    screen_pack_img_kernel<<<gr, 256, 0, st>>>(right, c, g, 1, ws.R16);
    VWB_LAUNCH_CHECK();
    screen_pack_qa_kernel<MODE><<<gq, 256, 0, st>>>(ws.rp, ws.Sr, c, g, qrows, ws.Qp, ws.Ap);
    VWB_LAUNCH_CHECK();
    screen_pack_b_kernel<MODE><<<gb, 256, 0, st>>>(ws.Sl, c, (double)K, g, ws.Bp);
    VWB_LAUNCH_CHECK();
  }
  // seeding stage (skipped when the half-resolution problem is outside what k1_fast handles)
  const float* T0 = nullptr;
  if (W >= 64 && H >= 64 && k1_fast_supported(VWB200_ABSOLUTE_DIFFERENCE, ws.kx2, ws.ky2, ws.sx2, ws.sy2, vmin, vmax, true) == VWB200_OK) {
    const int lw2 = ws.W2 + ws.kx2 - 1, lh2 = ws.H2 + ws.ky2 - 1, rw2 = lw2 + ws.sx2 - 1, rh2 = lh2 + ws.sy2 - 1;
    dim3 b2(32, 8);
    screen_subsample2_kernel<<<dim3((lw2 + 31) / 32, (lh2 + 7) / 8), b2, 0, st>>>(left, g.lox, g.loy, lw2, lh2, ws.L2);
    VWB_LAUNCH_CHECK();
    screen_subsample2_kernel<<<dim3((rw2 + 31) / 32, (rh2 + 7) / 8), b2, 0, st>>>(right, g.rox, g.roy, rw2, rh2, ws.R2);
    VWB_LAUNCH_CHECK();
    VWB_TRY(k1_fast_launch(VWB200_ABSOLUTE_DIFFERENCE, ImgF{ws.L2, lw2, lh2, lw2}, ImgF{ws.R2, rw2, rh2, rw2}, ws.W2, ws.H2, ws.sx2, ws.sy2,
                           ws.kx2, ws.ky2, vmin, ws.d2, ws.W2, ws.ws2, ws.ws2_bytes, st));
    screen_seed_kernel<MODE><<<dim3((W + 31) / 32, (H + 7) / 8), b2, 0, st>>>(left, right, ws.d2, ws.W2, g, c, K, ws.Sl, ws.Sr, ws.rp, ws.T0);
    VWB_LAUNCH_CHECK();
    T0 = ws.T0;
  }
  ScreenCtx cx{ws.lp, ws.rp, ws.Sl, ws.Sr, ws.nanflag, W, H, ow, c, K, T0};
  int dev = 0, nsm = 148;
  VWB_CUDA(cudaGetDevice(&dev));
  VWB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
  if (nsm > 148) nsm = 148;
  const int items = g.NS * g.NB * g.J;
  const int grid = items < nsm ? items : nsm;
  const size_t smem = screen_smem_bytes(g, MODE);
  void (*kern)(const int16_t*, const int16_t*, const float*, const float*, const float*, FastGeom, int, ScreenCtx, unsigned long long*, int*,
               uint4*, int, vwb200_dispi*, ptrdiff_t, unsigned long long*, int*) = nullptr;
  switch (kx) {
#define KCASE(K) case K: kern = k1_screen_kernel<K, MODE>; break;
    KCASE(3) KCASE(5) KCASE(7) KCASE(9) KCASE(11) KCASE(13) KCASE(15) KCASE(17) KCASE(19) KCASE(21) KCASE(23) KCASE(25)
    KCASE(27) KCASE(29) KCASE(31)
#undef KCASE
    default: set_error("k1_screen: unsupported kernel width %d", kx); return VWB200_ENOIMPL;
  }
  VWB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));   // per-function state shared by all host threads: device maximum
  if (ev && ev->e0) cudaEventRecord(ev->e0, st);
  kern<<<grid, F_THREADS, smem, st>>>(ws.L16, ws.R16, ws.Qp, ws.Ap, ws.Bp, g, qrows, cx, ws.bk, ws.bi, ws.list, ws.cap, out, opitch, ws.pk, ws.pi);
  VWB_LAUNCH_CHECK();
  if (ev && ev->e1) cudaEventRecord(ev->e1, st);
  dim3 b(32, 8), gg((W + 31) / 32, (H + 7) / 8);
  if (g.J > 1) {
    k1_screen_merge_kernel<<<gg, b, 0, st>>>(g, ws.pk, ws.pi, ws.nanflag, out, opitch);
    VWB_LAUNCH_CHECK();
  }
  k1_screen_allequal_fixup<MODE><<<gg, b, 0, st>>>(left, right, g, ws.lp, ws.rp, out, opitch);
  VWB_LAUNCH_CHECK();
  // pixels marked for replay (valid == 2): the reference's sequential best/worst state machine
  {
    Zone z{};
    z.obase = 0; z.opitch = (int)opitch; z.w = W; z.h = H; z.lx = g.lox; z.ly = g.loy; z.rx = g.rox; z.ry = g.roy; z.sx = sx; z.sy = sy;
    z.addx = g.addx; z.addy = g.addy; z.nchunks = 1; z.sbase = 0;
    screen_set_zone_kernel<<<1, 1, 0, st>>>(ws.zone, z);
    VWB_LAUNCH_CHECK();
    NccMaps maps{ws.lp, g.lox, g.loy, W, H, ws.rp, g.rox, g.roy, ow, oh};
    const long long px = (long long)W * H;
    const int gridx = (int)std::min<long long>((px + 127) / 128, 148 * 16);
    VWB_TRY(k1_nan_fixup_launch(MODE == M_NCC ? VWB200_CROSS_CORRELATION : VWB200_SQUARED_DIFFERENCE, left, right, ws.zone, 1, kx, ky, maps, out,
                                st, gridx));
  }
  return VWB200_OK;
}

int k1_screen_launch(int cost, ImgF left, ImgF right, int W, int H, int sx, int sy, int kx, int ky, float vmin, float vmax,
                     vwb200_dispi* out, ptrdiff_t opitch, void* workspace, cudaStream_t st, const KEvents* ev, const FastOrigin* org) {
  if (cost == VWB200_CROSS_CORRELATION) return screen_launch_t<M_NCC>(left, right, W, H, sx, sy, kx, ky, vmin, vmax, out, opitch, workspace, st, ev, org);
  if (cost == VWB200_SQUARED_DIFFERENCE) return screen_launch_t<M_SQ>(left, right, W, H, sx, sy, kx, ky, vmin, vmax, out, opitch, workspace, st, ev, org);
  set_error("k1_screen: cost type %d not handled", cost);
  return VWB200_ENOIMPL;
}

}  // namespace vwb200
