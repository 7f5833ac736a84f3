// k1_fast_common.cuh -- pieces shared by the exact-integer fast kernels (k1_fast.cu: AbsoluteCost / SquaredCost,
// k1_fast_ncc.cu: NCC): tile geometry, mbarrier + TMA bulk-copy PTX wrappers, shuffle-based window sums.
#pragma once
#include "common.cuh"

namespace vwb200 {

static constexpr int F_TH = 32;        // output rows per band
static constexpr int F_COLS = 256;     // padded columns per strip (32 lanes x 8)
static constexpr int F_WARPS = 8;       // 4 dx subsets x 2 row halves (2 warps per SM sub-partition)
static constexpr int F_SUBSETS = 4;
static constexpr int F_HALVES = F_WARPS / F_SUBSETS;
static constexpr int F_RH = F_TH / F_HALVES;      // output rows per warp
static constexpr int F_THREADS = F_WARPS * 32;
static constexpr int F_B = 8;          // consecutive dx per thread (one "octet"); keys are cost*8 + b
static constexpr uint32_t S_INIT = 0x7ffffff8u;

// ---- geometry -----------------------------------------------------------------------------------------
struct FastGeom {
  int W, H, sx, sy, kx, ky;
  int out_cols;      // output columns per strip = 256 - (kx-1)
  int NS, NB;        // strips, bands
  int lrows, rrows;  // padded row counts of the packed arrays
  int ltile_rows;    // F_TH + ky - 1
  int ring_slots;    // F_TH + ky
  int rw;            // u16 per packed right row = 256 + sx (multiple of 8)
  int scale;                // values are packed as (v - vmin) * scale: 8 for AbsoluteCost (keys = cost*8+b), 1 for SquaredCost
  int J, dy_per;            // the dy range is split into J chunks of dy_per rows (more, smaller work items for small rasters)
  int lox, loy, rox, roy;   // origin of the (logical) left / right rasters inside the images passed to the pack kernels
  int addx, addy;           // constant added to the output disparities
  int sd;                   // k1_screen: dy rows per synchronisation period (ring depth)
};
static inline FastGeom make_geom(int W, int H, int sx, int sy, int kx, int ky) {
  FastGeom g;
  g.W = W; g.H = H; g.sx = sx; g.sy = sy; g.kx = kx; g.ky = ky;
  g.out_cols = F_COLS - (kx - 1);
  g.NS = (W + g.out_cols - 1) / g.out_cols;
  g.NB = (H + F_TH - 1) / F_TH;
  g.ltile_rows = F_TH + ky - 1;
  g.ring_slots = F_TH + ky;
  g.lrows = g.NB * F_TH + ky - 1;
  g.rrows = g.NB * F_TH + ky - 1 + sy;
  g.rw = ((F_COLS + sx + 7) / 8) * 8 + 8;
  g.lox = g.loy = g.rox = g.roy = 0; g.addx = g.addy = 0; g.scale = F_B; g.sd = 1;
  // The work items (strip x band x dy-chunk) are dealt round-robin to 148 persistent CTAs, so the last partial wave idles
  // part of the chip: 1120 items = 7.57 waves run as 8 (efficiency 0.946 -- the 8-GPU share of the 8192^2 raster).  Split
  // the dy range into J chunks (merged by k1_fast_merge) so that items * J fills its last wave: pick the J with the best
  // wave efficiency, charging each extra chunk the measured ~0.4 % for its partial planes and the merge pass.  Small
  // rasters additionally want >= ~6 waves for balance.
  g.J = 1;
  const int items = g.NS * g.NB;
  const int jmax = sy / 8 < 1 ? 1 : (sy / 8 > 8 ? 8 : sy / 8);
  if (items < 64 * 148) {
    double best = -1.0;
    for (int J = 1; J <= jmax; ++J) {
      const double w = (double)items * J / 148.0;
      const long long full = (long long)((items * (long long)J + 147) / 148);
      double eff = w / (double)full * (1.0 - 0.004 * (J - 1));
      if (w < 6.0) eff *= 0.5 + w / 12.0;          // few waves: uneven items (edge strips / bands) are not averaged out
      if (eff > best + 1e-9) { best = eff; g.J = J; }
    }
  }
  g.dy_per = (sy + g.J - 1) / g.J;
  g.J = (sy + g.dy_per - 1) / g.dy_per;
  return g;
}
static inline size_t fast_smem_bytes(const FastGeom& g) {
  return (size_t)F_SUBSETS * F_TH * F_COLS * 4 + (size_t)g.ltile_rows * F_COLS * 2 + (size_t)g.ring_slots * g.rw * 2 + 64;
}

// ---- PTX helpers: mbarrier + TMA bulk copy -----------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@!p bra WAIT_%=;\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- horizontal kx-window sums of 8 per-lane columns via in-lane prefix + warp shuffles -----------------------
// p[a] = inclusive prefix of the lane's 8 column sums.  out[r] = sum of the KX columns starting at
// column 8*lane + r.  Static structure for a given KX (all loops unrolled).
template <int KX>
__device__ __forceinline__ void window_sums(const int (&p)[8], int (&out)[8]) {
  const int T = p[7];
  constexpr int MAXL = (KX - 1) / 8;            // most full following lanes any window needs
  // W[k] = T_l + T_{l+1} + ... + T_{l+k}
  int W[MAXL + 1];
  W[0] = T;
#pragma unroll
  for (int k = 1; k <= MAXL; ++k) W[k] = W[k - 1] + __shfl_down_sync(0xffffffffu, T, k);
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int own = 8 - r;                      // columns available in the own lane from r
    if (KX <= own) {
      out[r] = r ? p[r + KX - 1] - p[r - 1] : p[KX - 1];
    } else {
      const int rem = KX - own;                 // columns still needed from the following lanes
      const int full = rem / 8, part = rem % 8;
      if (part) {
        const int q = __shfl_down_sync(0xffffffffu, p[part - 1], full + 1);
        out[r] = r ? (W[full] + q) - p[r - 1] : W[full] + q;      // one IADD3
      } else {
        out[r] = r ? W[full] - p[r - 1] : W[full];
      }
    }
  }
}


}  // namespace vwb200
