// k1_zone_int.cu -- the zone kernel of the pyramid level loop for INTEGER-valued imagery (level 0 of 8-bit rasters):
// the same fused cost-volume + arg-best as k1_generic.cu (semantics of vw::stereo::best_of_search_convolution,
// Stereo/Correlation.cc:33-137, driven by the zone table of Stereo/CorrelationView.cc:607-648), but in exact int32
// arithmetic, with no shared-memory round trip inside the disparity loop.
//
// Exactness: the reference computes the per-pixel cost in float and sums it in double; with integer-valued pixels whose
// range fits 16 bits every term and every window sum is an integer below 2^31, so int32 sums are the same numbers.
//
// One WARP per tile of a zone (<= 33-K columns x 16 rows), four independent warps per CTA:
//   * a lane owns two adjacent columns of the K-1 padded tile; lanes 0-15 work on disparity d, lanes 16-31 on d+1
//   * the tile's left columns live in registers (packed u16 pairs; WIDE: in shared memory); the right search patch is
//     staged once in shared memory as u16 (edge clamping applied during the copy)
//   * per disparity: a running vertical window sum per column (the costs leaving the window come from a register ring,
//     packed u16 pairs), the horizontal window through 6 lane shuffles per row for the lane's two outputs
//   * running best per output = min over (cost << ib | d - d_begin): strict '<' in ascending raster order of d, i.e. the
//     first disparity wins ties, like the reference; running max for the "all costs equal -> invalid" rule (:121-133)
// WIDE (SquaredCost on imagery wider than 8 bits, e.g. the 12-bit pairs of SURVEY 8d): window sums use all 32 bits
// (K^2 * range^2 < 2^32), so the running best is kept as separate (u32 cost, 8-bit index packed four to a register) and
// the "costs differ" rule as one bit per output (set when a cost differs from the running minimum before it).
// Zones with more than 2^ib disparities are split into chunks and finished by k1_generic_merge_kernel (same scratch planes).
#include "common.cuh"

namespace vwb200 {

static constexpr int ZI_TH = 16, ZI_WARPS = 4, ZI_RB = 4;
static constexpr int ZI_FLAG_DIFF = 0x40000000;
static constexpr long long ZI_MAX_U16 = 28672;      // 56 KB of staged right patch per warp (x4 warps <= 227 KB)

__device__ __forceinline__ int zi_clamp(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
__device__ __forceinline__ float zi_ld(const ImgF& im, int x, int y) {
  return __ldg(im.p + (ptrdiff_t)zi_clamp(y, 0, im.h - 1) * im.pitch + zi_clamp(x, 0, im.w - 1));
}

// sum of p over the lanes l .. l+M-1 (binary decomposition of M: floor(log2 M) doublings + popcount(M)-1 pieces)
template <int M>
__device__ __forceinline__ unsigned lane_window(unsigned p) {
  unsigned acc = 0, s = p;
  int off = 0;
#pragma unroll
  for (int bit = 0; (1 << bit) <= M; ++bit) {
    if (M & (1 << bit)) { acc += off == 0 ? s : __shfl_down_sync(0xffffffffu, s, off); off += 1 << bit; }
    if ((2 << bit) <= M) s += __shfl_down_sync(0xffffffffu, s, 1 << bit);
  }
  return acc;
}

template <int COST>
__device__ __forceinline__ int zi_cost(int a, int b) {
  const int e = a - b;
  return COST == VWB200_SQUARED_DIFFERENCE ? e * e : abs(e);
}

__device__ __forceinline__ unsigned put_byte(unsigned word, unsigned v, int pos) {   // byte pos of word := low byte of v
  return __byte_perm(word, v, pos == 0 ? 0x3214 : (pos == 1 ? 0x3240 : (pos == 2 ? 0x3410 : 0x4210)));   // pos is a constant after unrolling
}

// WIDE also reads the left columns from shared memory instead of registers, and its ring keeps |a-b| (two to a register,
// squared again when the row leaves the window): ~100 registers instead of 168, four CTAs per SM instead of three.  The
// narrow kernel would spill at 128 registers, so it keeps the left columns in registers at three CTAs per SM.
template <int COST, int K, bool WIDE>
__global__ void __launch_bounds__(ZI_WARPS * 32, WIDE ? 4 : 3)
k1_zone_int_kernel(ImgF L, ImgF R, const Zone* __restrict__ zones, const Tile* __restrict__ tiles, int ntiles, float vmin, int ib,
                   int warp_u16, vwb200_dispi* __restrict__ out, double* __restrict__ scratch_cost, int* __restrict__ scratch_idx,
                   int* __restrict__ zone_flag) {
  constexpr int M = K / 2, PH = ZI_TH + K - 1, TW = 33 - K;
  extern __shared__ __align__(16) unsigned short zi_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, half = lane >> 4, hl = lane & 15;
  const int ti = blockIdx.x * ZI_WARPS + warp;
  if (ti >= ntiles) return;                                    // warps are independent: no CTA-wide barrier below
  unsigned* sL = reinterpret_cast<unsigned*>(zi_smem + (size_t)warp * warp_u16);     // WIDE: [PH][16] column pairs of the left tile
  unsigned short* sR = zi_smem + (size_t)warp * warp_u16 + (WIDE ? PH * 32 : 0);
  const Tile t = tiles[ti];
  const Zone z = zones[t.zone];
  const int ntx = (z.w + TW - 1) / TW, twb = (z.w + ntx - 1) / ntx;           // balanced split of the zone (host: same formula)
  const int nty = (z.h + ZI_TH - 1) / ZI_TH, thb = (z.h + nty - 1) / nty;
  const int tw = min(twb, z.w - t.tx), th = min(thb, z.h - t.ty);
  const int ph = th + K - 1;
  const int nd_all = z.sx * z.sy, csz = 1 << ib;
  const int d_begin = t.chunk * csz;
  const int nd = z.nchunks > 1 ? min(nd_all, d_begin + csz) : nd_all;          // this warp covers [d_begin, nd)
  const int dy_lo = d_begin / z.sx, dy_hi = (nd - 1) / z.sx;
  const int rph = ph + dy_hi - dy_lo, rpitch = 32 + z.sx;
  const int lx0 = z.lx + t.tx, ly0 = z.ly + t.ty, rx0 = z.rx + t.tx, ry0 = z.ry + t.ty;

  unsigned Lp[WIDE ? 1 : PH];                                  // the lane's two left columns, all padded rows
  bool frac = false;                                           // a non-integer pixel (the mean that replaced a masked one)
#pragma unroll
  for (int r = 0; r < PH; ++r) {
    const int rr = min(r, ph - 1);
    const float f0 = zi_ld(L, lx0 + 2 * hl, ly0 + rr), f1 = zi_ld(L, lx0 + 2 * hl + 1, ly0 + rr);
    frac |= f0 != rintf(f0) || f1 != rintf(f1);
    const unsigned pr = (unsigned)(int)(f0 - vmin) | ((unsigned)(int)(f1 - vmin) << 16);
    if (WIDE) { if (!half) sL[r * 16 + hl] = pr; } else Lp[r] = pr;
  }
  for (int r = 0; r < rph; ++r) {
    const int gy = ry0 + dy_lo + r;
    for (int c = lane; c < rpitch; c += 32) {
      const float f = zi_ld(R, rx0 + c, gy);
      frac |= f != rintf(f);
      sR[r * rpitch + c] = (unsigned short)(int)(f - vmin);
    }
  }
  if (__any_sync(0xffffffffu, frac)) {                         // not exact in integers: the fp64 kernel redoes the whole zone
    if (lane == 0) zone_flag[t.zone] = 1;
    return;
  }
  __syncwarp();

  unsigned bmin[ZI_TH][2];
  int bmax[WIDE ? 1 : ZI_TH][2];                               // narrow: running max
  unsigned bidx[WIDE ? ZI_TH / 2 : 1];                         // wide: 8-bit disparity index of output (y, j) in byte (2y+j)&3 of word (2y+j)>>2
  unsigned dmask = 0;                                          // wide: bit 2y+j = some cost differed from the running minimum
#pragma unroll
  for (int y = 0; y < ZI_TH; ++y) { bmin[y][0] = bmin[y][1] = 0xffffffffu; if (!WIDE) bmax[y][0] = bmax[y][1] = 0; }
#pragma unroll
  for (int i = 0; i < (WIDE ? ZI_TH / 2 : 1); ++i) bidx[i] = 0;

  const int niter = (nd - d_begin + 1) >> 1;
  for (int it = 0; it < niter; ++it) {
    int d = d_begin + 2 * it + half;
    if (d >= nd) d = nd - 1;                                   // odd count: the upper half repeats the last disparity (harmless)
    const int dy = d / z.sx, dx = d - dy * z.sx;
    const unsigned short* rp = sR + (dy - dy_lo) * rpitch + 2 * hl + dx;
    const unsigned didx = (unsigned)(d - d_begin);
    unsigned v0 = 0, v1 = 0;
    unsigned ring[ZI_TH];                                      // costs that will leave the window: rows 0 .. TH-1 only
#pragma unroll
    for (int r = 0; r < K - 1; ++r) {                          // rows above the first window (ph >= K: always present)
      const unsigned lp = WIDE ? sL[r * 16 + hl] : Lp[r];
      const int e0 = (int)(lp & 0xffffu) - (int)rp[r * rpitch], e1 = (int)(lp >> 16) - (int)rp[r * rpitch + 1];
      const unsigned c0 = (unsigned)(COST == VWB200_SQUARED_DIFFERENCE ? e0 * e0 : abs(e0));
      const unsigned c1 = (unsigned)(COST == VWB200_SQUARED_DIFFERENCE ? e1 * e1 : abs(e1));
      if (r < ZI_TH) {
        if (WIDE) ring[r] = (unsigned)abs(e0) | ((unsigned)abs(e1) << 16);
        else ring[r] = c0 | (c1 << 16);
      }
      v0 += c0; v1 += c1;
    }
#pragma unroll
    for (int yb = 0; yb < ZI_TH; yb += ZI_RB) {
      if (yb < th) {                                           // warp-uniform, one branch per block of ZI_RB rows: the rows of a block
#pragma unroll                                                 // interleave; rows past th inside the last block work on stale data
        for (int y = yb; y < yb + ZI_RB; ++y) {                // (shared memory rows that exist, outputs never written)
          const int r = y + K - 1;
          const unsigned lp = WIDE ? sL[r * 16 + hl] : Lp[r];
          const int e0 = (int)(lp & 0xffffu) - (int)rp[r * rpitch], e1 = (int)(lp >> 16) - (int)rp[r * rpitch + 1];
          const unsigned c0 = (unsigned)(COST == VWB200_SQUARED_DIFFERENCE ? e0 * e0 : abs(e0));
          const unsigned c1 = (unsigned)(COST == VWB200_SQUARED_DIFFERENCE ? e1 * e1 : abs(e1));
          if (r < ZI_TH) {
            if (WIDE) ring[r] = (unsigned)abs(e0) | ((unsigned)abs(e1) << 16);
            else ring[r] = c0 | (c1 << 16);
          }
          v0 += c0; v1 += c1;
          // K = 2M+1 columns: output 2l = M pairs (l .. l+M-1) + column 2(l+M); output 2l+1 = column 2l+1 + M pairs (l+1 .. l+M)
          const unsigned pm = lane_window<M>(v0 + v1);
          const unsigned h0 = pm + __shfl_down_sync(0xffffffffu, v0, M);
          const unsigned h1 = v1 + __shfl_down_sync(0xffffffffu, pm, 1);
          if (WIDE) {
            if (h0 != bmin[y][0]) dmask |= 1u << (2 * y);
            if (h1 != bmin[y][1]) dmask |= 2u << (2 * y);
            if (h0 < bmin[y][0]) bidx[y / 2] = put_byte(bidx[y / 2], didx, (2 * y) & 3);
            if (h1 < bmin[y][1]) bidx[y / 2] = put_byte(bidx[y / 2], didx, (2 * y + 1) & 3);
            bmin[y][0] = min(bmin[y][0], h0);
            bmin[y][1] = min(bmin[y][1], h1);
            const unsigned a0 = ring[y] & 0xffffu, a1 = ring[y] >> 16;
            v0 -= a0 * a0;
            v1 -= a1 * a1;
          } else {
            bmin[y][0] = min(bmin[y][0], (h0 << ib) | didx);
            bmin[y][1] = min(bmin[y][1], (h1 << ib) | didx);
            bmax[y][0] = max(bmax[y][0], (int)h0);
            bmax[y][1] = max(bmax[y][1], (int)h1);
            v0 -= ring[y] & 0xffffu;
            v1 -= ring[y] >> 16;
          }
        }
      }
    }
    if (WIDE && it == 0) dmask = 0;                            // the first disparity only set the baseline
  }
  // the two half warps saw different disparities of the same pixels; outputs: lanes 0-15
  const unsigned o_dmask = __shfl_xor_sync(0xffffffffu, dmask, 16);
  unsigned o_bidx[WIDE ? ZI_TH / 2 : 1];
#pragma unroll
  for (int i = 0; i < (WIDE ? ZI_TH / 2 : 1); ++i) o_bidx[i] = WIDE ? __shfl_xor_sync(0xffffffffu, bidx[i], 16) : 0u;
#pragma unroll
  for (int y = 0; y < ZI_TH; ++y) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const unsigned o_min = __shfl_xor_sync(0xffffffffu, bmin[y][j], 16);
      int o_max = 0;
      if (!WIDE) o_max = __shfl_xor_sync(0xffffffffu, bmax[y][j], 16);
      if (half || y >= th) continue;
      const int x = 2 * hl + j;
      if (x >= tw) continue;
      unsigned best; int d; bool diff;
      if (WIDE) {
        const int sh = 8 * ((2 * y + j) & 3);
        const unsigned i0 = (bidx[y / 2] >> sh) & 0xffu, i1 = (o_bidx[y / 2] >> sh) & 0xffu;
        diff = (((dmask | o_dmask) >> (2 * y + j)) & 1u) || bmin[y][j] != o_min;
        const bool other = o_min < bmin[y][j] || (o_min == bmin[y][j] && i1 < i0);     // equal costs: the earlier disparity
        best = other ? o_min : bmin[y][j];
        d = d_begin + (int)(other ? i1 : i0);
      } else {
        const unsigned m = min(bmin[y][j], o_min);
        best = m >> ib;
        d = d_begin + (int)(m & (unsigned)(csz - 1));
        diff = (unsigned)max(bmax[y][j], o_max) != best;
      }
      if (z.nchunks > 1) {
        const long long s = z.sbase + ((long long)t.chunk * z.h + (t.ty + y)) * z.w + (t.tx + x);
        scratch_cost[s] = (double)best;
        scratch_idx[s] = d | (diff ? ZI_FLAG_DIFF : 0);
      } else {
        vwb200_dispi o;
        o.dy = d / z.sx;
        o.dx = d - o.dy * z.sx + z.addx;
        o.dy += z.addy;
        o.valid = diff ? 1 : 0;
        out[z.obase + (ptrdiff_t)(t.ty + y) * z.opitch + (t.tx + x)] = o;
      }
    }
  }
}

// ---- host side ------------------------------------------------------------------------------------------------------
// supported: Abs / Sq, square odd kernel 3..25, pixel range that keeps a per-pixel cost in 16 bits and a window sum (shifted
// left by the disparity-index bits) in 32.  *ib_out = log2 of the disparity chunk a warp covers.
// Returns 0 (unsupported), 1 (narrow) or 2 (wide).
int k1_zone_int_mode(int cost, int kx, int ky, long long range, int* ib_out) {
  if (cost != VWB200_ABSOLUTE_DIFFERENCE && cost != VWB200_SQUARED_DIFFERENCE) return 0;
  if (kx != ky || kx < 3 || kx > 25 || !(kx & 1) || range < 0 || range > 65535) return 0;
  // |a-b| <= 4095 keeps the reference's FLOAT product (a-b)*(a-b) exact (< 2^24)
  if (cost == VWB200_SQUARED_DIFFERENCE && range > 4095) return 0;
  const long long per_pixel = cost == VWB200_SQUARED_DIFFERENCE ? range * range : range;
  const long long maxh = per_pixel * kx * ky;
  if (ib_out) *ib_out = 8;                  // 256 disparities per warp = K1G_DCHUNK: split zones share the fp64 kernel's scratch layout
  if (per_pixel <= 65535 && maxh < (1ll << 24)) return 1;
  if (cost == VWB200_SQUARED_DIFFERENCE && maxh < 0xffffffffll) return 2;
  return 0;
}
bool k1_zone_int_supported(int cost, int kx, int ky, long long range, int* ib_out) { return k1_zone_int_mode(cost, kx, ky, range, ib_out) != 0; }
int k1_zone_int_tile_w(int k) { return 33 - k; }
int k1_zone_int_tile_h() { return ZI_TH; }
// u16 elements of right search patch one warp stages for a tile of this zone (upper bound over its tiles)
long long k1_zone_int_stage_u16(int k, int sx, int sy, int nchunks, int ib) {
  const int span = nchunks > 1 ? std::min(sy, ((1 << ib) + sx - 1) / sx + 1) : sy;
  return (long long)(ZI_TH + k - 1 + span - 1) * (32 + sx) + (ZI_TH + k - 1) * 32;      // + the left tile (wide)
}
long long k1_zone_int_stage_max() { return ZI_MAX_U16; }

int k1_zone_int_launch(int cost, ImgF left, ImgF right, const Zone* d_zones, const Tile* d_tiles, int ntiles, int k, float vmin, float vmax,
                       int warp_u16, vwb200_dispi* out, double* scratch_cost, int* scratch_idx, int* zone_flag, cudaStream_t st,
                       const KEvents* ev) {
  if (ntiles <= 0) return VWB200_OK;
  int ib = 0;
  const int mode = k1_zone_int_mode(cost, k, k, (long long)vmax - (long long)vmin, &ib);
  if (!mode) { set_error("integer zone kernel: unsupported configuration"); return VWB200_ELOGIC; }
  void (*kern)(ImgF, ImgF, const Zone*, const Tile*, int, float, int, int, vwb200_dispi*, double*, int*, int*) = nullptr;
#define ZI_CASE(KK)                                                                                                          \
  case KK:                                                                                                                   \
    kern = mode == 2 ? k1_zone_int_kernel<VWB200_SQUARED_DIFFERENCE, KK, true>                                               \
         : (cost == VWB200_SQUARED_DIFFERENCE ? k1_zone_int_kernel<VWB200_SQUARED_DIFFERENCE, KK, false>                     \
                                              : k1_zone_int_kernel<VWB200_ABSOLUTE_DIFFERENCE, KK, false>);                  \
    break;
  switch (k) {
    ZI_CASE(3) ZI_CASE(5) ZI_CASE(7) ZI_CASE(9) ZI_CASE(11) ZI_CASE(13) ZI_CASE(15) ZI_CASE(17) ZI_CASE(19) ZI_CASE(21) ZI_CASE(23) ZI_CASE(25)
    default: set_error("integer zone kernel: kernel size %d not instantiated", k); return VWB200_ELOGIC;
  }
#undef ZI_CASE
  warp_u16 = (warp_u16 + 7) & ~7;
  const size_t smem = (size_t)ZI_WARPS * warp_u16 * sizeof(unsigned short);
  if (smem > 227 * 1024) { set_error("integer zone kernel needs %zu bytes of shared memory", smem); return VWB200_ELOGIC; }
  // per-function state shared by all host threads: always the device maximum, never the per-launch size
  VWB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  if (ev && ev->e0) cudaEventRecord(ev->e0, st);
  kern<<<(ntiles + ZI_WARPS - 1) / ZI_WARPS, ZI_WARPS * 32, smem, st>>>(left, right, d_zones, d_tiles, ntiles, vmin, ib, warp_u16, out,
                                                                      scratch_cost, scratch_idx, zone_flag);
  VWB_LAUNCH_CHECK();
  if (ev && ev->e1) cudaEventRecord(ev->e1, st);
  return VWB200_OK;
}

}  // namespace vwb200
