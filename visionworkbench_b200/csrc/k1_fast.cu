// k1_fast.cu -- exact-integer fast path of the fused cost-volume + arg-best kernel (AbsoluteCost).
//
// When both rasters are integer valued with (max-min)*8 < 2^16 (8..13-bit imagery), every quantity
// of best_of_search_convolution (Stereo/Correlation.cc:33-137) is an exact integer: the float
// per-pixel cost |a-b|, the double box sums and therefore the comparison results.  The kernel below
// evaluates the same cost volume in int32 and applies the same selection rule (strict '<', dy-major /
// dx-minor order => first disparity wins ties; all-equal => invalid), so it is bit-identical to the
// reference while doing ~10 issue slots per (pixel, disparity) instead of ~70 bytes of DRAM traffic.
//
// Decomposition (persistent CTAs of 4 warps, one CTA per SM; work item = 236-column x 32-row band):
//   * values are pre-packed (pack kernels) as u16 (v-vmin)*8, one contiguous row per strip, so that a
//     lane fetches its 8 left / 16 right columns with conflict-free 16-byte LDS.128 loads
//   * the left tile (32+ky-1 rows) and a ring of right rows are staged in shared memory with TMA bulk
//     copies (cp.async.bulk + mbarrier); one new right row is prefetched per dy while the CTA computes
//   * lane l owns padded columns 8l..8l+7 and 8 consecutive dx: V[8][8] vertical sliding sums live in
//     registers (VABSDIFF accumulate: +new row, -old row)
//   * the kx-wide horizontal sums are formed without shared memory: in-lane prefix sums + 9 warp
//     shuffles per 8 outputs (blocked-prefix scheme), 3-input IADD3
//   * arg-best: costs are pre-scaled by 8 so key = cost*8 + b; min over the 8 dx is 7 VIADDMNMX;
//     the running best (cost only) sits in shared memory, the index goes to a global scratch plane
//     on the (rare) improvements; warps cover disjoint dx subsets and are merged at the end of the band
//   * pixels whose arg-best is disparity (0,0) are re-checked by a small kernel for the
//     "every disparity gave the same cost => invalid" rule (Correlation.cc:121-133)
#include "k1_fast_common.cuh"

namespace vwb200 {

// ---- min / max / integer-valuedness reduction -------------------------------------------------------
__global__ void image_stats_kernel(ImgF img, float* __restrict__ result) {
  float mn = INFINITY, mx = -INFINITY; int allint = 1;
  const long long n = (long long)img.w * img.h;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
    const float v = img.p[(ptrdiff_t)(k / img.w) * img.pitch + (k % img.w)];
    mn = fminf(mn, v); mx = fmaxf(mx, v);
    if (!(v == rintf(v))) allint = 0;          // NaN/inf -> not integer
  }
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    allint &= __shfl_xor_sync(0xffffffffu, allint, o);
  }
  if ((threadIdx.x & 31) == 0) {
    // order-preserving float->int mapping so integer atomics can be used
    atomicMin(reinterpret_cast<int*>(result) + 0, mn >= 0 ? __float_as_int(mn) : (int)(0x80000000u - (unsigned)__float_as_int(mn)));
    atomicMax(reinterpret_cast<int*>(result) + 1, mx >= 0 ? __float_as_int(mx) : (int)(0x80000000u - (unsigned)__float_as_int(mx)));
    if (!allint) atomicExch(reinterpret_cast<int*>(result) + 2, 0);
  }
}
__global__ void image_stats_init(float* result) {
  reinterpret_cast<int*>(result)[0] = INT_MAX; reinterpret_cast<int*>(result)[1] = INT_MIN; reinterpret_cast<int*>(result)[2] = 1;
}
__global__ void image_stats_fini(float* result) {
  int* r = reinterpret_cast<int*>(result);
  for (int i = 0; i < 2; ++i) {
    const int o = r[i];
    result[i] = o >= 0 ? __int_as_float(o) : __int_as_float((int)(0x80000000u - (unsigned)o));
  }
  result[2] = r[2] ? 1.0f : 0.0f;
}
int image_stats_launch(ImgF img, float* d_result3, cudaStream_t st) {
  image_stats_init<<<1, 1, 0, st>>>(d_result3);
  VWB_LAUNCH_CHECK();
  image_stats_kernel<<<296, 256, 0, st>>>(img, d_result3);
  VWB_LAUNCH_CHECK();
  image_stats_fini<<<1, 1, 0, st>>>(d_result3);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

int k1_fast_supported(int cost, int kx, int ky, int sx, int sy, float vmin, float vmax, bool integer_valued) {
  if (cost != VWB200_ABSOLUTE_DIFFERENCE && cost != VWB200_SQUARED_DIFFERENCE) return VWB200_ENOIMPL;
  if (!integer_valued) return VWB200_ENOIMPL;
  if (cost == VWB200_SQUARED_DIFFERENCE) {        // window sums of (a-b)^2 must fit uint32
    const double r = (double)vmax - (double)vmin;
    // |a-b| <= 4095 keeps the reference's FLOAT (a-b)*(a-b) exact (< 2^24); beyond that it rounds and only the
    // general kernel (which issues the same float multiply) reproduces it
    if (!(r <= 4095.0) || !(r * r * kx * ky < 4294967295.0)) return VWB200_ENOIMPL;
  } else if (!(vmax - vmin <= 8191.0f)) return VWB200_ENOIMPL;
  if ( !(fabsf(vmin) < 1.0e6f) || !(fabsf(vmax) < 1.0e6f)) return VWB200_ENOIMPL;
  if (kx < 3 || kx > 31 || ky < 1 || ky > 41) return VWB200_ENOIMPL;
  if (sx < F_B || sx > 512 || sy < 1) return VWB200_ENOIMPL;
  if ((long long)sx * sy > 65536) return VWB200_ENOIMPL;
  if ((long long)sx * sy < 64) return VWB200_ENOIMPL;      // tiny searches: the generic kernel is as good
  FastGeom g = make_geom(256, 32, sx, sy, kx, ky);
  if (fast_smem_bytes(g) > 227 * 1024) return VWB200_ENOIMPL;
  return VWB200_OK;
}

size_t k1_fast_workspace_bytes(int W, int H, int sx, int sy, int kx, int ky) {
  FastGeom g = make_geom(W, H, sx, sy, kx, ky);
  size_t l = (size_t)g.NS * g.lrows * F_COLS * 2;
  size_t r = (size_t)g.NS * g.rrows * g.rw * 2;
  size_t idx = (size_t)1024 * F_SUBSETS * F_TH * F_COLS * 2;    // per-CTA index planes (<= 1024 CTAs)
  size_t part = g.J > 1 ? (size_t)g.J * W * H * 6 + 64 : 0;      // per-dy-chunk partial (cost u32, index u16)
  return l + r + idx + part + 512;
}

// ---- pack kernels: float raster -> u16 (v - vmin) * 4 in the lane-transposed strip layout ------------
__global__ void pack_left_kernel(ImgF img, float vmin, FastGeom g, uint16_t* __restrict__ out) {
  const int row = blockIdx.x, strip = blockIdx.y;
  const int s0 = strip * g.out_cols;
  uint16_t* o = out + ((size_t)strip * g.lrows + row) * F_COLS;
  for (int c = threadIdx.x; c < F_COLS; c += blockDim.x) {      // c = strip-relative padded column (coalesced reads)
    const int gx = s0 + c;
    uint16_t v = 0;      // logical raster = (W+kx-1) x (H+ky-1) at (lox,loy); constant edge extension of the image beyond it
    if (row < g.H + g.ky - 1 && gx < g.W + g.kx - 1) {
      const int iy = min(max(g.loy + row, 0), img.h - 1), ix = min(max(g.lox + gx, 0), img.w - 1);
      v = (uint16_t)((int)(img.p[(ptrdiff_t)iy * img.pitch + ix] - vmin) * g.scale);
    }
    o[c] = v;
  }
}
__global__ void pack_right_kernel(ImgF img, float vmin, FastGeom g, uint16_t* __restrict__ out) {
  const int row = blockIdx.x, strip = blockIdx.y;
  const int s0 = strip * g.out_cols;
  uint16_t* o = out + ((size_t)strip * g.rrows + row) * g.rw;
  for (int c = threadIdx.x; c < g.rw; c += blockDim.x) {
    const int gx = s0 + c;
    uint16_t v = 0;
    if (row < g.H + g.ky - 1 + g.sy - 1 && gx < g.W + g.kx - 1 + g.sx - 1) {
      const int iy = min(max(g.roy + row, 0), img.h - 1), ix = min(max(g.rox + gx, 0), img.w - 1);
      v = (uint16_t)((int)(img.p[(ptrdiff_t)iy * img.pitch + ix] - vmin) * g.scale);
    }
    o[c] = v;
  }
}

// ---- one pass: 8 consecutive dx (octet g) x 8 columns per lane, sliding down the warp's rows ----------------
__device__ __forceinline__ void unpack8(const uint4 v, int (&o)[8]) {
  o[0] = v.x & 0xffff; o[1] = v.x >> 16; o[2] = v.y & 0xffff; o[3] = v.y >> 16;
  o[4] = v.z & 0xffff; o[5] = v.z >> 16; o[6] = v.w & 0xffff; o[7] = v.w >> 16;
}
__device__ __forceinline__ void load_row(const uint16_t* lrow, const uint16_t* rrow, int (&Lv)[8], int (&Rv)[16]) {
  unpack8(*reinterpret_cast<const uint4*>(lrow), Lv);
  int t[8];
  unpack8(*reinterpret_cast<const uint4*>(rrow), t);
#pragma unroll
  for (int i = 0; i < 8; ++i) Rv[i] = t[i];
  unpack8(*reinterpret_cast<const uint4*>(rrow + 8), t);
#pragma unroll
  for (int i = 0; i < 8; ++i) Rv[8 + i] = t[i];
}

template <int KX, bool FULL>
__device__ __forceinline__ void fast_pass(const uint16_t* __restrict__ ltile, const uint16_t* __restrict__ rring,
                                          uint32_t* __restrict__ state, uint16_t* __restrict__ idxp,
                                          int lane, int g, int ky, int ring_slots, int rw, int ring_base, int idx_base, int row0, int nb) {
  int V[8][F_B];
  const uint16_t* lp = ltile + row0 * F_COLS + 8 * lane;       // + row*256            (16-byte aligned)
  const uint16_t* rp = rring + 8 * (lane + g);                 // + slot*rw            (16-byte aligned)
  int slot_new = ring_base;                                     // ring slot of right row (dy + row0 + t)
  // ---- seed: first ky rows
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < F_B; ++b) V[a][b] = 0;
  for (int t = 0; t < ky; ++t) {
    int Lv[8], Rv[16];
    load_row(lp + t * F_COLS, rp + slot_new * rw, Lv, Rv);
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = 0; b < F_B; ++b) V[a][b] = __sad(Lv[a], Rv[a + b], V[a][b]);
    if (++slot_new == ring_slots) slot_new = 0;
  }
  int slot_old = ring_base;
  for (int y = 0; y < F_RH; ++y) {
    if (y > 0) {
      {
        int Lv[8], Rv[16];
        load_row(lp + (y + ky - 1) * F_COLS, rp + slot_new * rw, Lv, Rv);
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < F_B; ++b) V[a][b] = __sad(Lv[a], Rv[a + b], V[a][b]);
      }
      {
        int Lo[8], Ro[16];
        load_row(lp + (y - 1) * F_COLS, rp + slot_old * rw, Lo, Ro);
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < F_B; ++b) V[a][b] -= __sad(Lo[a], Ro[a + b], 0);
      }
      if (++slot_new == ring_slots) slot_new = 0;
      if (++slot_old == ring_slots) slot_old = 0;
    }
    // ---- horizontal window sums + min over the 8 dx (keys = cost*8 + b) ----
    int m[8];
#pragma unroll
    for (int b = 0; b < F_B; ++b) {
      if (!FULL && b >= nb) break;      // last octet of a search width that is not a multiple of 8 (warp uniform)
      int p[8], o[8];
      p[0] = V[0][b];
#pragma unroll
      for (int a = 1; a < 8; ++a) p[a] = p[a - 1] + V[a][b];
      window_sums<KX>(p, o);
#pragma unroll
      for (int r = 0; r < 8; ++r) m[r] = (b == 0) ? o[r] : min(o[r] + b, m[r]);
    }
    // ---- running best (shared memory), index plane (global) on improvement ----
    uint32_t* srow = state + y * F_COLS + lane;
    uint32_t s8[8];
    bool improved = false;
#pragma unroll
    for (int r = 0; r < 8; ++r) { s8[r] = srow[r * 32]; improved |= ((uint32_t)m[r] < s8[r]); }
    if (improved) {            // rare once the search has seen the neighbourhood of the true match
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        if ((uint32_t)m[r] < s8[r]) {
          srow[r * 32] = (uint32_t)m[r] & ~7u;
          idxp[y * F_COLS + r * 32 + lane] = (uint16_t)(idx_base + (m[r] & 7));
        }
      }
    }
  }
}

// ---- SquaredCost variant of the integer pass ----------------------------------------------------------------
// (a-b)^2 of integer imagery is an exact integer in the reference's float arithmetic as long as |a-b| < 4096, and
// the double window sums are exact; here they are uint32 (the host checks kx*ky*range^2 < 2^32).  Costs do not
// leave room for the key trick, so the arg-min over the octet is tracked with compare/select.
template <int KX>
__device__ __forceinline__ void fast_pass_sq(const uint16_t* __restrict__ ltile, const uint16_t* __restrict__ rring,
                                             uint32_t* __restrict__ state, uint16_t* __restrict__ idxp,
                                             int lane, int g, int ky, int ring_slots, int rw, int ring_base, int idx_base, int row0, int nb) {
  int V[8][F_B];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < F_B; ++b) V[a][b] = 0;
  const uint16_t* lp = ltile + row0 * F_COLS + 8 * lane;
  const uint16_t* rp = rring + 8 * (lane + g);
  int slot_new = ring_base;
  for (int t = 0; t < ky; ++t) {
    int Lv[8], Rv[16];
    load_row(lp + t * F_COLS, rp + slot_new * rw, Lv, Rv);
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = 0; b < F_B; ++b) { const int d = Lv[a] - Rv[a + b]; V[a][b] += d * d; }
    if (++slot_new == ring_slots) slot_new = 0;
  }
  int slot_old = ring_base;
  for (int y = 0; y < F_RH; ++y) {
    if (y > 0) {
      {
        int Lv[8], Rv[16];
        load_row(lp + (y + ky - 1) * F_COLS, rp + slot_new * rw, Lv, Rv);
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < F_B; ++b) { const int d = Lv[a] - Rv[a + b]; V[a][b] += d * d; }
      }
      {
        int Lo[8], Ro[16];
        load_row(lp + (y - 1) * F_COLS, rp + slot_old * rw, Lo, Ro);
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < F_B; ++b) { const int d = Lo[a] - Ro[a + b]; V[a][b] -= d * d; }
      }
      if (++slot_new == ring_slots) slot_new = 0;
      if (++slot_old == ring_slots) slot_old = 0;
    }
    uint32_t m[8];
    int mb[8];
#pragma unroll
    for (int b = 0; b < F_B; ++b) {
      if (b >= nb) break;
      int p[8], o[8];
      p[0] = V[0][b];
#pragma unroll
      for (int a = 1; a < 8; ++a) p[a] = p[a - 1] + V[a][b];     // wraps mod 2^32 like the uint32 sums they stand for
      window_sums<KX>(p, o);
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const uint32_t c = (uint32_t)o[r];
        if (b == 0) { m[r] = c; mb[r] = 0; }
        else if (c < m[r]) { m[r] = c; mb[r] = b; }
      }
    }
    uint32_t* srow = state + y * F_COLS + lane;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      if (m[r] < srow[r * 32]) {
        srow[r * 32] = m[r];
        idxp[y * F_COLS + r * 32 + lane] = (uint16_t)(idx_base + mb[r]);
      }
    }
  }
}

template <int KX, bool SQ>
__global__ void __launch_bounds__(F_THREADS, 1)
k1_fast_abs_kernel(const uint16_t* __restrict__ L16, const uint16_t* __restrict__ R16, FastGeom G,
                   uint16_t* __restrict__ idx_scratch, vwb200_dispi* __restrict__ out, ptrdiff_t opitch,
                   uint32_t* __restrict__ part_cost, uint16_t* __restrict__ part_idx) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint32_t* state = reinterpret_cast<uint32_t*>(smem);                                  // [4][32][8][32]
  uint16_t* ltile = reinterpret_cast<uint16_t*>(smem + (size_t)F_SUBSETS * F_TH * F_COLS * 4);
  uint16_t* rring = ltile + (size_t)G.ltile_rows * F_COLS;
  uint64_t* bars = reinterpret_cast<uint64_t*>(rring + (size_t)G.ring_slots * G.rw);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int sub = w & (F_SUBSETS - 1), half = w / F_SUBSETS, row0 = half * F_RH;
  const int ngroups = (G.sx + F_B - 1) / F_B;
  uint16_t* idxp_block = idx_scratch + (size_t)blockIdx.x * F_SUBSETS * F_TH * F_COLS;
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  __syncthreads();
  uint32_t ph0 = 0, ph1 = 0;
  const uint32_t lbytes = (uint32_t)G.ltile_rows * F_COLS * 2, rrow_bytes = (uint32_t)G.rw * 2;
  for (int item = blockIdx.x; item < G.NS * G.NB * G.J; item += gridDim.x) {
    const int chunk = item % G.J, rest = item / G.J;
    const int strip = rest % G.NS, band = rest / G.NS;
    const int y0 = band * F_TH;
    const int dy0 = chunk * G.dy_per, ndy = min(G.sy, dy0 + G.dy_per) - dy0;
    const uint16_t* lsrc = L16 + ((size_t)strip * G.lrows + y0) * F_COLS;
    const uint16_t* rsrc = R16 + ((size_t)strip * G.rrows + y0 + dy0) * G.rw;
    if (tid == 0) {
      fence_proxy_async();
      mbar_expect_tx(&bars[0], lbytes + (uint32_t)G.ltile_rows * rrow_bytes);
      tma_load_1d(ltile, lsrc, lbytes, &bars[0]);
      tma_load_1d(rring, rsrc, (uint32_t)G.ltile_rows * rrow_bytes, &bars[0]);     // right rows y0 .. y0+ltile_rows-1 -> slots 0..
    }
    for (int k = tid; k < F_SUBSETS * F_TH * F_COLS; k += F_THREADS) state[k] = SQ ? 0xffffffffu : S_INIT;     // max cost / max key
    __syncthreads();
    mbar_wait(&bars[0], ph0); ph0 ^= 1;
    uint32_t* wstate = state + ((size_t)sub * F_TH + row0) * F_COLS;       // this warp's rows of its subset plane
    uint16_t* widx = idxp_block + ((size_t)sub * F_TH + row0) * F_COLS;
    for (int dy = 0; dy < ndy; ++dy) {         // dy relative to the chunk's first row dy0
      const int ring_base = (dy + row0) % G.ring_slots;
      if (tid == 0 && dy + 1 < ndy) {        // prefetch the row iteration dy+1 adds, into the slot iteration dy-1 freed
        fence_proxy_async();
        mbar_expect_tx(&bars[1], rrow_bytes);
        tma_load_1d(rring + (size_t)((dy + G.ltile_rows) % G.ring_slots) * G.rw, rsrc + (size_t)(dy + G.ltile_rows) * G.rw, rrow_bytes, &bars[1]);
      }
      for (int g = sub; g < ngroups; g += F_SUBSETS) {
        if (SQ) fast_pass_sq<KX>(ltile, rring, wstate, widx, lane, g, G.ky, G.ring_slots, G.rw, ring_base, (dy0 + dy) * G.sx + F_B * g, row0,
                                 min(F_B, G.sx - F_B * g));
        else if (G.sx - F_B * g >= F_B)
          fast_pass<KX, true>(ltile, rring, wstate, widx, lane, g, G.ky, G.ring_slots, G.rw, ring_base, (dy0 + dy) * G.sx + F_B * g, row0, F_B);
        else
          fast_pass<KX, false>(ltile, rring, wstate, widx, lane, g, G.ky, G.ring_slots, G.rw, ring_base, (dy0 + dy) * G.sx + F_B * g, row0,
                               G.sx - F_B * g);
      }
      if (dy + 1 < ndy) { mbar_wait(&bars[1], ph1); ph1 ^= 1; }
      __syncthreads();
    }
    // ---- merge the 4 warps' private bests and write {dx, dy, valid} ----
    const int nw = ngroups < F_SUBSETS ? ngroups : F_SUBSETS;
    const int s0 = strip * G.out_cols;
    for (int pix = tid; pix < F_TH * G.out_cols; pix += F_THREADS) {
      const int x = pix % G.out_cols, y = pix / G.out_cols;
      const int gx = s0 + x, gy = y0 + y;
      if (gx >= G.W || gy >= G.H) continue;
      const int off = y * F_COLS + (x & 7) * 32 + (x >> 3);
      uint32_t best = state[off];
      int bidx = idxp_block[off];
      for (int ww = 1; ww < nw; ++ww) {
        const uint32_t c = state[(size_t)ww * F_TH * F_COLS + off];
        const int i = idxp_block[(size_t)ww * F_TH * F_COLS + off];
        if (c < best || (c == best && i < bidx)) { best = c; bidx = i; }
      }
      if (G.J > 1) {             // partial result of this dy chunk; k1_fast_merge_kernel finishes the pixel
        const size_t pk = ((size_t)chunk * G.H + gy) * G.W + gx;
        part_cost[pk] = best; part_idx[pk] = (uint16_t)bidx;
        continue;
      }
      vwb200_dispi o;
      o.dx = bidx % G.sx + G.addx; o.dy = bidx / G.sx + G.addy; o.valid = 1;
      out[(ptrdiff_t)gy * opitch + gx] = o;
    }
    __syncthreads();
  }
}

// merge of the dy chunks (ascending chunk = ascending raster order: an equal cost keeps the earlier chunk)
__global__ void k1_fast_merge_kernel(FastGeom G, const uint32_t* __restrict__ part_cost, const uint16_t* __restrict__ part_idx,
                                     vwb200_dispi* __restrict__ out, ptrdiff_t opitch) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= G.W || y >= G.H) return;
  const size_t plane = (size_t)G.W * G.H, k = (size_t)y * G.W + x;
  uint32_t best = part_cost[k];
  int bidx = part_idx[k];
  for (int c = 1; c < G.J; ++c) {
    const uint32_t cc = part_cost[c * plane + k];
    if (cc < best) { best = cc; bidx = part_idx[c * plane + k]; }
  }
  vwb200_dispi o;
  o.dx = bidx % G.sx + G.addx; o.dy = bidx / G.sx + G.addy; o.valid = 1;
  out[(ptrdiff_t)y * opitch + x] = o;
}

// ---- "every disparity gave the same cost" fix-up for pixels whose arg-best is (0,0) --------------------------
__global__ void k1_fast_allequal_fixup(ImgF L, ImgF R, FastGeom g, vwb200_dispi* __restrict__ out, ptrdiff_t opitch) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= g.W || y >= g.H) return;
  vwb200_dispi* o = out + (ptrdiff_t)y * opitch + x;
  if (o->dx != g.addx || o->dy != g.addy) return;
  // arg-best (0,0): valid iff some disparity has a different (necessarily larger) cost.  Integer-valued inputs:
  // exact integer arithmetic.  Reads follow the pack kernels (constant edge extension around the logical rasters).
  auto lv = [&](int xx, int yy) { return (int)L.p[(ptrdiff_t)min(max(g.loy + yy, 0), L.h - 1) * L.pitch + min(max(g.lox + xx, 0), L.w - 1)]; };
  auto rv = [&](int xx, int yy) { return (int)R.p[(ptrdiff_t)min(max(g.roy + yy, 0), R.h - 1) * R.pitch + min(max(g.rox + xx, 0), R.w - 1)]; };
  long long c0 = 0;
  for (int j = 0; j < g.ky; ++j)
    for (int i = 0; i < g.kx; ++i) { const long long d = lv(x + i, y + j) - rv(x + i, y + j); c0 += g.scale == 1 ? d * d : (d < 0 ? -d : d); }
  for (int dy = 0; dy < g.sy; ++dy)
    for (int dx = 0; dx < g.sx; ++dx) {
      if (dx == 0 && dy == 0) continue;
      long long c = 0;
      for (int j = 0; j < g.ky; ++j)
        for (int i = 0; i < g.kx; ++i) { const long long d = lv(x + i, y + j) - rv(x + i + dx, y + j + dy); c += g.scale == 1 ? d * d : (d < 0 ? -d : d); }
      if (c != c0) return;      // not all equal -> stays valid
    }
  o->valid = 0;
}

int k1_fast_launch(int cost, ImgF left, ImgF right, int W, int H, int sx, int sy, int kx, int ky, float vmin,
                   vwb200_dispi* out, ptrdiff_t opitch, void* workspace, size_t workspace_bytes, cudaStream_t st,
                   const KEvents* ev, const FastOrigin* org) {
  (void)workspace_bytes;
  const bool sq = cost == VWB200_SQUARED_DIFFERENCE;
  FastGeom g = make_geom(W, H, sx, sy, kx, ky);
  g.scale = sq ? 1 : F_B;
  if (org) { g.lox = org->lox; g.loy = org->loy; g.rox = org->rox; g.roy = org->roy; g.addx = org->addx; g.addy = org->addy; }
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  uint16_t* L16 = reinterpret_cast<uint16_t*>(ws);
  uint16_t* R16 = L16 + (size_t)g.NS * g.lrows * F_COLS;
  uint16_t* idx = R16 + (size_t)g.NS * g.rrows * g.rw;
  uint32_t* part_cost = reinterpret_cast<uint32_t*>(reinterpret_cast<uintptr_t>(idx + (size_t)1024 * F_SUBSETS * F_TH * F_COLS + 31) & ~(uintptr_t)63);
  uint16_t* part_idx = reinterpret_cast<uint16_t*>(part_cost + (size_t)g.J * W * H);
  {
    dim3 gl(g.lrows, g.NS), gr(g.rrows, g.NS);
    pack_left_kernel<<<gl, 256, 0, st>>>(left, vmin, g, L16);
    VWB_LAUNCH_CHECK();
    pack_right_kernel<<<gr, 256, 0, st>>>(right, vmin, g, R16);
    VWB_LAUNCH_CHECK();
  }
  int dev = 0, nsm = 148;
  VWB_CUDA(cudaGetDevice(&dev));
  VWB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
  const int items = g.NS * g.NB * g.J;
  const int grid = items < nsm ? items : nsm;
  const size_t smem = fast_smem_bytes(g);
  void (*kern)(const uint16_t*, const uint16_t*, FastGeom, uint16_t*, vwb200_dispi*, ptrdiff_t, uint32_t*, uint16_t*) = nullptr;
  switch (kx) {
#define KCASE(K) case K: kern = sq ? k1_fast_abs_kernel<K, true> : k1_fast_abs_kernel<K, false>; break;
    KCASE(3) KCASE(5) KCASE(7) KCASE(9) KCASE(11) KCASE(13) KCASE(15) KCASE(17) KCASE(19) KCASE(21) KCASE(23) KCASE(25)
    KCASE(27) KCASE(29) KCASE(31)
#undef KCASE
    default: set_error("k1_fast: unsupported kernel width %d", kx); return VWB200_ENOIMPL;
  }
  VWB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));   // per-function state shared by all host threads: device maximum
  if (ev && ev->e0) cudaEventRecord(ev->e0, st);
  kern<<<grid, F_THREADS, smem, st>>>(L16, R16, g, idx, out, opitch, part_cost, part_idx);
  VWB_LAUNCH_CHECK();
  if (ev && ev->e1) cudaEventRecord(ev->e1, st);
  if (g.J > 1) {
    dim3 mb(32, 8), mg((W + 31) / 32, (H + 7) / 8);
    k1_fast_merge_kernel<<<mg, mb, 0, st>>>(g, part_cost, part_idx, out, opitch);
    VWB_LAUNCH_CHECK();
  }
  dim3 b(32, 8), gg((W + 31) / 32, (H + 7) / 8);
  k1_fast_allequal_fixup<<<gg, b, 0, st>>>(left, right, g, out, opitch);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

}  // namespace vwb200
