// k5_sgm.cu -- SemiGlobalMatcher on the device (SURVEY section 8, row a10): everything but the path accumulation.
//
// vw::stereo::calc_disparity_sgm (Stereo/SGM.cc:167-230) -> SemiGlobalMatcher::semi_global_matching_func (:2387-2448):
//   u8_convert                       sgm_u8_kernel            HBM bound, 4 B read + 1 B written per pixel
//   census / ternary census          sgm_census_kernel        k*k L1 reads, 8 B written per pixel (Image/CensusTransform.h)
//   populate_disp_bound_image        sgm_rmask_*_kernel, sgm_populate_bounds_kernel   (:241-455)  per-pixel search boxes from
//   constrain_disp_bound_image       sgm_hull_rows_kernel, sgm_hull_cols_kernel       (:502-668)  masks + previous disparity
//   calc_main_buf_size               sgm_count_kernel, sgm_scan_blocks_kernel, sgm_meta_kernel (:677-731) exclusive scan
//   get_hamming_distance_costs       sgm_cost_kernel          1 B written per (pixel, d), ragged (:39-73)
//   accum_sgm / accum_mgm            k5_sgm_paths.cu
//   create_disparity_view[_subpixel] sgm_wta_kernel           2 B read per (pixel, d) (:1159-1346, 1402-1614)
// Everything is integer / bit arithmetic except u8_convert's stretch, the tie smoothing of select_best_disparity and
// the sub-pixel models, which use the reference's double operations one by one.
#include "k5_sgm.cuh"
#include <cmath>
#include <mutex>

namespace vwb200 {

// ---- vw::u8_convert (Image/ImageThresh.h:274-286, Image/Algorithms.h:106-126) --------------------------------------
__global__ void sgm_u8_kernel(ImgF img, const float* __restrict__ stats /* min, max */, uint8_t* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= img.w || y >= img.h) return;
  double mn = (double)stats[0], mx = (double)stats[1];
  if (mx == mn) mx = __dadd_rn(mn, 1.0);
  const float old_min = (float)mn, old_max = (float)mx;
  const double ratio = (old_max == old_min) ? 0.0 : __ddiv_rn(255.0, (double)__fsub_rn(old_max, old_min));
  float v = img.p[(ptrdiff_t)y * img.pitch + x];
  if (v < old_min) v = old_min;
  if (v > old_max) v = old_max;
  const float n = __double2float_rn(__dadd_rn(__dmul_rn((double)__fsub_rn(v, old_min), ratio), 0.0));
  out[(size_t)y * img.w + x] = (uint8_t)n;
}

// ---- census signatures (Image/CensusTransform.h:64-160 binary, :167-340 ternary) ---------------------------------------
__constant__ int c_c9_cols[32] = {0, 4, 8, 1, 3, 5, 7, 2, 4, 6, 1, 4, 7, 0, 2, 3, 5, 6, 8, 1, 4, 7, 2, 4, 6, 1, 3, 5, 7, 0, 4, 8};
__constant__ int c_c9_rows[32] = {0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 3, 3, 3, 4, 4, 4, 4, 4, 4, 5, 5, 5, 6, 6, 6, 7, 7, 7, 7, 8, 8, 8};
__constant__ int c_t7_cols[32] = {0, 2, 3, 4, 6, 1, 3, 5, 0, 2, 3, 4, 6, 0, 1, 2, 4, 5, 6, 0, 2, 3, 4, 6, 1, 3, 5, 0, 2, 3, 4, 6};
__constant__ int c_t7_rows[32] = {0, 0, 0, 0, 0, 1, 1, 1, 2, 2, 2, 2, 2, 3, 3, 3, 3, 3, 3, 4, 4, 4, 4, 4, 5, 5, 5, 6, 6, 6, 6, 6};

// ternary: 2 bits per neighbour: 00 below centre - t, 01 inside the band, 11 above centre + t.  The reference stores the
// signatures in the integer type the binary census of the same kernel needs: the 48-bit ternary 5x5 signature is truncated
// to 32 bits (SGM.cc:1789-1803, ImageView<uint32>) -- kept.
__global__ void sgm_census_kernel(const uint8_t* __restrict__ img, int w, int h, int k, int ternary, int thr,
                                  unsigned long long* __restrict__ out) {
  const int hk = (k - 1) / 2, cw = w - 2 * hk, ch = h - 2 * hk;
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
  if (c >= cw || r >= ch) return;
  const int col = c + hk, row = r + hk;
  const int center = img[(size_t)row * w + col];
  unsigned long long sig = 0;
  if (!ternary) {
    unsigned long long addend = 1;
    if (k == 9) {
      for (int i = 0; i < 32; ++i) {
        if ((int)img[(size_t)(row + c_c9_rows[i] - 4) * w + (col + c_c9_cols[i] - 4)] > center) sig += addend;
        addend *= 2;
      }
    } else {
      for (int rr = row + hk; rr >= row - hk; --rr)
        for (int cc = col + hk; cc >= col - hk; --cc) {
          if (rr == row && cc == col) continue;
          if ((int)img[(size_t)rr * w + cc] > center) sig += addend;
          addend *= 2;
        }
    }
  } else {
    const int lo = center - thr, hi = center + thr;
    int shift = 0;
    auto code = [&](int val) {
      if (val >= lo) sig += (val > hi ? 3ull : 1ull) << shift;
      shift += 2;
    };
    if (k == 9 || k == 7) {
      const int* cs = k == 9 ? c_c9_cols : c_t7_cols;
      const int* rs = k == 9 ? c_c9_rows : c_t7_rows;
      for (int i = 0; i < 32; ++i) code((int)img[(size_t)(row + rs[i] - hk) * w + (col + cs[i] - hk)]);
    } else {
      for (int rr = row + hk; rr >= row - hk; --rr)
        for (int cc = col + hk; cc >= col - hk; --cc) {
          if (rr == row && cc == col) continue;
          if (shift < 64) code((int)img[(size_t)rr * w + cc]);
        }
      if (k == 5) sig &= 0xFFFFFFFFull;
    }
  }
  out[(size_t)r * cw + c] = sig;
}

// ---- populate_disp_bound_image (SGM.cc:241-455) --------------------------------------------------------------------
// extents of the valid right-mask pixels: ext[0] = min_valid_right_row (init rmh - 1), ext[1] = max_valid_right_row (init 0);
// only the first ow columns are looked at and row 0 never counts as a maximum (:303-331, loops kept as they are)
__global__ void sgm_rmask_cols_kernel(ImgB rm, int ow, int* __restrict__ ext) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ow) return;
  for (int i = rm.h - 1; i > 0; --i)
    if (rm.p[(ptrdiff_t)i * rm.pitch + c] > 0) { atomicMax(&ext[1], i); break; }
  for (int i = 0; i < rm.h; ++i)
    if (rm.p[(ptrdiff_t)i * rm.pitch + c] > 0) { atomicMin(&ext[0], i); break; }
}
// per output row: {min_valid_right_column, max_valid_right_column} = {-1, -2} when the row has no valid pixel right of
// column 0 (:343-359); one warp per row
__global__ void sgm_rmask_rows_kernel(ImgB rm, int oh, int2* __restrict__ rowext) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= oh) return;
  const uint8_t* row = rm.p + (ptrdiff_t)r * rm.pitch;
  int max_vc = -2, min_vc = -1;
  for (int base = rm.w - 1; base > 0; base -= 32) {
    const int i = base - lane;
    const unsigned b = __ballot_sync(0xffffffffu, i > 0 && row[i] > 0);
    if (b) { max_vc = base - (__ffs(b) - 1); break; }
  }
  if (max_vc > 0)
    for (int base = 0; base < rm.w; base += 32) {
      const int i = base + lane;
      const unsigned b = __ballot_sync(0xffffffffu, i < rm.w && row[i] > 0);
      if (b) { min_vc = base + (__ffs(b) - 1); break; }
    }
  if (lane == 0) rowext[r] = make_int2(min_vc, max_vc);
}

struct BoundsArgs {
  int ow, oh, sx, sy, buf_x, buf_y;
  const vwb200_dispi* prev; int pw, ph; ptrdiff_t ppitch;
  ImgB lmask, rmask;
  const int* ext; const int2* rowext;
};
__global__ void sgm_populate_bounds_kernel(BoundsArgs a, short4* __restrict__ bounds, uint8_t* __restrict__ full, unsigned* __restrict__ nfull) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
  if (c >= a.ow || r >= a.oh) return;
  const size_t pix = (size_t)r * a.ow + c;
  const short4 ZERO = make_short4(0, 0, -1, -1);
  uint8_t is_full = 0;
  short4 res;
  if (a.lmask.p && a.lmask.p[(ptrdiff_t)r * a.lmask.pitch + c] == 0) {                       // (:372-376)
    res = ZERO;
  } else {
    const bool check_x_edge = a.sx + 1 >= 10, check_y_edge = a.sy + 1 >= 10;                 // (:286-289)
    bool good = false;
    int dxs = 0, dys = 0;
    const int c_in = c / 2, r_in = r / 2;
    if (a.prev && c_in < a.pw && r_in < a.ph) {                                              // (:385-403)
      const vwb200_dispi d = a.prev[(ptrdiff_t)r_in * a.ppitch + c_in];
      dxs = d.dx * 2; dys = d.dy * 2;
      const bool on_edge = (check_x_edge && (dxs <= 0 || dxs >= a.sx)) || (check_y_edge && (dys <= 0 || dys >= a.sy));
      good = d.valid != 0 && !on_edge;
    }
    int b0, b1, b2, b3;
    if (good) {                                                                              // (:407-422)
      b0 = max(dxs - a.buf_x, 0); b2 = min(dxs + a.buf_x, a.sx);
      b1 = max(dys - a.buf_y, 0); b3 = min(dys + a.buf_y, a.sy);
    } else {
      b0 = 0; b1 = 0; b2 = a.sx; b3 = a.sy;
      is_full = 255;
    }
    if (a.rmask.p) {                                                                         // (:431-452)
      const int2 re = a.rowext[r];
      const int v0 = max(re.x - c, b0), v1 = max(a.ext[0] - r, b1), v2 = min(re.y - c, b2), v3 = min(a.ext[1] - r, b3);
      if (v0 > v2 || v1 > v3) { res = ZERO; is_full = 0; }
      else res = make_short4((short)v0, (short)v1, (short)v2, (short)v3);
    } else res = make_short4((short)b0, (short)b1, (short)b2, (short)b3);
  }
  bounds[pix] = res;
  full[pix] = is_full;
  if (is_full && a.prev) atomicAdd(nfull, 1u);      // one counter: "is there anything to constrain"
}

// ---- constrain_disp_bound_image (SGM.cc:502-668): hull of the boxes of the trusted pixels within +-range -----------
// separable: rows first (every pixel), then columns (full-search pixels only).  Sentinel = BBox2i() (empty).
__global__ void sgm_hull_rows_kernel(const short4* __restrict__ bounds, const uint8_t* __restrict__ full, int ow, int oh, int range,
                                     short4* __restrict__ hull) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c >= ow) return;
  int x0 = 32767, y0 = 32767, x1 = -32768, y1 = -32768;
  const int c0 = max(c - range, 0), c1 = min(c + range, ow - 1);
  const size_t row = (size_t)r * ow;
  for (int cs = c0; cs <= c1; ++cs) {
    if (full[row + cs]) continue;
    const short4 v = bounds[row + cs];
    if (v.x == 0 && v.y == 0 && v.z == -1 && v.w == -1) continue;
    x0 = min(x0, (int)v.x); y0 = min(y0, (int)v.y); x1 = max(x1, (int)v.z); y1 = max(y1, (int)v.w);
    // grow(min corner) and grow(max corner): the corners are ordered, so the hull's min comes from the mins
    x0 = min(x0, (int)v.z); y0 = min(y0, (int)v.w); x1 = max(x1, (int)v.x); y1 = max(y1, (int)v.y);
  }
  hull[row + c] = make_short4((short)x0, (short)y0, (short)x1, (short)y1);
}
__global__ void sgm_hull_cols_kernel(const short4* __restrict__ hull, const uint8_t* __restrict__ full, int ow, int oh, int range,
                                     int conserve, int sx, int sy, short4* __restrict__ bounds) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c >= ow) return;
  const size_t pix = (size_t)r * ow + c;
  if (!full[pix]) return;
  int x0 = 32767, y0 = 32767, x1 = -32768, y1 = -32768;
  const int r0 = max(r - range, 0), r1 = min(r + range, oh - 1);
  for (int rs = r0; rs <= r1; ++rs) {
    const short4 v = hull[(size_t)rs * ow + c];
    x0 = min(x0, (int)v.x); y0 = min(y0, (int)v.y); x1 = max(x1, (int)v.z); y1 = max(y1, (int)v.w);
  }
  if (x0 >= x1 || y0 >= y1) {                        // BBox2i::empty(): no estimate (also when all corners coincide in an axis)
    if (conserve > 0) bounds[pix] = make_short4(0, 0, -1, -1);
    return;
  }
  x0 = max(x0 - 2, 0); y0 = max(y0 - 2, 0); x1 = min(x1 + 2, sx); y1 = min(y1 + 2, sy);     // expand(2), crop(max range)
  bounds[pix] = make_short4((short)x0, (short)y0, (short)x1, (short)y1);
}

__global__ void sgm_bounds_from_ints_kernel(const int* __restrict__ in, size_t npix, int sx, int sy, short4* __restrict__ out, int* __restrict__ bad) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const int b0 = in[4 * i], b1 = in[4 * i + 1], b2 = in[4 * i + 2], b3 = in[4 * i + 3];
  if (sgm_box_n(b0, b1, b2, b3) == 0) { out[i] = make_short4(0, 0, -1, -1); return; }
  if (b0 < 0 || b1 < 0 || b2 > sx || b3 > sy) { *bad = 1; out[i] = make_short4(0, 0, -1, -1); return; }
  out[i] = make_short4((short)b0, (short)b1, (short)b2, (short)b3);
}
__global__ void sgm_bounds_to_ints_kernel(const short4* __restrict__ in, size_t npix, int* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const short4 v = in[i];
  out[4 * i] = v.x; out[4 * i + 1] = v.y; out[4 * i + 2] = v.z; out[4 * i + 3] = v.w;
}
__global__ void sgm_fill_bounds_kernel(short4* __restrict__ b, size_t npix, short4 v) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < npix) b[i] = v;
}

// ---- calc_main_buf_size (SGM.cc:677-731): exclusive scan of the box areas -> meta records ---------------------------
static constexpr int SCAN_BLOCK = 1024;      // pixels per block (256 threads x 4)
__device__ __forceinline__ unsigned box_n4(short4 v) { return (unsigned)sgm_box_n(v.x, v.y, v.z, v.w); }

__global__ void __launch_bounds__(256) sgm_count_kernel(const short4* __restrict__ bounds, size_t npix, unsigned long long* __restrict__ block_sums) {
  __shared__ unsigned long long red[8];
  const size_t base = (size_t)blockIdx.x * SCAN_BLOCK + threadIdx.x * 4;
  unsigned long long s = 0;
  for (int i = 0; i < 4; ++i) if (base + i < npix) s += box_n4(bounds[base + i]);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) { unsigned long long t = 0; for (int i = 0; i < 8; ++i) t += red[i]; block_sums[blockIdx.x] = t; }
}
// one CTA: exclusive scan of the block sums in place; totals[0] = total
__global__ void __launch_bounds__(1024) sgm_scan_blocks_kernel(unsigned long long* __restrict__ block_sums, int nblocks, unsigned long long* __restrict__ totals) {
  __shared__ unsigned long long part[1024];
  const int per = (nblocks + 1023) / 1024, b0 = threadIdx.x * per, b1 = min(b0 + per, nblocks);
  unsigned long long s = 0;
  for (int i = b0; i < b1; ++i) s += block_sums[i];
  part[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) { unsigned long long run = 0; for (int i = 0; i < 1024; ++i) { const unsigned long long t = part[i]; part[i] = run; run += t; } totals[0] = run; }
  __syncthreads();
  unsigned long long run = part[threadIdx.x];
  for (int i = b0; i < b1; ++i) { const unsigned long long t = block_sums[i]; block_sums[i] = run; run += t; }
}
__global__ void __launch_bounds__(256) sgm_meta_kernel(const short4* __restrict__ bounds, size_t npix, const unsigned long long* __restrict__ block_offs,
                                                       const uint8_t* __restrict__ left8, SgmGeom g, SgmMeta* __restrict__ meta,
                                                       unsigned* __restrict__ max_n) {
  __shared__ unsigned wsum[8];
  const size_t base = (size_t)blockIdx.x * SCAN_BLOCK + threadIdx.x * 4;
  short4 v[4]; unsigned n[4], s = 0;
  for (int i = 0; i < 4; ++i) {
    v[i] = base + i < npix ? bounds[base + i] : make_short4(0, 0, -1, -1);
    n[i] = base + i < npix ? box_n4(v[i]) : 0u;
    s += n[i];
  }
  unsigned incl = s;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  if (lane == 31) wsum[wid] = incl;
  __syncthreads();
  unsigned woff = 0;
  for (int i = 0; i < wid; ++i) woff += wsum[i];
  unsigned long long run = block_offs[blockIdx.x] + woff + (incl - s);
  unsigned mx = 0, mw = 0, mh = 0;
  for (int i = 0; i < 4; ++i) {
    if (base + i < npix) {
      const size_t pix = base + i;
      const int c = (int)(pix % g.ow), r = (int)(pix / g.ow);
      SgmMeta m;
      m.b0 = v[i].x; m.b1 = v[i].y; m.b2 = v[i].z; m.b3 = v[i].w;
      m.start = (unsigned)run;
      m.val_n = (unsigned)left8[(size_t)(r + g.min_row) * g.lw + (c + g.min_col)] | (n[i] << 8);
      meta[pix] = m;
      mx = max(mx, n[i]);
      if (n[i]) { mw = max(mw, (unsigned)(v[i].z - v[i].x + 1)); mh = max(mh, (unsigned)(v[i].w - v[i].y + 1)); }
    }
    run += n[i];
  }
  for (int o = 16; o > 0; o >>= 1) {
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    mw = max(mw, __shfl_xor_sync(0xffffffffu, mw, o));
    mh = max(mh, __shfl_xor_sync(0xffffffffu, mh, o));
  }
  if (lane == 0 && mx) { atomicMax(max_n, mx); atomicMax(max_n + 1, mw); atomicMax(max_n + 2, mh); }
}

// ---- Hamming costs (get_hamming_distance_costs, SGM.cc:39-73) ---------------------------------------------------------
// one warp per 32 consecutive pixels: lane i fetches record i (coalesced), then the warp walks the 32 pixels with
// lanes = the pixel's disparities (coalesced byte stores into the ragged volume); 4 pixels in flight per iteration
// warps whose 32 pixels all have <= 32 entries are skipped: sgm_cost_lanes_kernel does those
__global__ void __launch_bounds__(256) sgm_cost_kernel(const unsigned long long* __restrict__ lc, const unsigned long long* __restrict__ rc,
                                                       const SgmMeta* __restrict__ meta, SgmGeom g, sgm_cost_t* __restrict__ cost) {
  const int lane = threadIdx.x & 31;
  const size_t npix = (size_t)g.ow * g.oh;
  const size_t p0 = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32;
  if (p0 >= npix) return;
  const size_t mine = p0 + lane;
  uint4 mq = make_uint4(0xffff0000u, 0xffffu, 0u, 0u);
  unsigned long long l = 0;
  int br = 0, bc = 0;
  if (mine < npix) mq = __ldg(reinterpret_cast<const uint4*>(meta) + mine);
  if (!__any_sync(0xffffffffu, (mq.w >> 8) > 32u)) return;
  if (mine < npix) {
    const int c = (int)(mine % g.ow), r = (int)(mine / g.ow);
    br = r + g.min_row - g.hk; bc = c + g.min_col - g.hk;
    l = lc[(size_t)br * g.clw + bc];
  }
  const unsigned lhi = (unsigned)(l >> 32), llo = (unsigned)l;
  for (int j0 = 0; j0 < 32; j0 += 4) {
    unsigned long long v[4]; size_t dst[4]; bool ok[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = j0 + u;
      const unsigned bx = __shfl_sync(0xffffffffu, mq.x, j), by = __shfl_sync(0xffffffffu, mq.y, j);
      const unsigned st = __shfl_sync(0xffffffffu, mq.z, j), n = __shfl_sync(0xffffffffu, mq.w, j) >> 8;
      const int pbr = __shfl_sync(0xffffffffu, br, j), pbc = __shfl_sync(0xffffffffu, bc, j);
      const unsigned long long pl = ((unsigned long long)__shfl_sync(0xffffffffu, lhi, j) << 32) | __shfl_sync(0xffffffffu, llo, j);
      const int b0 = (short)(bx & 0xffff), b1 = (short)(bx >> 16), b2 = (short)(by & 0xffff);
      const int w = max(b2 - b0 + 1, 1);
      ok[u] = (unsigned)lane < n;
      const int y = lane / w, x = lane - y * w;
      dst[u] = (size_t)st + lane;
      v[u] = ok[u] ? (pl ^ rc[(size_t)(pbr + b1 + y) * g.crw + (pbc + b0 + x)]) : 0ull;
      if (n > 32u)                                                     // a large box: finish it warp-strided right here
        for (unsigned e = lane + 32; e < n; e += 32) {
          const int yy = (int)e / w, xx = (int)e - yy * w;
          cost[(size_t)st + e] = (sgm_cost_t)__popcll(pl ^ rc[(size_t)(pbr + b1 + yy) * g.crw + (pbc + b0 + xx)]);
        }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) if (ok[u]) cost[dst[u]] = (sgm_cost_t)__popcll(v[u]);
  }
}

// The common case (every pixel of the warp has <= 32 entries, e.g. the 5x5 boxes of a pyramid level): lane = pixel.  A lane
// walks its own box (the loads of neighbouring lanes fall on neighbouring census words), the costs are staged in shared
// memory at the offsets they have in the ragged volume -- the 32 pixels of a warp own ONE contiguous byte range of it --
// and the range goes out with aligned 4-byte stores.  ~2.7x fewer instructions than the walk above.
__global__ void __launch_bounds__(256) sgm_cost_lanes_kernel(const unsigned long long* __restrict__ lc, const unsigned long long* __restrict__ rc,
                                                             const SgmMeta* __restrict__ meta, SgmGeom g, sgm_cost_t* __restrict__ cost) {
  __shared__ __align__(16) unsigned char stage[8][1040];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t npix = (size_t)g.ow * g.oh;
  const size_t p0 = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32;
  if (p0 >= npix) return;
  const size_t mine = p0 + lane;
  uint4 mq = make_uint4(0xffff0000u, 0xffffu, 0u, 0u);
  if (mine < npix) mq = __ldg(reinterpret_cast<const uint4*>(meta) + mine);
  const unsigned n = mine < npix ? (mq.w >> 8) : 0u;
  if (__any_sync(0xffffffffu, n > 32u)) return;                          // sgm_cost_kernel takes this warp
  const unsigned st0 = __shfl_sync(0xffffffffu, mq.z, 0);                 // pixel p0 always exists
  unsigned end = n ? mq.z + n : st0;
  for (int o = 16; o > 0; o >>= 1) end = max(end, __shfl_xor_sync(0xffffffffu, end, o));
  const unsigned a = st0 & 3u, total = end - st0;                         // <= 1024 bytes
  unsigned char* s = stage[warp];
  if (n) {
    const int c = (int)(mine % g.ow), r = (int)(mine / g.ow);
    const int br = r + g.min_row - g.hk, bc = c + g.min_col - g.hk;
    const unsigned long long l = lc[(size_t)br * g.clw + bc];
    const int b0 = (short)(mq.x & 0xffff), b1 = (short)(mq.x >> 16), b2 = (short)(mq.y & 0xffff);
    const int w = max(b2 - b0 + 1, 1);
    const unsigned long long* rrow = rc + (size_t)(br + b1) * g.crw + (bc + b0);
    unsigned char* d = s + a + (mq.z - st0);
    int x = 0;
    for (unsigned e = 0; e < n; ++e) {
      d[e] = (unsigned char)__popcll(l ^ rrow[x]);
      if (++x == w) { x = 0; rrow += g.crw; }
    }
  }
  __syncwarp();
  unsigned char* gbase = reinterpret_cast<unsigned char*>(cost) + (st0 - a);      // 4-byte aligned (the volume is, and st0 - a is)
  const unsigned nb = a + total, w_lo = a ? 1u : 0u, w_hi = nb >> 2;
  for (unsigned i = w_lo + lane; i < w_hi; i += 32) reinterpret_cast<unsigned*>(gbase)[i] = reinterpret_cast<const unsigned*>(s)[i];
  if (a) for (unsigned b = a + lane; b < min(4u, nb); b += 32) gbase[b] = s[b];                   // head of a partial first word
  for (unsigned b = max(w_hi << 2, w_lo << 2) + lane; b < nb; b += 32) gbase[b] = s[b];          // tail
}

// ---- create_disparity_view / select_best_disparity (SGM.cc:1159-1346) + create_disparity_view_subpixel (:1402-1614) ----
__device__ __forceinline__ double sgm_fit(double x, int mode) {
  const double PI = 3.14159265359;
  const double lin = __ddiv_rn(x, 2.0);
  if (mode == 3) return __ddiv_rn(__dadd_rn(__dmul_rn(__dmul_rn(__dmul_rn(x, x), x), x), x), 4.0);      // poly4Fit
  const double cf = __dsub_rn(1.0, cos(__ddiv_rn(__dmul_rn(x, PI), 3.0)));                               // cosFit
  if (mode == 4) return cf;
  if (mode == 5) {                                                                                        // lcBlendFit
    const double factor = __dsub_rn(1.195, cos(__dmul_rn(x, PI / 2.3)));
    return __dadd_rn(__dmul_rn(cf, factor), __dmul_rn(lin, __dsub_rn(1.0, factor)));
  }
  return lin;
}
__device__ __forceinline__ double sgm_subpixel_offset(int prev, int center, int next, bool left_bound, bool right_bound, int mode) {
  const double ld = (double)(prev - center), rd = (double)(next - center);
  if (rd == 0 && ld == 0) return 0.0;
  if (left_bound) return __dmul_rn(0.5, __ddiv_rn((double)center, (double)next));                  // two_value_subpixel
  if (right_bound) return __dmul_rn(-1.0, __dmul_rn(0.5, __ddiv_rn((double)center, (double)prev)));
  double x = __ddiv_rn(rd, ld), mult = -1.0;
  if (ld < rd) { x = __ddiv_rn(ld, rd); mult = 1.0; }
  return __dmul_rn(__dsub_rn(sgm_fit(x, mode), 0.5), mult);
}
// ParabolaFit2d::find_peak (SGMAssist.h:99-134): the 6x9 pseudo-inverse is stored as FLOAT (Matrix<float,6,9>) and
// multiplied with the double z vector; the raw offset passes through a Vector2f
__constant__ float c_pinv[54];
static const double H_PINV[54] = {
    1.0 / 6, -1.0 / 3, 1.0 / 6, 1.0 / 6, -1.0 / 3, 1.0 / 6, 1.0 / 6, -1.0 / 3, 1.0 / 6,
    1.0 / 6, 1.0 / 6, 1.0 / 6, -1.0 / 3, -1.0 / 3, -1.0 / 3, 1.0 / 6, 1.0 / 6, 1.0 / 6,
    1.0 / 4, 0.0, -1.0 / 4, 0.0, 0.0, 0.0, -1.0 / 4, 0.0, 1.0 / 4,
    -1.0 / 6, 0.0, 1.0 / 6, -1.0 / 6, 0.0, 1.0 / 6, -1.0 / 6, 0.0, 1.0 / 6,
    -1.0 / 6, -1.0 / 6, -1.0 / 6, 0.0, 0.0, 0.0, 1.0 / 6, 1.0 / 6, 1.0 / 6,
    -1.0 / 9, 2.0 / 9, -1.0 / 9, 2.0 / 9, 5.0 / 9, 2.0 / 9, -1.0 / 9, 2.0 / 9, -1.0 / 9};
__device__ __forceinline__ bool sgm_parabola_peak(const double* z, double* dx, double* dy) {
  double vals[6];
  for (int i = 0; i < 6; ++i) {
    double s = 0.0;
    for (int j = 0; j < 9; ++j) s = __dadd_rn(s, __dmul_rn((double)c_pinv[i * 9 + j], z[j]));
    vals[i] = s;
  }
  const double denom = __dsub_rn(__dmul_rn(__dmul_rn(4.0, vals[0]), vals[1]), __dmul_rn(vals[2], vals[2]));
  if (fabs(denom) < 0.01) return false;
  const float ox = (float)__ddiv_rn(__dsub_rn(__dmul_rn(vals[2], vals[4]), __dmul_rn(__dmul_rn(2.0, vals[1]), vals[3])), denom);
  const float oy = (float)__ddiv_rn(__dsub_rn(__dmul_rn(vals[2], vals[3]), __dmul_rn(__dmul_rn(2.0, vals[0]), vals[4])), denom);
  const double sX = 0.34574, sY = 0.38944;
  double x = __ddiv_rn(erf(__ddiv_rn((double)ox, __dmul_rn(sX, sqrt(2.0)))), 2.0);
  double y = __ddiv_rn(erf(__ddiv_rn((double)oy, __dmul_rn(sY, sqrt(2.0)))), 2.0);
  const double nrm = sqrt(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)));
  if (nrm >= 0.5) { const double scale = __ddiv_rn(nrm, 0.5); x = __ddiv_rn(x, scale); y = __ddiv_rn(y, scale); }
  *dx = x; *dy = y;
  return true;
}

// total of the four partial volumes of the concurrent directions (uint16 wrapping adds, like the reference's in-place
// accumulation), 8 entries per thread, into the first volume: HBM bound, 4 x 2 B read + 2 B written per entry
__global__ void __launch_bounds__(256) sgm_sum4_kernel(uint4* __restrict__ a0, const uint4* __restrict__ a1, const uint4* __restrict__ a2,
                                                       const uint4* __restrict__ a3, size_t nvec) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
    uint4 v = a0[i];
    const uint4 x = a1[i], y = a2[i], z = a3[i];
    v.x = __vadd2(__vadd2(v.x, x.x), __vadd2(y.x, z.x)); v.y = __vadd2(__vadd2(v.y, x.y), __vadd2(y.y, z.y));
    v.z = __vadd2(__vadd2(v.z, x.z), __vadd2(y.z, z.z)); v.w = __vadd2(__vadd2(v.w, x.w), __vadd2(y.w, z.w));
    a0[i] = v;
  }
}

// accum = the first partial volume (it receives the totals of the pixels that need them re-read: ties, sub-pixel), a1..a3 =
// the other partial volumes of the concurrent directions (NULL: accum already holds the total)
// staged != 0 (with a1..a3): a warp's 32 consecutive pixels own one contiguous range of the ragged volumes; when every one of
// them has <= 32 entries the warp adds the four partial volumes with coalesced word loads into shared memory and the
// winner / sub-pixel stages read the totals from there (nothing is written back unless a pixel needs the tie smoothing).
__global__ void __launch_bounds__(128) sgm_wta_kernel(sgm_accum_t* __restrict__ accum, const sgm_accum_t* __restrict__ a1,
                                                      const sgm_accum_t* __restrict__ a2, const sgm_accum_t* __restrict__ a3,
                                                      sgm_accum_t* __restrict__ scratch,
                                                      const SgmMeta* __restrict__ meta, SgmGeom g, vwb200_dispi* __restrict__ out,
                                                      ptrdiff_t opitch, int want_sub, int mode, float* __restrict__ out_sub, ptrdiff_t sub_pitch,
                                                      int staged) {
  __shared__ __align__(16) sgm_accum_t tot[4][1024 + 8];
  const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t npix = (size_t)g.ow * g.oh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint4 mq = make_uint4(0xffff0000u, 0xffffu, 0u, 0u);
  if (pix < npix) mq = __ldg(reinterpret_cast<const uint4*>(meta) + pix);
  const int num = pix < npix ? (int)(mq.w >> 8) : 0;
  const sgm_accum_t* tot_vec = nullptr;                                 // != NULL: this pixel's totals in shared memory
  if (staged && a1 && !__any_sync(0xffffffffu, num > 32)) {
    const unsigned st0 = __shfl_sync(0xffffffffu, mq.z, 0);              // the warp's first pixel exists (pix - lane < npix)
    unsigned end = num ? mq.z + (unsigned)num : st0;
    for (int o = 16; o > 0; o >>= 1) end = max(end, __shfl_xor_sync(0xffffffffu, end, o));
    const unsigned a = st0 & 1u, nw = (a + (end - st0) + 1) >> 1;       // words from the even entry st0 - a; <= 513
    const unsigned* w0 = reinterpret_cast<const unsigned*>(accum + (st0 - a));
    const unsigned* w1 = reinterpret_cast<const unsigned*>(a1 + (st0 - a));
    const unsigned* w2 = reinterpret_cast<const unsigned*>(a2 + (st0 - a));
    const unsigned* w3 = reinterpret_cast<const unsigned*>(a3 + (st0 - a));
    unsigned* t = reinterpret_cast<unsigned*>(tot[warp]);
    for (unsigned i = lane; i < nw; i += 32) t[i] = __vadd2(__vadd2(w0[i], w1[i]), __vadd2(w2[i], w3[i]));   // uint16 wrapping sums
    __syncwarp();
    tot_vec = tot[warp] + a + (mq.z - st0);
  }
  if (pix >= npix) return;
  const int oi = (int)(pix % g.ow), oj = (int)(pix / g.ow);
  const int b0 = (short)(mq.x & 0xffff), b1 = (short)(mq.x >> 16), b2 = (short)(mq.y & 0xffff), b3 = (short)(mq.y >> 16);
  vwb200_dispi o;
  float* f = want_sub ? out_sub + (ptrdiff_t)oj * sub_pitch + 3 * oi : nullptr;
  if (num == 0) {                                                       // never valid (:1317-1321)
    o.dx = 0; o.dy = 0; o.valid = 0;
    if (out) out[(ptrdiff_t)oj * opitch + oi] = o;
    if (f) { f[0] = 0.0f; f[1] = 0.0f; f[2] = 0.0f; }
    return;
  }
  sgm_accum_t* accum_vec = accum + mq.z;
  sgm_accum_t* buffer = scratch + mq.z;
  const int width = b2 - b0 + 1, height = b3 - b1 + 1;
  int min_count = 0, min_index = 0;
  unsigned min_val = 65535;
  const bool parts = a1 != nullptr && !tot_vec;
  const bool need_total = parts && want_sub && mode != 0;              // the sub-pixel stage re-reads neighbours of the winner
  for (int i = 0; i < num; ++i) {
    unsigned v = tot_vec ? tot_vec[i] : accum_vec[i];
    if (parts) {                                                        // uint16 wrapping sum, like the reference's in-place adds
      v = (v + a1[mq.z + i] + a2[mq.z + i] + a3[mq.z + i]) & 0xffffu;
      if (need_total) accum_vec[i] = (sgm_accum_t)v;
    }
    if (v == min_val) ++min_count;
    if (v < min_val) { min_index = i; min_val = v; min_count = 1; }
  }
  bool in_global = !tot_vec;                                            // where the totals of this pixel are
  if (min_count > 1) {                                                  // tie smoothing (:1196-1288), rare
    if (tot_vec) { for (int i = 0; i < num; ++i) accum_vec[i] = tot_vec[i]; in_global = true; }
    if (parts && !need_total)
      for (int i = 0; i < num; ++i) accum_vec[i] = (sgm_accum_t)((accum_vec[i] + a1[mq.z + i] + a2[mq.z + i] + a3[mq.z + i]) & 0xffffu);
    for (int i = 0; i < num; ++i) buffer[i] = accum_vec[i];
    sgm_accum_t* input_array = accum_vec;
    sgm_accum_t* output_array = buffer;
    const double third = 1.0 / 3.0;
    int iter_count = 0, index = 0;
    while (min_count > 1) {
      sgm_accum_t* sw = input_array; input_array = output_array; output_array = sw;
      index = 0; min_count = 0; min_val = 65535; min_index = 0;
      for (int row = 0; row < height; ++row)
        for (int col = 0; col < width; ++col) {
          int mn = -1, mx = 1;
          double result = 0.0, weight_total = 0.0;
          if (iter_count < 5) {
            if (mn + col < 0) mn = 0;
            if (mx + col >= width) mx = 0;
            for (int k = mn; k <= mx; ++k) { result = __dadd_rn(result, __dmul_rn((double)input_array[index + k], third)); weight_total = __dadd_rn(weight_total, third); }
          } else {
            if (mn + row < 0) mn = 0;
            if (mx + row >= height) mx = 0;
            for (int k = mn; k <= mx; ++k) { result = __dadd_rn(result, __dmul_rn((double)input_array[index + k * width], third)); weight_total = __dadd_rn(weight_total, third); }
          }
          const unsigned v = (unsigned)(sgm_accum_t)round(__ddiv_rn(result, weight_total));
          if (v == min_val) ++min_count;
          if (v < min_val) { min_index = index; min_val = v; min_count = 1; }
          output_array[index] = (sgm_accum_t)v;
          ++index;
        }
      if (++iter_count >= 6) break;
    }
    if (iter_count > 0 && iter_count % 2 == 0)
      for (int i = 0; i < index; ++i) input_array[i] = output_array[i];
  }
  const int dyi = min_index / width;
  const int dx = min_index - dyi * width + b0, dy = dyi + b1;          // disp_index_to_xy (:2737-2745)
  o.dx = dx; o.dy = dy; o.valid = 1;
  if (out) out[(ptrdiff_t)oj * opitch + oi] = o;
  if (!f) return;
  f[2] = 1.0f;
  if (mode == 0) { f[0] = (float)dx; f[1] = (float)dy; return; }
  int x_left = -1, x_right = 1, y_up = -width, y_down = width;
  bool lb = false, rb = false, tb = false, bb = false;
  if (dx == b0) { x_left = 0; lb = true; }
  if (dx == b2) { x_right = 0; rb = true; }
  if (dy == b1) { y_up = 0; tb = true; }
  if (dy == b3) { y_down = 0; bb = true; }
  const sgm_accum_t* av = in_global ? accum_vec : tot_vec;
  double ddx, ddy;
  if (mode == 1) {                                                      // SUBPIXEL_PARABOLA (:1566-1576)
    double z[9];
    z[0] = av[min_index + x_left + y_up];   z[1] = av[min_index + y_up];   z[2] = av[min_index + x_right + y_up];
    z[3] = av[min_index + x_left];          z[4] = av[min_index];          z[5] = av[min_index + x_right];
    z[6] = av[min_index + x_left + y_down]; z[7] = av[min_index + y_down]; z[8] = av[min_index + x_right + y_down];
    if (!sgm_parabola_peak(z, &ddx, &ddy)) { f[0] = (float)dx; f[1] = (float)dy; return; }
  } else {
    ddx = sgm_subpixel_offset(av[min_index + x_left], av[min_index], av[min_index + x_right], lb, rb, mode);
    ddy = sgm_subpixel_offset(av[min_index + y_up], av[min_index], av[min_index + y_down], tb, bb, mode);
  }
  f[0] = (float)__dadd_rn((double)dx, ddx);
  f[1] = (float)__dadd_rn((double)dy, ddy);
}

// ---- host side -----------------------------------------------------------------------------------------------------
int image_stats_launch(ImgF img, float* d_result3, cudaStream_t st);

int sgm_output_size(int lw, int lh, int rw, int rh, int sx, int sy, int k, int* ow, int* oh) {
  const int hk = (k - 1) / 2;                      // semi_global_matching_func (:2397-2420) with min_disp = 0
  const int min_row = hk, min_col = hk;
  int max_row = std::min(lh - 1 - hk, rh - 1 - (hk + sy));
  int max_col = std::min(lw - 1 - hk, rw - 1 - (hk + sx));
  max_row = std::min(max_row, lh - 1); max_col = std::min(max_col, lw - 1);
  *ow = std::max(0, max_col - min_col + 1); *oh = std::max(0, max_row - min_row + 1);
  return VWB200_OK;
}

// search boxes into d_b (short4 per pixel) + full-search flags; returns the number of full-search pixels with a prior
struct BoundsState { short4* b = nullptr; uint8_t* full = nullptr; short4* hull = nullptr; unsigned nfull = 0; bool derived = false; };

static int bounds_populate(const SgmArgs& a, int ow, int oh, BoundsState& bs, Arena& ar, cudaStream_t st) {
  const size_t npix = (size_t)ow * oh;
  VWB_TRY(ar.alloc(&bs.b, npix));
  if (a.bounds_in) {
    int* d_bad;
    VWB_TRY(ar.alloc(&d_bad, 1));
    VWB_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    sgm_bounds_from_ints_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(a.bounds_in, npix, a.sx, a.sy, bs.b, d_bad);
    VWB_LAUNCH_CHECK();
    int bad = 0;
    VWB_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
    if (bad) { set_error("sgm: a search box lies outside [0, search]"); return VWB200_EARG; }
    return VWB200_OK;
  }
  if (a.lmask.p && (a.lmask.w != ow || a.lmask.h != oh)) { set_error("Left mask size does not match the output size."); return VWB200_ELOGIC; }   // :250-256
  if (a.rmask.p && !(a.rmask.w >= ow + a.sx && a.rmask.h >= oh + a.sy)) {
    set_error("Right mask size is not large enough to support search range.");                                                                      // :262-268
    return VWB200_ELOGIC;
  }
  bs.derived = true;
  VWB_TRY(ar.alloc(&bs.full, npix));
  int* d_ext = nullptr; int2* d_rowext = nullptr; unsigned* d_nfull;
  VWB_TRY(ar.alloc(&d_nfull, 1));
  VWB_CUDA(cudaMemsetAsync(d_nfull, 0, sizeof(unsigned), st));
  if (a.rmask.p) {
    VWB_TRY(ar.alloc(&d_ext, 2));
    VWB_TRY(ar.alloc(&d_rowext, (size_t)oh));
    const int init[2] = {a.rmask.h - 1, 0};
    VWB_CUDA(cudaMemcpyAsync(d_ext, init, sizeof(init), cudaMemcpyHostToDevice, st));
    VWB_CUDA(cudaStreamSynchronize(st));
    sgm_rmask_cols_kernel<<<(ow + 127) / 128, 128, 0, st>>>(a.rmask, ow, d_ext);
    VWB_LAUNCH_CHECK();
    sgm_rmask_rows_kernel<<<(oh + 7) / 8, 256, 0, st>>>(a.rmask, oh, d_rowext);
    VWB_LAUNCH_CHECK();
  }
  BoundsArgs ba{ow, oh, a.sx, a.sy, a.buf_x, a.buf_y, a.prev, a.pw, a.ph, a.ppitch, a.lmask, a.rmask, d_ext, d_rowext};
  sgm_populate_bounds_kernel<<<dim3((ow + 31) / 32, (oh + 7) / 8), dim3(32, 8), 0, st>>>(ba, bs.b, bs.full, d_nfull);
  VWB_LAUNCH_CHECK();
  if (a.prev) {
    VWB_CUDA(cudaMemcpyAsync(&bs.nfull, d_nfull, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
  }
  return VWB200_OK;
}
// one pass of constrain_disp_bound_image at a conservation level.  Re-running it at a higher level on its own output is
// what the reference's retry loop does: trusted pixels never change and every full-search pixel is rewritten (level > 0).
static int bounds_constrain(const SgmArgs& a, int ow, int oh, int level, BoundsState& bs, Arena& ar, cudaStream_t st) {
  if (!bs.derived || !a.prev || bs.nfull == 0) return VWB200_OK;
  const int range = level == 1 ? 25 : (level == 2 ? 3 : (level == 3 ? 0 : 10));
  if (!bs.hull) VWB_TRY(ar.alloc(&bs.hull, (size_t)ow * oh));
  sgm_hull_rows_kernel<<<dim3((ow + 127) / 128, oh), 128, 0, st>>>(bs.b, bs.full, ow, oh, range, bs.hull);
  VWB_LAUNCH_CHECK();
  sgm_hull_cols_kernel<<<dim3((ow + 127) / 128, oh), 128, 0, st>>>(bs.hull, bs.full, ow, oh, range, level, a.sx, a.sy, bs.b);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

struct ScanState { unsigned long long* block_sums = nullptr; unsigned long long* totals = nullptr; int nblocks = 0; };
static int bounds_total(const short4* b, size_t npix, ScanState& ss, unsigned long long* total, Arena& ar, cudaStream_t st) {
  ss.nblocks = (int)((npix + SCAN_BLOCK - 1) / SCAN_BLOCK);
  if (!ss.block_sums) { VWB_TRY(ar.alloc(&ss.block_sums, (size_t)ss.nblocks)); VWB_TRY(ar.alloc(&ss.totals, 2)); }
  sgm_count_kernel<<<ss.nblocks, 256, 0, st>>>(b, npix, ss.block_sums);
  VWB_LAUNCH_CHECK();
  sgm_scan_blocks_kernel<<<1, 1024, 0, st>>>(ss.block_sums, ss.nblocks, ss.totals);
  VWB_LAUNCH_CHECK();
  VWB_CUDA(cudaMemcpyAsync(total, ss.totals, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  VWB_CUDA(cudaStreamSynchronize(st));
  return VWB200_OK;
}
// calc_main_buf_size's memory check (SGM.cc:693-729)
static bool fits_memory(const SgmArgs& a, int ow, int oh, unsigned long long main_buf) {
  if (main_buf < 6) main_buf = 6;
  const double nd = (double)(a.sx + 1) * (a.sy + 1);
  double small_elems;
  if (a.use_mgm) {
    const double v = std::min((double)oh * nd, (double)main_buf), h = std::min((double)ow * nd, (double)main_buf);
    small_elems = v * 4 + h * 4;
  } else {
    const int line = (int)(std::sqrt((double)(ow * ow + oh * oh)) + 1);       // int arithmetic of one_buf_size (SGMAssist.h:565-583)
    small_elems = std::min((double)line * nd, (double)main_buf) * a.assumed_threads;
  }
  const double mb = 1024.0 * 1024.0;
  return (double)main_buf * (3.0 / mb) + small_elems * (2.0 / mb) <= a.memory_limit_mb;
}

// derive the boxes like populate_disp_bound_image incl. its retry loop; returns total entries (or ok = false when even
// the most conservative level does not fit)
static int bounds_derive(const SgmArgs& a, int ow, int oh, BoundsState& bs, ScanState& ss, unsigned long long* total, bool* ok,
                         Arena& ar, cudaStream_t st) {
  const size_t npix = (size_t)ow * oh;
  VWB_TRY(bounds_populate(a, ow, oh, bs, ar, st));
  *ok = true;
  if (!bs.derived) return bounds_total(bs.b, npix, ss, total, ar, st);
  if (a.conserve_level >= 0) {
    VWB_TRY(bounds_constrain(a, ow, oh, a.conserve_level, bs, ar, st));
    return bounds_total(bs.b, npix, ss, total, ar, st);
  }
  for (int level = 0; level <= 3; ++level) {
    VWB_TRY(bounds_constrain(a, ow, oh, level, bs, ar, st));
    VWB_TRY(bounds_total(bs.b, npix, ss, total, ar, st));
    if (fits_memory(a, ow, oh, *total)) return VWB200_OK;
  }
  *ok = false;
  return VWB200_OK;
}

int sgm_bounds_run(const SgmArgs& a, int ow, int oh, int* d_bounds, Arena& ar, cudaStream_t st) {
  if (a.sx > 32767 || a.sy > 32767) { set_error("sgm: search range exceeds 32767"); return VWB200_ENOIMPL; }
  BoundsState bs; ScanState ss; unsigned long long total = 0; bool ok = true;
  VWB_TRY(bounds_derive(a, ow, oh, bs, ss, &total, &ok, ar, st));
  const size_t npix = (size_t)ow * oh;
  sgm_bounds_to_ints_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(bs.b, npix, d_bounds);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

int sgm_run(const SgmArgs& a, Arena& /*callers_arena*/, cudaStream_t st) {
  Arena ar(st);                 // everything allocated here is released (stream-ordered) when the call returns
  const int k = a.k;
  if (k != 3 && k != 5 && k != 7 && k != 9) {
    set_error("Census transforms are only available in size 3, 5, 7, and 9.");       // SGM.cc:1885-1888
    return VWB200_ENOIMPL;
  }
  if (a.sx < 0 || a.sy < 0) { set_error("sgm: negative search volume"); return VWB200_EARG; }
  if (a.sx > 32767 || a.sy > 32767) { set_error("sgm: search range exceeds 32767"); return VWB200_ENOIMPL; }
  int p1 = a.p1, p2 = a.p2;
  if (p1 <= 0) p1 = a.ternary ? (k == 3 ? 12 : k == 5 ? 30 : 40) : (k == 3 ? 3 : k == 5 ? 15 : k == 7 ? 30 : 20);            // set_parameters (:106-130)
  if (p2 <= 0) p2 = a.ternary ? (k == 3 ? 600 : k == 5 ? 1500 : 2000) : (k == 3 ? 70 : k == 5 ? 750 : k == 7 ? 1500 : 1000);   // (:135-157)
  SgmGeom g;
  g.sx = a.sx; g.sy = a.sy; g.ndx = a.sx + 1; g.ndy = a.sy + 1;
  const long long nd = (long long)g.ndx * g.ndy;
  if (nd > (1ll << 24) - 1) { set_error("Number of disparities is too large for data type."); return VWB200_ENOIMPL; }       // (:102-103)
  g.nd = (int)nd; g.p1 = p1; g.p2 = p2;
  g.hk = (k - 1) / 2; g.min_col = g.hk; g.min_row = g.hk; g.lw = a.left.w;
  sgm_output_size(a.left.w, a.left.h, a.right.w, a.right.h, a.sx, a.sy, k, &g.ow, &g.oh);
  if (g.ow <= 0 || g.oh <= 0) return VWB200_OK;
  g.clw = a.left.w - 2 * g.hk; g.crw = a.right.w - 2 * g.hk;
  const size_t npix = (size_t)g.ow * g.oh;
  if (p1 > p2 || p2 > 30000) {     // the kernels rely on every path cost staying <= 255 + P2 (no uint16 wrap in dJ)
    set_error("sgm: penalties outside the supported range (need p1 <= p2 <= 30000), got p1 = %d, p2 = %d", p1, p2);
    return VWB200_ENOIMPL;
  }
  {
    static float pf[54];
    static std::once_flag pinv_once;
    std::call_once(pinv_once, [] { for (int i = 0; i < 54; ++i) pf[i] = (float)H_PINV[i]; });
    VWB_CUDA(cudaMemcpyToSymbolAsync(c_pinv, pf, sizeof(pf), 0, cudaMemcpyHostToDevice, st));
  }
  // u8 stretch + census signatures
  uint8_t *l8, *r8; unsigned long long *lc, *rc; float* stats;
  VWB_TRY(ar.alloc(&l8, (size_t)a.left.w * a.left.h));
  VWB_TRY(ar.alloc(&r8, (size_t)a.right.w * a.right.h));
  VWB_TRY(ar.alloc(&lc, (size_t)a.left.w * a.left.h));
  VWB_TRY(ar.alloc(&rc, (size_t)a.right.w * a.right.h));
  VWB_TRY(ar.alloc(&stats, 8));
  const dim3 b(32, 8);
  VWB_TRY(image_stats_launch(a.left, stats, st));
  VWB_TRY(image_stats_launch(a.right, stats + 3, st));
  sgm_u8_kernel<<<dim3((a.left.w + 31) / 32, (a.left.h + 7) / 8), b, 0, st>>>(a.left, stats, l8);
  VWB_LAUNCH_CHECK();
  sgm_u8_kernel<<<dim3((a.right.w + 31) / 32, (a.right.h + 7) / 8), b, 0, st>>>(a.right, stats + 3, r8);
  VWB_LAUNCH_CHECK();
  sgm_census_kernel<<<dim3((g.clw + 31) / 32, (a.left.h - 2 * g.hk + 7) / 8), b, 0, st>>>(l8, a.left.w, a.left.h, k, a.ternary, a.ternary_threshold, lc);
  VWB_LAUNCH_CHECK();
  sgm_census_kernel<<<dim3((g.crw + 31) / 32, (a.right.h - 2 * g.hk + 7) / 8), b, 0, st>>>(r8, a.right.w, a.right.h, k, a.ternary, a.ternary_threshold, rc);
  VWB_LAUNCH_CHECK();
  // search boxes -> ragged layout
  BoundsState bs; ScanState ss; unsigned long long total = 0; bool ok = true;
  VWB_TRY(bounds_derive(a, g.ow, g.oh, bs, ss, &total, &ok, ar, st));
  if (a.bounds_out) {
    sgm_bounds_to_ints_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(bs.b, npix, a.bounds_out);
    VWB_LAUNCH_CHECK();
  }
  auto all_invalid = [&]() -> int {                                    // (:2430-2436)
    if (a.out) VWB_CUDA(cudaMemset2DAsync(a.out, (size_t)a.opitch * sizeof(vwb200_dispi), 0, (size_t)g.ow * sizeof(vwb200_dispi), g.oh, st));
    if (a.out_sub) VWB_CUDA(cudaMemset2DAsync(a.out_sub, (size_t)a.sub_pitch * 4, 0, (size_t)g.ow * 12, g.oh, st));
    return VWB200_OK;
  };
  if (!ok) return all_invalid();
  if (total > 0xFFFFFFF0ull) {
    set_error("SGM: %llu (pixel, disparity) entries exceed the 2^32 this engine indexes; reduce the search range or the tile", total);
    return VWB200_ENOMEM;
  }
  if (total == 0) return all_invalid();
  SgmMeta* meta; unsigned* d_maxn; sgm_cost_t* cost; sgm_accum_t *accum, *scratch;
  sgm_accum_t* parts[4] = {nullptr, nullptr, nullptr, nullptr};
  VWB_TRY(ar.alloc(&meta, npix));
  VWB_TRY(ar.alloc(&d_maxn, 4));          // max entries, max box width, max box height
  VWB_CUDA(cudaMemsetAsync(d_maxn, 0, 4 * sizeof(unsigned), st));
  sgm_meta_kernel<<<ss.nblocks, 256, 0, st>>>(bs.b, npix, ss.block_sums, l8, g, meta, d_maxn);
  VWB_LAUNCH_CHECK();
  unsigned maxes[4] = {0, 0, 0, 0};
  VWB_CUDA(cudaMemcpyAsync(maxes, d_maxn, sizeof(maxes), cudaMemcpyDeviceToHost, st));
  // 64 entries of padding in front of and behind the ragged volumes (the rows-in-lanes kernel fetches rows with aligned
  // word loads that may start one entry early and end a few entries late)
  VWB_TRY(ar.alloc(&cost, (size_t)total + 192));
  VWB_TRY(ar.alloc(&accum, (size_t)total + 192));
  VWB_TRY(ar.alloc(&scratch, (size_t)total + 64));
  VWB_CUDA(cudaMemsetAsync(cost, 0, 64, st));
  VWB_CUDA(cudaMemsetAsync(accum, 0, 64 * sizeof(sgm_accum_t), st));
  cost += 64; accum += 64;
  parts[0] = accum;
  const int naccum = a.use_mgm ? 1 : 4;       // partial volumes of the concurrent SGM directions; MGM sums into accum
  for (int k = 1; k < naccum; ++k) {
    VWB_TRY(ar.alloc(&parts[k], (size_t)total + 192));
    VWB_CUDA(cudaMemsetAsync(parts[k], 0, 64 * sizeof(sgm_accum_t), st));
    parts[k] += 64;
  }
  static_assert(sizeof(sgm_cost_t) == 1, "the staged copy moves bytes");
  sgm_cost_lanes_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(lc, rc, meta, g, cost);
  VWB_LAUNCH_CHECK();
  sgm_cost_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(lc, rc, meta, g, cost);
  VWB_LAUNCH_CHECK();
  VWB_CUDA(cudaStreamSynchronize(st));                                  // max_n
  if (a.use_mgm) {
    VWB_CUDA(cudaMemsetAsync(accum, 0, ((size_t)total + 64) * sizeof(sgm_accum_t), st));
    VWB_TRY(mgm_paths_launch(meta, cost, accum, l8, g, (size_t)total, ar, st));
  } else {
    VWB_TRY(sgm_paths_launch(meta, cost, parts, g, maxes[0], maxes[1], maxes[2], ar, st));
  }
  const bool fused_wta = naccum == 4 && maxes[0] <= 32;   // every pixel has <= 32 entries
  if (naccum == 4 && !fused_wta) {
    const size_t nvec = ((size_t)total + 7) / 8;              // the volumes are 16-byte aligned and padded
    sgm_sum4_kernel<<<148 * 8, 256, 0, st>>>(reinterpret_cast<uint4*>(accum), reinterpret_cast<const uint4*>(parts[1]),
                                             reinterpret_cast<const uint4*>(parts[2]), reinterpret_cast<const uint4*>(parts[3]), nvec);
    VWB_LAUNCH_CHECK();
  }
  sgm_wta_kernel<<<(unsigned)((npix + 127) / 128), 128, 0, st>>>(accum, fused_wta ? parts[1] : nullptr, fused_wta ? parts[2] : nullptr,
                                                                 fused_wta ? parts[3] : nullptr, scratch, meta, g, a.out, a.opitch,
                                                                 a.out_sub != nullptr, a.subpixel_mode, a.out_sub, a.sub_pitch, fused_wta ? 1 : 0);
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

}  // namespace vwb200
