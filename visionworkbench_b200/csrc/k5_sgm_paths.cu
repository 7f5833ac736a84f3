// k5_sgm_paths.cu -- path accumulation of SemiGlobalMatcher with a search box per pixel (SURVEY section 8, row a10).
//
// SGM (accum_sgm_multithread, Stereo/SGM.cc:2462-2611; PixelPassTask, SGMAssist.h:691-832; evaluate_path SSE flavour,
// SGM.cc:1014-1141): along each of the 8 directions every pixel lies on exactly one line; a line is a sequential chain.
//   sgm_lines_kernel: ONE WARP PER LINE, lanes = the disparities of the pixel's search box (the common case: <= 32,
//   e.g. the 5 x 5 box around a half-resolution prior).  The previous pixel's path costs stay in registers in the layout of
//   ITS box; the reference scatters them into a full-size array filled with BAD and looks up the 8 adjacent disparities
//   (+ the same one) there -- here that is a 3 x 3 minimum over the intersection with the previous box:
//     min(min8 + P1, centre) == min(min9 + P1, centre)   (P1 > 0, saturating add is monotonic)
//   so the separable form needs 4 shuffles when the box did not move and 6 when it did (the lane then gathers, from the
//   clamped position in the old box, one of {v, row-min3, column-min3, 3x3-min} according to which axis was clamped).
//   min over the previous pixel = one REDUX.  Meta records (16 B), cost bytes and accumulated costs are prefetched
//   PF / 2*PF pixels ahead in registers.  Diagonal lines are wrapped around the image edge (line L owns column
//   (L + t) mod ow of row t and restarts at the edge), which makes all lines equally long and keeps the warps of a CTA on
//   neighbouring pixels of the same row (shared sectors in L1/L2).
//   Boxes with more than 32 disparities (full-search pixels) take a general warp-strided step through a per-warp scratch
//   line in global memory.
// Algorithmic bytes per (pixel, disparity) and direction: 1 (cost) + 2 + 2 (accum read / write); the first direction
// does not read accum.  Per pixel and direction: 16 B meta.
//
// MGM (accum_mgm_multithread, SGM.cc:2619-2700; SmoothPathAccumTask, SGMAssist.h:835-1239): eight sweeps; a pixel's
// path cost is the truncating mean of evaluate_path from TWO predecessors, so a sweep is a wavefront over the image
// (rows, columns or anti-diagonals).  mgm_sweep_kernel: persistent cooperative grid, one grid barrier per wavefront,
// a warp per pixel.
#include "k5_sgm.cuh"
#include <cooperative_groups.h>

namespace vwb200 {
namespace cg = cooperative_groups;

__constant__ unsigned short c_recip[33] = {0, 1024, 512, 342, 256, 205, 171, 147, 128, 114, 103, 94, 86, 79, 74, 69, 64, 61,
                                           57, 54, 52, 49, 47, 45, 43, 41, 40, 38, 37, 36, 35, 34, 32};   // ceil(1024 / w)

struct MetaR { int b0, b1, b2, b3; unsigned start; int val; int n; };
__device__ __forceinline__ MetaR unpack_meta(uint4 q) {
  MetaR m;
  m.b0 = (short)(q.x & 0xffff); m.b1 = (short)(q.x >> 16); m.b2 = (short)(q.y & 0xffff); m.b3 = (short)(q.y >> 16);
  m.start = q.z; m.val = (int)(q.w & 255u); m.n = (int)(q.w >> 8);
  return m;
}
__device__ __forceinline__ unsigned sat_add16(unsigned a, unsigned b) { return min(a + b, 65535u); }
__device__ __forceinline__ unsigned sat_sub16(unsigned a, unsigned b) { return a > b ? a - b : 0u; }

// evaluate_path for one pixel whose box (b, n entries) and whose predecessor's box (pb, pn entries, packed costs in
// prior[]) are arbitrary: warp-strided over the entries.  emit(e, value) receives the path cost of entry e.
template <bool CG, class Emit>
__device__ __forceinline__ void eval_path_general(const MetaR& m, int pb0, int pb1, int pb2, int pb3, int pn, const sgm_accum_t* prior,
                                                  const sgm_cost_t* __restrict__ cost, unsigned p1, unsigned p2_mod, unsigned BAD, int lane,
                                                  Emit emit) {
  unsigned mp = BAD;
  auto ld = [&](int i) -> unsigned { return CG ? (unsigned)__ldcg(prior + i) : (unsigned)prior[i]; };   // CG: written by other SMs
  for (int i = lane; i < pn; i += 32) mp = min(mp, ld(i));
  mp = __reduce_min_sync(0xffffffffu, mp);
  const unsigned dJ = (mp + p2_mod) & 0xffffu;
  const int w = m.b2 - m.b0 + 1, pw = pb2 - pb0 + 1;
  for (int e = lane; e < m.n; e += 32) {
    const int y = e / w, x = e - y * w, X = m.b0 + x, Y = m.b1 + y;
    unsigned nb = BAD, centre = BAD;
    if (pn > 0) {
      const int y0 = max(Y - 1, pb1), y1 = min(Y + 1, pb3), x0 = max(X - 1, pb0), x1 = min(X + 1, pb2);
      for (int yy = y0; yy <= y1; ++yy)
        for (int xx = x0; xx <= x1; ++xx) {
          const unsigned v = ld((yy - pb1) * pw + (xx - pb0));
          nb = min(nb, v);
          if (xx == X && yy == Y) centre = v;
        }
    }
    unsigned res = sat_add16(nb, p1);
    res = min(res, min(centre, dJ));
    res = sat_add16(res, (unsigned)cost[(size_t)m.start + e]);
    emit(e, sat_sub16(res, mp));
  }
}

// ---- the general step: a box with more than 32 disparities is involved (rare: full-search pixels) ---------------------
struct LineState {
  unsigned pv;                 // previous pixel's path cost of this lane's entry (layout of ITS box); BAD = no entry
  int pn;                      // previous pixel's number of entries (0 also stands for "line starts here")
  int pb0, pb1, pb2, pb3;      // previous pixel's box
  int prev_in_buf;             // pn > 32: the previous costs live in bufA
  sgm_accum_t *bufA, *bufB;
};
__device__ __noinline__ void sgm_general_step(LineState* s, uint4 mq, const sgm_cost_t* __restrict__ cost, sgm_accum_t* __restrict__ accum,
                                              unsigned p1, unsigned p2_mod, unsigned BAD, int first_dir, int lane) {
  const MetaR m = unpack_meta(mq);
  if (!s->prev_in_buf) { if (lane < s->pn) s->bufA[lane] = (sgm_accum_t)s->pv; __syncwarp(); }
  sgm_accum_t* bufB = s->bufB;
  eval_path_general<false>(m, s->pb0, s->pb1, s->pb2, s->pb3, s->pn, s->bufA, cost, p1, p2_mod, BAD, lane, [&](int e, unsigned v) {
    bufB[e] = (sgm_accum_t)v;
    const unsigned a0 = first_dir ? 0u : (unsigned)accum[(size_t)m.start + e];
    accum[(size_t)m.start + e] = (sgm_accum_t)(a0 + v);
  });
  __syncwarp();
  s->bufB = s->bufA; s->bufA = bufB;
  s->prev_in_buf = m.n > 32;
  s->pv = (m.n <= 32 && lane < m.n) ? (unsigned)bufB[lane] : BAD;
  s->pn = m.n; s->pb0 = m.b0; s->pb1 = m.b1; s->pb2 = m.b2; s->pb3 = m.b3;
}

__device__ __forceinline__ uint4 lds128(unsigned addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint2 lds64(unsigned addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}

// Per-warp shared-memory rings: 64 meta records (the current and the next 32-pixel epoch; lane i fetches the record of pixel
// 32 * epoch + i two epochs ahead) and DR data slots (cost byte | accumulated cost << 16 of this lane's entry), filled
// DR - 1 pixels ahead through a two-step register delay so that the loads have landed when they are written to the ring.
// The loop is not unrolled: the body is ~90 instructions and the kernel is issue bound, not latency bound.
// A line start is handled as "the previous pixel had no search area": with every predecessor cost = BAD the recurrence
// returns exactly the local cost (BAD + cost - BAD), which is what the reference does for the first pixel (SGMAssist.h:756-759).
// MODE: 0 horizontal lines, 1 vertical, 2 diagonal (wrapped).  FIRST: the first direction writes accum without reading it.
__device__ __forceinline__ unsigned opaque(unsigned v) { asm volatile("mov.u32 %0, %0;" : "+r"(v)); return v; }   // pin in a register
template <class T> __device__ __forceinline__ T* opaque_ptr(T* p) { asm volatile("mov.u64 %0, %0;" : "+l"(p)); return p; }
template <int WARPS, int MODE, bool FIRST>
__global__ void __launch_bounds__(WARPS * 32, 28 / WARPS) sgm_lines_kernel(const SgmMeta* __restrict__ meta, const sgm_cost_t* __restrict__ cost,
                                                               sgm_accum_t* __restrict__ accum, SgmGeom g, int sc, int sr,
                                                               sgm_accum_t* __restrict__ scratch, unsigned scratch_per_warp) {
  constexpr int first_dir = FIRST ? 1 : 0;
  constexpr int DR = 16, P = DR - 1;
  __shared__ unsigned short s_p2mod[256];
  __shared__ uint4 s_ring[WARPS][64];
  __shared__ unsigned s_data[WARPS][DR][32];
  for (unsigned d = threadIdx.x; d < 256; d += blockDim.x) {          // p2_mod as a function of the grey-value step (:1026-1031)
    const unsigned p2u = (unsigned)g.p2 & 0xffffu;                   // (accum_t)p2
    unsigned v = d ? p2u / d : p2u;
    if (v < (unsigned)g.p1) v = (unsigned)g.p1;
    s_p2mod[d] = (unsigned short)v;
  }
  __syncthreads();
  const int lane = (int)opaque(threadIdx.x & 31), wid = threadIdx.x >> 5;
  const int line = blockIdx.x * WARPS + wid;
  constexpr bool horiz = MODE == 0;
  const int ow = g.ow, oh = g.oh;
  const int NL = horiz ? oh : ow, NS = horiz ? ow : oh;
  if (line >= NL) return;
  const unsigned BAD = opaque((unsigned)((255 + g.p2) & 0xffff));    // get_bad_accum_val (SGM.h:240) as accum_t
  const unsigned p1 = opaque((unsigned)g.p1);
  const unsigned ring_s = opaque((unsigned)__cvta_generic_to_shared(&s_ring[wid][0]));
  const unsigned data_s = opaque((unsigned)__cvta_generic_to_shared(&s_data[wid][0][lane]));
  const unsigned p2mod_s = opaque((unsigned)__cvta_generic_to_shared(&s_p2mod[0]));
  const sgm_cost_t* cost_l = opaque_ptr(cost + lane);
  sgm_accum_t* accum_l = opaque_ptr(accum + lane);
  const uint4 MZ = make_uint4(0xffff0000u, 0xffffu, 0u, 0u);         // box (0,0,-1,-1), n = 0

  // pixel of step t on this line: horizontal (line, t) or the wrapped column (line + sc * t) mod ow of row t
  int lc;                                                             // this lane's column cursor for the meta fetches
  if (horiz) lc = sc > 0 ? lane : ow - 1 - lane;
  else { lc = (line + sc * lane) % ow; if (lc < 0) lc += ow; }
  auto fetch_meta = [&](int epoch) -> uint4 {                        // record of step 32 * epoch + lane; advances the cursor by 32 steps
    const int t = 32 * epoch + lane;
    uint4 q = MZ;
    if (t < NS) {
      const int r = horiz ? line : (sr > 0 ? t : oh - 1 - t);
      q = __ldg(reinterpret_cast<const uint4*>(meta) + ((size_t)r * ow + lc));
    }
    lc += 32 * sc;
    if (!horiz) { while (lc >= ow) lc -= ow; while (lc < 0) lc += ow; }
    return q;
  };
  s_ring[wid][lane] = fetch_meta(0);
  s_ring[wid][32 + lane] = fetch_meta(1);
  uint4 mnext = fetch_meta(2);
  __syncwarp();

  auto load_data = [&](int t) -> unsigned {                           // cost | accum << 16 of this lane's entry of the pixel of step t
    const uint2 q = lds64(ring_s + ((t & 63) << 4) + 8);              // (its record is in the meta ring)
    unsigned v = 0u;
    if ((unsigned)lane < (q.y >> 8) && q.y < (33u << 8)) {
      unsigned c, a = 0u;
      asm("ld.global.nc.u8 %0, [%1];" : "=r"(c) : "l"(cost_l + q.x));
      if (!first_dir) asm volatile("ld.global.u16 %0, [%1];" : "=r"(a) : "l"(accum_l + q.x) : "memory");
      v = c | (a << 16);
    }
    return v;
  };
  for (int t = 0; t < P - 2; ++t) asm volatile("st.shared.u32 [%0], %1;" ::"r"(data_s + ((t & (DR - 1)) << 7)), "r"(load_data(t)));
  unsigned d1 = load_data(P - 2), d0 = load_data(P - 1);              // written to the ring at steps 0 and 1

  // chain state (see LineState); x, y, w, h: this lane's position in the previous pixel's box; o?: 0xffff where the
  // neighbour on that side is outside the box (a masked neighbour may read as 0xffff instead of BAD: the result is the
  // same because min(.., centre, dJ) never exceeds BAD < BAD + P1)
  unsigned pv = BAD, pkx = 0xffffffffu, pky = 0xffffffffu;
  int pn = 0, last_val = 0, pb0 = 0, pb1 = 0, pb2 = -1, pb3 = -1, w = 1;
  unsigned oL = 0xffffu, oR = 0xffffu, oU = 0xffffffffu, oD = 0xffffffffu;
  int prev_in_buf = 0;
  sgm_accum_t* bufA = scratch ? scratch + (size_t)line * scratch_per_warp : nullptr;
  sgm_accum_t* bufB = bufA ? bufA + scratch_per_warp / 2 : nullptr;
  // wrapped diagonals: steps until the line reaches the image edge and restarts
  constexpr bool wraps = MODE == 2;
  int to_edge = wraps ? (sc > 0 ? ow - line : line + 1) : 0x7fffffff;

#pragma unroll 1
  for (int t = 0; t < NS; ++t) {
    if ((t & 31) == 0 && t) {              // epoch start: publish the records of the next epoch, start fetching the one after
      s_ring[wid][((t + 32) & 63) + lane] = mnext;
      mnext = fetch_meta((t >> 5) + 2);
      __syncwarp();
    }
    // data ring: the loads issued two steps ago go in, the loads for pixel t + P go out
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(data_s + (((t + P - 2) & (DR - 1)) << 7)), "r"(d1));
    d1 = d0;
    d0 = load_data(t + P);
    const uint4 mq = lds128(ring_s + ((t & 63) << 4));
    unsigned dat;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(dat) : "r"(data_s + ((t & (DR - 1)) << 7)));
    const int n = (int)(mq.w >> 8), val = (int)(mq.w & 255u);
    if (wraps && to_edge == 0) { pv = BAD; pn = 0; prev_in_buf = 0; to_edge = ow; }      // the line restarts at the image edge
    unsigned p2_mod;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(p2_mod) : "r"(p2mod_s + 2u * (unsigned)abs(val - last_val)));
    if (n <= 32 && pn <= 32) {
      // ---------------- register path ----------------
      const unsigned mp = __reduce_min_sync(0xffffffffu, pv);      // lanes without an entry hold BAD
      const unsigned dJ = (mp + p2_mod) & 0xffffu;
      const unsigned vl = __shfl_up_sync(0xffffffffu, pv, 1), vr = __shfl_down_sync(0xffffffffu, pv, 1);
      const unsigned hmin = min(min(vl | oL, pv), vr | oR);
      unsigned nb, centre;
      if (mq.x == pkx && mq.y == pky) {                              // same box as the previous pixel
        const unsigned hu = __shfl_up_sync(0xffffffffu, hmin, w), hd = __shfl_down_sync(0xffffffffu, hmin, w);
        nb = min(min(hu | oU, hmin), hd | oD);
        centre = pv;
      } else {
        const MetaR m = unpack_meta(mq);
        const unsigned q = pv | (hmin << 16);
        const unsigned qu = __shfl_up_sync(0xffffffffu, q, w) | oU, qd = __shfl_down_sync(0xffffffffu, q, w) | oD;
        const unsigned wm = __vimin3_u16x2(qu, q, qd);             // lo: column min3 of v, hi: 3 x 3 min
        const int nw = max(m.b2 - m.b0 + 1, 1), nh = m.b3 - m.b1 + 1;
        const int ny = (lane * (int)c_recip[min(nw, 32)]) >> 10, nx = lane - ny * nw;
        const int X = m.b0 + nx, Y = m.b1 + ny;
        const int sxp = min(max(X, pb0), pb2), syp = min(max(Y, pb1), pb3);
        const int ddx = X - sxp, ddy = Y - syp;
        const int src = ((syp - pb1) * w + (sxp - pb0)) & 31;
        const unsigned g1 = __shfl_sync(0xffffffffu, q, src), g2 = __shfl_sync(0xffffffffu, wm, src);
        const bool reach = pn > 0 && (unsigned)(ddx + 1) <= 2u && (unsigned)(ddy + 1) <= 2u;
        centre = BAD;
        if (!reach) nb = BAD;
        else if (ddx == 0 && ddy == 0) { nb = g2 >> 16; centre = g1 & 0xffffu; }
        else if (ddy == 0) nb = g2 & 0xffffu;
        else if (ddx == 0) nb = g1 >> 16;
        else nb = g1 & 0xffffu;
        // the new box becomes the layout
        pkx = mq.x; pky = mq.y; pb0 = m.b0; pb1 = m.b1; pb2 = m.b2; pb3 = m.b3; w = nw;
        oL = nx > 0 ? 0u : 0xffffu; oR = nx < nw - 1 ? 0u : 0xffffu;
        oU = ny > 0 ? 0u : 0xffffffffu; oD = ny < nh - 1 ? 0u : 0xffffffffu;
      }
      unsigned res = sat_add16(nb, p1);
      res = min(res, min(centre, dJ));
      res = sat_add16(res, dat & 0xffu);
      const unsigned cur = sat_sub16(res, mp);
      pv = BAD;
      if (lane < n) {                                                  // update_accum_buffer, uint16 wrap
        asm volatile("st.global.u16 [%0], %1;" ::"l"(accum_l + mq.z), "r"((dat >> 16) + cur) : "memory");
        pv = cur;
      }
      pn = n;
    } else {
      LineState st{pv, pn, pb0, pb1, pb2, pb3, prev_in_buf, bufA, bufB};
      sgm_general_step(&st, mq, cost, accum, p1, p2_mod, BAD, first_dir, lane);
      pv = st.pv; pn = st.pn; pb0 = st.pb0; pb1 = st.pb1; pb2 = st.pb2; pb3 = st.pb3; prev_in_buf = st.prev_in_buf; bufA = st.bufA; bufB = st.bufB;
      pkx = mq.x; pky = mq.y;
      w = max(pb2 - pb0 + 1, 1);
      const int h = pb3 - pb1 + 1, y = (lane * (int)c_recip[min(w, 32)]) >> 10, x = lane - y * w;
      oL = x > 0 ? 0u : 0xffffu; oR = x < w - 1 ? 0u : 0xffffu;
      oU = y > 0 ? 0u : 0xffffffffu; oD = y < h - 1 ? 0u : 0xffffffffu;
    }
    last_val = val;
    if (wraps) --to_edge;
  }
}

// ---- rows-in-lanes variant: FOUR lines per warp ------------------------------------------------------------------------------
// When no search box of the image is wider or higher than 8 (the regime of config 4 and of every pyramid level below the
// top: boxes of (2 * buffer + 1)^2 around the doubled previous disparity), a lane owns one ROW of its line's box: eight lanes
// = the rows of one line, four lines per warp, and the up-to-8 path costs of a row sit in NR registers as packed u16 pairs.
// Path costs are kept in COMPLEMENT form c = 0x7fff - v, so that "outside the previous box" is simply 0 (shifts and
// out-of-range shuffles fill with zeros) and every minimum becomes a packed maximum:
//   vertical 3-max   : the previous pixel's rows Y-1, Y, Y+1 arrive by three shuffles per register (rows = lanes)
//   horizontal 3-max : 16-bit funnel shifts inside the row + VIMNMX3.U16x2
//   realignment      : the row is shifted by (box.min_x - previous box.min_x) elements when a box moved (64-bit shifts)
//   min over the previous pixel = max of the complements: in-lane, then 3 xor-shuffles inside the 8-lane group
//   recurrence       : __viaddmin_u16x2 / __vimin3_u16x2 on two disparities at a time (no 16-bit overflow: P2 <= 30000)
// 0x7fff instead of BAD for a neighbour outside the box gives the same result as long as the centre is clamped to BAD
// (min(.., centre, dJ) <= BAD < BAD + P1).  Per line-step this issues ~40 instructions instead of ~110.
__device__ __forceinline__ void shift_row(unsigned (&r)[4], int s) {      // r[x] <- r[x + s] (halfword elements), zeros shifted in
  unsigned long long lo = ((unsigned long long)r[1] << 32) | r[0], hi = ((unsigned long long)r[3] << 32) | r[2];
  unsigned long long nlo, nhi;
  if (s >= 0) {
    const int k = 16 * s;
    if (k == 0) { nlo = lo; nhi = hi; }
    else if (k < 64) { nlo = (lo >> k) | (hi << (64 - k)); nhi = hi >> k; }
    else if (k < 128) { nlo = hi >> (k - 64); nhi = 0; }
    else { nlo = 0; nhi = 0; }
  } else {
    const int k = -16 * s;
    if (k < 64) { nhi = (hi << k) | (lo >> (64 - k)); nlo = lo << k; }
    else if (k < 128) { nhi = lo << (k - 64); nlo = 0; }
    else { nlo = 0; nhi = 0; }
  }
  r[0] = (unsigned)nlo; r[1] = (unsigned)(nlo >> 32); r[2] = (unsigned)nhi; r[3] = (unsigned)(nhi >> 32);
}

// Register layout of a row: element 0 is a margin (the column left of the box, always empty), elements 1..w are the box
// columns, so the 3-wide horizontal maximum of the previous row also exists for the column just left and just right of
// the previous box (w <= 6).  The ragged buffers carry 64 entries of padding in front for the margin's loads.
template <int MODE, bool FIRST>
__global__ void __launch_bounds__(64) sgm_rows_kernel(const SgmMeta* __restrict__ meta, const sgm_cost_t* __restrict__ cost,
                                                      sgm_accum_t* __restrict__ accum, SgmGeom g, int sc, int sr) {
  constexpr int WPC = 2, DR = 8, P = DR - 1;
  constexpr unsigned K = 0x7fff7fffu;
  __shared__ unsigned short s_p2mod[256];
  __shared__ uint4 s_meta[WPC][4][64];
  __shared__ uint4 s_data[WPC][DR][32][2];
  for (unsigned d = threadIdx.x; d < 256; d += blockDim.x) {
    const unsigned p2u = (unsigned)g.p2 & 0xffffu;
    unsigned v = d ? p2u / d : p2u;
    if (v < (unsigned)g.p1) v = (unsigned)g.p1;
    s_p2mod[d] = (unsigned short)v;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int gl = lane >> 3, ry = lane & 7;
  constexpr bool horiz = MODE == 0, wraps = MODE == 2;
  const int ow = g.ow, oh = g.oh;
  const int NL = horiz ? oh : ow, NS = horiz ? ow : oh;
  const int line0 = (blockIdx.x * WPC + wid) * 4;
  if (line0 >= NL) return;
  const int line = line0 + gl;
  const unsigned BAD = (unsigned)((255 + g.p2) & 0xffff), BB = BAD * 0x10001u, P1P1 = (unsigned)g.p1 * 0x10001u;
  const uint4 MZ = make_uint4(0xffff0000u, 0xffffu, 0u, 0u);
  const unsigned* cost32 = reinterpret_cast<const unsigned*>(cost);
  const unsigned* accum32 = reinterpret_cast<const unsigned*>(accum);
  // meta fetch: lane i brings the record of step 32 * epoch + i of each of the warp's four lines
  int lc[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (horiz) lc[q] = sc > 0 ? lane : ow - 1 - lane;
    else { lc[q] = (line0 + q + sc * lane) % ow; if (lc[q] < 0) lc[q] += ow; }
  }
  auto fetch_meta = [&](int epoch) {
    const int t = 32 * epoch + lane;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint4 m = MZ;
      if (t < NS && line0 + q < NL) {
        const int r = horiz ? line0 + q : (sr > 0 ? t : oh - 1 - t);
        m = __ldg(reinterpret_cast<const uint4*>(meta) + ((size_t)r * ow + lc[q]));
      }
      s_meta[wid][q][(t & 63)] = m;
      lc[q] += 32 * sc;
      if (!horiz) { while (lc[q] >= ow) lc[q] -= ow; while (lc[q] < 0) lc[q] += ow; }
    }
  };
  fetch_meta(0);
  fetch_meta(1);
  __syncwarp();
  // this lane's row of the pixel of step t, RAW: the three aligned words that hold its cost bytes and the four that hold its
  // accumulated costs (element e = column e - 1).  Nothing here depends on the loaded values -- they rest in registers for
  // two steps, then in the ring, and are only shifted into place (funnel shifts by the row's misalignment) when the step
  // is computed; whatever lies outside the row is masked there.
  auto load_data = [&](int t, uint4& cq, uint4& aq) {
    const uint4 q = s_meta[wid][gl][t & 63];
    const int b0 = (short)(q.x & 0xffff), b1 = (short)(q.x >> 16), b2 = (short)(q.y & 0xffff), b3 = (short)(q.y >> 16);
    const int w = (q.w >> 8) ? b2 - b0 + 1 : 0, h = b3 - b1 + 1;
    cq = make_uint4(0u, 0u, 0u, 0u); aq = cq;
    if (ry < h && w > 0) {
      const long long A = (long long)q.z + (long long)(ry * w) - 1;   // entry of element 0 (the margin; -1 for the very first row:
      const unsigned* cw = cost32 + (A >> 2);                         // the front padding makes it valid)
      cq.x = __ldg(cw); cq.y = __ldg(cw + 1); cq.z = __ldg(cw + 2);
      if (!FIRST) {
        const unsigned* aw = accum32 + (A >> 1);
        aq.x = aw[0]; aq.y = aw[1]; aq.z = aw[2]; aq.w = aw[3];
      }
    }
  };
  uint4 d1c, d1a, d0c, d0a;
  for (int t = 0; t < P - 2; ++t) {
    uint4 c, a;
    load_data(t, c, a);
    s_data[wid][t & (DR - 1)][lane][0] = c;
    s_data[wid][t & (DR - 1)][lane][1] = a;
  }
  load_data(P - 2, d1c, d1a);
  load_data(P - 1, d0c, d0a);

  unsigned pc[4] = {0u, 0u, 0u, 0u};     // previous pixel's path costs of this lane's row, complement form, 0 = no entry
  int pb0 = 0, pb1 = 0, ph = 0, last_val = 0;
  int to_edge = wraps ? (sc > 0 ? ow - line : line + 1) : 0x7fffffff;

#pragma unroll 1
  for (int t = 0; t < NS; ++t) {
    if ((t & 31) == 0 && t) { fetch_meta((t >> 5) + 1); __syncwarp(); }
    // data ring: the loads issued two steps ago go in, the loads for step t + P go out
    s_data[wid][(t + P - 2) & (DR - 1)][lane][0] = d1c;
    s_data[wid][(t + P - 2) & (DR - 1)][lane][1] = d1a;
    d1c = d0c; d1a = d0a;
    load_data(t + P, d0c, d0a);
    const uint4 mq = s_meta[wid][gl][t & 63];
    const uint4 dcq = s_data[wid][t & (DR - 1)][lane][0], daq = s_data[wid][t & (DR - 1)][lane][1];
    const int b0 = (short)(mq.x & 0xffff), b1 = (short)(mq.x >> 16), b2 = (short)(mq.y & 0xffff), b3 = (short)(mq.y >> 16);
    const int n = (int)(mq.w >> 8), val = (int)(mq.w & 255u);
    const int w = n ? b2 - b0 + 1 : 0, h = n ? b3 - b1 + 1 : 0;
    unsigned cst[4], acc[4];
    {   // shift the raw words into place: element e <- entry A + e
      const long long A = (long long)mq.z + (long long)(ry * w) - 1;
      const unsigned sh = (unsigned)(A & 3) * 8u, s2 = (unsigned)(A & 1) * 16u;
      const unsigned B0 = __funnelshift_r(dcq.x, dcq.y, sh), B1 = __funnelshift_r(dcq.y, dcq.z, sh);
      cst[0] = __byte_perm(B0, 0u, 0x4140); cst[1] = __byte_perm(B0, 0u, 0x4342); cst[2] = __byte_perm(B1, 0u, 0x4140); cst[3] = __byte_perm(B1, 0u, 0x4342);
      acc[0] = __funnelshift_r(daq.x, daq.y, s2); acc[1] = __funnelshift_r(daq.y, daq.z, s2);
      acc[2] = __funnelshift_r(daq.z, daq.w, s2); acc[3] = __funnelshift_r(daq.w, 0u, s2);
    }
    if (wraps && to_edge == 0) { pc[0] = pc[1] = pc[2] = pc[3] = 0u; ph = 0; to_edge = ow; }      // the line restarts at the image edge
    const unsigned p2_mod = s_p2mod[abs(val - last_val)];
    // min over the previous pixel (all rows of the group)
    unsigned mx = __vimax3_u16x2(pc[0], pc[1], pc[2]);
    mx = __vimax3_u16x2(mx, pc[3], pc[3]);
    mx = max(mx & 0xffffu, mx >> 16);
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
    const unsigned mp = min(0x7fffu - mx, BAD);
    const unsigned dJ = mp + p2_mod;
    // rows Y - 1, Y, Y + 1 of the previous pixel (Y = this lane's row of the current box)
    const int sy = b1 - pb1, sx = b0 - pb0;
    unsigned v3[4], cr[4];
    {
      const int r0 = ry + sy - 1, r1 = ry + sy, r2 = ry + sy + 1;
      const int base = lane & 24;
      const bool k0 = (unsigned)r0 < (unsigned)ph, k1 = (unsigned)r1 < (unsigned)ph, k2 = (unsigned)r2 < (unsigned)ph;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        unsigned u0 = __shfl_sync(0xffffffffu, pc[j], base | (r0 & 7));
        unsigned u1 = __shfl_sync(0xffffffffu, pc[j], base | (r1 & 7));
        unsigned u2 = __shfl_sync(0xffffffffu, pc[j], base | (r2 & 7));
        if (!k0) u0 = 0u;
        if (!k1) u1 = 0u;
        if (!k2) u2 = 0u;
        v3[j] = __vimax3_u16x2(u0, u1, u2);
        cr[j] = u1;
      }
    }
    // horizontal 3-max inside the row (previous box's columns, with the margins)
    unsigned h9[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const unsigned below = j > 0 ? v3[j - 1] : 0u, above = j < 3 ? v3[j + 1] : 0u;
      const unsigned vl = __funnelshift_l(below, v3[j], 16), vr = __funnelshift_r(v3[j], above, 16);
      h9[j] = __vimax3_u16x2(vl, v3[j], vr);
    }
    if (__any_sync(0xffffffffu, sx != 0)) {      // a box moved sideways: bring the row into the current box's columns
      shift_row(h9, sx);
      shift_row(cr, sx);
    }
    // recurrence on pairs of disparities
    const unsigned dJdJ = dJ * 0x10001u, mpmp = mp * 0x10001u;
    const bool rowok = ry < h;
    sgm_accum_t* arow = accum + (size_t)mq.z + (size_t)(ry * w) - 1;          // entry of element 0
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool e0 = rowok && 2 * j >= 1 && 2 * j <= w, e1 = rowok && 2 * j + 1 <= w;
      const unsigned em = (e0 ? 0xffffu : 0u) | (e1 ? 0xffff0000u : 0u);
      const unsigned nb = K - h9[j];
      const unsigned centre = __vimin3_u16x2(K - cr[j], BB, BB);
      unsigned tt = __viaddmin_u16x2(nb, P1P1, centre);
      tt = __vimin3_u16x2(tt, dJdJ, dJdJ);
      const unsigned cur = tt + (cst[j] & em) - mpmp;
      const unsigned na = __vadd2(acc[j], cur);             // update_accum_buffer: uint16 wrap per entry
      if (e0) arow[2 * j] = (sgm_accum_t)(na & 0xffffu);
      if (e1) arow[2 * j + 1] = (sgm_accum_t)(na >> 16);
      pc[j] = (K - cur) & em;
    }
    pb0 = b0; pb1 = b1; ph = h; last_val = val;
    if (wraps) --to_edge;
  }
}

// One direction: the rows-in-lanes kernel when no box is wider than 6 or higher than 8, else the lane-per-disparity kernel.
static int sgm_direction_launch(bool rows, const SgmMeta* meta, const sgm_cost_t* cost, sgm_accum_t* accum, const SgmGeom& g, int sc, int sr,
                                bool first, sgm_accum_t* scratch, unsigned per_warp, cudaStream_t st) {
  const int lines = sr == 0 ? g.oh : g.ow;
  if (rows) {
    const dim3 grid((lines + 7) / 8), blk(64);
    if (sr == 0) { if (first) sgm_rows_kernel<0, true><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr); else sgm_rows_kernel<0, false><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr); }
    else if (sc == 0) { if (first) sgm_rows_kernel<1, true><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr); else sgm_rows_kernel<1, false><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr); }
    else { if (first) sgm_rows_kernel<2, true><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr); else sgm_rows_kernel<2, false><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr); }
  } else {
    constexpr int WPB = 4;                                             // warps (= neighbouring lines) per CTA
    const dim3 grid((lines + WPB - 1) / WPB), blk(WPB * 32);
    if (sr == 0) { if (first) sgm_lines_kernel<WPB, 0, true><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr, scratch, per_warp); else sgm_lines_kernel<WPB, 0, false><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr, scratch, per_warp); }
    else if (sc == 0) { if (first) sgm_lines_kernel<WPB, 1, true><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr, scratch, per_warp); else sgm_lines_kernel<WPB, 1, false><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr, scratch, per_warp); }
    else { if (first) sgm_lines_kernel<WPB, 2, true><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr, scratch, per_warp); else sgm_lines_kernel<WPB, 2, false><<<grid, blk, 0, st>>>(meta, cost, accum, g, sc, sr, scratch, per_warp); }
  }
  VWB_LAUNCH_CHECK();
  return VWB200_OK;
}

// The eight directions of accum_sgm_multithread (:2462-2611).  A direction is a set of sequential chains -- 4096 lines keep
// a B200 far from full -- and the reference only ever ADDS the per-direction results (uint16, wrapping), so the directions
// are independent: they run FOUR AT A TIME on four streams, each pair of directions into its own partial volume
// (accum[k] receives directions k and k + 4; the first one stores without reading), and the winner-takes-all kernel sums
// the four partial volumes on the fly.
int sgm_paths_launch(const SgmMeta* meta, const sgm_cost_t* cost, sgm_accum_t* const* accum, const SgmGeom& g, unsigned max_n,
                     unsigned max_w, unsigned max_h, Arena& ar, cudaStream_t st) {
  static const int DIRS[8][2] = {{1, 0}, {0, 1}, {1, 1}, {-1, 1}, {-1, 0}, {0, -1}, {1, -1}, {-1, -1}};
  const bool rows = max_w <= 6 && max_h <= 8 && !getenv("VWB200_SGM_LANES_PER_ENTRY");
  const int nlines = std::max(g.ow, g.oh);
  sgm_accum_t* scratch[4] = {nullptr, nullptr, nullptr, nullptr};
  unsigned per_warp = 0;
  if (!rows && max_n > 32) {
    per_warp = 2 * ((max_n + 31u) & ~31u);
    for (int k = 0; k < 4; ++k) VWB_TRY(ar.alloc(&scratch[k], (size_t)per_warp * nlines));
  }
  struct Side { cudaStream_t s = nullptr; cudaEvent_t e = nullptr; ~Side() { if (e) cudaEventDestroy(e); if (s) cudaStreamDestroy(s); } } side[3];
  cudaEvent_t fork;
  VWB_CUDA(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
  struct EvGuard { cudaEvent_t e; ~EvGuard() { cudaEventDestroy(e); } } fg{fork};
  VWB_CUDA(cudaEventRecord(fork, st));
  for (int k = 0; k < 4; ++k) {
    cudaStream_t sk = st;
    if (k > 0) {
      VWB_CUDA(cudaStreamCreateWithFlags(&side[k - 1].s, cudaStreamNonBlocking));
      VWB_CUDA(cudaEventCreateWithFlags(&side[k - 1].e, cudaEventDisableTiming));
      sk = side[k - 1].s;
      VWB_CUDA(cudaStreamWaitEvent(sk, fork, 0));
    }
    VWB_TRY(sgm_direction_launch(rows, meta, cost, accum[k], g, DIRS[k][0], DIRS[k][1], true, scratch[k], per_warp, sk));
    VWB_TRY(sgm_direction_launch(rows, meta, cost, accum[k], g, DIRS[k + 4][0], DIRS[k + 4][1], false, scratch[k], per_warp, sk));
    if (k > 0) VWB_CUDA(cudaEventRecord(side[k - 1].e, sk));
  }
  for (int k = 0; k < 3; ++k) VWB_CUDA(cudaStreamWaitEvent(st, side[k].e, 0));
  return VWB200_OK;
}

// ---- MGM -------------------------------------------------------------------------------------------------------------
struct MgmTask { int p1c, p1r, p2c, p2r, dirx, diry, need_r_gt0, need_r_lt, need_c_gt0, need_c_lt, wf; };
// wf: wavefront index  0: c + r   1: (ow-1-c) + (oh-1-r)   2: r   3: oh-1-r   4: r + (ow-1-c)   5: (oh-1-r) + c   6: ow-1-c   7: c
__constant__ MgmTask c_mgm_tasks[8] = {
    /* L  */ {-1, 0, 0, -1, -1, 0, 1, 0, 1, 0, 0},
    /* R  */ {1, 0, 0, 1, 1, 0, 0, 1, 0, 1, 1},
    /* TL */ {-1, -1, 1, -1, -1, -1, 1, 0, 1, 1, 2},
    /* BR */ {1, 1, -1, 1, 1, 1, 0, 1, 1, 1, 3},
    /* T  */ {0, -1, 1, 0, 0, -1, 1, 0, 0, 1, 4},
    /* B  */ {0, 1, -1, 0, 0, 1, 0, 1, 1, 0, 5},
    /* TR */ {1, -1, 1, 1, 1, -1, 1, 1, 0, 1, 6},
    /* BL */ {-1, 1, -1, -1, -1, 1, 1, 1, 1, 0, 7},
};

__global__ void __launch_bounds__(256) mgm_sweep_kernel(const SgmMeta* __restrict__ meta, const sgm_cost_t* __restrict__ cost,
                                                        sgm_accum_t* __restrict__ accum, sgm_accum_t* path, const uint8_t* __restrict__ left8,
                                                        SgmGeom g, int task) {
  cg::grid_group grid = cg::this_grid();
  const MgmTask t = c_mgm_tasks[task];
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const unsigned BAD = (unsigned)((255 + g.p2) & 0xffff), p1 = (unsigned)g.p1, p2u = (unsigned)g.p2 & 0xffffu;
  const int last_c = g.ow - 1, last_r = g.oh - 1;
  const int nfronts = t.wf < 2 || t.wf == 4 || t.wf == 5 ? g.ow + g.oh - 1 : (t.wf == 2 || t.wf == 3 ? g.oh : g.ow);
  for (int f = 0; f < nfronts; ++f) {
    // pixels of this wavefront: parametrised by k
    int k0 = 0, k1 = 0;                    // k range [k0, k1)
    if (t.wf == 2 || t.wf == 3) { k1 = g.ow; }
    else if (t.wf == 6 || t.wf == 7) { k1 = g.oh; }
    else { k0 = max(0, f - (g.oh - 1)); k1 = min(g.ow - 1, f) + 1; }      // k = column-like coordinate u, v = f - u
    for (int k = k0 + warp; k < k1; k += nwarps) {
      int c, r;
      switch (t.wf) {
        case 0: c = k; r = f - k; break;
        case 1: c = last_c - k; r = last_r - (f - k); break;
        case 2: c = k; r = f; break;
        case 3: c = k; r = last_r - f; break;
        case 4: c = last_c - k; r = f - k; break;
        case 5: c = k; r = last_r - (f - k); break;
        case 6: c = last_c - f; r = k; break;
        default: c = f; r = k; break;
      }
      const size_t pix = (size_t)r * g.ow + c;
      const MetaR m = unpack_meta(__ldg(reinterpret_cast<const uint4*>(meta) + pix));
      if (m.n == 0) continue;
      sgm_accum_t* out = path + m.start;
      const bool ok = (!t.need_r_gt0 || r > 0) && (!t.need_r_lt || r < last_r) && (!t.need_c_gt0 || c > 0) && (!t.need_c_lt || c < last_c);
      if (!ok) {
        for (int e = lane; e < m.n; e += 32) {
          const unsigned v = cost[(size_t)m.start + e];
          out[e] = (sgm_accum_t)v;
          accum[(size_t)m.start + e] = (sgm_accum_t)(accum[(size_t)m.start + e] + v);
        }
        continue;
      }
      // get_path_pixel_diff (SGM.cc:2715-2721) looks at the pixel OPPOSITE to the direction it is given -- kept
      // (it may lie in the kernel padding outside the output area, hence the image and not the meta record)
      const int diff = abs(m.val - (int)left8[(size_t)(r - t.diry + g.min_row) * g.lw + (c - t.dirx + g.min_col)]);
      unsigned p2_mod = diff > 0 ? p2u / (unsigned)diff : p2u;
      if (p2_mod < p1) p2_mod = p1;
      const MetaR q1 = unpack_meta(__ldg(reinterpret_cast<const uint4*>(meta) + ((size_t)(r + t.p1r) * g.ow + (c + t.p1c))));
      const MetaR q2 = unpack_meta(__ldg(reinterpret_cast<const uint4*>(meta) + ((size_t)(r + t.p2r) * g.ow + (c + t.p2c))));
      eval_path_general<true>(m, q1.b0, q1.b1, q1.b2, q1.b3, q1.n, path + q1.start, cost, p1, p2_mod, BAD, lane,
                        [&](int e, unsigned v) { out[e] = (sgm_accum_t)v; });
      __syncwarp();
      eval_path_general<true>(m, q2.b0, q2.b1, q2.b2, q2.b3, q2.n, path + q2.start, cost, p1, p2_mod, BAD, lane, [&](int e, unsigned v) {
        const unsigned mean = ((unsigned)out[e] + v) / 2u;
        out[e] = (sgm_accum_t)mean;
        accum[(size_t)m.start + e] = (sgm_accum_t)(accum[(size_t)m.start + e] + mean);
      });
    }
    __threadfence();
    grid.sync();
  }
}

int mgm_paths_launch(const SgmMeta* meta, const sgm_cost_t* cost, sgm_accum_t* accum, const uint8_t* left8, const SgmGeom& g, size_t total,
                     Arena& ar, cudaStream_t st) {
  sgm_accum_t* path;
  VWB_TRY(ar.alloc(&path, total + 64));
  int dev = 0, sms = 0, per_sm = 0;
  VWB_CUDA(cudaGetDevice(&dev));
  VWB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  VWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mgm_sweep_kernel, 256, 0));
  if (per_sm < 1) { set_error("mgm: the sweep kernel does not fit on an SM"); return VWB200_ECUDA; }
  const int blocks = sms * std::min(per_sm, 4);
  for (int task = 0; task < 8; ++task) {
    SgmGeom gg = g;
    void* args[] = {(void*)&meta, (void*)&cost, (void*)&accum, (void*)&path, (void*)&left8, (void*)&gg, (void*)&task};
    VWB_CUDA(cudaLaunchCooperativeKernel((void*)mgm_sweep_kernel, dim3(blocks), dim3(256), args, 0, st));
    VWB_LAUNCH_CHECK();
  }
  return VWB200_OK;
}

}  // namespace vwb200
