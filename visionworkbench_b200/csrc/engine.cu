// engine.cu -- host side of the vwb200 engine: error plumbing, the extern "C" ABI of
// include/vwb200.h, and the per-tile level loop of PyramidCorrelationView::prerasterize
// (behaviour of Stereo/CorrelationView.cc:273-886, block-matching branch) driving the CUDA kernels.
//
// Everything here is re-entrant: no mutable globals except the launch counter; each rasterize call
// owns a stream and stream-ordered allocations (VW calls prerasterize concurrently from its tile
// thread pool, Image/ImageIO.h:228-235).
#include "common.cuh"
#include <chrono>
#include "k5_sgm.cuh"
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <algorithm>
#include <mutex>
#include <vector>

namespace vwb200 {

std::atomic<long long> g_launches{0};
static thread_local char t_error[512] = "";
static thread_local vwb200_k1_stats t_k1_stats = {0, 0, 0.0f, 0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_error, sizeof(t_error), fmt, ap);
  va_end(ap);
}

int ensure_device() {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    set_error("no CUDA device available (%s); the vwb200 engine has no CPU path",
              e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    cudaGetLastError();
    return VWB200_ENODEVICE;
  }
  // keep stream-ordered allocations cached in the pool between calls (the default threshold of 0
  // returns the memory to the driver at every synchronisation: ~100 ms per call at 8K x 8K)
  static std::atomic<unsigned long long> configured{0};
  int dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess && dev < 64 && !(configured.load() & (1ull << dev))) {
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      unsigned long long thr = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    configured.fetch_or(1ull << dev);
  }
  return VWB200_OK;
}

int zone_post_launch(const Tile* d_tiles, int ntiles, const Zone* d_zones, const Zone* d_rlzones, const int2* d_post_add,
                     vwb200_dispi* disp, const vwb200_dispi* rl, float thr, int tile_w, int tile_h, cudaStream_t st, float* diff = nullptr,
                     ptrdiff_t dpitch = 0, int dox = 0, int doy = 0);

// ---------------------------------------------------------------------------------------------------
// small RAII helpers: stream-ordered device buffers, an owned-or-borrowed stream
// ---------------------------------------------------------------------------------------------------
struct StreamGuard {
  cudaStream_t st = nullptr; bool own = false;
  // device-resident inputs are produced on the caller's stream: a NULL stream then means the legacy default stream
  // (which is what e.g. torch's default stream is), never a private one -- otherwise the kernels could start before the
  // producer of their inputs has finished.  Host-resident calls with no stream get a private non-blocking stream.
  int init(void* user, int device_resident = 0) {
    if (user) { st = static_cast<cudaStream_t>(user); return VWB200_OK; }
    if (device_resident) { st = cudaStreamLegacy; return VWB200_OK; }
    VWB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    own = true;
    return VWB200_OK;
  }
  ~StreamGuard() { if (own && st) cudaStreamDestroy(st); }
};

static void make_tiles(const std::vector<Zone>& zones, int tile_w, int tile_h, std::vector<Tile>& tiles, bool with_chunks) {
  tiles.clear();
  for (size_t zi = 0; zi < zones.size(); ++zi)
    for (int c = 0; c < (with_chunks ? zones[zi].nchunks : 1); ++c)
      for (int ty = 0; ty < zones[zi].h; ty += tile_h)
        for (int tx = 0; tx < zones[zi].w; tx += tile_w) tiles.push_back(Tile{(int)zi, tx, ty, c});
}

// ---------------------------------------------------------------------------------------------------
// K1 dispatch for one batch of zones (generic path).  NCC maps are built over the bounding domain of
// the window origins the zones touch.
// ---------------------------------------------------------------------------------------------------
static int run_k1_zones(int cost, ImgF left, ImgF right, std::vector<Zone> zones, int kx, int ky,
                        vwb200_dispi* d_out, Arena& ar, cudaStream_t st, const Zone** d_zones_out = nullptr,
                        const Tile** d_tiles_out = nullptr, int* ntiles_out = nullptr, const KEvents* ev = nullptr,
                        const std::vector<char>* skip = nullptr, const ZoneIntMode* zim = nullptr) {
  if (zones.empty()) { if (ntiles_out) *ntiles_out = 0; return VWB200_OK; }
  // integer-valued imagery (level 0 of 8-bit rasters): the int32 warp-per-tile kernel takes every zone whose search patch fits
  int ib = 0;
  const bool int_mode = zim && zim->on && !getenv("VWB200_NO_ZONE_INT") &&
                        k1_zone_int_supported(cost, kx, ky, (long long)zim->vmax - (long long)zim->vmin, &ib);
  std::vector<char> zint(zones.size(), 0);
  // split the disparity range of zones with many disparities over several CTAs (load balance: a zone whose
  // range was reset to the full search window would otherwise be one CTA's serial loop)
  std::vector<int> split;
  long long scratch_elems = 0;
  bool clamp_reads = false;
  for (size_t zi = 0; zi < zones.size(); ++zi) {
    Zone& z = zones[zi];
    const int nd = z.sx * z.sy;
    const bool skipped = skip && (*skip)[zi];
    z.nchunks = skipped ? 1 : (nd + K1G_DCHUNK - 1) / K1G_DCHUNK;     // zones the fast kernel took are not ours
    if (int_mode && !skipped) {
      const int nci = (nd + (1 << ib) - 1) >> ib;
      if (k1_zone_int_stage_u16(kx, z.sx, z.sy, nci, ib) <= k1_zone_int_stage_max() &&
          (nci == 1 || (long long)z.w * z.h * nci < (1ll << 29))) { zint[zi] = 1; z.nchunks = nci; }
    }
    z.sbase = 0;
    if (z.nchunks > 1 && (long long)z.w * z.h * z.nchunks < (1ll << 29)) {
      z.sbase = scratch_elems; scratch_elems += (long long)z.nchunks * z.w * z.h; split.push_back((int)zi);
    } else z.nchunks = 1;
    if (z.lx < 0 || z.ly < 0 || z.lx + z.w + kx - 1 > left.w || z.ly + z.h + ky - 1 > left.h ||
        z.rx < 0 || z.ry < 0 || z.rx + z.w + kx - 1 + z.sx - 1 > right.w || z.ry + z.h + ky - 1 + z.sy - 1 > right.h) clamp_reads = true;
  }
  std::vector<Tile> tiles, tiles_post, tiles_int;
  make_tiles(zones, k1_generic_tile_w(kx), k1_generic_tile_h(ky), tiles, true);
  tiles.erase(std::remove_if(tiles.begin(), tiles.end(), [&](const Tile& t) { return (skip && (*skip)[t.zone] != 0) || zint[t.zone]; }), tiles.end());
  // zone-int tiles: balanced split of each zone (the kernel derives the tile size from the zone with the same formula),
  // in up to three launches by the size of the staged right patch, heaviest tiles first inside a launch
  static constexpr long long ZI_CLS[2] = {3072, 12288};
  int ni_cls[3] = {0, 0, 0};
  long long ri_max[3] = {0, 0, 0};
  if (int_mode) {
    const int TW = k1_zone_int_tile_w(kx), TH = k1_zone_int_tile_h();
    for (size_t zi = 0; zi < zones.size(); ++zi) {
      if (!zint[zi]) continue;
      const Zone& z = zones[zi];
      const int ntx = (z.w + TW - 1) / TW, twb = (z.w + ntx - 1) / ntx, nty = (z.h + TH - 1) / TH, thb = (z.h + nty - 1) / nty;
      for (int c = 0; c < z.nchunks; ++c)
        for (int ty = 0; ty < z.h; ty += thb)
          for (int tx = 0; tx < z.w; tx += twb) tiles_int.push_back(Tile{(int)zi, tx, ty, c});
    }
    auto need = [&](const Tile& t) { const Zone& z = zones[t.zone]; return k1_zone_int_stage_u16(kx, z.sx, z.sy, z.nchunks, ib); };
    auto icls = [&](const Tile& t) { const long long n = need(t); return n <= ZI_CLS[0] ? 0 : (n <= ZI_CLS[1] ? 1 : 2); };
    auto work = [&](const Tile& t) {
      const Zone& z = zones[t.zone];
      const int nd = z.sx * z.sy;
      return z.nchunks > 1 ? std::min(1 << ib, nd - (t.chunk << ib)) : nd;
    };
    std::stable_sort(tiles_int.begin(), tiles_int.end(), [&](const Tile& a, const Tile& b) {
      const int ca = icls(a), cb = icls(b);
      return ca != cb ? ca < cb : work(a) > work(b);
    });
    for (const Tile& t : tiles_int) { const int c = icls(t); ++ni_cls[c]; ri_max[c] = std::max(ri_max[c], need(t)); }
  }
  // three launches: tiles with a small right search patch (staged; little shared memory -> 2-3 CTAs per SM), tiles with
  // a large one (staged, 1 CTA per SM), and tiles whose patch does not fit (reads through L1)
  static constexpr long long SMALL_R = 6144;
  auto cls = [&](const Tile& t) {
    const Zone& z = zones[t.zone];
    const long long f = k1_generic_stage_floats(kx, ky, z.sx, z.sy, z.nchunks);
    return !k1_generic_can_stage(kx, ky, z.sx, z.sy, z.nchunks) ? 2 : (f <= SMALL_R ? 0 : 1);
  };
  std::stable_sort(tiles.begin(), tiles.end(), [&](const Tile& a, const Tile& b) { return cls(a) < cls(b); });
  int n_cls[3] = {0, 0, 0};
  long long r_max[3] = {0, 0, 0};
  for (const Tile& t : tiles) {
    const int c = cls(t);
    const Zone& z = zones[t.zone];
    ++n_cls[c];
    r_max[c] = std::max(r_max[c], k1_generic_stage_floats(kx, ky, z.sx, z.sy, z.nchunks));
  }
  Zone* d_zones; Tile* d_tiles;
  double* d_sc = nullptr; int* d_si = nullptr; int* d_split = nullptr;
  if (!split.empty()) {
    VWB_TRY(ar.alloc(&d_sc, (size_t)scratch_elems)); VWB_TRY(ar.alloc(&d_si, (size_t)scratch_elems)); VWB_TRY(ar.alloc(&d_split, split.size()));
    VWB_CUDA(cudaMemcpyAsync(d_split, split.data(), split.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  }
  VWB_TRY(ar.alloc(&d_zones, zones.size()));
  VWB_TRY(ar.alloc(&d_tiles, tiles.size() + 1));
  VWB_CUDA(cudaMemcpyAsync(d_zones, zones.data(), zones.size() * sizeof(Zone), cudaMemcpyHostToDevice, st));
  if (!tiles.empty()) VWB_CUDA(cudaMemcpyAsync(d_tiles, tiles.data(), tiles.size() * sizeof(Tile), cudaMemcpyHostToDevice, st));
  bool ev_used = false;
  std::vector<Tile> tiles_gated;
  const NccMaps no_ncc = {};
  if (!tiles_int.empty()) {
    Tile* d_ti; int* d_flag;
    VWB_TRY(ar.alloc(&d_ti, tiles_int.size()));
    VWB_TRY(ar.alloc(&d_flag, zones.size()));
    VWB_CUDA(cudaMemcpyAsync(d_ti, tiles_int.data(), tiles_int.size() * sizeof(Tile), cudaMemcpyHostToDevice, st));
    VWB_CUDA(cudaMemsetAsync(d_flag, 0, zones.size() * sizeof(int), st));
    int off = 0;
    for (int c = 0; c < 3; ++c) {
      if (!ni_cls[c]) continue;
      VWB_TRY(k1_zone_int_launch(cost, left, right, d_zones, d_ti + off, ni_cls[c], kx, zim->vmin, zim->vmax, (int)ri_max[c], d_out, d_sc, d_si,
                                 d_flag, st, ev_used ? nullptr : ev));
      ev_used = true;
      off += ni_cls[c];
    }
    if (zim->checked) {
      // zones that met a mean-filled (non-integer) pixel: the fp64 kernel over the tiles of every integer zone, gated by the flag
      make_tiles(zones, k1_generic_tile_w(kx), k1_generic_tile_h(ky), tiles_gated, true);
      tiles_gated.erase(std::remove_if(tiles_gated.begin(), tiles_gated.end(), [&](const Tile& t) { return !zint[t.zone]; }), tiles_gated.end());
      std::stable_sort(tiles_gated.begin(), tiles_gated.end(), [&](const Tile& a, const Tile& b) { return cls(a) < cls(b); });
      int ng[3] = {0, 0, 0};
      long long rg[3] = {0, 0, 0};
      for (const Tile& t : tiles_gated) {
        const int c = cls(t);
        const Zone& z = zones[t.zone];
        ++ng[c];
        rg[c] = std::max(rg[c], k1_generic_stage_floats(kx, ky, z.sx, z.sy, z.nchunks));
      }
      Tile* d_tg;
      VWB_TRY(ar.alloc(&d_tg, tiles_gated.size()));
      VWB_CUDA(cudaMemcpyAsync(d_tg, tiles_gated.data(), tiles_gated.size() * sizeof(Tile), cudaMemcpyHostToDevice, st));
      int goff = 0;
      for (int c = 0; c < 3; ++c) {
        if (!ng[c]) continue;
        VWB_TRY(k1_generic_launch(cost, left, right, d_zones, d_tg + goff, ng[c], kx, ky, no_ncc, d_out, d_sc, d_si, clamp_reads,
                                  c == 2 ? 0 : (int)rg[c], st, nullptr, d_flag));
        goff += ng[c];
      }
    }
  }
  NccMaps ncc = {};
  if (cost == VWB200_CROSS_CORRELATION) {
    int lx0 = INT_MAX, ly0 = INT_MAX, lx1 = INT_MIN, ly1 = INT_MIN, rx0 = INT_MAX, ry0 = INT_MAX, rx1 = INT_MIN, ry1 = INT_MIN;
    for (const Zone& z : zones) {
      lx0 = std::min(lx0, z.lx); ly0 = std::min(ly0, z.ly); lx1 = std::max(lx1, z.lx + z.w); ly1 = std::max(ly1, z.ly + z.h);
      rx0 = std::min(rx0, z.rx); ry0 = std::min(ry0, z.ry);
      rx1 = std::max(rx1, z.rx + z.w + z.sx - 1); ry1 = std::max(ry1, z.ry + z.h + z.sy - 1);
    }
    double *il, *ir;
    VWB_TRY(ar.alloc(&il, (size_t)(lx1 - lx0) * (ly1 - ly0)));
    VWB_TRY(ar.alloc(&ir, (size_t)(rx1 - rx0) * (ry1 - ry0)));
    VWB_TRY(box_sq_inv_launch(left, kx, ky, lx0, ly0, lx1 - lx0, ly1 - ly0, il, st));
    VWB_TRY(box_sq_inv_launch(right, kx, ky, rx0, ry0, rx1 - rx0, ry1 - ry0, ir, st));
    ncc = NccMaps{il, lx0, ly0, lx1 - lx0, ly1 - ly0, ir, rx0, ry0, rx1 - rx0, ry1 - ry0};
  }
  {
    int off = 0;
    for (int c = 0; c < 3; ++c) {
      if (!n_cls[c]) continue;
      VWB_TRY(k1_generic_launch(cost, left, right, d_zones, d_tiles + off, n_cls[c], kx, ky, ncc, d_out, d_sc, d_si, clamp_reads,
                                c == 2 ? 0 : (int)r_max[c], st, ev_used ? nullptr : ev));
      ev_used = true;
      off += n_cls[c];
    }
  }
  VWB_TRY(k1_generic_merge_launch(cost, d_zones, d_split, (int)split.size(), d_sc, d_si, d_out, st));
  if (cost == VWB200_CROSS_CORRELATION)
    VWB_TRY(k1_nan_fixup_launch(cost, left, right, d_zones, (int)zones.size(), kx, ky, ncc, d_out, st));
  if (d_zones_out) *d_zones_out = d_zones;
  if (d_tiles_out) {          // chunk-free tile table for the per-pixel post pass
    make_tiles(zones, k1_generic_tile_w(kx), k1_generic_tile_h(ky), tiles_post, false);
    Tile* d_tp;
    VWB_TRY(ar.alloc(&d_tp, tiles_post.size()));
    VWB_CUDA(cudaMemcpyAsync(d_tp, tiles_post.data(), tiles_post.size() * sizeof(Tile), cudaMemcpyHostToDevice, st));
    VWB_CUDA(cudaStreamSynchronize(st));      // tiles_post is a local
    *d_tiles_out = d_tp;
    if (ntiles_out) *ntiles_out = (int)tiles_post.size();
  } else if (ntiles_out) *ntiles_out = (int)tiles.size();
  VWB_CUDA(cudaStreamSynchronize(st));        // zones / tiles / split are locals of this frame
  return VWB200_OK;
}

// ---------------------------------------------------------------------------------------------------
// host-side quad-tree search-range refinement.  Behaviour of vw::stereo::subdivide_regions
// (Stereo/Correlation.cc:139-328): see DESIGN.md "zones".  Box arithmetic follows vw::BBox2i
// (Math/BBox.tcc): half-open, "empty" when min >= max in any axis.
// ---------------------------------------------------------------------------------------------------
namespace {
struct Range { bool any = false; int x0 = 0, y0 = 0, x1 = 0, y1 = 0; };   // [min, max+1) of valid disparities
inline bool same_range(const Range& a, const Range& b) {
  if (a.any != b.any) return false;
  return !a.any || (a.x0 == b.x0 && a.y0 == b.y0 && a.x1 == b.x1 && a.y1 == b.y1);
}
inline int32_t wmul(int32_t a, int32_t b) { return (int32_t)((uint32_t)a * (uint32_t)b); }
inline int32_t wadd(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }

struct Subdivider {
  const vwb200_dispi* d; int w, h, kx, ky;
  std::vector<HostZone>* out;

  Range scan(Box b) const {
    Range r;
    for (int y = b.y0; y < b.y1; ++y) {
      const vwb200_dispi* row = d + (size_t)y * w;
      for (int x = b.x0; x < b.x1; ++x) {
        if (!row[x].valid) continue;
        const int vx = row[x].dx, vy = row[x].dy;
        if (!r.any) { r.any = true; r.x0 = vx; r.x1 = vx + 1; r.y0 = vy; r.y1 = vy + 1; }
        else { r.x0 = std::min(r.x0, vx); r.x1 = std::max(r.x1, vx + 1); r.y0 = std::min(r.y0, vy); r.y1 = std::max(r.y1, vy + 1); }
      }
    }
    return r;
  }
  static Box to_box(const Range& r) {
    if (!r.any) return Box{INT_MAX - 1, INT_MAX - 1, -(INT_MAX - 1), -(INT_MAX - 1)};   // default (empty) BBox2i
    return Box{r.x0, r.y0, r.x1, r.y1};
  }
  void emit(Box img, const Range& r) const { out->push_back(HostZone{img, to_box(r)}); }
  static int area(const Range& r) { return r.any ? (r.x1 - r.x0) * (r.y1 - r.y0) : 0; }
  static Range merge(Range a, const Range& b) {
    if (!b.any) return a;
    if (!a.any) return b;
    a.x0 = std::min(a.x0, b.x0); a.y0 = std::min(a.y0, b.y0); a.x1 = std::max(a.x1, b.x1); a.y1 = std::max(a.y1, b.y1);
    return a;
  }
  static Box hull(Box a, Box b) { return Box{std::min(a.x0, b.x0), std::min(a.y0, b.y0), std::max(a.x1, b.x1), std::max(a.y1, b.y1)}; }

  // returns false only for "second failure" (the caller then treats the quadrant as unsplittable)
  bool run(Box cur, int fails) const {
    const int cw = cur.x1 - cur.x0, ch = cur.y1 - cur.y0;
    if (cw * ch <= 200 || cw < 16 || ch < 16) {
      Box e{std::max(cur.x0 - 1, 0), std::max(cur.y0 - 1, 0), std::min(cur.x1 + 1, w), std::min(cur.y1 + 1, h)};
      Range r = scan(e);
      if (r.any) emit(cur, r);
      return true;
    }
    const int mx = cur.x0 + cw / 2, my = cur.y0 + ch / 2;
    const Box q[4] = {{cur.x0, cur.y0, mx, my}, {mx, cur.y0, cur.x1, my}, {cur.x0, my, mx, cur.y1}, {mx, my, cur.x1, cur.y1}};
    Range rq[4], all;
    int32_t split_cost = 0;
    for (int i = 0; i < 4; ++i) {
      rq[i] = scan(q[i]);
      if (rq[i].any) split_cost = wadd(split_cost, wmul(area(rq[i]), wmul(q[i].x1 - q[i].x0 + kx, q[i].y1 - q[i].y0 + ky)));
      all = merge(all, rq[i]);
    }
    const int32_t whole_cost = wmul(area(all), wmul(cw + kx, ch + ky));
    const bool worthwhile = !((double)split_cost > (double)whole_cost * 0.8);
    if (worthwhile) {
      for (int i = 0; i < 4; ++i) run(q[i], 0);
      return true;
    }
    if (fails > 0) return false;
    // first failure: give every quadrant one more chance, then deal with the ones that refused
    int bad[4], nbad = 0;
    for (int i = 0; i < 4; ++i) if (!run(q[i], fails + 1)) bad[nbad++] = i;
    auto adjacent_same = [&](int a, int b) {
      return (q[a].x0 == q[b].x0 || q[a].y0 == q[b].y0) && same_range(rq[a], rq[b]);
    };
    if (nbad == 4) { emit(cur, all); return true; }
    if (nbad == 3) {
      const int pairs[3][3] = {{0, 1, 2}, {1, 2, 0}, {0, 2, 1}};      // (merge a, merge b, leftover)
      for (const auto& p : pairs)
        if (adjacent_same(bad[p[0]], bad[p[1]])) {
          out->push_back(HostZone{hull(q[bad[p[0]]], q[bad[p[1]]]), to_box(rq[bad[p[0]]])});
          emit(q[bad[p[2]]], rq[bad[p[2]]]);
          return true;
        }
      for (int i = 0; i < 3; ++i) emit(q[bad[i]], rq[bad[i]]);
    } else if (nbad == 2) {
      if (adjacent_same(bad[0], bad[1])) out->push_back(HostZone{hull(q[bad[0]], q[bad[1]]), to_box(rq[bad[0]])});
      else { emit(q[bad[0]], rq[bad[0]]); emit(q[bad[1]], rq[bad[1]]); }
    } else if (nbad == 1) {
      emit(q[bad[0]], rq[bad[0]]);
    }
    return true;
  }
};
}  // namespace

void subdivide_regions_host(const vwb200_dispi* disp, int w, int h, int kx, int ky, std::vector<HostZone>& out) {
  Subdivider s{disp, w, h, kx, ky, &out};
  s.run(Box{0, 0, w, h}, 0);
}

// ---------------------------------------------------------------------------------------------------
// stereo pre-filter (behaviour of Stereo/PreFilter.h:45-95).  Gaussian taps: erf differences over unit
// bins, normalised, stored as float (Image/Filter.tcc:36-79; default size 7*sigma made odd, >= 3,
// Image/Filter.cc:31-37).  In place on a dense w x h float image.
// ---------------------------------------------------------------------------------------------------
static std::vector<float> gaussian_taps(double sigma) {
  std::vector<float> k;
  if (sigma == 0) return k;
  int size = (int)(7 * sigma);
  if (size < 3) size = 3; else if (size % 2 == 0) size -= 1;
  k.resize(size);
  const int c = size / 2;
  const double z = 1 / (std::sqrt(2.0) * sigma);
  double sum = 0.0;
  for (int i = 1; i <= c; ++i) {
    const double t = std::erf((i + 0.5) * z) - std::erf((i - 0.5) * z);
    sum += t;
    k[c + i] = k[c - i] = (float)t;
  }
  sum *= 2.0;
  const double t0 = std::erf(0.5 * z) - std::erf(-0.5 * z);
  sum += t0;
  k[c] = (float)t0;
  const double norm = 1.0 / sum;
  for (float& v : k) v = (float)(v * norm);
  return k;
}
static int prefilter_inplace(float* img, int w, int h, int mode, float width, Arena& ar, cudaStream_t st) {
  if (mode == VWB200_PREFILTER_NONE) return VWB200_OK;
  if (mode != VWB200_PREFILTER_LOG && mode != VWB200_PREFILTER_MEANSUB) { set_error("unknown prefilter mode %d", mode); return VWB200_EARG; }
  const std::vector<float> taps = gaussian_taps((double)width);
  float *d_taps, *work, *g;
  VWB_TRY(ar.alloc(&d_taps, taps.size() + 1));
  VWB_TRY(ar.alloc(&work, (size_t)w * h));
  VWB_TRY(ar.alloc(&g, (size_t)w * h));
  const ImgF im{img, w, h, w};
  if (taps.empty()) {          // sigma 0: no smoothing, the view is the (edge-extended) image itself
    VWB_CUDA(cudaMemcpyAsync(g, img, (size_t)w * h * sizeof(float), cudaMemcpyDeviceToDevice, st));
  } else {
    VWB_CUDA(cudaMemcpyAsync(d_taps, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    VWB_CUDA(cudaStreamSynchronize(st));       // taps live on this frame's stack
    VWB_TRY(sepconv_launch(im, d_taps, (int)taps.size(), work, g, st));
  }
  VWB_TRY(prefilter_final_launch(im, g, mode, work, st));
  VWB_CUDA(cudaMemcpyAsync(img, work, (size_t)w * h * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return VWB200_OK;
}

// prefilter.filter(image) over an arbitrary region of the lazily edge-extended view (what
// crop(prefilter.filter(img), region) yields in ParabolaSubpixelView::prerasterize, .cc:296-327).
static int filtered_region(ImgF img, int mode, float width, Box reg, float** out, Arena& ar, cudaStream_t st) {
  const int w = reg.x1 - reg.x0, h = reg.y1 - reg.y0;
  float* o;
  VWB_TRY(ar.alloc(&o, (size_t)w * h));
  *out = o;
  if (mode == VWB200_PREFILTER_NONE) return crop_extend_f32_launch(img, reg.x0, reg.y0, w, h, o, w, st);
  if (mode != VWB200_PREFILTER_LOG && mode != VWB200_PREFILTER_MEANSUB) { set_error("unknown prefilter mode %d", mode); return VWB200_EARG; }
  const std::vector<float> taps = gaussian_taps((double)width);
  const int n = (int)taps.size();
  float* d_taps;
  VWB_TRY(ar.alloc(&d_taps, taps.size() + 1));
  if (n) { VWB_CUDA(cudaMemcpyAsync(d_taps, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice, st)); VWB_CUDA(cudaStreamSynchronize(st)); }
  auto clampi = [](int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); };
  Box big;
  if (mode == VWB200_PREFILTER_MEANSUB) big = Box{reg.x0 - n, reg.y0 - n, reg.x1 + n, reg.y1 + n};
  else {
    const Box need{clampi(reg.x0 - 1, 0, img.w - 1), clampi(reg.y0 - 1, 0, img.h - 1), clampi(reg.x1, 0, img.w - 1) + 1, clampi(reg.y1, 0, img.h - 1) + 1};
    big = Box{need.x0 - n, need.y0 - n, need.x1 + n, need.y1 + n};
  }
  const int ew = big.x1 - big.x0, eh = big.y1 - big.y0;
  float *e, *g, *work;
  VWB_TRY(ar.alloc(&e, (size_t)ew * eh)); VWB_TRY(ar.alloc(&g, (size_t)ew * eh)); VWB_TRY(ar.alloc(&work, (size_t)ew * eh));
  VWB_TRY(crop_extend_f32_launch(img, big.x0, big.y0, ew, eh, e, ew, st));
  if (n) VWB_TRY(sepconv_launch(ImgF{e, ew, eh, ew}, d_taps, n, work, g, st));
  else VWB_CUDA(cudaMemcpyAsync(g, e, (size_t)ew * eh * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (mode == VWB200_PREFILTER_MEANSUB) return meansub_region_launch(e, g, ew, n, w, h, o, st);
  return log_region_launch(g, ew, big.x0, big.y0, img.w, img.h, reg.x0, reg.y0, w, h, o, st);
}

// ---------------------------------------------------------------------------------------------------
// the view handle
// ---------------------------------------------------------------------------------------------------
}  // namespace vwb200

using namespace vwb200;

struct LevelImgsT;
struct vwb200_corr {
  vwb200_corr_params p;
  int max_level_by_search = 0;
  // inputs in HBM
  const float* L = nullptr; const float* R = nullptr; const uint8_t* Lm = nullptr; const uint8_t* Rm = nullptr;
  int lcols = 0, lrows = 0, rcols = 0, rrows = 0;
  ptrdiff_t lpitch = 0, rpitch = 0, lmpitch = 0, rmpitch = 0;
  bool owned = false;
  bool streamed = false;       // L / R / Lm / Rm are HOST pointers; every rasterize call uploads its own region of interest
  int device = 0;
  ~vwb200_corr() { release(); }
  void release() {
    if (owned) { cudaFree((void*)L); cudaFree((void*)R); cudaFree((void*)Lm); cudaFree((void*)Rm); }
    L = R = nullptr; Lm = Rm = nullptr; owned = false; streamed = false;
  }
  int num_levels(int bw, int bh) const {
    // CorrelationView.cc:301-310: log(int) is double, log(2.0f) is float
    const int smallest = std::min(bw, bh), largest_kernel = std::max(p.kernel_x, p.kernel_y);
    int levels = (int)std::floor(std::log((double)smallest) / (double)std::log(2.0f) - std::log((double)largest_kernel) / (double)std::log(2.0f));
    if (max_level_by_search < levels) levels = max_level_by_search;
    if (levels < 1) levels = 0;
    return levels;
  }
  // optional lr_disp_diff output (CorrelationView.h:67-68): PixelMask<float> pairs, caller-owned
  float* diff = nullptr; int diff_cols = 0, diff_rows = 0; ptrdiff_t diff_pitch = 0; int diff_on_device = 0;
  struct DiffTile { float* d = nullptr; ptrdiff_t pitch = 0; int ox = 0, oy = 0; };   // device view of the processed box's window
  int prerasterize(Box bbox, vwb200_dispi** d_disp_out, float** d_sub_out, int* all_invalid, const DiffTile& df, Arena& ar, cudaStream_t st) const;
  int prerasterize_sgm(Box bbox, const std::vector<struct LevelImgsT>& py, int levels, vwb200_dispi** d_disp_out, float** d_sub_out,
                       const DiffTile& df, Arena& ar, cudaStream_t st) const;
};

namespace {
inline Box bexpand(Box b, int ex, int ey) { if (b.x0 >= b.x1 || b.y0 >= b.y1) return b; return Box{b.x0 - ex, b.y0 - ey, b.x1 + ex, b.y1 + ey}; }
inline bool bempty(Box b) { return b.x0 >= b.x1 || b.y0 >= b.y1; }
}
struct LevelImgsT { float* l; float* r; uint8_t* lm; uint8_t* rm; int lw, lh, rw, rh, lmw, lmh, rmw, rmh; };
typedef LevelImgsT LevelImgs;

// The per-tile pipeline.  Result: integer disparity (bw x bh, dense) in device memory, WITHOUT the
// final "+ search_region.min()" (finalize_kernel adds it while casting to float).
int vwb200_corr::prerasterize(Box bbox, vwb200_dispi** d_disp_out, float** d_sub_out, int* all_invalid, const DiffTile& df, Arena& ar,
                              cudaStream_t st) const {
  *d_sub_out = nullptr;
  const int bw = bbox.x1 - bbox.x0, bh = bbox.y1 - bbox.y0;
  const int kx = p.kernel_x, ky = p.kernel_y, hkx = kx / 2, hky = ky / 2;
  const int ssx = p.search_x1 - p.search_x0, ssy = p.search_y1 - p.search_y0;
  const int levels = num_levels(bw, bh);
  const int up = 1 << levels;
  *all_invalid = 0;

  // ---- build_image_pyramids (CorrelationView.cc:67-239) ----
  const Box lg = bexpand(bbox, hkx * up, hky * up);
  Box rg{lg.x0 + p.search_x0, lg.y0 + p.search_y0, lg.x1 + p.search_x0 + ssx, lg.y1 + p.search_y0 + ssy};
  std::vector<LevelImgs> py(levels + 1);
  LevelImgs& b0 = py[0];
  b0.lw = lg.x1 - lg.x0; b0.lh = lg.y1 - lg.y0; b0.rw = rg.x1 - rg.x0; b0.rh = rg.y1 - rg.y0;
  VWB_TRY(ar.alloc(&b0.l, (size_t)b0.lw * b0.lh));
  VWB_TRY(ar.alloc(&b0.r, (size_t)b0.rw * b0.rh));
  ImgF Lin{L, lcols, lrows, lpitch}, Rin{R, rcols, rrows, rpitch};
  ImgB Lmin{Lm, lcols, lrows, lmpitch}, Rmin{Rm, rcols, rrows, rmpitch};
  int lox = 0, loy = 0, rox_ = 0, roy_ = 0;          // origin of the device-resident part of the rasters
  if (streamed) {
    // the tile feeder (SURVEY 8f n3; Image/ImageIO.h:150-314 is the caller pattern): the rasters stay on the host and only
    // this tile's region of interest -- the padded left box and the right box grown by the search window, clipped to the
    // image -- goes up.  Clamping to the ROI equals clamping to the image: the ROI reaches the image edge wherever the
    // needed region crosses it, and coordinates inside the image but outside the ROI are never requested.
    auto clip = [](Box b, int w, int h) {
      Box r{std::min(std::max(b.x0, 0), w - 1), std::min(std::max(b.y0, 0), h - 1), std::max(std::min(b.x1, w), 1), std::max(std::min(b.y1, h), 1)};
      if (r.x1 <= r.x0) r.x1 = r.x0 + 1;
      if (r.y1 <= r.y0) r.y1 = r.y0 + 1;
      return r;
    };
    const Box lr_ = clip(lg, lcols, lrows), rr_ = clip(rg, rcols, rrows);
    const int lw_ = lr_.x1 - lr_.x0, lh_ = lr_.y1 - lr_.y0, rw_ = rr_.x1 - rr_.x0, rh_ = rr_.y1 - rr_.y0;
    float *dl_, *dr_; uint8_t *dlm_, *drm_;
    VWB_TRY(ar.alloc(&dl_, (size_t)lw_ * lh_)); VWB_TRY(ar.alloc(&dr_, (size_t)rw_ * rh_));
    VWB_TRY(ar.alloc(&dlm_, (size_t)lw_ * lh_)); VWB_TRY(ar.alloc(&drm_, (size_t)rw_ * rh_));
    VWB_CUDA(cudaMemcpy2DAsync(dl_, (size_t)lw_ * 4, L + (ptrdiff_t)lr_.y0 * lpitch + lr_.x0, (size_t)lpitch * 4, (size_t)lw_ * 4, lh_, cudaMemcpyHostToDevice, st));
    VWB_CUDA(cudaMemcpy2DAsync(dr_, (size_t)rw_ * 4, R + (ptrdiff_t)rr_.y0 * rpitch + rr_.x0, (size_t)rpitch * 4, (size_t)rw_ * 4, rh_, cudaMemcpyHostToDevice, st));
    VWB_CUDA(cudaMemcpy2DAsync(dlm_, (size_t)lw_, Lm + (ptrdiff_t)lr_.y0 * lmpitch + lr_.x0, (size_t)lmpitch, (size_t)lw_, lh_, cudaMemcpyHostToDevice, st));
    VWB_CUDA(cudaMemcpy2DAsync(drm_, (size_t)rw_, Rm + (ptrdiff_t)rr_.y0 * rmpitch + rr_.x0, (size_t)rmpitch, (size_t)rw_, rh_, cudaMemcpyHostToDevice, st));
    Lin = ImgF{dl_, lw_, lh_, lw_}; Rin = ImgF{dr_, rw_, rh_, rw_};
    Lmin = ImgB{dlm_, lw_, lh_, lw_}; Rmin = ImgB{drm_, rw_, rh_, rw_};
    lox = lr_.x0; loy = lr_.y0; rox_ = rr_.x0; roy_ = rr_.y0;
  }
  VWB_TRY(crop_extend_f32_launch(Lin, lg.x0 - lox, lg.y0 - loy, b0.lw, b0.lh, b0.l, b0.lw, st));
  VWB_TRY(crop_extend_f32_launch(Rin, rg.x0 - rox_, rg.y0 - roy_, b0.rw, b0.rh, b0.r, b0.rw, st));
  // level-0 imagery statistics, taken BEFORE the mean fill (the mean of pixels lies inside their range, so vmin / vmax
  // still bound the filled image): integer-valued rasters with a small range -> the exact-integer kernels take level 0.
  // any_filled: some pixel of the padded tile is masked and becomes the (non-integer) mean -- the integer zone kernel then
  // checks what it reads and hands the zones that touch such pixels to the fp64 kernel; the whole-zone fast kernels are off.
  float hstats[6] = {0, 0, 0, 0, 0, 0};
  int any_filled = 0;
  const bool want_stats = p.cost_type == VWB200_ABSOLUTE_DIFFERENCE || p.cost_type == VWB200_SQUARED_DIFFERENCE;
  {  // mean fill of masked pixels (:116-149); masks here are constant-edge-extended over the padded ROI
    uint8_t *lmb, *rmb; double* acc;
    float* d_stats = nullptr; int* d_filled = nullptr;
    VWB_TRY(ar.alloc(&lmb, (size_t)b0.lw * b0.lh));
    VWB_TRY(ar.alloc(&rmb, (size_t)b0.rw * b0.rh));
    VWB_TRY(ar.alloc(&acc, 2 * (2 + 2 * 256)));
    VWB_TRY(crop_extend_u8_launch(Lmin, lg.x0 - lox, lg.y0 - loy, b0.lw, b0.lh, 0, lmb, b0.lw, st));
    VWB_TRY(crop_extend_u8_launch(Rmin, rg.x0 - rox_, rg.y0 - roy_, b0.rw, b0.rh, 0, rmb, b0.rw, st));
    double* acc_r = acc + (2 + 2 * 256);
    VWB_TRY(masked_mean_launch(ImgF{b0.l, b0.lw, b0.lh, b0.lw}, ImgB{lmb, b0.lw, b0.lh, b0.lw}, acc, st));
    VWB_TRY(masked_mean_launch(ImgF{b0.r, b0.rw, b0.rh, b0.rw}, ImgB{rmb, b0.rw, b0.rh, b0.rw}, acc_r, st));
    double hacc[4];
    VWB_CUDA(cudaMemcpyAsync(hacc, acc, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaMemcpyAsync(hacc + 2, acc_r, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (want_stats) {
      VWB_TRY(ar.alloc(&d_stats, 6));
      VWB_TRY(ar.alloc(&d_filled, 1));
      VWB_TRY(image_stats_launch(ImgF{b0.l, b0.lw, b0.lh, b0.lw}, d_stats, st));
      VWB_TRY(image_stats_launch(ImgF{b0.r, b0.rw, b0.rh, b0.rw}, d_stats + 3, st));
      VWB_CUDA(cudaMemsetAsync(d_filled, 0, sizeof(int), st));
      VWB_TRY(mask_any_zero_launch(ImgB{lmb, b0.lw, b0.lh, b0.lw}, d_filled, st));
      VWB_TRY(mask_any_zero_launch(ImgB{rmb, b0.rw, b0.rh, b0.rw}, d_filled, st));
      VWB_CUDA(cudaMemcpyAsync(hstats, d_stats, sizeof(hstats), cudaMemcpyDeviceToHost, st));
      VWB_CUDA(cudaMemcpyAsync(&any_filled, d_filled, sizeof(int), cudaMemcpyDeviceToHost, st));
    }
    VWB_CUDA(cudaStreamSynchronize(st));
    if (hacc[1] == 0.0 || hacc[3] == 0.0) { *all_invalid = 1; *d_disp_out = nullptr; return VWB200_OK; }   // :137-142, :320-331
    VWB_TRY(mean_fill_launch(b0.l, b0.lw, b0.lh, b0.lw, ImgB{lmb, b0.lw, b0.lh, b0.lw}, acc, st));
    VWB_TRY(mean_fill_launch(b0.r, b0.rw, b0.rh, b0.rw, ImgB{rmb, b0.rw, b0.rh, b0.rw}, acc_r, st));
  }
  const float tile_vmin = std::min(hstats[0], hstats[3]), tile_vmax = std::max(hstats[1], hstats[4]);
  const bool raster_integer = want_stats && hstats[2] != 0.0f && hstats[5] != 0.0f && p.prefilter_mode == VWB200_PREFILTER_NONE;
  const bool tile_integer = raster_integer && !any_filled;          // every pixel of the level-0 images is an integer
  // final masks: zero edge extension, no kernel padding (:192-197)
  b0.lmw = bw; b0.lmh = bh; b0.rmw = bw + ssx; b0.rmh = bh + ssy;
  VWB_TRY(ar.alloc(&b0.lm, (size_t)b0.lmw * b0.lmh));
  VWB_TRY(ar.alloc(&b0.rm, (size_t)b0.rmw * b0.rmh));
  VWB_TRY(crop_extend_u8_launch(Lmin, bbox.x0 - lox, bbox.y0 - loy, b0.lmw, b0.lmh, 1, b0.lm, b0.lmw, st));
  VWB_TRY(crop_extend_u8_launch(Rmin, bbox.x0 + p.search_x0 - rox_, bbox.y0 + p.search_y0 - roy_, b0.rmw, b0.rmh, 1, b0.rm, b0.rmw, st));
  for (int i = 1; i <= levels; ++i) {   // :209-216
    const LevelImgs& a = py[i - 1];
    LevelImgs& b = py[i];
    b.lw = 1 + (a.lw - 1) / 2; b.lh = 1 + (a.lh - 1) / 2; b.rw = 1 + (a.rw - 1) / 2; b.rh = 1 + (a.rh - 1) / 2;
    b.lmw = 1 + (a.lmw - 1) / 2; b.lmh = 1 + (a.lmh - 1) / 2; b.rmw = 1 + (a.rmw - 1) / 2; b.rmh = 1 + (a.rmh - 1) / 2;
    VWB_TRY(ar.alloc(&b.l, (size_t)b.lw * b.lh));
    VWB_TRY(ar.alloc(&b.r, (size_t)b.rw * b.rh));
    VWB_TRY(ar.alloc(&b.lm, (size_t)b.lmw * b.lmh));
    VWB_TRY(ar.alloc(&b.rm, (size_t)b.rmw * b.rmh));
    VWB_TRY(pyramid_down_launch(ImgF{a.l, a.lw, a.lh, a.lw}, b.l, b.lw, st));
    VWB_TRY(pyramid_down_launch(ImgF{a.r, a.rw, a.rh, a.rw}, b.r, b.rw, st));
    VWB_TRY(subsample_mask_launch(ImgB{a.lm, a.lmw, a.lmh, a.lmw}, b.lm, b.lmw, st));
    VWB_TRY(subsample_mask_launch(ImgB{a.rm, a.rmw, a.rmh, a.rmw}, b.rm, b.rmw, st));
  }

  const int prefilter_mode = p.algorithm != VWB200_CORRELATION_BM ? VWB200_PREFILTER_NONE : p.prefilter_mode;   // CorrelationView.h:96-97
  for (int i = 0; i <= levels; ++i) {   // :233-236 prefilter every level
    VWB_TRY(prefilter_inplace(py[i].l, py[i].lw, py[i].lh, prefilter_mode, p.prefilter_width, ar, st));
    VWB_TRY(prefilter_inplace(py[i].r, py[i].rw, py[i].rh, prefilter_mode, p.prefilter_width, ar, st));
  }
  if (p.algorithm != VWB200_CORRELATION_BM) return prerasterize_sgm(bbox, py, levels, d_disp_out, d_sub_out, df, ar, st);

  // ---- level loop (CorrelationView.cc:363-830) ----
  const bool prof = getenv("VWB200_PROFILE") != nullptr;      // host-side wall-clock split of this call, one line on stderr
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms_since = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double, std::milli>(now() - t).count(); };
  const auto t_loop = now();
  double ms_zones = 0, ms_d2h = 0, ms_subdiv = 0;
  std::vector<HostZone> zones;
  zones.push_back(HostZone{Box{0, 0, py[levels].lmw, py[levels].lmh}, Box{0, 0, ssx / up + 1, ssy / up + 1}});   // :338-342
  vwb200_dispi* disp = nullptr;
  std::vector<vwb200_dispi> hdisp;
  const int tile_w = k1_generic_tile_w(kx), tile_h = k1_generic_tile_h(ky);
  for (int level = levels; level >= 0; --level) {
    const LevelImgs& lv = py[level];
    const int scaling = 1 << level;
    const int dw = lv.lmw, dh = lv.lmh;
    VWB_TRY(ar.alloc(&disp, (size_t)dw * dh));
    VWB_CUDA(cudaMemsetAsync(disp, 0, (size_t)dw * dh * sizeof(vwb200_dispi), st));    // fresh ImageView: (0,0) invalid
    const int rox = up * hkx / scaling, roy = up * hky / scaling;                     // :381
    std::vector<Zone> zl, zr;
    std::vector<int2> post;
    const bool check = (p.consistency_threshold >= 0 && level == 0);
    long long rl_elems = 0;
    for (const HostZone& hz : zones) {
      const int zw = hz.img.x1 - hz.img.x0, zh = hz.img.y1 - hz.img.y0;
      if (zw <= 0 || zh <= 0) continue;
      const int dsx = hz.disp.x1 - hz.disp.x0, dsy = hz.disp.y1 - hz.disp.y0;
      if (dsx <= 0 || dsy <= 0) { set_error("zone with empty disparity range"); return VWB200_ELOGIC; }
      Zone z{};
      z.obase = (long long)hz.img.y0 * dw + hz.img.x0; z.opitch = dw; z.w = zw; z.h = zh;
      z.lx = hz.img.x0 + rox - hkx; z.ly = hz.img.y0 + roy - hky;                      // :611-612 (expand by half kernel)
      z.rx = z.lx + hz.disp.x0; z.ry = z.ly + hz.disp.y0;                             // :615
      z.sx = dsx; z.sy = dsy; z.addx = 0; z.addy = 0;
      zl.push_back(z);
      post.push_back(make_int2(hz.disp.x0, hz.disp.y0));
      if (check) {   // R->L (:669-675): reference = right crop, search in left shifted by -size
        Zone q{};
        q.obase = rl_elems; q.opitch = zw + dsx; q.w = zw + dsx; q.h = zh + dsy;
        q.lx = z.rx; q.ly = z.ry; q.rx = z.lx - dsx; q.ry = z.ly - dsy;
        q.sx = dsx; q.sy = dsy; q.addx = -dsx; q.addy = -dsy;
        rl_elems += (long long)q.w * q.h;
        zr.push_back(q);
      }
    }
    if (getenv("VWB200_DEBUG")) {
      long long evals = 0, maxd = 0, big = 0; int nbig = 0;
      for (const Zone& z : zl) { long long e = (long long)z.w * z.h * z.sx * z.sy; evals += e; if ((long long)z.sx * z.sy > maxd) maxd = (long long)z.sx * z.sy; if ((long long)z.sx * z.sy > 400) { ++nbig; big += e; } }
      fprintf(stderr, "[vwb200] level %d: %zu zones, %lld evals, max search %lld, %d zones with >400 disparities (%lld evals)\n", level, zl.size(), evals, maxd, nbig, big);
    }
    const ImgF Ll{lv.l, lv.lw, lv.lh, lv.lw}, Rl{lv.r, lv.rw, lv.rh, lv.rw};
    vwb200_dispi* rl = nullptr;
    if (check && !zr.empty()) VWB_TRY(ar.alloc(&rl, (size_t)rl_elems));
    // large level-0 zones of integer imagery go to the exact-integer fast kernel, everything else to the zone kernel
    std::vector<char> fast_l(zl.size(), 0), fast_r(zr.size(), 0);
    if (level == 0 && tile_integer) {
      auto try_fast = [&](const Zone& z, ImgF a, ImgF b, vwb200_dispi* dst, char& flag) -> int {
        if ((long long)z.w * z.h < 128 * 128 || (long long)z.sx * z.sy < 256) return VWB200_OK;
        const FastOrigin org{z.lx, z.ly, z.rx, z.ry, z.addx, z.addy};
        unsigned char* ws;
        if (k1_fast_supported(p.cost_type, kx, ky, z.sx, z.sy, tile_vmin, tile_vmax, true) == VWB200_OK) {
          const size_t wb = k1_fast_workspace_bytes(z.w, z.h, z.sx, z.sy, kx, ky);
          VWB_TRY(ar.alloc(&ws, wb));
          VWB_TRY(k1_fast_launch(p.cost_type, a, b, z.w, z.h, z.sx, z.sy, kx, ky, tile_vmin, dst + z.obase, z.opitch, ws, wb, st, nullptr, &org));
          flag = 1;
        } else if (k1_screen_supported(p.cost_type, kx, ky, z.sx, z.sy, tile_vmin, tile_vmax, true) == VWB200_OK) {
          VWB_TRY(ar.alloc(&ws, k1_screen_workspace_bytes(p.cost_type, z.w, z.h, z.sx, z.sy, kx, ky)));
          VWB_TRY(k1_screen_launch(p.cost_type, a, b, z.w, z.h, z.sx, z.sy, kx, ky, tile_vmin, tile_vmax, dst + z.obase, z.opitch, ws, st, nullptr, &org));
          flag = 1;
          if (getenv("VWB200_DEBUG")) fprintf(stderr, "[vwb200] level 0 zone %dx%d search %dx%d -> k1_screen\n", z.w, z.h, z.sx, z.sy);
        }
        return VWB200_OK;
      };
      for (size_t i = 0; i < zl.size(); ++i) VWB_TRY(try_fast(zl[i], Ll, Rl, disp, fast_l[i]));
      for (size_t i = 0; i < zr.size(); ++i) VWB_TRY(try_fast(zr[i], Rl, Ll, rl, fast_r[i]));
    }
    const Zone* d_zl = nullptr; const Tile* d_tl = nullptr; int ntl = 0;
    const ZoneIntMode zim{level == 0 && raster_integer, tile_vmin, tile_vmax, any_filled != 0};
    const auto t_z = now();
    VWB_TRY(run_k1_zones(p.cost_type, Ll, Rl, zl, kx, ky, disp, ar, st, &d_zl, &d_tl, &ntl, nullptr, &fast_l, &zim));
    const Zone* d_zr = nullptr;
    if (check && !zr.empty()) VWB_TRY(run_k1_zones(p.cost_type, Rl, Ll, zr, kx, ky, rl, ar, st, &d_zr, nullptr, nullptr, nullptr, &fast_r, &zim));
    ms_zones += ms_since(t_z);
    if (!zl.empty()) {
      int2* d_post;
      VWB_TRY(ar.alloc(&d_post, post.size()));
      VWB_CUDA(cudaMemcpyAsync(d_post, post.data(), post.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
      VWB_TRY(zone_post_launch(d_tl, ntl, d_zl, d_zr, d_post, disp, rl, p.consistency_threshold, tile_w, tile_h, st,
                               (level == 0 && check) ? df.d : nullptr, df.pitch, df.ox, df.oy));
    }
    if (p.filter_half_kernel > 0) {   // :713-744
      const int fh = p.filter_half_kernel;
      vwb200_dispi *t1, *t2;
      VWB_TRY(ar.alloc(&t2, (size_t)dw * dh));
      if (level != 0) {
        VWB_TRY(ar.alloc(&t1, (size_t)(dw + 2) * (dh + 2)));
        VWB_TRY(rm_outliers_launch(disp, dw, dh, fh, fh, 3.0, 0.5, -1, -1, dw + 2, dh + 2, t1, st));
        VWB_TRY(cleanup_pass2_launch(t1, dw, dh, t2, st));
      } else {
        VWB_TRY(rm_outliers_launch(disp, dw, dh, fh, fh, 3.0, 0.5, 0, 0, dw, dh, t2, st));
      }
      VWB_TRY(disparity_mask_launch(t2, dw, dh, ImgB{lv.lm, lv.lmw, lv.lmh, lv.lmw}, ImgB{lv.rm, lv.rmw, lv.rmh, lv.rmw}, disp, st));
    }
    if (p.blob_filter_area / scaling >= 1) {   // :746-749, disparity_blob_filter (:242-271)
      int* work;
      VWB_TRY(ar.alloc(&work, (size_t)2 * dw * dh));
      VWB_TRY(blob_filter_launch(disp, dw, dh, p.blob_filter_area / scaling, work, st));
    }
    if (level != 0) {   // :754-799 refine the search zones on the host (zones are O(10^3), data dependent)
      const auto t_d = now();
      hdisp.resize((size_t)dw * dh);
      VWB_CUDA(cudaMemcpyAsync(hdisp.data(), disp, hdisp.size() * sizeof(vwb200_dispi), cudaMemcpyDeviceToHost, st));
      VWB_CUDA(cudaStreamSynchronize(st));
      ms_d2h += ms_since(t_d);
      const auto t_s = now();
      zones.clear();
      subdivide_regions_host(hdisp.data(), dw, dh, kx, ky, zones);
      ms_subdiv += ms_since(t_s);
      const LevelImgs& nl = py[level - 1];
      const Box scale_search{0, 0, nl.rw - nl.lw, nl.rh - nl.lh};
      for (HostZone& z : zones) {
        if (!bempty(z.img)) { z.img.x0 *= 2; z.img.y0 *= 2; z.img.x1 *= 2; z.img.y1 *= 2; }
        z.img.x0 = std::max(z.img.x0, 0); z.img.y0 = std::max(z.img.y0, 0);
        z.img.x1 = std::min(z.img.x1, nl.lmw); z.img.y1 = std::min(z.img.y1, nl.lmh);
        if (!bempty(z.disp)) { z.disp.x0 *= 2; z.disp.y0 *= 2; z.disp.x1 *= 2; z.disp.y1 *= 2; }
        z.disp = bexpand(z.disp, 2, 2);
        z.disp.x0 = std::max(z.disp.x0, scale_search.x0); z.disp.y0 = std::max(z.disp.y0, scale_search.y0);
        z.disp.x1 = std::min(z.disp.x1, scale_search.x1); z.disp.y1 = std::min(z.disp.y1, scale_search.y1);
        if (bempty(z.disp)) z.disp = Box{0, 0, ssx, ssy};
      }
    }
  }
  const LevelImgs& l0 = py[0];
  if (l0.lmw != bw || l0.lmh != bh) { set_error("PyramidCorrelation: Solved disparity doesn't match requested bbox size."); return VWB200_EMATH; }
  if (df.d) VWB_TRY(diff_invalidate_launch(disp, bw, bh, df.d, df.pitch, df.ox, df.oy, st));   // :848-857
  if (prof) {
    const double enq = ms_since(t_loop);
    cudaStreamSynchronize(st);
    fprintf(stderr, "[vwb200] tile %d,%d: level loop %.2f ms host (zone tables+launch+sync %.2f, D2H+wait %.2f, subdivide %.2f), %.2f ms until the stream drained\n",
            bbox.x0, bbox.y0, enq, ms_zones, ms_d2h, ms_subdiv, ms_since(t_loop));
  }
  *d_disp_out = disp;
  return VWB200_OK;
}

// The SGM / MGM / FINAL_MGM branch of the level loop (CorrelationView.cc:392-595, 700-750, 859-871): one calc_disparity_sgm
// per level over the whole padded tile, seeded by the previous level's filtered disparity; an R->L pass + consistency check
// at the levels >= min_consistency_level; the sub-pixel view is made at level 0 BEFORE the check and the filters.
int vwb200_corr::prerasterize_sgm(Box bbox, const std::vector<LevelImgs>& py, int levels, vwb200_dispi** d_disp_out, float** d_sub_out,
                                  const DiffTile& df, Arena& ar, cudaStream_t st) const {
  const int bw = bbox.x1 - bbox.x0, bh = bbox.y1 - bbox.y0;
  const int kx = p.kernel_x, ky = p.kernel_y, hkx = kx / 2, hky = ky / 2;
  const int ssx = p.search_x1 - p.search_x0, ssy = p.search_y1 - p.search_y0;
  const int up = 1 << levels;
  if (kx != ky) { set_error("SGM needs a square kernel (SemiGlobalMatcher takes kernel_size[0], SGM.cc:213-215)"); return VWB200_EARG; }
  vwb200_dispi *disp = nullptr, *disp_rl = nullptr, *prev = nullptr, *prev_rl = nullptr;
  int dw = 0, dh = 0, pw = 0, ph = 0, rlw = 0, rlh = 0, prlw = 0, prlh = 0;
  float* sub = nullptr;
  for (int level = levels; level >= 0; --level) {
    const LevelImgs& lv = py[level];
    const int use_mgm = p.algorithm == VWB200_CORRELATION_MGM || (p.algorithm == VWB200_CORRELATION_FINAL_MGM && level == 0);   // :366-367
    const int scaling = 1 << level;
    prev = disp; pw = dw; ph = dh; prev_rl = disp_rl; prlw = rlw; prlh = rlh;                    // :373-376
    disp = nullptr; disp_rl = nullptr;
    dw = lv.lmw; dh = lv.lmh;
    const int rox = up * hkx / scaling, roy = up * hky / scaling;
    const int dsx = ssx / scaling, dsy = ssy / scaling;                                          // :395-396
    const Box lr{rox - hkx, roy - hky, dw + rox + hkx, dh + roy + hky};                          // :404-405
    const Box rr{lr.x0, lr.y0, lr.x1 + dsx, lr.y1 + dsy};                                       // :406-407
    const int lcw = lr.x1 - lr.x0, lch = lr.y1 - lr.y0, rcw = rr.x1 - rr.x0, rch = rr.y1 - rr.y0;
    float *lc, *rc;
    VWB_TRY(ar.alloc(&lc, (size_t)lcw * lch));
    VWB_TRY(ar.alloc(&rc, (size_t)rcw * rch));
    VWB_TRY(crop_extend_f32_launch(ImgF{lv.l, lv.lw, lv.lh, lv.lw}, lr.x0, lr.y0, lcw, lch, lc, lcw, st));
    VWB_TRY(crop_extend_f32_launch(ImgF{lv.r, lv.rw, lv.rh, lv.rw}, rr.x0, rr.y0, rcw, rch, rc, rcw, st));
    SgmArgs a;
    a.left = ImgF{lc, lcw, lch, lcw}; a.right = ImgF{rc, rcw, rch, rcw};
    a.sx = dsx; a.sy = dsy; a.k = kx;
    a.ternary = p.cost_type == VWB200_TERNARY_CENSUS_TRANSFORM; a.ternary_threshold = 5;
    a.use_mgm = use_mgm; a.subpixel_mode = p.sgm_subpixel_mode;
    a.buf_x = p.sgm_search_buffer_x; a.buf_y = p.sgm_search_buffer_y;
    a.memory_limit_mb = p.memory_limit_mb > 0 ? p.memory_limit_mb : 6000.0;
    a.assumed_threads = p.sgm_threads > 0 ? p.sgm_threads : 4;
    a.lmask = ImgB{lv.lm, lv.lmw, lv.lmh, lv.lmw}; a.rmask = ImgB{lv.rm, lv.rmw, lv.rmh, lv.rmw};
    if (level < levels) { a.prev = prev; a.pw = pw; a.ph = ph; a.ppitch = pw; }
    int ow = 0, oh = 0;
    sgm_output_size(lcw, lch, rcw, rch, dsx, dsy, kx, &ow, &oh);
    if (ow != dw || oh != dh) { set_error("PyramidCorrelation(SGM): level %d disparity is %dx%d, expected %dx%d", level, ow, oh, dw, dh); return VWB200_EMATH; }
    VWB_TRY(ar.alloc(&disp, (size_t)dw * dh));
    a.out = disp; a.opitch = dw;
    if (level == 0) { VWB_TRY(ar.alloc(&sub, (size_t)dw * dh * 3)); a.out_sub = sub; a.sub_pitch = (ptrdiff_t)dw * 3; }
    VWB_TRY(sgm_run(a, ar, st));
    bool check_rl = false;
    uint8_t *rrm = nullptr, *lrm = nullptr; int lrmw = 0, lrmh = 0;
    if (p.consistency_threshold >= 0.0f && level >= p.min_consistency_level) {                  // :438-590
      check_rl = true;
      const Box llr{lr.x0 - dsx, lr.y0 - dsy, lr.x1 + dsx, lr.y1 + dsy};                         // :453-455
      const int l2w = llr.x1 - llr.x0, l2h = llr.y1 - llr.y0;
      float* l2;
      VWB_TRY(ar.alloc(&l2, (size_t)l2w * l2h));
      VWB_TRY(crop_extend_f32_launch(ImgF{lv.l, lv.lw, lv.lh, lv.lw}, llr.x0, llr.y0, l2w, l2h, l2, l2w, st));
      rlw = rcw - 2 * hkx; rlh = rch - 2 * hky;                                                  // masks of the reversed problem (:496-508)
      lrmw = l2w - 2 * hkx; lrmh = l2h - 2 * hky;
      VWB_TRY(ar.alloc(&rrm, (size_t)rlw * rlh));
      VWB_TRY(ar.alloc(&lrm, (size_t)lrmw * lrmh));
      VWB_TRY(crop_extend_u8_launch(ImgB{lv.rm, lv.rmw, lv.rmh, lv.rmw}, 0, 0, rlw, rlh, 1, rrm, rlw, st));
      VWB_TRY(crop_extend_u8_launch(ImgB{lv.lm, lv.lmw, lv.lmh, lv.lmw}, -dsx, -dsy, lrmw, lrmh, 1, lrm, lrmw, st));
      SgmArgs b = a;
      b.left = ImgF{rc, rcw, rch, rcw}; b.right = ImgF{l2, l2w, l2h, l2w};
      b.lmask = ImgB{rrm, rlw, rlh, rlw}; b.rmask = ImgB{lrm, lrmw, lrmh, lrmw};
      b.prev = nullptr; b.pw = b.ph = 0; b.ppitch = 0;
      if (level < levels) { b.prev = prev_rl; b.pw = prlw; b.ph = prlh; b.ppitch = prlw; }
      int ow2 = 0, oh2 = 0;
      sgm_output_size(rcw, rch, l2w, l2h, dsx, dsy, kx, &ow2, &oh2);
      if (ow2 != rlw || oh2 != rlh) { set_error("PyramidCorrelation(SGM): R->L size mismatch"); return VWB200_EMATH; }
      VWB_TRY(ar.alloc(&disp_rl, (size_t)rlw * rlh));
      b.out = disp_rl; b.opitch = rlw; b.out_sub = nullptr; b.subpixel_mode = 0;
      VWB_TRY(sgm_run(b, ar, st));
      // the R->L disparity enters the check shifted by -size and goes on un-shifted (:548-549, 586)
      VWB_TRY(consistency_launch(disp, dw, dh, dw, disp_rl, rlw, rlh, rlw, p.consistency_threshold, st, -dsx, -dsy,
                                 level == 0 ? df.d : nullptr, df.pitch, df.ox, df.oy));
    }
    if (p.filter_half_kernel > 0) {                                                             // :713-744
      const int fh = p.filter_half_kernel;
      vwb200_dispi *t1, *t2;
      VWB_TRY(ar.alloc(&t2, (size_t)dw * dh));
      if (level != 0) {
        VWB_TRY(ar.alloc(&t1, (size_t)(dw + 2) * (dh + 2)));
        VWB_TRY(rm_outliers_launch(disp, dw, dh, fh, fh, 3.0, 0.5, -1, -1, dw + 2, dh + 2, t1, st));
        VWB_TRY(cleanup_pass2_launch(t1, dw, dh, t2, st));
      } else {
        VWB_TRY(rm_outliers_launch(disp, dw, dh, fh, fh, 3.0, 0.5, 0, 0, dw, dh, t2, st));
      }
      VWB_TRY(disparity_mask_launch(t2, dw, dh, ImgB{lv.lm, lv.lmw, lv.lmh, lv.lmw}, ImgB{lv.rm, lv.rmw, lv.rmh, lv.rmw}, disp, st));
      if (level != 0 && check_rl) {
        vwb200_dispi *u1, *u2;
        VWB_TRY(ar.alloc(&u1, (size_t)(rlw + 2) * (rlh + 2)));
        VWB_TRY(ar.alloc(&u2, (size_t)rlw * rlh));
        VWB_TRY(rm_outliers_launch(disp_rl, rlw, rlh, fh, fh, 3.0, 0.5, -1, -1, rlw + 2, rlh + 2, u1, st));
        VWB_TRY(cleanup_pass2_launch(u1, rlw, rlh, u2, st));
        VWB_TRY(disparity_mask_launch(u2, rlw, rlh, ImgB{rrm, rlw, rlh, rlw}, ImgB{lrm, lrmw, lrmh, lrmw}, disp_rl, st));
      }
    }
    const int area = p.blob_filter_area / scaling;                                               // :747-749
    if (area >= 1) {
      int* work;
      VWB_TRY(ar.alloc(&work, (size_t)2 * std::max(dw * dh, check_rl ? rlw * rlh : 0)));
      VWB_TRY(blob_filter_launch(disp, dw, dh, area, work, st));
      if (check_rl && level != 0) VWB_TRY(blob_filter_launch(disp_rl, rlw, rlh, area, work, st));
    }
  }
  if (dw != bw || dh != bh) { set_error("PyramidCorrelation: Solved disparity doesn't match requested bbox size."); return VWB200_EMATH; }
  if (df.d) VWB_TRY(diff_invalidate_launch(disp, bw, bh, df.d, df.pitch, df.ox, df.oy, st));
  *d_disp_out = disp; *d_sub_out = sub;
  return VWB200_OK;
}

// stage a host image into HBM (or pass a device image through)
template <class T>
static int stage_in(const T* src, int w, int h, ptrdiff_t pitch, int on_device, Arena& ar, cudaStream_t st, const T** out, ptrdiff_t* opitch) {
  if (on_device) { *out = src; *opitch = pitch; return VWB200_OK; }
  T* d;
  VWB_TRY(ar.alloc(&d, (size_t)w * h));
  VWB_CUDA(cudaMemcpy2DAsync(d, (size_t)w * sizeof(T), src, (size_t)pitch * sizeof(T), (size_t)w * sizeof(T), h, cudaMemcpyHostToDevice, st));
  *out = d; *opitch = w;
  return VWB200_OK;
}


// ===================================================================================================
// extern "C" ABI
// ===================================================================================================
extern "C" {

const char* vwb200_last_error(void) { return t_error; }
const char* vwb200_version(void) { return "vwb200 0.1 (sm_100a)"; }
int vwb200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
long long vwb200_kernel_launches(void) { return g_launches.load(); }
// the engine keeps its stream-ordered scratch cached in the device's default memory pool between calls (ensure_device raises
// the release threshold); a host application that wants the memory back -- e.g. before a torch allocation burst -- calls this
int vwb200_trim(void) {
  VWB_TRY(ensure_device());
  int dev = 0;
  VWB_CUDA(cudaGetDevice(&dev));
  cudaMemPool_t pool;
  VWB_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
  VWB_CUDA(cudaDeviceSynchronize());
  VWB_CUDA(cudaMemPoolTrimTo(pool, 0));
  return VWB200_OK;
}
int vwb200_last_k1_stats(vwb200_k1_stats* out) { if (!out) return VWB200_EARG; *out = t_k1_stats; return VWB200_OK; }

// calc_disparity on device-resident rasters: statistics -> kernel choice -> launch(es).  Results are bit-identical
// whichever kernel runs, so callers may split a raster into bands freely.
static int calc_disparity_device(int cost_type, ImgF Li, ImgF Ri, int W, int H, int sx, int sy, int kx, int ky, vwb200_dispi* dout, ptrdiff_t dop,
                                 Arena& ar, cudaStream_t st, const KEvents* kev, int* path_out) {
  int path = 1;
  float* d_stats; float hs[6];
  VWB_TRY(ar.alloc(&d_stats, 6));
  VWB_TRY(image_stats_launch(Li, d_stats, st));
  VWB_TRY(image_stats_launch(Ri, d_stats + 3, st));
  VWB_CUDA(cudaMemcpyAsync(hs, d_stats, sizeof(hs), cudaMemcpyDeviceToHost, st));
  VWB_CUDA(cudaStreamSynchronize(st));
  const float vmin = std::min(hs[0], hs[3]), vmax = std::max(hs[1], hs[4]);
  const bool integer = hs[2] != 0.0f && hs[5] != 0.0f;
  // exact-integer fast path when the imagery allows it
  const bool force_zone_int = getenv("VWB200_K1_ZONE_INT") && integer;      // test hook: the level loop's integer zone kernel
  if (force_zone_int) {
  } else if (k1_fast_supported(cost_type, kx, ky, sx, sy, vmin, vmax, integer) == VWB200_OK) {
    const size_t wb = k1_fast_workspace_bytes(W, H, sx, sy, kx, ky);
    unsigned char* ws;
    VWB_TRY(ar.alloc(&ws, wb));
    VWB_TRY(k1_fast_launch(cost_type, Li, Ri, W, H, sx, sy, kx, ky, vmin, dout, dop, ws, wb, st, kev));
    path = 0;
  } else if (k1_screen_supported(cost_type, kx, ky, sx, sy, vmin, vmax, integer) == VWB200_OK) {
    unsigned char* ws;
    VWB_TRY(ar.alloc(&ws, k1_screen_workspace_bytes(cost_type, W, H, sx, sy, kx, ky)));
    VWB_TRY(k1_screen_launch(cost_type, Li, Ri, W, H, sx, sy, kx, ky, vmin, vmax, dout, dop, ws, st, kev));
    path = 0;
  }
  if (path == 1) {
    std::vector<Zone> zones(1);
    Zone& z = zones[0];
    z.obase = 0; z.opitch = (int)dop; z.w = W; z.h = H; z.lx = 0; z.ly = 0; z.rx = 0; z.ry = 0; z.sx = sx; z.sy = sy; z.addx = 0; z.addy = 0;
    const ZoneIntMode zim{force_zone_int, vmin, vmax, false};
    VWB_TRY(run_k1_zones(cost_type, Li, Ri, zones, kx, ky, dout, ar, st, nullptr, nullptr, nullptr, kev, nullptr, &zim));
  }
  *path_out = path;
  return VWB200_OK;
}

namespace {
struct EventGuard {              // RAII for the cudaEvents of one call (they used to leak on the error paths)
  std::vector<cudaEvent_t> ev;
  int make(cudaEvent_t* out, unsigned flags = cudaEventDefault) {
    cudaEvent_t e;
    VWB_CUDA(cudaEventCreateWithFlags(&e, flags));
    ev.push_back(e); *out = e;
    return VWB200_OK;
  }
  ~EventGuard() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
};
struct ExtraStream {
  cudaStream_t s = nullptr;
  int init() { VWB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)); return VWB200_OK; }
  ~ExtraStream() { if (s) cudaStreamDestroy(s); }
};
}  // namespace

// Host-resident rasters (the tile feeder, SURVEY 8f n3; caller pattern Image/ImageIO.h:150-314): the output rows are cut
// into bands; band b's input rows go up on a copy stream while band b-1 is correlated and band b-2's result comes down on
// a third stream.  Three band-sized buffer sets rotate, so the rasters never have to be resident as a whole.
static int calc_disparity_host_pipelined(int cost_type, const float* left, int lw, int lh, ptrdiff_t lpitch, const float* right, ptrdiff_t rpitch,
                                         int sx, int sy, int kx, int ky, vwb200_dispi* out, ptrdiff_t opitch, cudaStream_t st, int* path_out,
                                         float* kernel_ms_out) {
  const int W = lw - kx + 1, H = lh - ky + 1, rw = lw + sx - 1;
  // band schedule: a short first band (the kernels start after ~1 ms of upload), a short last band (only ~1 ms of
  // download is left when the kernels end), and in between bands as tall as a quarter of the free HBM allows -- tall
  // bands keep the persistent kernels' wave efficiency, the copies of a tall band hide behind its neighbours' kernels
  std::vector<int> ys;          // band b = output rows [ys[b], ys[b + 1])
  {
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const size_t row_bytes = (size_t)lw * 4 + (size_t)rw * 4 + (size_t)W * sizeof(vwb200_dispi);
    long long cap = (long long)(free_b / 4 / (3 * row_bytes));
    cap = std::max<long long>(256, cap / 32 * 32);
    int edge = 512;
    if (const char* e = getenv("VWB200_BAND_ROWS")) { edge = std::max(32, atoi(e)); cap = edge; }
    ys.push_back(0);
    if (H > 3 * edge) {
      ys.push_back(edge);
      int y = edge;
      const int mid_end = H - edge;
      while (y < mid_end) { y = (int)std::min<long long>(mid_end, y + cap); ys.push_back(y); }
      ys.push_back(H);
    } else {
      for (int y = edge; y < H; y += edge) ys.push_back(y);
      ys.push_back(H);
    }
  }
  const int NB = (int)ys.size() - 1;
  int BH = 0;
  for (int b = 0; b < NB; ++b) BH = std::max(BH, ys[b + 1] - ys[b]);
  constexpr int NBUF = 3;
  ExtraStream s_in, s_out;
  VWB_TRY(s_in.init()); VWB_TRY(s_out.init());
  EventGuard evs;
  std::vector<cudaEvent_t> in_done(NB), comp_done(NB), out_done(NB), k0(NB), k1(NB);
  for (int b = 0; b < NB; ++b) {
    VWB_TRY(evs.make(&in_done[b], cudaEventDisableTiming)); VWB_TRY(evs.make(&comp_done[b], cudaEventDisableTiming));
    VWB_TRY(evs.make(&out_done[b], cudaEventDisableTiming)); VWB_TRY(evs.make(&k0[b])); VWB_TRY(evs.make(&k1[b]));
  }
  Arena ar(st);
  const int lrows_max = BH + ky - 1, rrows_max = lrows_max + sy - 1;
  float* bl[NBUF]; float* br[NBUF]; vwb200_dispi* bo[NBUF];
  for (int i = 0; i < std::min(NBUF, NB); ++i) {
    VWB_TRY(ar.alloc(&bl[i], (size_t)lrows_max * lw));
    VWB_TRY(ar.alloc(&br[i], (size_t)rrows_max * rw));
    VWB_TRY(ar.alloc(&bo[i], (size_t)BH * W));
  }
  cudaEvent_t alloc_done;
  VWB_TRY(evs.make(&alloc_done, cudaEventDisableTiming));
  VWB_CUDA(cudaEventRecord(alloc_done, st));
  VWB_CUDA(cudaStreamWaitEvent(s_in.s, alloc_done, 0));
  auto upload = [&](int b) -> int {
    const int y0 = ys[b], h = ys[b + 1] - ys[b], buf = b % NBUF;
    if (b >= NBUF) VWB_CUDA(cudaStreamWaitEvent(s_in.s, comp_done[b - NBUF], 0));       // the buffers are free again
    VWB_CUDA(cudaMemcpy2DAsync(bl[buf], (size_t)lw * 4, left + (ptrdiff_t)y0 * lpitch, (size_t)lpitch * 4, (size_t)lw * 4, h + ky - 1,
                               cudaMemcpyHostToDevice, s_in.s));
    VWB_CUDA(cudaMemcpy2DAsync(br[buf], (size_t)rw * 4, right + (ptrdiff_t)y0 * rpitch, (size_t)rpitch * 4, (size_t)rw * 4, h + ky - 1 + sy - 1,
                               cudaMemcpyHostToDevice, s_in.s));
    VWB_CUDA(cudaEventRecord(in_done[b], s_in.s));
    return VWB200_OK;
  };
  for (int b = 0; b < std::min(NBUF, NB); ++b) VWB_TRY(upload(b));
  int path = 0;
  for (int b = 0; b < NB; ++b) {
    const int y0 = ys[b], h = ys[b + 1] - ys[b], buf = b % NBUF;
    VWB_CUDA(cudaStreamWaitEvent(st, in_done[b], 0));
    if (b >= NBUF) VWB_CUDA(cudaStreamWaitEvent(st, out_done[b - NBUF], 0));             // its output buffer has been read back
    const ImgF Li{bl[buf], lw, h + ky - 1, lw}, Ri{br[buf], rw, h + ky - 1 + sy - 1, rw};
    KEvents kev; kev.e0 = k0[b]; kev.e1 = k1[b];
    int pth = 1;
    {
      Arena band(st);            // the band's workspace is returned to the pool as soon as its kernels are queued
      VWB_TRY(calc_disparity_device(cost_type, Li, Ri, W, h, sx, sy, kx, ky, bo[buf], W, band, st, &kev, &pth));
    }
    path = std::max(path, pth);
    VWB_CUDA(cudaEventRecord(comp_done[b], st));
    VWB_CUDA(cudaStreamWaitEvent(s_out.s, comp_done[b], 0));
    VWB_CUDA(cudaMemcpy2DAsync(out + (ptrdiff_t)y0 * opitch, (size_t)opitch * sizeof(vwb200_dispi), bo[buf], (size_t)W * sizeof(vwb200_dispi),
                               (size_t)W * sizeof(vwb200_dispi), h, cudaMemcpyDeviceToHost, s_out.s));
    VWB_CUDA(cudaEventRecord(out_done[b], s_out.s));
    if (b + NBUF < NB) VWB_TRY(upload(b + NBUF));
  }
  VWB_CUDA(cudaStreamSynchronize(s_out.s));
  VWB_CUDA(cudaStreamSynchronize(st));
  float total = 0.0f;
  for (int b = 0; b < NB; ++b) { float ms = 0.0f; if (cudaEventElapsedTime(&ms, k0[b], k1[b]) == cudaSuccess) total += ms; else cudaGetLastError(); }
  *kernel_ms_out = total; *path_out = path;
  return VWB200_OK;
}

int vwb200_calc_disparity(int cost_type, const float* left, int lw, int lh, ptrdiff_t lpitch,
                          const float* right, int rw, int rh, ptrdiff_t rpitch,
                          int sx, int sy, int kx, int ky, vwb200_dispi* out, ptrdiff_t opitch,
                          int on_device, void* stream) {
  // argument checks of calc_disparity (Stereo/Correlation.cc:340-353)
  if (kx % 2 != 1 || ky % 2 != 1) { set_error("calc_disparity: Kernel input not sized with odd values."); return VWB200_EARG; }
  if (kx > lw || ky > lh) { set_error("calc_disparity: Kernel size too large of active region."); return VWB200_EARG; }
  if (sx <= 0 || sy <= 0) { set_error("calc_disparity: Search volume must be greater than 0."); return VWB200_EARG; }
  if (rw < lw + sx - 1 || rh < lh + sy - 1) { set_error("calc_disparity: right raster smaller than region + search volume - 1."); return VWB200_EARG; }
  if (cost_type < 0 || cost_type > 2) { set_error("calc_disparity: unsupported cost type %d", cost_type); return VWB200_EARG; }
  if (!left || !right || !out) { set_error("calc_disparity: null pointer"); return VWB200_EARG; }
  if (lpitch < lw || rpitch < lw + sx - 1 || opitch < lw - kx + 1) { set_error("calc_disparity: a row pitch is smaller than its row"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  const long long launches0 = g_launches.load();
  const int W = lw - kx + 1, H = lh - ky + 1;
  int path = 1;
  float kernel_ms = 0.0f;
  if (!on_device && (H > 1024 || getenv("VWB200_BAND_ROWS")) && !getenv("VWB200_NO_PIPELINE")) {
    VWB_TRY(calc_disparity_host_pipelined(cost_type, left, lw, lh, lpitch, right, rpitch, sx, sy, kx, ky, out, opitch, st, &path, &kernel_ms));
  } else {
    EventGuard evs;
    KEvents kev;
    VWB_TRY(evs.make(&kev.e0)); VWB_TRY(evs.make(&kev.e1));
    {
      Arena ar(st);
      const float *dl, *dr; ptrdiff_t dlp, drp;
      VWB_TRY(stage_in(left, lw, lh, lpitch, on_device, ar, st, &dl, &dlp));
      VWB_TRY(stage_in(right, lw + sx - 1, lh + sy - 1, rpitch, on_device, ar, st, &dr, &drp));
      vwb200_dispi* dout = out; ptrdiff_t dop = opitch;
      if (!on_device) { VWB_TRY(ar.alloc(&dout, (size_t)W * H)); dop = W; }
      const ImgF Li{dl, lw, lh, dlp}, Ri{dr, lw + sx - 1, lh + sy - 1, drp};
      VWB_TRY(calc_disparity_device(cost_type, Li, Ri, W, H, sx, sy, kx, ky, dout, dop, ar, st, &kev, &path));
      if (!on_device)
        VWB_CUDA(cudaMemcpy2DAsync(out, (size_t)opitch * sizeof(vwb200_dispi), dout, (size_t)W * sizeof(vwb200_dispi),
                                   (size_t)W * sizeof(vwb200_dispi), H, cudaMemcpyDeviceToHost, st));
    }
    VWB_CUDA(cudaStreamSynchronize(st));
    if (cudaEventElapsedTime(&kernel_ms, kev.e0, kev.e1) != cudaSuccess) { kernel_ms = 0.0f; cudaGetLastError(); }
  }
  t_k1_stats.path = path;
  t_k1_stats.launches = (int)(g_launches.load() - launches0);
  t_k1_stats.kernel_ms = kernel_ms;
  return VWB200_OK;
}

int vwb200_pyramid_down(const float* in, int w, int h, ptrdiff_t pitch, float* out, ptrdiff_t opitch, int on_device, void* stream) {
  if (!in || !out || w <= 0 || h <= 0) { set_error("pyramid_down: bad arguments"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    const int ow = 1 + (w - 1) / 2, oh = 1 + (h - 1) / 2;
    const float* din; ptrdiff_t dp;
    VWB_TRY(stage_in(in, w, h, pitch, on_device, ar, st, &din, &dp));
    float* dout = out; ptrdiff_t dop = opitch;
    if (!on_device) { VWB_TRY(ar.alloc(&dout, (size_t)ow * oh)); dop = ow; }
    VWB_TRY(pyramid_down_launch(ImgF{din, w, h, dp}, dout, dop, st));
    if (!on_device)
      VWB_CUDA(cudaMemcpy2DAsync(out, (size_t)opitch * sizeof(float), dout, (size_t)ow * sizeof(float), (size_t)ow * sizeof(float), oh, cudaMemcpyDeviceToHost, st));
  }
  VWB_CUDA(cudaStreamSynchronize(st));
  return VWB200_OK;
}

int vwb200_prefilter(const float* in, int w, int h, ptrdiff_t pitch, int mode, float width, float* out, ptrdiff_t opitch, int on_device, void* stream) {
  if (!in || !out || w <= 0 || h <= 0) { set_error("prefilter: bad arguments"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    float* buf;
    VWB_TRY(ar.alloc(&buf, (size_t)w * h));
    VWB_CUDA(cudaMemcpy2DAsync(buf, (size_t)w * 4, in, (size_t)pitch * 4, (size_t)w * 4, h, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    VWB_TRY(prefilter_inplace(buf, w, h, mode, width, ar, st));
    VWB_CUDA(cudaMemcpy2DAsync(out, (size_t)opitch * 4, buf, (size_t)w * 4, (size_t)w * 4, h, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
  }
  return VWB200_OK;
}

// calc_disparity_sgm behind the C ABI: stage the inputs, run vwb200::sgm_run, copy the results back
static int sgm_abi_run(const vwb200_sgm_params* sp, const float* left, int lw, int lh, ptrdiff_t lpitch, const float* right, int rw, int rh,
                       ptrdiff_t rpitch, const uint8_t* lmask, ptrdiff_t lmpitch, const uint8_t* rmask, int rmw, int rmh, ptrdiff_t rmpitch,
                       const vwb200_dispi* prev, int pw, int ph, ptrdiff_t ppitch, const int32_t* bounds, vwb200_dispi* out, ptrdiff_t opitch,
                       float* out_sub, ptrdiff_t sub_pitch, int32_t* bounds_out, int* out_w, int* out_h, int on_device, void* stream) {
  if (!sp || !left || !right || lw <= 0 || lh <= 0 || rw <= 0 || rh <= 0 || !out_w || !out_h) { set_error("sgm_calc_disparity: bad arguments"); return VWB200_EARG; }
  const int kernel_size = sp->kernel_size, search_x = sp->search_x, search_y = sp->search_y;
  if (kernel_size % 2 != 1) { set_error("calc_disparity_sgm: Kernel input not sized with odd values."); return VWB200_EARG; }       // SGM.cc:184-185
  if (kernel_size > lw || kernel_size > lh) { set_error("calc_disparity_sgm: Kernel size too large of active region."); return VWB200_EARG; }
  if (search_x < 0 || search_y < 0) { set_error("calc_disparity_sgm: negative search volume"); return VWB200_EARG; }
  if (sp->cost_type != VWB200_CENSUS_TRANSFORM && sp->cost_type != VWB200_TERNARY_CENSUS_TRANSFORM) {
    set_error("With SGM/MGM, only the census transform cost mode gives good results.");                                                // SGM.cc:1888-1892
    return VWB200_ENOIMPL;
  }
  if (out_sub && (sp->subpixel_mode < 0 || sp->subpixel_mode > 5)) { set_error("sgm: unknown sub-pixel mode %d", sp->subpixel_mode); return VWB200_EARG; }
  VWB_TRY(sgm_output_size(lw, lh, rw, rh, search_x, search_y, kernel_size, out_w, out_h));
  if (!out && !out_sub && !bounds_out) return VWB200_OK;           // size query
  const int W = *out_w, H = *out_h;
  if ((out && opitch < W) || (out_sub && sub_pitch < W)) { set_error("sgm_calc_disparity: output pitch smaller than the output width"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    SgmArgs a;
    const float *dl, *dr; ptrdiff_t dlp, drp;
    VWB_TRY(stage_in(left, lw, lh, lpitch, on_device, ar, st, &dl, &dlp));
    VWB_TRY(stage_in(right, rw, rh, rpitch, on_device, ar, st, &dr, &drp));
    a.left = ImgF{dl, lw, lh, dlp}; a.right = ImgF{dr, rw, rh, drp};
    a.sx = search_x; a.sy = search_y; a.k = kernel_size;
    a.ternary = sp->cost_type == VWB200_TERNARY_CENSUS_TRANSFORM; a.ternary_threshold = sp->ternary_threshold;
    a.p1 = sp->p1; a.p2 = sp->p2; a.use_mgm = sp->use_mgm; a.subpixel_mode = out_sub ? sp->subpixel_mode : 0;
    a.buf_x = sp->search_buffer_x; a.buf_y = sp->search_buffer_y; a.conserve_level = sp->conserve_level;
    a.memory_limit_mb = sp->memory_limit_mb > 0 ? sp->memory_limit_mb : 6000.0;
    a.assumed_threads = sp->assumed_threads > 0 ? sp->assumed_threads : 4;
    if (W > 0 && H > 0) {
      if (lmask) {
        const uint8_t* d; ptrdiff_t dp;
        VWB_TRY(stage_in(lmask, W, H, lmpitch, on_device, ar, st, &d, &dp));
        a.lmask = ImgB{d, W, H, dp};
      }
      if (rmask) {
        const uint8_t* d; ptrdiff_t dp;
        VWB_TRY(stage_in(rmask, rmw, rmh, rmpitch, on_device, ar, st, &d, &dp));
        a.rmask = ImgB{d, rmw, rmh, dp};
      }
      if (prev) {
        if (pw <= 0 || ph <= 0) { set_error("sgm: empty previous disparity"); return VWB200_EARG; }
        const vwb200_dispi* d; ptrdiff_t dp;
        VWB_TRY(stage_in(prev, pw, ph, ppitch, on_device, ar, st, &d, &dp));
        a.prev = d; a.pw = pw; a.ph = ph; a.ppitch = dp;
      }
      if (bounds) {
        const int32_t* d; ptrdiff_t dp;
        VWB_TRY(stage_in(bounds, W * 4, H, (ptrdiff_t)W * 4, on_device, ar, st, &d, &dp));
        a.bounds_in = d;
      }
      vwb200_dispi* dout = out; ptrdiff_t dop = opitch;
      if (!on_device || !out) { VWB_TRY(ar.alloc(&dout, (size_t)W * H)); dop = W; }
      float* dsub = out_sub; ptrdiff_t dsp = sub_pitch * 3;
      if (out_sub && !on_device) { VWB_TRY(ar.alloc(&dsub, (size_t)W * H * 3)); dsp = (ptrdiff_t)W * 3; }
      int32_t* dbo = bounds_out;
      if (bounds_out && !on_device) VWB_TRY(ar.alloc(&dbo, (size_t)W * H * 4));
      a.out = dout; a.opitch = dop; a.out_sub = out_sub ? dsub : nullptr; a.sub_pitch = dsp; a.bounds_out = dbo;
      VWB_TRY(sgm_run(a, ar, st));
      if (!on_device && out)
        VWB_CUDA(cudaMemcpy2DAsync(out, (size_t)opitch * sizeof(vwb200_dispi), dout, (size_t)W * sizeof(vwb200_dispi),
                                   (size_t)W * sizeof(vwb200_dispi), H, cudaMemcpyDeviceToHost, st));
      if (!on_device && out_sub)
        VWB_CUDA(cudaMemcpy2DAsync(out_sub, (size_t)sub_pitch * 12, dsub, (size_t)W * 12, (size_t)W * 12, H, cudaMemcpyDeviceToHost, st));
      if (!on_device && bounds_out)
        VWB_CUDA(cudaMemcpyAsync(bounds_out, dbo, (size_t)W * H * 16, cudaMemcpyDeviceToHost, st));
    }
    VWB_CUDA(cudaStreamSynchronize(st));
  }
  return VWB200_OK;
}

static vwb200_sgm_params sgm_default_params(int search_x, int search_y, int kernel_size, int p1, int p2, int subpixel_mode) {
  vwb200_sgm_params sp{};
  sp.search_x = search_x; sp.search_y = search_y; sp.kernel_size = kernel_size; sp.cost_type = VWB200_CENSUS_TRANSFORM; sp.ternary_threshold = 5;
  sp.p1 = p1; sp.p2 = p2; sp.use_mgm = 0; sp.subpixel_mode = subpixel_mode; sp.search_buffer_x = 2; sp.search_buffer_y = 2; sp.conserve_level = -1;
  sp.memory_limit_mb = 1e12; sp.assumed_threads = 4;
  return sp;
}
int vwb200_sgm_calc_disparity(const float* left, int lw, int lh, ptrdiff_t lpitch, const float* right, int rw, int rh, ptrdiff_t rpitch,
                              int search_x, int search_y, int kernel_size, int p1, int p2, vwb200_dispi* out, ptrdiff_t opitch,
                              int* out_w, int* out_h, int on_device, void* stream) {
  const vwb200_sgm_params sp = sgm_default_params(search_x, search_y, kernel_size, p1, p2, 0);
  return sgm_abi_run(&sp, left, lw, lh, lpitch, right, rw, rh, rpitch, nullptr, 0, nullptr, 0, 0, 0, nullptr, 0, 0, 0, nullptr, out, opitch, nullptr, 0,
                     nullptr, out_w, out_h, on_device, stream);
}
int vwb200_sgm_calc_disparity_subpixel(const float* left, int lw, int lh, ptrdiff_t lpitch, const float* right, int rw, int rh, ptrdiff_t rpitch,
                                       int search_x, int search_y, int kernel_size, int p1, int p2, int subpixel_mode,
                                       vwb200_dispi* out, ptrdiff_t opitch, float* out_sub, ptrdiff_t sub_pitch,
                                       int* out_w, int* out_h, int on_device, void* stream) {
  if (subpixel_mode < 0 || subpixel_mode > 5) { set_error("sgm: unknown sub-pixel mode %d", subpixel_mode); return VWB200_EARG; }
  const vwb200_sgm_params sp = sgm_default_params(search_x, search_y, kernel_size, p1, p2, subpixel_mode);
  return sgm_abi_run(&sp, left, lw, lh, lpitch, right, rw, rh, rpitch, nullptr, 0, nullptr, 0, 0, 0, nullptr, 0, 0, 0, nullptr, out, opitch, out_sub,
                     sub_pitch, nullptr, out_w, out_h, on_device, stream);
}
int vwb200_sgm_calc_disparity_ex(const vwb200_sgm_params* params, const float* left, int lw, int lh, ptrdiff_t lpitch,
                                 const float* right, int rw, int rh, ptrdiff_t rpitch,
                                 const uint8_t* lmask, ptrdiff_t lmpitch, const uint8_t* rmask, int rmw, int rmh, ptrdiff_t rmpitch,
                                 const vwb200_dispi* prev, int pw, int ph, ptrdiff_t ppitch, const int32_t* bounds,
                                 vwb200_dispi* out, ptrdiff_t opitch, float* out_sub, ptrdiff_t sub_pitch, int32_t* bounds_out,
                                 int* out_w, int* out_h, int on_device, void* stream) {
  return sgm_abi_run(params, left, lw, lh, lpitch, right, rw, rh, rpitch, lmask, lmpitch, rmask, rmw, rmh, rmpitch, prev, pw, ph, ppitch, bounds, out,
                     opitch, out_sub, sub_pitch, bounds_out, out_w, out_h, on_device, stream);
}
int vwb200_sgm_disp_bounds(const vwb200_sgm_params* sp, const vwb200_dispi* prev, int pw, int ph, ptrdiff_t ppitch,
                           const uint8_t* lmask, ptrdiff_t lmpitch, const uint8_t* rmask, int rmw, int rmh, ptrdiff_t rmpitch,
                           int ow, int oh, int32_t* bounds, int on_device, void* stream) {
  if (!sp || !bounds || ow <= 0 || oh <= 0 || sp->search_x < 0 || sp->search_y < 0) { set_error("sgm_disp_bounds: bad arguments"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    SgmArgs a;
    a.sx = sp->search_x; a.sy = sp->search_y; a.buf_x = sp->search_buffer_x; a.buf_y = sp->search_buffer_y; a.conserve_level = sp->conserve_level;
    a.use_mgm = sp->use_mgm; a.memory_limit_mb = sp->memory_limit_mb > 0 ? sp->memory_limit_mb : 6000.0;
    a.assumed_threads = sp->assumed_threads > 0 ? sp->assumed_threads : 4;
    if (lmask) { const uint8_t* d; ptrdiff_t dp; VWB_TRY(stage_in(lmask, ow, oh, lmpitch, on_device, ar, st, &d, &dp)); a.lmask = ImgB{d, ow, oh, dp}; }
    if (rmask) { const uint8_t* d; ptrdiff_t dp; VWB_TRY(stage_in(rmask, rmw, rmh, rmpitch, on_device, ar, st, &d, &dp)); a.rmask = ImgB{d, rmw, rmh, dp}; }
    if (prev) { const vwb200_dispi* d; ptrdiff_t dp; VWB_TRY(stage_in(prev, pw, ph, ppitch, on_device, ar, st, &d, &dp)); a.prev = d; a.pw = pw; a.ph = ph; a.ppitch = dp; }
    int32_t* db = bounds;
    if (!on_device) VWB_TRY(ar.alloc(&db, (size_t)ow * oh * 4));
    VWB_TRY(sgm_bounds_run(a, ow, oh, db, ar, st));
    if (!on_device) VWB_CUDA(cudaMemcpyAsync(bounds, db, (size_t)ow * oh * 16, cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
  }
  return VWB200_OK;
}

int vwb200_parabola_subpixel(const float* disparity, int cols, int rows, const float* left, ptrdiff_t lpitch,
                             const float* right, int rcols, int rrows, ptrdiff_t rpitch, int kx, int ky,
                             int prefilter_mode, float prefilter_width, int x0, int y0, int x1, int y1,
                             float* dest, ptrdiff_t dest_pitch, int on_device, void* stream) {
  if (!disparity || !left || !right || !dest) { set_error("parabola_subpixel: null pointer"); return VWB200_EARG; }
  if (x1 <= x0 || y1 <= y0 || x0 < 0 || y0 < 0 || x1 > cols || y1 > rows) { set_error("parabola_subpixel: bbox outside the disparity image"); return VWB200_EARG; }
  if (kx % 2 != 1 || ky % 2 != 1 || kx < 1 || ky < 1) { set_error("parabola_subpixel: kernel size must be odd"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    const int bw = x1 - x0, bh = y1 - y0;
    const float *dd, *dl, *dr; ptrdiff_t p0, p1, p2;
    VWB_TRY(stage_in(disparity, cols * 3, rows, (ptrdiff_t)cols * 3, on_device, ar, st, &dd, &p0));
    VWB_TRY(stage_in(left, cols, rows, lpitch, on_device, ar, st, &dl, &p1));
    VWB_TRY(stage_in(right, rcols, rrows, rpitch, on_device, ar, st, &dr, &p2));
    int* d_r; int hr[5];
    VWB_TRY(ar.alloc(&d_r, 5));
    VWB_TRY(disp_range_launch(dd, cols, x0, y0, bw, bh, d_r, st));
    VWB_CUDA(cudaMemcpyAsync(hr, d_r, sizeof(hr), cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
    if (!hr[4]) { hr[0] = hr[1] = hr[2] = hr[3] = 0; }
    // entire_search_range: max += 1, expand(1)  (ParabolaSubpixelView.cc:296-299)
    const Box sr{hr[0] - 1, hr[1] - 1, hr[2] + 2, hr[3] + 2};
    const int hkx = kx / 2, hky = ky / 2;
    const Box lreg{x0 - hkx, y0 - hky, x1 + hkx, y1 + hky};
    const Box rreg{lreg.x0 + sr.x0, lreg.y0 + sr.y0, lreg.x1 + sr.x0 + (sr.x1 - sr.x0), lreg.y1 + sr.y0 + (sr.y1 - sr.y0)};
    float *Lf, *Rf;
    VWB_TRY(filtered_region(ImgF{dl, cols, rows, p1}, prefilter_mode, prefilter_width, lreg, &Lf, ar, st));
    VWB_TRY(filtered_region(ImgF{dr, rcols, rrows, p2}, prefilter_mode, prefilter_width, rreg, &Rf, ar, st));
    float* dout = dest;
    if (!on_device || dest_pitch != bw) VWB_TRY(ar.alloc(&dout, (size_t)bw * bh * 3));
    VWB_TRY(parabola_launch(dd, cols, x0, y0, bw, bh, Lf, lreg.x1 - lreg.x0, Rf, rreg.x1 - rreg.x0, sr.x0, sr.y0, kx, ky, dout, st));
    if (dout != dest)
      VWB_CUDA(cudaMemcpy2DAsync(dest, (size_t)dest_pitch * 12, dout, (size_t)bw * 12, (size_t)bw * 12, bh,
                                 on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
  }
  return VWB200_OK;
}

// ---- K6: PyramidSubpixelView and the level functions -------------------------------------------------------------
static thread_local vwb200_subpixel_stats t_subpixel_stats = {0, 0, 0, 0, 0, 0};

int vwb200_last_subpixel_stats(vwb200_subpixel_stats* out) { if (!out) return VWB200_EARG; *out = t_subpixel_stats; return VWB200_OK; }

static int subpixel_check_algorithm(int algorithm, const char* who) {
  if (algorithm == VWB200_SUBPIXEL_PHASE) { set_error("%s: SUBPIXEL_PHASE is not implemented", who); return VWB200_ENOIMPL; }
  if (algorithm < VWB200_SUBPIXEL_LUCAS_KANADE || algorithm > VWB200_SUBPIXEL_BAYES_EM) {
    set_error("%s: invalid algorithm %d", who, algorithm);
    return VWB200_ENOIMPL;
  }
  return VWB200_OK;
}

int vwb200_pyramid_subpixel(const float* disparity, int cols, int rows, const float* left, ptrdiff_t lpitch,
                            const float* right, int rcols, int rrows, ptrdiff_t rpitch, int kx, int ky,
                            int prefilter_mode, float prefilter_width, int x0, int y0, int x1, int y1,
                            float* dest, ptrdiff_t dest_pitch, int on_device, void* stream,
                            int max_pyramid_levels, int algorithm) {
  t_subpixel_stats = vwb200_subpixel_stats{0, 0, 0, 0, 0, 0};
  if (!disparity || !left || !right || !dest) { set_error("pyramid_subpixel: null pointer"); return VWB200_EARG; }
  if (x1 <= x0 || y1 <= y0 || x0 < 0 || y0 < 0 || x1 > cols || y1 > rows) { set_error("pyramid_subpixel: bbox outside the disparity image"); return VWB200_EARG; }
  if (kx % 2 != 1 || ky % 2 != 1 || kx < 3 || ky < 3) { set_error("pyramid_subpixel: kernel size must be odd and >= 3"); return VWB200_EARG; }
  if (prefilter_mode < VWB200_PREFILTER_NONE || prefilter_mode > VWB200_PREFILTER_MEANSUB) { set_error("unknown prefilter mode %d", prefilter_mode); return VWB200_EARG; }
  VWB_TRY(subpixel_check_algorithm(algorithm, "pyramid_subpixel"));
  const int levels = max_pyramid_levels < 0 ? 0 : max_pyramid_levels;
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    const int bw = x1 - x0, bh = y1 - y0;
    const float *dd, *dl, *dr; ptrdiff_t p0, p1, p2;
    VWB_TRY(stage_in(disparity, cols * 3, rows, (ptrdiff_t)cols * 3, on_device, ar, st, &dd, &p0));
    VWB_TRY(stage_in(left, cols, rows, lpitch, on_device, ar, st, &dl, &p1));
    VWB_TRY(stage_in(right, rcols, rrows, rpitch, on_device, ar, st, &dr, &p2));
    // get_disparity_range over the bbox crop: the only host round trip of the pipeline
    int* d_r; int hr[5];
    VWB_TRY(ar.alloc(&d_r, 5));
    VWB_TRY(k6_range_launch(dd, cols, x0, y0, bw, bh, d_r, st));
    VWB_CUDA(cudaMemcpyAsync(hr, d_r, sizeof(hr), cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
    if (hr[4]) { set_error("pyramid_subpixel: disparity values in the bbox must be finite and below 2^24 in magnitude"); return VWB200_EARG; }
    // SubpixelView.cc:45-61: right = bbox + range, left widened to the right's size, both grown by the kernel size
    const Box rreg{x0 + hr[0] - kx, y0 + hr[1] - ky, x1 + hr[2] + kx, y1 + hr[3] + ky};
    const int pw = rreg.x1 - rreg.x0, ph = rreg.y1 - rreg.y0;
    const Box lreg{x0 - kx, y0 - ky, x0 - kx + pw, y0 - ky + ph};
    float *Lf, *Rf, *D;
    VWB_TRY(filtered_region(ImgF{dl, cols, rows, p1}, prefilter_mode, prefilter_width, lreg, &Lf, ar, st));
    VWB_TRY(filtered_region(ImgF{dr, rcols, rrows, p2}, prefilter_mode, prefilter_width, rreg, &Rf, ar, st));
    VWB_TRY(ar.alloc(&D, (size_t)pw * ph * 3));
    VWB_TRY(k6_disp_crop_launch(dd, cols, rows, lreg.x0, lreg.y0, pw, ph, (float)hr[0], (float)hr[1], D, st));
    VWB_TRY(k6_pyramid_run(algorithm, D, Lf, Rf, pw, ph, kx, ky, bw, bh, levels, ar, st, &t_subpixel_stats));
    float* dout = dest;
    ptrdiff_t opitch = dest_pitch;
    if (!on_device) { VWB_TRY(ar.alloc(&dout, (size_t)bw * bh * 3)); opitch = bw; }
    VWB_TRY(k6_disp_out_launch(D, pw, kx, ky, (float)hr[0], (float)hr[1], bw, bh, dout, opitch, st));
    if (dout != dest)
      VWB_CUDA(cudaMemcpy2DAsync(dest, (size_t)dest_pitch * 12, dout, (size_t)bw * 12, (size_t)bw * 12, bh, cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
  }
  return VWB200_OK;
}

int vwb200_subpixel_refine(int algorithm, float* disparity, int cols, int rows, ptrdiff_t dpitch,
                           const float* left, ptrdiff_t lpitch, const float* right, int rcols, int rrows, ptrdiff_t rpitch,
                           int kx, int ky, int x0, int y0, int x1, int y1, int do_h, int do_v, int on_device, void* stream) {
  t_subpixel_stats = vwb200_subpixel_stats{0, 0, 0, 0, 0, 0};
  if (!disparity || !left || !right) { set_error("subpixel_refine: null pointer"); return VWB200_EARG; }
  if (cols <= 0 || rows <= 0 || rcols <= 0 || rrows <= 0) { set_error("subpixel_refine: empty image"); return VWB200_EARG; }
  if (kx % 2 != 1 || ky % 2 != 1 || kx < 3 || ky < 3) { set_error("subpixel_refine: kernel size must be odd and >= 3"); return VWB200_EARG; }
  VWB_TRY(subpixel_check_algorithm(algorithm, "subpixel_refine"));
  if (!do_h && !do_v) return VWB200_OK;                                            // Correlate.cc:512, :861, :1213
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    const float *dl, *dr; ptrdiff_t p1, p2;
    VWB_TRY(stage_in(left, cols, rows, lpitch, on_device, ar, st, &dl, &p1));
    VWB_TRY(stage_in(right, rcols, rrows, rpitch, on_device, ar, st, &dr, &p2));
    float *D, *L = const_cast<float*>(dl), *R = const_cast<float*>(dr);
    VWB_TRY(ar.alloc(&D, (size_t)cols * rows * 3));
    VWB_CUDA(cudaMemcpy2DAsync(D, (size_t)cols * 12, disparity, (size_t)dpitch * 12, (size_t)cols * 12, rows,
                               on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    if (p1 != cols) {
      VWB_TRY(ar.alloc(&L, (size_t)cols * rows));
      VWB_CUDA(cudaMemcpy2DAsync(L, (size_t)cols * 4, dl, (size_t)p1 * 4, (size_t)cols * 4, rows, cudaMemcpyDeviceToDevice, st));
    }
    if (p2 != rcols) {
      VWB_TRY(ar.alloc(&R, (size_t)rcols * rrows));
      VWB_CUDA(cudaMemcpy2DAsync(R, (size_t)rcols * 4, dr, (size_t)p2 * 4, (size_t)rcols * 4, rrows, cudaMemcpyDeviceToDevice, st));
    }
    VWB_TRY(k6_level_run(algorithm, D, L, cols, rows, R, rcols, rrows, kx, ky, x0, y0, x1, y1, ar, st, &t_subpixel_stats));
    VWB_CUDA(cudaMemcpy2DAsync(disparity, (size_t)dpitch * 12, D, (size_t)cols * 12, (size_t)cols * 12, rows,
                               on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
  }
  return VWB200_OK;
}

// ---- K7: CorrEval ------------------------------------------------------------------------------------------------
int vwb200_corr_eval(const float* left, int lw, int lh, ptrdiff_t lpitch, const float* right, int rw, int rh, ptrdiff_t rpitch,
                     const float* disparity, ptrdiff_t dpitch, int kx, int ky, int metric, int sample_rate, int round_to_int,
                     float prefilter_kernel_width, int x0, int y0, int x1, int y1, float* dest, ptrdiff_t dest_pitch,
                     int on_device, void* stream) {
  if (!left || !right || !disparity || !dest) { set_error("corr_eval: null pointer"); return VWB200_EARG; }
  if (lw <= 0 || lh <= 0 || rw <= 0 || rh <= 0) { set_error("corr_eval: empty image"); return VWB200_EARG; }
  if (!(kx > 0 && kx % 2 == 1 && ky > 0 && ky % 2 == 1)) { set_error("CorrEval: The kernel dimensions must be positive and odd."); return VWB200_EARG; }
  if (metric < VWB200_CORR_EVAL_NCC || metric > VWB200_CORR_EVAL_CRAMER_RAO) { set_error("CorrEval: Invalid metric: %d.", metric); return VWB200_EARG; }
  if (sample_rate < 1) { set_error("CorrEval: the sample rate must be at least 1"); return VWB200_EARG; }
  if (x1 <= x0 || y1 <= y0 || x0 < 0 || y0 < 0 || x1 > lw || y1 > lh) { set_error("corr_eval: bbox outside the left image"); return VWB200_EARG; }
  // m_extra_padding = (int)ceil(prefilter_kernel_width) + 5 (CorrEval.h:77)
  const float pad = ceilf(prefilter_kernel_width) + 5.0f;
  if (!(pad >= 0.0f && pad <= 1048576.0f)) { set_error("corr_eval: prefilter_kernel_width must give a padding ceil(w) + 5 in [0, 2^20]"); return VWB200_EARG; }
  const bool curvature = metric == VWB200_CORR_EVAL_PARABOLA_CURVATURE || metric == VWB200_CORR_EVAL_CRAMER_RAO;
  const int margin = 1 + 2 + (int)pad + (curvature ? 1 : 0);   // CorrEval.cc:205-214
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  const int bw = x1 - x0, bh = y1 - y0;
  int bad = 0;
  {
    Arena ar(st);
    const float *dl, *dr, *dd; ptrdiff_t pl, pr, pd;
    VWB_TRY(stage_in(left, lw * 2, lh, lpitch * 2, on_device, ar, st, &dl, &pl));
    VWB_TRY(stage_in(right, rw * 2, rh, rpitch * 2, on_device, ar, st, &dr, &pr));
    VWB_TRY(stage_in(disparity, lw * 3, lh, dpitch * 3, on_device, ar, st, &dd, &pd));
    int* d_org;
    VWB_TRY(ar.alloc(&d_org, 3));
    VWB_TRY(k7_origin_launch(dd, pd / 3, x0, y0, bw, bh, sample_rate, round_to_int, d_org, st));
    float* dout = dest;
    ptrdiff_t opitch = dest_pitch;
    if (!on_device) { VWB_TRY(ar.alloc(&dout, (size_t)bw * bh * 2)); opitch = bw; }
    VWB_TRY(k7_corr_eval_launch(dl, lw, lh, pl / 2, dr, rw, rh, pr / 2, dd, pd / 3, x0, y0, bw, bh, kx, ky, metric, sample_rate,
                                round_to_int, margin, d_org, dout, opitch, st));
    VWB_CUDA(cudaMemcpyAsync(&bad, d_org + 2, sizeof(int), cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
    if (!bad && dout != dest) {
      VWB_CUDA(cudaMemcpy2DAsync(dest, (size_t)dest_pitch * 8, dout, (size_t)bw * 8, (size_t)bw * 8, bh, cudaMemcpyDeviceToHost, st));
      VWB_CUDA(cudaStreamSynchronize(st));
    }
  }
  if (bad) { set_error("corr_eval: sampled valid disparities in the bbox must be finite and below 2^24 in magnitude"); return VWB200_EARG; }
  return VWB200_OK;
}

int vwb200_subsample_mask_by_two(const uint8_t* in, int w, int h, ptrdiff_t pitch, uint8_t* out, ptrdiff_t opitch, int on_device, void* stream) {
  if (!in || !out || w <= 0 || h <= 0) { set_error("subsample_mask_by_two: bad arguments"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    const int ow = 1 + (w - 1) / 2, oh = 1 + (h - 1) / 2;
    const uint8_t* din; ptrdiff_t dp;
    VWB_TRY(stage_in(in, w, h, pitch, on_device, ar, st, &din, &dp));
    uint8_t* dout = out; ptrdiff_t dop = opitch;
    if (!on_device) { VWB_TRY(ar.alloc(&dout, (size_t)ow * oh)); dop = ow; }
    VWB_TRY(subsample_mask_launch(ImgB{din, w, h, dp}, dout, dop, st));
    if (!on_device)
      VWB_CUDA(cudaMemcpy2DAsync(out, (size_t)opitch, dout, (size_t)ow, (size_t)ow, oh, cudaMemcpyDeviceToHost, st));
  }
  VWB_CUDA(cudaStreamSynchronize(st));
  return VWB200_OK;
}

int vwb200_cross_corr_consistency_check(vwb200_dispi* l2r, int lw, int lh, ptrdiff_t lpitch, const vwb200_dispi* r2l, int rw, int rh,
                                        ptrdiff_t rpitch, float threshold, int on_device, void* stream) {
  if (!l2r || !r2l) { set_error("cross_corr_consistency_check: null pointer"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    vwb200_dispi* dl = l2r; const vwb200_dispi* dr = r2l; ptrdiff_t dlp = lpitch, drp = rpitch;
    if (!on_device) {
      VWB_TRY(ar.alloc(&dl, (size_t)lw * lh));
      VWB_CUDA(cudaMemcpy2DAsync(dl, (size_t)lw * 12, l2r, (size_t)lpitch * 12, (size_t)lw * 12, lh, cudaMemcpyHostToDevice, st));
      dlp = lw;
      VWB_TRY(stage_in(r2l, rw, rh, rpitch, 0, ar, st, &dr, &drp));
    }
    VWB_TRY(consistency_launch(dl, lw, lh, dlp, dr, rw, rh, drp, threshold, st));
    if (!on_device)
      VWB_CUDA(cudaMemcpy2DAsync(l2r, (size_t)lpitch * 12, dl, (size_t)lw * 12, (size_t)lw * 12, lh, cudaMemcpyDeviceToHost, st));
  }
  VWB_CUDA(cudaStreamSynchronize(st));
  return VWB200_OK;
}

static int filter_common(int which, const vwb200_dispi* in, int w, int h, int hx, int hy, double pt, double rt,
                         const uint8_t* lm, const uint8_t* rm, int rmw, int rmh, vwb200_dispi* out, int on_device, void* stream) {
  if (!in || !out || w <= 0 || h <= 0) { set_error("disparity filter: bad arguments"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  StreamGuard sg; VWB_TRY(sg.init(stream, on_device));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    const vwb200_dispi* din; ptrdiff_t dp;
    VWB_TRY(stage_in(in, w, h, (ptrdiff_t)w, on_device, ar, st, &din, &dp));
    vwb200_dispi* dout = out;
    if (!on_device) VWB_TRY(ar.alloc(&dout, (size_t)w * h));
    if (which == 0) {
      VWB_TRY(rm_outliers_launch(din, w, h, hx, hy, pt, rt, 0, 0, w, h, dout, st));
    } else if (which == 1) {
      vwb200_dispi* t1;
      VWB_TRY(ar.alloc(&t1, (size_t)(w + 2) * (h + 2)));
      VWB_TRY(rm_outliers_launch(din, w, h, hx, hy, pt, rt, -1, -1, w + 2, h + 2, t1, st));
      VWB_TRY(cleanup_pass2_launch(t1, w, h, dout, st));
    } else {
      const uint8_t *dlm, *drm; ptrdiff_t p1, p2;
      VWB_TRY(stage_in(lm, w, h, (ptrdiff_t)w, on_device, ar, st, &dlm, &p1));
      VWB_TRY(stage_in(rm, rmw, rmh, (ptrdiff_t)rmw, on_device, ar, st, &drm, &p2));
      VWB_TRY(disparity_mask_launch(din, w, h, ImgB{dlm, w, h, p1}, ImgB{drm, rmw, rmh, p2}, dout, st));
    }
    if (!on_device) VWB_CUDA(cudaMemcpyAsync(out, dout, (size_t)w * h * sizeof(vwb200_dispi), cudaMemcpyDeviceToHost, st));
  }
  VWB_CUDA(cudaStreamSynchronize(st));
  return VWB200_OK;
}
int vwb200_rm_outliers_using_thresh(const vwb200_dispi* in, int w, int h, int hx, int hy, double pt, double rt, vwb200_dispi* out, int on_device, void* stream) {
  return filter_common(0, in, w, h, hx, hy, pt, rt, nullptr, nullptr, 0, 0, out, on_device, stream);
}
int vwb200_disparity_cleanup_using_thresh(const vwb200_dispi* in, int w, int h, int hx, int hy, double pt, double rt, vwb200_dispi* out, int on_device, void* stream) {
  return filter_common(1, in, w, h, hx, hy, pt, rt, nullptr, nullptr, 0, 0, out, on_device, stream);
}
int vwb200_disparity_mask(const vwb200_dispi* in, int w, int h, const uint8_t* lm, const uint8_t* rm, int rmw, int rmh, vwb200_dispi* out, int on_device, void* stream) {
  if (!lm || !rm) { set_error("disparity_mask: null mask"); return VWB200_EARG; }
  return filter_common(2, in, w, h, 1, 1, 0, 0, lm, rm, rmw, rmh, out, on_device, stream);
}

// ---- the view -------------------------------------------------------------------------------------
int vwb200_corr_create(const vwb200_corr_params* p, vwb200_corr** out) {
  if (!p || !out) { set_error("corr_create: null pointer"); return VWB200_EARG; }
  const double w = (double)p->search_x1 - p->search_x0, h = (double)p->search_y1 - p->search_y0;
  if (!(w * h == w * h)) { set_error("PyramidCorrelationView: Invalid search region"); return VWB200_EARG; }   // CorrelationView.h:88-94
  if (p->search_x1 <= p->search_x0 || p->search_y1 <= p->search_y0) { set_error("PyramidCorrelationView: empty search region"); return VWB200_EARG; }
  if (p->kernel_x % 2 != 1 || p->kernel_y % 2 != 1 || p->kernel_x < 1 || p->kernel_y < 1) { set_error("PyramidCorrelationView: kernel size must be odd"); return VWB200_EARG; }
  if (p->algorithm < VWB200_CORRELATION_BM || p->algorithm > VWB200_CORRELATION_FINAL_MGM) { set_error("unknown correlation algorithm %d", p->algorithm); return VWB200_EARG; }
  if (p->cost_type < 0 || p->cost_type > VWB200_TERNARY_CENSUS_TRANSFORM) { set_error("unknown cost type %d", p->cost_type); return VWB200_EARG; }
  vwb200_corr* h_ = new vwb200_corr();
  h_->p = *p;
  // CorrelationView.h:96-105 (float maths)
  const int largest_search = std::max(p->search_x1 - p->search_x0, p->search_y1 - p->search_y0);
  int m = (int)(std::floor(std::log((float)largest_search) / std::log(2.0f)) - 1);
  if (m > p->max_pyramid_levels) m = p->max_pyramid_levels;
  if (m < 0) m = 0;
  h_->max_level_by_search = m;
  *out = h_;
  return VWB200_OK;
}

int vwb200_corr_set_inputs(vwb200_corr* h, const float* left, int lcols, int lrows, ptrdiff_t lpitch,
                           const float* right, int rcols, int rrows, ptrdiff_t rpitch,
                           const uint8_t* lmask, ptrdiff_t lmpitch, const uint8_t* rmask, ptrdiff_t rmpitch, int on_device) {
  if (!h || !left || !right || !lmask || !rmask || lcols <= 0 || lrows <= 0 || rcols <= 0 || rrows <= 0) { set_error("corr_set_inputs: bad arguments"); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  h->release();
  VWB_CUDA(cudaGetDevice(&h->device));
  h->lcols = lcols; h->lrows = lrows; h->rcols = rcols; h->rrows = rrows;
  if (on_device == VWB200_INPUTS_STREAMED) {          // host rasters, fed tile by tile
    h->L = left; h->R = right; h->Lm = lmask; h->Rm = rmask;
    h->lpitch = lpitch; h->rpitch = rpitch; h->lmpitch = lmpitch; h->rmpitch = rmpitch;
    h->streamed = true;
    return VWB200_OK;
  }
  if (on_device) {
    h->L = left; h->R = right; h->Lm = lmask; h->Rm = rmask;
    h->lpitch = lpitch; h->rpitch = rpitch; h->lmpitch = lmpitch; h->rmpitch = rmpitch;
    return VWB200_OK;
  }
  float *dl, *dr; uint8_t *dlm, *drm;
  VWB_CUDA(cudaMalloc(&dl, (size_t)lcols * lrows * 4)); VWB_CUDA(cudaMalloc(&dr, (size_t)rcols * rrows * 4));
  VWB_CUDA(cudaMalloc(&dlm, (size_t)lcols * lrows)); VWB_CUDA(cudaMalloc(&drm, (size_t)rcols * rrows));
  h->L = dl; h->R = dr; h->Lm = dlm; h->Rm = drm; h->owned = true;
  h->lpitch = lcols; h->rpitch = rcols; h->lmpitch = lcols; h->rmpitch = rcols;
  VWB_CUDA(cudaMemcpy2D(dl, (size_t)lcols * 4, left, (size_t)lpitch * 4, (size_t)lcols * 4, lrows, cudaMemcpyHostToDevice));
  VWB_CUDA(cudaMemcpy2D(dr, (size_t)rcols * 4, right, (size_t)rpitch * 4, (size_t)rcols * 4, rrows, cudaMemcpyHostToDevice));
  VWB_CUDA(cudaMemcpy2D(dlm, (size_t)lcols, lmask, (size_t)lmpitch, (size_t)lcols, lrows, cudaMemcpyHostToDevice));
  VWB_CUDA(cudaMemcpy2D(drm, (size_t)rcols, rmask, (size_t)rmpitch, (size_t)rcols, rrows, cudaMemcpyHostToDevice));
  return VWB200_OK;
}

int vwb200_corr_cols(const vwb200_corr* h) { return h ? h->lcols : 0; }
int vwb200_corr_rows(const vwb200_corr* h) { return h ? h->lrows : 0; }
int vwb200_corr_num_levels(const vwb200_corr* h, int bw, int bh) { return h ? h->num_levels(bw, bh) : VWB200_EARG; }

static int corr_rasterize_impl(vwb200_corr* h, int x0, int y0, int x1, int y1, float* dest, ptrdiff_t dest_pitch, int dest_on_device, void* stream,
                               bool with_collar) {
  if (!h || !dest) { set_error("corr_rasterize: null pointer"); return VWB200_EARG; }
  if (!h->L) { set_error("corr_rasterize: inputs not set"); return VWB200_ELOGIC; }
  if (x1 <= x0 || y1 <= y0) { set_error("corr_rasterize: empty bbox"); return VWB200_EARG; }
  const bool sgm = h->p.algorithm != VWB200_CORRELATION_BM;
  if (sgm && h->p.cost_type != VWB200_CENSUS_TRANSFORM && h->p.cost_type != VWB200_TERNARY_CENSUS_TRANSFORM) {
    // NoImplErr of SGM.cc:1888-1892, re-thrown as ArgumentErr by calc_disparity_sgm (:221-226)
    set_error("Failed to compute the correlation. Detailed error message: With SGM/MGM, only the census transform cost mode gives good results.");
    return VWB200_EARG;
  }
  if (!sgm && h->p.cost_type > VWB200_CROSS_CORRELATION) { set_error("cost type %d is only valid for SGM", h->p.cost_type); return VWB200_EARG; }
  VWB_TRY(ensure_device());
  int prev_dev = -1;
  cudaGetDevice(&prev_dev);
  struct DevRestore { int d; ~DevRestore() { if (d >= 0) cudaSetDevice(d); } } restore{prev_dev != h->device ? prev_dev : -1};
  VWB_CUDA(cudaSetDevice(h->device));
  StreamGuard sg; VWB_TRY(sg.init(stream, ((h->owned || h->streamed) ? dest_on_device : 1)));
  cudaStream_t st = sg.st;
  {
    Arena ar(st);
    const int bw = x1 - x0, bh = y1 - y0;
    Box proc{x0, y0, x1, y1};
    if (with_collar && h->p.collar_size > 0) proc = bexpand(proc, h->p.collar_size, h->p.collar_size);   // CorrelationView.h:128-131
    const int pw = proc.x1 - proc.x0, ph = proc.y1 - proc.y0;
    vwb200_corr::DiffTile df;
    float* host_diff_window = nullptr;
    if (h->diff) {                                                                                        // CorrelationView.cc:276-283
      const int ulx = h->p.region_ul_x, uly = h->p.region_ul_y;
      if (!(proc.x0 >= ulx && proc.y0 >= uly && proc.x1 <= ulx + h->diff_cols && proc.y1 <= uly + h->diff_rows)) {
        set_error("The L-R to R-L difference image domain does not contain the current tile.");
        return VWB200_EARG;
      }
      if (h->diff_on_device) { df.d = h->diff; df.pitch = h->diff_pitch; df.ox = proc.x0 - ulx; df.oy = proc.y0 - uly; }
      else {                        // stage the tile's window (pixels the tile does not write keep their content)
        host_diff_window = h->diff + ((ptrdiff_t)(proc.y0 - uly) * h->diff_pitch + (proc.x0 - ulx)) * 2;
        VWB_TRY(ar.alloc(&df.d, (size_t)pw * ph * 2));
        df.pitch = pw; df.ox = 0; df.oy = 0;
        VWB_CUDA(cudaMemcpy2DAsync(df.d, (size_t)pw * 8, host_diff_window, (size_t)h->diff_pitch * 8, (size_t)pw * 8, ph, cudaMemcpyHostToDevice, st));
      }
    }
    vwb200_dispi* disp = nullptr; float* sub = nullptr; int all_invalid = 0;
    VWB_TRY(h->prerasterize(proc, &disp, &sub, &all_invalid, df, ar, st));
    float* dout = dest; ptrdiff_t dop = dest_pitch;
    if (!dest_on_device) { VWB_TRY(ar.alloc(&dout, (size_t)bw * bh * 3)); dop = bw; }
    if (all_invalid) {
      VWB_CUDA(cudaMemset2DAsync(dout, (size_t)dop * 12, 0, (size_t)bw * 12, bh, st));
    } else if (sgm) {
      VWB_TRY(sgm_finalize_launch(sub, disp, pw, h->p.search_x0, h->p.search_y0, dout, dop, x0 - proc.x0, y0 - proc.y0, bw, bh, st));
    } else {
      VWB_TRY(finalize_launch(disp, pw, ph, h->p.search_x0, h->p.search_y0, dout, dop, x0 - proc.x0, y0 - proc.y0, bw, bh, st));
    }
    if (!dest_on_device)
      VWB_CUDA(cudaMemcpy2DAsync(dest, (size_t)dest_pitch * 12, dout, (size_t)bw * 12, (size_t)bw * 12, bh, cudaMemcpyDeviceToHost, st));
    if (host_diff_window && !all_invalid)
      VWB_CUDA(cudaMemcpy2DAsync(host_diff_window, (size_t)h->diff_pitch * 8, df.d, (size_t)pw * 8, (size_t)pw * 8, ph, cudaMemcpyDeviceToHost, st));
    VWB_CUDA(cudaStreamSynchronize(st));
  }
  return VWB200_OK;
}
int vwb200_corr_rasterize(vwb200_corr* h, int x0, int y0, int x1, int y1, float* dest, ptrdiff_t dest_pitch, int dest_on_device, void* stream) {
  return corr_rasterize_impl(h, x0, y0, x1, y1, dest, dest_pitch, dest_on_device, stream, true);
}
int vwb200_corr_prerasterize(vwb200_corr* h, int x0, int y0, int x1, int y1, float* dest, ptrdiff_t dest_pitch, int dest_on_device, void* stream) {
  return corr_rasterize_impl(h, x0, y0, x1, y1, dest, dest_pitch, dest_on_device, stream, false);
}
int vwb200_corr_set_lr_disp_diff(vwb200_corr* h, float* diff, int cols, int rows, ptrdiff_t pitch, int on_device) {
  if (!h || (diff && (cols <= 0 || rows <= 0 || pitch < cols))) { set_error("corr_set_lr_disp_diff: bad arguments"); return VWB200_EARG; }
  h->diff = diff; h->diff_cols = cols; h->diff_rows = rows; h->diff_pitch = pitch; h->diff_on_device = on_device;
  return VWB200_OK;
}

void vwb200_corr_destroy(vwb200_corr* h) { delete h; }

}  // extern "C"
