// test_subpixel_shim.cpp -- exercises include/vwb200/PyramidSubpixelView.h the way Vision Workbench code would
// (crop(view, bbox) rasterised into an ImageView, tiles from several threads) and checks every float bit against the CPU
// oracle.  Exit codes: 0 ok, 1 mismatch, 3 no CUDA device (expected on a machine without a GPU).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <thread>
#include <vector>
#include "vwb200/PyramidSubpixelView.h"
#include "../../oracle/vw_subpixel_oracle.h"

using namespace vw;
using namespace vw::stereo;

int main() {
  const int W = 160, H = 128;
  ImageView<PixelGray<float>> left(W, H), right(W, H);
  ImageView<PixelMask<Vector2f>> disp(W, H);
  for (int y = 0; y < H; ++y)
    for (int x = 0; x < W; ++x) {
      left(x, y) = 0.5f + 0.25f * std::sin(x / 3.1f) * std::cos(y / 4.3f);
      right(x, y) = 0.5f + 0.25f * std::sin((x - 1.4f) / 3.1f) * std::cos((y + 0.3f) / 4.3f);
      disp(x, y) = PixelMask<Vector2f>(Vector2f(1.0f, 0.0f));
      if ((x * 7 + y * 13) % 23 == 0) disp(x, y).invalidate();
    }
  const Vector2i kernel(7, 7);
  try {
    bool threw = false;
    try { B200PyramidSubpixelView(disp, left, right, PREFILTER_NONE, 0.f, kernel, 2, SUBPIXEL_PHASE).prerasterize(BBox2i(0, 0, 8, 8)); }
    catch (NoImplErr const&) { threw = true; }
    if (!threw) { std::printf("FAIL: SUBPIXEL_PHASE accepted\n"); return 1; }

    long bad = 0, moved = 0;
    const int tile = 64;
    B200PyramidSubpixelView views[3] = {b200_lk_subpixel(disp, left, right, PREFILTER_LOG, 1.4f, kernel),
                                        b200_affine_subpixel(disp, left, right, PREFILTER_LOG, 1.4f, kernel),
                                        b200_bayes_em_subpixel(disp, left, right, PREFILTER_LOG, 1.4f, kernel)};
    { ImageView<PixelMask<Vector2f>> probe = crop(views[2], BBox2i(0, 0, 16, 16)); }   // a missing device throws here
    for (int a = 0; a < 3; ++a) {
      ImageView<PixelMask<Vector2f>> out(W, H);
      std::vector<std::thread> th;
      for (int ty = 0; ty < H; ty += tile)
        for (int tx = 0; tx < W; tx += tile)
          th.emplace_back([&, tx, ty] {
            const BBox2i b(tx, ty, std::min(tile, W - tx), std::min(tile, H - ty));
            ImageView<PixelMask<Vector2f>> t = crop(views[a], b);
            for (int y = 0; y < b.height(); ++y)
              for (int x = 0; x < b.width(); ++x) out(tx + x, ty + y) = t(x, y);
          });
      for (auto& t : th) t.join();
      for (int ty = 0; ty < H; ty += tile)
        for (int tx = 0; tx < W; tx += tile) {
          const int bw = std::min(tile, W - tx), bh = std::min(tile, H - ty);
          std::vector<float> ref(size_t(bw) * bh * 3);
          if (vwso_pyramid_subpixel(reinterpret_cast<const float*>(disp.data()), W, H, reinterpret_cast<const float*>(left.data()), W,
                                    reinterpret_cast<const float*>(right.data()), W, H, W, 7, 7, 1, 1.4f, tx, ty, tx + bw, ty + bh,
                                    2, a, ref.data())) return 1;
          for (int y = 0; y < bh; ++y)
            for (int x = 0; x < bw; ++x) {
              const PixelMask<Vector2f>& g = out(tx + x, ty + y);
              const float* r = &ref[(size_t(y) * bw + x) * 3];
              const float gv[3] = {g.child()[0], g.child()[1], is_valid(g) ? 1.f : 0.f};
              if (std::memcmp(gv, r, sizeof(gv))) ++bad;
              if (is_valid(g) && g.child()[0] != 1.0f) ++moved;
            }
        }
    }
    std::printf("subpixel shim: %ld mismatches, %ld refined of %d\n", bad, moved, 3 * W * H);
    return bad || !moved ? 1 : 0;
  } catch (LogicErr const& e) {
    std::printf("NODEVICE-or-CUDA: %s\n", e.what());
    return 3;
  }
}
