// test_corr_eval_shim.cpp -- exercises include/vwb200/CorrEval.h the way Vision Workbench code would (crop(view, bbox)
// rasterised into an ImageView, tiles from several threads) and checks every float bit against the CPU oracle.
// Exit codes: 0 ok, 1 mismatch, 3 no CUDA device (expected on a machine without a GPU).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <thread>
#include <vector>
#include "vwb200/CorrEval.h"
#include "../../oracle/vw_corr_eval_oracle.h"

using namespace vw;
using namespace vw::stereo;

int main() {
  const int W = 150, H = 110, RW = 170, RH = 100;
  ImageView<PixelMask<float>> left(W, H), right(RW, RH);
  ImageView<PixelMask<Vector2f>> disp(W, H);
  for (int y = 0; y < H; ++y)
    for (int x = 0; x < W; ++x) {
      left(x, y) = PixelMask<float>(std::sin(x / 3.1f) * std::cos(y / 4.3f) + 0.1f * std::sin(0.7f * x * y));
      if ((x * 5 + y * 11) % 29 == 0) left(x, y).invalidate();
      disp(x, y) = PixelMask<Vector2f>(Vector2f(1.3f + 0.01f * x, -0.4f + 0.02f * y));
      if ((x * 7 + y * 13) % 23 == 0) disp(x, y).invalidate();
    }
  for (int y = 0; y < RH; ++y)
    for (int x = 0; x < RW; ++x) {
      right(x, y) = PixelMask<float>(std::sin((x - 1.4f) / 3.1f) * std::cos((y + 0.3f) / 4.3f));
      if ((x * 3 + y * 7) % 31 == 0) right(x, y).invalidate();
    }
  const Vector2i kernel(7, 5);
  const char* metrics[4] = {"ncc", "stddev", "parabola_curvature", "cramer_rao"};
  try {
    bool threw = false;
    try { B200CorrEval(left, right, disp, kernel, "phase", 1, false); } catch (ArgumentErr const&) { threw = true; }
    if (!threw) { std::printf("FAIL: an unknown metric was accepted\n"); return 1; }
    threw = false;
    try { B200CorrEval(left, right, disp, Vector2i(4, 5), "ncc", 1, false); } catch (ArgumentErr const&) { threw = true; }
    if (!threw) { std::printf("FAIL: an even kernel was accepted\n"); return 1; }
    threw = false;
    try { B200CorrEval(left, right, disp, kernel, "ncc", 1, false)(0, 0); } catch (NoImplErr const&) { threw = true; }
    if (!threw) { std::printf("FAIL: operator() did not throw NoImplErr\n"); return 1; }

    { ImageView<PixelMask<float>> probe = crop(b200_corr_eval(left, right, disp, kernel, "ncc", 1, false), BBox2i(0, 0, 8, 8)); }  // a missing device throws here
    long bad = 0, valid = 0;
    const int tile = 48;
    for (int m = 0; m < 4; ++m)
      for (int round = 0; round < 2; ++round) {
        const B200CorrEval view = b200_corr_eval(left, right, disp, kernel, metrics[m], 2, round != 0, 1, 1.4f);
        ImageView<PixelMask<float>> out(W, H);
        std::vector<std::thread> th;
        for (int ty = 0; ty < H; ty += tile)
          for (int tx = 0; tx < W; tx += tile)
            th.emplace_back([&, tx, ty] {
              const BBox2i b(tx, ty, std::min(tile, W - tx), std::min(tile, H - ty));
              ImageView<PixelMask<float>> t = crop(view, b);
              for (int y = 0; y < b.height(); ++y)
                for (int x = 0; x < b.width(); ++x) out(tx + x, ty + y) = t(x, y);
            });
        for (auto& t : th) t.join();
        for (int ty = 0; ty < H; ty += tile)
          for (int tx = 0; tx < W; tx += tile) {
            const int bw = std::min(tile, W - tx), bh = std::min(tile, H - ty);
            std::vector<float> ref(size_t(bw) * bh * 2);
            if (vwce_corr_eval(reinterpret_cast<const float*>(left.data()), W, H, W, reinterpret_cast<const float*>(right.data()), RW, RH, RW,
                               reinterpret_cast<const float*>(disp.data()), W, kernel[0], kernel[1], m, 2, round, 1.4f,
                               tx, ty, tx + bw, ty + bh, ref.data(), bw)) return 1;
            for (int y = 0; y < bh; ++y)
              for (int x = 0; x < bw; ++x) {
                const PixelMask<float>& g = out(tx + x, ty + y);
                const float gv[2] = {g.child(), is_valid(g) ? 1.f : 0.f};
                if (std::memcmp(gv, &ref[(size_t(y) * bw + x) * 2], sizeof(gv))) ++bad;
                if (is_valid(g)) ++valid;
              }
          }
      }
    std::printf("corr_eval shim: %ld mismatches, %ld valid of %d\n", bad, valid, 8 * W * H);
    return bad || !valid ? 1 : 0;
  } catch (LogicErr const& e) {
    std::printf("NODEVICE-or-CUDA: %s\n", e.what());
    return 3;
  }
}
