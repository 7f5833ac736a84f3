// vw_standin.h -- minimal stand-ins for the Vision Workbench types the shim touches, with the same
// names, member layout and semantics, so that include/vwb200/PyramidCorrelationView.h compiles and is
// testable WITHOUT the reference tree (which needs Boost/GDAL).  When the shim is dropped into
// src/vw/Stereo, define VWB200_USE_REAL_VW and include the real headers instead; nothing else changes.
//
// Mirrors (reference file:line under src/vw/):
//   Vector2i/Vector2f           Math/Vector.h           (fixed-size POD vectors, operator[])
//   BBox2i                      Math/BBox.h, BBox.tcc:37-285   (half-open, min()/max()/width()/height()/expand)
//   PixelGray<T>, PixelMask<T>  Image/PixelTypes.h, Image/PixelMask.h:48-160  (child + valid channel)
//   ImageViewBase<ImplT>        Image/ImageViewBase.h:57-122   (CRTP base)
//   ImageView<PixelT>           Image/ImageView.h:67-297       (shared buffer, cols/rows, operator(), set_size)
//   ImageViewRef<PixelT>        Image/ImageViewRef.h           (any view behind one pixel type; held rasterised here)
//   CropView<ImageT>            Image/Manipulation.h:82-146
//   vw::rasterize               Image/ImageViewBase.h:283-316
//   Exception hierarchy         Core/Exception.h:201-253
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>

namespace vw {

typedef int32_t int32;
typedef uint8_t uint8;

// ---- exceptions (Core/Exception.h) ---------------------------------------------------------------
struct Exception : public std::exception {
  std::string m_desc;
  Exception() {}
  explicit Exception(std::string const& s) : m_desc(s) {}
  const char* what() const noexcept override { return m_desc.c_str(); }
  template <class T> Exception& operator<<(T const& t) { std::ostringstream o; o << t; m_desc += o.str(); return *this; }
};
#define VWB200_STANDIN_EXC(name) \
  struct name : public Exception { name() {} explicit name(std::string const& s) : Exception(s) {} \
    template <class T> name& operator<<(T const& t) { Exception::operator<<(t); return *this; } }
VWB200_STANDIN_EXC(ArgumentErr);
VWB200_STANDIN_EXC(MathErr);
VWB200_STANDIN_EXC(LogicErr);
VWB200_STANDIN_EXC(NoImplErr);
VWB200_STANDIN_EXC(IOErr);
template <class E> [[noreturn]] inline void vw_throw(E const& e) { throw e; }

// ---- math ------------------------------------------------------------------------------------------
template <class T> struct Vector2 {
  T v[2];
  Vector2() { v[0] = v[1] = T(); }
  Vector2(T a, T b) { v[0] = a; v[1] = b; }
  T& operator[](size_t i) { return v[i]; }
  T const& operator[](size_t i) const { return v[i]; }
  T& x() { return v[0]; } T& y() { return v[1]; }
  T const& x() const { return v[0]; } T const& y() const { return v[1]; }
};
typedef Vector2<int32> Vector2i;
typedef Vector2<float> Vector2f;

class BBox2i {
  Vector2i m_min, m_max;
public:
  BBox2i() : m_min(2147483646, 2147483646), m_max(-2147483646, -2147483646) {}          // BBox.tcc:37-44
  BBox2i(int32 x, int32 y, int32 w, int32 h) : m_min(x, y), m_max(x + w, y + h) {}      // BBox.tcc:55-59
  BBox2i(Vector2i const& mn, Vector2i const& mx) : m_min(mn), m_max(mx) {}
  Vector2i& min() { return m_min; } Vector2i& max() { return m_max; }
  Vector2i const& min() const { return m_min; } Vector2i const& max() const { return m_max; }
  bool empty() const { return m_min[0] >= m_max[0] || m_min[1] >= m_max[1]; }
  int32 width() const { return empty() ? 0 : m_max[0] - m_min[0]; }
  int32 height() const { return empty() ? 0 : m_max[1] - m_min[1]; }
  Vector2i size() const { return Vector2i(m_max[0] - m_min[0], m_max[1] - m_min[1]); }
  double area() const { return empty() ? 0.0 : double(m_max[0] - m_min[0]) * double(m_max[1] - m_min[1]); }
  void expand(int32 o) { if (empty()) return; m_min[0] -= o; m_min[1] -= o; m_max[0] += o; m_max[1] += o; }
};

// ---- pixels -----------------------------------------------------------------------------------------
template <class T> struct PixelGray { T v; PixelGray() : v() {} PixelGray(T a) : v(a) {} operator T() const { return v; } };
template <class ChildT> struct PixelMaskChannel;
template <> struct PixelMaskChannel<Vector2f> { typedef float type; static float valid_max() { return 1.0f; } };
template <> struct PixelMaskChannel<Vector2i> { typedef int32 type; static int32 valid_max() { return 2147483647; } };
template <> struct PixelMaskChannel<float> { typedef float type; static float valid_max() { return 1.0f; } };
template <class ChildT> struct PixelMask {                      // Image/PixelMask.h:48-160: {child, valid}
  typedef typename PixelMaskChannel<ChildT>::type channel_type;
private:
  ChildT m_child; channel_type m_valid;
public:
  PixelMask() : m_child(), m_valid(0) {}
  PixelMask(ChildT const& c) : m_child(c), m_valid(PixelMaskChannel<ChildT>::valid_max()) {}
  channel_type valid() const { return m_valid; }
  void invalidate() { m_valid = 0; }
  void validate() { m_valid = PixelMaskChannel<ChildT>::valid_max(); }
  ChildT& child() { return m_child; } ChildT const& child() const { return m_child; }
  channel_type& operator[](size_t i) { return i == 2 ? m_valid : m_child[i]; }
  channel_type const& operator[](size_t i) const { return i == 2 ? m_valid : m_child[i]; }
};
template <class C> inline bool is_valid(PixelMask<C> const& p) { return p.valid() != 0; }
static_assert(sizeof(PixelMask<Vector2f>) == 12, "PixelMask<Vector2f> must be 3 floats (Image/PixelMask.h:52-54)");

// ---- views -------------------------------------------------------------------------------------------
template <class ImplT> struct ImageViewBase {                     // Image/ImageViewBase.h:57-64
  ImplT& impl() { return static_cast<ImplT&>(*this); }
  ImplT const& impl() const { return static_cast<ImplT const&>(*this); }
};

template <class PixelT> class ImageView : public ImageViewBase<ImageView<PixelT>> {
  std::shared_ptr<PixelT> m_data; int32 m_cols, m_rows, m_planes; PixelT* m_origin; ptrdiff_t m_rstride;
public:
  typedef PixelT pixel_type; typedef PixelT& result_type;
  ImageView() : m_cols(0), m_rows(0), m_planes(0), m_origin(nullptr), m_rstride(0) {}
  ImageView(int32 c, int32 r, int32 p = 1) : m_cols(0), m_rows(0), m_planes(0), m_origin(nullptr), m_rstride(0) { set_size(c, r, p); }
  template <class ViewT> ImageView(ImageViewBase<ViewT> const& view) : m_cols(0), m_rows(0), m_planes(0), m_origin(nullptr), m_rstride(0) {
    set_size(view.impl().cols(), view.impl().rows(), view.impl().planes());                 // Image/ImageView.h:114-118
    view.impl().rasterize(*this, BBox2i(0, 0, view.impl().cols(), view.impl().rows()));
  }
  void set_size(int32 c, int32 r, int32 p = 1) {                                            // Image/ImageView.h:175-215
    if (c == m_cols && r == m_rows && p == m_planes) return;
    if (c < 0 || r < 0 || p < 0) vw_throw(ArgumentErr() << "Cannot allocate image with negative pixel count");
    size_t n = size_t(c) * size_t(r) * size_t(p);
    m_data.reset(n ? new PixelT[n]() : nullptr, std::default_delete<PixelT[]>());
    m_cols = c; m_rows = r; m_planes = p; m_origin = m_data.get(); m_rstride = c;
  }
  int32 cols() const { return m_cols; } int32 rows() const { return m_rows; } int32 planes() const { return m_planes; }
  PixelT* data() const { return m_origin; }
  ptrdiff_t rstride() const { return m_rstride; }
  PixelT& operator()(int32 c, int32 r, int32 = 0) const { return m_origin[ptrdiff_t(r) * m_rstride + c]; }
  template <class DestT> void rasterize(DestT const& dest, BBox2i const& bbox) const {
    for (int32 r = 0; r < bbox.height(); ++r)
      for (int32 c = 0; c < bbox.width(); ++c) dest(c, r) = (*this)(bbox.min()[0] + c, bbox.min()[1] + r);
  }
  typedef ImageView prerasterize_type;
  prerasterize_type prerasterize(BBox2i const&) const { return *this; }
};

// Image/ImageViewRef.h: a view of any type behind one pixel type.  The stand-in holds the view rasterised into an
// ImageView, which is what a consumer that rasterises its inputs (the shims) observes.
template <class PixelT> class ImageViewRef : public ImageViewBase<ImageViewRef<PixelT>> {
  ImageView<PixelT> m_view;
public:
  typedef PixelT pixel_type; typedef PixelT result_type;
  template <class ViewT> ImageViewRef(ImageViewBase<ViewT> const& view) : m_view(view) {}
  int32 cols() const { return m_view.cols(); } int32 rows() const { return m_view.rows(); } int32 planes() const { return m_view.planes(); }
  result_type operator()(int32 c, int32 r, int32 p = 0) const { return m_view(c, r, p); }
  template <class DestT> void rasterize(DestT const& dest, BBox2i const& bbox) const { m_view.rasterize(dest, bbox); }
};

template <class ImageT> class CropView : public ImageViewBase<CropView<ImageT>> {             // Image/Manipulation.h:82-146
  ImageT m_child; int32 m_ci, m_cj, m_di, m_dj;
public:
  typedef typename ImageT::pixel_type pixel_type; typedef pixel_type& result_type;
  CropView(ImageT const& image, int32 upper_left_i, int32 upper_left_j, int32 width, int32 height)
    : m_child(image), m_ci(upper_left_i), m_cj(upper_left_j), m_di(width), m_dj(height) {}
  int32 cols() const { return m_di; } int32 rows() const { return m_dj; } int32 planes() const { return m_child.planes(); }
  result_type operator()(int32 i, int32 j, int32 p = 0) const { return m_child(m_ci + i, m_cj + j, p); }
  ImageT const& child() const { return m_child; }
  // Image/Manipulation.h:138-146: rasterisation is delegated to the child over the shifted box
  template <class DestT> void rasterize(DestT const& dest, BBox2i const& bbox) const {
    m_child.rasterize(dest, BBox2i(bbox.min()[0] + m_ci, bbox.min()[1] + m_cj, bbox.width(), bbox.height()));
  }
};
template <class ImageT> inline CropView<ImageT> crop(ImageViewBase<ImageT> const& v, BBox2i const& b) {
  return CropView<ImageT>(v.impl(), b.min()[0], b.min()[1], b.width(), b.height());
}

// vw::rasterize(src, dest, bbox): Image/ImageViewBase.h:283-316
template <class SrcT, class DestT> inline void rasterize(SrcT const& src, DestT const& dest, BBox2i const& bbox) {
  if (dest.cols() != bbox.width() || dest.rows() != bbox.height())
    vw_throw(ArgumentErr() << "rasterize: Source and destination must have same dimensions.");
  src.rasterize(dest, bbox);
}

// Image/PixelAccessors.h:119-156: the accessor of views whose pixels are computed by operator()
template <class ViewT> class ProceduralPixelAccessor {
  ViewT const& m_view; int32 m_c, m_r, m_p;
public:
  typedef typename ViewT::pixel_type pixel_type; typedef typename ViewT::result_type result_type;
  ProceduralPixelAccessor(ViewT const& view) : m_view(view), m_c(0), m_r(0), m_p(0) {}
  ProceduralPixelAccessor(ViewT const& view, int32 c, int32 r, int32 p = 0) : m_view(view), m_c(c), m_r(r), m_p(p) {}
  ProceduralPixelAccessor& next_col() { ++m_c; return *this; } ProceduralPixelAccessor& prev_col() { --m_c; return *this; }
  ProceduralPixelAccessor& next_row() { ++m_r; return *this; } ProceduralPixelAccessor& prev_row() { --m_r; return *this; }
  ProceduralPixelAccessor& advance(int32 dc, int32 dr, ptrdiff_t dp = 0) { m_c += dc; m_r += dr; m_p += int32(dp); return *this; }
  result_type operator*() const { return m_view(m_c, m_r, m_p); }
};

namespace stereo {
struct SemiGlobalMatcher {                                                                    // Stereo/SGM.h:93-99
  enum SgmSubpixelMode { SUBPIXEL_NONE = 0, SUBPIXEL_PARABOLA = 1, SUBPIXEL_LINEAR = 2, SUBPIXEL_POLY4 = 3, SUBPIXEL_COSINE = 4, SUBPIXEL_LC_BLEND = 5 };
};
enum CostFunctionType { ABSOLUTE_DIFFERENCE, SQUARED_DIFFERENCE, CROSS_CORRELATION, CENSUS_TRANSFORM, TERNARY_CENSUS_TRANSFORM };  // Stereo/CostFunctions.h:143-149
enum PrefilterModeType { PREFILTER_NONE = 0, PREFILTER_LOG = 1, PREFILTER_MEANSUB = 2 };                                           // Stereo/PrefilterEnum.h:24-28
enum CorrelationAlgorithm { VW_CORRELATION_BM = 0, VW_CORRELATION_SGM = 1, VW_CORRELATION_MGM = 2, VW_CORRELATION_FINAL_MGM = 3 };
enum PyramidSubpixelView_Algorithm {                                                                 // Stereo/SubpixelView.h:35-40
  SUBPIXEL_LUCAS_KANADE = 0, SUBPIXEL_FAST_AFFINE = 1, SUBPIXEL_BAYES_EM = 2, SUBPIXEL_PHASE = 3 };
}  // namespace stereo
}  // namespace vw
