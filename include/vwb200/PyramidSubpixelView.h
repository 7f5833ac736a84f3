// PyramidSubpixelView.h -- C++ shim: vw::stereo::PyramidSubpixelView's lazy-view interface (Stereo/SubpixelView.h:42-150)
// over the C ABI entry vwb200_pyramid_subpixel.
//
//   * derives ImageViewBase<Self>, pixel_type = PixelMask<Vector2f>, cols/rows/planes of the disparity
//   * the reference constructor (:57-85), phase_subpixel_accuracy defaulting to 20; the disparity must match the left image
//   * operator() throws NoImplErr; prerasterize(bbox) returns an owning bbox-sized buffer wrapped as
//     CropView(buf, -bbox.min, cols, rows) (SubpixelView.cc:220-223), rasterize(dest, bbox) = vw::rasterize(prerasterize(bbox), ...)
//   * factories b200_lk_subpixel / b200_affine_subpixel / b200_bayes_em_subpixel with max_pyramid_levels = 2 (:117-145)
// SUBPIXEL_PHASE or an unknown algorithm throws NoImplErr at rasterisation, like the reference (SubpixelView.cc:158-159).
// The inputs are rasterised once at construction and sent with every tile call; the refinement runs on the device and is
// bit-identical to the sequential reference order (DESIGN.md section K6).
#pragma once
#include "PyramidCorrelationView.h"

namespace vw { namespace stereo {

class B200PyramidSubpixelView : public ImageViewBase<B200PyramidSubpixelView> {
public:
  typedef PixelMask<Vector2f> pixel_type;
  typedef pixel_type result_type;

  template <class DispT, class LeftT, class RightT>
  B200PyramidSubpixelView(ImageViewBase<DispT> const& disparity_map, ImageViewBase<LeftT> const& left_image,
                          ImageViewBase<RightT> const& right_image, PrefilterModeType prefilter_mode, float prefilter_width,
                          Vector2i const& kernel_size, int max_pyramid_levels, PyramidSubpixelView_Algorithm algorithm,
                          int phase_subpixel_accuracy = 20)
    : m_disparity(disparity_map.impl()), m_left(left_image.impl()), m_right(right_image.impl()), m_kernel(kernel_size),
      m_prefilter_mode(prefilter_mode), m_prefilter_width(prefilter_width), m_max_pyramid_levels(max_pyramid_levels),
      m_algorithm(algorithm), m_phase_subpixel_accuracy(phase_subpixel_accuracy) {
    static_assert(sizeof(pixel_type) == 12, "PixelMask<Vector2f> must be {dx, dy, valid} floats");
    static_assert(sizeof(PixelGray<float>) == sizeof(float), "PixelGray<float> must be a bare float");
    if (m_disparity.cols() != m_left.cols() || m_disparity.rows() != m_left.rows())
      vw_throw(ArgumentErr() << "SubpixelView: Disparity image must match left image.");
  }

  inline int32 cols() const { return m_disparity.cols(); }
  inline int32 rows() const { return m_disparity.rows(); }
  inline int32 planes() const { return 1; }
  inline pixel_type operator()(int32 /*i*/, int32 /*j*/, int32 /*p*/ = 0) const {
    vw_throw(NoImplErr() << "PyramidSubpixelView::operator() is not implemented.");
    return pixel_type();
  }

  typedef CropView<ImageView<pixel_type>> prerasterize_type;
  inline prerasterize_type prerasterize(BBox2i const& bbox) const {
    ImageView<pixel_type> buf(bbox.width(), bbox.height());
    b200_detail::check(vwb200_pyramid_subpixel(
        reinterpret_cast<const float*>(m_disparity.data()), m_disparity.cols(), m_disparity.rows(),
        reinterpret_cast<const float*>(m_left.data()), m_left.cols(),
        reinterpret_cast<const float*>(m_right.data()), m_right.cols(), m_right.rows(), m_right.cols(),
        m_kernel[0], m_kernel[1], int(m_prefilter_mode), m_prefilter_width,
        bbox.min()[0], bbox.min()[1], bbox.max()[0], bbox.max()[1],
        reinterpret_cast<float*>(buf.data()), buf.cols(), /*on_device=*/0, nullptr, m_max_pyramid_levels, int(m_algorithm)));
    return prerasterize_type(buf, -bbox.min()[0], -bbox.min()[1], cols(), rows());
  }
  template <class DestT>
  inline void rasterize(DestT const& dest, BBox2i const& bbox) const { vw::rasterize(prerasterize(bbox), dest, bbox); }

private:
  ImageView<pixel_type> m_disparity;
  ImageView<PixelGray<float>> m_left, m_right;
  Vector2i m_kernel;
  PrefilterModeType m_prefilter_mode;
  float m_prefilter_width;
  int m_max_pyramid_levels;
  PyramidSubpixelView_Algorithm m_algorithm;
  int m_phase_subpixel_accuracy;   // kept for the reference's constructor; SUBPIXEL_PHASE is not implemented
};

/// vw::stereo::lk_subpixel's twin (Stereo/SubpixelView.h:117-125)
template <class DispT, class LeftT, class RightT>
inline B200PyramidSubpixelView
b200_lk_subpixel(ImageViewBase<DispT> const& disparity_map, ImageViewBase<LeftT> const& left_image,
                 ImageViewBase<RightT> const& right_image, PrefilterModeType prefilter_mode, float prefilter_width,
                 Vector2i const& kernel_size, int max_pyramid_levels = 2) {
  return B200PyramidSubpixelView(disparity_map, left_image, right_image, prefilter_mode, prefilter_width, kernel_size,
                                 max_pyramid_levels, SUBPIXEL_LUCAS_KANADE);
}
/// vw::stereo::affine_subpixel's twin (Stereo/SubpixelView.h:127-135)
template <class DispT, class LeftT, class RightT>
inline B200PyramidSubpixelView
b200_affine_subpixel(ImageViewBase<DispT> const& disparity_map, ImageViewBase<LeftT> const& left_image,
                     ImageViewBase<RightT> const& right_image, PrefilterModeType prefilter_mode, float prefilter_width,
                     Vector2i const& kernel_size, int max_pyramid_levels = 2) {
  return B200PyramidSubpixelView(disparity_map, left_image, right_image, prefilter_mode, prefilter_width, kernel_size,
                                 max_pyramid_levels, SUBPIXEL_FAST_AFFINE);
}
/// vw::stereo::bayes_em_subpixel's twin (Stereo/SubpixelView.h:137-145)
template <class DispT, class LeftT, class RightT>
inline B200PyramidSubpixelView
b200_bayes_em_subpixel(ImageViewBase<DispT> const& disparity_map, ImageViewBase<LeftT> const& left_image,
                       ImageViewBase<RightT> const& right_image, PrefilterModeType prefilter_mode, float prefilter_width,
                       Vector2i const& kernel_size, int max_pyramid_levels = 2) {
  return B200PyramidSubpixelView(disparity_map, left_image, right_image, prefilter_mode, prefilter_width, kernel_size,
                                 max_pyramid_levels, SUBPIXEL_BAYES_EM);
}

}}  // namespace vw::stereo
