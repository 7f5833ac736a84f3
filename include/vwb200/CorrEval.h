// CorrEval.h -- C++ shim: vw::stereo::CorrEval's lazy-view interface (Stereo/CorrEval.h:56-129) over the C ABI entry
// vwb200_corr_eval.
//
//   * derives ImageViewBase<Self>, pixel_type = result_type = PixelMask<float>, cols/rows/planes of the left image
//   * the reference constructor (:66-91) with its argument checks: the left image and the disparity of the same size, a
//     positive odd kernel and one of the metrics "ncc", "stddev", "parabola_curvature", "cramer_rao" (ArgumentErr)
//   * operator() throws NoImplErr; prerasterize(bbox) returns an owning bbox-sized buffer wrapped as
//     CropView(buf, -bbox.min, cols, rows) (CorrEval.cc:315-316), rasterize(dest, bbox) = vw::rasterize(prerasterize(bbox), ...)
//   * the factory b200_corr_eval (:117-128)
// The inputs are rasterised once at construction and sent with every tile call; the evaluation runs on the device and is
// bit-identical to the sequential reference order (DESIGN.md section K7).
#pragma once
#include "PyramidCorrelationView.h"

namespace vw { namespace stereo {

class B200CorrEval : public ImageViewBase<B200CorrEval> {
public:
  typedef PixelMask<float> pixel_type;
  typedef PixelMask<float> result_type;
  typedef ProceduralPixelAccessor<B200CorrEval> pixel_accessor;

  B200CorrEval(ImageViewRef<PixelMask<float>> left, ImageViewRef<PixelMask<float>> right,
               ImageViewRef<PixelMask<Vector2f>> disp, Vector2i const& kernel_size, std::string const& metric,
               int sample_rate, bool round_to_int, int prefilter_mode = 0, float prefilter_kernel_width = 0.0)
    : m_left(left), m_right(right), m_disp(disp), m_kernel_size(kernel_size), m_metric(metric), m_sample_rate(sample_rate),
      m_round_to_int(round_to_int), m_prefilter_mode(prefilter_mode), m_prefilter_kernel_width(prefilter_kernel_width) {
    static_assert(sizeof(PixelMask<float>) == 8, "PixelMask<float> must be {value, valid} floats");
    static_assert(sizeof(PixelMask<Vector2f>) == 12, "PixelMask<Vector2f> must be {dx, dy, valid} floats");
    if (m_left.cols() != m_disp.cols() || m_left.rows() != m_disp.rows())
      vw_throw(ArgumentErr() << "CorrEval: Left image and disparity must have the same dimensions.\n");
    if (!(m_kernel_size[0] > 0 && m_kernel_size[0] % 2 == 1 && m_kernel_size[1] > 0 && m_kernel_size[1] % 2 == 1))
      vw_throw(ArgumentErr() << "CorrEval: The kernel dimensions must be positive and odd.\n");
    if (m_metric == "ncc") m_metric_id = VWB200_CORR_EVAL_NCC;
    else if (m_metric == "stddev") m_metric_id = VWB200_CORR_EVAL_STDDEV;
    else if (m_metric == "parabola_curvature") m_metric_id = VWB200_CORR_EVAL_PARABOLA_CURVATURE;
    else if (m_metric == "cramer_rao") m_metric_id = VWB200_CORR_EVAL_CRAMER_RAO;
    else vw_throw(ArgumentErr() << "CorrEval: Invalid metric: " << m_metric << ".\n");
  }

  inline int32 cols() const { return m_left.cols(); }
  inline int32 rows() const { return m_left.rows(); }
  inline int32 planes() const { return 1; }
  inline pixel_accessor origin() const { return pixel_accessor(*this, 0, 0); }
  inline pixel_type operator()(double /*i*/, double /*j*/, int32 /*p*/ = 0) const {
    vw_throw(NoImplErr() << "CorrEval::operator() is not implemented.");
    return pixel_type();
  }

  typedef CropView<ImageView<pixel_type>> prerasterize_type;
  inline prerasterize_type prerasterize(BBox2i const& bbox) const {
    ImageView<pixel_type> buf(bbox.width(), bbox.height());
    b200_detail::check(vwb200_corr_eval(
        reinterpret_cast<const float*>(m_left.data()), m_left.cols(), m_left.rows(), m_left.cols(),
        reinterpret_cast<const float*>(m_right.data()), m_right.cols(), m_right.rows(), m_right.cols(),
        reinterpret_cast<const float*>(m_disp.data()), m_disp.cols(), m_kernel_size[0], m_kernel_size[1], m_metric_id,
        m_sample_rate, m_round_to_int ? 1 : 0, m_prefilter_kernel_width,
        bbox.min()[0], bbox.min()[1], bbox.max()[0], bbox.max()[1],
        reinterpret_cast<float*>(buf.data()), buf.cols(), /*on_device=*/0, nullptr));
    return prerasterize_type(buf, -bbox.min()[0], -bbox.min()[1], cols(), rows());
  }
  template <class DestT>
  inline void rasterize(DestT const& dest, BBox2i const& bbox) const { vw::rasterize(prerasterize(bbox), dest, bbox); }

private:
  ImageView<PixelMask<float>> m_left, m_right;
  ImageView<PixelMask<Vector2f>> m_disp;
  Vector2i m_kernel_size;
  std::string m_metric;
  int m_metric_id = VWB200_CORR_EVAL_NCC;
  int m_sample_rate;
  bool m_round_to_int;
  int m_prefilter_mode;            // accepted and unused, as in the reference
  float m_prefilter_kernel_width;  // sets the crop padding ceil(width) + 5 (CorrEval.h:77)
};

/// vw::stereo::corr_eval's twin (Stereo/CorrEval.h:117-128)
inline B200CorrEval b200_corr_eval(ImageViewRef<PixelMask<float>> left, ImageViewRef<PixelMask<float>> right,
                                   ImageViewRef<PixelMask<Vector2f>> disp, Vector2i const& kernel_size, std::string const& metric,
                                   int sample_rate, bool round_to_int, int prefilter_mode = 0, float prefilter_kernel_width = 0.0) {
  return B200CorrEval(left, right, disp, kernel_size, metric, sample_rate, round_to_int, prefilter_mode, prefilter_kernel_width);
}

}}  // namespace vw::stereo
