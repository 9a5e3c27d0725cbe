// ORACLE -- test infrastructure only.  depth_image_proc's convert<T> (depth_conversions.h; PointCloudXyzrgbNodelet's
// XYZ arithmetic is the same) restated literally, with fromPCLPointCloud2<PointXYZ>'s padding float 1.0f: the cloud
// that kinect2_bridge publishes on /kinect2/qhd/points, built from one depth image and its pinhole model.  Neither
// image_pipeline nor iai_kinect2 is available to build here; this restatement and the independent numpy one in
// depth_util.py pin the semantics.  Built like the pipeline oracle (g++ -O2 -ffp-contract=off -fno-fast-math), so every
// float op is rounded in turn and none is contracted.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>

#include "pcop.h"

namespace {

template <class T>
struct DepthTraits;
template <>
struct DepthTraits<uint16_t> {
  static bool valid(uint16_t depth) { return depth != 0; }
  static float toMeters(uint16_t depth) { return depth * 0.001f; }  // millimetres
};
template <>
struct DepthTraits<float> {
  static bool valid(float depth) { return std::isfinite(depth); }
  static float toMeters(float depth) { return depth; }
};

template <class T>
void convert(const pcop_depth_image& im, float* out) {
  // PinholeCameraModel::cx() .. fy() are doubles; the nodelet keeps the centre as float
  const float center_x = (float)im.cx;
  const float center_y = (float)im.cy;
  const double unit_scaling = DepthTraits<T>::toMeters(T(1));
  const float constant_x = unit_scaling / im.fx;
  const float constant_y = unit_scaling / im.fy;
  const float bad_point = std::numeric_limits<float>::quiet_NaN();
  for (int v = 0; v < im.height; ++v) {
    const unsigned char* row = im.data + (size_t)v * (size_t)im.step;
    for (int u = 0; u < im.width; ++u) {
      T depth;
      std::memcpy(&depth, row + (size_t)u * sizeof(T), sizeof(T));  // (little-endian host, as the image)
      float* p = out + 4 * ((size_t)v * (size_t)im.width + (size_t)u);
      if (!DepthTraits<T>::valid(depth)) {
        p[0] = p[1] = p[2] = bad_point;
      } else {
        p[0] = (u - center_x) * depth * constant_x;
        p[1] = (v - center_y) * depth * constant_y;
        p[2] = DepthTraits<T>::toMeters(depth);
      }
      p[3] = 1.0f;
    }
  }
}

}  // namespace

extern "C" int pcop_oracle_depth_image_to_xyz(const pcop_depth_image* im, float* out_xyzw) {
  if (!im || im->width < 0 || im->height < 0) return PCOP_ERR_BAD_PARAM;
  if ((long long)im->width * im->height == 0) return PCOP_OK;
  if (!im->data || !out_xyzw) return PCOP_ERR_BAD_PARAM;
  if (im->encoding == PCOP_DEPTH_16UC1 && im->step >= 2 * im->width)
    convert<uint16_t>(*im, out_xyzw);
  else if (im->encoding == PCOP_DEPTH_32FC1 && im->step >= 4 * im->width)
    convert<float>(*im, out_xyzw);
  else
    return PCOP_ERR_BAD_PARAM;
  return PCOP_OK;
}
