// RGB-D back-projection of one keypoint pixel (camera_models.py:781-799, 835-860, 203-212; pose_est_tools.py:612-620),
// shared by rgbd_backproject_kernel (geometry.cu) and the front-end's rgbd_store_kernel (frontend.cu) so that the two
// give the same bits.
#pragma once
#include <math_constants.h>
#include <stdint.h>

#include "sosfront.h"

struct RgbdP {
  double v[SOS_RGBD_NPARAMS];
};

__device__ __forceinline__ double rgbd_depth_z(const RgbdP& c, double d, double u, double v) {
  if (c.v[SOS_RGBD_DEPTH_IS_Z] != 0.0) return d;
  const double f = c.v[SOS_RGBD_FOCAL_M];
  const double xi = (f / c.v[SOS_RGBD_FX]) * (u - c.v[SOS_RGBD_CX]);
  const double yi = (f / c.v[SOS_RGBD_FY]) * (v - c.v[SOS_RGBD_CY]);
  return f * d / sqrt(xi * xi + yi * yi + f * f);
}

// Pixel (u, v) of the frame's depth map [h, w] -> xyz and unit bearing (float64 arithmetic rounded to float32), and
// whether the keypoint passes the reference's gate: Z not NaN (a pixel outside the map or zero depth gives NaN,
// camera_models.py:846) and, for zmin / zmax > 0, zmin <= |Z| <= zmax (pose_est_tools.py:570-592 gates |Z|).
__device__ __forceinline__ bool rgbd_point(const RgbdP& c, const float* __restrict__ depth, int h, int w, int u, int v,
                                           double zmin, double zmax, float* __restrict__ xyz, float* __restrict__ bearing) {
  double Z = CUDART_NAN;
  if (u >= 0 && u < w && v >= 0 && v < h) {
    const double d = (double)depth[(size_t)v * w + u];
    const double zz = rgbd_depth_z(c, d, (double)u, (double)v);
    if (zz != 0.0) Z = zz;
  }
  const double X = ((double)u - c.v[SOS_RGBD_CX]) * Z / c.v[SOS_RGBD_FX];
  const double Y = ((double)v - c.v[SOS_RGBD_CY]) * Z / c.v[SOS_RGBD_FY];
  const double nrm = sqrt(X * X + Y * Y + Z * Z);
  xyz[0] = (float)X; xyz[1] = (float)Y; xyz[2] = (float)Z;
  bearing[0] = (float)(X / nrm); bearing[1] = (float)(Y / nrm); bearing[2] = (float)(Z / nrm);
  bool ok = !isnan(Z);
  const double az = fabs(Z);
  if (zmin > 0.0) ok = ok && az >= zmin;
  if (zmax > 0.0) ok = ok && az <= zmax;
  return ok;
}
