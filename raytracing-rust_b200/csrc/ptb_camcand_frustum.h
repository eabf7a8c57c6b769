// The f64 camera of the per-pixel candidate lists' frustum test and its error margins (ptb_camcand.cuh states the
// argument). Plain C++ with no CUDA dependency, so that the CPU statement of the lists (scripts/camcand_ref.cpp) uses the
// very margins and camera bound the device uses, and its directed frustum check guards them.
#pragma once
#include <math.h>

#ifdef __CUDACC__
#define PTB_CC_HD __host__ __device__ __forceinline__
#else
#define PTB_CC_HD inline
#endif

namespace ptb {

struct CamCandCamera {  // f64 camera of the frustum test (cam_cand_camera)
  double o[3], ll[3], h[3], vv[3];
  double f[3];   // unit normal of the image plane, away from the apex
  double sin_a;  // bound on the angle between a computed camera direction and the exact cone (ptb_camcand.cuh)
};
constexpr double kCcEps = 1.0 / 8388608.0;
constexpr double kCcUvMargin = 1.0 / 1048576.0;
constexpr double kCcBoxGrow = 1.0 / 65536.0;
constexpr double kCcKeySlack = 1.0 / 65536.0;

PTB_CC_HD void cc_cross(const double a[3], const double b[3], double r[3]) {
  r[0] = a[1] * b[2] - a[2] * b[1];
  r[1] = a[2] * b[0] - a[0] * b[2];
  r[2] = a[0] * b[1] - a[1] * b[0];
}
PTB_CC_HD double cc_dot(const double a[3], const double b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// host: the f64 camera of the frustum test from the f32 camera vectors (origin, lower_left, horizontal, vertical)
inline CamCandCamera cam_cand_camera(const float o[3], const float ll[3], const float h[3], const float vv[3]) {
  CamCandCamera c;
  const float* src[4] = {o, ll, h, vv};
  double* dst[4] = {c.o, c.ll, c.h, c.vv};
  for (int i = 0; i < 4; ++i)
    for (int k = 0; k < 3; ++k) dst[i][k] = src[i][k];
  double s2 = 0.0;
  for (int k = 0; k < 3; ++k) {
    const double s = fabs(c.ll[k]) + 2.0 * fabs(c.h[k]) + 2.0 * fabs(c.vv[k]) + fabs(c.o[k]);
    s2 += s * s;
  }
  cc_cross(c.h, c.vv, c.f);
  const double fm = sqrt(cc_dot(c.f, c.f));
  for (int k = 0; k < 3; ++k) c.f[k] /= fm;
  const double llo[3] = {c.ll[0] - c.o[0], c.ll[1] - c.o[1], c.ll[2] - c.o[2]};
  double dmin = cc_dot(llo, c.f);
  if (dmin < 0.0) { for (int k = 0; k < 3; ++k) c.f[k] = -c.f[k]; dmin = -dmin; }
  c.sin_a = 8.0 * kCcEps * sqrt(s2) / dmin + 2.0 * kCcEps;
  return c;
}

}  // namespace ptb
