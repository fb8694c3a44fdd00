// Geometry helpers of utils/projections.py: RGB-D back-projection and (un-truncated) forward
// projection, fp64 like the reference's numpy code.
//
// Reference: depth_to_pointcloud utils/projections.py:67-86 (x = ((u - cx) / fx) * z with u an
// int64 pixel index, promoted to fp64; a fp32 depth map is promoted to fp64 by the multiply),
// _cvt_regrad_coord :89-92 / _cvt_blender_coord :95-97, transform_pointcloud_to_world_frame
// utils/transforms.py:43-49 (np.dot(pose, [p;1]) -> k-ascending FMA chain, pose promoted from
// fp32), pointcloud_to_pixel utils/projections.py:59-64.
#include "geometry_math.cuh"

namespace {

__global__ void __launch_bounds__(256) backproject_kernel(const float* __restrict__ depths, int n_views, int height, int width,
                                                          const double* __restrict__ k4, int flip_y, int flip_z,
                                                          const double* __restrict__ poses, double* __restrict__ out) {
  const int64_t hw = (int64_t)height * width;
  const int64_t total = hw * n_views;
  const double fx = k4[0], fy = k4[1], cx = k4[2], cy = k4[3];
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int v = (int)(t / hw);
    const int64_t pix = t - (int64_t)v * hw;
    const int y = (int)(pix / width), x = (int)(pix - (int64_t)y * width);
    double w[3];
    dc::backproject_pixel(x, y, (double)depths[t], fx, fy, cx, cy, flip_y, flip_z, poses ? poses + (int64_t)v * 16 : nullptr, w);
    out[3 * t] = w[0];
    out[3 * t + 1] = w[1];
    out[3 * t + 2] = w[2];
  }
}

__global__ void __launch_bounds__(256) points_to_pixels_kernel(const double* __restrict__ pts, int64_t n,
                                                               const double* __restrict__ k4, double* __restrict__ pix) {
  const double fx = k4[0], fy = k4[1], cx = k4[2], cy = k4[3];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
    // fx * x / z + cx  evaluates left to right: (fx * x) / z, then + cx
    pix[2 * i] = __dadd_rn(__ddiv_rn(__dmul_rn(fx, x), z), cx);
    pix[2 * i + 1] = __dadd_rn(__ddiv_rn(__dmul_rn(fy, y), z), cy);
  }
}

struct Mat12 { double m[12]; };

__global__ void __launch_bounds__(256) transform_points_kernel(const double* __restrict__ pts, int64_t n, Mat12 M,
                                                               double* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      double acc = __dmul_rn(M.m[4 * r], x);
      acc = __fma_rn(M.m[4 * r + 1], y, acc);
      acc = __fma_rn(M.m[4 * r + 2], z, acc);
      out[3 * i + r] = __dadd_rn(M.m[4 * r + 3], acc);
    }
  }
}

unsigned grid_for(int64_t n) {
  int64_t b = dc::ceil_div<int64_t>(n, 256);
  const int64_t cap = (int64_t)dc::sm_count() * 16;
  return (unsigned)(b < cap ? (b < 1 ? 1 : b) : cap);
}

}  // namespace

extern "C" {

int dc_backproject(const float* depths, int n_views, int height, int width, const double* fxfycxcy, int flip_y, int flip_z,
                   const double* poses, double* out, dc_stream_t stream) {
  DC_CHECK_ARG(depths && fxfycxcy && out, "dc_backproject: null pointer argument");
  if (n_views <= 0 || height <= 0 || width <= 0) return DC_OK;
  backproject_kernel<<<grid_for((int64_t)n_views * height * width), 256, 0, dc::as_stream(stream)>>>(
      depths, n_views, height, width, fxfycxcy, flip_y, flip_z, poses, out);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

int dc_transform_points(const double* points, int64_t n, const double* matrix_host, double* out, dc_stream_t stream) {
  DC_CHECK_ARG(points && matrix_host && out, "dc_transform_points: null pointer argument");
  if (n <= 0) return DC_OK;
  Mat12 M;
  for (int i = 0; i < 12; ++i) M.m[i] = matrix_host[i];
  transform_points_kernel<<<grid_for(n), 256, 0, dc::as_stream(stream)>>>(points, n, M, out);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

int dc_points_to_pixels(const double* cam_points, int64_t n, const double* fxfycxcy, double* pixels, dc_stream_t stream) {
  DC_CHECK_ARG(cam_points && fxfycxcy && pixels, "dc_points_to_pixels: null pointer argument");
  if (n <= 0) return DC_OK;
  points_to_pixels_kernel<<<grid_for(n), 256, 0, dc::as_stream(stream)>>>(cam_points, n, fxfycxcy, pixels);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

}  // extern "C"
