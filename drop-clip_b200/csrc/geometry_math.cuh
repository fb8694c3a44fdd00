// Per-point arithmetic shared by the geometry kernels (geometry.cu, sortpool.cu, aggregate.cu). Every operation is
// rounded on its own (no contraction), in the order the reference's numpy / Open3D code evaluates it.
#pragma once
#include "common.cuh"

namespace dc {

// Back-projection of pixel (x, y) at depth z. flip_y bit 1: Open3D create_from_rgbd_image rounding, (u - cx) * z / fx;
// otherwise utils/projections.py:75-81, ((u - cx) / fx) * z. flip_y bit 0 / flip_z negate y / z. pose (row-major 3x4
// of a 4x4, fp64) may be null: camera -> world as np.dot(pose, [p; 1]), a k-ascending FMA chain.
__device__ __forceinline__ void backproject_pixel(int x, int y, double z, double fx, double fy, double cx, double cy, int flip_y,
                                                  int flip_z, const double* pose, double out[3]) {
  double px, py;
  if (flip_y & 2) {
    px = __ddiv_rn(__dmul_rn(__dsub_rn((double)x, cx), z), fx);
    py = __ddiv_rn(__dmul_rn(__dsub_rn((double)y, cy), z), fy);
  } else {
    px = __dmul_rn(__ddiv_rn(__dsub_rn((double)x, cx), fx), z);
    py = __dmul_rn(__ddiv_rn(__dsub_rn((double)y, cy), fy), z);
  }
  double pz = z;
  if (flip_y & 1) py = -py;
  if (flip_z) pz = -pz;
  if (pose) {
    double w[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      double acc = __dmul_rn(pose[4 * r], px);
      acc = __fma_rn(pose[4 * r + 1], py, acc);
      acc = __fma_rn(pose[4 * r + 2], pz, acc);
      w[r] = __dadd_rn(pose[4 * r + 3], acc);
    }
    px = w[0]; py = w[1]; pz = w[2];
  }
  out[0] = px;
  out[1] = py;
  out[2] = pz;
}

// Ordered-integer image of a double, so that an unsigned atomicMin / atomicMax orders negative values too.
__device__ __forceinline__ unsigned long long double_to_ordered(double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double ordered_to_double(unsigned long long b) {
  b = (b & 0x8000000000000000ull) ? (b & 0x7fffffffffffffffull) : ~b;
  return __longlong_as_double((long long)b);
}

// Open3D voxel index along one axis: floor((p - voxel_min_bound) / voxel_size), bound = min - size / 2.
__device__ __forceinline__ double voxel_coord(double p, double bound, double voxel) {
  return floor(__ddiv_rn(__dsub_rn(p, bound), voxel));
}
// The 21-bit range of the packed voxel key; a point outside it (or NaN) takes key 0.
__device__ __forceinline__ bool voxel_coord_ok(double f) { return f >= 0 && f < 2097152.0; }

}  // namespace dc
