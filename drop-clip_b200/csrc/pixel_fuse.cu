// Pixel-level fusion (the `use_obj_prior=0` ablation path).
//
// Reference: MultiviewFeatureFusion.aggregate_features utils/feature_fusion.py:138-250 and the final
// division of fuse_points :266-268. Per view the reference bicubically upsamples the (ph,pw,C)
// patch map to (H,W,C) (943.7 MB at 480x640x768 fp32), L2-normalises every pixel, multiplies the
// whole map with the query matrix, builds a per-pixel similarity metric, and finally gathers the
// visible projected pixels. Only those gathered pixels matter, so this kernel evaluates the 16
// bicubic taps directly at each visible (point, view), in registers, and never materialises the
// map. Rows are accumulated over the views in view order (same order as `sum_features[mask] += feat3d`)
// and written once. The query similarity of an interpolated feature comes from a per-view table of
// (patch cell . query) dots interpolated with the same weights (patch_query_dots_kernel).
//
// Bicubic weights follow ATen's upsample_bicubic2d (align_corners=False, A=-0.75, source index
// scale*(dst+0.5)-0.5 un-clamped, taps clamped to the border).
#include <algorithm>

#include "common.cuh"
#include "umma.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxPerLane = 32;  // channels per lane: dim <= 1024

struct PixParams {
  const double* points;
  const int64_t* point_off;
  const int64_t* view_off;
  const double* inv_poses;
  const double* intrinsics;
  const int64_t* mask_off;
  const uint8_t* visible;
  const void* seg;
  int seg_dtype;
  const float* patch;
  int ph, pw, dim;
  const float* queries;
  const int64_t* query_off;
  int sim_kernel, norm_feat;
  int height, width;
  const int64_t* perm;
  float* out_sum;
  float* out_weight;
  double* dots;  // [total_views][ph * pw][q_stride] fp64: patch row . query, see patch_query_dots_kernel
  int q_stride;
  int normalize;  // divide the sums by sum_v weight (similarity) or by the number of views that see the point
};

__device__ __forceinline__ float cubic1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }

__device__ __forceinline__ void cubic_taps(int dst, float scale, int in_size, int (&idx)[4], float (&w)[4]) {
  const float A = -0.75f;
  const float src = scale * ((float)dst + 0.5f) - 0.5f;
  const float fl = floorf(src);
  const float t = src - fl;
  const int i0 = (int)fl;
  w[0] = cubic2(t + 1.f, A);
  w[1] = cubic1(t, A);
  w[2] = cubic1(1.f - t, A);
  w[3] = cubic2(2.f - t, A);
#pragma unroll
  for (int k = 0; k < 4; ++k) idx[k] = min(max(i0 - 1 + k, 0), in_size - 1);
}

// The same taps with fp64 weights (ATen's formulas evaluated in double precision, as F.interpolate does for fp64
// input): used for the similarity chain only, see "similarity weights in fp64" below.
__device__ __forceinline__ double cubic1d(double x, double A) { return ((A + 2.0) * x - (A + 3.0)) * x * x + 1.0; }
__device__ __forceinline__ double cubic2d(double x, double A) { return ((A * x - 5.0 * A) * x + 8.0 * A) * x - 4.0 * A; }
__device__ __forceinline__ int cubic_weights64(int dst, int in_size, int out_size, double (&w)[4]) {
  const double A = -0.75;
  const double src = ((double)in_size / (double)out_size) * ((double)dst + 0.5) - 0.5;
  const double fl = floor(src);
  const double t = src - fl;
  w[0] = cubic2d(t + 1.0, A);
  w[1] = cubic1d(t, A);
  w[2] = cubic1d(1.0 - t, A);
  w[3] = cubic2d(2.0 - t, A);
  return (int)fl;  // first tap is at index i0 - 1 (clamped by the caller)
}
// Taps of one axis with EXACT weights: the fp64 coefficients (for the similarity chain) and their fp32 roundings
// (for the fp32 feature fold). ATen's own fp32 evaluation of `scale * (dst + 0.5) - 0.5` carries an absolute error
// of ~1e-6 in the source coordinate (and depends on how its compiler contracted the expression into FMAs), which
// moves interpolated features by ~2e-7 - already 1e-3 of the smallest magnitudes the parity metric resolves
// (profiles/r02_reference_fp32_noise.md). Evaluating the coordinate in fp64 puts this kernel next to the exact
// value of the reference's formula rather than next to one particular build's rounding of it.
__device__ __forceinline__ void cubic_taps_exact(int dst, int in_size, int out_size, int (&idx)[4], float (&w)[4], double (&w64)[4]) {
  const int i0 = cubic_weights64(dst, in_size, out_size, w64);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    idx[k] = min(max(i0 - 1 + k, 0), in_size - 1);
    w[k] = (float)w64[k];
  }
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ int seg_at(const void* seg, int dtype, int64_t idx) {
  if (dtype == DC_U8) return (int)__ldg(reinterpret_cast<const uint8_t*>(seg) + idx);
  if (dtype == DC_I32) return __ldg(reinterpret_cast<const int32_t*>(seg) + idx);
  const long long v = __ldg(reinterpret_cast<const long long*>(seg) + idx);
  return (v < 0 || v > 0x7fffffff) ? -1 : (int)v;
}

// The similarity of an interpolated feature with a query is linear in the taps:
//   f . q = sum_t w_t (T_t . q),   f = sum_t w_t T_t  (16 bicubic taps T_t of the patch map)
// so the (patch cell, query) dot products are computed ONCE per view (ph * pw * Q dots, 16 M FMA at 24x32x21x768)
// instead of Q x C FMA and 64 KB of query reads per visible (point, view). The normalisation of `norm_feat`
// divides the similarity by |f| afterwards ((f / |f|) . q = (f . q) / |f|). Warp per patch cell, lanes over channels.
__global__ void __launch_bounds__(kThreads) patch_query_dots_kernel(PixParams p) {
  const int scene = blockIdx.y;
  const int64_t v0 = p.view_off[scene];
  const int n_views = (int)(p.view_off[scene + 1] - v0);
  const int n_q = (int)(p.query_off[scene + 1] - p.query_off[scene]);
  const float* q = p.queries + p.query_off[scene] * p.dim;
  const int lane = threadIdx.x & 31;
  const int64_t n_cells = (int64_t)p.ph * p.pw, n_rows = n_cells * n_views;
  for (int64_t r = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); r < n_rows; r += (int64_t)gridDim.x * kWarps) {
    const float* row = p.patch + (v0 * n_cells + r) * p.dim;
    double* out = p.dots + (v0 * n_cells + r) * p.q_stride;
    float t[kMaxPerLane];
#pragma unroll
    for (int k = 0; k < kMaxPerLane; ++k) t[k] = (k * 32 + lane < p.dim) ? __ldg(row + k * 32 + lane) : 0.f;
    for (int o = 0; o < n_q; o += 4) {  // four queries per round: their loads overlap (the kernel is latency-bound)
      double d[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (o + j < n_q) {
          const float* qo = q + (int64_t)(o + j) * p.dim;
#pragma unroll
          for (int k = 0; k < kMaxPerLane; ++k)
            if (k * 32 + lane < p.dim) d[j] = fma((double)t[k], (double)__ldg(qo + k * 32 + lane), d[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) d[j] = warp_sum_d(d[j]);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (lane == 0 && o + j < n_q) out[o + j] = d[j];
    }
  }
}

// The same table for the CLIP widths (dim = 32 * kPer), four patch cells per warp: a query chunk is loaded once per four
// cells and the four fp64 chains (and their shuffle reductions) overlap. Same per-lane summation order as above, so the
// table is bit-identical. (The one-cell version is latency-bound: 0.44 ms for 73 x 768 cells x 21 queries.)
template <int kPer>
__global__ void __launch_bounds__(kThreads) patch_query_dots4_kernel(PixParams p) {
  const int scene = blockIdx.y;
  const int64_t v0 = p.view_off[scene];
  const int n_views = (int)(p.view_off[scene + 1] - v0);
  const int n_q = (int)(p.query_off[scene + 1] - p.query_off[scene]);
  const float* q = p.queries + p.query_off[scene] * p.dim;
  const int lane = threadIdx.x & 31;
  const int64_t n_cells = (int64_t)p.ph * p.pw, n_rows = n_cells * n_views;
  for (int64_t r0 = ((int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5)) * 4; r0 < n_rows; r0 += (int64_t)gridDim.x * kWarps * 4) {
    float t[4][kPer];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int64_t r = r0 + c < n_rows ? r0 + c : n_rows - 1;  // a ragged last group repeats the last row (not stored)
      const float* row = p.patch + (v0 * n_cells + r) * p.dim;
#pragma unroll
      for (int k = 0; k < kPer; ++k) t[c][k] = __ldg(row + k * 32 + lane);
    }
    for (int o = 0; o < n_q; ++o) {
      const float* qo = q + (int64_t)o * p.dim;
      double d[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int k = 0; k < kPer; ++k) {
        const double qv = (double)__ldg(qo + k * 32 + lane);
#pragma unroll
        for (int c = 0; c < 4; ++c) d[c] = fma((double)t[c][k], qv, d[c]);
      }
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1) {
#pragma unroll
        for (int c = 0; c < 4; ++c) d[c] += __shfl_xor_sync(0xffffffffu, d[c], sh);
      }
      if (lane < 4 && r0 + lane < n_rows) {
        const double mine = lane == 0 ? d[0] : lane == 1 ? d[1] : lane == 2 ? d[2] : d[3];
        p.dots[(v0 * n_cells + r0 + lane) * p.q_stride + o] = mine;
      }
    }
  }
}

// Similarity weights in fp64. The weight of a visible (point, view) is clip(pos - max|mean(neg), 1e-6) of the
// similarities of its (normalised) interpolated feature with the scene's queries (calculate_sim,
// feature_fusion.py:65-73,182-196). On surfaces whose best two queries tie, pos - neg is a difference of two numbers
// ~1 that lands near the 1e-6 clip, and the fused feature of a point whose views all do that is a mean with weights
// of relative accuracy eps_fp32 / 1e-6: the reference's own fp32 result is then several percent away from the exact
// value of its formulas (profiles/r02_reference_fp32_noise.md: 0.7 % of the rows of a 480x640, V=8 scene are off by
// more than 1e-3). An fp32 evaluation here would add its own, different, noise on top, so the whole chain is exact
// instead: fp64 (patch . query) table, fp64 bicubic weights, pos - red(neg) in fp64, ONE division by |f| at the end
// ((pos - neg) / |f| = pos / |f| - neg / |f|, and max commutes with the positive scale), one rounding to fp32.
// What remains between this and the reference is the reference's rounding noise alone.
// interp_dot: lane l interpolates query o's dots (issued before the tap loads); finish_weight reduces over queries.
// Scenes with more than 32 queries take further rounds of interp_dot inside finish_weight.
__device__ __forceinline__ double interp_dot(const PixParams& p, const double* __restrict__ dots_view, const int (&iy)[4],
                                             const int (&ix)[4], const double (&wy)[4], const double (&wx)[4], int o, int n_q) {
  double mine = 0.0;
  if (o < n_q) {
#pragma unroll
    for (int ty = 0; ty < 4; ++ty) {
      const double* row = dots_view + ((int64_t)iy[ty] * p.pw) * p.q_stride + o;
      double r = __ldg(row + ix[0] * p.q_stride) * wx[0];
      r = fma(__ldg(row + ix[1] * p.q_stride), wx[1], r);
      r = fma(__ldg(row + ix[2] * p.q_stride), wx[2], r);
      r = fma(__ldg(row + ix[3] * p.q_stride), wx[3], r);
      mine = fma(r, wy[ty], mine);
    }
  }
  return mine;
}

template <typename More>
__device__ __forceinline__ float finish_weight(const PixParams& p, double first, float nrm, int id, int n_q, int lane, More&& more) {
  double pos = 0.0, red = (p.sim_kernel == DC_SIM_MAX) ? -INFINITY : 0.0;
  bool nan_seen = false;
  for (int o0 = 0; o0 < n_q; o0 += 32) {
    const int o = o0 + lane;
    const double mine = o0 == 0 ? first : more(o);
    if (id >= o0 && id < o0 + 32) pos = __shfl_sync(0xffffffffu, mine, id - o0);
    const bool is_neg = o < n_q && o != id;
    nan_seen |= __any_sync(0xffffffffu, is_neg && (mine != mine));
    if (p.sim_kernel == DC_SIM_MAX) red = fmax(red, warp_max_d(is_neg ? mine : -INFINITY));
    else red += warp_sum_d(is_neg ? mine : 0.0);
  }
  if (p.sim_kernel == DC_SIM_MEAN) red = red / (double)(n_q - 1);
  if (nan_seen) red = __longlong_as_double(0x7ff8000000000000ll);
  double w = pos - red;
  if (p.norm_feat) w = w / (double)nrm;  // nrm = 0 (an all-zero feature): 0 / 0 = NaN like the reference's f / |f|
  float weight = (float)w;
  if (weight == weight) weight = fmaxf(weight, 1e-6f);
  return weight;
}

// seg_at in two halves: the load (requested early) and the range check / narrowing (done where the id is needed), so
// that the scoreboard wait for this cold, scattered load sits behind the tap arithmetic.
__device__ __forceinline__ long long seg_raw(const void* seg, int dtype, int64_t idx) {
  long long v;
  if (dtype == DC_U8) v = (long long)__ldg(reinterpret_cast<const uint8_t*>(seg) + idx);
  else if (dtype == DC_I32) v = (long long)__ldg(reinterpret_cast<const int32_t*>(seg) + idx);
  else v = __ldg(reinterpret_cast<const long long*>(seg) + idx);
  return v;
}
__device__ __forceinline__ int seg_id(long long v) { return (v < 0 || v > 0x7fffffff) ? -1 : (int)v; }

__global__ void __launch_bounds__(kThreads) pixel_fuse_kernel(PixParams p) {
  extern __shared__ double s_cam[];  // [n_views][12] + [9]
  const int scene = blockIdx.y;
  const int64_t p0 = p.point_off[scene];
  const int64_t n_pts = p.point_off[scene + 1] - p0;
  const int64_t v0 = p.view_off[scene];
  const int n_views = (int)(p.view_off[scene + 1] - v0);
  for (int i = threadIdx.x; i < n_views * 12; i += kThreads) {
    const int v = i / 12, e = i - v * 12;
    s_cam[i] = __ldg(p.inv_poses + (v0 + v) * 16 + e);
  }
  double* s_K = s_cam + n_views * 12;
  if (threadIdx.x < 9) s_K[threadIdx.x] = __ldg(p.intrinsics + (int64_t)scene * 9 + threadIdx.x);
  __syncthreads();

  const int lane = threadIdx.x & 31;
  const int per_lane = p.dim / 32;  // host guarantees dim % 32 == 0, dim <= 1024
  const int n_q = p.sim_kernel != DC_SIM_NONE ? (int)(p.query_off[scene + 1] - p.query_off[scene]) : 0;
  const int64_t hw = (int64_t)p.height * p.width;
  const uint8_t* vis_scene = p.visible + p.mask_off[scene];
  float* w_scene = p.out_weight ? p.out_weight + p.mask_off[scene] : nullptr;

  for (int64_t s_pos = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); s_pos < n_pts; s_pos += (int64_t)gridDim.x * kWarps) {
    const int64_t i = p.perm ? __ldg(p.perm + p0 + s_pos) : s_pos;  // spatially sorted processing order, original indexing
    const double x = __ldg(p.points + 3 * (p0 + i)), y = __ldg(p.points + 3 * (p0 + i) + 1),
                 z = __ldg(p.points + 3 * (p0 + i) + 2);
    float acc[kMaxPerLane];
#pragma unroll
    for (int k = 0; k < kMaxPerLane; ++k) acc[k] = 0.f;
    for (int v = 0; v < n_views; ++v) {
      const bool vis = vis_scene[(int64_t)v * n_pts + i] != 0;  // warp-uniform
      if (!vis) {
        if (w_scene && lane == 0) w_scene[(int64_t)v * n_pts + i] = 0.f;
        continue;
      }
      // same projection arithmetic as visibility.cu (the point is visible, so it is inside)
      const double* m = s_cam + v * 12;
      double cx = __dadd_rn(m[3], __fma_rn(m[2], z, __fma_rn(m[1], y, __dmul_rn(m[0], x))));
      double cy = __dadd_rn(m[7], __fma_rn(m[6], z, __fma_rn(m[5], y, __dmul_rn(m[4], x))));
      double cz = __dadd_rn(m[11], __fma_rn(m[10], z, __fma_rn(m[9], y, __dmul_rn(m[8], x))));
      cy = -cy;
      cz = -cz;
      const double qx = __fma_rn(s_K[2], cz, __fma_rn(s_K[1], cy, __dmul_rn(s_K[0], cx)));
      const double qy = __fma_rn(s_K[5], cz, __fma_rn(s_K[4], cy, __dmul_rn(s_K[3], cx)));
      const double qz = __fma_rn(s_K[8], cz, __fma_rn(s_K[7], cy, __dmul_rn(s_K[6], cx)));
      int pu = 0, pv = 0;
      if (qz != 0.0) {
        pu = (int)__ddiv_rn(qx, qz);
        pv = (int)__ddiv_rn(qy, qz);
      }
      int iy[4], ix[4];
      float wy[4], wx[4];
      double wy64[4], wx64[4];
      cubic_taps_exact(pv, p.ph, p.height, iy, wy, wy64);
      cubic_taps_exact(pu, p.pw, p.width, ix, wx, wx64);
      const float* pm = p.patch + (v0 + v) * (int64_t)p.ph * p.pw * p.dim;
      const double* dots_view = p.dots + (v0 + v) * (int64_t)p.ph * p.pw * p.q_stride;
      auto sim_dot = [&](int o) { return interp_dot(p, dots_view, iy, ix, wy64, wx64, o, n_q); };
      const double first_dot = p.sim_kernel != DC_SIM_NONE ? sim_dot(lane) : 0.0;
      float f[kMaxPerLane];
#pragma unroll
      for (int k = 0; k < kMaxPerLane; ++k) f[k] = 0.f;
      // ATen order: interpolate along x inside each of the 4 rows, then along y
#pragma unroll
      for (int ty = 0; ty < 4; ++ty) {
        const float* row = pm + (int64_t)iy[ty] * p.pw * p.dim;
        const float* t0 = row + (int64_t)ix[0] * p.dim;
        const float* t1 = row + (int64_t)ix[1] * p.dim;
        const float* t2 = row + (int64_t)ix[2] * p.dim;
        const float* t3 = row + (int64_t)ix[3] * p.dim;
#pragma unroll
        for (int k = 0; k < kMaxPerLane; ++k) {
          if (k < per_lane) {
            const int c = k * 32 + lane;
            const float r = __ldg(t0 + c) * wx[0] + __ldg(t1 + c) * wx[1] + __ldg(t2 + c) * wx[2] + __ldg(t3 + c) * wx[3];
            f[k] = fmaf(r, wy[ty], f[k]);
          }
        }
      }
      float nrm = 1.f;
      if (p.norm_feat) {
        float ss = 0.f;
#pragma unroll
        for (int k = 0; k < kMaxPerLane; ++k)
          if (k < per_lane) ss = fmaf(f[k], f[k], ss);
        nrm = sqrtf(dc::warp_sum(ss));
#pragma unroll
        for (int k = 0; k < kMaxPerLane; ++k)
          if (k < per_lane) f[k] = f[k] / nrm;
      }
      float weight = 1.f;
      if (p.sim_kernel != DC_SIM_NONE) {
        const int id = seg_at(p.seg, p.seg_dtype, (v0 + v) * hw + (int64_t)pv * p.width + pu);
        weight = 0.f;  // pixels whose id has no query keep metric 0 (quirk q13)
        if (id >= 0 && id < n_q)
          weight = finish_weight(p, first_dot, nrm, id, n_q, lane, sim_dot);
        if (w_scene && lane == 0) w_scene[(int64_t)v * n_pts + i] = weight;
#pragma unroll
        for (int k = 0; k < kMaxPerLane; ++k)
          if (k < per_lane) acc[k] += f[k] * weight;  // feat2d[ys,xs] * metric, then +=  (two roundings)
      } else {
#pragma unroll
        for (int k = 0; k < kMaxPerLane; ++k)
          if (k < per_lane) acc[k] += f[k];
      }
    }
    float* dst = p.out_sum + (p0 + i) * p.dim;
#pragma unroll
    for (int k = 0; k < kMaxPerLane; ++k)
      if (k < per_lane) dst[k * 32 + lane] = acc[k];
  }
}

// The fast path (dim = 128 * kChunks: CLIP widths 512 / 768 / 1024). A lane owns 4 consecutive channels of every
// 128-channel chunk (128-bit tap loads). A CTA owns kTilePts consecutive points of the (Morton-sorted) processing
// order and walks the views IN STEP (one barrier per view that sees any of them). Neighbouring points project into
// the same patch cells of a view, so while the CTA is on view v its warps keep hitting the same ~50 KB of taps in
// L1. A point-major version (one warp per point, all its views) let every warp drift through the views at its own
// pace: its ncu capture showed 43 % L1 hits, 10 GB of L2 reads per 8-view scene and 6.6 long-scoreboard stall cycles
// per issue; this kernel: 79 % L1 hits, 3.4 GB, 4.0 (profiles/r01_pixel_fuse.md).
// The per-point accumulators live in shared memory (kTilePts x dim fp32) so that the visible points of a view can
// be dealt to the warps round-robin whatever their position in the tile; a point is touched by one warp per view
// and the barrier orders the views, so every row is accumulated in view order exactly like `sum_features[mask] +=`.
constexpr int kTilePts = 32;

template <int kChunks>
__global__ void __launch_bounds__(kThreads, 2) pixel_fuse_tile_kernel(PixParams p) {
  extern __shared__ double s_cam[];  // [n_views][12] + [9], then the accumulators
  constexpr int kDim = 128 * kChunks;
  const int scene = blockIdx.y;
  const int64_t p0 = p.point_off[scene];
  const int64_t n_pts = p.point_off[scene + 1] - p0;
  const int64_t v0 = p.view_off[scene];
  const int n_views = (int)(p.view_off[scene + 1] - v0);
  const int64_t tile0 = (int64_t)blockIdx.x * kTilePts;
  if (tile0 >= n_pts) return;
  const int n_tile = (int)min((int64_t)kTilePts, n_pts - tile0);
  for (int i = threadIdx.x; i < n_views * 12; i += kThreads) {
    const int v = i / 12, e = i - v * 12;
    s_cam[i] = __ldg(p.inv_poses + (v0 + v) * 16 + e);
  }
  double* s_K = s_cam + n_views * 12;
  if (threadIdx.x < 9) s_K[threadIdx.x] = __ldg(p.intrinsics + (int64_t)scene * 9 + threadIdx.x);
  float4* s_acc = reinterpret_cast<float4*>(s_cam + (((size_t)n_views * 12 + 9 + 1) & ~(size_t)1));  // 16-byte aligned
  float* s_den = reinterpret_cast<float*>(s_acc + kTilePts * (kDim / 4));  // [kTilePts] denominators of fuse_points :266-268
  // per slot and view: the 8 exact (fp64) bicubic weights (y taps, x taps) and the first tap indices, written by the
  // lane that owns the slot, read by the warp that processes the pair
  double* s_tw = reinterpret_cast<double*>(s_den + kTilePts);  // [kTilePts][8]
  int* s_ti = reinterpret_cast<int*>(s_tw + kTilePts * 8);     // [kTilePts][2]
  for (int i = threadIdx.x; i < kTilePts * (kDim / 4); i += kThreads) s_acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (threadIdx.x < kTilePts) s_den[threadIdx.x] = 0.f;
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_q = p.sim_kernel != DC_SIM_NONE ? (int)(p.query_off[scene + 1] - p.query_off[scene]) : 0;
  const int64_t hw = (int64_t)p.height * p.width;
  const uint8_t* vis_scene = p.visible + p.mask_off[scene];
  float* w_scene = p.out_weight ? p.out_weight + p.mask_off[scene] : nullptr;
  // lane l <-> tile slot l: original index of the point at sorted position tile0 + l
  const int64_t my_i = lane < n_tile ? (p.perm ? __ldg(p.perm + p0 + tile0 + lane) : tile0 + lane) : 0;
  const double px = __ldg(p.points + 3 * (p0 + my_i)), py = __ldg(p.points + 3 * (p0 + my_i) + 1), pz = __ldg(p.points + 3 * (p0 + my_i) + 2);

  for (int v = 0; v < n_views; ++v) {
    const bool vis = lane < n_tile && vis_scene[(int64_t)v * n_pts + my_i] != 0;
    const unsigned m = __ballot_sync(0xffffffffu, vis);  // identical in every warp of the CTA
    if (m == 0) continue;
    const int n_vis = __popc(m);
    const float4* pm = reinterpret_cast<const float4*>(p.patch + (v0 + v) * (int64_t)p.ph * p.pw * kDim);
    const double* dots_view = p.dots + (v0 + v) * (int64_t)p.ph * p.pw * p.q_stride;
    // lane-parallel projection: every lane projects ITS slot's point once per view (the same fp64 arithmetic as
    // visibility.cu; the point is visible, so it is inside); the pair loop below fetches pixels by shuffle
    const double* cam = s_cam + v * 12;
    int my_pu = 0, my_pv = 0;
    {
      double cx = __dadd_rn(cam[3], __fma_rn(cam[2], pz, __fma_rn(cam[1], py, __dmul_rn(cam[0], px))));
      double cy = __dadd_rn(cam[7], __fma_rn(cam[6], pz, __fma_rn(cam[5], py, __dmul_rn(cam[4], px))));
      double cz = __dadd_rn(cam[11], __fma_rn(cam[10], pz, __fma_rn(cam[9], py, __dmul_rn(cam[8], px))));
      cy = -cy;
      cz = -cz;
      const double qx = __fma_rn(s_K[2], cz, __fma_rn(s_K[1], cy, __dmul_rn(s_K[0], cx)));
      const double qy = __fma_rn(s_K[5], cz, __fma_rn(s_K[4], cy, __dmul_rn(s_K[3], cx)));
      const double qz = __fma_rn(s_K[8], cz, __fma_rn(s_K[7], cy, __dmul_rn(s_K[6], cx)));
      if (vis && qz != 0.0) {
        my_pu = (int)__ddiv_rn(qx, qz);
        my_pv = (int)__ddiv_rn(qy, qz);
      }
      // every warp computes and writes the same values (m, the pixels and hence these are identical in all warps);
      // the __syncthreads() that ends the previous visible view orders them against that view's readers
      if (vis) {
        double wy64[4], wx64[4];
        s_ti[2 * lane] = cubic_weights64(my_pv, p.ph, p.height, wy64);
        s_ti[2 * lane + 1] = cubic_weights64(my_pu, p.pw, p.width, wx64);
#pragma unroll
        for (int t4 = 0; t4 < 4; ++t4) {
          s_tw[8 * lane + t4] = wy64[t4];
          s_tw[8 * lane + 4 + t4] = wx64[t4];
        }
      }
      __syncwarp();
    }
    for (int k = warp; k < n_vis; k += kWarps) {
      const int slot = __fns(m, 0, k + 1);
      const int64_t i = __shfl_sync(0xffffffffu, my_i, slot);
      const int pu = __shfl_sync(0xffffffffu, my_pu, slot), pv = __shfl_sync(0xffffffffu, my_pv, slot);
      int iy[4], ix[4];
      float wy[4], wx[4];
      {
        const int iy0 = s_ti[2 * slot], ix0 = s_ti[2 * slot + 1];
#pragma unroll
        for (int t4 = 0; t4 < 4; ++t4) {
          iy[t4] = min(max(iy0 - 1 + t4, 0), p.ph - 1);
          ix[t4] = min(max(ix0 - 1 + t4, 0), p.pw - 1);
          wy[t4] = (float)s_tw[8 * slot + t4];
          wx[t4] = (float)s_tw[8 * slot + 4 + t4];
        }
      }
      // the instance id and the first round of query dots are requested before the taps: both are cold loads whose
      // latency then hides behind the 96 tap loads instead of sitting in front of the accumulator update
      long long raw_id = p.sim_kernel != DC_SIM_NONE ? seg_raw(p.seg, p.seg_dtype, (v0 + v) * hw + (int64_t)pv * p.width + pu) : -1;
      // the fp64 weights are re-read from shared memory inside the lambda (broadcast loads; nothing stays live)
      auto sim_dot = [&](int o) {
        double wy64[4], wx64[4];
#pragma unroll
        for (int t4 = 0; t4 < 4; ++t4) {
          wy64[t4] = s_tw[8 * slot + t4];
          wx64[t4] = s_tw[8 * slot + 4 + t4];
        }
        return interp_dot(p, dots_view, iy, ix, wy64, wx64, o, n_q);
      };
      const double first_dot = p.sim_kernel != DC_SIM_NONE ? sim_dot(lane) : 0.0;
      // Chunk-major: the 16 taps of one 128-channel chunk are requested back to back (16 independent 128-bit loads
      // in flight per lane) and folded in the ATen order (along x inside each row, then along y); finished chunks
      // occupy 4 registers each, so the loads of the next chunk have room without spilling.
      float4 f[kChunks];
      int row_off[4], col_off[4];
#pragma unroll
      for (int t4 = 0; t4 < 4; ++t4) {
        row_off[t4] = iy[t4] * p.pw * (kDim / 4) + lane;
        col_off[t4] = ix[t4] * (kDim / 4);
      }
#pragma unroll
      for (int c = 0; c < kChunks; ++c) {
        float4 t[4][4];
#pragma unroll
        for (int ty = 0; ty < 4; ++ty)
#pragma unroll
          for (int tx = 0; tx < 4; ++tx) t[ty][tx] = __ldg(pm + (row_off[ty] + col_off[tx] + c * 32));
        // two-wide fp32 (fma.rn.f32x2): the same multiply-add chain per channel, half the instructions
        float2 lo = make_float2(0.f, 0.f), hi = lo;
#pragma unroll
        for (int ty = 0; ty < 4; ++ty) {
          const float2 w0 = make_float2(wx[0], wx[0]), w1 = make_float2(wx[1], wx[1]), w2 = make_float2(wx[2], wx[2]),
                       w3 = make_float2(wx[3], wx[3]), wv = make_float2(wy[ty], wy[ty]);
          float2 r = __fmul2_rn(make_float2(t[ty][0].x, t[ty][0].y), w0);
          r = __ffma2_rn(make_float2(t[ty][1].x, t[ty][1].y), w1, r);
          r = __ffma2_rn(make_float2(t[ty][2].x, t[ty][2].y), w2, r);
          r = __ffma2_rn(make_float2(t[ty][3].x, t[ty][3].y), w3, r);
          lo = __ffma2_rn(r, wv, lo);
          float2 q = __fmul2_rn(make_float2(t[ty][0].z, t[ty][0].w), w0);
          q = __ffma2_rn(make_float2(t[ty][1].z, t[ty][1].w), w1, q);
          q = __ffma2_rn(make_float2(t[ty][2].z, t[ty][2].w), w2, q);
          q = __ffma2_rn(make_float2(t[ty][3].z, t[ty][3].w), w3, q);
          hi = __ffma2_rn(q, wv, hi);
        }
        const float4 acc4 = make_float4(lo.x, lo.y, hi.x, hi.y);
        f[c] = acc4;
      }
      float nrm = 1.f;
      if (p.norm_feat) {
        float ss = 0.f;
#pragma unroll
        for (int c = 0; c < kChunks; ++c) ss = fmaf(f[c].x, f[c].x, fmaf(f[c].y, f[c].y, fmaf(f[c].z, f[c].z, fmaf(f[c].w, f[c].w, ss))));
        nrm = sqrtf(dc::warp_sum(ss));
        // one correctly rounded reciprocal and 4 * kChunks multiplications instead of as many IEEE divisions (8-10
        // instructions each): the quotients differ from `feat2d /= norm` by at most 1 ulp, far inside the 1e-3 bar
        const float inv = __frcp_rn(nrm);
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
          f[c].x = f[c].x * inv;
          f[c].y = f[c].y * inv;
          f[c].z = f[c].z * inv;
          f[c].w = f[c].w * inv;
        }
      }
      float4* acc = s_acc + slot * (kDim / 4) + lane;
      if (p.sim_kernel != DC_SIM_NONE) {
        asm volatile("" : "+l"(raw_id));  // keeps the narrowing (and the wait for the load) down here
        const int id = seg_id(raw_id);
        float weight = 0.f;  // pixels whose id has no query keep metric 0 (quirk q13)
        if (id >= 0 && id < n_q)
          weight = finish_weight(p, first_dot, nrm, id, n_q, lane, sim_dot);
        if (w_scene && lane == 0) w_scene[(int64_t)v * n_pts + i] = weight;
        if (lane == 0) s_den[slot] += weight;
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {  // feat2d[ys,xs] * metric, then +=  (two roundings)
          float4 a = acc[c * 32];
          a.x += f[c].x * weight;
          a.y += f[c].y * weight;
          a.z += f[c].z * weight;
          a.w += f[c].w * weight;
          acc[c * 32] = a;
        }
      } else {
        if (lane == 0) s_den[slot] += 1.f;
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
          float4 a = acc[c * 32];
          a.x += f[c].x;
          a.y += f[c].y;
          a.z += f[c].z;
          a.w += f[c].w;
          acc[c * 32] = a;
        }
      }
    }
    __syncthreads();  // the next view may hand a point to another warp
  }
  for (int slot = warp; slot < n_tile; slot += kWarps) {
    const int64_t i = __shfl_sync(0xffffffffu, my_i, slot);
    float4* dst = reinterpret_cast<float4*>(p.out_sum + (p0 + i) * kDim) + lane;
    const float den = s_den[slot];
#pragma unroll
    for (int c = 0; c < kChunks; ++c) {
      float4 a = s_acc[slot * (kDim / 4) + c * 32 + lane];
      if (p.normalize) a = make_float4(a.x / den, a.y / den, a.z / den, a.w / den);
      dst[c * 32] = a;
    }
  }
}

// similarity_mask entries of invisible (point, view) pairs are 0 (:238 writes visible pairs only into a zero tensor).
// The tile kernel writes the visible ones; this pass fills the rest with coalesced stores (the point-major kernels
// write them from inside their view loop, which in Morton order is one scattered 4-byte store per pair).
__global__ void __launch_bounds__(kThreads) zero_invisible_weights_kernel(const uint8_t* __restrict__ visible,
                                                                          const int64_t* __restrict__ mask_off,
                                                                          float* __restrict__ weight) {
  const int64_t begin = mask_off[blockIdx.y], end = mask_off[blockIdx.y + 1];
  for (int64_t j = begin + (int64_t)blockIdx.x * kThreads + threadIdx.x; j < end; j += (int64_t)gridDim.x * kThreads)
    if (!visible[j]) weight[j] = 0.f;
}

// feat[j,:] /= denom[j], denom = sum_v weight[v,j] (similarity) or sum_v visible[v,j]
__global__ void __launch_bounds__(kThreads) pixel_normalize_kernel(float* __restrict__ sums, const int64_t* __restrict__ point_off,
                                                                   const int64_t* __restrict__ view_off,
                                                                   const int64_t* __restrict__ mask_off,
                                                                   const uint8_t* __restrict__ visible,
                                                                   const float* __restrict__ weight, int dim) {
  const int scene = blockIdx.y;
  const int64_t p0 = point_off[scene];
  const int64_t n_pts = point_off[scene + 1] - p0;
  const int n_views = (int)(view_off[scene + 1] - view_off[scene]);
  const int lane = threadIdx.x & 31;
  for (int64_t i = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); i < n_pts; i += (int64_t)gridDim.x * kWarps) {
    float denom = 0.f;
    if (weight) {
      const float* w = weight + mask_off[scene];
      for (int v = 0; v < n_views; ++v) denom += w[(int64_t)v * n_pts + i];
    } else {
      const uint8_t* m = visible + mask_off[scene];
      int c = 0;
      for (int v = 0; v < n_views; ++v) c += m[(int64_t)v * n_pts + i] != 0;
      denom = (float)c;
    }
    float* row = sums + (p0 + i) * dim;
    for (int c = lane; c < dim; c += 32) row[c] = row[c] / denom;
  }
}

// generate_view_clip (data/dataset_blender.py:132-171): every point of a cloud is projected into ONE view
// (fp64 pose - the json world_matrix is inverted in fp64 there -, truncation toward zero, pixel (0,0) when the
// projected z is 0), the pixel is CLIPPED into the image instead of tested (:158-159), and the bicubically
// upsampled patch feature of that pixel is gathered (:151-156,165). No visibility, no weights. The reference
// materialises the (h, w, C) map per view; here the 16 taps are evaluated per point. Warp per (point, view);
// lanes stride over channels in float4 when the rows allow it.
template <bool kVec>
__global__ void __launch_bounds__(kThreads) view_clip_gather_kernel(const double* __restrict__ points, int64_t n_pts,
                                                                    const double* __restrict__ inv_poses,
                                                                    const double* __restrict__ intrinsics,
                                                                    const float* __restrict__ patch, int ph, int pw, int dim,
                                                                    int height, int width, float* __restrict__ out) {
  const int view = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const double* m = inv_poses + (int64_t)view * 16;
  const double* K = intrinsics;
  const float scale_y = (float)ph / (float)height, scale_x = (float)pw / (float)width;
  const float* pm = patch + (int64_t)view * ph * pw * dim;
  for (int64_t i = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); i < n_pts; i += (int64_t)gridDim.x * kWarps) {
    const double x = __ldg(points + 3 * i), y = __ldg(points + 3 * i + 1), z = __ldg(points + 3 * i + 2);
    const double cx = __dadd_rn(__ldg(m + 3), __fma_rn(__ldg(m + 2), z, __fma_rn(__ldg(m + 1), y, __dmul_rn(__ldg(m), x))));
    const double cy = -__dadd_rn(__ldg(m + 7), __fma_rn(__ldg(m + 6), z, __fma_rn(__ldg(m + 5), y, __dmul_rn(__ldg(m + 4), x))));
    const double cz = -__dadd_rn(__ldg(m + 11), __fma_rn(__ldg(m + 10), z, __fma_rn(__ldg(m + 9), y, __dmul_rn(__ldg(m + 8), x))));
    const double qx = __fma_rn(__ldg(K + 2), cz, __fma_rn(__ldg(K + 1), cy, __dmul_rn(__ldg(K), cx)));
    const double qy = __fma_rn(__ldg(K + 5), cz, __fma_rn(__ldg(K + 4), cy, __dmul_rn(__ldg(K + 3), cx)));
    const double qz = __fma_rn(__ldg(K + 8), cz, __fma_rn(__ldg(K + 7), cy, __dmul_rn(__ldg(K + 6), cx)));
    int pu = 0, pv = 0;
    if (qz != 0.0) {
      // fp64 -> int64 assignment: truncation; NaN, +-inf and anything beyond int64 become INT64_MIN, which np.clip turns into 0
      const double uq = __ddiv_rn(qx, qz), vq = __ddiv_rn(qy, qz);
      if (fabs(uq) < 9.2e18) pu = (int)max(0ll, min((long long)(width - 1), __double2ll_rz(uq)));
      if (fabs(vq) < 9.2e18) pv = (int)max(0ll, min((long long)(height - 1), __double2ll_rz(vq)));
    }
    int iy[4], ix[4];
    float wy[4], wx[4];
    cubic_taps(pv, scale_y, ph, iy, wy);
    cubic_taps(pu, scale_x, pw, ix, wx);
    float* row_out = out + ((int64_t)view * n_pts + i) * dim;
    if (kVec) {
      for (int c = lane; c < dim / 4; c += 32) {
        float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int ty = 0; ty < 4; ++ty) {
          const float* row = pm + (int64_t)iy[ty] * pw * dim;
          const float4 a = __ldg(reinterpret_cast<const float4*>(row + (int64_t)ix[0] * dim) + c);
          const float4 b = __ldg(reinterpret_cast<const float4*>(row + (int64_t)ix[1] * dim) + c);
          const float4 d = __ldg(reinterpret_cast<const float4*>(row + (int64_t)ix[2] * dim) + c);
          const float4 e = __ldg(reinterpret_cast<const float4*>(row + (int64_t)ix[3] * dim) + c);
          f.x = fmaf(a.x * wx[0] + b.x * wx[1] + d.x * wx[2] + e.x * wx[3], wy[ty], f.x);
          f.y = fmaf(a.y * wx[0] + b.y * wx[1] + d.y * wx[2] + e.y * wx[3], wy[ty], f.y);
          f.z = fmaf(a.z * wx[0] + b.z * wx[1] + d.z * wx[2] + e.z * wx[3], wy[ty], f.z);
          f.w = fmaf(a.w * wx[0] + b.w * wx[1] + d.w * wx[2] + e.w * wx[3], wy[ty], f.w);
        }
        __stcs(reinterpret_cast<float4*>(row_out) + c, f);  // written once, never re-read here
      }
    } else {
      for (int c = lane; c < dim; c += 32) {
        float f = 0.f;
#pragma unroll
        for (int ty = 0; ty < 4; ++ty) {
          const float* row = pm + (int64_t)iy[ty] * pw * dim + c;
          const float r = __ldg(row + (int64_t)ix[0] * dim) * wx[0] + __ldg(row + (int64_t)ix[1] * dim) * wx[1] +
                          __ldg(row + (int64_t)ix[2] * dim) * wx[2] + __ldg(row + (int64_t)ix[3] * dim) * wx[3];
          f = fmaf(r, wy[ty], f);
        }
        row_out[c] = f;
      }
    }
  }
}


// =====================================================================================================================
// Pixel-level fusion on the tensor cores (tcgen05).
//
// The 16-tap bicubic fold of one visible (point, view) pair is a 16 x C contraction: f = sum_t w_t T_t. Pairs that
// share a bicubic FOOTPRINT - the same view and the same first source cell (iy0, ix0), (ph + 1)(pw + 1) = 825 of them per
// view at 24 x 32 - share their 16 taps, so the pairs are counting-sorted by (view, footprint) and every 128 consecutive
// sorted pairs become one MMA tile:
//     D[128 pairs x C] = sum over the footprint segments g of the tile   A_g[128 x 16] . B_g[16 x C]
// A_g holds the pairs' 16 tap weights (zero rows outside segment g), B_g the segment's taps. fp32 accuracy on the fp16
// tensor path comes from hi/lo planes (A_hi.B_hi + A_hi.B_lo + A_lo.B_hi), as in gemm.cuh. B_g is an MN-major operand
// (taps are rows of C contiguous channels in memory) in the no-swizzle core-matrix layout, filled with 16-byte cp.async;
// A_g is K-major, written from registers. C is walked in 256-column chunks with two TMEM accumulators in flight.
// Pass NORM (only under norm_feat): the epilogue reduces sum f^2 per pair. A warp-per-pair kernel then evaluates the
// similarity weight (fp64 chain of finish_weight) and the pair's scale = weight / |f|. Pass ACCUM: the epilogue scales
// the row and adds it to the point's output row with red.global.add.v4.f32 (rows of one point come from different tiles;
// the order of the additions is not fixed, the sums differ from a view-ordered sum by fp32 rounding only).
// =====================================================================================================================
inline int query_stride_(int max_queries) { return (max_queries + 3) & ~3; }

namespace mma {

using namespace dc::umma;

constexpr int kStages = 6;
constexpr int kABytes = 4096;    // one plane of A: [2 k-halves][16 row groups][8 rows][16 B]
constexpr int kBBytes = 8192;    // one plane of B: [2 k-groups][32 column groups][8 taps][16 B]   (N = 256)
constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;
constexpr int kLoaderThreads = 128;
constexpr int kMmaWarp = 4;
constexpr int kEpiWarp0 = 8;
constexpr int kEpiWarps = 8;       // two groups of four (TMEM lane quarters): group h owns columns [128 h, 128 h + 128) of a chunk
constexpr int kThreadsMma = (kEpiWarp0 + kEpiWarps) * 32;
constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 512 /*barriers*/ + 1024 /*row keys*/ + kEpiWarps * 32 * 36 * 4 /*epilogue transposition*/;

struct Footprints {
  int ph, pw, height, width;
  // Sort key = (region, global view, footprint). A region is a contiguous range of the scene's Morton order (rank from
  // dc_spatial_sort): all tiles of region 0 (every view) come first, then region 1, ... so that the output rows the
  // accumulate pass adds to at any time (one region: N / n_regions rows) stay resident in L2; being spatially compact, a
  // region keeps the pairs-per-footprint density of the whole scene. rank == nullptr: one region.
  int n_regions;
  int64_t total_views;
  const int64_t* rank;
  __host__ __device__ int per_view() const { return (ph + 1) * (pw + 1); }
  __device__ int region_of(int64_t global_point, int64_t n_pts) const {
    if (!rank || n_regions <= 1) return 0;
    const int r = (int)((rank[global_point] * n_regions) / n_pts);
    return r < n_regions ? r : n_regions - 1;
  }
  __device__ int key_of(int region, int64_t v_glob, int fp) const { return (int)((region * total_views + v_glob) * per_view() + fp); }
  __device__ int view_of_key(int key) const { return (int)((key / per_view()) % total_views); }
};

// first source cell of the bicubic footprint of destination pixel `dst` (ATen: floor(scale * (dst + 0.5) - 0.5)), in [-1, in - 1]
__device__ __forceinline__ int first_cell(int dst, int in_size, int out_size) {
  const double src = ((double)in_size / (double)out_size) * ((double)dst + 0.5) - 0.5;
  return (int)floor(src);
}
__device__ __forceinline__ int footprint_of(const Footprints& f, int pu, int pv) {
  return (first_cell(pv, f.ph, f.height) + 1) * (f.pw + 1) + (first_cell(pu, f.pw, f.width) + 1);
}

// the projection of visibility.cu / pixel_fuse_tile_kernel (the pair is visible, hence inside the image)
__device__ __forceinline__ void project_pixel(const double* __restrict__ m, const double* __restrict__ K, double x, double y,
                                              double z, int& pu, int& pv) {
  double cx = __dadd_rn(m[3], __fma_rn(m[2], z, __fma_rn(m[1], y, __dmul_rn(m[0], x))));
  double cy = __dadd_rn(m[7], __fma_rn(m[6], z, __fma_rn(m[5], y, __dmul_rn(m[4], x))));
  double cz = __dadd_rn(m[11], __fma_rn(m[10], z, __fma_rn(m[9], y, __dmul_rn(m[8], x))));
  cy = -cy;
  cz = -cz;
  const double qx = __fma_rn(K[2], cz, __fma_rn(K[1], cy, __dmul_rn(K[0], cx)));
  const double qy = __fma_rn(K[5], cz, __fma_rn(K[4], cy, __dmul_rn(K[3], cx)));
  const double qz = __fma_rn(K[8], cz, __fma_rn(K[7], cy, __dmul_rn(K[6], cx)));
  pu = 0;
  pv = 0;
  if (qz != 0.0) {
    pu = (int)__ddiv_rn(qx, qz);
    pv = (int)__ddiv_rn(qy, qz);
  }
}

// thread per point, loop over the scene's views: pixel of every visible pair (stashed in mask layout) and the histogram
// of (global view, footprint) keys
__global__ void __launch_bounds__(kThreads) pair_count_kernel(PixParams p, Footprints fp, uint32_t* __restrict__ pix,
                                                              unsigned* __restrict__ counts) {
  const int scene = blockIdx.y;
  const int64_t p0 = p.point_off[scene], n_pts = p.point_off[scene + 1] - p0;
  const int64_t v0 = p.view_off[scene];
  const int n_views = (int)(p.view_off[scene + 1] - v0);
  const uint8_t* vis = p.visible + p.mask_off[scene];
  uint32_t* px = pix + p.mask_off[scene];
  double K[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) K[e] = __ldg(p.intrinsics + (int64_t)scene * 9 + e);
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n_pts; i += (int64_t)gridDim.x * kThreads) {
    const double x = __ldg(p.points + 3 * (p0 + i)), y = __ldg(p.points + 3 * (p0 + i) + 1), z = __ldg(p.points + 3 * (p0 + i) + 2);
    const int region = fp.region_of(p0 + i, n_pts);
    for (int v = 0; v < n_views; ++v) {
      if (!vis[(int64_t)v * n_pts + i]) continue;
      double m[12];
#pragma unroll
      for (int e = 0; e < 12; ++e) m[e] = __ldg(p.inv_poses + (v0 + v) * 16 + e);
      int pu, pv;
      project_pixel(m, K, x, y, z, pu, pv);
      // a pair the visibility kernels marked visible projects inside the image; a hand-made mask must not index outside
      pu = min(max(pu, 0), p.width - 1);
      pv = min(max(pv, 0), p.height - 1);
      px[(int64_t)v * n_pts + i] = (uint32_t)pu | ((uint32_t)pv << 16);
      atomicAdd(counts + fp.key_of(region, v0 + v, footprint_of(fp, pu, pv)), 1u);
    }
  }
}

// exclusive scan of `n` counters (three launches): per-block sums, scan of the block sums by one CTA, local scans + bases.
constexpr int kScanBlock = 1024;
__global__ void __launch_bounds__(kScanBlock) scan_sums_kernel(const unsigned* __restrict__ in, int64_t n, unsigned* __restrict__ sums) {
  __shared__ unsigned s_w[32];
  const int64_t i = (int64_t)blockIdx.x * kScanBlock + threadIdx.x;
  unsigned v = i < n ? in[i] : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    unsigned t = s_w[threadIdx.x];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) sums[blockIdx.x] = t;
  }
}
__global__ void __launch_bounds__(kScanBlock) scan_bases_kernel(unsigned* __restrict__ sums, int64_t n_blocks, unsigned* __restrict__ total) {
  __shared__ unsigned s_w[32];
  __shared__ unsigned s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int64_t b0 = 0; b0 < n_blocks; b0 += kScanBlock) {
    const int64_t i = b0 + threadIdx.x;
    const unsigned v = i < n_blocks ? sums[i] : 0u;
    unsigned incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned up = __shfl_up_sync(0xffffffffu, incl, o);
      if ((threadIdx.x & 31) >= o) incl += up;
    }
    if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      const unsigned t = s_w[threadIdx.x];
      unsigned ti = t;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned up = __shfl_up_sync(0xffffffffu, ti, o);
        if (threadIdx.x >= o) ti += up;
      }
      s_w[threadIdx.x] = ti - t;
    }
    __syncthreads();
    const unsigned base = s_carry + s_w[threadIdx.x >> 5];
    if (i < n_blocks) sums[i] = base + incl - v;
    __syncthreads();
    if (threadIdx.x == kScanBlock - 1) s_carry = base + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = s_carry;
}
__global__ void __launch_bounds__(kScanBlock) scan_apply_kernel(unsigned* __restrict__ data, int64_t n, const unsigned* __restrict__ bases) {
  __shared__ unsigned s_w[32];
  const int64_t i = (int64_t)blockIdx.x * kScanBlock + threadIdx.x;
  const unsigned v = i < n ? data[i] : 0u;
  unsigned incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned up = __shfl_up_sync(0xffffffffu, incl, o);
    if ((threadIdx.x & 31) >= o) incl += up;
  }
  if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = incl;
  __syncthreads();
  if (threadIdx.x < 32) {
    const unsigned t = s_w[threadIdx.x];
    unsigned ti = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned up = __shfl_up_sync(0xffffffffu, ti, o);
      if (threadIdx.x >= o) ti += up;
    }
    s_w[threadIdx.x] = ti - t;
  }
  __syncthreads();
  if (i < n) data[i] = bases[blockIdx.x] + s_w[threadIdx.x >> 5] + incl - v;
}

// sorted pair records: global point index, packed pixel, key; and the pair's 16 tap weights as fp16 hi/lo planes
// (w_t = wy[ty] * wx[tx] from the fp64 coefficients of cubic_weights64, t = 4 ty + tx)
__global__ void __launch_bounds__(kThreads) pair_scatter_kernel(PixParams p, Footprints fp, const uint32_t* __restrict__ pix,
                                                                unsigned* __restrict__ cursor, int* __restrict__ rec_point,
                                                                uint32_t* __restrict__ rec_pix, int* __restrict__ rec_key,
                                                                __half* __restrict__ arec) {
  const int scene = blockIdx.y;
  const int64_t p0 = p.point_off[scene], n_pts = p.point_off[scene + 1] - p0;
  const int64_t v0 = p.view_off[scene];
  const int n_views = (int)(p.view_off[scene + 1] - v0);
  const uint8_t* vis = p.visible + p.mask_off[scene];
  const uint32_t* px = pix + p.mask_off[scene];
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n_pts; i += (int64_t)gridDim.x * kThreads) {
    const int region = fp.region_of(p0 + i, n_pts);
    for (int v = 0; v < n_views; ++v) {
      if (!vis[(int64_t)v * n_pts + i]) continue;
      const uint32_t pp = px[(int64_t)v * n_pts + i];
      const int pu = (int)(pp & 0xffffu), pv = (int)(pp >> 16);
      const int key = fp.key_of(region, v0 + v, footprint_of(fp, pu, pv));
      const unsigned pos = atomicAdd(cursor + key, 1u);
      rec_point[pos] = (int)(p0 + i);
      rec_pix[pos] = pp;
      rec_key[pos] = key;
      double wy[4], wx[4];
      cubic_weights64(pv, fp.ph, fp.height, wy);
      cubic_weights64(pu, fp.pw, fp.width, wx);
      __half hi[16], lo[16];
#pragma unroll
      for (int ty = 0; ty < 4; ++ty)
#pragma unroll
        for (int tx = 0; tx < 4; ++tx) {
          const float w = (float)(wy[ty] * wx[tx]);
          const __half h = __float2half_rn(w);
          hi[ty * 4 + tx] = h;
          lo[ty * 4 + tx] = __float2half_rn(w - __half2float(h));
        }
      int4* dst = reinterpret_cast<int4*>(arec + (int64_t)pos * 32);
      dst[0] = reinterpret_cast<const int4*>(hi)[0];
      dst[1] = reinterpret_cast<const int4*>(hi)[1];
      dst[2] = reinterpret_cast<const int4*>(lo)[0];
      dst[3] = reinterpret_cast<const int4*>(lo)[1];
    }
  }
}

// ---- descriptors (cute/atom/mma_traits_sm100.hpp documents the canonical layouts; no-swizzle = "INTERLEAVE")
// K-major, no swizzle:  ((8, m), (8, 2)) : ((16 B, SBO), (1 elem, LBO))  - 8 x 16 B core matrices, SBO between row groups,
//                       LBO between the two k-halves.        MN-major, no swizzle: ((8, m), (8, k)) : ((1 elem, SBO), (16 B, LBO))
__device__ __forceinline__ uint64_t smem_desc_noswizzle(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;  // version
  return d;                // layout type 0 = no swizzle
}
// MN-major, SWIZZLE_128B:  ((8, 8, m), (8, k)) : ((1 elem, 16 B, LBO), (128 B, SBO)) with Swizzle<3,4,3> - LBO between the
// 64-element atoms along N, SBO between the 8-row groups along K
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;  // version
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}
// fp32 accumulator, fp16 A (K-major) and B (MN-major: bit 16)
__host__ __device__ constexpr uint32_t idesc_f16_f32_bmn(int m, int n) {
  return (1u << 4) | (1u << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
// 16 bytes from global memory, or 16 zero bytes when !take (src-size 0: nothing is read)
__device__ __forceinline__ void cp_async16_or_zero(void* smem_dst, const void* gsrc, bool take) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(take ? 16 : 0) : "memory");
}
// arrival on the mbarrier once all cp.async of this thread issued so far have landed (counts against the expected arrivals)
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

struct MmaParams {
  const int* rec_point;
  const int* rec_key;
  const __half* arec;       // [pairs][32]: 16 hi, 16 lo
  const __half* plane_hi;   // [total_views * ph * pw][dim]
  const __half* plane_lo;
  const unsigned* n_pairs;  // device scalar
  int ph, pw, dim, nfp;     // nfp = footprints per view
  int total_views;          // key = (region * total_views + view) * nfp + footprint
  float* norm2;             // [pairs]  (pass NORM)
  const float* scale;       // [pairs]  (pass ACCUM)
  float* out;               // [total_points][dim]
};

template <bool kAccum>
__global__ void __launch_bounds__(kThreadsMma, 1) pixel_mma_kernel(const MmaParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);  // SWIZZLE_128B operand atoms need 1024-byte alignment
  uint8_t* stages = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* full = bars;                 // [kStages]  128 loader arrivals
  uint64_t* empty = bars + kStages;      // [kStages]  MMA commit
  uint64_t* tmem_full = bars + 2 * kStages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;       // [2]  4 epilogue warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  unsigned* s_mask = reinterpret_cast<unsigned*>(tmem_slot + 2);  // [2 tile slots][4 warps]
  int* s_last = reinterpret_cast<int*>(s_mask + 8);               // [kStages] 1 when the stage holds the last segment of its (tile, chunk)
  int* s_keys = reinterpret_cast<int*>(smem + kStages * kStageBytes + 512);       // [2 tile slots][128] sort keys of the tile's rows
  float* s_trans = reinterpret_cast<float*>(smem + kStages * kStageBytes + 512 + 1024);  // [4 epilogue warps][32][36] transposition blocks

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned n_pairs = *p.n_pairs;
  const int n_tiles = (int)((n_pairs + 127u) / 128u);
  const int n_chunks = p.dim / 256;
  const int ncell = p.ph * p.pw;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full + s, kLoaderThreads + 1);  // 128 cp.async completions + thread 0's arrival behind the segment flag
      mbar_init(empty + s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tmem_full + a, 1);
      mbar_init(tmem_empty + a, kEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ===================== loaders: thread r <-> row r of the tile =====================
    const int r = threadIdx.x;
    int stage = 0;
    uint32_t phase = 0;

    int local_tile = 0;
    // rows of a tile: sort key, the key of the row before (segment starts) and the 16 tap weights (hi / lo). They are
    // fetched one tile AHEAD, so that a tile's first stage is not issued behind two dependent global-load latencies.
    struct Rows { int key, prev; };
    auto fetch_rows = [&](int tile) -> Rows {
      Rows t{-1, -2};
      const unsigned row = (unsigned)tile * 128u + (unsigned)r;
      if (tile < n_tiles && row < n_pairs) {
        t.key = __ldg(p.rec_key + row);
        if (r != 0) t.prev = __ldg(p.rec_key + row - 1);
      }
      return t;
    };
    Rows next = fetch_rows(blockIdx.x);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++local_tile) {
      const int slot = local_tile & 1;
      const Rows cur = next;
      next = fetch_rows(tile + gridDim.x);
      const int key = cur.key;
      const unsigned starts = __ballot_sync(0xffffffffu, key >= 0 && key != cur.prev);
      // my row's 16 tap weights (hi, lo) in global memory; rows past the end are never inside a segment
      const __half* my_arec = p.arec + (int64_t)(key >= 0 ? (unsigned)tile * 128u + (unsigned)r : 0u) * 32;
      if (lane == 0) s_mask[slot * 4 + warp] = starts;
      s_keys[slot * 128 + r] = key;  // a segment's key is read from here (a global load per stage sat on the critical path)
      asm volatile("bar.sync 2, 128;" ::: "memory");
      unsigned m[4];
      int nseg = 0;
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        m[w] = s_mask[slot * 4 + w];
        nseg += __popc(m[w]);
      }
      const int n_rows = (int)min(128u, n_pairs - (unsigned)tile * 128u);
      for (int c = 0; c < n_chunks; ++c) {
        int w = 0;
        unsigned bits = m[0];
        int seg_start = -1;
        // walk the segment starts in row order; the segment [seg_start, next start) is emitted when its end is known
        for (;;) {
          int next;
          while (w < 4 && bits == 0) { ++w; bits = w < 4 ? m[w] : 0u; }
          if (w < 4) {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            next = w * 32 + b;
          } else {
            next = n_rows;
          }
          if (seg_start >= 0) {
            const int seg_end = next;
            const int seg_key = s_keys[slot * 128 + seg_start];
            uint8_t* st = stages + stage * kStageBytes;
            mbar_wait(empty + stage, phase ^ 1);
            if (r == 0) {  // read by the MMA warp behind this stage's full barrier (a plain arrival: release)
              s_last[stage] = (seg_end >= n_rows) ? 1 : 0;
              mbar_arrive(full + stage);
            }
            // A: my row's 16 weights, or zeros outside the segment - also by cp.async (zero-fill form), so that the loader
            // never touches the stage through the generic proxy and never has to wait for its own copies
            const bool mine = r >= seg_start && r < seg_end;
            uint8_t* arow = st + (r >> 3) * 128 + (r & 7) * 16;
            cp_async16_or_zero(arow, my_arec, mine);
            cp_async16_or_zero(arow + 2048, my_arec + 8, mine);
            cp_async16_or_zero(arow + kABytes, my_arec + 16, mine);
            cp_async16_or_zero(arow + kABytes + 2048, my_arec + 24, mine);
            // B: 16 taps x 256 channels of both planes, 16 bytes per copy
            const int vk = seg_key / p.nfp, f = seg_key - vk * p.nfp;
            const int v_glob = vk % p.total_views;
            const int iy0 = f / (p.pw + 1) - 1, ix0 = f - (f / (p.pw + 1)) * (p.pw + 1) - 1;
            uint8_t* bh = st + 2 * kABytes;
            uint8_t* bl = bh + kBBytes;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int idx = r + 128 * j;
              const int t = idx >> 5, g8 = idx & 31;
              const int cy = min(max(iy0 - 1 + (t >> 2), 0), p.ph - 1), cx = min(max(ix0 - 1 + (t & 3), 0), p.pw - 1);
              const int64_t src = ((int64_t)v_glob * ncell + cy * p.pw + cx) * p.dim + c * 256 + g8 * 8;
              // MN-major SWIZZLE_128B: atoms of 8 taps x 64 channels (8 rows of 128 B, 16-byte chunk index XOR tap row),
              // four atoms along N (1024 B apart), two tap groups (4096 B apart). The no-swizzle core-matrix layout put the
              // 32 column groups of a tap row 128 B apart - every operand fetch of the tensor core hit the same banks.
              const int dst = (t >> 3) * 4096 + (g8 >> 3) * 1024 + (t & 7) * 128 + (((g8 & 7) ^ (t & 7)) << 4);
              cp_async16(bh + dst, p.plane_hi + src);
              cp_async16(bl + dst, p.plane_lo + src);
            }
            cp_async_arrive_noinc(full + stage);  // arrives when this thread's copies of the stage have landed
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
          if (next >= n_rows) break;
          seg_start = next;
        }
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = idesc_f16_f32_bmn(128, 256);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int local_tile = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++local_tile) {
        for (int c = 0; c < n_chunks; ++c) {
          mbar_wait(tmem_empty + acc, acc_phase ^ 1);
          fence_after_sync();
          const uint32_t d_tmem = tmem_base + (uint32_t)(acc * 256);
          bool last = false;
          for (int g = 0; !last; ++g) {
            mbar_wait(full + stage, phase);
            // the stage was written by the loaders' cp.async (generic proxy); the MMA reads it through the async proxy
#ifndef DC_EXPERIMENT_NO_PROXY_FENCE
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#endif
            fence_after_sync();
            last = *reinterpret_cast<volatile int*>(s_last + stage) != 0;
            const uint32_t a_hi = smem_u32(stages + stage * kStageBytes), a_lo = a_hi + kABytes;
            const uint32_t b_hi = a_hi + 2 * kABytes, b_lo = b_hi + kBBytes;
            const uint64_t da_hi = smem_desc_noswizzle(a_hi, 2048, 128), da_lo = smem_desc_noswizzle(a_lo, 2048, 128);
            const uint64_t db_hi = smem_desc_mn_sw128(b_hi, 1024, 4096), db_lo = smem_desc_mn_sw128(b_lo, 1024, 4096);
            mma_f16_ss(d_tmem, da_hi, db_hi, idesc, g ? 1u : 0u);
            mma_f16_ss(d_tmem, da_hi, db_lo, idesc, 1u);
            mma_f16_ss(d_tmem, da_lo, db_hi, idesc, 1u);
            mma_commit(empty + stage);
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
          mma_commit(tmem_full + acc);
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ===================== epilogue: thread <-> row, warp group h <-> column half h of the chunk =====================
    const int quarter = warp & 3;
    const int half = (warp - kEpiWarp0) >> 2;
    const int r = quarter * 32 + lane;
    float* tb = s_trans + (warp - kEpiWarp0) * (32 * 36);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const unsigned row = (unsigned)tile * 128u + (unsigned)r;
      const bool valid = row < n_pairs;
      const int point = valid ? __ldg(p.rec_point + row) : -1;
      const float sc = (kAccum && valid) ? __ldg(p.scale + row) : 0.f;
      float ss = 0.f;
      for (int c = 0; c < n_chunks; ++c) {
        mbar_wait(tmem_full + acc, acc_phase);
        fence_after_sync();
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 256 + half * 128);
        const int col0 = c * 256 + half * 128;
        // four 32-column blocks, the TMEM load of block cc + 1 in flight while block cc is processed
        uint32_t va[32], vb[32];
        tmem_ld_32x32(taddr, va);
        tmem_ld_wait();
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          uint32_t(&v)[32] = (cc & 1) ? vb : va;
          uint32_t(&nx)[32] = (cc & 1) ? va : vb;
          if (cc + 1 < 4) tmem_ld_32x32(taddr + (uint32_t)((cc + 1) * 32), nx);
          if (kAccum) {
            // thread = row out of TMEM, but a warp-wide red of one row segment per thread would touch 32 half-used sectors:
            // the 32 x 32 block goes through shared memory (row stride 36 floats) and comes back with 8 lanes per row,
            // so one red instruction adds 4 rows x 128 contiguous bytes (16 full sectors)
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              *reinterpret_cast<float4*>(tb + lane * 36 + i) = make_float4(__uint_as_float(v[i]) * sc, __uint_as_float(v[i + 1]) * sc,
                                                                          __uint_as_float(v[i + 2]) * sc, __uint_as_float(v[i + 3]) * sc);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int rr = i * 4 + (lane >> 3);
              const int pt = __shfl_sync(0xffffffffu, point, rr);
              const float4 q = *reinterpret_cast<const float4*>(tb + rr * 36 + (lane & 7) * 4);
              if (pt >= 0) red_add_v4(p.out + (int64_t)pt * p.dim + col0 + cc * 32 + (lane & 7) * 4, q.x, q.y, q.z, q.w);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) ss = fmaf(__uint_as_float(v[i]), __uint_as_float(v[i]), ss);
          }
          if (cc + 1 < 4) tmem_ld_wait();
        }
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(tmem_empty + acc);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (!kAccum && valid) atomicAdd(p.norm2 + row, ss);  // the two column halves of a row meet here (norm2 starts at zero)
    }
  }

  fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) {
    __syncwarp();
    fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

// thread per sorted pair: similarity weight and the scale the ACCUM pass applies (weight / |f| under norm_feat, weight
// otherwise; weight = 1 without similarity); also writes similarity_mask. Same fp64 chain as finish_weight (table of
// (patch cell . query) dots interpolated with the fp64 bicubic weights, pos - max|mean(neg), one division by |f|, clip),
// organised per thread: neighbouring pairs of the sorted order share their footprint, so the 16 x Q table loads of a warp
// are broadcasts.
__global__ void __launch_bounds__(kThreads) pair_weight_kernel(PixParams p, Footprints fp, int n_scenes, const int* __restrict__ rec_point,
                                                               const uint32_t* __restrict__ rec_pix, const int* __restrict__ rec_key,
                                                               const unsigned* __restrict__ n_pairs_dev, const float* __restrict__ norm2,
                                                               float* __restrict__ scale, float* __restrict__ den) {
  const unsigned n_pairs = *n_pairs_dev;
  const int64_t hw = (int64_t)p.height * p.width;
  for (unsigned pair = blockIdx.x * kThreads + threadIdx.x; pair < n_pairs; pair += gridDim.x * kThreads) {
    const int key = __ldg(rec_key + pair);
    const int v_glob = fp.view_of_key(key);
    const uint32_t pp = __ldg(rec_pix + pair);
    const int pu = (int)(pp & 0xffffu), pv = (int)(pp >> 16);
    const float nrm = p.norm_feat ? sqrtf(__ldg(norm2 + pair)) : 1.f;
    float weight = 1.f;
    if (p.sim_kernel != DC_SIM_NONE) {
      int lo = 0, hi = n_scenes;  // scene of the view: last s with view_off[s] <= v_glob
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (p.view_off[mid] <= v_glob) lo = mid; else hi = mid;
      }
      const int scene = lo;
      const int n_q = (int)(p.query_off[scene + 1] - p.query_off[scene]);
      const int id = seg_at(p.seg, p.seg_dtype, (int64_t)v_glob * hw + (int64_t)pv * p.width + pu);
      weight = 0.f;  // pixels whose id has no query keep metric 0 (quirk q13)
      if (id >= 0 && id < n_q) {
        double wy64[4], wx64[4];
        const int iy0 = cubic_weights64(pv, p.ph, p.height, wy64), ix0 = cubic_weights64(pu, p.pw, p.width, wx64);
        const double* dots_view = p.dots + (int64_t)v_glob * p.ph * p.pw * p.q_stride;
        const double* cell[16];
#pragma unroll
        for (int ty = 0; ty < 4; ++ty)
#pragma unroll
          for (int tx = 0; tx < 4; ++tx) {
            const int cy = min(max(iy0 - 1 + ty, 0), p.ph - 1), cx = min(max(ix0 - 1 + tx, 0), p.pw - 1);
            cell[ty * 4 + tx] = dots_view + ((int64_t)cy * p.pw + cx) * p.q_stride;
          }
        double pos = 0.0, red = (p.sim_kernel == DC_SIM_MAX) ? -INFINITY : 0.0;
        bool nan_seen = false;
        for (int o = 0; o < n_q; ++o) {
          // the association of interp_dot: along x inside each row of taps, then along y
          double mine = 0.0;
#pragma unroll
          for (int ty = 0; ty < 4; ++ty) {
            double r = __ldg(cell[ty * 4] + o) * wx64[0];
            r = fma(__ldg(cell[ty * 4 + 1] + o), wx64[1], r);
            r = fma(__ldg(cell[ty * 4 + 2] + o), wx64[2], r);
            r = fma(__ldg(cell[ty * 4 + 3] + o), wx64[3], r);
            mine = fma(r, wy64[ty], mine);
          }
          if (o == id) pos = mine;
          else {
            nan_seen |= (mine != mine);
            if (p.sim_kernel == DC_SIM_MAX) red = fmax(red, mine); else red += mine;
          }
        }
        if (p.sim_kernel == DC_SIM_MEAN) red = red / (double)(n_q - 1);
        if (nan_seen) red = __longlong_as_double(0x7ff8000000000000ll);
        double w = pos - red;
        if (p.norm_feat) w = w / (double)nrm;  // nrm = 0 (an all-zero feature): 0 / 0 = NaN like the reference's f / |f|
        weight = (float)w;
        if (weight == weight) weight = fmaxf(weight, 1e-6f);
      }
      if (p.out_weight) {
        const int64_t p0 = p.point_off[scene], n_pts = p.point_off[scene + 1] - p0;
        const int v_local = (int)(v_glob - p.view_off[scene]);
        p.out_weight[p.mask_off[scene] + (int64_t)v_local * n_pts + (__ldg(rec_point + pair) - p0)] = weight;
      }
    }
    scale[pair] = p.norm_feat ? weight / nrm : weight;  // (f / |f|) * weight; 0 / 0 = NaN like the reference
    if (den) atomicAdd(den + __ldg(rec_point + pair), weight);  // denominator of fuse_points :266-268 (sum of weights / view count)
  }
}

// normalize: the division of fuse_points is folded into the pair scales (sum_v s_v f_v / den = sum_v (s_v / den) f_v), and the
// rows of points nobody sees become 0 / 0 = NaN like the separate division pass would leave them
__global__ void __launch_bounds__(kThreads) pair_scale_div_kernel(const int* __restrict__ rec_point, const unsigned* __restrict__ n_pairs_dev,
                                                                  const float* __restrict__ den, float* __restrict__ scale) {
  const unsigned n_pairs = *n_pairs_dev;
  for (unsigned pair = blockIdx.x * kThreads + threadIdx.x; pair < n_pairs; pair += gridDim.x * kThreads)
    scale[pair] = scale[pair] / __ldg(den + __ldg(rec_point + pair));
}
__global__ void __launch_bounds__(kThreads) nan_unseen_rows_kernel(const float* __restrict__ den, int64_t total_points, int dim,
                                                                   float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  for (int64_t i = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); i < total_points; i += (int64_t)gridDim.x * kWarps) {
    if (__ldg(den + i) != 0.f) continue;  // (a NaN denominator already made the row NaN through its scales)
    float* row = out + i * dim;
    for (int c = lane; c < dim; c += 32) row[c] = __int_as_float(0x7fc00000);
  }
}

struct Workspace {
  size_t dots, pix, counts, sums, total, rec_point, rec_pix, rec_key, arec, norm2, scale, den, plane_hi, plane_lo, bytes;
  int64_t n_keys, n_scan_blocks;
};
constexpr int kMaxRegions = 32;
Workspace layout(int64_t total_views, int64_t mask_elems, int ph, int pw, int dim, int max_q) {
  Workspace w{};
  size_t off = 0;
  auto take = [&](size_t b) { const size_t o = off; off = (off + b + 255) / 256 * 256; return o; };
  const int64_t pairs = mask_elems > 0 ? mask_elems : 1;
  w.n_keys = (int64_t)kMaxRegions * total_views * (ph + 1) * (pw + 1);  // sized for the most regions; a call scans what it uses
  w.n_scan_blocks = (w.n_keys + kScanBlock - 1) / kScanBlock;
  w.dots = take(max_q > 0 ? (size_t)total_views * ph * pw * query_stride_(max_q) * sizeof(double) : 0);
  w.pix = take((size_t)pairs * 4);
  w.counts = take((size_t)(w.n_keys > 0 ? w.n_keys : 1) * 4);
  w.sums = take((size_t)(w.n_scan_blocks > 0 ? w.n_scan_blocks : 1) * 4);
  w.total = take(256);
  w.rec_point = take((size_t)pairs * 4);
  w.rec_pix = take((size_t)pairs * 4);
  w.rec_key = take((size_t)pairs * 4);
  w.arec = take((size_t)pairs * 64);
  w.norm2 = take((size_t)pairs * 4);
  w.scale = take((size_t)pairs * 4);
  w.den = take((size_t)pairs * 4);  // per point (<= pairs)
  w.plane_hi = take((size_t)total_views * ph * pw * dim * 2);
  w.plane_lo = take((size_t)total_views * ph * pw * dim * 2);
  w.bytes = off;
  return w;
}

}  // namespace mma

unsigned blocks_for(int64_t max_points, int n_scenes) {
  int64_t want = dc::ceil_div<int64_t>(max_points, kWarps);
  int64_t cap = dc::ceil_div<int64_t>((int64_t)dc::sm_count() * 16, n_scenes);
  if (want > cap) want = cap;
  return (unsigned)(want < 1 ? 1 : want);
}

int query_stride(int max_queries) { return (max_queries + 3) & ~3; }  // whole 32-byte sectors per (cell) row of doubles

}  // namespace

extern "C" {

size_t dc_pixel_fuse_workspace(int64_t total_views, int patch_h, int patch_w, int max_queries_per_scene) {
  if (total_views <= 0 || patch_h <= 0 || patch_w <= 0 || max_queries_per_scene <= 0) return 0;
  return (size_t)total_views * patch_h * patch_w * query_stride(max_queries_per_scene) * sizeof(double);
}

int dc_pixel_fuse(const double* points, const int64_t* point_off, const int64_t* view_off, const double* inv_poses,
                  const double* intrinsics, const int64_t* mask_off, const uint8_t* visible, const void* seg, int seg_dtype,
                  const float* patch_feats, int patch_h, int patch_w, int dim, const float* queries,
                  const int64_t* query_off, int sim_kernel, int norm_feat, int n_scenes, int64_t max_points_per_scene,
                  int max_views_per_scene, int height, int width, const int64_t* perm, float* out_sum, float* out_weight,
                  int normalize, int64_t total_views, int max_queries_per_scene, void* workspace, size_t workspace_bytes,
                  dc_stream_t stream) {
  DC_CHECK_ARG(points && point_off && view_off && inv_poses && intrinsics && mask_off && visible && patch_feats && out_sum,
               "dc_pixel_fuse: null pointer argument");
  DC_CHECK_ARG(sim_kernel >= DC_SIM_NONE && sim_kernel <= DC_SIM_MEAN, "dc_pixel_fuse: Please set method in [mean, max]");
  DC_CHECK_ARG(sim_kernel == DC_SIM_NONE || (queries && query_off && seg), "dc_pixel_fuse: similarity needs queries and seg");
  DC_CHECK_ARG(dim > 0 && dim % 32 == 0 && dim <= 32 * kMaxPerLane, "dc_pixel_fuse: dim must be a multiple of 32, <= %d",
               32 * kMaxPerLane);
  DC_CHECK_ARG(patch_h > 0 && patch_w > 0 && height > 0 && width > 0, "dc_pixel_fuse: bad sizes");
  if (n_scenes <= 0 || max_points_per_scene <= 0) return DC_OK;
  DC_CHECK_ARG(n_scenes <= 65535, "dc_pixel_fuse: at most 65535 scenes per call");
  const size_t smem = ((size_t)max_views_per_scene * 12 + 9) * sizeof(double);
  DC_CHECK_ARG(smem <= 48 * 1024, "dc_pixel_fuse: too many views per scene (%d)", max_views_per_scene);
  PixParams p{points, point_off, view_off, inv_poses, intrinsics, mask_off, visible, seg, seg_dtype, patch_feats, patch_h,
              patch_w, dim, queries, query_off, sim_kernel, norm_feat, height, width, perm, out_sum, out_weight, nullptr, 0, normalize};
  dim3 grid(blocks_for(max_points_per_scene, n_scenes), (unsigned)n_scenes);
  const bool aligned = (((uintptr_t)patch_feats | (uintptr_t)out_sum) & 15) == 0;
  cudaStream_t st = dc::as_stream(stream);
  if (sim_kernel != DC_SIM_NONE) {
    DC_CHECK_ARG(total_views >= 0 && max_queries_per_scene >= 0, "dc_pixel_fuse: bad extents");
    const size_t need = dc_pixel_fuse_workspace(total_views, patch_h, patch_w, max_queries_per_scene);
    DC_CHECK_ARG(workspace && workspace_bytes >= need, "dc_pixel_fuse: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    DC_CHECK_ARG(((uintptr_t)workspace & 7) == 0, "dc_pixel_fuse: workspace must be 8-byte aligned");
    p.dots = static_cast<double*>(workspace);
    p.q_stride = query_stride(max_queries_per_scene);
    if (total_views > 0 && max_queries_per_scene > 0) {
      const int64_t rows = (int64_t)max_views_per_scene * patch_h * patch_w;
      dim3 dgrid(blocks_for(rows, n_scenes), (unsigned)n_scenes);
      patch_query_dots_kernel<<<dgrid, kThreads, 0, st>>>(p);
      DC_LAUNCH_CHECK();
    }
  }
  if (aligned && (dim == 768 || dim == 512 || dim == 1024)) {  // CLIP ViT-L/14, ViT-B, ViT-H widths
    const size_t cam_doubles = ((size_t)max_views_per_scene * 12 + 9 + 1) & ~(size_t)1;
    const size_t tsmem = cam_doubles * sizeof(double) + (size_t)kTilePts * dim * sizeof(float) + kTilePts * sizeof(float) +
                         kTilePts * (8 * sizeof(double) + 2 * sizeof(int));
    dim3 tgrid((unsigned)dc::ceil_div<int64_t>(max_points_per_scene, kTilePts), (unsigned)n_scenes);
    DC_CHECK_ARG(tsmem <= 200 * 1024, "dc_pixel_fuse: too many views per scene (%d)", max_views_per_scene);
    // the attribute belongs to the (function, device) pair, so it is set on every call for the device in use
    const void* fn = dim == 768 ? (const void*)pixel_fuse_tile_kernel<6>
                   : dim == 512 ? (const void*)pixel_fuse_tile_kernel<4> : (const void*)pixel_fuse_tile_kernel<8>;
    DC_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    if (dim == 768) pixel_fuse_tile_kernel<6><<<tgrid, kThreads, tsmem, st>>>(p);
    else if (dim == 512) pixel_fuse_tile_kernel<4><<<tgrid, kThreads, tsmem, st>>>(p);
    else pixel_fuse_tile_kernel<8><<<tgrid, kThreads, tsmem, st>>>(p);
    if (out_weight) {
      DC_LAUNCH_CHECK();
      dim3 zgrid((unsigned)std::min<int64_t>(dc::ceil_div<int64_t>(max_points_per_scene * max_views_per_scene, kThreads * 8), 4096),
                 (unsigned)n_scenes);
      zero_invisible_weights_kernel<<<zgrid, kThreads, 0, st>>>(visible, mask_off, out_weight);
    }
  }
  else {
    pixel_fuse_kernel<<<grid, kThreads, smem, st>>>(p);
    if (normalize) {
      DC_LAUNCH_CHECK();
      DC_CHECK_ARG(sim_kernel == DC_SIM_NONE || out_weight, "dc_pixel_fuse: normalize needs out_weight on this path");
      pixel_normalize_kernel<<<grid, kThreads, 0, st>>>(out_sum, point_off, view_off, mask_off, visible,
                                                        sim_kernel != DC_SIM_NONE ? out_weight : nullptr, dim);
    }
  }
  DC_LAUNCH_CHECK();
  return DC_OK;
}

size_t dc_pixel_fuse_mma_workspace(int64_t total_views, int64_t mask_elems, int patch_h, int patch_w, int dim,
                                   int max_queries_per_scene) {
  if (total_views <= 0 || patch_h <= 0 || patch_w <= 0 || dim <= 0) return 0;
  return mma::layout(total_views, mask_elems, patch_h, patch_w, dim, max_queries_per_scene).bytes;
}

int dc_pixel_fuse_mma(const double* points, const int64_t* point_off, const int64_t* view_off, const double* inv_poses,
                      const double* intrinsics, const int64_t* mask_off, const uint8_t* visible, const void* seg, int seg_dtype,
                      const float* patch_feats, int patch_h, int patch_w, int dim, const float* queries,
                      const int64_t* query_off, int sim_kernel, int norm_feat, int n_scenes, int64_t max_points_per_scene,
                      int max_views_per_scene, int height, int width, const int64_t* rank, float* out_sum, float* out_weight,
                      int normalize, int64_t total_views, int64_t total_points, int64_t mask_elems, int max_queries_per_scene,
                      void* workspace, size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(points && point_off && view_off && inv_poses && intrinsics && mask_off && visible && patch_feats && out_sum && workspace,
               "dc_pixel_fuse_mma: null pointer argument");
  DC_CHECK_ARG(sim_kernel >= DC_SIM_NONE && sim_kernel <= DC_SIM_MEAN, "dc_pixel_fuse_mma: Please set method in [mean, max]");
  DC_CHECK_ARG(sim_kernel == DC_SIM_NONE || (queries && query_off && seg && out_weight),
               "dc_pixel_fuse_mma: similarity needs queries, seg and out_weight");
  DC_CHECK_ARG(dim == 512 || dim == 768 || dim == 1024, "dc_pixel_fuse_mma: dim must be 512, 768 or 1024 (got %d)", dim);
  DC_CHECK_ARG(patch_h > 0 && patch_w > 0 && height > 0 && width > 0 && height < 65536 && width < 65536, "dc_pixel_fuse_mma: bad sizes");
  DC_CHECK_ARG((((uintptr_t)patch_feats | (uintptr_t)out_sum | (uintptr_t)workspace) & 255) == 0 || (((uintptr_t)workspace & 255) == 0 &&
               (((uintptr_t)patch_feats | (uintptr_t)out_sum) & 15) == 0), "dc_pixel_fuse_mma: buffers must be 16-byte (workspace 256-byte) aligned");
  if (n_scenes <= 0 || max_points_per_scene <= 0 || total_points <= 0) return DC_OK;
  DC_CHECK_ARG(n_scenes <= 65535, "dc_pixel_fuse_mma: at most 65535 scenes per call");
  DC_CHECK_ARG(total_points < (1ll << 31) && mask_elems < (1ll << 31), "dc_pixel_fuse_mma: too many points / pairs for one call");
  // regions: the rows one region adds to should fit well inside the 126 MB L2 (~24 MB per region), while every scene keeps
  // enough points per region for full tiles
  int n_regions = 1;
  if (rank) {
    const int64_t row_bytes = (int64_t)dim * 4;
    const int64_t want = dc::ceil_div<int64_t>(max_points_per_scene * n_scenes * row_bytes, (int64_t)24 << 20);
    n_regions = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(want, mma::kMaxRegions), max_points_per_scene / 2048));
  }
  DC_CHECK_ARG((int64_t)n_regions * total_views * (int64_t)(patch_h + 1) * (patch_w + 1) < (1ll << 31), "dc_pixel_fuse_mma: too many views for one call");
  mma::Workspace w = mma::layout(total_views, mask_elems, patch_h, patch_w, dim, sim_kernel != DC_SIM_NONE ? max_queries_per_scene : 0);
  if (workspace_bytes < w.bytes) return dc::fail(DC_ERR_WORKSPACE, "dc_pixel_fuse_mma: workspace %zu < %zu", workspace_bytes, w.bytes);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  cudaStream_t st = dc::as_stream(stream);
  PixParams p{points, point_off, view_off, inv_poses, intrinsics, mask_off, visible, seg, seg_dtype, patch_feats, patch_h,
              patch_w, dim, queries, query_off, sim_kernel, norm_feat, height, width, nullptr, out_sum, out_weight, nullptr, 0, normalize};
  const mma::Footprints fp{patch_h, patch_w, height, width, n_regions, total_views, rank};
  w.n_keys = (int64_t)n_regions * total_views * fp.per_view();
  w.n_scan_blocks = (w.n_keys + mma::kScanBlock - 1) / mma::kScanBlock;
  unsigned* counts = reinterpret_cast<unsigned*>(ws + w.counts);
  unsigned* sums = reinterpret_cast<unsigned*>(ws + w.sums);
  unsigned* total = reinterpret_cast<unsigned*>(ws + w.total);
  uint32_t* pix = reinterpret_cast<uint32_t*>(ws + w.pix);
  int* rec_point = reinterpret_cast<int*>(ws + w.rec_point);
  uint32_t* rec_pix = reinterpret_cast<uint32_t*>(ws + w.rec_pix);
  int* rec_key = reinterpret_cast<int*>(ws + w.rec_key);
  __half* arec = reinterpret_cast<__half*>(ws + w.arec);
  float* norm2 = reinterpret_cast<float*>(ws + w.norm2);
  float* scale = reinterpret_cast<float*>(ws + w.scale);
  __half* plane_hi = reinterpret_cast<__half*>(ws + w.plane_hi);
  __half* plane_lo = reinterpret_cast<__half*>(ws + w.plane_lo);
  DC_CUDA(cudaMemsetAsync(counts, 0, (size_t)w.n_keys * 4, st));
  DC_CUDA(cudaMemsetAsync(out_sum, 0, (size_t)total_points * dim * sizeof(float), st));
  if (out_weight) DC_CUDA(cudaMemsetAsync(out_weight, 0, (size_t)mask_elems * sizeof(float), st));
  if (sim_kernel != DC_SIM_NONE) {
    p.dots = reinterpret_cast<double*>(ws + w.dots);
    p.q_stride = query_stride(max_queries_per_scene);
    if (total_views > 0 && max_queries_per_scene > 0) {
      const int64_t rows = (int64_t)max_views_per_scene * patch_h * patch_w;
      dim3 dgrid(blocks_for((rows + 3) / 4, n_scenes), (unsigned)n_scenes);
      if (dim == 768) patch_query_dots4_kernel<24><<<dgrid, kThreads, 0, st>>>(p);
      else if (dim == 512) patch_query_dots4_kernel<16><<<dgrid, kThreads, 0, st>>>(p);
      else patch_query_dots4_kernel<32><<<dgrid, kThreads, 0, st>>>(p);
      DC_LAUNCH_CHECK();
    }
  }
  // fp16 hi / lo planes of the patch maps (the B operands)
  int rc = dc_row_normalize(const_cast<float*>(patch_feats), DC_F32, total_views * patch_h * patch_w, dim, 0, plane_hi, plane_lo, stream);
  if (rc) return rc;
  // pairs sorted by (view, footprint)
  int64_t chunks = dc::ceil_div<int64_t>(max_points_per_scene, kThreads);
  const int64_t cap = dc::ceil_div<int64_t>((int64_t)dc::sm_count() * 16, n_scenes);
  if (chunks > cap) chunks = cap;
  dim3 pgrid((unsigned)(chunks < 1 ? 1 : chunks), (unsigned)n_scenes);
  mma::pair_count_kernel<<<pgrid, kThreads, 0, st>>>(p, fp, pix, counts);
  mma::scan_sums_kernel<<<(unsigned)w.n_scan_blocks, mma::kScanBlock, 0, st>>>(counts, w.n_keys, sums);
  mma::scan_bases_kernel<<<1, mma::kScanBlock, 0, st>>>(sums, w.n_scan_blocks, total);
  mma::scan_apply_kernel<<<(unsigned)w.n_scan_blocks, mma::kScanBlock, 0, st>>>(counts, w.n_keys, sums);
  mma::pair_scatter_kernel<<<pgrid, kThreads, 0, st>>>(p, fp, pix, counts, rec_point, rec_pix, rec_key, arec);
  DC_LAUNCH_CHECK();
  mma::MmaParams mp{rec_point, rec_key, arec, plane_hi, plane_lo, total, patch_h, patch_w, dim, fp.per_view(), (int)total_views, norm2, scale, out_sum};
  DC_CUDA(cudaFuncSetAttribute(mma::pixel_mma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mma::kSmemBytes));
  DC_CUDA(cudaFuncSetAttribute(mma::pixel_mma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mma::kSmemBytes));
  const int64_t max_tiles = dc::ceil_div<int64_t>(mask_elems, 128);
  const unsigned mgrid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(max_tiles, dc::sm_count()));
  if (norm_feat) {
    DC_CUDA(cudaMemsetAsync(norm2, 0, (size_t)mask_elems * sizeof(float), st));
    mma::pixel_mma_kernel<false><<<mgrid, mma::kThreadsMma, mma::kSmemBytes, st>>>(mp);
  }
  const unsigned wgrid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(dc::ceil_div<int64_t>(mask_elems, kThreads), (int64_t)dc::sm_count() * 16));
  float* den = normalize ? reinterpret_cast<float*>(ws + w.den) : nullptr;
  if (den) DC_CUDA(cudaMemsetAsync(den, 0, (size_t)total_points * sizeof(float), st));
  mma::pair_weight_kernel<<<wgrid, kThreads, 0, st>>>(p, fp, n_scenes, rec_point, rec_pix, rec_key, total, norm2, scale, den);
  if (den) mma::pair_scale_div_kernel<<<wgrid, kThreads, 0, st>>>(rec_point, total, den, scale);
  mma::pixel_mma_kernel<true><<<mgrid, mma::kThreadsMma, mma::kSmemBytes, st>>>(mp);
  if (den) {
    const unsigned ngrid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(dc::ceil_div<int64_t>(total_points, kWarps), (int64_t)dc::sm_count() * 16));
    mma::nan_unseen_rows_kernel<<<ngrid, kThreads, 0, st>>>(den, total_points, dim, out_sum);
  }
  DC_LAUNCH_CHECK();
  return DC_OK;
}

int dc_pixel_normalize(float* sums, const int64_t* point_off, const int64_t* view_off, const int64_t* mask_off,
                       const uint8_t* visible, const float* weight, int n_scenes, int64_t max_points_per_scene, int dim,
                       dc_stream_t stream) {
  DC_CHECK_ARG(sums && point_off && view_off && mask_off && (visible || weight), "dc_pixel_normalize: null pointer argument");
  if (n_scenes <= 0 || max_points_per_scene <= 0) return DC_OK;
  dim3 grid(blocks_for(max_points_per_scene, n_scenes), (unsigned)n_scenes);
  pixel_normalize_kernel<<<grid, kThreads, 0, dc::as_stream(stream)>>>(sums, point_off, view_off, mask_off, visible, weight, dim);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

int dc_view_clip_gather(const double* points, int64_t n_points, const double* inv_poses, const double* intrinsics,
                        const float* patch_feats, int n_views, int patch_h, int patch_w, int dim, int height, int width,
                        float* out, dc_stream_t stream) {
  DC_CHECK_ARG(points && inv_poses && intrinsics && patch_feats && out, "dc_view_clip_gather: null pointer argument");
  DC_CHECK_ARG(patch_h > 0 && patch_w > 0 && dim > 0 && height > 0 && width > 0, "dc_view_clip_gather: bad sizes");
  if (n_points <= 0 || n_views <= 0) return DC_OK;
  DC_CHECK_ARG(n_views <= 65535, "dc_view_clip_gather: at most 65535 views per call");
  dim3 grid(blocks_for(n_points, n_views), (unsigned)n_views);
  const bool vec = dim % 4 == 0 && (((uintptr_t)patch_feats | (uintptr_t)out) & 15) == 0;
  cudaStream_t st = dc::as_stream(stream);
  if (vec) view_clip_gather_kernel<true><<<grid, kThreads, 0, st>>>(points, n_points, inv_poses, intrinsics, patch_feats, patch_h,
                                                                    patch_w, dim, height, width, out);
  else view_clip_gather_kernel<false><<<grid, kThreads, 0, st>>>(points, n_points, inv_poses, intrinsics, patch_feats, patch_h,
                                                                  patch_w, dim, height, width, out);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

}  // extern "C"
