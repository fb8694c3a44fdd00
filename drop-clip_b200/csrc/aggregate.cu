// aggregate_views_blender_new (utils/geometry.py:120-204) for a batch of scenes at several voxel sizes.
//
//   1. compaction: every view of every scene at once. A pixel is labelled when depth < trunc and becomes a point
//      when 0 < depth < trunc (the reference compacts the two by different masks, so a pixel with depth <= 0 shifts
//      the labels against the points). Rows come out scene -> view -> row-major: the world point (Open3D
//      back-projection, Blender flip, fp64 world matrix), the colour / 255 and the label at its own index.
//   2. segmented voxel-down-trace over the (voxel size, scene) segments: min / max bound per scene, the packed voxel
//      key of Open3D's voxel index, an LSD radix sort of (segment, key) that uses only the key bits the segments'
//      grid extents need (counted on the device; passes beyond them return at once), heads, and per voxel the mean
//      point and colour (members summed in ascending point index) and the majority label.
// dc_voxel_down_trace is the one-scene, one-size case. Nothing here waits for the device.
#include <stdlib.h>

#include <algorithm>

#include "geometry_math.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kItems = 16;
constexpr int kTile = kThreads * kItems;  // pixels per compaction chunk, sort elements per radix / head tile
constexpr int kScanThreads = 1024;
constexpr int kScanItems = 8;

unsigned grid_for(int64_t n) {
  int64_t b = dc::ceil_div<int64_t>(n, kThreads);
  const int64_t cap = (int64_t)dc::sm_count() * 16;
  return (unsigned)(b < 1 ? 1 : (b < cap ? b : cap));
}

// exclusive scan of one value per thread over the block; returns the block total in *total
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* total) {
  __shared__ T warp_sums[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  T incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    T w = lane < n_warps ? warp_sums[lane] : T(0);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const T t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    warp_sums[lane] = w;  // inclusive over warps
  }
  __syncthreads();
  const T base = warp > 0 ? warp_sums[warp - 1] : T(0);
  *total = warp_sums[n_warps - 1];
  __syncthreads();  // warp_sums is reused by the next call
  return base + incl - v;
}

// exclusive scan in place of rows of `len` entries (one CTA per row, blockIdx.x = row); totals[row] = row sum
__device__ __forceinline__ void scan_row(uint32_t* __restrict__ data, int64_t len, uint32_t* __restrict__ totals) {
  uint32_t* row = data + (int64_t)blockIdx.x * len;
  uint32_t carry = 0;
  for (int64_t c0 = 0; c0 < len; c0 += (int64_t)kScanThreads * kScanItems) {
    const int64_t b = c0 + (int64_t)threadIdx.x * kScanItems;
    uint32_t v[kScanItems], loc = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
      v[k] = b + k < len ? row[b + k] : 0u;
      loc += v[k];
    }
    uint32_t chunk;
    uint32_t run = carry + block_exclusive_scan<uint32_t>(loc, &chunk);
#pragma unroll
    for (int k = 0; k < kScanItems; ++k)
      if (b + k < len) {
        row[b + k] = run;
        run += v[k];
      }
    carry += chunk;
  }
  if (threadIdx.x == 0) totals[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(kScanThreads) scan_rows_kernel(uint32_t* __restrict__ data, int64_t len, uint32_t* __restrict__ totals) {
  scan_row(data, len, totals);
}

// ------------------------------------------------------------------ 1. compaction
struct Views {
  const int64_t* pix_off;  // [V + 1]
  const int32_t* hw;       // [2V] height, width
  const double* poses;     // [16V] fp64 world matrices
  const double* k4;        // fx, fy, cx, cy
  int n_views;
  int chunks;              // chunks per view (of the largest view)
};

__device__ __forceinline__ void pixel_flags(float d, float trunc, bool& valid, bool& kept) {
  valid = d < trunc;               // seg_ins_2d[depth < trunc]
  kept = !(d >= trunc) && d > 0;   // Open3D: depth >= trunc -> 0, then keeps depth > 0
}

// per (view, chunk): number of labelled and of kept pixels -> counts[0][v * chunks + c], counts[1][...]
__global__ void __launch_bounds__(kThreads) count_pixels_kernel(const float* __restrict__ depths, Views vw, float trunc,
                                                               uint32_t* __restrict__ counts) {
  const int v = blockIdx.x;
  const int64_t p0 = vw.pix_off[v], np = vw.pix_off[v + 1] - p0;
  const int64_t len = (int64_t)vw.n_views * vw.chunks;
  for (int c = blockIdx.y; c < vw.chunks; c += gridDim.y) {
    const int64_t b = (int64_t)c * kTile + (int64_t)threadIdx.x * kItems;
    uint32_t nv = 0, nk = 0;
    for (int k = 0; k < kItems; ++k)
      if (b + k < np) {
        bool valid, kept;
        pixel_flags(depths[p0 + b + k], trunc, valid, kept);
        nv += valid;
        nk += kept;
      }
    uint32_t tv, tk;
    block_exclusive_scan<uint32_t>(nv, &tv);
    block_exclusive_scan<uint32_t>(nk, &tk);
    if (threadIdx.x == 0) {
      counts[(int64_t)v * vw.chunks + c] = tv;
      counts[len + (int64_t)v * vw.chunks + c] = tk;
    }
  }
}

// label_off[s] / point_off[s] = first label / point of scene s (from the scanned chunk counts)
__global__ void scene_offsets_kernel(const uint32_t* __restrict__ scanned, const uint32_t* __restrict__ totals, int64_t len,
                                     const int32_t* __restrict__ scene_view_off, int n_scenes, int chunks,
                                     int64_t* __restrict__ label_off, int64_t* __restrict__ point_off) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s > n_scenes) return;
  const int64_t i = (int64_t)scene_view_off[s] * chunks;
  label_off[s] = i < len ? scanned[i] : totals[0];
  point_off[s] = i < len ? scanned[len + i] : totals[1];
}

template <typename SegT, typename RgbT>
__global__ void __launch_bounds__(kThreads) compact_pixels_kernel(const float* __restrict__ depths, const SegT* __restrict__ segs,
                                                                 const RgbT* __restrict__ rgbs, Views vw, float trunc,
                                                                 const uint32_t* __restrict__ scanned, double* __restrict__ points,
                                                                 double* __restrict__ colors, long long* __restrict__ labels) {
  const int v = blockIdx.x;
  const int64_t p0 = vw.pix_off[v], np = vw.pix_off[v + 1] - p0;
  const int width = vw.hw[2 * v + 1];
  const int64_t len = (int64_t)vw.n_views * vw.chunks;
  const double fx = vw.k4[0], fy = vw.k4[1], cx = vw.k4[2], cy = vw.k4[3];
  const double* pose = vw.poses + 16 * (int64_t)v;
  for (int c = blockIdx.y; c < vw.chunks; c += gridDim.y) {
    const int64_t b = (int64_t)c * kTile + (int64_t)threadIdx.x * kItems;
    uint32_t nv = 0, nk = 0;
    for (int k = 0; k < kItems; ++k)
      if (b + k < np) {
        bool valid, kept;
        pixel_flags(depths[p0 + b + k], trunc, valid, kept);
        nv += valid;
        nk += kept;
      }
    uint32_t tv, tk;
    int64_t li = scanned[(int64_t)v * vw.chunks + c] + block_exclusive_scan<uint32_t>(nv, &tv);
    int64_t pi = scanned[len + (int64_t)v * vw.chunks + c] + block_exclusive_scan<uint32_t>(nk, &tk);
    for (int k = 0; k < kItems; ++k) {
      const int64_t pix = b + k;
      if (pix >= np) break;
      const float d = depths[p0 + pix];
      bool valid, kept;
      pixel_flags(d, trunc, valid, kept);
      if (valid) labels[li++] = (long long)segs[p0 + pix];
      if (kept) {
        const int y = (int)(pix / width), x = (int)(pix - (int64_t)y * width);
        double w[3];
        dc::backproject_pixel(x, y, (double)d, fx, fy, cx, cy, 3, 1, pose, w);  // Open3D rounding, * [1, -1, -1], world
        const RgbT* rgb = rgbs + 3 * (p0 + pix);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          points[3 * pi + a] = w[a];
          colors[3 * pi + a] = __ddiv_rn((double)rgb[a], 255.0);  // numpy's `/ 255.0`
        }
        ++pi;
      }
    }
  }
}

// ------------------------------------------------------------------ 2. segmented voxel-down-trace
// Sort element e stands for point p = e - u * stride at voxel size u. Points [point_off[S], stride) pad every size's
// range; they form an extra segment after the scenes of that size, so segment (u, s) keeps the positions
// [u * stride + point_off[s], u * stride + point_off[s + 1]) through the sort.
struct Segs {
  const double* pts;
  const double* cols;         // may be null
  const long long* labels;    // may be null; point p of scene s votes with labels[label_off[s] + p - point_off[s]]
  const int64_t* point_off;   // [S + 1]
  const int64_t* label_off;   // [S + 1]
  const double* voxel;        // [U]
  int n_scenes, n_sizes;
  int64_t stride;
  int64_t n_elems;            // U * stride
  int g_bits;                 // bits of the virtual segment id u * (S + 1) + s
};

struct SortWs {
  unsigned long long* keys[2];
  int* vals[2];
  int* vstart;             // sorted position of each voxel's first member
  uint32_t* hist;          // [256][n_tiles]
  uint32_t* tile_heads;    // [n_tiles]
  uint32_t* totals;        // [256]
  unsigned long long* mn;  // [3S] ordered images
  unsigned long long* mx;  // [3S]
  int* seg_bits;           // [U * S][3]
  int* lbits;              // max local key bits over the segments
  int64_t n_tiles;
};

__device__ __forceinline__ int scene_of(int64_t p, const int64_t* __restrict__ point_off, int n_scenes) {
  if (p >= point_off[n_scenes]) return n_scenes;  // padding
  int lo = 0, hi = n_scenes - 1;                  // largest s with point_off[s] <= p
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (point_off[mid] <= p) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(kThreads) bounds_kernel(Segs sg, unsigned long long* __restrict__ mn, unsigned long long* __restrict__ mx) {
  const int s = blockIdx.y;
  const int64_t a = sg.point_off[s], b = sg.point_off[s + 1];
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t i = a + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < b; i += (int64_t)gridDim.x * blockDim.x)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      lo[k] = fmin(lo[k], sg.pts[3 * i + k]);
      hi[k] = fmax(hi[k], sg.pts[3 * i + k]);
    }
#pragma unroll
  for (int k = 0; k < 3; ++k)
    for (int o = 16; o > 0; o >>= 1) {
      lo[k] = fmin(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o));
      hi[k] = fmax(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o));
    }
  if ((threadIdx.x & 31) == 0)
    for (int k = 0; k < 3; ++k) {
      atomicMin(mn + 3 * s + k, dc::double_to_ordered(lo[k]));
      atomicMax(mx + 3 * s + k, dc::double_to_ordered(hi[k]));
    }
}

__device__ __forceinline__ double voxel_bound(const unsigned long long* mn, int s, int k, double voxel) {
  return dc::ordered_to_double(mn[3 * s + k]) - voxel * 0.5;
}

// bits of each axis of segment (u, s): enough for the voxel index of the scene's max bound (the index is monotone in
// the coordinate); 21 when that index is out of range
__global__ void segment_bits_kernel(Segs sg, const unsigned long long* __restrict__ mn, const unsigned long long* __restrict__ mx,
                                    int* __restrict__ seg_bits, int* __restrict__ lbits) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= sg.n_sizes * sg.n_scenes) return;
  const int u = g / sg.n_scenes, s = g - u * sg.n_scenes;
  const double voxel = sg.voxel[u];
  int total = 0;
  for (int k = 0; k < 3; ++k) {
    const double f = dc::voxel_coord(dc::ordered_to_double(mx[3 * s + k]), voxel_bound(mn, s, k, voxel), voxel);
    int bits = 21;
    if (dc::voxel_coord_ok(f)) {
      const unsigned long long top = (unsigned long long)f;
      bits = top == 0 ? 0 : 64 - __clzll((long long)top);
    }
    seg_bits[3 * g + k] = bits;
    total += bits;
  }
  atomicMax(lbits, total);
}

__global__ void __launch_bounds__(kThreads) voxel_keys_kernel(Segs sg, const unsigned long long* __restrict__ mn,
                                                             const int* __restrict__ seg_bits, unsigned long long* __restrict__ keys,
                                                             int* __restrict__ vals) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < sg.n_elems; e += (int64_t)gridDim.x * blockDim.x) {
    const int u = (int)(e / sg.stride);
    const int64_t p = e - u * sg.stride;
    const int s = scene_of(p, sg.point_off, sg.n_scenes);
    unsigned long long key = 0;
    if (s < sg.n_scenes) {
      const double voxel = sg.voxel[u];
      const double fx = dc::voxel_coord(sg.pts[3 * p], voxel_bound(mn, s, 0, voxel), voxel);
      const double fy = dc::voxel_coord(sg.pts[3 * p + 1], voxel_bound(mn, s, 1, voxel), voxel);
      const double fz = dc::voxel_coord(sg.pts[3 * p + 2], voxel_bound(mn, s, 2, voxel), voxel);
      if (dc::voxel_coord_ok(fx) && dc::voxel_coord_ok(fy) && dc::voxel_coord_ok(fz)) {
        const int* bits = seg_bits + 3 * (u * sg.n_scenes + s);
        key = ((unsigned long long)fx << (bits[1] + bits[2])) | ((unsigned long long)fy << bits[2]) | (unsigned long long)fz;
      }
    }
    keys[e] = key;
    vals[e] = (int)e;
  }
}

__device__ __forceinline__ unsigned radix_digit(unsigned long long key, int e, const Segs& sg, int lbits, int shift) {
  unsigned __int128 k = key;
  if (shift + 8 > lbits) {  // the digit reaches the segment id
    const int u = (int)(e / sg.stride);
    const int s = scene_of(e - u * sg.stride, sg.point_off, sg.n_scenes);
    k |= (unsigned __int128)((unsigned long long)u * (sg.n_scenes + 1) + s) << lbits;
  }
  return (unsigned)(k >> shift) & 255u;
}

__global__ void __launch_bounds__(kThreads) radix_hist_kernel(Segs sg, const unsigned long long* __restrict__ keys,
                                                             const int* __restrict__ vals, const int* __restrict__ lbits_p, int shift,
                                                             uint32_t* __restrict__ hist, int64_t n_tiles) {
  const int lbits = *lbits_p;
  if (shift >= lbits + sg.g_bits) return;
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * kTile;
  for (int k = 0; k < kItems; ++k) {
    const int64_t i = base + k * kThreads + threadIdx.x;
    if (i < sg.n_elems) atomicAdd(&h[radix_digit(keys[i], vals[i], sg, lbits, shift)], 1u);
  }
  __syncthreads();
  hist[(int64_t)threadIdx.x * n_tiles + blockIdx.x] = h[threadIdx.x];
}

__global__ void __launch_bounds__(kScanThreads) radix_scan_kernel(const int* __restrict__ lbits_p, int g_bits, int shift,
                                                                 uint32_t* __restrict__ hist, int64_t n_tiles, uint32_t* __restrict__ totals) {
  if (shift >= *lbits_p + g_bits) return;
  scan_row(hist, n_tiles, totals);
}

// stable scatter of one tile: 16 rounds of 256 consecutive elements; an element's rank = elements of its digit in
// earlier rounds + in earlier warps of its round + in earlier lanes of its warp
__global__ void __launch_bounds__(kThreads) radix_scatter_kernel(Segs sg, const unsigned long long* __restrict__ keys_in,
                                                                const int* __restrict__ vals_in, const int* __restrict__ lbits_p,
                                                                int shift, const uint32_t* __restrict__ hist, int64_t n_tiles,
                                                                const uint32_t* __restrict__ totals,
                                                                unsigned long long* __restrict__ keys_out, int* __restrict__ vals_out) {
  const int lbits = *lbits_p;
  if (shift >= lbits + sg.g_bits) return;
  constexpr int kWarps = kThreads / 32;
  __shared__ uint32_t run[256];
  __shared__ uint32_t wcnt[kWarps][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t dummy;
  const uint32_t digit_base = block_exclusive_scan<uint32_t>(totals[threadIdx.x], &dummy);
  run[threadIdx.x] = digit_base + hist[(int64_t)threadIdx.x * n_tiles + blockIdx.x];
#pragma unroll
  for (int w = 0; w < kWarps; ++w) wcnt[w][threadIdx.x] = 0;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * kTile;
  const unsigned lt = (1u << lane) - 1u;
  for (int r = 0; r < kItems; ++r) {
    const int64_t i = base + r * kThreads + threadIdx.x;
    const bool live = i < sg.n_elems;
    unsigned long long key = 0;
    int val = 0;
    unsigned d = 256;
    if (live) {
      key = keys_in[i];
      val = vals_in[i];
      d = radix_digit(key, val, sg, lbits, shift);
    }
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    if (live && lane == __ffs(peers) - 1) wcnt[warp][d] = __popc(peers);
    __syncthreads();
    if (live) {
      uint32_t pos = run[d] + __popc(peers & lt);
      for (int w = 0; w < warp; ++w) pos += wcnt[w][d];
      keys_out[pos] = key;
      vals_out[pos] = val;
    }
    __syncthreads();
    uint32_t add = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      add += wcnt[w][threadIdx.x];
      wcnt[w][threadIdx.x] = 0;
    }
    run[threadIdx.x] += add;
    __syncthreads();
  }
}

__device__ __forceinline__ int sorted_buffer(const int* lbits_p, int g_bits) { return (((*lbits_p + g_bits) + 7) / 8) & 1; }

// position i is a voxel's first member: it lies in a scene's range and starts that range or a new key
__device__ __forceinline__ bool is_head(int64_t i, const Segs& sg, const unsigned long long* keys, bool* seg_start, int* g) {
  const int u = (int)(i / sg.stride);
  const int64_t p = i - u * sg.stride;
  const int s = scene_of(p, sg.point_off, sg.n_scenes);
  *seg_start = false;
  if (s >= sg.n_scenes) return false;
  *g = u * sg.n_scenes + s;
  *seg_start = p == sg.point_off[s];
  return *seg_start || keys[i] != keys[i - 1];
}

__global__ void __launch_bounds__(kThreads) count_heads_kernel(Segs sg, const unsigned long long* __restrict__ k0, const unsigned long long* __restrict__ k1,
                                                              const int* __restrict__ lbits_p, uint32_t* __restrict__ tile_heads) {
  const unsigned long long* keys = sorted_buffer(lbits_p, sg.g_bits) ? k1 : k0;
  const int64_t b = (int64_t)blockIdx.x * kTile + (int64_t)threadIdx.x * kItems;
  uint32_t n = 0;
  for (int k = 0; k < kItems; ++k) {
    bool st;
    int g;
    if (b + k < sg.n_elems) n += is_head(b + k, sg, keys, &st, &g);
  }
  uint32_t total;
  block_exclusive_scan<uint32_t>(n, &total);
  if (threadIdx.x == 0) tile_heads[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kThreads) write_heads_kernel(Segs sg, const unsigned long long* __restrict__ k0,
                                                              const unsigned long long* __restrict__ k1, const int* __restrict__ lbits_p,
                                                              const uint32_t* __restrict__ tile_off, int* __restrict__ vstart,
                                                              int64_t* __restrict__ vox_off) {
  const unsigned long long* keys = sorted_buffer(lbits_p, sg.g_bits) ? k1 : k0;
  const int64_t b = (int64_t)blockIdx.x * kTile + (int64_t)threadIdx.x * kItems;
  uint32_t n = 0;
  for (int k = 0; k < kItems; ++k) {
    bool st;
    int g;
    if (b + k < sg.n_elems) n += is_head(b + k, sg, keys, &st, &g);
  }
  uint32_t total;
  int64_t vid = tile_off[blockIdx.x] + block_exclusive_scan<uint32_t>(n, &total);
  for (int k = 0; k < kItems && b + k < sg.n_elems; ++k) {
    bool st;
    int g;
    if (!is_head(b + k, sg, keys, &st, &g)) continue;
    if (st) vox_off[g] = vid;
    vstart[vid++] = (int)(b + k);
  }
}

// vox_off[U * S] = voxel total; an empty segment starts where the next one does
__global__ void finish_offsets_kernel(int64_t* __restrict__ vox_off, int n_segs, const uint32_t* __restrict__ total,
                                      int64_t* __restrict__ n_voxels) {
  int64_t next = total ? *total : 0;
  vox_off[n_segs] = next;
  for (int g = n_segs - 1; g >= 0; --g) {
    if (vox_off[g] < 0) vox_off[g] = next;
    next = vox_off[g];
  }
  if (n_voxels) *n_voxels = vox_off[n_segs];
}

// one thread per voxel: members summed in ascending point index (the sort is stable) and divided by their count,
// Open3D's AccumulatedPointForTrace; the label is Counter(labels).most_common()[0][0] - the most frequent, ties to
// the one met first. Up to kSlots distinct labels are counted in one pass (a scene of MV-TOD has at most 22: 21
// objects and the background; with 8 slots, voxels that 73 views see spent seconds in the quadratic scan that
// more distinct labels fall back to).
__global__ void __launch_bounds__(kThreads) voxel_trace_kernel(Segs sg, const int* __restrict__ v0, const int* __restrict__ v1,
                                                              const int* __restrict__ lbits_p, const int* __restrict__ vstart,
                                                              const int64_t* __restrict__ vox_off, double* __restrict__ out_pts,
                                                              double* __restrict__ out_cols, long long* __restrict__ out_labels,
                                                              int64_t* __restrict__ first_index, int64_t* __restrict__ counts) {
  constexpr int kSlots = 32;
  const int* order = sorted_buffer(lbits_p, sg.g_bits) ? v1 : v0;
  const int64_t n_vox = vox_off[(int64_t)sg.n_sizes * sg.n_scenes];
  for (int64_t vid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; vid < n_vox; vid += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = vstart[vid];
    const int u = (int)(order[i] / sg.stride);
    const int64_t ubase = u * sg.stride;
    const int s = scene_of(order[i] - ubase, sg.point_off, sg.n_scenes);
    int64_t end = ubase + sg.point_off[s + 1];
    if (vid + 1 < n_vox && vstart[vid + 1] < end) end = vstart[vid + 1];
    const long long* labs = sg.labels ? sg.labels + (sg.label_off[s] - sg.point_off[s]) : nullptr;
    double sx = 0, sy = 0, sz = 0, cr = 0, cg = 0, cb = 0;
    long long lab[kSlots];
    int cnt[kSlots];
    int used = 0;
    bool overflow = false;
    for (int64_t k = i; k < end; ++k) {
      const int64_t j = order[k] - ubase;
      sx += sg.pts[3 * j];
      sy += sg.pts[3 * j + 1];
      sz += sg.pts[3 * j + 2];
      if (sg.cols) {
        cr += sg.cols[3 * j];
        cg += sg.cols[3 * j + 1];
        cb += sg.cols[3 * j + 2];
      }
      if (labs && !overflow) {
        const long long l = labs[j];
        int q = 0;
        while (q < used && lab[q] != l) ++q;
        if (q < used) ++cnt[q];
        else if (used < kSlots) { lab[used] = l; cnt[used] = 1; ++used; }
        else overflow = true;
      }
    }
    const int64_t c = end - i;
    const double dc_ = (double)c;
    out_pts[3 * vid] = sx / dc_;
    out_pts[3 * vid + 1] = sy / dc_;
    out_pts[3 * vid + 2] = sz / dc_;
    if (sg.cols) {
      out_cols[3 * vid] = cr / dc_;
      out_cols[3 * vid + 1] = cg / dc_;
      out_cols[3 * vid + 2] = cb / dc_;
    }
    if (first_index) first_index[vid] = order[i] - ubase;
    if (counts) counts[vid] = c;
    if (labs) {
      long long best = 0;
      int64_t best_n = -1;
      if (!overflow) {
        for (int q = 0; q < used; ++q)  // slots are in first-seen order: strict > keeps the earliest on ties
          if (cnt[q] > best_n) { best_n = cnt[q]; best = lab[q]; }
      } else {
        for (int64_t a = i; a < end; ++a) {
          const long long l = labs[order[a] - ubase];
          bool seen = false;
          for (int64_t b = i; b < a && !seen; ++b) seen = labs[order[b] - ubase] == l;
          if (seen) continue;
          int64_t m = 0;
          for (int64_t b = a; b < end; ++b) m += labs[order[b] - ubase] == l;
          if (m > best_n) { best_n = m; best = l; }
        }
      }
      out_labels[vid] = best;
    }
  }
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Carve {
  size_t off = 0;
  uint8_t* base;
  explicit Carve(void* ws) : base(reinterpret_cast<uint8_t*>(ws)) {}
  template <typename T>
  T* take(size_t n) {
    const size_t o = off;
    off = align_up(off + n * sizeof(T), 256);
    return base ? reinterpret_cast<T*>(base + o) : nullptr;
  }
};

SortWs carve_sort(Carve& c, int n_scenes, int n_sizes, int64_t n_elems) {
  SortWs w{};
  w.n_tiles = dc::ceil_div<int64_t>(n_elems, kTile);
  const size_t ne = (size_t)(n_elems > 0 ? n_elems : 1);
  w.keys[0] = c.take<unsigned long long>(ne);
  w.keys[1] = c.take<unsigned long long>(ne);
  w.vals[0] = c.take<int>(ne);
  w.vals[1] = c.take<int>(ne);
  w.vstart = c.take<int>(ne);
  w.hist = c.take<uint32_t>(256 * (size_t)(w.n_tiles > 0 ? w.n_tiles : 1));
  w.tile_heads = c.take<uint32_t>((size_t)(w.n_tiles > 0 ? w.n_tiles : 1));
  w.totals = c.take<uint32_t>(256);
  w.mn = c.take<unsigned long long>(3 * (size_t)n_scenes);
  w.mx = c.take<unsigned long long>(3 * (size_t)n_scenes);
  w.seg_bits = c.take<int>(3 * (size_t)n_scenes * n_sizes);
  w.lbits = c.take<int>(1);
  return w;
}

int bits_for(int64_t n) {  // bits of n - 1
  int b = 0;
  while (b < 62 && (1ll << b) < n) ++b;
  return b;
}

// the segmented trace on stream st; vox_off[U * S + 1] (device) receives the voxel layout
int segmented_trace(Segs sg, SortWs& w, int64_t* vox_off, double* out_pts, double* out_cols, long long* out_labels,
                    int64_t* first_index, int64_t* counts, int64_t* n_voxels, cudaStream_t st) {
  const int n_segs = sg.n_scenes * sg.n_sizes;
  DC_CUDA(cudaMemsetAsync(vox_off, 0xFF, sizeof(int64_t) * (size_t)n_segs, st));
  if (sg.n_elems == 0) {
    finish_offsets_kernel<<<1, 1, 0, st>>>(vox_off, n_segs, nullptr, n_voxels);
    DC_LAUNCH_CHECK();
    return DC_OK;
  }
  DC_CUDA(cudaMemsetAsync(w.mn, 0xFF, sizeof(unsigned long long) * 3 * (size_t)sg.n_scenes, st));
  DC_CUDA(cudaMemsetAsync(w.mx, 0, sizeof(unsigned long long) * 3 * (size_t)sg.n_scenes, st));
  DC_CUDA(cudaMemsetAsync(w.lbits, 0, sizeof(int), st));
  const unsigned bx = (unsigned)dc::ceil_div<int64_t>((int64_t)dc::sm_count() * 8, sg.n_scenes);
  bounds_kernel<<<dim3(bx, (unsigned)sg.n_scenes), kThreads, 0, st>>>(sg, w.mn, w.mx);
  segment_bits_kernel<<<(unsigned)dc::ceil_div(n_segs, 128), 128, 0, st>>>(sg, w.mn, w.mx, w.seg_bits, w.lbits);
  voxel_keys_kernel<<<grid_for(sg.n_elems), kThreads, 0, st>>>(sg, w.mn, w.seg_bits, w.keys[0], w.vals[0]);
  const unsigned tiles = (unsigned)w.n_tiles;
  for (int pass = 0; pass * 8 < 63 + sg.g_bits; ++pass) {  // passes past the device's key width return at once
    const int in = pass & 1, shift = pass * 8;
    radix_hist_kernel<<<tiles, kThreads, 0, st>>>(sg, w.keys[in], w.vals[in], w.lbits, shift, w.hist, w.n_tiles);
    radix_scan_kernel<<<256, kScanThreads, 0, st>>>(w.lbits, sg.g_bits, shift, w.hist, w.n_tiles, w.totals);
    radix_scatter_kernel<<<tiles, kThreads, 0, st>>>(sg, w.keys[in], w.vals[in], w.lbits, shift, w.hist, w.n_tiles, w.totals,
                                                     w.keys[in ^ 1], w.vals[in ^ 1]);
  }
  count_heads_kernel<<<tiles, kThreads, 0, st>>>(sg, w.keys[0], w.keys[1], w.lbits, w.tile_heads);
  scan_rows_kernel<<<1, kScanThreads, 0, st>>>(w.tile_heads, w.n_tiles, w.totals);
  write_heads_kernel<<<tiles, kThreads, 0, st>>>(sg, w.keys[0], w.keys[1], w.lbits, w.tile_heads, w.vstart, vox_off);
  finish_offsets_kernel<<<1, 1, 0, st>>>(vox_off, n_segs, w.totals, n_voxels);
  voxel_trace_kernel<<<grid_for(sg.n_elems), kThreads, 0, st>>>(sg, w.vals[0], w.vals[1], w.lbits, w.vstart, vox_off, out_pts,
                                                                out_cols, out_labels, first_index, counts);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

// host tables of dc_aggregate_views, staged with one copy
struct Tables {
  int64_t* pix_off;
  int32_t* hw;
  int32_t* scene_view_off;
  double* poses;
  double* k4;
  double* voxel;
  int64_t* pad_off;  // [2] for the one-scene trace
};

Tables carve_tables(Carve& c, int n_scenes, int n_views, int n_sizes) {
  Tables t{};
  t.pix_off = c.take<int64_t>((size_t)n_views + 1);
  t.hw = c.take<int32_t>(2 * (size_t)n_views);
  t.scene_view_off = c.take<int32_t>((size_t)n_scenes + 1);
  t.poses = c.take<double>(16 * (size_t)n_views);
  t.k4 = c.take<double>(4);
  t.voxel = c.take<double>((size_t)n_sizes);
  t.pad_off = c.take<int64_t>(2);
  return t;
}

int max_chunks(const int64_t* pix_off, int n_views) {
  int64_t m = 1;
  for (int v = 0; v < n_views; ++v) m = std::max<int64_t>(m, dc::ceil_div<int64_t>(pix_off[v + 1] - pix_off[v], kTile));
  return (int)m;
}

}  // namespace

extern "C" {

size_t dc_aggregate_views_workspace(int n_scenes, int n_views, int64_t n_pixels, int n_sizes) {
  if (n_scenes < 0 || n_views < 0 || n_pixels < 0 || n_sizes < 0) return 0;
  Carve c(nullptr);
  carve_tables(c, n_scenes, n_views, n_sizes);
  c.take<uint32_t>(2 * ((size_t)n_views * dc::ceil_div<int64_t>(n_pixels > 0 ? n_pixels : 1, kTile) + 1));
  c.take<uint32_t>(2);
  carve_sort(c, n_scenes, n_sizes, (int64_t)n_sizes * n_pixels);
  return c.off;
}

int dc_aggregate_views(const float* depths, const void* segs, int seg_dtype, const void* rgbs, int rgb_dtype, const int64_t* view_pix_off,
                       const int32_t* view_hw, const int32_t* scene_view_off, const double* poses, const double* fxfycxcy,
                       float depth_trunc, const double* voxel_sizes, int n_scenes, int n_views, int n_sizes, double* points,
                       double* colors, int64_t* labels, int64_t* point_off, int64_t* label_off, double* vox_points,
                       double* vox_colors, int64_t* vox_labels, int64_t* vox_off, void* workspace, size_t workspace_bytes,
                       dc_stream_t stream) {
  DC_CHECK_ARG(view_pix_off && view_hw && scene_view_off && fxfycxcy && point_off && label_off && workspace,
               "dc_aggregate_views: null pointer argument");
  DC_CHECK_ARG(n_scenes >= 1 && n_scenes <= 65535 && n_views >= 0 && n_sizes >= 0, "dc_aggregate_views: bad counts");
  DC_CHECK_ARG(seg_dtype == DC_U8 || seg_dtype == DC_I64, "dc_aggregate_views: instance maps must be uint8 or int64");
  DC_CHECK_ARG(rgb_dtype == DC_U8 || rgb_dtype == DC_F64, "dc_aggregate_views: colours must be uint8 or fp64");
  DC_CHECK_ARG(scene_view_off[0] == 0 && scene_view_off[n_scenes] == n_views && view_pix_off[0] == 0,
               "dc_aggregate_views: bad scene / view offsets");
  for (int s = 0; s < n_scenes; ++s)
    DC_CHECK_ARG(scene_view_off[s + 1] >= scene_view_off[s], "dc_aggregate_views: scene view offsets must not decrease");
  for (int v = 0; v < n_views; ++v)
    DC_CHECK_ARG(view_hw[2 * v] >= 0 && view_hw[2 * v + 1] >= 0 &&
                     view_pix_off[v + 1] - view_pix_off[v] == (int64_t)view_hw[2 * v] * view_hw[2 * v + 1],
                 "dc_aggregate_views: view %d: pixel offsets do not match its size", v);
  const int64_t n_pixels = view_pix_off[n_views];
  DC_CHECK_ARG(n_pixels < (1ll << 31) && (int64_t)n_sizes * n_pixels < (1ll << 31),
               "dc_aggregate_views: pixels x voxel sizes must stay below 2^31");
  if (n_pixels > 0) DC_CHECK_ARG(depths && segs && rgbs && points && colors && labels, "dc_aggregate_views: null pointer argument");
  if (n_sizes > 0) {
    DC_CHECK_ARG(voxel_sizes && vox_off && vox_points && vox_colors && vox_labels, "dc_aggregate_views: null pointer argument");
    DC_CHECK_ARG(depth_trunc == depth_trunc, "dc_aggregate_views: depth_trunc is NaN (no pixel would be labelled)");
    for (int u = 0; u < n_sizes; ++u) DC_CHECK_ARG(voxel_sizes[u] > 0.0, "dc_aggregate_views: voxel_size must be positive");
  }
  const size_t need = dc_aggregate_views_workspace(n_scenes, n_views, n_pixels, n_sizes);
  if (workspace_bytes < need) return dc::fail(DC_ERR_WORKSPACE, "dc_aggregate_views: workspace %zu < %zu", workspace_bytes, need);
  cudaStream_t st = dc::as_stream(stream);

  Carve c(workspace);
  Tables t = carve_tables(c, n_scenes, n_views, n_sizes);
  const size_t tables_bytes = c.off;
  {  // one host -> device copy of every table
    uint8_t* host = static_cast<uint8_t*>(malloc(tables_bytes));
    if (!host) return dc::fail(DC_ERR_INVALID, "dc_aggregate_views: out of host memory");
    uint8_t* b = static_cast<uint8_t*>(workspace);
    auto put = [&](void* dev, const void* src, size_t bytes) {
      if (bytes) memcpy(host + (static_cast<uint8_t*>(dev) - b), src, bytes);
    };
    put(t.pix_off, view_pix_off, sizeof(int64_t) * ((size_t)n_views + 1));
    put(t.hw, view_hw, sizeof(int32_t) * 2 * (size_t)n_views);
    put(t.scene_view_off, scene_view_off, sizeof(int32_t) * ((size_t)n_scenes + 1));
    if (n_views) put(t.poses, poses, sizeof(double) * 16 * (size_t)n_views);
    put(t.k4, fxfycxcy, sizeof(double) * 4);
    if (n_sizes) put(t.voxel, voxel_sizes, sizeof(double) * (size_t)n_sizes);
    const cudaError_t e = cudaMemcpyAsync(workspace, host, tables_bytes, cudaMemcpyHostToDevice, st);
    free(host);  // a pageable source is staged before the call returns
    DC_CUDA(e);
  }
  const int chunks = max_chunks(view_pix_off, n_views);
  const int64_t len = (int64_t)n_views * chunks;
  uint32_t* counts = c.take<uint32_t>(2 * ((size_t)n_views * dc::ceil_div<int64_t>(n_pixels > 0 ? n_pixels : 1, kTile) + 1));
  uint32_t* totals = c.take<uint32_t>(2);
  SortWs w = carve_sort(c, n_scenes, n_sizes, (int64_t)n_sizes * n_pixels);

  Views vw{t.pix_off, t.hw, t.poses, t.k4, n_views, chunks};
  if (n_views > 0) {
    const dim3 grid((unsigned)n_views, (unsigned)std::min(chunks, 65535));
    count_pixels_kernel<<<grid, kThreads, 0, st>>>(depths, vw, depth_trunc, counts);
    scan_rows_kernel<<<2, kScanThreads, 0, st>>>(counts, len, totals);
  } else {
    DC_CUDA(cudaMemsetAsync(totals, 0, 2 * sizeof(uint32_t), st));
  }
  scene_offsets_kernel<<<(unsigned)dc::ceil_div(n_scenes + 1, 128), 128, 0, st>>>(counts, totals, len, t.scene_view_off, n_scenes,
                                                                                  chunks, label_off, point_off);
  if (n_views > 0) {
    const dim3 grid((unsigned)n_views, (unsigned)std::min(chunks, 65535));
    long long* lab = reinterpret_cast<long long*>(labels);
    if (seg_dtype == DC_U8 && rgb_dtype == DC_U8)
      compact_pixels_kernel<uint8_t, uint8_t><<<grid, kThreads, 0, st>>>(depths, (const uint8_t*)segs, (const uint8_t*)rgbs, vw,
                                                                         depth_trunc, counts, points, colors, lab);
    else if (seg_dtype == DC_U8)
      compact_pixels_kernel<uint8_t, double><<<grid, kThreads, 0, st>>>(depths, (const uint8_t*)segs, (const double*)rgbs, vw,
                                                                        depth_trunc, counts, points, colors, lab);
    else if (rgb_dtype == DC_U8)
      compact_pixels_kernel<int64_t, uint8_t><<<grid, kThreads, 0, st>>>(depths, (const int64_t*)segs, (const uint8_t*)rgbs, vw,
                                                                         depth_trunc, counts, points, colors, lab);
    else
      compact_pixels_kernel<int64_t, double><<<grid, kThreads, 0, st>>>(depths, (const int64_t*)segs, (const double*)rgbs, vw,
                                                                        depth_trunc, counts, points, colors, lab);
  }
  DC_LAUNCH_CHECK();
  if (n_sizes == 0) return DC_OK;
  Segs sg{points, colors, reinterpret_cast<const long long*>(labels), point_off, label_off, t.voxel, n_scenes, n_sizes,
          n_pixels, (int64_t)n_sizes * n_pixels, bits_for((int64_t)n_sizes * (n_scenes + 1))};
  return segmented_trace(sg, w, vox_off, vox_points, vox_colors, reinterpret_cast<long long*>(vox_labels), nullptr, nullptr,
                         nullptr, st);
}

size_t dc_voxel_down_trace_workspace(int64_t n) {
  Carve c(nullptr);
  carve_tables(c, 1, 0, 1);
  c.take<int64_t>(2);
  carve_sort(c, 1, 1, n > 0 ? n : 0);
  return c.off;
}

int dc_voxel_down_trace(const double* points, const double* colors, const int64_t* labels, int64_t n, double voxel_size,
                        double* out_points, double* out_colors, int64_t* out_labels, int64_t* first_index, int64_t* counts,
                        int64_t* n_voxels, void* workspace, size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(points && out_points && n_voxels && workspace, "dc_voxel_down_trace: null pointer argument");
  DC_CHECK_ARG((!colors || out_colors) && (!labels || out_labels), "dc_voxel_down_trace: output missing for an optional input");
  DC_CHECK_ARG(voxel_size > 0.0, "dc_voxel_down_trace: voxel_size must be positive");
  DC_CHECK_ARG(n >= 0 && n < (1ll << 31), "dc_voxel_down_trace: too many points");
  const size_t need = dc_voxel_down_trace_workspace(n);
  if (workspace_bytes < need) return dc::fail(DC_ERR_WORKSPACE, "dc_voxel_down_trace: workspace %zu < %zu", workspace_bytes, need);
  cudaStream_t st = dc::as_stream(stream);
  Carve c(workspace);
  Tables t = carve_tables(c, 1, 0, 1);
  int64_t* vox_off = c.take<int64_t>(2);
  SortWs w = carve_sort(c, 1, 1, n);
  struct {
    int64_t off[2];
    double voxel;
  } host = {{0, n}, voxel_size};
  DC_CUDA(cudaMemcpyAsync(t.pad_off, host.off, sizeof(host.off), cudaMemcpyHostToDevice, st));
  DC_CUDA(cudaMemcpyAsync(t.voxel, &host.voxel, sizeof(double), cudaMemcpyHostToDevice, st));
  Segs sg{points, colors, reinterpret_cast<const long long*>(labels), t.pad_off, t.pad_off, t.voxel, 1, 1, n, n, bits_for(2)};
  return segmented_trace(sg, w, vox_off, out_points, out_colors, reinterpret_cast<long long*>(out_labels), first_index, counts,
                         n_voxels, st);
}

}  // extern "C"
