// Sort-based building blocks for the REGRAD-style helpers of utils/projections.py:
//   * lexicographic sort of (N,3) fp64 rows + unique + segmented max  -> pool_multiview_features
//     (utils/projections.py:245-261: np.unique(axis=0) + np.maximum.reduceat)
//   * voxel-grid down-sampling with per-voxel mean in point order     -> pc_voxel_down
//     (utils/geometry.py:350-352 -> Open3D voxel_down_sample, parity unpinned: Open3D absent);
//     the traced variant with the label vote lives in aggregate.cu
//   * exact nearest neighbour (fp64, brute force, tiled through smem) -> find_closest_indices
//     (utils/geometry.py:390-401 -> scipy cKDTree.query, k = 1)
// The sort is a bitonic network over an index array (power-of-two padded with sentinels); steps
// whose partner distance fits a CTA run in shared memory, the rest in global memory. Keys are
// fetched through the index (gather) so that any key type can be sorted by the same kernels.
#include "geometry_math.cuh"

namespace {

constexpr int kSortThreads = 512;
constexpr int kSortChunk = 2 * kSortThreads;  // elements sorted per CTA in shared memory

struct LessRow3 {  // lexicographic (x, y, z), ties by index; -1 = +inf sentinel
  const double* p;
  __device__ __forceinline__ bool operator()(int a, int b) const {
    if (a < 0 || b < 0) return b < 0 && a >= 0;
    const double ax = p[3 * (int64_t)a], bx = p[3 * (int64_t)b];
    if (ax < bx) return true;
    if (ax > bx) return false;
    const double ay = p[3 * (int64_t)a + 1], by = p[3 * (int64_t)b + 1];
    if (ay < by) return true;
    if (ay > by) return false;
    const double az = p[3 * (int64_t)a + 2], bz = p[3 * (int64_t)b + 2];
    if (az < bz) return true;
    if (az > bz) return false;
    return a < b;
  }
};

struct LessKey64 {
  const unsigned long long* k;
  __device__ __forceinline__ bool operator()(int a, int b) const {
    if (a < 0 || b < 0) return b < 0 && a >= 0;
    const unsigned long long ka = k[a], kb = k[b];
    if (ka != kb) return ka < kb;
    return a < b;
  }
};

template <class Less>
__device__ __forceinline__ void cmp_swap(int& a, int& b, bool ascending, const Less& less) {
  if (less(b, a) == ascending) {
    const int t = a;
    a = b;
    b = t;
  }
}

// all steps with partner distance < kSortChunk for stage size k (k_first..k_last), in shared memory
template <class Less>
__global__ void __launch_bounds__(kSortThreads) bitonic_smem_kernel(int* __restrict__ idx, int64_t k_first, int64_t k_last,
                                                                    Less less) {
  __shared__ int s[kSortChunk];
  const int64_t base = (int64_t)blockIdx.x * kSortChunk;
  s[threadIdx.x] = idx[base + threadIdx.x];
  s[threadIdx.x + kSortThreads] = idx[base + threadIdx.x + kSortThreads];
  __syncthreads();
  for (int64_t k = k_first; k <= k_last; k <<= 1) {
    int64_t j = k >> 1;
    if (j >= kSortChunk) j = kSortChunk >> 1;
    for (; j > 0; j >>= 1) {
      const int t = threadIdx.x;
      const int lo = (int)(((t / j) * 2 * j) + (t % j));  // lower element of the pair
      const int hi = lo + (int)j;
      const bool asc = (((base + lo) & k) == 0);
      cmp_swap(s[lo], s[hi], asc, less);
      __syncthreads();
    }
  }
  idx[base + threadIdx.x] = s[threadIdx.x];
  idx[base + threadIdx.x + kSortThreads] = s[threadIdx.x + kSortThreads];
}

template <class Less>
__global__ void __launch_bounds__(256) bitonic_global_kernel(int* __restrict__ idx, int64_t n_pairs, int64_t j, int64_t k, Less less) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_pairs) return;
  const int64_t lo = ((t / j) * 2 * j) + (t % j);
  const int64_t hi = lo + j;
  const bool asc = ((lo & k) == 0);
  int a = idx[lo], b = idx[hi];
  const int a0 = a;
  cmp_swap(a, b, asc, less);
  if (a != a0) {
    idx[lo] = a;
    idx[hi] = b;
  }
}

__global__ void iota_pad_kernel(int* idx, int64_t n, int64_t n_pad) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pad; i += (int64_t)gridDim.x * blockDim.x)
    idx[i] = i < n ? (int)i : -1;
}

int64_t pad_pow2(int64_t n) {
  int64_t p = kSortChunk;
  while (p < n) p <<= 1;
  return p;
}

unsigned grid_for(int64_t n, int threads = 256) {
  int64_t b = dc::ceil_div<int64_t>(n, threads);
  const int64_t cap = (int64_t)dc::sm_count() * 16;
  return (unsigned)(b < 1 ? 1 : (b < cap ? b : cap));
}

template <class Less>
int bitonic_sort(int* idx, int64_t n, Less less, cudaStream_t st) {
  const int64_t n_pad = pad_pow2(n);
  iota_pad_kernel<<<grid_for(n_pad), 256, 0, st>>>(idx, n, n_pad);
  const unsigned chunks = (unsigned)(n_pad / kSortChunk);
  bitonic_smem_kernel<Less><<<chunks, kSortThreads, 0, st>>>(idx, 2, kSortChunk, less);
  for (int64_t k = 2 * (int64_t)kSortChunk; k <= n_pad; k <<= 1) {
    for (int64_t j = k >> 1; j >= kSortChunk; j >>= 1)
      bitonic_global_kernel<Less><<<(unsigned)dc::ceil_div<int64_t>(n_pad / 2, 256), 256, 0, st>>>(idx, n_pad / 2, j, k, less);
    bitonic_smem_kernel<Less><<<chunks, kSortThreads, 0, st>>>(idx, k, k, less);
  }
  DC_LAUNCH_CHECK();
  return DC_OK;
}

// ------------------------------------------------------------------ unique + segmented max
__global__ void row_heads_kernel(const double* __restrict__ pts, const int* __restrict__ order, int64_t n, uint8_t* __restrict__ head) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    bool h = true;
    if (i > 0) {
      const int64_t a = order[i - 1], b = order[i];
      h = !(pts[3 * a] == pts[3 * b] && pts[3 * a + 1] == pts[3 * b + 1] && pts[3 * a + 2] == pts[3 * b + 2]);
    }
    head[i] = h ? 1 : 0;
  }
}

__global__ void key_heads_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ order, int64_t n,
                                 uint8_t* __restrict__ head) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    head[i] = (i == 0 || keys[order[i - 1]] != keys[order[i]]) ? 1 : 0;
}

// single-CTA exclusive scan of head flags -> segment id per sorted position, total in *count.
// (these helpers serve the peripheral REGRAD path; N is at most a few million)
__global__ void __launch_bounds__(1024) scan_heads_kernel(const uint8_t* __restrict__ head, int64_t n, int64_t* __restrict__ seg,
                                                          int64_t* __restrict__ count) {
  __shared__ int64_t s[1024];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int64_t per = 16;
  for (int64_t c0 = 0; c0 < n; c0 += 1024 * per) {
    const int64_t b = c0 + (int64_t)threadIdx.x * per;
    int64_t loc = 0;
    for (int64_t k = 0; k < per; ++k)
      if (b + k < n) loc += head[b + k];
    s[threadIdx.x] = loc;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      const int64_t add = threadIdx.x >= o ? s[threadIdx.x - o] : 0;
      __syncthreads();
      s[threadIdx.x] += add;
      __syncthreads();
    }
    int64_t run = carry + s[threadIdx.x] - loc;
    for (int64_t k = 0; k < per; ++k)
      if (b + k < n) {
        run += head[b + k];
        seg[b + k] = run - 1;  // id of the segment this position belongs to (heads start a new one)
      }
    __syncthreads();
    if (threadIdx.x == 1023) carry += s[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = carry;
}

template <typename T>
__global__ void __launch_bounds__(256) unique_max_pool_kernel(const double* __restrict__ pts, const T* __restrict__ feats, int dim,
                                                              const int* __restrict__ order, const uint8_t* __restrict__ head,
                                                              const int64_t* __restrict__ seg, int64_t n,
                                                              double* __restrict__ out_pts, T* __restrict__ out_feats) {
  // one warp per sorted position that is a segment head; it walks its segment
  const int lane = threadIdx.x & 31;
  for (int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); i < n; i += (int64_t)gridDim.x * 8) {
    if (!head[i]) continue;
    const int64_t u = seg[i];
    const int64_t first = order[i];
    if (lane < 3) out_pts[3 * u + lane] = pts[3 * first + lane] + 0.0;  // -0.0 -> +0.0 like the sorted representative
    int64_t end = i + 1;
    while (end < n && !head[end]) ++end;
    for (int c = lane; c < dim; c += 32) {
      T m = feats[first * dim + c];
      for (int64_t k = i + 1; k < end; ++k) {
        const T v = feats[(int64_t)order[k] * dim + c];
        m = (v > m || v != v) ? v : m;  // np.maximum propagates NaN
      }
      out_feats[u * dim + c] = m;
    }
  }
}

// ------------------------------------------------------------------ voxel down-sampling (Open3D semantics)
__global__ void __launch_bounds__(256) min_bound_kernel(const double* __restrict__ pts, int64_t n, unsigned long long* __restrict__ mn) {
  // ordered-integer image of a double so that atomicMin works for negative values too
  double lx = INFINITY, ly = INFINITY, lz = INFINITY;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    lx = fmin(lx, pts[3 * i]);
    ly = fmin(ly, pts[3 * i + 1]);
    lz = fmin(lz, pts[3 * i + 2]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    lx = fmin(lx, __shfl_xor_sync(0xffffffffu, lx, o));
    ly = fmin(ly, __shfl_xor_sync(0xffffffffu, ly, o));
    lz = fmin(lz, __shfl_xor_sync(0xffffffffu, lz, o));
  }
  if ((threadIdx.x & 31) == 0) {
    const double v[3] = {lx, ly, lz};
    for (int a = 0; a < 3; ++a) atomicMin(mn + a, dc::double_to_ordered(v[a]));
  }
}

__global__ void __launch_bounds__(256) voxel_keys_kernel(const double* __restrict__ pts, int64_t n, double voxel,
                                                         const unsigned long long* __restrict__ mn, unsigned long long* __restrict__ keys,
                                                         int* __restrict__ error) {
  const double bx = dc::ordered_to_double(mn[0]) - voxel * 0.5, by = dc::ordered_to_double(mn[1]) - voxel * 0.5,
               bz = dc::ordered_to_double(mn[2]) - voxel * 0.5;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    // Open3D: ref_coord = (point - voxel_min_bound) / voxel_size; voxel_index = floor(ref_coord)
    const double fx = dc::voxel_coord(pts[3 * i], bx, voxel);
    const double fy = dc::voxel_coord(pts[3 * i + 1], by, voxel);
    const double fz = dc::voxel_coord(pts[3 * i + 2], bz, voxel);
    if (!(dc::voxel_coord_ok(fx) && dc::voxel_coord_ok(fy) && dc::voxel_coord_ok(fz))) {
      atomicExch(error, 1);
      keys[i] = 0;
      continue;
    }
    keys[i] = ((unsigned long long)fx << 42) | ((unsigned long long)fy << 21) | (unsigned long long)fz;
  }
}

// one thread per voxel: sequential sum of its members in ascending point index (the sort breaks
// ties by index), then / count - the accumulation order of Open3D's AccumulatedPoint
__global__ void __launch_bounds__(256) voxel_mean_kernel(const double* __restrict__ pts, const int* __restrict__ order,
                                                         const uint8_t* __restrict__ head, const int64_t* __restrict__ seg, int64_t n,
                                                         double* __restrict__ out, int64_t* __restrict__ first_index) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (!head[i]) continue;
    double sx = 0, sy = 0, sz = 0;
    int64_t c = 0, k = i;
    do {
      const int64_t j = order[k];
      sx += pts[3 * j];
      sy += pts[3 * j + 1];
      sz += pts[3 * j + 2];
      ++c;
      ++k;
    } while (k < n && !head[k]);
    const int64_t u = seg[i];
    out[3 * u] = sx / (double)c;
    out[3 * u + 1] = sy / (double)c;
    out[3 * u + 2] = sz / (double)c;
    first_index[u] = order[i];
  }
}

// ------------------------------------------------------------------ nearest neighbour
constexpr int kNNTile = 1024;
__global__ void __launch_bounds__(256) nearest_kernel(const double* __restrict__ query, int64_t m, const double* __restrict__ ref,
                                                      int64_t n, int64_t* __restrict__ out, double* __restrict__ out_d2) {
  __shared__ double s[kNNTile * 3];
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = q < m;
  const double x = live ? query[3 * q] : 0, y = live ? query[3 * q + 1] : 0, z = live ? query[3 * q + 2] : 0;
  double best = INFINITY;
  int64_t arg = -1;
  for (int64_t t0 = 0; t0 < n; t0 += kNNTile) {
    const int cnt = (int)((n - t0) < kNNTile ? (n - t0) : kNNTile);
    __syncthreads();
    for (int i = threadIdx.x; i < cnt * 3; i += blockDim.x) s[i] = ref[3 * t0 + i];
    __syncthreads();
    if (live) {
#pragma unroll 4
      for (int i = 0; i < cnt; ++i) {
        const double dx = s[3 * i] - x, dy = s[3 * i + 1] - y, dz = s[3 * i + 2] - z;
        const double d2 = dx * dx + dy * dy + dz * dz;
        if (d2 < best) {  // strict: the smallest index wins ties
          best = d2;
          arg = t0 + i;
        }
      }
    }
  }
  if (live) {
    out[q] = arg;
    if (out_d2) out_d2[q] = best;
  }
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct SortWs {
  int* order;
  uint8_t* head;
  int64_t* seg;
  unsigned long long* keys;
  unsigned long long* mn;
  int* error;
  size_t total;
};

SortWs carve(void* ws, int64_t n) {
  const int64_t n_pad = pad_pow2(n > 0 ? n : 1);
  size_t off = 0;
  auto take = [&](size_t b) { size_t o = off; off = align_up(off + b, 256); return o; };
  const size_t o_order = take(4 * (size_t)n_pad), o_head = take((size_t)n_pad), o_seg = take(8 * (size_t)n_pad),
               o_keys = take(8 * (size_t)n_pad), o_mn = take(32), o_err = take(8);
  SortWs w{};
  w.total = off;
  if (ws) {
    uint8_t* b = reinterpret_cast<uint8_t*>(ws);
    w.order = reinterpret_cast<int*>(b + o_order);
    w.head = b + o_head;
    w.seg = reinterpret_cast<int64_t*>(b + o_seg);
    w.keys = reinterpret_cast<unsigned long long*>(b + o_keys);
    w.mn = reinterpret_cast<unsigned long long*>(b + o_mn);
    w.error = reinterpret_cast<int*>(b + o_err);
  }
  return w;
}

}  // namespace

extern "C" {

size_t dc_sort_workspace(int64_t n) { return carve(nullptr, n).total; }

int dc_unique_max_pool(const double* points, const void* feats, int feat_dtype, int dim, int64_t n, double* out_points,
                       void* out_feats, int64_t* n_unique, void* workspace, size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(points && feats && out_points && out_feats && n_unique && workspace, "dc_unique_max_pool: null pointer argument");
  DC_CHECK_ARG(feat_dtype == DC_F32 || feat_dtype == DC_F64, "dc_unique_max_pool: features must be fp32 or fp64");
  DC_CHECK_ARG(n < (1ll << 30) && dim > 0, "dc_unique_max_pool: bad sizes");
  SortWs w = carve(workspace, n);
  if (workspace_bytes < w.total) return dc::fail(DC_ERR_WORKSPACE, "dc_unique_max_pool: workspace %zu < %zu", workspace_bytes, w.total);
  cudaStream_t st = dc::as_stream(stream);
  if (n <= 0) {
    DC_CUDA(cudaMemsetAsync(n_unique, 0, sizeof(int64_t), st));
    return DC_OK;
  }
  int rc = bitonic_sort(w.order, n, LessRow3{points}, st);
  if (rc) return rc;
  row_heads_kernel<<<grid_for(n), 256, 0, st>>>(points, w.order, n, w.head);
  scan_heads_kernel<<<1, 1024, 0, st>>>(w.head, n, w.seg, n_unique);
  if (feat_dtype == DC_F32)
    unique_max_pool_kernel<float><<<grid_for(n * 32), 256, 0, st>>>(points, (const float*)feats, dim, w.order, w.head, w.seg, n,
                                                                   out_points, (float*)out_feats);
  else
    unique_max_pool_kernel<double><<<grid_for(n * 32), 256, 0, st>>>(points, (const double*)feats, dim, w.order, w.head, w.seg, n,
                                                                    out_points, (double*)out_feats);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

int dc_voxel_down_mean(const double* points, int64_t n, double voxel_size, double* out_points, int64_t* first_index,
                       int64_t* n_voxels, void* workspace, size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(points && out_points && first_index && n_voxels && workspace, "dc_voxel_down_mean: null pointer argument");
  DC_CHECK_ARG(voxel_size > 0.0, "dc_voxel_down_mean: voxel_size must be positive");
  DC_CHECK_ARG(n < (1ll << 30), "dc_voxel_down_mean: too many points");
  SortWs w = carve(workspace, n);
  if (workspace_bytes < w.total) return dc::fail(DC_ERR_WORKSPACE, "dc_voxel_down_mean: workspace %zu < %zu", workspace_bytes, w.total);
  cudaStream_t st = dc::as_stream(stream);
  if (n <= 0) {
    DC_CUDA(cudaMemsetAsync(n_voxels, 0, sizeof(int64_t), st));
    return DC_OK;
  }
  DC_CUDA(cudaMemsetAsync(w.mn, 0xFF, 24, st));
  DC_CUDA(cudaMemsetAsync(w.error, 0, 4, st));
  min_bound_kernel<<<grid_for(n), 256, 0, st>>>(points, n, w.mn);
  voxel_keys_kernel<<<grid_for(n), 256, 0, st>>>(points, n, voxel_size, w.mn, w.keys, w.error);
  int rc = bitonic_sort(w.order, n, LessKey64{w.keys}, st);
  if (rc) return rc;
  key_heads_kernel<<<grid_for(n), 256, 0, st>>>(w.keys, w.order, n, w.head);
  scan_heads_kernel<<<1, 1024, 0, st>>>(w.head, n, w.seg, n_voxels);
  voxel_mean_kernel<<<grid_for(n), 256, 0, st>>>(points, w.order, w.head, w.seg, n, out_points, first_index);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

int dc_nearest_index(const double* query, int64_t m, const double* ref, int64_t n, int64_t* out_index, double* out_dist2,
                     dc_stream_t stream) {
  DC_CHECK_ARG(query && ref && out_index, "dc_nearest_index: null pointer argument");
  DC_CHECK_ARG(n >= 1, "dc_nearest_index: empty reference set");
  if (m <= 0) return DC_OK;
  nearest_kernel<<<(unsigned)dc::ceil_div<int64_t>(m, 256), 256, 0, dc::as_stream(stream)>>>(query, m, ref, n, out_index, out_dist2);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

}  // extern "C"
