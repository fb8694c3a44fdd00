// (1) Projection + visibility with spatially sorted points.
//
// Why: the reference's point cloud arrives in Open3D hash order, so the 32 lanes of a warp gather
// 32 unrelated depth pixels = 32 distinct 128-B lines per load. ncu on the direct kernel
// (profiles/r01_ncu_project_visibility_v1_raw.csv) shows DRAM at 6 %, L2 hit rate 84 % and the
// time set by L1TEX line replays (~2 cycles per line). Sorting the points of a scene by a coarse
// Morton cell makes neighbouring lanes project to neighbouring pixels (~8 lines per load).
//
// Pipeline (all kernels scene-batched, results bit-identical to the direct kernel):
//   1. bbox per scene (fp32 is enough: cells only steer locality, never results)
//   2. counting sort by 15-bit Morton cell: histogram -> per-scene scan -> scatter (perm, rank)
//   3. visibility in sorted order - an fp32 filter with rigorous error bounds decides ~99.8 % of the
//      (point, view) pairs, the rest is re-evaluated with the literal fp64 sequence from a per-warp
//      queue (see "fp32 filter + exact fp64 queue" below); results bit-packed per point (one
//      32-bit word per 32 views, plane-major so that lanes store contiguous words)
//   4. unpack: a thread per original point reads its words through `rank` and writes the
//      (V,N) mask rows coalesced - or, fused with the removal of never-visible points, writes the
//      compacted (V,N') mask directly (the form fuse_obj_prior returns, utils/feature_fusion.py
//      :277-281), so the full mask never touches HBM.
#include <mutex>
#include <type_traits>

#include "visibility_math.cuh"

namespace {

using namespace dc::vis;

constexpr int kThreads = 256;
constexpr int kCellBits = 5;                    // per axis
constexpr int kCells = 1 << (3 * kCellBits);    // 32768 bins per scene
constexpr float kHuge = 1e15f;                  // coordinates beyond this never enter the fp32 filter

struct SortedWs {
  float* bbox;        // [n_scenes][6] min xyz, max xyz
  int* counts;        // [n_scenes][kCells]
  int64_t* perm;      // [total_points] scene-local point index at each sorted position
  void* view_consts;  // [n_scenes][max_views] ViewConst
  size_t total;
};

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

SortedWs carve(void* ws, int64_t total_points, int n_scenes, int max_views) {
  size_t off = 0;
  auto take = [&](size_t b) { size_t o = off; off = align_up(off + b, 256); return o; };
  const size_t o_bbox = take(sizeof(float) * 6 * (size_t)n_scenes);
  const size_t o_counts = take(sizeof(int) * (size_t)kCells * (size_t)n_scenes);
  const size_t o_perm = take(sizeof(int64_t) * (size_t)(total_points > 0 ? total_points : 1));
  const size_t o_vc = take((size_t)80 * (size_t)n_scenes * (size_t)(max_views > 0 ? max_views : 1));
  SortedWs w{};
  w.total = off;
  if (ws) {
    uint8_t* b = reinterpret_cast<uint8_t*>(ws);
    w.bbox = reinterpret_cast<float*>(b + o_bbox);
    w.counts = reinterpret_cast<int*>(b + o_counts);
    w.perm = reinterpret_cast<int64_t*>(b + o_perm);
    w.view_consts = b + o_vc;
  }
  return w;
}

__device__ __forceinline__ void atomic_min_f(float* a, float v) {
  if (v >= 0) atomicMin(reinterpret_cast<int*>(a), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned*>(a), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f(float* a, float v) {
  if (v >= 0) atomicMax(reinterpret_cast<int*>(a), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned*>(a), __float_as_uint(v));
}

__global__ void init_bbox_kernel(float* bbox, int n_scenes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_scenes * 6) bbox[i] = (i % 6 < 3) ? INFINITY : -INFINITY;
}

__device__ __forceinline__ float finite_or(double v, float alt) {
  const float f = (float)v;
  return (fabsf(f) < kHuge) ? f : alt;  // NaN / inf / huge coordinates do not stretch the grid (exact path only)
}

__global__ void __launch_bounds__(kThreads) bbox_kernel(const double* __restrict__ points, const int64_t* __restrict__ point_off,
                                                        float* __restrict__ bbox) {
  const int scene = blockIdx.y;
  const int64_t p0 = point_off[scene], n = point_off[scene + 1] - p0;
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double v = __ldg(points + 3 * (p0 + i) + a);
      lo[a] = fminf(lo[a], finite_or(v, INFINITY));
      hi[a] = fmaxf(hi[a], finite_or(v, -INFINITY));
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    lo[a] = dc::warp_min(lo[a]);
    hi[a] = dc::warp_max(hi[a]);
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (lo[a] != INFINITY) atomic_min_f(bbox + scene * 6 + a, lo[a] + 0.0f);
      if (hi[a] != -INFINITY) atomic_max_f(bbox + scene * 6 + 3 + a, hi[a] + 0.0f);
    }
  }
}

__device__ __forceinline__ unsigned spread3(unsigned v) {  // 5 bits -> every third bit
  v &= 0x1f;
  v = (v | (v << 8)) & 0x100f;
  v = (v | (v << 4)) & 0x10c3;
  v = (v | (v << 2)) & 0x1249;
  return v;
}

__device__ __forceinline__ int cell_of(const double* __restrict__ points, int64_t j, const float* __restrict__ bb) {
  const float ext = fmaxf(fmaxf(bb[3] - bb[0], bb[4] - bb[1]), fmaxf(bb[5] - bb[2], 1e-20f));
  const float inv = (float)(1 << kCellBits) / ext;  // isotropic cells
  unsigned c[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float f = (finite_or(__ldg(points + 3 * j + a), bb[a]) - bb[a]) * inv;
    int q = (int)f;
    q = q < 0 ? 0 : (q > (1 << kCellBits) - 1 ? (1 << kCellBits) - 1 : q);
    c[a] = (unsigned)q;
  }
  return (int)(spread3(c[0]) | (spread3(c[1]) << 1) | (spread3(c[2]) << 2));
}

__global__ void __launch_bounds__(kThreads) cell_count_kernel(const double* __restrict__ points, const int64_t* __restrict__ point_off,
                                                              const float* __restrict__ bbox, int* __restrict__ counts) {
  const int scene = blockIdx.y;
  const int64_t p0 = point_off[scene], n = point_off[scene + 1] - p0;
  const float* bb = bbox + scene * 6;
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads)
    atomicAdd(counts + (int64_t)scene * kCells + cell_of(points, p0 + i, bb), 1);
}

// one CTA per scene: exclusive scan of its kCells counters, in place. Warp w owns the 1024 consecutive
// counters [w * 1024, (w + 1) * 1024) and walks them 32 at a time (coalesced), scanning with shuffles;
// the 32 warp totals are scanned once and added in a second coalesced pass.
__global__ void __launch_bounds__(1024) cell_scan_kernel(int* __restrict__ counts) {
  static_assert(kCells == 32 * 1024, "one warp per 1024 counters");
  __shared__ int s_warp[32];
  int* c = counts + (int64_t)blockIdx.x * kCells + (threadIdx.x >> 5) * 1024;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int carry = 0;
#pragma unroll 4
  for (int it = 0; it < 32; ++it) {
    const int v = c[it * 32 + lane];
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += up;
    }
    c[it * 32 + lane] = carry + incl - v;  // exclusive inside the warp's range
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) s_warp[warp] = carry;
  __syncthreads();
  if (warp == 0) {
    const int t = s_warp[lane];
    int incl = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += up;
    }
    s_warp[lane] = incl - t;
  }
  __syncthreads();
  const int base = s_warp[warp];
  if (base != 0) {
#pragma unroll 4
    for (int it = 0; it < 32; ++it) c[it * 32 + lane] += base;
  }
}

__global__ void __launch_bounds__(kThreads) cell_scatter_kernel(const double* __restrict__ points, const int64_t* __restrict__ point_off,
                                                                const float* __restrict__ bbox, int* __restrict__ counts,
                                                                int64_t* __restrict__ perm, int64_t* __restrict__ rank) {
  const int scene = blockIdx.y;
  const int64_t p0 = point_off[scene], n = point_off[scene + 1] - p0;
  const float* bb = bbox + scene * 6;
  int* c = counts + (int64_t)scene * kCells;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  // four returning atomics in flight per thread: the slot reservation is a round trip to L2
  for (; i + 3 * stride < n; i += 4 * stride) {
    int cell[4], pos[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) cell[k] = cell_of(points, p0 + i + k * stride, bb);
#pragma unroll
    for (int k = 0; k < 4; ++k) pos[k] = atomicAdd(c + cell[k], 1);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      perm[p0 + pos[k]] = i + k * stride;  // order inside a cell depends on scheduling; results do not (they are un-permuted)
      rank[p0 + i + k * stride] = pos[k];
    }
  }
  for (; i < n; i += stride) {
    const int pos = atomicAdd(c + cell_of(points, p0 + i, bb), 1);
    perm[p0 + pos] = i;
    rank[p0 + i] = pos;
  }
}

// ---------------------------------------------------------------------------------------------
// fp32 filter + exact fp64 queue
//
// The reference's arithmetic is fp64 (oracle/visibility_ref.c) and the result must match it bit for
// bit, but only two facts per (point, view) are observable: the integer pixel and the outcome of
// |depth - z| <= threshold. Both are decided here from an fp32 evaluation with a rigorous error
// bound; a pair whose fp32 interval straddles a decision boundary (pixel edge, image border,
// threshold) is pushed to a per-warp queue and re-evaluated later with the literal fp64 sequence
// (`literal_pixel`), with all 32 lanes busy. On MV-TOD-shaped scenes ~0.2 % of the pairs take the
// exact path (benchmarks/fp32_filter_model.py), so the fp64 pipe (1/2 rate, ~35 instructions per
// pair in the previous kernel) is off the critical path.
//
// Error model (eps = 2^-24, u = 2^-53; x~ denotes fp32 quantities):
//   P = K * [R|t]' (3x4, evaluated once per view in fp64, rows 1,2 of the inverse pose negated),
//   q~_r = fp32 dot(P~_r, [p~;1]).  Rounding P and p to fp32 costs 2 eps per product, the chain at
//   most 5 more roundings, the reference's own fp64 roundings ~10 u:  |q~_r - q_r| <= E_r :=
//   8 eps * (sum_j A_rj * B_j + A_r3), A_rj = |K_r0||M_0j| + |K_r2||M_2j| >= |P_rj| (no cancellation, so the
//   same sum times 8 u also bounds the reference's fp64 roundings), B = per-scene bound on |coordinate|.
//   r~ = rcp.approx(q~_z) (1 ulp) = (1 + eta) / q_z with |eta| <= rho := 1.03 E_z r~ + 5 eps, valid while
//   q~_z >= zmin := max(1024 E_z, 4 E_x, 4 E_y)  (points behind or within ~2 cm of the camera plane take
//   the exact path; then rho <= 1.01e-3 and E_x r~ <= 0.26).   u~ = q~_x * r~  =>
//   |u~ - u| <= 1.02 (|u~| rho + E_x r~)                     (same for v with E_y).
//   With f = floor(u~) (exact, by the 1.5 * 2^23 trick) and c = (W - 1) / 2 a pair is, per axis,
//     "not near"  |f - c| > NL := c + 2 + 0.0014 W : the true u lies outside [-1, W) whatever the error
//                 (relative part <= 1.3e-3 |u~|, additive part <= 0.26) -> decided, outside;
//     otherwise |u~| <= U := c + NL + 1 and the bound becomes linear in r~:
//                 e_u = A_u r~ + B_u,  A_u = 1.02 (E_x + 1.03 U E_z),  B_u = 1.02 * 5 eps * U.
//   The pixel is decided when the fractional part t = u~ - |f| lies in (e_u, 1 - e_u) on both axes (no
//   integer between u~ and the reference's correctly rounded quotient); then floor(u_ref) = f and the
//   reference's "trunc toward zero into [0, W)" test is 0 <= f <= W - 1. Using |f| makes t fall outside
//   [0, 1) for f < 0, so u in (-1, 0) - which the reference maps to column 0 (quirk q1) - is never
//   decided here and is evaluated exactly.
//   The depth test is decided when | |d - q~_z| - threshold | > E_z (+ fp32 rounding slack).
// Anything non-finite, huge or degenerate fails a comparison and ends up in the exact queue.
//
// Arithmetic is packed two-wide where both axes share an operation (fma.rn.f32x2 etc. on sm_100a: the
// x and y image rows of P, the floor trick, the border tests), the point coordinates are kept
// duplicated in register pairs for that, and the camera table is laid out so that one 64-bit constant
// load yields the (x-row, y-row) operand pair.
struct ViewConst {        // 20 floats = 80 B; 819 views fit the 64 KB constant bank
  float2 Pxy[4];          // (P_0j, P_1j): x and y image rows of K * inverse pose (rows 1,2 negated), fp32
  float Pz[4];            // z row
  float2 nA;              // (-A_u, -A_v)
  float zmin;             // +inf disables the filter for this view (non-pinhole K, overflow)
  float thr_lo, thr_hi;   // threshold -/+ E_z with directed rounding
  float pad0, pad1, pad2;
};
static_assert(sizeof(ViewConst) == 80, "ViewConst layout");
constexpr int kConstViews = 65536 / (int)sizeof(ViewConst);  // 819
__constant__ ViewConst c_views[kConstViews];

constexpr int kPts = 4;                        // points per thread
constexpr int kTile = kThreads * kPts;         // points per CTA
constexpr int kQueue = 256;                    // exact-path queue entries per warp
constexpr float kMagic = 12582912.0f;          // 1.5 * 2^23: x + kMagic (round down) = floor(x) + kMagic for |x| < 2^22

__host__ __device__ inline double near_limit(int limit) { return 0.5 * (limit - 1) + 2.0 + 0.0014 * limit; }   // NL
__host__ __device__ inline double coord_bound(int limit) { return 0.5 * (limit - 1) + near_limit(limit) + 1.0; }  // U

// one thread per (scene, view slot): fp64 set-up of the filter constants
__global__ void camera_prep_kernel(const double* __restrict__ inv_poses, const double* __restrict__ intrinsics,
                                   const int64_t* __restrict__ view_off, const float* __restrict__ bbox, int n_scenes,
                                   int max_views, int height, int width, double threshold, ViewConst* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_scenes * max_views) return;
  const int scene = i / max_views, v = i - scene * max_views;
  ViewConst c;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    c.Pxy[j] = make_float2(0.f, 0.f);
    c.Pz[j] = 0.f;
  }
  c.nA = make_float2(0.f, 0.f);
  c.zmin = INFINITY;
  c.thr_lo = -INFINITY;
  c.thr_hi = INFINITY;
  c.pad0 = c.pad1 = c.pad2 = 0.f;
  const int64_t v0 = view_off[scene];
  const int n_views = (int)(view_off[scene + 1] - v0);
  if (v < n_views) {
    double m[12];
    bool ok = true;
#pragma unroll
    for (int e = 0; e < 12; ++e) {
      const double val = __ldg(inv_poses + (v0 + v) * 16 + e);
      ok &= fabs(val) < 1e30;
      m[e] = (e >= 4) ? -val : val;
    }
    double K[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) {
      K[e] = __ldg(intrinsics + (int64_t)scene * 9 + e);
      ok &= fabs(K[e]) < 1e30;
    }
    ok &= (K[1] == 0.0 && K[3] == 0.0 && K[6] == 0.0 && K[7] == 0.0 && K[8] == 1.0);
    const float* bb = bbox + scene * 6;
    double B[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double lo = bb[a], hi = bb[3 + a];
      B[a] = (lo <= hi) ? fmax(fabs(lo), fabs(hi)) * (1.0 + 1e-6) : 0.0;  // bbox holds fp32-rounded coordinates
    }
    double P[12], E[3];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      P[j] = K[0] * m[j] + K[2] * m[8 + j];
      P[4 + j] = K[4] * m[4 + j] + K[5] * m[8 + j];
      P[8 + j] = m[8 + j];
    }
    const double eps = 5.9604644775390625e-08;  // 2^-24
#pragma unroll
    // magnitude sums WITHOUT cancellation between the two products of a row of K * M: they bound the fp32
    // error of q~ (|P_rj| <= A_rj) and, times 8 u, the rounding of the reference's own two-step fp64 evaluation
    double A[12];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      A[j] = fabs(K[0]) * fabs(m[j]) + fabs(K[2]) * fabs(m[8 + j]);
      A[4 + j] = fabs(K[4]) * fabs(m[4 + j]) + fabs(K[5]) * fabs(m[8 + j]);
      A[8 + j] = fabs(m[8 + j]);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const double S = A[4 * r] * B[0] + A[4 * r + 1] * B[1] + A[4 * r + 2] * B[2] + A[4 * r + 3];
      ok &= S < 1e30;
      E[r] = fmax(8.0 * eps * S * (1.0 + 1e-6), 1e-30);
    }
    if (ok) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        c.Pxy[j] = make_float2((float)P[j], (float)P[4 + j]);
        c.Pz[j] = (float)P[8 + j];
      }
      c.nA = make_float2(-__double2float_ru(1.02 * (E[0] + 1.03 * coord_bound(width) * E[2])),
                         -__double2float_ru(1.02 * (E[1] + 1.03 * coord_bound(height) * E[2])));
      c.zmin = __double2float_ru(fmax(1024.0 * E[2], fmax(4.0 * E[0], 4.0 * E[1])));
      const double lo = threshold - E[2], hi = threshold + E[2];
      c.thr_lo = __double2float_rd(lo - 4.0 * eps * fabs(lo) - 1e-30);   // NaN threshold: every comparison fails
      c.thr_hi = __double2float_ru(hi + 4.0 * eps * fabs(hi) + 1e-30);
    }
  }
  out[i] = c;
}

struct FastParams {
  const double* points;
  const int64_t* point_off;
  const int64_t* view_off;
  const float* depths;
  const double* inv_poses;
  const double* intrinsics;
  const int64_t* perm;
  int64_t total_points;
  int scene0, max_views;
  int height, width;
  float wf;                 // width
  unsigned idx_max;         // height * width - 1
  float2 centre;            // ((W - 1) / 2, (H - 1) / 2): |floor - centre| <= centre  <=>  0 <= floor <= limit - 1
  float2 near;              // NL per axis
  float2 h0;                // 0.499999 - B per axis
  double threshold;
  uint32_t* records;  // [n_words][total_points], indexed by sorted position
  uint8_t* any_visible;
};

// Exact re-evaluation of the queued pairs of one warp (all lanes busy). Results are OR-ed into the
// warp's slice of s_rec. Kept out of line so that its fp64 registers do not weigh on the filter loop.
// `pts` / `perm` point at the scene's first point, `poses` / `depths` at its first view, `K` at its intrinsics.
static __device__ __noinline__ void drain_queue(const uint32_t* __restrict__ queue, int count, int n_tile, const double* __restrict__ pts,
                                                const int64_t* __restrict__ perm_tile, const double* __restrict__ poses,
                                                const double* __restrict__ Kp, const float* __restrict__ depths, int width,
                                                int height, double threshold, uint32_t* __restrict__ s_rec) {
  const int lane = threadIdx.x & 31;
  double K[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) K[e] = __ldg(Kp + e);
  const int64_t hw = (int64_t)height * width;
  for (int i = lane; i < count; i += 32) {
    const uint32_t entry = queue[i];
    const int v = (int)(entry >> 12), local = (int)(entry & 4095u);
    const int64_t orig = __ldg(perm_tile + (local < n_tile ? local : n_tile - 1));  // padding slots repeat the last point
    const double x = __ldg(pts + 3 * orig), y = __ldg(pts + 3 * orig + 1), z = __ldg(pts + 3 * orig + 2);
    double m[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) {
      const double val = __ldg(poses + (int64_t)v * 16 + e);
      m[e] = (e >= 4) ? -val : val;
    }
    int pix;
    double qz;
    bool vis = literal_pixel(m, K, x, y, z, width, height, pix, qz);
    if (vis) vis = fabs((double)__ldg(depths + (int64_t)v * hw + pix) - qz) <= threshold;
    if (vis) atomicOr(s_rec + (v >> 5) * kTile + local, 1u << (v & 31));
  }
}

// Stage A of one view for the kPts points of a thread: fp32 projection, pixel decision, and the depth
// gather ISSUED as a 4-byte cp.async into the thread's own shared-memory slot. The loop below tests it
// three stages later behind cp.async.wait_group, so the L2/DRAM latency of the gather is covered by
// the arithmetic of the next views instead of by occupancy. (Plain loads cannot do this: ptxas puts
// every LDG of the loop on one scoreboard, so a consumer of the oldest gather also waits for the
// newest - measured as 18-28 % of all stall samples on that one instruction.)
__device__ __forceinline__ void cp_async_f32(float* smem_dst, const float* gmem_base, unsigned index) {
  asm volatile(
      "{\n\t.reg .u64 a;\n\t"
      "mad.wide.u32 a, %2, 4, %1;\n\t"
      "cp.async.ca.shared.global [%0], [a], 4;\n\t}"
      ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(__cvta_generic_to_global(gmem_base)), "r"(index)
      : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void stage_project(const ViewConst& c, const FastParams& p, const float* __restrict__ depth,
                                              const float2 (&x)[kPts], const float2 (&y)[kPts], const float2 (&z)[kPts],
                                              float (&qz_out)[kPts], float* __restrict__ s_slot) {
  asm volatile("" : "+l"(depth));  // keep the view's base pointer in a register pair (one IMAD.WIDE per gather)
  const float2 magic = make_float2(kMagic, kMagic), neg_magic = make_float2(-kMagic, -kMagic);
  const float2 neg_half = make_float2(-0.5f, -0.5f), neg_centre = make_float2(-p.centre.x, -p.centre.y);
#pragma unroll
  for (int k = 0; k < kPts; ++k) {
    // (x, y image rows) two-wide; x[k] = (x, x) etc.
    const float2 qxy = __ffma2_rn(c.Pxy[0], x[k], __ffma2_rn(c.Pxy[1], y[k], __ffma2_rn(c.Pxy[2], z[k], c.Pxy[3])));
    const float qz = fmaf(c.Pz[0], x[k].x, fmaf(c.Pz[1], y[k].x, fmaf(c.Pz[2], z[k].x, c.Pz[3])));
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(qz));
    const float2 rr = make_float2(r, r);
    const float2 uw = __fmul2_rn(qxy, rr);                       // (u~, v~)
    const float2 h = __ffma2_rn(c.nA, rr, p.h0);                 // 0.5 - e per axis (r > 0 whenever the pair is sane)
    const float2 f = __fadd2_rn(__fadd2_rd(uw, magic), neg_magic);  // floor, exact while |u~| < 2^22
    const float tu = uw.x - fabsf(f.x), tv = uw.y - fabsf(f.y);     // fractional part; outside [0, 1) when floor < 0
    const float2 g = __fadd2_rn(make_float2(tu, tv), neg_half);
    const float2 a = __fadd2_rn(f, neg_centre);
    const bool not_near = (fabsf(a.x) > p.near.x) || (fabsf(a.y) > p.near.y);
    const bool frac_ok = (fabsf(g.x) < h.x) && (fabsf(g.y) < h.y);
    const bool decided = (qz >= c.zmin) && (not_near || frac_ok);
    const bool inside = (fabsf(a.x) <= p.centre.x) && (fabsf(a.y) <= p.centre.y);
    // The gather is issued unconditionally (no predicate has to outlive the arithmetic) at a pixel index
    // forced into the image: for a pair inside the image fv * W + fu is an integer-valued float < 2^23
    // whose index is the low mantissa bits of idx + 2^23 (no conversion instruction); anything else
    // (negative, NaN, huge) yields arbitrary bits that the unsigned min clamps to a valid pixel.
    const unsigned pix = min((unsigned)__float_as_int(fmaf(f.y, p.wf, f.x) + 8388608.0f) & 0x7fffffu, p.idx_max);
    cp_async_f32(s_slot + k * kThreads, depth, pix);
    // No flag travels with the gather either. A pixel decided to be outside the image records
    // z = +inf: |depth - inf| fails "<= thr_lo" and passes "> thr_hi" (decided, not visible). An
    // undecided pixel records z = NaN, which fails both tests (-> exact queue), exactly like a NaN
    // depth pixel would.
    qz_out[k] = decided ? (inside ? qz : INFINITY) : __int_as_float(0x7fc00000);
  }
  cp_async_commit();
}

__global__ void __launch_bounds__(kThreads, 3) visibility_filter_kernel(const __grid_constant__ FastParams p) {
  extern __shared__ uint32_t s_dyn[];  // [n_words][kTile] records, [8][kQueue] queues, [3][kTile] gathered depths
  const int scene = p.scene0 + blockIdx.y;
  const int64_t p0 = p.point_off[scene];
  const int64_t n_pts = p.point_off[scene + 1] - p0;
  const int64_t tile0 = (int64_t)blockIdx.x * kTile;
  if (tile0 >= n_pts) return;
  const int n_tile = (int)((n_pts - tile0 < kTile) ? (n_pts - tile0) : kTile);  // valid points of this tile
  const int64_t v0 = p.view_off[scene];
  const int n_views = (int)(p.view_off[scene + 1] - v0);
  const int n_words = (n_views + 31) >> 5;
  uint32_t* s_rec = s_dyn;
  uint32_t* s_queue = s_dyn + (size_t)((p.max_views + 31) >> 5) * kTile + (threadIdx.x >> 5) * kQueue;
  float* s_sensor = reinterpret_cast<float*>(s_dyn + (size_t)((p.max_views + 31) >> 5) * kTile + (kThreads / 32) * kQueue) + threadIdx.x;
  const int lane = threadIdx.x & 31;

  // Slots past the end of the scene re-evaluate its last point (results are never written out), so
  // the loop carries no per-point validity test. Points that must not enter the filter (non-finite
  // or huge coordinates) carry NaN, which fails every comparison and lands in the exact queue.
  float2 x[kPts], y[kPts], z[kPts];  // each coordinate duplicated: operands of the two-wide instructions
  uint32_t word[kPts];
#pragma unroll
  for (int k = 0; k < kPts; ++k) {
    const int local = k * kThreads + threadIdx.x;
    const int64_t orig = p0 + __ldg(p.perm + p0 + tile0 + (local < n_tile ? local : n_tile - 1));
    const float fx = (float)__ldg(p.points + 3 * orig), fy = (float)__ldg(p.points + 3 * orig + 1),
                fz = (float)__ldg(p.points + 3 * orig + 2);
    const bool tame = fabsf(fx) < kHuge && fabsf(fy) < kHuge && fabsf(fz) < kHuge;  // NaN -> false; same rule as the bbox pass
    const float fx_or_nan = tame ? fx : __int_as_float(0x7fc00000);
    x[k] = make_float2(fx_or_nan, fx_or_nan);
    y[k] = make_float2(fy, fy);
    z[k] = make_float2(fz, fz);
    word[k] = 0;
    for (int w = 0; w < n_words; ++w) s_rec[w * kTile + local] = 0;
    for (int g = 0; g < 3; ++g) s_sensor[g * kTile + k * kThreads] = 0.f;  // slots never hold junk NaN/inf patterns
  }
  __syncwarp();
  const int64_t hw = (int64_t)p.height * p.width;
  const ViewConst* cviews = c_views + blockIdx.y * p.max_views;
  const float* depth = p.depths + v0 * hw;
  int qcount = 0;

  // stage B of view v: depth test on the gathers issued three stages earlier, queue pushes, record flush
  auto stage_test = [&](auto may_be_last, int v, const float (&qz)[kPts], const float* __restrict__ s_slot) -> bool {
    const uint32_t bit = 1u << (v & 31);
    const float thr_lo = cviews[v].thr_lo, thr_hi = cviews[v].thr_hi;
    cp_async_wait<2>();  // all but the two most recent groups have landed
    bool und[kPts], any_und = false;
#pragma unroll
    for (int k = 0; k < kPts; ++k) {
      const float delta = fabsf(s_slot[k * kThreads] - qz[k]);
      const bool yes = delta <= thr_lo;
      if (yes) word[k] |= bit;
      und[k] = !yes && !(delta > thr_hi);
      any_und |= und[k];
    }
    if (__any_sync(0xffffffffu, any_und)) {
#pragma unroll
      for (int k = 0; k < kPts; ++k) {
        const bool mine = und[k];
        const unsigned b = __ballot_sync(0xffffffffu, mine);
        if (mine) s_queue[qcount + __popc(b & ((1u << lane) - 1u))] = ((uint32_t)v << 12) | (uint32_t)(k * kThreads + threadIdx.x);
        qcount += __popc(b);
      }
    }
    if ((v & 31) == 31 || (decltype(may_be_last)::value && v == n_views - 1)) {
#pragma unroll
      for (int k = 0; k < kPts; ++k) {
        s_rec[(v >> 5) * kTile + k * kThreads + threadIdx.x] |= word[k];  // warp-private slots: no race with drain's atomicOr
        word[k] = 0;
      }
    }
    return qcount > kQueue - 32 * kPts;  // no room for another view's worth of entries: the caller drains
  };

  // Three gather groups rotate (the loop is unrolled by three): the gathers of view v + 3 are issued
  // right after view v has been tested, two views of arithmetic before they are needed - enough to
  // cover a DRAM miss. Every stage commits exactly one (possibly empty) group, so "all but the two
  // most recent groups" always names the view under test.
  // The exact queue is drained outside the pipelined loop (one call site, no call inside the hot loop): when
  // it fills up, the pipeline is abandoned after the current view, the queue is resolved, and the pipeline
  // restarts at the next view (re-issuing at most two views of gathers - rare: ~0.4 % of the pairs are queued).
  float qa[kPts], qb[kPts], qc[kPts];
  float* const sa = s_sensor;
  float* const sb = s_sensor + kTile;
  float* const sc = s_sensor + 2 * kTile;
  int v_begin = 0;
  for (;;) {
    const float* d = depth + (int64_t)v_begin * hw;
    if (v_begin < n_views) stage_project(cviews[v_begin], p, d, x, y, z, qa, sa); else cp_async_commit();
    if (v_begin + 1 < n_views) stage_project(cviews[v_begin + 1], p, d + hw, x, y, z, qb, sb); else cp_async_commit();
    if (v_begin + 2 < n_views) stage_project(cviews[v_begin + 2], p, d + 2 * hw, x, y, z, qc, sc); else cp_async_commit();
    d += 3 * hw;
    bool full = false;
    int v = v_begin;
    // steady state: six more views exist, no bounds checks on the stages
    for (; v + 5 < n_views; v += 3, d += 3 * hw) {
      if (stage_test(std::false_type{}, v, qa, sa)) { v_begin = v + 1; full = true; break; }
      stage_project(cviews[v + 3], p, d, x, y, z, qa, sa);
      if (stage_test(std::false_type{}, v + 1, qb, sb)) { v_begin = v + 2; full = true; break; }
      stage_project(cviews[v + 4], p, d + hw, x, y, z, qb, sb);
      if (stage_test(std::false_type{}, v + 2, qc, sc)) { v_begin = v + 3; full = true; break; }
      stage_project(cviews[v + 5], p, d + 2 * hw, x, y, z, qc, sc);
    }
    for (; !full && v < n_views; v += 3, d += 3 * hw) {
      if (stage_test(std::true_type{}, v, qa, sa)) { v_begin = v + 1; full = true; break; }
      if (v + 3 < n_views) stage_project(cviews[v + 3], p, d, x, y, z, qa, sa); else cp_async_commit();
      if (v + 1 < n_views && stage_test(std::true_type{}, v + 1, qb, sb)) { v_begin = v + 2; full = true; break; }
      if (v + 4 < n_views) stage_project(cviews[v + 4], p, d + hw, x, y, z, qb, sb); else cp_async_commit();
      if (v + 2 < n_views && stage_test(std::true_type{}, v + 2, qc, sc)) { v_begin = v + 3; full = true; break; }
      if (v + 5 < n_views) stage_project(cviews[v + 5], p, d + 2 * hw, x, y, z, qc, sc); else cp_async_commit();
    }
    cp_async_wait<0>();
    __syncwarp();
    if (qcount > 0)
      drain_queue(s_queue, qcount, n_tile, p.points + 3 * p0, p.perm + p0 + tile0, p.inv_poses + v0 * 16,
                  p.intrinsics + (int64_t)scene * 9, p.depths + v0 * hw, p.width, p.height, p.threshold, s_rec);
    __syncwarp();
    qcount = 0;
    if (!full || v_begin >= n_views) break;
  }
#pragma unroll
  for (int k = 0; k < kPts; ++k) {
    const int local = k * kThreads + threadIdx.x;
    if (local >= n_tile) continue;
    const int64_t s = tile0 + local;
    uint32_t any = 0;
    for (int w = 0; w < n_words; ++w) {
      const uint32_t bits = s_rec[w * kTile + local];
      p.records[(int64_t)w * p.total_points + p0 + s] = bits;
      any |= bits;
    }
    if (p.any_visible) p.any_visible[p0 + __ldg(p.perm + p0 + s)] = any ? 1 : 0;
  }
}

// thread per original point; TOut mask element. kCompact: write only kept points at their rank.
template <typename TOut, bool kCompact>
__global__ void __launch_bounds__(kThreads) unpack_kernel(const uint32_t* __restrict__ records, const int64_t* __restrict__ rank,
                                                          const int64_t* __restrict__ point_off, const int64_t* __restrict__ view_off,
                                                          const int64_t* __restrict__ mask_off, int64_t total_points,
                                                          const uint8_t* __restrict__ any_visible,
                                                          const int64_t* __restrict__ new_index, const int64_t* __restrict__ kept_off,
                                                          TOut* __restrict__ out) {
  const int scene = blockIdx.y;
  const int64_t p0 = point_off[scene];
  const int64_t n = point_off[scene + 1] - p0;
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= n) return;
  if (kCompact && !any_visible[p0 + i]) return;
  const int n_v = (int)(view_off[scene + 1] - view_off[scene]);
  const int64_t s = p0 + rank[p0 + i];
  int64_t stride = n, col = i;
  if (kCompact) {
    const int64_t kept0 = kept_off[scene];
    stride = kept_off[scene + 1] - kept0;
    col = new_index[p0 + i] - kept0;
  }
  TOut* dst = out + mask_off[scene] + col;
  for (int w = 0; w * 32 < n_v; ++w) {
    const uint32_t bits = __ldg(records + (int64_t)w * total_points + s);
    const int lim = min(32, n_v - w * 32);
#pragma unroll 8
    for (int b = 0; b < lim; ++b) dst[(int64_t)(w * 32 + b) * stride] = (TOut)((bits >> b) & 1u);
  }
}



// ---- wide uint8 unpack of the compacted masks -------------------------------------------------------------------
// The thread-per-point kernel above writes one byte per (point, view): 32-byte warp stores, ~5 instructions per byte,
// L2 write transactions at 70 % (ncu). Here a thread owns FOUR consecutive output columns of a scene: the same byte
// of their four record words is gathered into one register (PRMT), one shift + mask then yields the four mask bytes
// of a view as a 32-bit word, and a warp writes 124 contiguous bytes per view with 4-byte stores. Rows of the
// compacted mask start at arbitrary byte addresses (stride = number of kept points), so the word a thread stores is
// funnel-shifted together from its own columns and its right neighbour's (lane 31 of a warp repeats lane 0 of the
// next warp and stores nothing); the few bytes in front of the first aligned word and at the end of a row are
// written one by one.
__global__ void __launch_bounds__(kThreads) kept_positions_kernel(const int64_t* __restrict__ rank, const int64_t* __restrict__ point_off,
                                                                  const uint8_t* __restrict__ any_visible,
                                                                  const int64_t* __restrict__ new_index, uint32_t* __restrict__ src_pos) {
  const int scene = blockIdx.y;
  const int64_t p0 = point_off[scene], n = point_off[scene + 1] - p0;
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= n || !any_visible[p0 + i]) return;
  src_pos[new_index[p0 + i]] = (uint32_t)(p0 + rank[p0 + i]);  // sorted position of the point behind output column new_index
}

__global__ void __launch_bounds__(kThreads) unpack_compact_wide_kernel(const uint32_t* __restrict__ records,
                                                                       const uint32_t* __restrict__ src_pos,
                                                                       const int64_t* __restrict__ view_off,
                                                                       const int64_t* __restrict__ kept_off,
                                                                       const int64_t* __restrict__ out_off, int64_t total_points,
                                                                       uint8_t* __restrict__ out) {
  const int scene = blockIdx.y;
  const int64_t kept0 = kept_off[scene];
  const int64_t n_kept = kept_off[scene + 1] - kept0;
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  const int64_t g = warp * 31 + lane;  // group of four columns; lane 31 repeats lane 0 of the next warp
  if (warp * 31 * 4 >= n_kept) return;  // whole warp beyond the scene
  const int n_v = (int)(view_off[scene + 1] - view_off[scene]);
  const int64_t c0 = 4 * g;
  int64_t pos[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) pos[k] = (c0 + k < n_kept) ? (int64_t)__ldg(src_pos + kept0 + c0 + k) : -1;
  uint8_t* base = out + out_off[scene];
  // Interior warps (every column of the warp and of its right neighbour group exists, and the warp does not hold the
  // row start) run a lean loop: no per-byte code, the address and the funnel shift advance by additions only.
  if (warp > 0 && (warp * 31 + 32) * 4 <= n_kept) {
    uint8_t* ptr = base + c0;                    // my first column in row v (advanced by n_kept per view)
    unsigned low = (unsigned)(uintptr_t)ptr;     // its low address bits: they alone decide the alignment
    const unsigned step = (unsigned)n_kept;
    // one view: my four bytes, my right neighbour's, and the aligned word they form at or after my first column
    // (byte shift by PRMT: selector 0x3210 + 0x1111 * off takes my bytes off..3 and the neighbour's bytes 0..off-1)
    auto emit = [&](uint32_t mine) {
      const uint32_t next = __shfl_down_sync(0xffffffffu, mine, 1);
      const unsigned off = (0u - low) & 3u;
      const uint32_t word = __byte_perm(mine, next, 0x3210u + 0x1111u * off);
      if (lane < 31) *reinterpret_cast<uint32_t*>(ptr + off) = word;
      ptr += n_kept;
      low += step;
    };
    for (int w = 0; w * 32 < n_v; ++w) {
      uint32_t r[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) r[k] = __ldg(records + (int64_t)w * total_points + pos[k]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int left = n_v - (w * 32 + j * 8);  // views left in this byte (warp-uniform)
        if (left <= 0) break;
        const uint32_t lo2 = __byte_perm(r[0], r[1], 0x0040 + j * 0x11);
        const uint32_t hi2 = __byte_perm(r[2], r[3], 0x0040 + j * 0x11);
        const uint32_t packed = __byte_perm(lo2, hi2, 0x5410);
        if (left >= 8) {
#pragma unroll
          for (int i = 0; i < 8; ++i) emit((packed >> i) & 0x01010101u);
        } else {
          for (int i = 0; i < left; ++i) emit((packed >> i) & 0x01010101u);
        }
      }
    }
    return;
  }
  for (int w = 0; w * 32 < n_v; ++w) {
    uint32_t r[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) r[k] = pos[k] >= 0 ? __ldg(records + (int64_t)w * total_points + pos[k]) : 0u;
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
      if (w * 32 + j * 8 >= n_v) break;  // warp-uniform
      // byte j of the four records side by side: bits i of the four bytes are view 32 w + 8 j + i of the four columns
      const uint32_t lo2 = __byte_perm(r[0], r[1], 0x0040 + j * 0x11);  // (r0.byte j, r1.byte j, -, -)
      const uint32_t hi2 = __byte_perm(r[2], r[3], 0x0040 + j * 0x11);
      const uint32_t packed = __byte_perm(lo2, hi2, 0x5410);
#pragma unroll 1
      for (int i = 0; i < 8; ++i) {
        const int v = w * 32 + j * 8 + i;
        if (v >= n_v) break;  // warp-uniform
        const uint32_t mine = (packed >> i) & 0x01010101u;
        const uint32_t next = __shfl_down_sync(0xffffffffu, mine, 1);
        uint8_t* row = base + (int64_t)v * n_kept;
        const int m = (int)((uintptr_t)row & 3);  // misalignment of the row start (warp-uniform)
        if (m == 0) {
          if (lane < 31) {
            if (c0 + 3 < n_kept) *reinterpret_cast<uint32_t*>(row + c0) = mine;
            else
              for (int k = 0; k < 4; ++k)
                if (c0 + k < n_kept) row[c0 + k] = (uint8_t)(mine >> (8 * k));
          }
        } else {
          // aligned word holding columns c0 + 4 - m .. c0 + 7 - m: my last m bytes below my neighbour's first 4 - m
          const uint32_t word = __funnelshift_r(mine, next, 8 * (4 - m));
          const int64_t first = c0 + 4 - m;
          if (lane < 31) {
            if (first + 3 < n_kept) *reinterpret_cast<uint32_t*>(row + first) = word;
            else
              for (int k = 0; k < 4; ++k)
                if (first + k < n_kept) row[first + k] = (uint8_t)(word >> (8 * k));
          }
          if (g == 0)  // the bytes in front of the first aligned word
            for (int k = 0; k < 4 - m; ++k)
              if (k < n_kept) row[k] = (uint8_t)(mine >> (8 * k));
        }
      }
    }
  }
}

// Serialises the users of c_views on one device: holds a process-wide mutex while work is enqueued, makes the
// caller's stream wait for the previous user's last kernel, and records the new "last use" event on release.
struct ConstBankTurn {
  static constexpr int kMaxDevices = 64;
  static std::mutex& mutex() { static std::mutex m; return m; }
  static cudaEvent_t* events() { static cudaEvent_t e[kMaxDevices] = {}; return e; }
  std::unique_lock<std::mutex> lock;
  cudaStream_t stream;
  cudaError_t status = cudaSuccess;
  int device = 0;
  explicit ConstBankTurn(cudaStream_t st) : lock(mutex()), stream(st) {
    status = cudaGetDevice(&device);
    if (status != cudaSuccess) return;
    if (device < 0 || device >= kMaxDevices) { status = cudaErrorInvalidDevice; return; }
    cudaEvent_t& ev = events()[device];
    if (!ev) status = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    else status = cudaStreamWaitEvent(stream, ev, 0);
  }
  // Records the "last use" event. Also runs from the destructor, so an error return between the constructor and the
  // explicit release() still orders the next user of the bank behind the kernels this call did enqueue.
  cudaError_t release() {
    if (released || status != cudaSuccess) return cudaSuccess;
    released = true;
    return cudaEventRecord(events()[device], stream);
  }
  ~ConstBankTurn() { (void)release(); }
  bool released = false;
};

// scenes per filter launch: bounded by the constant bank and by one full wave of CTAs; balanced
int64_t scenes_per_group(int n_scenes, int64_t max_points_per_scene, int max_views_per_scene) {
  const int64_t ctas_per_scene = dc::ceil_div<int64_t>(max_points_per_scene, kTile);
  int64_t group = kConstViews / (max_views_per_scene > 0 ? max_views_per_scene : 1);
  const int64_t wave = ((int64_t)dc::sm_count() * 8) / (ctas_per_scene > 0 ? ctas_per_scene : 1);  // a few CTAs per slot
  if (wave >= 1 && group > wave) group = wave;
  if (group < 1) group = 1;
  const int64_t n_groups = dc::ceil_div<int64_t>(n_scenes, group);
  return dc::ceil_div<int64_t>(n_scenes, n_groups);
}

}  // namespace

extern "C" {

int dc_visibility_sorted_groups(int n_scenes, int64_t max_points_per_scene, int max_views_per_scene) {
  if (n_scenes <= 0 || max_points_per_scene <= 0 || max_views_per_scene <= 0) return 0;
  return (int)dc::ceil_div<int64_t>(n_scenes, scenes_per_group(n_scenes, max_points_per_scene, max_views_per_scene));
}

size_t dc_visibility_sorted_workspace(int64_t total_points, int n_scenes, int max_views_per_scene) {
  return carve(nullptr, total_points, n_scenes > 0 ? n_scenes : 1, max_views_per_scene).total;
}

size_t dc_spatial_sort_workspace(int n_scenes) {
  const size_t ns = (size_t)(n_scenes > 0 ? n_scenes : 1);
  return ((sizeof(float) * 6 * ns + 255) / 256) * 256 + sizeof(int) * (size_t)kCells * ns;
}

int dc_spatial_sort(const double* points, const int64_t* point_off, int n_scenes, int64_t total_points,
                    int64_t max_points_per_scene, int64_t* perm, int64_t* rank, void* workspace, size_t workspace_bytes,
                    dc_stream_t stream) {
  DC_CHECK_ARG(points && point_off && perm && rank && workspace, "dc_spatial_sort: null pointer argument");
  if (n_scenes <= 0 || max_points_per_scene <= 0 || total_points <= 0) return DC_OK;
  DC_CHECK_ARG(n_scenes <= 65535, "dc_spatial_sort: at most 65535 scenes per call");
  if (workspace_bytes < dc_spatial_sort_workspace(n_scenes))
    return dc::fail(DC_ERR_WORKSPACE, "dc_spatial_sort: workspace %zu < %zu", workspace_bytes, dc_spatial_sort_workspace(n_scenes));
  float* bbox = reinterpret_cast<float*>(workspace);
  int* counts = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(workspace) + ((sizeof(float) * 6 * (size_t)n_scenes + 255) / 256) * 256);
  cudaStream_t st = dc::as_stream(stream);
  init_bbox_kernel<<<dc::ceil_div(n_scenes * 6, 128), 128, 0, st>>>(bbox, n_scenes);
  DC_CUDA(cudaMemsetAsync(counts, 0, sizeof(int) * (size_t)kCells * n_scenes, st));
  int64_t chunks = dc::ceil_div<int64_t>(max_points_per_scene, kThreads * 4);
  const int64_t cap = dc::ceil_div<int64_t>((int64_t)dc::sm_count() * 8, n_scenes);
  if (chunks > cap) chunks = cap;
  if (chunks < 1) chunks = 1;
  dim3 g1((unsigned)chunks, (unsigned)n_scenes);
  bbox_kernel<<<g1, kThreads, 0, st>>>(points, point_off, bbox);
  cell_count_kernel<<<g1, kThreads, 0, st>>>(points, point_off, bbox, counts);
  cell_scan_kernel<<<(unsigned)n_scenes, 1024, 0, st>>>(counts);
  cell_scatter_kernel<<<g1, kThreads, 0, st>>>(points, point_off, bbox, counts, perm, rank);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

int dc_project_visibility_sorted(const double* points, const int64_t* point_off, const int64_t* view_off, const float* depths,
                                 const double* inv_poses, const double* intrinsics, int n_scenes, int64_t total_points,
                                 int64_t max_points_per_scene, int max_views_per_scene, int height, int width,
                                 double threshold, uint32_t* records, int64_t* rank, uint8_t* any_visible, void* workspace,
                                 size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(points && point_off && view_off && depths && inv_poses && intrinsics && records && rank && workspace,
               "dc_project_visibility_sorted: null pointer argument");
  DC_CHECK_ARG(height > 0 && width > 0 && (int64_t)height * width < (1ll << 31), "dc_project_visibility_sorted: bad image size");
  if (n_scenes <= 0 || max_points_per_scene <= 0 || total_points <= 0) return DC_OK;
  DC_CHECK_ARG(n_scenes <= 65535, "dc_project_visibility_sorted: at most 65535 scenes per call");
  DC_CHECK_ARG(max_points_per_scene < (1ll << 31), "dc_project_visibility_sorted: at most 2^31 points per scene");
  DC_CHECK_ARG(max_views_per_scene > 0 && max_views_per_scene <= kConstViews && max_views_per_scene < (1 << 20),
               "dc_project_visibility_sorted: 1..%d views per scene (%d)", kConstViews, max_views_per_scene);
  DC_CHECK_ARG((int64_t)height * width <= (1 << 23), "dc_project_visibility_sorted: image too large for the fp32 pixel index");
  const int n_words = (max_views_per_scene + 31) / 32;
  const size_t smem = sizeof(uint32_t) * ((size_t)n_words * kTile + (size_t)(kThreads / 32) * kQueue + 3 * (size_t)kTile);
  DC_CHECK_ARG(smem <= 200 * 1024, "dc_project_visibility_sorted: too many views per scene (%d)", max_views_per_scene);
  SortedWs w = carve(workspace, total_points, n_scenes, max_views_per_scene);
  if (workspace_bytes < w.total)
    return dc::fail(DC_ERR_WORKSPACE, "dc_project_visibility_sorted: workspace %zu < %zu", workspace_bytes, w.total);
  cudaStream_t st = dc::as_stream(stream);
  init_bbox_kernel<<<dc::ceil_div(n_scenes * 6, 128), 128, 0, st>>>(w.bbox, n_scenes);
  DC_CUDA(cudaMemsetAsync(w.counts, 0, sizeof(int) * (size_t)kCells * n_scenes, st));
  int64_t chunks = dc::ceil_div<int64_t>(max_points_per_scene, kThreads * 4);
  const int64_t cap = dc::ceil_div<int64_t>((int64_t)dc::sm_count() * 8, n_scenes);
  if (chunks > cap) chunks = cap;
  if (chunks < 1) chunks = 1;
  dim3 g1((unsigned)chunks, (unsigned)n_scenes);
  bbox_kernel<<<g1, kThreads, 0, st>>>(points, point_off, w.bbox);
  cell_count_kernel<<<g1, kThreads, 0, st>>>(points, point_off, w.bbox, w.counts);
  cell_scan_kernel<<<(unsigned)n_scenes, 1024, 0, st>>>(w.counts);
  cell_scatter_kernel<<<g1, kThreads, 0, st>>>(points, point_off, w.bbox, w.counts, w.perm, rank);
  ViewConst* vc = reinterpret_cast<ViewConst*>(w.view_consts);
  camera_prep_kernel<<<dc::ceil_div(n_scenes * max_views_per_scene, 128), 128, 0, st>>>(
      inv_poses, intrinsics, view_off, w.bbox, n_scenes, max_views_per_scene, height, width, threshold, vc);
  DC_LAUNCH_CHECK();
  static dc::FuncAttrCache smem_attr, carve_attr;
  if (smem > 48 * 1024) DC_CUDA(smem_attr.set(visibility_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // two-stream mode: the instance-histogram ring kernel of the object branch (csrc/seg_table.cu) shares the SMs with this
  // kernel, and an SM cannot change its shared-memory carve-out while CTAs are resident: both ask for the same one
  DC_CUDA(carve_attr.set(visibility_filter_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                         dc::stream_overlap() ? dc::kOverlapCarveoutPct : cudaSharedmemCarveoutDefault));
  // The per-view constants live in the constant bank (uniform operands instead of 24 shared-memory
  // wavefronts per view and warp), refreshed per group of scenes by a device-to-device copy in
  // stream order. A group is at most one full wave of CTAs.
  const int64_t ctas_per_scene = dc::ceil_div<int64_t>(max_points_per_scene, kTile);
  const int64_t group = scenes_per_group(n_scenes, max_points_per_scene, max_views_per_scene);
  // The constant bank is one per device: calls on different streams (or from different host threads) take
  // turns on it. The lock covers the enqueue, the event chain covers the execution on the device.
  ConstBankTurn turn(st);
  if (turn.status != cudaSuccess) return dc::fail(DC_ERR_CUDA, "dc_project_visibility_sorted: %s", cudaGetErrorString(turn.status));
  for (int s0 = 0; s0 < n_scenes; s0 += (int)group) {
    const int ns = (int)((n_scenes - s0 < group) ? (n_scenes - s0) : group);
    DC_CUDA(cudaMemcpyToSymbolAsync(c_views, vc + (size_t)s0 * max_views_per_scene,
                                    sizeof(ViewConst) * (size_t)ns * max_views_per_scene, 0, cudaMemcpyDeviceToDevice, st));
    FastParams p{points, point_off, view_off, depths, inv_poses, intrinsics, w.perm, total_points, s0,
                 max_views_per_scene, height, width, (float)width, (unsigned)((int64_t)height * width - 1),
                 make_float2(0.5f * (float)(width - 1), 0.5f * (float)(height - 1)),
                 make_float2((float)near_limit(width), (float)near_limit(height)),
                 make_float2((float)(0.499999 - 1.02 * 5.0 * 5.9604644775390625e-08 * coord_bound(width)),
                             (float)(0.499999 - 1.02 * 5.0 * 5.9604644775390625e-08 * coord_bound(height))),
                 threshold, records, any_visible};
    dim3 grid((unsigned)ctas_per_scene, (unsigned)ns);
    visibility_filter_kernel<<<grid, kThreads, smem, st>>>(p);
  }
  DC_LAUNCH_CHECK();
  DC_CUDA(turn.release());
  return DC_OK;
}

int dc_unpack_visibility(const uint32_t* records, const int64_t* rank, const int64_t* point_off, const int64_t* view_off,
                         const int64_t* mask_off, int n_scenes, int64_t total_points, int64_t max_points_per_scene, void* mask,
                         int mask_elem_size, dc_stream_t stream) {
  DC_CHECK_ARG(records && rank && point_off && view_off && mask_off && mask, "dc_unpack_visibility: null pointer argument");
  DC_CHECK_ARG(mask_elem_size == 1 || mask_elem_size == 8, "dc_unpack_visibility: mask_elem_size must be 1 or 8");
  if (n_scenes <= 0 || max_points_per_scene <= 0) return DC_OK;
  dim3 grid((unsigned)dc::ceil_div<int64_t>(max_points_per_scene, kThreads), (unsigned)n_scenes);
  cudaStream_t st = dc::as_stream(stream);
  if (mask_elem_size == 1)
    unpack_kernel<uint8_t, false><<<grid, kThreads, 0, st>>>(records, rank, point_off, view_off, mask_off, total_points, nullptr,
                                                             nullptr, nullptr, (uint8_t*)mask);
  else
    unpack_kernel<long long, false><<<grid, kThreads, 0, st>>>(records, rank, point_off, view_off, mask_off, total_points, nullptr,
                                                               nullptr, nullptr, (long long*)mask);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

size_t dc_unpack_compact_workspace(int64_t total_points, int out_elem_size) {
  return out_elem_size == 1 && total_points > 0 ? sizeof(uint32_t) * (size_t)total_points : 0;
}

int dc_unpack_visibility_compact(const uint32_t* records, const int64_t* rank, const int64_t* point_off, const int64_t* view_off,
                                 const uint8_t* any_visible, const int64_t* new_index, const int64_t* kept_off,
                                 const int64_t* out_off, int n_scenes, int64_t total_points, int64_t max_points_per_scene,
                                 void* out, int out_elem_size, void* workspace, size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(records && rank && point_off && view_off && any_visible && new_index && kept_off && out_off && out,
               "dc_unpack_visibility_compact: null pointer argument");
  DC_CHECK_ARG(out_elem_size == 1 || out_elem_size == 8, "dc_unpack_visibility_compact: out_elem_size must be 1 or 8");
  if (n_scenes <= 0 || max_points_per_scene <= 0) return DC_OK;
  dim3 grid((unsigned)dc::ceil_div<int64_t>(max_points_per_scene, kThreads), (unsigned)n_scenes);
  cudaStream_t st = dc::as_stream(stream);
  const size_t need = dc_unpack_compact_workspace(total_points, out_elem_size);
  const bool wide = out_elem_size == 1 && workspace && workspace_bytes >= need && total_points < (1ll << 32) &&
                    ((uintptr_t)out & 3) == 0;
  if (wide) {
    uint32_t* src_pos = static_cast<uint32_t*>(workspace);
    kept_positions_kernel<<<grid, kThreads, 0, st>>>(rank, point_off, any_visible, new_index, src_pos);
    DC_LAUNCH_CHECK();
    const int64_t groups = dc::ceil_div<int64_t>(max_points_per_scene, 4);
    const int64_t warps = dc::ceil_div<int64_t>(groups, 31);
    dim3 wgrid((unsigned)dc::ceil_div<int64_t>(warps, kThreads / 32), (unsigned)n_scenes);
    unpack_compact_wide_kernel<<<wgrid, kThreads, 0, st>>>(records, src_pos, view_off, kept_off, out_off, total_points, (uint8_t*)out);
  } else if (out_elem_size == 1)
    unpack_kernel<uint8_t, true><<<grid, kThreads, 0, st>>>(records, rank, point_off, view_off, out_off, total_points, any_visible,
                                                            new_index, kept_off, (uint8_t*)out);
  else
    unpack_kernel<long long, true><<<grid, kThreads, 0, st>>>(records, rank, point_off, view_off, out_off, total_points, any_visible,
                                                              new_index, kept_off, (long long*)out);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

}  // extern "C"
