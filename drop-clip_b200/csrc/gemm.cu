// (3) view scoring and (6) grounding: operand preparation, tcgen05 GEMM launches and epilogues.
//
// Reference: utils/feature_fusion.py:311-313 (feat_v_norm @ query.T), models/similarity.py:28-101
// (vis_feats @ text.T, paired softmax, min-max, threshold), engine/distil.py:244-246.
#include <algorithm>
#include <cstring>
#include <mutex>
#include <type_traits>
#include <vector>

#include "gemm.cuh"

namespace dc {
namespace gemm {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  return fn;
}

int encode_plane_map(CUtensorMap* out, const void* base, int64_t rows, int k, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(DC_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  if (((uintptr_t)base & 15) != 0) return fail(DC_ERR_INVALID, "GEMM operand plane must be 16-byte aligned");
  if (rows < 1) rows = 1;
  cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)k * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DC_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return DC_OK;
}

}  // namespace gemm
}  // namespace dc

namespace {

using dc::gemm::Params;
using dc::gemm::Tile;

// ---------------------------------------------------------------------------- row normalisation
// One warp per row. torch semantics per dtype:
//   fp16: norm = fp16(sqrt(sum x^2)); y = fp16(float(x) / float(norm))       (rounded twice)
//   fp32: norm = sqrt(sum x^2);       y = x / norm
// The sum of squares is accumulated in fp64, so the norm is the CORRECTLY ROUNDED one. torch accumulates in fp32
// in an order that depends on the kernel (CPU vector width / CUDA block shape); its fp16 norm then lands on the
// neighbouring fp16 value whenever the exact norm sits within ~1e-7 of a rounding boundary - 3.5 rows in 10 000
// (measured: 70 of 200 000 random 768-d rows), and such a flip moves every similarity of the row by 5e-4. No fp32
// order can follow all of torch's builds; the exactly rounded norm is the value they all approximate.
// Writes y back in place when `normalize`, and the fp16 operand planes when requested.
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <typename T>
__device__ __forceinline__ float rounded_norm(double sum_sq) {
  const double nrm = sqrt(sum_sq);
  return sizeof(T) == 2 ? __half2float(__double2half(nrm)) : (float)nrm;
}
template <typename T, bool kInPlace>
__global__ void __launch_bounds__(256) row_normalize_kernel(T* __restrict__ x, int64_t n_rows, int dim, int normalize,
                                                            __half* __restrict__ hi, __half* __restrict__ lo) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int lane = threadIdx.x & 31;
  T* xr = x + row * dim;
  float inv_scale_num = 1.f;  // divide by this
  if (normalize) {
    double ss = 0.0;
    for (int c = lane; c < dim; c += 32) {
      const double v = (double)(float)xr[c];
      ss = fma(v, v, ss);
    }
    inv_scale_num = rounded_norm<T>(warp_sum_f64(ss));
  }
  for (int c = lane; c < dim; c += 32) {
    float v = (float)xr[c];
    if (normalize) {
      v = v / inv_scale_num;  // IEEE division, like torch
      if (sizeof(T) == 2) v = __half2float(__float2half_rn(v));
      if (kInPlace) xr[c] = (T)v;
    }
    if (hi) {
      const __half h = __float2half_rn(v);
      hi[row * dim + c] = h;
      if (lo) lo[row * dim + c] = __float2half_rn(v - __half2float(h));
    }
  }
}

// Same arithmetic, organised for bandwidth: a warp keeps its whole row in registers (128-bit loads,
// kChunks x 8 fp16 or kChunks x 4 fp32 per lane), reduces, scales and writes it back once. Used when
// dim == 32 * kChunks * (16 / sizeof(T)) and the rows are 16-byte aligned (dim = 768: fp16 3 chunks,
// fp32 6 chunks). The generic kernel above reads the row twice with 2- or 4-byte accesses.
template <typename T, bool kInPlace, int kChunks>
__global__ void __launch_bounds__(256) row_normalize_vec_kernel(T* __restrict__ x, int64_t n_rows, int normalize,
                                                                __half* __restrict__ hi, __half* __restrict__ lo) {
  constexpr int kPer = 16 / (int)sizeof(T);       // elements per 128-bit access
  constexpr int kDim = 32 * kChunks * kPer;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int lane = threadIdx.x & 31;
  T* xr = x + row * kDim;
  float v[kChunks][kPer];
#pragma unroll
  for (int k = 0; k < kChunks; ++k) {
    const int4 raw = dc::ld_stream(reinterpret_cast<const int4*>(xr) + k * 32 + lane);
    if (sizeof(T) == 2) {
      const __half2* h2 = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(h2[j]);
        v[k][2 * j] = f.x;
        v[k][2 * j + 1] = f.y;
      }
    } else {
      const float* f = reinterpret_cast<const float*>(&raw);
#pragma unroll
      for (int j = 0; j < kPer; ++j) v[k][j] = f[j];
    }
  }
  if (normalize) {
    float nrm;
    bool exact = false;
    if (sizeof(T) == 2) {
      // fp16 rows: the squares are exact in fp32 (11-bit significands) and every partial sum is positive, so an fp32
      // accumulation (4 chains + 5 shuffle rounds) + sqrt stays within 20 eps = 1.2e-6 of the exact norm. If both ends of
      // that interval round to the same fp16 value (99 % of the rows), it IS the correctly rounded norm; otherwise the
      // fp64 accumulation below decides. (The fp64 chain on every row cost 25 % of this kernel's time.)
      float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < kChunks; ++k)
#pragma unroll
        for (int j = 0; j < kPer; ++j) s[j & 3] = fmaf(v[k][j], v[k][j], s[j & 3]);
      const float tot = dc::warp_sum((s[0] + s[1]) + (s[2] + s[3]));
      const float n32 = sqrtf(tot);
      const __half lo = __float2half_rn(n32 * (1.0f - 1.5e-6f)), hi = __float2half_rn(n32 * (1.0f + 1.5e-6f));
      nrm = __half2float(lo);
      exact = (__half_as_ushort(lo) == __half_as_ushort(hi)) && n32 < 60000.f && tot > 1e-12f;
    }
    if (!exact) {
      double ss = 0.0;
#pragma unroll
      for (int k = 0; k < kChunks; ++k)
#pragma unroll
        for (int j = 0; j < kPer; ++j) ss = fma((double)v[k][j], (double)v[k][j], ss);
      nrm = rounded_norm<T>(warp_sum_f64(ss));
    }
    if (sizeof(T) == 2 && nrm > 0.f && nrm < INFINITY) {
      // x / nrm correctly rounded without the division sequence: with the correctly rounded reciprocal r, q = x * r, the
      // exact remainder x - q * nrm and one fma give RN(x / nrm) (Markstein; nrm is an fp16 value, so its significand is
      // never all ones; quotients of fp16 values never leave the fp32 normal range)
      const float r = 1.0f / nrm;
#pragma unroll
      for (int k = 0; k < kChunks; ++k)
#pragma unroll
        for (int j = 0; j < kPer; ++j) {
          const float q0 = v[k][j] * r;
          // copysign: (+0) + (-0) = +0 in the last fma would lose the sign of a -0 entry (IEEE division keeps it)
          v[k][j] = copysignf(__half2float(__float2half_rn(fmaf(fmaf(-q0, nrm, v[k][j]), r, q0))), v[k][j]);
        }
    } else {
#pragma unroll
      for (int k = 0; k < kChunks; ++k)
#pragma unroll
        for (int j = 0; j < kPer; ++j) {
          float q = v[k][j] / nrm;  // IEEE division, like torch
          if (sizeof(T) == 2) q = __half2float(__float2half_rn(q));
          v[k][j] = q;
        }
    }
  }
#pragma unroll
  for (int k = 0; k < kChunks; ++k) {
    if (sizeof(T) == 2) {
      int4 packed;
      __half2* h2 = reinterpret_cast<__half2*>(&packed);
#pragma unroll
      for (int j = 0; j < 4; ++j) h2[j] = __floats2half2_rn(v[k][2 * j], v[k][2 * j + 1]);
      if (normalize && kInPlace) dc::st_stream(reinterpret_cast<int4*>(xr) + k * 32 + lane, packed);
      if (hi) dc::st_stream(reinterpret_cast<int4*>(hi + row * kDim) + k * 32 + lane, packed);
    } else {
      if (normalize && kInPlace) {
        int4 packed;
        float* f = reinterpret_cast<float*>(&packed);
#pragma unroll
        for (int j = 0; j < kPer; ++j) f[j] = v[k][j];
        dc::st_stream(reinterpret_cast<int4*>(xr) + k * 32 + lane, packed);
      }
      if (hi) {
        // 4 fp32 -> 4 fp16 (+ 4 fp16 residuals): 8-byte stores, still fully coalesced per warp
        __half2 h[2], l[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          h[j] = __floats2half2_rn(v[k][2 * j], v[k][2 * j + 1]);
          const float2 back = __half22float2(h[j]);
          l[j] = __floats2half2_rn(v[k][2 * j] - back.x, v[k][2 * j + 1] - back.y);
        }
        *reinterpret_cast<uint2*>(hi + row * kDim + (k * 32 + lane) * 4) = *reinterpret_cast<uint2*>(h);
        if (lo) *reinterpret_cast<uint2*>(lo + row * kDim + (k * 32 + lane) * 4) = *reinterpret_cast<uint2*>(l);
      }
    }
  }
}

int launch_row_normalize(void* x, int dtype, int64_t n_rows, int dim, int normalize, bool in_place, void* hi, void* lo,
                         cudaStream_t st) {
  if (n_rows <= 0) return DC_OK;
  const unsigned grid = (unsigned)dc::ceil_div<int64_t>(n_rows, 8);
  const bool aligned = ((uintptr_t)x & 15) == 0 && ((uintptr_t)hi & 15) == 0 && ((uintptr_t)lo & 15) == 0;
  if (aligned && dim == 768) {  // the CLIP ViT-L/14 width of every caller (models/features/clip); other widths: generic kernel
    __half* h = (__half*)hi;
    __half* l = (__half*)lo;
    if (dtype == DC_F16) {
      if (in_place) row_normalize_vec_kernel<__half, true, 3><<<grid, 256, 0, st>>>((__half*)x, n_rows, normalize, h, nullptr);
      else row_normalize_vec_kernel<__half, false, 3><<<grid, 256, 0, st>>>((__half*)x, n_rows, normalize, h, nullptr);
    } else {
      if (in_place) row_normalize_vec_kernel<float, true, 6><<<grid, 256, 0, st>>>((float*)x, n_rows, normalize, h, l);
      else row_normalize_vec_kernel<float, false, 6><<<grid, 256, 0, st>>>((float*)x, n_rows, normalize, h, l);
    }
    DC_LAUNCH_CHECK();
    return DC_OK;
  }
  if (dtype == DC_F16) {
    if (in_place) row_normalize_kernel<__half, true><<<grid, 256, 0, st>>>((__half*)x, n_rows, dim, normalize, (__half*)hi, nullptr);
    else row_normalize_kernel<__half, false><<<grid, 256, 0, st>>>((__half*)x, n_rows, dim, normalize, (__half*)hi, nullptr);
  } else {
    if (in_place) row_normalize_kernel<float, true><<<grid, 256, 0, st>>>((float*)x, n_rows, dim, normalize, (__half*)hi, (__half*)lo);
    else row_normalize_kernel<float, false><<<grid, 256, 0, st>>>((float*)x, n_rows, dim, normalize, (__half*)hi, (__half*)lo);
  }
  DC_LAUNCH_CHECK();
  return DC_OK;
}

// ---------------------------------------------------------------------------- epilogues
// raw store: out[row, col] for valid rows/cols
struct EpiStore {
  float* out;
  int ld;
  __device__ __forceinline__ void row(const Tile& t, int r, int c0, const float (&v)[32]) {
    if (r >= t.rows) return;
    float* dst = out + (int64_t)(t.a_row + r) * ld + c0;
    const int n = min(32, min(t.cols, ld) - c0);
    if (n == 32 && (ld & 3) == 0) {
#pragma unroll
      for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (i < n) dst[i] = v[i];
    }
  }
  __device__ __forceinline__ void begin(const Tile&, int, float) {}
  __device__ __forceinline__ void finish(const Tile&, int, int, int, float*) {}
};

__device__ __forceinline__ void atomic_min_f(float* a, float v) {
  v += 0.0f;
  if (v >= 0) atomicMin(reinterpret_cast<int*>(a), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned*>(a), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f(float* a, float v) {
  v += 0.0f;
  if (v >= 0) atomicMax(reinterpret_cast<int*>(a), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned*>(a), __float_as_uint(v));
}

// Grounding epilogue. A thread owns one point (row) and one half of the prompt axis, walked in
// 32-column chunks, so the N x P similarity matrix never leaves the SM unless mode == RAW. The two
// halves of a row meet in shared memory (finish).
//   paired:  out = 1 / (Nneg + sum_neg exp((neg - pos) / T))   (closed form of models/similarity.py:51-61)
//   argmax:  out = pos - mean(neg), pred = (pos >= max(neg))    (:91-101)
// exp is evaluated as ex2((v - pos) * log2(e) / T) with four independent partial sums; a result below
// 2^-126 flushes to zero and one above 2^128 gives inf -> out = 0, the limits of the closed form.
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct EpiGround {
  int mode;
  int n_prompts;   // columns of THIS launch (<= 256)
  float inv_temp;
  float* out;
  int out_ld;
  uint8_t* pred;
  float* minmax;  // [0] min(out) [1] max(out) [2] min(raw) [3] max(raw)
  // prompt axis cut into blocks of <= 256 columns (one launch each): this launch covers the global columns
  // [col_base, col_base + n_prompts) of n_total; `carry` [n_points, 4] hands (pos, partial sum, running max, arg max)
  // from block to block, the last block finishes the row. One block: col_base = 0, last = 1, carry unused.
  int col_base, n_total, last;
  float* carry;
  int64_t* argmax_idx;  // DC_GROUND_CLASS: index of the row maximum (torch.max(sims, 1)[1], engine/distil.py:290)
  // per-thread running state
  float pos, scale, bias, acc[4], neg_max, raw_min, raw_max;
  int best_idx;

  __device__ __forceinline__ void begin(const Tile& t, int r, float col0) {
    pos = col0;
    if (col_base > 0 && mode != DC_GROUND_RAW && mode != DC_GROUND_CLASS)
      pos = (r < t.rows) ? carry[((int64_t)t.a_row + r) * 4] : 0.f;
    scale = inv_temp * 1.4426950408889634f;  // log2(e) / T
    bias = -pos * scale;
    acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
    neg_max = -INFINITY;
    raw_min = INFINITY;
    raw_max = -INFINITY;
    best_idx = 0x7fffffff;
  }

  template <bool kMasked>
  __device__ __forceinline__ void chunk(int c0, const float (&v)[32]) {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const bool valid = !kMasked || (c0 + i < n_prompts);
      const bool neg = !kMasked || (valid && col_base + c0 + i > 0);
      if (valid) {
        raw_min = fminf(raw_min, v[i]);
        raw_max = fmaxf(raw_max, v[i]);
      }
      if (neg) {
        if (mode == DC_GROUND_PAIRED) acc[i & 3] += ex2_approx(fmaf(v[i], scale, bias));
        else { acc[i & 3] += v[i]; neg_max = fmaxf(neg_max, v[i]); }
      }
    }
  }

  __device__ __forceinline__ void row(const Tile& t, int r, int c0, const float (&v)[32]) {
    if (r >= t.rows) return;
    if (mode == DC_GROUND_RAW || mode == DC_GROUND_CLASS) {
      const int n = min(32, n_prompts - c0);
      if (mode == DC_GROUND_CLASS) {
        // first index of the maximum; a NaN is the maximum (torch.max propagates NaN)
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < n) {
            const bool take = (v[i] > neg_max) || (v[i] != v[i] && neg_max == neg_max) || best_idx == 0x7fffffff;
            if (take) { neg_max = v[i]; best_idx = col_base + c0 + i; }
          }
      }
      if (out) {
        float* dst = out + (int64_t)(t.a_row + r) * out_ld + c0;
        if (n == 32 && (out_ld & 3) == 0 && ((uintptr_t)out & 15) == 0) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < n) dst[i] = v[i];
        }
      }
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (i < n) {
          raw_min = fminf(raw_min, v[i]);
          raw_max = fmaxf(raw_max, v[i]);
        }
      return;
    }
    if ((c0 > 0 || col_base > 0) && c0 + 32 <= n_prompts) chunk<false>(c0, v);  // interior chunk: no masks
    else chunk<true>(c0, v);                                                     // holds the positive column or the ragged end
  }

  __device__ __forceinline__ void finish(const Tile& t, int r, int half, int n_halves, float* scratch) {
    float sum = (acc[0] + acc[1]) + (acc[2] + acc[3]);
    if (n_halves == 2) {
      // half 1 hands its partials to half 0 through shared memory; barrier 1 is private to the 8 epilogue warps
      float* slot = scratch + r * 8;
      asm volatile("bar.sync 1, 256;" ::: "memory");  // previous tile's readers are done with the scratch
      if (half == 1) {
        slot[0] = sum;
        slot[1] = neg_max;
        slot[2] = raw_min;
        slot[3] = raw_max;
        slot[4] = __int_as_float(best_idx);
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (half == 1) return;
      sum += slot[0];
      if (mode == DC_GROUND_CLASS) {  // half 1 holds the higher indices: it wins only with a strictly larger value (or a NaN)
        const float o_max = slot[1];
        const int o_idx = __float_as_int(slot[4]);
        if (o_idx != 0x7fffffff && (best_idx == 0x7fffffff || o_max > neg_max || (o_max != o_max && neg_max == neg_max))) {
          neg_max = o_max;
          best_idx = o_idx;
        }
      } else {
        neg_max = fmaxf(neg_max, slot[1]);
      }
      raw_min = fminf(raw_min, slot[2]);
      raw_max = fmaxf(raw_max, slot[3]);
    }
    const bool have = r < t.rows;
    const int64_t gr = (int64_t)t.a_row + r;
    if (have && carry && mode != DC_GROUND_RAW) {
      float* cr = carry + gr * 4;
      if (col_base > 0) {
        if (mode == DC_GROUND_CLASS) {  // earlier blocks hold the lower indices
          const float p_max = cr[2];
          const int p_idx = __float_as_int(cr[3]);
          if (!(neg_max > p_max || (neg_max != neg_max && p_max == p_max))) { neg_max = p_max; best_idx = p_idx; }
        } else {
          sum += cr[1];
          neg_max = fmaxf(neg_max, cr[2]);
        }
      }
      if (!last) {
        cr[0] = pos;
        cr[1] = sum;
        cr[2] = neg_max;
        cr[3] = __int_as_float(best_idx);
      }
    }
    float o = 0.f;
    const bool final_row = have && last;
    if (final_row && mode == DC_GROUND_CLASS) argmax_idx[gr] = best_idx;
    if (final_row && (mode == DC_GROUND_PAIRED || mode == DC_GROUND_ARGMAX)) {
      const float n_neg = (float)(n_total - 1);
      if (mode == DC_GROUND_PAIRED) {
        o = 1.f / (n_neg + sum);
        if (o != o) o = 0.f;  // nan_to_num
      } else {
        o = pos - sum / n_neg;
        pred[gr] = (pos >= neg_max) ? 1 : 0;  // argmax == 0 (first index wins ties)
      }
      out[gr] = o;
    }
    const bool raw_like = (mode == DC_GROUND_RAW || mode == DC_GROUND_CLASS);
    float a = INFINITY, b = -INFINITY, c = INFINITY, d = -INFINITY;
    if (have) {
      if (raw_like) { a = raw_min; b = raw_max; }
      else if (last) { a = o; b = o; }
      c = raw_min;
      d = raw_max;
    }
    a = dc::warp_min(a); b = dc::warp_max(b); c = dc::warp_min(c); d = dc::warp_max(d);
    if ((threadIdx.x & 31) == 0) {
      if (a != INFINITY) atomic_min_f(minmax + 0, a);
      if (b != -INFINITY) atomic_max_f(minmax + 1, b);
      if (c != INFINITY) atomic_min_f(minmax + 2, c);
      if (d != -INFINITY) atomic_max_f(minmax + 3, d);
    }
  }
};

// ---------------------------------------------------------------------------- view-score helpers
// Tile list: every scene's feature rows cut into 128-row tiles, B tile = that scene's queries.
__global__ void __launch_bounds__(1024) build_score_tiles_kernel(const int64_t* __restrict__ feat_off, const int64_t* __restrict__ view_off,
                                                                 const int64_t* __restrict__ query_off, int n_scenes,
                                                                 int4* __restrict__ tiles, int* __restrict__ tile_count, int max_tiles) {
  // one CTA: thread s owns scenes s, s + 1024, ...; an inclusive block scan of the per-thread tile counts gives
  // every scene its slot range (the single-thread version of this loop cost 53 us for 64 scenes: two dependent
  // global loads per scene, serialised)
  __shared__ int s_scan[1024];
  const int t = threadIdx.x;
  int mine = 0;
  for (int s = t; s < n_scenes; s += 1024) {
    const int64_t r0 = feat_off[view_off[s]], r1 = feat_off[view_off[s + 1]];
    mine += (int)((r1 - r0 + dc::gemm::kBlockM - 1) / dc::gemm::kBlockM);
  }
  s_scan[t] = mine;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int add = t >= o ? s_scan[t - o] : 0;
    __syncthreads();
    s_scan[t] += add;
    __syncthreads();
  }
  // tiles are listed thread-major (thread 0's scenes first); the GEMM treats tiles independently, so the
  // order only matters for load balance
  int n = s_scan[t] - mine;
  for (int s = t; s < n_scenes; s += 1024) {
    const int64_t r0 = feat_off[view_off[s]], r1 = feat_off[view_off[s + 1]];
    const int q = (int)(query_off[s + 1] - query_off[s]);
    for (int64_t r = r0; r < r1; r += dc::gemm::kBlockM) {
      if (n < max_tiles) tiles[n] = make_int4((int)r, (int)query_off[s], (int)min((int64_t)dc::gemm::kBlockM, r1 - r), q);
      ++n;
    }
  }
  if (t == 1023) *tile_count = s_scan[1023] < max_tiles ? s_scan[1023] : max_tiles;
}

// One warp per view: global min/max of the view's (rows x Q) block, then the weight of each bound row.
__global__ void __launch_bounds__(128) view_weights_kernel(
    const float* __restrict__ sims, int sims_ld, const int64_t* __restrict__ feat_off, const int32_t* __restrict__ view_scene,
    const int64_t* __restrict__ view_off, const int64_t* __restrict__ query_off, const int64_t* __restrict__ wobj_off,
    const int32_t* __restrict__ row_object, const uint32_t* __restrict__ counts, int nbins, int64_t total_views,
    int sim_kernel, int use_visibility, float* __restrict__ weight_obj, float* __restrict__ view_minmax,
    int* __restrict__ refine_list, float refine_below) {
  const int64_t g = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (g >= total_views) return;
  const int lane = threadIdx.x & 31;
  const int s = view_scene[g];
  const int n_q = (int)(query_off[s + 1] - query_off[s]);
  const int n_v = (int)(view_off[s + 1] - view_off[s]);
  const int v_local = (int)(g - view_off[s]);
  const int64_t r0 = feat_off[g], r1 = feat_off[g + 1];
  float* w_scene = weight_obj + wobj_off[s];
  float mn = INFINITY, mx = -INFINITY;
  bool any_nan = false;
  if (sim_kernel != DC_SIM_NONE) {
    const int64_t cells = (r1 - r0) * n_q;
    for (int64_t i = lane; i < cells; i += 32) {
      const float v = sims[(r0 + i / n_q) * sims_ld + (i % n_q)];
      any_nan |= (v != v);
      mn = fminf(mn, v);
      mx = fmaxf(mx, v);
    }
    mn = dc::warp_min(mn);
    mx = dc::warp_max(mx);
    any_nan = __any_sync(0xffffffffu, any_nan);
    if (any_nan) mn = mx = __int_as_float(0x7fc00000);  // torch min()/max() propagate NaN
    if (view_minmax && lane == 0) {
      view_minmax[2 * g] = mn;
      view_minmax[2 * g + 1] = mx;
    }
  }
  const float range = mx - mn;
  for (int64_t r = r0 + lane; r < r1; r += 32) {
    const int obj = row_object[r];
    if (obj < 0) continue;
    float w = 1.0f;
    if (use_visibility) w = (float)counts[g * nbins + obj];
    if (sim_kernel != DC_SIM_NONE) {
      const float* srow = sims + r * sims_ld;
      const float pos = (srow[obj] - mn) / range;
      float red = (sim_kernel == DC_SIM_MAX) ? -INFINITY : 0.f;
      bool nan_seen = false;
      for (int o = 0; o < n_q; ++o) {
        if (o == obj) continue;
        const float v = (srow[o] - mn) / range;
        nan_seen |= (v != v);
        if (sim_kernel == DC_SIM_MAX) red = fmaxf(red, v);
        else red += v;
      }
      if (sim_kernel == DC_SIM_MEAN) red = red / (float)(n_q - 1);
      if (nan_seen) red = __int_as_float(0x7fc00000);
      w = pos - red;
      // torch.clip(x, min=eps): NaN stays NaN
      if (w == w) w = fmaxf(w, 1e-6f);
      // rows whose weight the GEMM's ~1e-7 of absolute noise does not resolve: queued for refine_weights_kernel
      if (refine_list && !(w >= refine_below)) {
        const int slot = atomicAdd(refine_list, 1);
        refine_list[1 + 2 * slot] = (int)r;
        refine_list[2 + 2 * slot] = (int)g;
      }
    }
    w_scene[(int64_t)obj * n_v + v_local] = w;
  }
}

// Exact similarity weights (second pass, one warp per feature row). The weight clip(pos - max|mean(neg), 1e-6) of
// the min-max normalised similarities equals (s_pos - red(s_neg)) / (max - min): the view's minimum cancels, the range
// only scales. What needs precision is the DIFFERENCE of two cosines ~1: the tensor-core GEMM (and the reference's own
// fp32 sgemm) carry ~1e-7 of absolute noise, which is a relative error of 10 % on a weight next to the 1e-6 clip, and
// the fused feature of an object whose views all score that low is a mean under such weights (measured at V = 73:
// 3e-3 off the reference on one object row, the reference itself being that far from the exact value of its own
// formulas). So the GEMM's similarities only SELECT here: the positive and every negative within `tol` of the
// arg-max (all negatives for the mean kernel) are re-evaluated as fp64 dot products of the normalised feature row
// (normalised the way torch does per dtype, like row_normalize_kernel) with the queries, and the weight is formed in
// fp64 and rounded once.
// `normed`: the fp16 plane of normalised rows dc_view_score left in its workspace (fp16 features: exactly the values
// the reference multiplies; then no norm and no division here) or nullptr (fp32 features: the row is normalised here
// from `feats`). kVec: dim is a multiple of 256 and the rows are 16-byte aligned - a lane owns 8 consecutive channels
// of every 256-channel chunk (128-bit loads). Only rows whose GEMM weight is below `refine_below` are re-evaluated
// (view_weights_kernel queues them): the GEMM's absolute noise of ~1e-7 is a relative error below 1e-5 on a weight
// above 0.02.
template <typename T, bool kVec>
__global__ void __launch_bounds__(256) refine_weights_kernel(
    const T* __restrict__ feats, const __half* __restrict__ normed, int dim, const float* __restrict__ queries,
    const float* __restrict__ sims, int sims_ld, const int64_t* __restrict__ feat_off, const int32_t* __restrict__ view_scene,
    const int64_t* __restrict__ view_off, const int64_t* __restrict__ query_off, const int64_t* __restrict__ wobj_off,
    const int32_t* __restrict__ row_object, const float* __restrict__ view_minmax, int sim_kernel,
    const int* __restrict__ refine_list, float* __restrict__ weight_obj) {
  constexpr int kMaxPerLane = 32;  // dim <= 1024
  // persistent warps over the (row, view) list view_weights_kernel queued
  const int lane = threadIdx.x & 31;
  const int n_items = refine_list[0];
  const int n_chunks = kVec ? dim / 256 : (dim + 31) / 32;  // per-lane groups of 8 (vector) or single (scalar) channels
  for (int item = blockIdx.x * 8 + (threadIdx.x >> 5); item < n_items; item += gridDim.x * 8) {
    const int64_t r = refine_list[1 + 2 * item], g = refine_list[2 + 2 * item];
    const int s = view_scene[g];
    const int n_q = (int)(query_off[s + 1] - query_off[s]);
    const int n_v = (int)(view_off[s + 1] - view_off[s]);
    const int v_local = (int)(g - view_off[s]);
    const float mn = view_minmax[2 * g], mx = view_minmax[2 * g + 1];
    const float tol = 1e-5f * fmaxf(fmaxf(fabsf(mn), fabsf(mx)), 1e-30f);
    const float* q0 = queries + query_off[s] * (int64_t)dim;
    const int obj = row_object[r];
    float* w_slot = weight_obj + wobj_off[s] + (int64_t)obj * n_v + v_local;
    const float* srow = sims + r * sims_ld;
    float y[kMaxPerLane];
#pragma unroll
    for (int k = 0; k < kMaxPerLane; ++k) y[k] = 0.f;
    if (normed) {
      const __half* yr = normed + r * dim;
      if (kVec) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (k < n_chunks) {
            const int4 raw = __ldg(reinterpret_cast<const int4*>(yr) + k * 32 + lane);
            const __half2* h2 = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 f = __half22float2(h2[j]);
              y[k * 8 + 2 * j] = f.x;
              y[k * 8 + 2 * j + 1] = f.y;
            }
          }
      } else {
#pragma unroll
        for (int k = 0; k < kMaxPerLane; ++k)
          if (k * 32 + lane < dim) y[k] = __half2float(yr[k * 32 + lane]);
      }
    } else {
      const T* x = feats + r * dim;
      double ss = 0.0;
      if (kVec) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (k < n_chunks) {
#pragma unroll
            for (int j = 0; j < 8; ++j) y[k * 8 + j] = (float)x[(k * 32 + lane) * 8 + j];
          }
      } else {
#pragma unroll
        for (int k = 0; k < kMaxPerLane; ++k)
          if (k * 32 + lane < dim) y[k] = (float)x[k * 32 + lane];
      }
#pragma unroll
      for (int k = 0; k < kMaxPerLane; ++k) ss = fma((double)y[k], (double)y[k], ss);
      const float nrm = rounded_norm<T>(warp_sum_f64(ss));  // same rule as row_normalize_kernel
#pragma unroll
      for (int k = 0; k < kMaxPerLane; ++k) {
        const float q = y[k] / nrm;  // IEEE division, like torch
        y[k] = sizeof(T) == 2 ? __half2float(__float2half_rn(q)) : q;
      }
    }
    // approximate arg-max of the negatives from the GEMM's fp32 similarities (lane o holds query o0 + o)
    float neg_max = -INFINITY;
    for (int o0 = 0; o0 < n_q; o0 += 32) {
      const int o = o0 + lane;
      neg_max = fmaxf(neg_max, (o < n_q && o != obj) ? srow[o] : -INFINITY);
    }
    neg_max = dc::warp_max(neg_max);
    double pos = 0.0, red = (sim_kernel == DC_SIM_MAX) ? -INFINITY : 0.0;
    bool nan_seen = false;
    for (int o0 = 0; o0 < n_q; o0 += 32) {
      const int o_mine = o0 + lane;
      const float so = o_mine < n_q ? srow[o_mine] : -INFINITY;
      // NaN similarities are taken (the comparison is false for them), so they propagate like in torch
      const bool take = o_mine < n_q && (o_mine == obj || sim_kernel == DC_SIM_MEAN || !(so < neg_max - tol));
      unsigned todo = __ballot_sync(0xffffffffu, take);
      while (todo) {
        const int o = o0 + __ffs(todo) - 1;
        todo &= todo - 1;
        const float* q = q0 + (int64_t)o * dim;
        double d = 0.0;
        if (kVec) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (k < n_chunks) {
              const float4 a = __ldg(reinterpret_cast<const float4*>(q) + (k * 32 + lane) * 2);
              const float4 b = __ldg(reinterpret_cast<const float4*>(q) + (k * 32 + lane) * 2 + 1);
              d = fma((double)y[k * 8 + 0], (double)a.x, d);
              d = fma((double)y[k * 8 + 1], (double)a.y, d);
              d = fma((double)y[k * 8 + 2], (double)a.z, d);
              d = fma((double)y[k * 8 + 3], (double)a.w, d);
              d = fma((double)y[k * 8 + 4], (double)b.x, d);
              d = fma((double)y[k * 8 + 5], (double)b.y, d);
              d = fma((double)y[k * 8 + 6], (double)b.z, d);
              d = fma((double)y[k * 8 + 7], (double)b.w, d);
            }
        } else {
#pragma unroll
          for (int k = 0; k < kMaxPerLane; ++k)
            if (k * 32 + lane < dim) d = fma((double)y[k], (double)__ldg(q + k * 32 + lane), d);
        }
        d = warp_sum_f64(d);
        if (o == obj) pos = d;
        else {
          nan_seen |= (d != d);
          if (sim_kernel == DC_SIM_MAX) red = fmax(red, d);
          else red += d;
        }
      }
    }
    if (sim_kernel == DC_SIM_MEAN) red = red / (double)(n_q - 1);
    if (nan_seen) red = __longlong_as_double(0x7ff8000000000000ll);
    float w = (float)((pos - red) / ((double)mx - (double)mn));  // NaN extrema (a NaN anywhere in the view) give NaN, like torch
    if (w == w) w = fmaxf(w, 1e-6f);
    if (lane == 0) *w_slot = w;
  }
}

__global__ void init_minmax_kernel(float* m) {
  if (threadIdx.x == 0) { m[0] = INFINITY; m[1] = -INFINITY; m[2] = INFINITY; m[3] = -INFINITY; }
}

// The ground-truth tables of a counting launch of minmax_threshold_kernel (dc_predict_many_iou). Query q's points carry
// the labels labels[point_row[q] + i]; its object ids are gt_ids[gt_off[q] .. gt_off[q+1]), sorted and unique.
struct IouCount {
  const void* labels;
  const int64_t* point_row;
  const int* gt_off;
  const int64_t* gt_ids;
  unsigned long long* inter;
  unsigned long long* uni;
};

// Whether `label` is one of ids[0 .. n) (ascending): a binary search through the read-only cache.
__device__ __forceinline__ bool id_listed(int64_t label, const int64_t* __restrict__ ids, int n) {
  const int64_t* end = ids + n;
  while (n > 0) {  // lower bound
    const int half = n >> 1;
    if (__ldg(ids + half) < label) { ids += half + 1; n -= half + 1; }
    else n = half;
  }
  return ids < end && __ldg(ids) == label;
}

// A single-row launch (gridDim.y == 1, no row table) normalises v [n] with the extrema mm [4]. With `row_off`, blockIdx.y
// selects query row y = v [row_off[y], row_off[y + 1]) with its own extrema mm [4 * y] (dc_predict_queries,
// dc_predict_many); `n` is then unused.
// Label != void (int32_t / int64_t, with a row table): count instead of writing. Point i of query y is predicted when
// the normalised score x > thr (or, when !pred_from_thr, its argmax byte pred[i] is set) and is ground truth when its
// label is one of the query's ids; the block adds |pred & gt| and |pred | gt| to cnt.inter[y] and cnt.uni[y]. Neither v
// nor pred is written.
template <class Label>
__global__ void __launch_bounds__(256) minmax_threshold_kernel(float* __restrict__ v, int64_t n, const float* __restrict__ mm,
                                                               int use_raw, float thr, int pred_from_thr,
                                                               uint8_t* __restrict__ pred,
                                                               const int64_t* __restrict__ row_off = nullptr,
                                                               IouCount cnt = {}) {
  constexpr bool kCount = !std::is_void<Label>::value;
  if (row_off) {
    const int64_t o = row_off[blockIdx.y];
    n = row_off[blockIdx.y + 1] - o;
    v += o;
    mm += 4 * blockIdx.y;
    if (pred) pred += o;
  }
  const float mn = mm[0], mx = mm[1];
  const bool differ = use_raw ? (mm[3] != mm[2]) : (mx != mn);
  const float range = mx - mn;
  if constexpr (!kCount) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      float x = v[i];
      x = differ ? (x - mn) / range : x / mx;
      v[i] = x;
      if (pred_from_thr) pred[i] = x > thr ? 1 : 0;
    }
  } else {
    const Label* __restrict__ labels = static_cast<const Label*>(cnt.labels) + cnt.point_row[blockIdx.y];
    const int g0 = cnt.gt_off[blockIdx.y], n_ids = cnt.gt_off[blockIdx.y + 1] - g0;
    const int64_t* __restrict__ ids = cnt.gt_ids + g0;
    unsigned both = 0, either = 0;  // < 2^31 points per query
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      bool p;
      if (pred_from_thr) {
        float x = v[i];
        x = differ ? (x - mn) / range : x / mx;
        p = x > thr;
      } else {
        p = pred[i] != 0;
      }
      const bool g = id_listed((int64_t)__ldg(labels + i), ids, n_ids);
      both += (p && g) ? 1u : 0u;
      either += (p || g) ? 1u : 0u;
    }
    __shared__ unsigned s_both[8], s_either[8];
    both = __reduce_add_sync(0xffffffffu, both);
    either = __reduce_add_sync(0xffffffffu, either);
    if ((threadIdx.x & 31) == 0) {
      s_both[threadIdx.x >> 5] = both;
      s_either[threadIdx.x >> 5] = either;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      both = 0;
      either = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
        both += s_both[w];
        either += s_either[w];
      }
      if (both) atomicAdd(cnt.inter + blockIdx.y, (unsigned long long)both);
      if (either) atomicAdd(cnt.uni + blockIdx.y, (unsigned long long)either);
    }
  }
}

constexpr int kSweepMaxThresholds = 1024;  // dc_predict_many_iou_sweep: two block histograms of <= 1025 bins, 8.2 KB

// The threshold pass of dc_predict_many_iou_sweep: query row y = v [row_off[y], row_off[y + 1]) with its extrema and
// ground truth as in the counting instances of minmax_threshold_kernel, and the same normalised score x. Instead of one
// threshold, the U ascending distinct levels u[0 .. U): point i falls into bin k = #{j : x > u_j} (0 for a NaN x;
// argmax: U when its byte is set, else 0), so x > u_r exactly when k > r. The block counts its points per (g, k) in
// shared memory, with one shared atomic per group of lanes of a warp that share the bin (most points of a query fall
// into one or two bins), and adds its non-zero bins to hist [n_queries][2][U + 1] (g = 0: not ground truth, 1: ground
// truth; 32 bits, < 2^31 points per query).
template <class Label>
__global__ void __launch_bounds__(256) threshold_sweep_kernel(const float* __restrict__ v, const float* __restrict__ mm,
                                                              int use_raw, int pred_from_thr,
                                                              const uint8_t* __restrict__ pred,
                                                              const int64_t* __restrict__ row_off,
                                                              const float* __restrict__ levels, int n_levels, IouCount cnt,
                                                              unsigned* __restrict__ hist) {
  extern __shared__ unsigned s_sweep[];
  const int bins = n_levels + 1;
  unsigned* s_hist = s_sweep;                                  // [2][bins]
  float* s_lv = reinterpret_cast<float*>(s_sweep + 2 * bins);  // [n_levels]
  for (int j = threadIdx.x; j < 2 * bins; j += blockDim.x) s_hist[j] = 0;
  for (int j = threadIdx.x; j < n_levels; j += blockDim.x) s_lv[j] = levels[j];
  __syncthreads();
  const int64_t o = row_off[blockIdx.y];
  const int64_t n = row_off[blockIdx.y + 1] - o;
  v += o;
  pred += o;
  mm += 4 * blockIdx.y;
  const float mn = mm[0], mx = mm[1];
  const bool differ = use_raw ? (mm[3] != mm[2]) : (mx != mn);
  const float range = mx - mn;
  const Label* __restrict__ labels = static_cast<const Label*>(cnt.labels) + cnt.point_row[blockIdx.y];
  const int g0 = cnt.gt_off[blockIdx.y], n_ids = cnt.gt_off[blockIdx.y + 1] - g0;
  const int64_t* __restrict__ ids = cnt.gt_ids + g0;
  const int lane = threadIdx.x & 31;
  // the loop runs warp-uniformly (lanes past the end take no bin), so every lane can join __match_any_sync
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x - lane); base < n;
       base += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = base + lane;
    int bin = -1;
    if (i < n) {
      int k;
      if (pred_from_thr) {
        float x = v[i];
        x = differ ? (x - mn) / range : x / mx;
        int lo = 0, hi = n_levels;  // k = #{j : u_j < x}: the comparison x > u_j, false for every u_j when x is NaN
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (s_lv[mid] < x) lo = mid + 1;
          else hi = mid;
        }
        k = lo;
      } else {
        k = pred[i] != 0 ? n_levels : 0;
      }
      bin = id_listed((int64_t)__ldg(labels + i), ids, n_ids) ? bins + k : k;
    }
    const unsigned same = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && lane == __ffs(same) - 1) atomicAdd(s_hist + bin, (unsigned)__popc(same));
  }
  __syncthreads();
  unsigned* h = hist + (int64_t)blockIdx.y * 2 * bins;
  for (int j = threadIdx.x; j < 2 * bins; j += blockDim.x)
    if (s_hist[j]) atomicAdd(h + j, s_hist[j]);
}

// The counts of dc_predict_many_iou_sweep from the histograms of threshold_sweep_kernel, one block per query q: with
// r = rank[t], inter[t][q] = sum_{k > r} hist[q][1][k] and uni[t][q] = |gt_q| + sum_{k > r} hist[q][0][k], where
// |gt_q| = sum_k hist[q][1][k]. One warp takes the suffix sums (each lane a run of bins), then the block writes T rows.
__global__ void __launch_bounds__(256) sweep_counts_kernel(const unsigned* __restrict__ hist, int n_levels,
                                                           const int* __restrict__ rank, int n_thr, int n_queries,
                                                           int64_t* __restrict__ inter, int64_t* __restrict__ uni) {
  extern __shared__ unsigned s_suffix[];  // [2][bins]: sum_{j >= k} hist[q][g][j]
  const int bins = n_levels + 1;
  const unsigned* h = hist + (int64_t)blockIdx.x * 2 * bins;
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    const int run = (bins + 31) / 32;
    const int j0 = min(bins, lane * run), j1 = min(bins, j0 + run);
    unsigned sn = 0, sg = 0;
    for (int j = j0; j < j1; ++j) {
      sn += h[j];
      sg += h[bins + j];
    }
    for (int d = 1; d < 32; d <<= 1) {  // inclusive suffix sums over the lanes
      const unsigned an = __shfl_down_sync(0xffffffffu, sn, d), ag = __shfl_down_sync(0xffffffffu, sg, d);
      if (lane + d < 32) {
        sn += an;
        sg += ag;
      }
    }
    unsigned rn = __shfl_down_sync(0xffffffffu, sn, 1), rg = __shfl_down_sync(0xffffffffu, sg, 1);
    if (lane == 31) rn = rg = 0;
    for (int j = j1 - 1; j >= j0; --j) {
      rn += h[j];
      rg += h[bins + j];
      s_suffix[j] = rn;
      s_suffix[bins + j] = rg;
    }
  }
  __syncthreads();
  const unsigned gt = s_suffix[bins];
  for (int t = threadIdx.x; t < n_thr; t += blockDim.x) {
    const int k = rank[t] + 1;  // in [1, U]
    inter[(int64_t)t * n_queries + blockIdx.x] = s_suffix[bins + k];
    uni[(int64_t)t * n_queries + blockIdx.x] = gt + s_suffix[k];
  }
}

__global__ void init_query_minmax_kernel(float* m, int n_slots) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 4 * n_slots; i += gridDim.x * blockDim.x)
    m[i] = (i & 1) ? -INFINITY : INFINITY;
}

// atomic_min_f / atomic_max_f skipped when a plain read already shows a value at least as extreme: the stored extremum
// only moves outwards, so a value that does not beat a stale read cannot beat the current one (most warps, once the
// extrema settle). NaN compares false and still takes the atomic, as in the epilogues.
__device__ __forceinline__ void atomic_min_f_if(float* a, float v) {
  if (!(v >= *(volatile float*)a)) atomic_min_f(a, v);
}
__device__ __forceinline__ void atomic_max_f_if(float* a, float v) {
  if (!(v <= *(volatile float*)a)) atomic_max_f(a, v);
}

// One scene of the scoring tables (dc_predict_queries: one, dc_predict_many: one per scene of the batch).
struct ScoreScene {
  int64_t s_row;    // the scene's first row of S
  int64_t out_off;  // start of the scene's [n_queries, n_points] block of v and pred
  int n_points;
  int n_prompts;    // the scene's columns of S: [0, n_prompts)
  int q0;           // the scene's first query
  int pad;
};
// One block of query_scores_kernel: rows [row0, row0 + rows) of scene `scene` (scene-local), queries [q0, q1).
struct ScoreBlock {
  int scene, row0, rows, q0, q1;
};

// Per-query scores from the raw similarity matrix S [rows, s_ld] (dc_predict_queries, dc_predict_many). Query q of
// scene s has the positive column pos[q] and the negative columns neg_cols[neg_off[q] .. neg_off[q+1]) (m of them),
// all in [0, P_s):
//   RAW    (m == 0): v = S[n, pos]
//   PAIRED (m >= 1): v = 1 / (m + sum_j exp((S[n, j] - S[n, pos]) / T)), NaN -> 0   (EpiGround's arithmetic)
//   ARGMAX (m >= 1): v = S[n, pos] - mean_j S[n, j], pred = S[n, pos] >= max_j S[n, j] (the positive wins ties)
// v: scene s's block [Q_s, N_s] at out_off; minmax [4 * q]: min/max of v, min/max of S over {pos} + negatives.
// A block stages its rows of S (at most `tile_rows`) in shared memory (coalesced: each row's P_s columns are
// contiguous in S; the row stride in shared memory is odd, so 32 lanes reading one column of 32 rows hit 32 banks).
// Thread t owns row t % tile_rows for the queries q0 + t / tile_rows, q0 + t / tile_rows + groups, ... of the block;
// a warp holds 32 rows of one query, so the stores of v are coalesced and the extrema reduce with shuffles. The
// blocks of one row tile are listed consecutively: the query chunks after the first re-read the tile from L2.
template <int kMode>
__global__ void __launch_bounds__(256) query_scores_kernel(const float* __restrict__ S, int s_ld,
                                                           const ScoreBlock* __restrict__ blocks,
                                                           const ScoreScene* __restrict__ scenes,
                                                           const int* __restrict__ pos, const int* __restrict__ neg_off,
                                                           const int* __restrict__ neg_cols, int tile_rows, float inv_temp,
                                                           float* __restrict__ v, uint8_t* __restrict__ pred,
                                                           float* __restrict__ minmax) {
  extern __shared__ float s_tile[];
  const ScoreBlock blk = blocks[blockIdx.x];
  const ScoreScene sc = scenes[blk.scene];
  const int n_prompts = sc.n_prompts;
  const int ld = n_prompts | 1;
  const int rows = blk.rows;
  const float* src = S + (sc.s_row + blk.row0) * (int64_t)s_ld;
  for (int i = threadIdx.x; i < rows * n_prompts; i += blockDim.x) {
    const int r = i / n_prompts;
    const int c = i - r * n_prompts;
    s_tile[r * ld + c] = src[(int64_t)r * s_ld + c];
  }
  __syncthreads();
  const int r = threadIdx.x % tile_rows;
  const int groups = blockDim.x / tile_rows;
  const bool have = r < rows;
  const float* srow = s_tile + r * ld;
  const int64_t n = blk.row0 + r;
  const float scale = inv_temp * 1.4426950408889634f;  // log2(e) / T
  v += sc.out_off - (int64_t)sc.q0 * sc.n_points;  // query q's row starts at q * n_points
  if (kMode == DC_GROUND_ARGMAX) pred += sc.out_off - (int64_t)sc.q0 * sc.n_points;
  const int64_t n_points = sc.n_points;
  for (int q = blk.q0 + threadIdx.x / tile_rows; q < blk.q1; q += groups) {  // warp-uniform
    const float sp = have ? srow[__ldg(pos + q)] : 0.f;
    const int j0 = __ldg(neg_off + q), j1 = __ldg(neg_off + q + 1);
    float raw_min = sp, raw_max = sp, acc[4] = {0.f, 0.f, 0.f, 0.f}, neg_max = -INFINITY;
    const float bias = -sp * scale;
    for (int j = j0; j < j1; ++j) {
      const float s = srow[__ldg(neg_cols + j)];
      raw_min = fminf(raw_min, s);
      raw_max = fmaxf(raw_max, s);
      if (kMode == DC_GROUND_PAIRED) acc[(j - j0) & 3] += ex2_approx(fmaf(s, scale, bias));
      else { acc[(j - j0) & 3] += s; neg_max = fmaxf(neg_max, s); }
    }
    const float sum = (acc[0] + acc[1]) + (acc[2] + acc[3]);
    const float m = (float)(j1 - j0);
    float o = sp;
    if (kMode == DC_GROUND_PAIRED) {
      o = 1.f / (m + sum);
      if (o != o) o = 0.f;  // nan_to_num
    } else if (kMode == DC_GROUND_ARGMAX) {
      o = sp - sum / m;
    }
    if (have) {
      v[(int64_t)q * n_points + n] = o;
      if (kMode == DC_GROUND_ARGMAX) pred[(int64_t)q * n_points + n] = (sp >= neg_max) ? 1 : 0;
    }
    float a = have ? o : INFINITY, b = have ? o : -INFINITY, c = have ? raw_min : INFINITY, d = have ? raw_max : -INFINITY;
    a = dc::warp_min(a); b = dc::warp_max(b); c = dc::warp_min(c); d = dc::warp_max(d);
    if ((threadIdx.x & 31) == 0) {
      float* mm = minmax + 4 * q;
      if (a != INFINITY) atomic_min_f_if(mm + 0, a);
      if (b != -INFINITY) atomic_max_f_if(mm + 1, b);
      if (c != INFINITY) atomic_min_f_if(mm + 2, c);
      if (d != -INFINITY) atomic_max_f_if(mm + 3, d);
    }
  }
}

constexpr int kQueryMaxPrompts = 1536;  // dc_predict_queries: 32 staged rows of S, 32 * 1537 * 4 = 197 KB of shared memory

template <class Epi>
int launch_bn(int bn, const void* a_hi, const void* a_lo, int64_t a_rows, const void* b_hi, const void* b_lo, int64_t b_rows,
              const Params& p, const Epi& epi, int max_tiles, cudaStream_t st) {
  switch (bn) {
    case 32: return dc::gemm::launch<32>(a_hi, a_lo, a_rows, b_hi, b_lo, b_rows, p, epi, max_tiles, st);
    case 64: return dc::gemm::launch<64>(a_hi, a_lo, a_rows, b_hi, b_lo, b_rows, p, epi, max_tiles, st);
    case 128: return dc::gemm::launch<128>(a_hi, a_lo, a_rows, b_hi, b_lo, b_rows, p, epi, max_tiles, st);
    case 256: return dc::gemm::launch<256>(a_hi, a_lo, a_rows, b_hi, b_lo, b_rows, p, epi, max_tiles, st);
  }
  return dc::fail(DC_ERR_UNSUPPORTED, "unsupported GEMM N tile %d", bn);
}

int pick_bn(int n) { return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : 256; }

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct ScoreWorkspace {
  size_t a_hi, a_lo, q_hi, q_lo, tiles, tile_count, total;
  int max_tiles;
};

ScoreWorkspace score_layout(int64_t total_rows, int64_t total_queries, int dim, int feat_dtype, int n_scenes_bound) {
  ScoreWorkspace w{};
  size_t off = 0;
  const size_t a_bytes = align_up((size_t)(total_rows > 0 ? total_rows : 1) * dim * 2, 1024);
  const size_t q_bytes = align_up((size_t)(total_queries > 0 ? total_queries : 1) * dim * 2, 1024);
  w.a_hi = off; off += a_bytes;
  w.a_lo = off; off += (feat_dtype == DC_F32) ? a_bytes : 0;
  w.q_hi = off; off += q_bytes;
  w.q_lo = off; off += q_bytes;
  w.max_tiles = (int)(total_rows / dc::gemm::kBlockM + n_scenes_bound + 1);
  w.tiles = off; off += align_up(sizeof(int4) * (size_t)w.max_tiles, 1024);
  w.tile_count = off; off += 1024;
  w.total = off;
  return w;
}

}  // namespace

extern "C" {

int dc_view_score_ld(int max_queries_per_scene) { return pick_bn(max_queries_per_scene); }

size_t dc_view_score_workspace(int64_t total_rows, int64_t total_queries, int dim, int feat_dtype) {
  // the tile list is bounded with total_queries >= n_scenes
  return score_layout(total_rows, total_queries, dim, feat_dtype, (int)total_queries).total;
}

int dc_view_score(const void* feats, int feat_dtype, int64_t total_rows, int dim, const int64_t* feat_off,
                  const int64_t* view_off, const float* queries, const int64_t* query_off, int64_t total_queries,
                  int n_scenes, int max_queries_per_scene, float* sims, int sims_ld, void* workspace,
                  size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(feats && feat_off && view_off && queries && query_off && sims && workspace,
               "dc_view_score: null pointer argument");
  DC_CHECK_ARG(feat_dtype == DC_F16 || feat_dtype == DC_F32, "dc_view_score: features must be fp16 or fp32");
  DC_CHECK_ARG(dim > 0 && dim % 64 == 0, "dc_view_score: feature dim must be a multiple of 64 (got %d)", dim);
  DC_CHECK_ARG(max_queries_per_scene >= 1 && max_queries_per_scene <= 256, "dc_view_score: 1..256 queries per scene");
  const int bn = pick_bn(max_queries_per_scene);
  DC_CHECK_ARG(sims_ld >= bn, "dc_view_score: sims_ld must be >= %d", bn);
  DC_CHECK_ARG(((uintptr_t)workspace & 1023) == 0, "dc_view_score: workspace must be 1024-byte aligned");
  DC_CHECK_ARG(total_rows < (1ll << 31) && total_queries < (1ll << 31), "dc_view_score: too many rows");
  if (total_rows <= 0 || n_scenes <= 0) return DC_OK;
  const ScoreWorkspace w = score_layout(total_rows, total_queries, dim, feat_dtype, (int)total_queries);
  if (workspace_bytes < w.total)
    return dc::fail(DC_ERR_WORKSPACE, "dc_view_score: workspace %zu < %zu", workspace_bytes, w.total);
  cudaStream_t st = dc::as_stream(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  void* a_hi = ws + w.a_hi;
  void* a_lo = feat_dtype == DC_F32 ? ws + w.a_lo : nullptr;
  void* q_hi = ws + w.q_hi;
  void* q_lo = ws + w.q_lo;
  int rc;
  // normalised copies of the feature rows (the reference keeps feat_v itself un-normalised, :311,333)
  if ((rc = launch_row_normalize(const_cast<void*>(feats), feat_dtype, total_rows, dim, 1, false, a_hi, a_lo, st))) return rc;
  if ((rc = launch_row_normalize(const_cast<float*>(queries), DC_F32, total_queries, dim, 0, false, q_hi, q_lo, st))) return rc;
  int4* tiles = reinterpret_cast<int4*>(ws + w.tiles);
  int* tile_count = reinterpret_cast<int*>(ws + w.tile_count);
  build_score_tiles_kernel<<<1, 1024, 0, st>>>(feat_off, view_off, query_off, n_scenes, tiles, tile_count, w.max_tiles);
  DC_LAUNCH_CHECK();
  Params p{tiles, tile_count, total_rows, bn, dim};
  dc::gemm::set_terms(p, a_lo, q_lo);
  EpiStore epi{sims, sims_ld};
  return launch_bn(bn, a_hi, a_lo, total_rows, q_hi, q_lo, total_queries, p, epi, w.max_tiles, st);
}

size_t dc_view_weights_scratch(int64_t total_views, int64_t total_rows) {
  return sizeof(float) * 2 * (size_t)(total_views > 0 ? total_views : 0) + sizeof(int) * (1 + 2 * (size_t)(total_rows > 0 ? total_rows : 0));
}

int dc_view_weights(const float* sims, int sims_ld, const int64_t* feat_off, const int32_t* view_scene,
                    const int64_t* view_off, const int64_t* query_off, const int64_t* wobj_off,
                    const int32_t* row_object, const uint32_t* counts, int nbins, int64_t total_views,
                    int sim_kernel, int use_visibility, float* weight_obj, const void* feats, int feat_dtype, int dim,
                    const float* queries, int64_t total_rows, void* scratch, const void* feats_normalized,
                    float refine_below, dc_stream_t stream) {
  DC_CHECK_ARG(feat_off && view_scene && view_off && query_off && wobj_off && row_object && weight_obj,
               "dc_view_weights: null pointer argument");
  DC_CHECK_ARG(sim_kernel == DC_SIM_NONE || sims, "dc_view_weights: sims required for a similarity kernel");
  DC_CHECK_ARG(!use_visibility || counts, "dc_view_weights: counts required for use_visibility");
  DC_CHECK_ARG(sim_kernel >= DC_SIM_NONE && sim_kernel <= DC_SIM_MEAN, "dc_view_weights: Please set method in [mean, max]");
  const bool refine = feats && sim_kernel != DC_SIM_NONE;
  DC_CHECK_ARG(!refine || (queries && scratch && dim > 0 && dim <= 1024 && (feat_dtype == DC_F16 || feat_dtype == DC_F32)),
               "dc_view_weights: exact weights need queries, scratch and fp16/fp32 features of dim <= 1024");
  DC_CHECK_ARG(!refine || ((uintptr_t)scratch & 3) == 0, "dc_view_weights: scratch must be 4-byte aligned");
  DC_CHECK_ARG(total_rows < (1ll << 31) && total_views < (1ll << 31), "dc_view_weights: too many rows");
  if (total_views <= 0) return DC_OK;
  cudaStream_t st = dc::as_stream(stream);
  float* view_minmax = refine ? static_cast<float*>(scratch) : nullptr;
  int* refine_list = refine ? reinterpret_cast<int*>(view_minmax + 2 * total_views) : nullptr;  // [0] count, then (row, view)
  if (refine) DC_CUDA(cudaMemsetAsync(refine_list, 0, sizeof(int), st));
  view_weights_kernel<<<(unsigned)dc::ceil_div<int64_t>(total_views, 4), 128, 0, st>>>(
      sims, sims_ld, feat_off, view_scene, view_off, query_off, wobj_off, row_object, counts, nbins, total_views,
      sim_kernel, use_visibility, weight_obj, view_minmax, refine_list, refine_below);
  DC_LAUNCH_CHECK();
  if (refine && total_rows > 0) {
    const unsigned grid = (unsigned)std::min<int64_t>(dc::ceil_div<int64_t>(total_rows, 8), (int64_t)dc::sm_count() * 2);
    const __half* normed = (const __half*)feats_normalized;
    const bool vec = dim % 256 == 0 && (((uintptr_t)feats | (uintptr_t)feats_normalized | (uintptr_t)queries) & 15) == 0;
#define DC_REFINE(T, V)                                                                                                     \
  refine_weights_kernel<T, V><<<grid, 256, 0, st>>>((const T*)feats, normed, dim, queries, sims, sims_ld, feat_off, view_scene, \
                                                    view_off, query_off, wobj_off, row_object, view_minmax, sim_kernel,       \
                                                    refine_list, weight_obj)
    if (feat_dtype == DC_F16) { if (vec) DC_REFINE(__half, true); else DC_REFINE(__half, false); }
    else { normed = nullptr; if (vec) DC_REFINE(float, true); else DC_REFINE(float, false); }
#undef DC_REFINE
    DC_LAUNCH_CHECK();
  }
  return DC_OK;
}

int dc_row_normalize(void* x, int dtype, int64_t n_rows, int dim, int normalize, void* plane_hi, void* plane_lo,
                     dc_stream_t stream) {
  DC_CHECK_ARG(x, "dc_row_normalize: null pointer argument");
  DC_CHECK_ARG(dtype == DC_F16 || dtype == DC_F32, "dc_row_normalize: dtype must be fp16 or fp32");
  DC_CHECK_ARG(dim > 0, "dc_row_normalize: bad dim");
  DC_CHECK_ARG(!plane_lo || plane_hi, "dc_row_normalize: plane_lo needs plane_hi");
  return launch_row_normalize(x, dtype, n_rows, dim, normalize, true, plane_hi, dtype == DC_F32 ? plane_lo : nullptr,
                              dc::as_stream(stream));
}

int dc_ground_init_minmax(float* minmax, dc_stream_t stream) {
  DC_CHECK_ARG(minmax, "dc_ground_init_minmax: null pointer argument");
  init_minmax_kernel<<<1, 32, 0, dc::as_stream(stream)>>>(minmax);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

size_t dc_ground_workspace(int64_t n_points, int n_prompts, int mode) {
  if (n_prompts <= 256 || mode == DC_GROUND_RAW || n_points <= 0) return 0;
  return (size_t)n_points * 4 * sizeof(float);
}

int dc_ground(const void* x_hi, const void* x_lo, int64_t n_points, const void* t_hi, const void* t_lo, int n_prompts,
              int dim, int mode, float softmax_temp, int normalize_fp16_rows, float* out, int out_ld, uint8_t* pred,
              int64_t* argmax_idx, float* minmax, void* workspace, size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(x_hi && t_hi && minmax, "dc_ground: null pointer argument");
  DC_CHECK_ARG(out || mode == DC_GROUND_CLASS, "dc_ground: null output");
  DC_CHECK_ARG(n_prompts >= 1, "dc_ground: at least one prompt (got %d)", n_prompts);
  DC_CHECK_ARG(dim > 0 && dim % 64 == 0, "dc_ground: feature dim must be a multiple of 64 (got %d)", dim);
  DC_CHECK_ARG(mode >= DC_GROUND_RAW && mode <= DC_GROUND_CLASS, "dc_ground: bad mode");
  DC_CHECK_ARG(mode != DC_GROUND_ARGMAX || pred, "dc_ground: argmax mode needs pred");
  DC_CHECK_ARG(mode != DC_GROUND_CLASS || argmax_idx, "dc_ground: class mode needs argmax_idx");
  DC_CHECK_ARG(mode == DC_GROUND_RAW || mode == DC_GROUND_CLASS || n_prompts >= 2,
               "dc_ground: paired/argmax need at least one negative prompt");
  DC_CHECK_ARG((mode != DC_GROUND_RAW && mode != DC_GROUND_CLASS) || !out || out_ld >= n_prompts, "dc_ground: out_ld < n_prompts");
  DC_CHECK_ARG(n_points < (1ll << 31), "dc_ground: too many points for one call");
  DC_CHECK_ARG(!normalize_fp16_rows || !x_lo, "dc_ground: normalize_fp16_rows is for fp16 features (x_lo must be NULL)");
  if (n_points <= 0) return DC_OK;
  // fp16 features to be normalised in place (models/similarity.py:77): a separate pass before the GEMM. Each row is a
  // dependent chain (sum of squares, shuffle reduction, sqrt, quotient) that the pass hides behind 64 resident warps per
  // SM, at the HBM rate. Next to the GEMM's operand ring only a few warps fit, and normalising there cost more than the
  // GEMM re-reading the rows.
  // Fused-normaliser experiment (bit-identical, 0.232 vs 0.177 ms on B200): profiles/r02_ground.md.
  if (normalize_fp16_rows) {
    const int rc = launch_row_normalize(const_cast<void*>(x_hi), DC_F16, n_points, dim, 1, true, nullptr, nullptr, dc::as_stream(stream));
    if (rc) return rc;
  }
  const size_t need = dc_ground_workspace(n_points, n_prompts, mode);
  if (need > 0 && (!workspace || workspace_bytes < need))
    return dc::fail(DC_ERR_WORKSPACE, "dc_ground: %zu workspace bytes needed for %d prompts, got %zu", need, n_prompts, workspace_bytes);
  const int max_tiles = (int)dc::ceil_div<int64_t>(n_points, dc::gemm::kBlockM);
  // the prompt axis in blocks of <= 256 columns (the widest UMMA N): partial sums / maxima of the paired softmax,
  // the mean of the negatives and the arg max combine across blocks through `carry` (models/similarity.py:47-61
  // has no prompt limit; tools/preprocess_data.py use_kernel_neg == 'all' concatenates the whole class table)
  for (int c0 = 0; c0 < n_prompts; c0 += 256) {
    const int cols = n_prompts - c0 < 256 ? n_prompts - c0 : 256;
    const int bn = pick_bn(cols);
    Params p{nullptr, nullptr, n_points, cols, dim};
    dc::gemm::set_terms(p, x_lo, t_lo);
    // after the separate normalisation pass the rows written last are still in L2 (126 MB): walk the tiles backwards
    p.reverse = (normalize_fp16_rows && c0 == 0) ? 1 : 0;
    EpiGround epi{};
    epi.mode = mode;
    epi.n_prompts = cols;
    epi.inv_temp = 1.0f / softmax_temp;
    epi.out = (mode == DC_GROUND_RAW || mode == DC_GROUND_CLASS) ? (out ? out + c0 : nullptr) : out;
    epi.out_ld = out_ld;
    epi.pred = pred;
    epi.minmax = minmax;
    epi.col_base = c0;
    epi.n_total = n_prompts;
    epi.last = (c0 + cols >= n_prompts) ? 1 : 0;
    epi.carry = need ? (float*)workspace : nullptr;
    epi.argmax_idx = argmax_idx;
    const char* th = (const char*)t_hi + (size_t)c0 * dim * 2;
    const char* tl = t_lo ? (const char*)t_lo + (size_t)c0 * dim * 2 : th;
    const int rc = launch_bn(bn, x_hi, x_lo, n_points, th, tl, cols, p, epi, max_tiles, dc::as_stream(stream));
    if (rc) return rc;
  }
  return DC_OK;
}

size_t dc_predict_workspace(int64_t n_points, int n_prompts, int dim, int feat_dtype, int text_dtype, int mode) {
  size_t b = 256;  // minmax
  if (text_dtype == DC_F32) b += 2 * align_up((size_t)n_prompts * dim * 2, 256);
  if (feat_dtype == DC_F32) b += 2 * align_up((size_t)(n_points > 0 ? n_points : 1) * dim * 2, 256);
  b += align_up(dc_ground_workspace(n_points, n_prompts, mode), 256);
  return b;
}

int dc_predict(void* feats, int feat_dtype, int64_t n_points, const void* text, int text_dtype, int n_prompts, int dim,
               int mode, float softmax_temp, int normalize, float threshold, float* out, uint8_t* pred, float** minmax_out,
               void* workspace, size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(feats && text && out && pred && workspace, "dc_predict: null pointer argument");
  DC_CHECK_ARG(feat_dtype == DC_F16 || feat_dtype == DC_F32, "dc_predict: features must be fp16 or fp32");
  DC_CHECK_ARG(text_dtype == DC_F16 || text_dtype == DC_F32, "dc_predict: prompt embeddings must be fp16 or fp32");
  DC_CHECK_ARG(mode == DC_GROUND_RAW || mode == DC_GROUND_PAIRED || mode == DC_GROUND_ARGMAX, "dc_predict: bad mode");
  DC_CHECK_ARG(mode != DC_GROUND_RAW || n_prompts == 1, "dc_predict: raw mode is the no-negatives case (one prompt)");
  DC_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "dc_predict: workspace must be 256-byte aligned");
  const size_t need = dc_predict_workspace(n_points, n_prompts, dim, feat_dtype, text_dtype, mode);
  if (workspace_bytes < need) return dc::fail(DC_ERR_WORKSPACE, "dc_predict: workspace %zu < %zu", workspace_bytes, need);
  uint8_t* w = static_cast<uint8_t*>(workspace);
  float* minmax = reinterpret_cast<float*>(w);
  w += 256;
  if (minmax_out) *minmax_out = minmax;
  int rc;
  if ((rc = dc_ground_init_minmax(minmax, stream))) return rc;
  if (n_points <= 0) return DC_OK;
  const void *t_hi = text, *t_lo = nullptr;
  if (text_dtype == DC_F32) {  // fp16 hi + lo planes of the (already normalised) prompt rows; fp16 prompts are used as they are
    const size_t pb = align_up((size_t)n_prompts * dim * 2, 256);
    if ((rc = launch_row_normalize(const_cast<void*>(text), DC_F32, n_prompts, dim, 0, false, w, w + pb, dc::as_stream(stream)))) return rc;
    t_hi = w;
    t_lo = w + pb;
    w += 2 * pb;
  }
  const void *x_hi = feats, *x_lo = nullptr;
  if (feat_dtype == DC_F32) {
    const size_t xb = align_up((size_t)n_points * dim * 2, 256);
    if ((rc = launch_row_normalize(feats, DC_F32, n_points, dim, normalize, true, w, w + xb, dc::as_stream(stream)))) return rc;
    x_hi = w;
    x_lo = w + xb;
    w += 2 * xb;
  }
  if ((rc = dc_ground(x_hi, x_lo, n_points, t_hi, t_lo, n_prompts, dim, mode, softmax_temp,
                      (feat_dtype == DC_F16 && normalize) ? 1 : 0, out, mode == DC_GROUND_RAW ? n_prompts : 1, pred, nullptr,
                      minmax, w, dc_ground_workspace(n_points, n_prompts, mode), stream)))
    return rc;
  // global min-max (+ threshold) of models/similarity.py:83-88; argmax branch :95-98 normalises pos - mean(neg) and keeps
  // the arg-max prediction the epilogue wrote
  return dc_minmax_threshold(out, n_points, minmax, mode == DC_GROUND_ARGMAX ? 1 : 0, threshold,
                             mode == DC_GROUND_ARGMAX ? 0 : 1, pred, stream);
}

}  // extern "C"

namespace {

// Host plan of the scoring pass of dc_predict_queries (one scene) and dc_predict_many (a batch): the workspace layout
// and the device tables - query rows, column CSR, scenes, score blocks and (dc_predict_many) the GEMM's tile lists -
// staged in one host buffer and copied into the workspace by one cudaMemcpyAsync. A scene without queries gets no
// blocks, no tiles and no normalisation.
// dc_predict_many_iou also stages its ground-truth tables (query q's first feature row, gt_off, gt_ids) in the table
// region, and keeps the scores and the argmax bytes in the workspace (`v`, `pred`). dc_predict_many_iou_sweep adds its
// threshold levels and ranks to the table region (room for n_thr each) and its histograms to the workspace (`hist`).
struct ScorePlan {
  size_t minmax, tables, t_planes, x_planes, sims, v, pred, hist, total;           // workspace byte offsets
  size_t t_qrow, t_pos, t_off, t_cols, t_scenes, t_blocks, t_counts, t_tiles;      // inside the table region
  size_t t_qpoint, t_gt_off, t_gt_ids, t_levels, t_rank, t_bytes;
  int n_queries = 0, minmax_slots = 0, max_prompts = 1, s_ld = 0, tile_rows = 0;  // max_prompts: over the scenes with queries
  int64_t n_rows = 0, n_text_rows = 0, n_neg = 0, max_points = 0;  // max_points: over the scenes with queries
  int64_t n_gt = -1;              // dc_predict_many_iou: the number of ground-truth ids; -1: no counting
  int n_thr = 0;                  // dc_predict_many_iou_sweep: the number of thresholds; 0: one threshold
  std::vector<float> levels;      // sweep: the distinct threshold levels, ascending (threshold_levels)
  std::vector<int> rank;          // sweep: [n_thr], threshold t's index in `levels`
  std::vector<int64_t> qrow_off;  // [n_queries + 1]: query q's row of v / pred
  std::vector<int64_t> qpoint;    // counting: [n_queries], the feature row of query q's first point
  std::vector<ScoreScene> scenes;
  std::vector<ScoreBlock> blocks;
  std::vector<int4> tiles;                            // the column blocks' tile lists, one after the other
  std::vector<int> tile_start, tile_count, tile_bn;   // per block of 256 prompt columns
};

// tile_list: dc_predict_many's GEMM (explicit tiles, S row stride = the widest scene rounded up to 4); otherwise
// dc_ground writes S [n_points, n_prompts] of the one scene densely. reverse: list the first column block's tiles last
// to first (the rows normalised last are still in L2, as in dc_ground). n_gt >= 0: the plan of dc_predict_many_iou with
// n_gt ground-truth ids; with n_thr > 0 as well, the plan of dc_predict_many_iou_sweep with n_thr thresholds.
ScorePlan score_plan(int n_scenes, const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off,
                     int64_t n_neg, int dim, int feat_dtype, int text_dtype, bool tile_list, bool reverse,
                     int64_t n_gt = -1, int n_thr = 0) {
  ScorePlan pl;
  pl.n_rows = point_off[n_scenes];
  pl.n_text_rows = prompt_off[n_scenes];
  pl.n_queries = query_off[n_scenes];
  pl.n_neg = n_neg;
  pl.n_gt = n_gt;
  pl.n_thr = n_thr;
  const bool count = n_gt >= 0;
  int& max_prompts = pl.max_prompts;
  int64_t out_off = 0;
  for (int s = 0; s < n_scenes; ++s) {
    const int64_t ns = point_off[s + 1] - point_off[s];
    const int ps = prompt_off[s + 1] - prompt_off[s], qs = query_off[s + 1] - query_off[s];
    pl.scenes.push_back(ScoreScene{point_off[s], out_off, (int)ns, ps, query_off[s], 0});
    for (int q = 0; q < qs; ++q) pl.qrow_off.push_back(out_off + q * ns);
    if (count) pl.qpoint.insert(pl.qpoint.end(), qs, point_off[s]);
    out_off += qs * ns;
    if (qs > 0) {
      max_prompts = std::max(max_prompts, ps);
      pl.max_points = std::max(pl.max_points, ns);
    }
  }
  pl.qrow_off.push_back(out_off);
  pl.s_ld = tile_list ? (max_prompts + 3) / 4 * 4 : max_prompts;
  // rows of S per block: as many as fit 48 KB of shared memory at the widest scene, 32 to 256
  pl.tile_rows = 256;
  while (pl.tile_rows > 32 && (size_t)pl.tile_rows * (max_prompts | 1) * sizeof(float) > 48 * 1024) pl.tile_rows >>= 1;
  int64_t score_tiles = 0;
  for (int s = 0; s < n_scenes; ++s)
    if (query_off[s + 1] > query_off[s]) score_tiles += dc::ceil_div<int64_t>(point_off[s + 1] - point_off[s], pl.tile_rows);
  // few row tiles (small scenes): split each scene's queries over more blocks, up to 4 blocks per SM in all
  const int64_t want = score_tiles ? dc::ceil_div<int64_t>(4 * (int64_t)dc::sm_count(), score_tiles) : 1;
  for (int s = 0; s < n_scenes; ++s) {
    const int64_t ns = point_off[s + 1] - point_off[s];
    const int qs = query_off[s + 1] - query_off[s], q0 = query_off[s];
    if (qs == 0) continue;
    const int q_per_chunk = (int)dc::ceil_div<int64_t>(qs, std::min<int64_t>(qs, want));
    for (int64_t r0 = 0; r0 < ns; r0 += pl.tile_rows)
      for (int c0 = 0; c0 < qs; c0 += q_per_chunk)
        pl.blocks.push_back(ScoreBlock{s, (int)r0, (int)std::min<int64_t>(pl.tile_rows, ns - r0), q0 + c0,
                                       q0 + std::min(qs, c0 + q_per_chunk)});
  }
  if (tile_list) {
    for (int c0 = 0; c0 < max_prompts; c0 += 256) {
      const int start = (int)pl.tiles.size();
      int widest = 1;
      for (int s = 0; s < n_scenes; ++s) {
        const int ps = prompt_off[s + 1] - prompt_off[s];
        if (query_off[s + 1] == query_off[s] || ps <= c0) continue;
        const int cols = std::min(256, ps - c0);
        widest = std::max(widest, cols);
        for (int64_t r0 = point_off[s]; r0 < point_off[s + 1]; r0 += dc::gemm::kBlockM)
          pl.tiles.push_back(make_int4((int)r0, prompt_off[s] + c0, (int)std::min<int64_t>(dc::gemm::kBlockM, point_off[s + 1] - r0),
                                       cols));
      }
      if (reverse && c0 == 0) std::reverse(pl.tiles.begin() + start, pl.tiles.end());
      pl.tile_start.push_back(start);
      pl.tile_count.push_back((int)pl.tiles.size() - start);
      pl.tile_bn.push_back(pick_bn(widest));
    }
  }
  const size_t q = (size_t)pl.n_queries;
  size_t t = 0;
  pl.t_qrow = t; t += align_up(sizeof(int64_t) * (q + 1), 16);
  pl.t_pos = t; t += align_up(sizeof(int) * q, 16);
  pl.t_off = t; t += align_up(sizeof(int) * (q + 1), 16);
  pl.t_cols = t; t += align_up(sizeof(int) * (size_t)n_neg, 16);
  pl.t_scenes = t; t += align_up(sizeof(ScoreScene) * pl.scenes.size(), 16);
  pl.t_blocks = t; t += align_up(sizeof(ScoreBlock) * pl.blocks.size(), 16);
  pl.t_counts = t; t += align_up(sizeof(int) * pl.tile_count.size(), 16);
  pl.t_tiles = t; t += align_up(sizeof(int4) * pl.tiles.size(), 16);
  pl.t_qpoint = t; if (count) t += align_up(sizeof(int64_t) * q, 16);
  pl.t_gt_off = t; if (count) t += align_up(sizeof(int) * (q + 1), 16);
  pl.t_gt_ids = t; if (count) t += sizeof(int64_t) * (size_t)n_gt;
  if (n_thr > 0) t = align_up(t, 16);
  pl.t_levels = t; t += sizeof(float) * (size_t)n_thr;
  pl.t_rank = t; t += sizeof(int) * (size_t)n_thr;
  pl.t_bytes = t;
  pl.minmax_slots = pl.n_queries + (tile_list ? 0 : 1);  // + dc_ground's extrema, unused
  size_t off = 0;
  pl.minmax = off; off += align_up(sizeof(float) * 4 * (size_t)pl.minmax_slots, 256);
  pl.tables = off; off += align_up(t, 256);
  pl.t_planes = off; if (text_dtype == DC_F32) off += 2 * align_up((size_t)pl.n_text_rows * dim * 2, 256);
  pl.x_planes = off; if (feat_dtype == DC_F32) off += 2 * align_up((size_t)(pl.n_rows > 0 ? pl.n_rows : 1) * dim * 2, 256);
  pl.sims = off; off += align_up((size_t)(pl.n_rows > 0 ? pl.n_rows : 1) * pl.s_ld * sizeof(float), 256);
  pl.v = off; if (count) off += align_up(sizeof(float) * (size_t)out_off, 256);
  pl.pred = off; if (count) off += align_up((size_t)out_off, 256);
  pl.hist = off; off += align_up(sizeof(unsigned) * 2 * (size_t)(n_thr > 0 ? n_thr + 1 : 0) * q, 256);
  pl.total = off;
  return pl;
}

// The column tables live in host memory: query q of scene s has its positive and negative columns in [0, P_s).
int check_columns(const char* fn, int n_scenes, const int32_t* prompt_off, const int32_t* query_off, const int32_t* pos,
                  const int32_t* neg_off, const int32_t* neg_cols, int mode) {
  DC_CHECK_ARG(neg_off[0] == 0, "%s: neg_off[0] must be 0", fn);
  for (int s = 0; s < n_scenes; ++s) {
    const int n_prompts = prompt_off[s + 1] - prompt_off[s];
    for (int q = query_off[s]; q < query_off[s + 1]; ++q) {
      const int m = neg_off[q + 1] - neg_off[q];
      DC_CHECK_ARG(pos[q] >= 0 && pos[q] < n_prompts, "%s: query %d: positive column %d outside [0, %d)", fn, q, pos[q],
                   n_prompts);
      DC_CHECK_ARG(m >= 0, "%s: neg_off must not decrease (query %d)", fn, q);
      DC_CHECK_ARG(mode != DC_GROUND_RAW || m == 0, "%s: raw mode is the no-negatives case (query %d has %d)", fn, q, m);
      DC_CHECK_ARG(mode == DC_GROUND_RAW || m >= 1, "%s: paired/argmax need a negative for every query (query %d)", fn, q);
    }
  }
  const int n_queries = query_off[n_scenes];
  DC_CHECK_ARG(neg_off[n_queries] == 0 || neg_cols, "%s: null pointer argument", fn);
  for (int s = 0; s < n_scenes; ++s) {
    const int n_prompts = prompt_off[s + 1] - prompt_off[s];
    for (int64_t j = neg_off[query_off[s]]; j < neg_off[query_off[s + 1]]; ++j)
      DC_CHECK_ARG(neg_cols[j] >= 0 && neg_cols[j] < n_prompts, "%s: negative column %d outside [0, %d)", fn, neg_cols[j],
                   n_prompts);
  }
  return DC_OK;
}

int stage_tables(const ScorePlan& pl, const int32_t* pos, const int32_t* neg_off, const int32_t* neg_cols, uint8_t* ws,
                 cudaStream_t st, const int32_t* gt_off = nullptr, const int64_t* gt_ids = nullptr) {
  std::vector<uint8_t> h(pl.t_bytes);
  auto put = [&](size_t at, const void* src, size_t bytes) {
    if (bytes) memcpy(h.data() + at, src, bytes);
  };
  const size_t q = (size_t)pl.n_queries;
  put(pl.t_qrow, pl.qrow_off.data(), sizeof(int64_t) * (q + 1));
  put(pl.t_pos, pos, sizeof(int) * q);
  put(pl.t_off, neg_off, sizeof(int) * (q + 1));
  put(pl.t_cols, neg_cols, sizeof(int) * (size_t)pl.n_neg);
  put(pl.t_scenes, pl.scenes.data(), sizeof(ScoreScene) * pl.scenes.size());
  put(pl.t_blocks, pl.blocks.data(), sizeof(ScoreBlock) * pl.blocks.size());
  put(pl.t_counts, pl.tile_count.data(), sizeof(int) * pl.tile_count.size());
  put(pl.t_tiles, pl.tiles.data(), sizeof(int4) * pl.tiles.size());
  if (pl.n_gt >= 0) {
    put(pl.t_qpoint, pl.qpoint.data(), sizeof(int64_t) * q);
    put(pl.t_gt_off, gt_off, sizeof(int) * (q + 1));
    put(pl.t_gt_ids, gt_ids, sizeof(int64_t) * (size_t)pl.n_gt);
  }
  put(pl.t_levels, pl.levels.data(), sizeof(float) * pl.levels.size());
  put(pl.t_rank, pl.rank.data(), sizeof(int) * pl.rank.size());
  // pageable source: cudaMemcpyAsync returns once it has staged the bytes, so `h` may go out of scope
  DC_CUDA(cudaMemcpyAsync(ws + pl.tables, h.data(), pl.t_bytes, cudaMemcpyHostToDevice, st));
  return DC_OK;
}

// Every query scored from its columns of S [n_rows, s_ld], then its min-max and threshold (one launch each). With `cnt`
// (dc_predict_many_iou) the second launch counts against the labels of dtype label_dtype instead of writing v and pred;
// a sweep plan (dc_predict_many_iou_sweep) replaces it with threshold_sweep_kernel into the zeroed histograms, then
// sweep_counts_kernel writes cnt.inter / cnt.uni [n_thr][n_queries].
int score_queries(const ScorePlan& pl, uint8_t* ws, int mode, float softmax_temp, float threshold, float* out,
                  uint8_t* pred, cudaStream_t st, const IouCount* cnt = nullptr, int label_dtype = DC_I64) {
  if (pl.blocks.empty()) return DC_OK;
  DC_CHECK_ARG(pl.blocks.size() < (1ull << 31), "too many score blocks for one launch");
  const uint8_t* tb = ws + pl.tables;
  const int64_t* qrow = reinterpret_cast<const int64_t*>(tb + pl.t_qrow);
  const int* d_pos = reinterpret_cast<const int*>(tb + pl.t_pos);
  const int* d_off = reinterpret_cast<const int*>(tb + pl.t_off);
  const int* d_cols = reinterpret_cast<const int*>(tb + pl.t_cols);
  const ScoreScene* scenes = reinterpret_cast<const ScoreScene*>(tb + pl.t_scenes);
  const ScoreBlock* blocks = reinterpret_cast<const ScoreBlock*>(tb + pl.t_blocks);
  const float* sims = reinterpret_cast<const float*>(ws + pl.sims);
  float* minmax = reinterpret_cast<float*>(ws + pl.minmax);
  const size_t smem = (size_t)pl.tile_rows * (pl.max_prompts | 1) * sizeof(float);
  const float inv_temp = 1.0f / softmax_temp;
  // the attribute belongs to the (function, device) pair: set for the device in use whenever a tile needs > 48 KB
  const void* fn = mode == DC_GROUND_PAIRED ? (const void*)query_scores_kernel<DC_GROUND_PAIRED>
                 : mode == DC_GROUND_ARGMAX ? (const void*)query_scores_kernel<DC_GROUND_ARGMAX>
                                            : (const void*)query_scores_kernel<DC_GROUND_RAW>;
  if (smem > 48 * 1024) DC_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned grid = (unsigned)pl.blocks.size();
#define DC_QUERY_SCORES(M)                                                                                             \
  query_scores_kernel<M><<<grid, 256, smem, st>>>(sims, pl.s_ld, blocks, scenes, d_pos, d_off, d_cols, pl.tile_rows, \
                                                  inv_temp, out, pred, minmax)
  if (mode == DC_GROUND_PAIRED) DC_QUERY_SCORES(DC_GROUND_PAIRED);
  else if (mode == DC_GROUND_ARGMAX) DC_QUERY_SCORES(DC_GROUND_ARGMAX);
  else DC_QUERY_SCORES(DC_GROUND_RAW);
#undef DC_QUERY_SCORES
  DC_LAUNCH_CHECK();
  // per-query min-max (+ threshold), every query in one launch (blockIdx.y = query, its row from the table)
  const int64_t blocks_x = dc::ceil_div<int64_t>(pl.max_points, 256);
  const int64_t per_query = std::max<int64_t>(1, dc::ceil_div<int64_t>((int64_t)dc::sm_count() * 8, pl.n_queries));
  const dim3 mm_grid((unsigned)std::min(blocks_x, per_query), (unsigned)pl.n_queries);
  const int use_raw = mode == DC_GROUND_ARGMAX ? 1 : 0, pred_from_thr = mode == DC_GROUND_ARGMAX ? 0 : 1;
  if (pl.n_thr > 0) {
    const int n_levels = (int)pl.levels.size();
    const float* levels = reinterpret_cast<const float*>(tb + pl.t_levels);
    unsigned* hist = reinterpret_cast<unsigned*>(ws + pl.hist);
    const size_t sweep_smem = sizeof(unsigned) * 2 * (n_levels + 1) + sizeof(float) * n_levels;
    if (label_dtype == DC_I32)
      threshold_sweep_kernel<int32_t><<<mm_grid, 256, sweep_smem, st>>>(out, minmax, use_raw, pred_from_thr, pred, qrow,
                                                                        levels, n_levels, *cnt, hist);
    else
      threshold_sweep_kernel<int64_t><<<mm_grid, 256, sweep_smem, st>>>(out, minmax, use_raw, pred_from_thr, pred, qrow,
                                                                        levels, n_levels, *cnt, hist);
    DC_LAUNCH_CHECK();
    sweep_counts_kernel<<<(unsigned)pl.n_queries, 256, sizeof(unsigned) * 2 * (n_levels + 1), st>>>(
        hist, n_levels, reinterpret_cast<const int*>(tb + pl.t_rank), pl.n_thr, pl.n_queries,
        reinterpret_cast<int64_t*>(cnt->inter), reinterpret_cast<int64_t*>(cnt->uni));
  } else if (!cnt)
    minmax_threshold_kernel<void><<<mm_grid, 256, 0, st>>>(out, 0, minmax, use_raw, threshold, pred_from_thr, pred, qrow);
  else if (label_dtype == DC_I32)
    minmax_threshold_kernel<int32_t><<<mm_grid, 256, 0, st>>>(out, 0, minmax, use_raw, threshold, pred_from_thr, pred, qrow,
                                                              *cnt);
  else
    minmax_threshold_kernel<int64_t><<<mm_grid, 256, 0, st>>>(out, 0, minmax, use_raw, threshold, pred_from_thr, pred, qrow,
                                                              *cnt);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

// fp32 prompt rows: their fp16 hi/lo operand planes in the workspace; fp16 prompts are used as they are
int prompt_planes(const ScorePlan& pl, const void* text, int text_dtype, int dim, uint8_t* ws, const void** t_hi,
                  const void** t_lo, cudaStream_t st) {
  *t_hi = text;
  *t_lo = nullptr;
  if (text_dtype != DC_F32) return DC_OK;
  const size_t pb = align_up((size_t)pl.n_text_rows * dim * 2, 256);
  int rc;
  if ((rc = launch_row_normalize(const_cast<void*>(text), DC_F32, pl.n_text_rows, dim, 0, false, ws + pl.t_planes,
                                 ws + pl.t_planes + pb, st)))
    return rc;
  *t_hi = ws + pl.t_planes;
  *t_lo = ws + pl.t_planes + pb;
  return DC_OK;
}

}  // namespace

extern "C" {

size_t dc_predict_queries_workspace(int64_t n_points, int n_prompts, int n_queries, int64_t n_neg_total, int dim,
                                    int feat_dtype, int text_dtype) {
  const int64_t point_off[2] = {0, n_points > 0 ? n_points : 0};
  const int32_t prompt_off[2] = {0, n_prompts}, query_off[2] = {0, n_queries};
  return score_plan(1, point_off, prompt_off, query_off, n_neg_total, dim, feat_dtype, text_dtype, false, false).total;
}

int dc_predict_queries(void* feats, int feat_dtype, int64_t n_points, const void* text, int text_dtype, int n_prompts,
                       int dim, const int32_t* pos, const int32_t* neg_off, const int32_t* neg_cols, int n_queries, int mode,
                       float softmax_temp, int normalize, float threshold, float* out, uint8_t* pred, void* workspace,
                       size_t workspace_bytes, dc_stream_t stream) {
  DC_CHECK_ARG(text && pos && neg_off && workspace, "dc_predict_queries: null pointer argument");
  DC_CHECK_ARG(n_points <= 0 || (feats && out && pred), "dc_predict_queries: null pointer argument");  // empty tensors have none
  DC_CHECK_ARG(feat_dtype == DC_F16 || feat_dtype == DC_F32, "dc_predict_queries: features must be fp16 or fp32");
  DC_CHECK_ARG(text_dtype == DC_F16 || text_dtype == DC_F32, "dc_predict_queries: prompt embeddings must be fp16 or fp32");
  DC_CHECK_ARG(mode == DC_GROUND_RAW || mode == DC_GROUND_PAIRED || mode == DC_GROUND_ARGMAX, "dc_predict_queries: bad mode");
  DC_CHECK_ARG(n_queries >= 1 && n_queries <= 65535, "dc_predict_queries: 1..65535 queries (got %d)", n_queries);
  DC_CHECK_ARG(n_prompts >= 1 && n_prompts <= kQueryMaxPrompts, "dc_predict_queries: 1..%d prompts (got %d)", kQueryMaxPrompts,
               n_prompts);
  DC_CHECK_ARG(dim > 0 && dim % 64 == 0, "dc_predict_queries: feature dim must be a multiple of 64 (got %d)", dim);
  DC_CHECK_ARG(n_points < (1ll << 31), "dc_predict_queries: too many points for one call");
  DC_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "dc_predict_queries: workspace must be 256-byte aligned");
  const int64_t point_off[2] = {0, n_points > 0 ? n_points : 0};
  const int32_t prompt_off[2] = {0, n_prompts}, query_off[2] = {0, n_queries};
  int rc;
  if ((rc = check_columns("dc_predict_queries", 1, prompt_off, query_off, pos, neg_off, neg_cols, mode))) return rc;
  const ScorePlan pl = score_plan(1, point_off, prompt_off, query_off, neg_off[n_queries], dim, feat_dtype, text_dtype,
                                  false, false);
  if (workspace_bytes < pl.total)
    return dc::fail(DC_ERR_WORKSPACE, "dc_predict_queries: workspace %zu < %zu", workspace_bytes, pl.total);
  cudaStream_t st = dc::as_stream(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  float* minmax = reinterpret_cast<float*>(ws + pl.minmax);
  init_query_minmax_kernel<<<1, 256, 0, st>>>(minmax, pl.minmax_slots);
  DC_LAUNCH_CHECK();
  if (n_points <= 0) return DC_OK;
  if ((rc = stage_tables(pl, pos, neg_off, neg_cols, ws, st))) return rc;
  // prologue of dc_predict: operand planes of fp32 prompts and fp32 features (normalised in place when asked); fp16
  // features are normalised in place by dc_ground
  const void *t_hi, *t_lo;
  if ((rc = prompt_planes(pl, text, text_dtype, dim, ws, &t_hi, &t_lo, st))) return rc;
  const void *x_hi = feats, *x_lo = nullptr;
  if (feat_dtype == DC_F32) {
    const size_t xb = align_up((size_t)n_points * dim * 2, 256);
    if ((rc = launch_row_normalize(feats, DC_F32, n_points, dim, normalize, true, ws + pl.x_planes, ws + pl.x_planes + xb, st)))
      return rc;
    x_hi = ws + pl.x_planes;
    x_lo = ws + pl.x_planes + xb;
  }
  // S = X . T^T once, every distinct prompt a column
  float* sims = reinterpret_cast<float*>(ws + pl.sims);
  if ((rc = dc_ground(x_hi, x_lo, n_points, t_hi, t_lo, n_prompts, dim, DC_GROUND_RAW, softmax_temp,
                      (feat_dtype == DC_F16 && normalize) ? 1 : 0, sims, n_prompts, nullptr, nullptr,
                      minmax + 4 * n_queries, nullptr, 0, stream)))
    return rc;
  return score_queries(pl, ws, mode, softmax_temp, threshold, out, pred, st);
}

}  // extern "C"

namespace {

// The ground-truth side of dc_predict_many_iou; with n_thresholds > 0, of dc_predict_many_iou_sweep (inter / uni are
// then [n_thresholds][sum Q]).
struct IouArgs {
  const void* labels;
  int label_dtype;
  const int32_t* gt_off;
  const int64_t* gt_ids;
  int64_t* inter;
  int64_t* uni;
  const float* thresholds;
  int n_thresholds;
};

size_t predict_many_workspace(int n_scenes, const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off,
                              int64_t n_neg_total, int dim, int feat_dtype, int text_dtype, int64_t n_gt, int n_thr = 0) {
  if (n_scenes < 0 || (n_scenes > 0 && !(point_off && prompt_off && query_off))) return 0;
  const int64_t zero64 = 0;
  const int32_t zero32 = 0;
  if (n_scenes == 0)
    return score_plan(0, &zero64, &zero32, &zero32, 0, dim, feat_dtype, text_dtype, true, false, n_gt >= 0 ? 0 : -1,
                      n_thr).total;
  return score_plan(n_scenes, point_off, prompt_off, query_off, n_neg_total, dim, feat_dtype, text_dtype, true, false,
                    n_gt, n_thr).total;
}

int check_thresholds(const char* fn, const float* thresholds, int n_thresholds) {
  DC_CHECK_ARG(n_thresholds >= 1 && n_thresholds <= kSweepMaxThresholds, "%s: 1..%d thresholds (got %d)", fn,
               kSweepMaxThresholds, n_thresholds);
  DC_CHECK_ARG(thresholds, "%s: null pointer argument", fn);
  return DC_OK;
}

// The sweep's threshold tables: the distinct values of thresholds[0 .. n) ascending, a NaN as +inf (x > NaN and
// x > +inf are false for every x), and rank[t] = the index of entry t's value among them. -0 and +0 are one level.
void threshold_levels(const float* thresholds, int n, std::vector<float>& levels, std::vector<int>& rank) {
  std::vector<float> vals(n);
  for (int t = 0; t < n; ++t) vals[t] = thresholds[t] != thresholds[t] ? INFINITY : thresholds[t];
  levels = vals;
  std::sort(levels.begin(), levels.end());
  levels.erase(std::unique(levels.begin(), levels.end()), levels.end());
  rank.resize(n);
  for (int t = 0; t < n; ++t) rank[t] = (int)(std::lower_bound(levels.begin(), levels.end(), vals[t]) - levels.begin());
}

// dc_predict_many (iou == nullptr: the scores and predictions go to out / pred) and dc_predict_many_iou (the scores and
// the argmax bytes stay in the workspace; the threshold pass counts against the ground truth instead). `fn` names the
// entry point in the error messages.
int predict_many(const char* fn, void* feats, int feat_dtype, const void* text, int text_dtype, int dim, int n_scenes,
                 const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off, const int32_t* pos,
                 const int32_t* neg_off, const int32_t* neg_cols, int mode, float softmax_temp, int normalize,
                 float threshold, float* out, uint8_t* pred, const IouArgs* iou, void* workspace, size_t workspace_bytes,
                 dc_stream_t stream) {
  DC_CHECK_ARG(n_scenes >= 0, "%s: negative scene count", fn);
  if (n_scenes == 0) return DC_OK;
  DC_CHECK_ARG(point_off && prompt_off && query_off && neg_off && workspace, "%s: null pointer argument", fn);
  DC_CHECK_ARG(feat_dtype == DC_F16 || feat_dtype == DC_F32, "%s: features must be fp16 or fp32", fn);
  DC_CHECK_ARG(text_dtype == DC_F16 || text_dtype == DC_F32, "%s: prompt embeddings must be fp16 or fp32", fn);
  DC_CHECK_ARG(mode == DC_GROUND_RAW || mode == DC_GROUND_PAIRED || mode == DC_GROUND_ARGMAX, "%s: bad mode", fn);
  DC_CHECK_ARG(dim > 0 && dim % 64 == 0, "%s: feature dim must be a multiple of 64 (got %d)", fn, dim);
  DC_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "%s: workspace must be 256-byte aligned", fn);
  DC_CHECK_ARG(point_off[0] == 0 && prompt_off[0] == 0 && query_off[0] == 0, "%s: offset tables must start at 0", fn);
  for (int s = 0; s < n_scenes; ++s) {
    const int64_t ns = point_off[s + 1] - point_off[s];
    const int ps = prompt_off[s + 1] - prompt_off[s], qs = query_off[s + 1] - query_off[s];
    DC_CHECK_ARG(ns >= 0 && ps >= 0 && qs >= 0, "%s: offset tables must not decrease (scene %d)", fn, s);
    DC_CHECK_ARG(ps <= kQueryMaxPrompts, "%s: scene %d: 0..%d prompts (got %d)", fn, s, kQueryMaxPrompts, ps);
    DC_CHECK_ARG(qs == 0 || ps >= 1, "%s: scene %d has queries but no prompts", fn, s);
  }
  const int64_t n_rows = point_off[n_scenes];
  const int n_queries = query_off[n_scenes];
  DC_CHECK_ARG(n_rows < (1ll << 31), "%s: too many points for one call (%lld)", fn, (long long)n_rows);
  DC_CHECK_ARG(n_queries <= 65535, "%s: at most 65535 queries in all (got %d)", fn, n_queries);
  DC_CHECK_ARG(n_rows == 0 || feats, "%s: null pointer argument", fn);
  DC_CHECK_ARG(prompt_off[n_scenes] == 0 || text, "%s: null pointer argument", fn);
  int64_t n_cells = 0;
  for (int s = 0; s < n_scenes; ++s)
    n_cells += (int64_t)(query_off[s + 1] - query_off[s]) * (point_off[s + 1] - point_off[s]);
  DC_CHECK_ARG(iou || n_cells == 0 || (out && pred), "%s: null pointer argument", fn);
  DC_CHECK_ARG(n_queries == 0 || pos, "%s: null pointer argument", fn);
  int rc;
  if ((rc = check_columns(fn, n_scenes, prompt_off, query_off, pos, neg_off, neg_cols, mode))) return rc;
  int64_t n_gt = -1;
  if (iou) {
    DC_CHECK_ARG(iou->label_dtype == DC_I32 || iou->label_dtype == DC_I64, "%s: labels must be int32 or int64", fn);
    DC_CHECK_ARG(n_queries == 0 || (iou->gt_off && iou->inter && iou->uni), "%s: null pointer argument", fn);
    DC_CHECK_ARG(n_cells == 0 || iou->labels, "%s: null pointer argument", fn);
    if (n_queries > 0) {
      const int32_t* g = iou->gt_off;
      DC_CHECK_ARG(g[0] == 0, "%s: gt_off[0] must be 0", fn);
      for (int q = 0; q < n_queries; ++q) {
        DC_CHECK_ARG(g[q + 1] >= g[q], "%s: gt_off must not decrease (query %d)", fn, q);
        for (int j = g[q] + 1; j < g[q + 1]; ++j)
          DC_CHECK_ARG(iou->gt_ids[j] > iou->gt_ids[j - 1], "%s: query %d: ground-truth ids must be strictly ascending", fn,
                       q);
      }
      n_gt = g[n_queries];
      DC_CHECK_ARG(n_gt == 0 || iou->gt_ids, "%s: null pointer argument", fn);
    }
  }
  if (n_queries == 0) return DC_OK;
  cudaStream_t st = dc::as_stream(stream);
  const int n_thr = iou ? iou->n_thresholds : 0;
  ScorePlan pl = score_plan(n_scenes, point_off, prompt_off, query_off, neg_off[n_queries], dim, feat_dtype, text_dtype,
                            true, feat_dtype == DC_F16 && normalize, n_gt, n_thr);
  if (workspace_bytes < pl.total) return dc::fail(DC_ERR_WORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, pl.total);
  if (n_thr > 0) threshold_levels(iou->thresholds, n_thr, pl.levels, pl.rank);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  IouCount cnt{};
  if (iou) {
    // every query reports 0 / 0 until its blocks add to it (a query of an empty scene gets none)
    const size_t rows = (size_t)std::max(n_thr, 1) * n_queries;
    DC_CUDA(cudaMemsetAsync(iou->inter, 0, sizeof(int64_t) * rows, st));
    DC_CUDA(cudaMemsetAsync(iou->uni, 0, sizeof(int64_t) * rows, st));
    if (n_thr > 0) DC_CUDA(cudaMemsetAsync(ws + pl.hist, 0, sizeof(unsigned) * 2 * (pl.levels.size() + 1) * n_queries, st));
    out = reinterpret_cast<float*>(ws + pl.v);
    pred = ws + pl.pred;
    const uint8_t* tb = ws + pl.tables;
    cnt = IouCount{iou->labels, reinterpret_cast<const int64_t*>(tb + pl.t_qpoint), reinterpret_cast<const int*>(tb + pl.t_gt_off),
                   reinterpret_cast<const int64_t*>(tb + pl.t_gt_ids), reinterpret_cast<unsigned long long*>(iou->inter),
                   reinterpret_cast<unsigned long long*>(iou->uni)};
  }
  float* minmax = reinterpret_cast<float*>(ws + pl.minmax);
  init_query_minmax_kernel<<<1, 256, 0, st>>>(minmax, pl.minmax_slots);
  DC_LAUNCH_CHECK();
  if (pl.blocks.empty()) return DC_OK;  // every scene with queries is empty
  if ((rc = stage_tables(pl, pos, neg_off, neg_cols, ws, st, iou ? iou->gt_off : nullptr, iou ? iou->gt_ids : nullptr)))
    return rc;
  const void *t_hi, *t_lo;
  if ((rc = prompt_planes(pl, text, text_dtype, dim, ws, &t_hi, &t_lo, st))) return rc;
  // the features of the scenes with queries, normalised in place (when asked) as dc_predict_queries does: fp32 rows
  // also get their operand planes. One launch per run of consecutive such scenes (one launch when every scene has
  // queries); the rows of a scene without queries stay untouched.
  const size_t xb = align_up((size_t)n_rows * dim * 2, 256);
  const size_t row_bytes = (size_t)dim * (feat_dtype == DC_F32 ? 4 : 2);
  const void *x_hi = feats, *x_lo = nullptr;
  if (feat_dtype == DC_F32) {
    x_hi = ws + pl.x_planes;
    x_lo = ws + pl.x_planes + xb;
  }
  if (feat_dtype == DC_F32 || normalize) {
    for (int s = 0; s < n_scenes;) {
      if (query_off[s + 1] == query_off[s]) { ++s; continue; }
      int e = s + 1;
      while (e < n_scenes && query_off[e + 1] > query_off[e]) ++e;
      const int64_t r0 = point_off[s], rows = point_off[e] - r0;
      uint8_t* hi = feat_dtype == DC_F32 ? ws + pl.x_planes + (size_t)r0 * dim * 2 : nullptr;
      uint8_t* lo = feat_dtype == DC_F32 ? hi + xb : nullptr;
      if ((rc = launch_row_normalize(static_cast<uint8_t*>(feats) + (size_t)r0 * row_bytes, feat_dtype, rows, dim, normalize,
                                     true, hi, lo, st)))
        return rc;
      s = e;
    }
  }
  // S = X . T^T of every scene with its own prompts: one tcgen05 GEMM per block of 256 prompt columns over the tile list
  // (a tile = 128 rows of one scene x that scene's columns of the block), written once at the row stride s_ld
  const uint8_t* tb = ws + pl.tables;
  float* sims = reinterpret_cast<float*>(ws + pl.sims);
  for (size_t cb = 0; cb < pl.tile_count.size(); ++cb) {
    if (pl.tile_count[cb] == 0) continue;
    Params p{reinterpret_cast<const int4*>(tb + pl.t_tiles) + pl.tile_start[cb],
             reinterpret_cast<const int*>(tb + pl.t_counts) + cb, n_rows, 0, dim};
    dc::gemm::set_terms(p, x_lo, t_lo);
    EpiStore epi{sims + 256 * cb, pl.s_ld};
    if ((rc = launch_bn(pl.tile_bn[cb], x_hi, x_lo, n_rows, t_hi, t_lo, pl.n_text_rows, p, epi,
                        pl.tile_count[cb], st)))
      return rc;
  }
  return score_queries(pl, ws, mode, softmax_temp, threshold, out, pred, st, iou ? &cnt : nullptr,
                       iou ? iou->label_dtype : DC_I64);
}

}  // namespace

extern "C" {

size_t dc_predict_many_workspace(int n_scenes, const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off,
                                 int64_t n_neg_total, int dim, int feat_dtype, int text_dtype) {
  return predict_many_workspace(n_scenes, point_off, prompt_off, query_off, n_neg_total, dim, feat_dtype, text_dtype, -1);
}

int dc_predict_many(void* feats, int feat_dtype, const void* text, int text_dtype, int dim, int n_scenes,
                    const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off, const int32_t* pos,
                    const int32_t* neg_off, const int32_t* neg_cols, int mode, float softmax_temp, int normalize,
                    float threshold, float* out, uint8_t* pred, void* workspace, size_t workspace_bytes,
                    dc_stream_t stream) {
  return predict_many("dc_predict_many", feats, feat_dtype, text, text_dtype, dim, n_scenes, point_off, prompt_off,
                      query_off, pos, neg_off, neg_cols, mode, softmax_temp, normalize, threshold, out, pred, nullptr,
                      workspace, workspace_bytes, stream);
}

size_t dc_predict_many_iou_workspace(int n_scenes, const int64_t* point_off, const int32_t* prompt_off,
                                     const int32_t* query_off, int64_t n_neg_total, int64_t n_gt_total, int dim,
                                     int feat_dtype, int text_dtype) {
  return predict_many_workspace(n_scenes, point_off, prompt_off, query_off, n_neg_total, dim, feat_dtype, text_dtype,
                                n_gt_total > 0 ? n_gt_total : 0);
}

int dc_predict_many_iou(void* feats, int feat_dtype, const void* text, int text_dtype, int dim, int n_scenes,
                        const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off, const int32_t* pos,
                        const int32_t* neg_off, const int32_t* neg_cols, const void* labels, int label_dtype,
                        const int32_t* gt_off, const int64_t* gt_ids, int mode, float softmax_temp, int normalize,
                        float threshold, int64_t* inter, int64_t* uni, void* workspace, size_t workspace_bytes,
                        dc_stream_t stream) {
  const IouArgs iou{labels, label_dtype, gt_off, gt_ids, inter, uni};
  return predict_many("dc_predict_many_iou", feats, feat_dtype, text, text_dtype, dim, n_scenes, point_off, prompt_off,
                      query_off, pos, neg_off, neg_cols, mode, softmax_temp, normalize, threshold, nullptr, nullptr, &iou,
                      workspace, workspace_bytes, stream);
}

size_t dc_predict_many_iou_sweep_workspace(int n_scenes, const int64_t* point_off, const int32_t* prompt_off,
                                           const int32_t* query_off, int64_t n_neg_total, int64_t n_gt_total,
                                           int n_thresholds, int dim, int feat_dtype, int text_dtype) {
  if (n_thresholds < 1 || n_thresholds > kSweepMaxThresholds) return 0;
  return predict_many_workspace(n_scenes, point_off, prompt_off, query_off, n_neg_total, dim, feat_dtype, text_dtype,
                                n_gt_total > 0 ? n_gt_total : 0, n_thresholds);
}

int dc_predict_many_iou_sweep(void* feats, int feat_dtype, const void* text, int text_dtype, int dim, int n_scenes,
                              const int64_t* point_off, const int32_t* prompt_off, const int32_t* query_off,
                              const int32_t* pos, const int32_t* neg_off, const int32_t* neg_cols, const void* labels,
                              int label_dtype, const int32_t* gt_off, const int64_t* gt_ids, int mode, float softmax_temp,
                              int normalize, const float* thresholds, int n_thresholds, int64_t* inter, int64_t* uni,
                              void* workspace, size_t workspace_bytes, dc_stream_t stream) {
  int rc;
  if ((rc = check_thresholds("dc_predict_many_iou_sweep", thresholds, n_thresholds))) return rc;
  const IouArgs iou{labels, label_dtype, gt_off, gt_ids, inter, uni, thresholds, n_thresholds};
  return predict_many("dc_predict_many_iou_sweep", feats, feat_dtype, text, text_dtype, dim, n_scenes, point_off,
                      prompt_off, query_off, pos, neg_off, neg_cols, mode, softmax_temp, normalize, 0.f, nullptr, nullptr,
                      &iou, workspace, workspace_bytes, stream);
}

int dc_sweep_levels(const float* thresholds, int n_thresholds, float* levels, int32_t* rank, int* n_levels) {
  int rc;
  if ((rc = check_thresholds("dc_sweep_levels", thresholds, n_thresholds))) return rc;
  DC_CHECK_ARG(levels && rank && n_levels, "dc_sweep_levels: null pointer argument");
  std::vector<float> lv;
  std::vector<int> rk;
  threshold_levels(thresholds, n_thresholds, lv, rk);
  std::copy(lv.begin(), lv.end(), levels);
  std::copy(rk.begin(), rk.end(), rank);
  *n_levels = (int)lv.size();
  return DC_OK;
}

int dc_minmax_threshold(float* values, int64_t n, const float* minmax, int use_raw_extrema_for_test, float threshold,
                        int pred_from_threshold, uint8_t* pred, dc_stream_t stream) {
  DC_CHECK_ARG(values && minmax, "dc_minmax_threshold: null pointer argument");
  DC_CHECK_ARG(!pred_from_threshold || pred, "dc_minmax_threshold: pred required");
  if (n <= 0) return DC_OK;
  const int64_t blocks = dc::ceil_div<int64_t>(n, 256);
  const unsigned grid = (unsigned)(blocks < (int64_t)dc::sm_count() * 8 ? blocks : (int64_t)dc::sm_count() * 8);
  minmax_threshold_kernel<void><<<grid, 256, 0, dc::as_stream(stream)>>>(values, n, minmax, use_raw_extrema_for_test, threshold,
                                                                  pred_from_threshold, pred);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

}  // extern "C"
