// Persistent, warp-specialised tcgen05 GEMM used by (3) view scoring and (6) grounding:
//     D[128 x BN] = sum over operand-plane terms  A_t[128 x K] . B_t[BN x K]^T     (fp32 in TMEM)
// A and B are fp16 K-major planes in global memory. fp32 inputs are represented by two planes
// (hi = fp16(x), lo = fp16(x - hi)); the kernel then runs the three products hi.hi + hi.lo +
// lo.hi into the same accumulator, which restores ~22 bits of operand precision while staying on
// the full-rate kind::f16 tensor path. With one fp32 operand only its lo product is added: hi.lo
// (fp32 B) or lo.hi (fp32 A, Params::a_lo_only).
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..9 = epilogue (TMEM -> registers -> global). Three pipelines: smem full/empty ring
// (TMA <-> MMA), TMEM full/empty double buffer (MMA <-> epilogue), persistent tile loop.
//
// Epilogue layout: a warp may only read the TMEM lane quarter (warp % 4), so the eight epilogue
// warps form two groups of four; group h handles the column half [h * BN/2, (h+1) * BN/2) of every
// row (for BN < 64 only group 0 works). A thread owns one row and walks its columns in 32-wide
// chunks with the tcgen05.ld of chunk c+1 in flight while chunk c is processed. Measured on the
// grounding shape (profiles/r01_ncu_gemm_ground_v1_raw.csv): with four single-row warps and a
// blocking load per chunk the tensor pipe was 18 % busy and the kernel spent its time in the
// epilogue's dependent instruction chains (issue slots 18 % used).
#pragma once
#include "common.cuh"
#include "umma.cuh"

namespace dc {
namespace gemm {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // 64 fp16 = 128 bytes = one swizzle row
constexpr int kUmmaK = 16;
constexpr int kThreads = 320;
constexpr int kEpilogueWarps = 8;
constexpr int kEpilogueWarp0 = 2;

struct Tile {
  int a_row;   // first row of the A tile
  int b_row;   // first row of the B tile
  int rows;    // valid rows (<= 128)
  int cols;    // valid columns (<= BN)
};

struct Params {
  const int4* tiles;      // explicit tile list (device) or nullptr for dense row tiling
  const int* tile_count;  // device tile count when `tiles` is given
  int64_t m_total;        // rows of A (dense tiling)
  int n_cols;             // valid columns (dense tiling)
  int k;                  // inner dimension (multiple of 64)
  int n_terms;            // 1: hi.hi   2: + hi.lo   3: + lo.hi
  int reverse;            // dense tiling: walk the row tiles last to first (the rows a preceding pass wrote last are still in L2)
  int a_lo_only;          // A has a lo plane and B has none (fp32 features, fp16 prompts): n_terms == 2 and term 1 is lo.hi
};

// The products whose planes exist: hi.hi, + hi.lo when B has a lo plane, + lo.hi when A has one.
inline void set_terms(Params& p, const void* a_lo, const void* b_lo) {
  p.n_terms = 1 + (a_lo ? 1 : 0) + (b_lo ? 1 : 0);
  p.a_lo_only = (a_lo && !b_lo) ? 1 : 0;
}

template <int BN>
struct Config {
  static constexpr int kStageBytesA = kBlockM * kBlockK * 2;
  static constexpr int kStageBytesB = BN * kBlockK * 2;
  static constexpr int kStageBytes = kStageBytesA + kStageBytesB;
  static constexpr int kBarrierBytes = 512;
  static constexpr int kScratchBytes = kBlockM * 8 * 4;                              // epilogue scratch
  static constexpr int kStages = (BN >= 256) ? 4 : (BN >= 128 ? 6 : 8);
  static constexpr int kTmemCols = (2 * BN < 32) ? 32 : 2 * BN;  // two accumulator buffers
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + kBarrierBytes + kScratchBytes;
  static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "invalid UMMA N");
  static_assert((kTmemCols & (kTmemCols - 1)) == 0 && kTmemCols <= 512, "TMEM columns must be a power of two");
  static_assert(kSmemBytes <= 227 * 1024, "not enough shared memory for the operand ring");
  static_assert((2 * kStages + 4) * 8 + 8 <= kBarrierBytes, "barrier region too small");
};

__device__ __forceinline__ Tile fetch_tile(const Params& p, int t) {
  if (p.tiles) {
    const int4 v = __ldg(p.tiles + t);
    return Tile{v.x, v.y, v.z, v.w};
  }
  if (p.reverse) t = (int)ceil_div<int64_t>(p.m_total, kBlockM) - 1 - t;
  const int64_t r0 = (int64_t)t * kBlockM;
  const int64_t left = p.m_total - r0;
  return Tile{(int)r0, 0, (int)(left < kBlockM ? left : kBlockM), p.n_cols};
}

// Epilogue functor contract (one instance per thread, copied from the kernel argument):
//   void begin(const Tile&, int row_in_tile, float col0_value);        // value of column 0 of this row
//   void row(const Tile&, int row_in_tile, int col0, const float (&v)[32]);   // 32 columns starting at col0
//   void finish(const Tile&, int row_in_tile, int half, int n_halves, float* scratch);
//        // after the last chunk; `scratch` = kBlockM * 8 floats of shared memory for combining the two
//        // column halves of a row (all epilogue threads of the active groups call finish together)
template <int BN, class Epi>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
            const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo, Params p, Epi epi) {
  using Cfg = Config<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = umma::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);  // SWIZZLE_128B tiles need 1024-B alignment
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + Cfg::kStages * Cfg::kStageBytesA;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* full = bars;                      // [kStages]
  uint64_t* empty = bars + Cfg::kStages;      // [kStages]
  uint64_t* tmem_full = bars + 2 * Cfg::kStages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* epi_scratch = reinterpret_cast<float*>(smem + Cfg::kStages * Cfg::kStageBytes + Cfg::kBarrierBytes);  // [kBlockM * 8]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tiles = p.tiles ? __ldg(p.tile_count) : (int)ceil_div<int64_t>(p.m_total, kBlockM);
  const int k_blocks = p.k / kBlockK;

  if (warp == 0 && lane == 0) {
    umma::prefetch_tmap(&tm_a_hi);
    umma::prefetch_tmap(&tm_b_hi);
    if (p.n_terms > 1 && !p.a_lo_only) umma::prefetch_tmap(&tm_b_lo);
    if (p.n_terms > 2 || p.a_lo_only) umma::prefetch_tmap(&tm_a_lo);
    for (int s = 0; s < Cfg::kStages; ++s) {
      umma::mbar_init(full + s, 1);
      umma::mbar_init(empty + s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      umma::mbar_init(tmem_full + a, 1);
      umma::mbar_init(tmem_empty + a, (BN >= 64) ? 8 : 4);  // one arrival per active epilogue warp
    }
    umma::fence_barrier_init();
  }
  if (warp == 1) {
    umma::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    umma::tmem_relinquish();
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const Tile tile = fetch_tile(p, t);
        for (int term = 0; term < p.n_terms; ++term) {
          const bool a_lo = term == 2 || (term == 1 && p.a_lo_only);
          const CUtensorMap* ta = a_lo ? &tm_a_lo : &tm_a_hi;
          const CUtensorMap* tb = (term == 1 && !p.a_lo_only) ? &tm_b_lo : &tm_b_hi;
          for (int kb = 0; kb < k_blocks; ++kb) {
            umma::mbar_wait(empty + stage, phase ^ 1);
            umma::mbar_expect_tx(full + stage, Cfg::kStageBytes);
            umma::tma_load_2d(smem_a + stage * Cfg::kStageBytesA, ta, full + stage, kb * kBlockK, tile.a_row);
            umma::tma_load_2d(smem_b + stage * Cfg::kStageBytesB, tb, full + stage, kb * kBlockK, tile.b_row);
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0) {
      constexpr uint32_t idesc = umma::idesc_f16_f32(kBlockM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        umma::mbar_wait(tmem_empty + acc, acc_phase ^ 1);
        umma::fence_after_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        const int total_kb = k_blocks * p.n_terms;
        for (int kb = 0; kb < total_kb; ++kb) {
          umma::mbar_wait(full + stage, phase);
          umma::fence_after_sync();
          const uint64_t da = umma::smem_desc_k_sw128(umma::smem_u32(smem_a + stage * Cfg::kStageBytesA));
          const uint64_t db = umma::smem_desc_k_sw128(umma::smem_u32(smem_b + stage * Cfg::kStageBytesB));
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k) {
            // advancing 16 fp16 (32 B) inside the swizzle row = +2 in the (addr >> 4) field
            umma::mma_f16_ss(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) ? 1u : 0u);
          }
          umma::mma_commit(empty + stage);  // frees the smem slot when these MMAs retire
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
        umma::mma_commit(tmem_full + acc);  // accumulator complete
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= kEpilogueWarp0) {
    // ===================== epilogue warps =====================
    constexpr int kHalves = (BN >= 64) ? 2 : 1;
    constexpr int kHalfCols = BN / kHalves;
    constexpr int kChunks = kHalfCols / 32;
    const int quarter = warp & 3;  // TMEM lane quarter this warp may access
    const int half = (warp - kEpilogueWarp0) >> 2;
    const int row_in_tile = quarter * 32 + lane;
    if (half < kHalves) {
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const Tile tile = fetch_tile(p, t);
        umma::mbar_wait(tmem_full + acc, acc_phase);
        umma::fence_after_sync();
        const uint32_t tacc = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN);
        const uint32_t taddr = tacc + (uint32_t)(half * kHalfCols);
        const int c_base = half * kHalfCols;
        uint32_t ra[32], rb[32], r0;
        __syncwarp();
        umma::tmem_ld_32x32_x1(tacc, r0);
        umma::tmem_ld_32x32(taddr, ra);
        umma::tmem_ld_wait();
        epi.begin(tile, row_in_tile, __uint_as_float(r0));
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
          uint32_t(&cur)[32] = (c & 1) ? rb : ra;
          uint32_t(&nxt)[32] = (c & 1) ? ra : rb;
          const bool more = (c + 1 < kChunks) && (c_base + (c + 1) * 32 < tile.cols);  // warp-uniform
          if (more) umma::tmem_ld_32x32(taddr + (uint32_t)((c + 1) * 32), nxt);
          if (c_base + c * 32 < tile.cols) {
            float v[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(cur[i]);
            epi.row(tile, row_in_tile, c_base + c * 32, v);
          }
          if (c + 1 < kChunks) umma::tmem_ld_wait();
        }
        umma::fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(tmem_empty + acc);  // TMEM buffer may be overwritten
        epi.finish(tile, row_in_tile, half, kHalves, epi_scratch);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  }

  umma::fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    umma::fence_after_sync();
    umma::tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---------------------------------------------------------------------------- host side
// cuTensorMapEncodeTiled is resolved through the runtime so the library has no link-time
// dependency on libcuda.
int encode_plane_map(CUtensorMap* out, const void* base, int64_t rows, int k, int box_rows);

template <int BN, class Epi>
int launch(const void* a_hi, const void* a_lo, int64_t a_rows, const void* b_hi, const void* b_lo, int64_t b_rows,
           const Params& p, const Epi& epi, int max_tiles, cudaStream_t st) {
  using Cfg = Config<BN>;
  CUtensorMap ta_hi, ta_lo, tb_hi, tb_lo;
  int rc;
  if ((rc = encode_plane_map(&ta_hi, a_hi, a_rows, p.k, kBlockM))) return rc;
  if ((rc = encode_plane_map(&ta_lo, a_lo ? a_lo : a_hi, a_rows, p.k, kBlockM))) return rc;
  if ((rc = encode_plane_map(&tb_hi, b_hi, b_rows, p.k, BN))) return rc;
  if ((rc = encode_plane_map(&tb_lo, b_lo ? b_lo : b_hi, b_rows, p.k, BN))) return rc;
  auto kern = gemm_kernel<BN, Epi>;
  DC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
  int grid = max_tiles < sm_count() ? max_tiles : sm_count();
  if (grid < 1) grid = 1;
  kern<<<grid, kThreads, Cfg::kSmemBytes, st>>>(ta_hi, ta_lo, tb_hi, tb_lo, p, epi);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

}  // namespace gemm
}  // namespace dc
