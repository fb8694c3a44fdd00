// (2) Per-view instance histograms and the row <-> object binding table.
//
// Reference: `np.unique(seg)[1:]` utils/feature_fusion.py:307, `(seg == obj).sum()` :320 and the
// `for i, obj in enumerate(obj_ids_2d)` binding :315,333. The reference runs one numpy sort per
// view on the host (np.unique of 307 200 int64) plus one full-image reduction per (object, view);
// here one streaming pass over all instance maps of the batch produces every count.
//
// Roofline: HBM-bound, reads each pixel once (8 B/pixel for the reference's int64 maps, 1 B for
// uint8 maps). Instance maps are piecewise constant, so a thread run-length-compresses what it
// reads and touches the shared-memory histogram only when the id changes.
#include <stdlib.h>

#include <algorithm>
#include <atomic>

#include "common.cuh"
#include "umma.cuh"  // mbarrier helpers

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

template <typename T> struct VecOf;
template <> struct VecOf<uint8_t> { static constexpr int n = 16; };
template <> struct VecOf<int32_t> { static constexpr int n = 4; };
template <> struct VecOf<long long> { static constexpr int n = 2; };

struct RunAcc {
  long long cur;
  unsigned cnt;
};

// Ids outside [0, nbins) are rare in valid data (a -1 background at most), so they go straight to the view's
// four global words: [0] pixels with id >= nbins, [1] pixels with id < 0, [2] smallest negative id (init 0),
// [3] largest negative id stored as id + 2^63 (init 0) - enough to tell whether the negative ids are ONE distinct
// value, which np.unique(seg)[1:] simply drops (utils/feature_fusion.py:307).
__device__ __forceinline__ void flush_run(RunAcc& r, unsigned* warp_hist, unsigned long long* outside, int nbins) {
  if (r.cnt) {
    if (r.cur >= 0 && r.cur < nbins) {
      atomicAdd(warp_hist + r.cur, r.cnt);
    } else if (r.cur >= 0) {
      atomicAdd(outside, (unsigned long long)r.cnt);
    } else {
      atomicAdd(outside + 1, (unsigned long long)r.cnt);
      atomicMin(reinterpret_cast<long long*>(outside + 2), r.cur);
      atomicMax(outside + 3, (unsigned long long)r.cur ^ 0x8000000000000000ull);
    }
  }
}

__device__ __forceinline__ void push(RunAcc& r, long long id, unsigned* warp_hist, unsigned long long* outside, int nbins) {
  if (id == r.cur) {
    ++r.cnt;
  } else {
    flush_run(r, warp_hist, outside, nbins);
    r.cur = id;
    r.cnt = 1;
  }
}

template <typename T>
__device__ __forceinline__ void consume_vector(const int4& raw, RunAcc& run, unsigned* hist, unsigned long long* outside, int nbins) {
  constexpr int VEC = VecOf<T>::n;
  const T* e = reinterpret_cast<const T*>(&raw);
  if (sizeof(T) < 8) {
    // narrow ids: a 16-byte vector that repeats one id (the usual case inside an object or on the table)
    // extends or starts a run with a handful of word compares instead of 16 / 4 element pushes
    const unsigned first = (unsigned)raw.x;
    const unsigned pat = sizeof(T) == 1 ? (first & 0xffu) * 0x01010101u : first;
    if (((unsigned)raw.x == pat) & ((unsigned)raw.y == pat) & ((unsigned)raw.z == pat) & ((unsigned)raw.w == pat)) {
      const long long id = (long long)e[0];
      if (id == run.cur) {
        run.cnt += VEC;
      } else {
        flush_run(run, hist, outside, nbins);
        run.cur = id;
        run.cnt = VEC;
      }
      return;
    }
  }
#pragma unroll
  for (int k = 0; k < VEC; ++k) push(run, (long long)e[k], hist, outside, nbins);
}

// One shared-memory histogram per CTA (run-length compression keeps the atomics on it rare), four 128-bit
// loads in flight per thread.
template <typename T>
__global__ void __launch_bounds__(kThreads) seg_histogram_kernel(const T* __restrict__ seg, int64_t pixels_per_view,
                                                                 int nbins, uint32_t* __restrict__ counts,
                                                                 unsigned long long* __restrict__ outside_out) {
  extern __shared__ unsigned s_hist[];  // [nbins]
  const int view = blockIdx.y;
  for (int i = threadIdx.x; i < nbins; i += kThreads) s_hist[i] = 0;
  __syncthreads();
  const T* base = seg + (int64_t)view * pixels_per_view;
  constexpr int VEC = VecOf<T>::n;
  // a view may start anywhere: scalar head up to the next 16-byte boundary, 128-bit body, scalar tail
  int64_t head = (int64_t)(((16 - ((uintptr_t)base & 15)) & 15) / sizeof(T));
  if (head > pixels_per_view) head = pixels_per_view;
  const int64_t n_vec = (pixels_per_view - head) / VEC;
  const int4* body = reinterpret_cast<const int4*>(base + head);
  RunAcc run{-1, 0};
  unsigned long long* outside = outside_out + 4 * (int64_t)view;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  for (; i + 3 * stride < n_vec; i += 4 * stride) {
    const int4 r0 = dc::ld_stream(body + i), r1 = dc::ld_stream(body + i + stride), r2 = dc::ld_stream(body + i + 2 * stride),
               r3 = dc::ld_stream(body + i + 3 * stride);
    consume_vector<T>(r0, run, s_hist, outside, nbins);
    consume_vector<T>(r1, run, s_hist, outside, nbins);
    consume_vector<T>(r2, run, s_hist, outside, nbins);
    consume_vector<T>(r3, run, s_hist, outside, nbins);
  }
  for (; i < n_vec; i += stride) consume_vector<T>(dc::ld_stream(body + i), run, s_hist, outside, nbins);
  if (blockIdx.x == 0) {
    for (int64_t j = threadIdx.x; j < head; j += kThreads) push(run, (long long)base[j], s_hist, outside, nbins);
    for (int64_t j = head + n_vec * VEC + threadIdx.x; j < pixels_per_view; j += kThreads)
      push(run, (long long)base[j], s_hist, outside, nbins);
  }
  flush_run(run, s_hist, outside, nbins);
  __syncthreads();
  for (int b = threadIdx.x; b < nbins; b += kThreads) {
    const unsigned t = s_hist[b];
    if (t) atomicAdd(counts + (int64_t)view * nbins + b, t);
  }
}

// ---------------------------------------------------------------------------------------------
// Ring variant for the reference's int64 maps (the dominant kernel of the object-level step).
//
// The histogram pass is HBM-bound and needs few issue slots; the visibility filter that shares the step
// is issue-bound and needs little HBM. The engine therefore runs the two on different streams, and this
// kernel is shaped to live BESIDE the filter on every SM instead of alternating with it:
//   * persistent, one CTA per SM, 12 warps x 64 registers and ~50 KB of shared memory: two filter CTAs (2 x 256 x 80
//     registers, 2 x 34 KB) fit next to it, with ~90 KB of the SM left to the L1 the filter's depth gathers live on;
//   * the bytes in flight that a streaming kernel needs (~50 KB per SM at 7 TB/s) come from shared-memory
//     rings filled by 1-D bulk copies (cp.async.bulk -> mbarrier complete_tx, L2 evict-first), not from the
//     registers of hundreds of resident threads;
//   * every warp runs its own ring (2 KB units, `depth` slots, its lane 0 is the producer), so a warp that
//     meets an object boundary (the slow, per-pixel path) does not hold up the other warps;
//   * a CTA takes whole views by atomic ticket (one view ahead, so the producers never drain at a view boundary),
//     deals the view's units to its warps round-robin and flushes its shared-memory histogram at the end of the view.
// Counting is the same run-length scheme as above. A lane owns 64 contiguous bytes = eight neighbouring pixels:
// "all eight equal" is an XOR/OR tree on the ALU, then one 64-bit compare against the current run.
constexpr int kUnit = 2048;  // bytes per warp unit: 32 lanes x 64 B
// 12 warps x 2 slots x 2 KB = 48 KB of ring, beside two filter CTAs in the shared carve-out (common.cuh).
// Alone: 6.7 TB/s (3 slots: 7.2, 8 warps: 5.8); the two-stream step: 2.75-2.78 ms with 2 slots, 2.80-2.85 with 3
// (B200, profiles/r02_seg_ring.md).
constexpr int kRingWarps = 12;
constexpr int kRingMinCtas = 3;
constexpr int kRingThreads = kRingWarps * 32;
constexpr int kRingDepth = 2;

__device__ __forceinline__ void bulk_load_evict_first(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar,
                                                      uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(dc::umma::smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(dc::umma::smem_u32(bar)), "l"(policy)
      : "memory");
}

// Waiting for a bulk copy with a suspend-time hint: the warp sleeps in the barrier unit instead of re-issuing try_wait.
// (This kernel is always waiting for HBM; with the plain spin loop 2/3 of its 1.08 G warp instructions per launch were
// try_wait re-issues - issue slots taken from the issue-bound filter that shares the SM; ncu: profiles/r02_seg_ring.md.)
__device__ __forceinline__ void mbar_wait_suspended(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(dc::umma::smem_u32(bar)), "r"(parity), "r"(20000u)
        : "memory");
  } while (!ok);
}

// acc | (x ^ ref) as ONE three-input logic instruction (written as C the compiler turns the equality test of eight
// 64-bit ids into a serial chain of 14 predicate-setting compares: ~180 cycles of dependent latency per unit)
__device__ __forceinline__ unsigned or_xor(unsigned acc, unsigned x, unsigned ref) {
  unsigned d;
  asm("lop3.b32 %0, %1, %2, %3, 0xBE;" : "=r"(d) : "r"(x), "r"(ref), "r"(acc));  // (a ^ b) | c
  return d;
}

// Views are handed out dynamically (one atomic ticket per view): CTAs that share their SM with more filter CTAs, or that
// were placed late because their SM was full at launch time, simply take fewer views. (With a static split of the
// batch the step time jumped between 2.8 and 4.0 ms depending on where the 148 CTAs had landed.)
constexpr int kTicketSlots = 64;
__device__ unsigned g_ring_tickets[kTicketSlots];

__global__ void __launch_bounds__(kRingThreads, kRingMinCtas)
seg_histogram_ring_kernel(const long long* __restrict__ seg, int64_t bytes_per_view, int units_per_view, int total_views,
                          int nbins, int depth, unsigned* __restrict__ ticket, uint32_t* __restrict__ counts,
                          unsigned long long* __restrict__ outside_out) {
  using namespace dc::umma;
  extern __shared__ __align__(128) unsigned char s_ring[];  // [warps][depth][2 KB], histogram, full[warps][depth], views[2]
  const size_t ring_bytes = (size_t)kRingWarps * depth * kUnit;
  unsigned* s_hist = reinterpret_cast<unsigned*>(s_ring + ring_bytes);
  uint64_t* full_all = reinterpret_cast<uint64_t*>(s_ring + ring_bytes + ((nbins * 4 + 15) & ~15));
  volatile int* s_view = reinterpret_cast<volatile int*>(full_all + kRingWarps * depth);  // the CTA's n-th view: s_view[n & 1]
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kRingWarps * depth; ++i) mbar_init(full_all + i, 1);
    fence_barrier_init();
    s_view[0] = (int)atomicAdd(ticket, 1u);
    s_view[1] = (int)atomicAdd(ticket, 1u);
  }
  for (int i = threadIdx.x; i < nbins; i += kRingThreads) s_hist[i] = 0;
  __syncthreads();

  const int last_bytes = (int)(bytes_per_view - (int64_t)(units_per_view - 1) * kUnit);  // of a view's last unit
  unsigned char* const my_ring = s_ring + (size_t)w * depth * kUnit;
  uint64_t* const full = full_all + w * depth;
  const char* const base = reinterpret_cast<const char*>(seg);
  // units w, w + warps, ... of every view are this warp's (the launcher guarantees units_per_view >= 4 * warps * depth,
  // so a warp's producer lane never runs two views ahead of its consumer)
  const int n_it = (units_per_view - w + kRingWarps - 1) / kRingWarps;
  const bool ends_partial = last_bytes != kUnit && w + (n_it - 1) * kRingWarps == units_per_view - 1;

  // ---- producer state (lane 0): the warp's next unit to load is unit pj of the CTA's pn-th view, at psrc, into slot pslot
  uint64_t policy = 0;
  int pn = 0, pj = w, pslot = 0;
  bool p_has = false;
  const char* psrc = nullptr;
  auto open_view = [&]() {
    const int pv = s_view[pn & 1];
    p_has = pv < total_views;
    psrc = base + (int64_t)pv * bytes_per_view + (int64_t)w * kUnit;
    pj = w;
  };
  auto issue = [&]() {
    const uint32_t bytes = (uint32_t)(pj == units_per_view - 1 ? last_bytes : kUnit);
    mbar_expect_tx(full + pslot, bytes);
    bulk_load_evict_first(my_ring + pslot * kUnit, psrc, bytes, full + pslot, policy);
    pslot = (pslot == depth - 1) ? 0 : pslot + 1;
    pj += kRingWarps;
    psrc += kRingWarps * kUnit;
    if (pj >= units_per_view) {  // on to the CTA's next view (claimed one view ahead, see the flush below)
      ++pn;
      open_view();
    }
  };
  if (lane == 0) {
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    open_view();
    for (int d = 0; d < depth && p_has; ++d) issue();
  }

  // ---- consumer: a lane owns 64 contiguous bytes of every unit; its four 16-byte reads are rotated by lane so that
  // the eight lanes of a shared-memory phase fall into eight different 16-byte bank groups
  int off[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    off[k] = 16 * (4 * lane + ((k + (lane >> 1)) & 3));
    asm volatile("" : "+r"(off[k]));  // keep the four offsets in registers (otherwise recomputed from the lane id per unit)
  }
  RunAcc run{-1, 0};
  int slot = 0;
  uint32_t parity = 0;
  const unsigned char* slot_ptr = my_ring;

  for (int n = 0;; ++n) {
    const int v = s_view[n & 1];
    if (v >= total_views) break;
    unsigned long long* outside = outside_out + 4 * (int64_t)v;
    for (int it = 0; it < n_it; ++it) {
      mbar_wait_suspended(full + slot, parity);
      if (!(ends_partial && it == n_it - 1)) {
        int4 r[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) r[k] = *reinterpret_cast<const int4*>(slot_ptr + off[k]);
        const unsigned lo0 = (unsigned)r[0].x, hi0 = (unsigned)r[0].y;
        unsigned dl = (unsigned)r[0].z ^ lo0, dh = (unsigned)r[0].w ^ hi0;
#pragma unroll
        for (int k = 1; k < 4; ++k) {
          dl = or_xor(or_xor(dl, (unsigned)r[k].x, lo0), (unsigned)r[k].z, lo0);
          dh = or_xor(or_xor(dh, (unsigned)r[k].y, hi0), (unsigned)r[k].w, hi0);
        }
        if ((dl | dh) == 0) {  // eight equal ids
          const long long id = (long long)(((unsigned long long)hi0 << 32) | lo0);
          if (id != run.cur) {
            flush_run(run, s_hist, outside, nbins);
            run.cur = id;
            run.cnt = 0;
          }
          run.cnt += 8;
        } else {
          // an object boundary inside the lane's eight pixels. The other lanes of the warp wait for this path, so it
          // is kept short and free of dependent chains: close the run, then one shared-memory atomic per pixel.
          flush_run(run, s_hist, outside, nbins);
          run.cur = -1;
          run.cnt = 0;
          const unsigned hi_any = (unsigned)r[0].y | (unsigned)r[0].w | (unsigned)r[1].y | (unsigned)r[1].w | (unsigned)r[2].y |
                                  (unsigned)r[2].w | (unsigned)r[3].y | (unsigned)r[3].w;
          const unsigned lo_max = max(max(max((unsigned)r[0].x, (unsigned)r[0].z), max((unsigned)r[1].x, (unsigned)r[1].z)),
                                      max(max((unsigned)r[2].x, (unsigned)r[2].z), max((unsigned)r[3].x, (unsigned)r[3].z)));
          if (hi_any == 0 && lo_max < (unsigned)nbins) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              atomicAdd(s_hist + (unsigned)r[k].x, 1u);
              atomicAdd(s_hist + (unsigned)r[k].z, 1u);
            }
          } else {  // ids outside the histogram (negative background, id >= nbins): the general path
#pragma unroll
            for (int k = 0; k < 4; ++k) consume_vector<long long>(r[k], run, s_hist, outside, nbins);
          }
        }
      } else {  // partial last unit of the view
        const int n_vec = last_bytes >> 4;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if ((off[k] >> 4) < n_vec)
            consume_vector<long long>(*reinterpret_cast<const int4*>(slot_ptr + off[k]), run, s_hist, outside, nbins);
      }
      // every lane has used its registers, so the shared-memory reads of the slot are complete: refill it
      __syncwarp();
      if (lane == 0 && p_has) issue();
      slot_ptr += kUnit;
      if (++slot == depth) {
        slot = 0;
        slot_ptr = my_ring;
        parity ^= 1u;
      }
    }
    // end of the view: all warps flush into the view's global row, and the CTA claims the view after the next one
    // (slot n & 1 of s_view is free: every warp has read it, and the producer lanes are already in view n + 1)
    flush_run(run, s_hist, outside, nbins);
    run.cur = -1;
    run.cnt = 0;
    __syncthreads();
    for (int bin = threadIdx.x; bin < nbins; bin += kRingThreads) {
      const unsigned t = s_hist[bin];
      if (t) {
        atomicAdd(counts + (int64_t)v * nbins + bin, t);
        s_hist[bin] = 0;
      }
    }
    if (threadIdx.x == 0) s_view[n & 1] = (int)atomicAdd(ticket, 1u);
    __syncthreads();
  }
}

inline bool ring_fits(int64_t bytes_per_view) {
  return dc::ceil_div<int64_t>(bytes_per_view, kUnit) >= (int64_t)4 * kRingWarps * kRingDepth;
}

int launch_ring(const void* seg, int64_t bytes_per_view, int64_t total_views, int nbins, uint32_t* counts, uint64_t* outside,
                cudaStream_t st) {
  const int upv = (int)dc::ceil_div<int64_t>(bytes_per_view, kUnit);
  const size_t smem = (size_t)kRingWarps * kRingDepth * kUnit + ((sizeof(unsigned) * nbins + 15) & ~(size_t)15) +
                      (size_t)kRingWarps * kRingDepth * sizeof(uint64_t) + 16;
  // a zeroed ticket counter per launch; launches in flight at the same time use different slots
  static std::atomic<unsigned> next_slot{0};
  static unsigned* tickets_of_device[dc::FuncAttrCache::kMaxDevices] = {nullptr};
  int dev = 0;
  DC_CUDA(cudaGetDevice(&dev));
  unsigned* tickets = (dev >= 0 && dev < dc::FuncAttrCache::kMaxDevices) ? tickets_of_device[dev] : nullptr;
  if (!tickets) {
    DC_CUDA(cudaGetSymbolAddress(reinterpret_cast<void**>(&tickets), g_ring_tickets));
    if (dev >= 0 && dev < dc::FuncAttrCache::kMaxDevices) tickets_of_device[dev] = tickets;
  }
  unsigned* ticket = tickets + next_slot.fetch_add(1) % kTicketSlots;
  DC_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned), st));
  static dc::FuncAttrCache smem_attr, carve_attr;
  DC_CUDA(smem_attr.set(seg_histogram_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // the SM's shared-memory carve-out is fixed while CTAs are resident: ask for one under which the filter's CTAs fit beside
  const int carve = dc::stream_overlap() ? dc::kOverlapCarveoutPct : cudaSharedmemCarveoutDefault;
  DC_CUDA(carve_attr.set(seg_histogram_ring_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
  const int grid = (int)std::min<int64_t>(dc::sm_count(), total_views);
  seg_histogram_ring_kernel<<<grid, kRingThreads, smem, st>>>((const long long*)seg, bytes_per_view, upv, (int)total_views, nbins,
                                                             kRingDepth, ticket, counts, (unsigned long long*)outside);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

// One warp per view: ids present (ascending) minus the smallest -> rows 0,1,2,... A lane looks at one bin of
// each 32-bin chunk and ballots give the ascending rank of every present id. Present ids are ascending, so every
// id below n_q is preceded only by ids below n_q: its row is simply its rank minus one (the dropped smallest id).
// (The one-thread-per-view version walked the 256 bins with dependent loads: 36 us for 4672 views.)
__global__ void __launch_bounds__(128) view_table_kernel(const uint32_t* __restrict__ counts, const unsigned long long* __restrict__ outside,
                                                         const int64_t* __restrict__ feat_off, const int32_t* __restrict__ view_scene,
                                                         const int64_t* __restrict__ view_off, const int64_t* __restrict__ query_off,
                                                         const int64_t* __restrict__ wobj_off, int64_t total_views, int nbins,
                                                         int32_t* __restrict__ row_object, int32_t* __restrict__ object_row,
                                                         int32_t* __restrict__ view_status) {
  const int64_t g = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (g >= total_views) return;
  const int lane = threadIdx.x & 31;
  const int s = view_scene[g];
  const int n_q = (int)(query_off[s + 1] - query_off[s]);
  const int n_v = (int)(view_off[s + 1] - view_off[s]);
  const int v_local = (int)(g - view_off[s]);
  const int64_t r0 = feat_off[g];
  const int64_t n_rows = feat_off[g + 1] - r0;
  // Ids outside the histogram: an id >= nbins (>= Q) is indexed by the reference's loop and raises IndexError
  // there (weight_obj[obj, v], :317). Negative ids: ONE distinct negative value is the smallest id of the view and
  // is dropped by np.unique(seg)[1:] (e.g. a -1 background) - then no id in [0, nbins) is dropped; two or more
  // distinct negative values would index weight_obj with a negative row (torch wraps it): reported as IndexError.
  const unsigned long long* o = outside + 4 * g;
  int status = o[0] ? 1 : 0;
  const bool has_negative = o[1] != 0;
  if (has_negative && (long long)o[2] != (long long)(o[3] ^ 0x8000000000000000ull)) status |= 1;
  const uint32_t* c = counts + g * nbins;
  int seen = has_negative ? 1 : 0;   // present ids met so far, the dropped smallest one included
  int bound = 0;  // rows bound by this lane
  for (int id0 = 0; id0 < nbins; id0 += 32) {
    const int id = id0 + lane;
    const bool present = id < nbins && c[id] != 0;
    const unsigned mask = __ballot_sync(0xffffffffu, present);
    if (present) {
      const int64_t row = (int64_t)seen + __popc(mask & ((1u << lane) - 1u)) - 1;
      if (row >= 0) {  // row < 0: the smallest present id, dropped like np.unique(seg)[1:]
        if (id >= n_q) status |= 1;
        else if (row >= n_rows) status |= 2;
        else {
          row_object[r0 + row] = id;
          object_row[wobj_off[s] + (int64_t)id * n_v + v_local] = (int32_t)(r0 + row);
          ++bound;
        }
      }
    }
    seen += __popc(mask);
  }
  status = __reduce_or_sync(0xffffffffu, status);
  const int next = __reduce_add_sync(0xffffffffu, bound);
  for (int64_t r = next + lane; r < n_rows; r += 32) row_object[r0 + r] = -1;  // feature rows no id is bound to
  if (lane == 0) view_status[g] = status;
}

}  // namespace

extern "C" int dc_seg_histogram(const void* seg, int seg_dtype, int64_t total_views, int64_t pixels_per_view,
                                int nbins, uint32_t* counts, uint64_t* outside, dc_stream_t stream) {
  DC_CHECK_ARG(seg && counts && outside, "dc_seg_histogram: null pointer argument");
  DC_CHECK_ARG(nbins > 0 && nbins <= 8192, "dc_seg_histogram: nbins must be in [1,8192]");
  DC_CHECK_ARG(seg_dtype == DC_U8 || seg_dtype == DC_I32 || seg_dtype == DC_I64,
               "dc_seg_histogram: seg dtype must be u8, i32 or i64");
  if (total_views <= 0 || pixels_per_view <= 0) return DC_OK;
  DC_CHECK_ARG(total_views <= 65535, "dc_seg_histogram: at most 65535 views per call");
  const int esize = seg_dtype == DC_U8 ? 1 : seg_dtype == DC_I32 ? 4 : 8;
  DC_CHECK_ARG((uintptr_t)seg % esize == 0, "dc_seg_histogram: seg is not aligned to its element size");
  cudaStream_t st = dc::as_stream(stream);
  DC_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * (size_t)total_views * nbins, st));
  DC_CUDA(cudaMemsetAsync(outside, 0, sizeof(uint64_t) * 4 * (size_t)total_views, st));
  // int64 maps with 16-byte aligned views, enough of them to give every SM a few MB: the ring kernel (bulk copies)
  const int64_t bytes_per_view = pixels_per_view * esize;
  // DC_SEG_MODE=ring forces the ring kernel wherever its preconditions hold, so that tests reach it at small sizes. It is
  // the library's only environment switch: every other launch decision follows from the arguments and the overlap mode.
  const char* mode = getenv("DC_SEG_MODE");
  const bool forced = mode && strcmp(mode, "ring") == 0;
  const bool want_ring = forced || (dc::stream_overlap() && total_views * bytes_per_view >= (int64_t)dc::sm_count() * (4 << 20));
  if (want_ring && seg_dtype == DC_I64 && (uintptr_t)seg % 16 == 0 && bytes_per_view % 16 == 0 && ring_fits(bytes_per_view))
    return launch_ring(seg, bytes_per_view, total_views, nbins, counts, outside, st);
  // CTAs of ~512 KB: enough of them per view to fill the machine a few times over when there are few views, and small
  // enough that the last wave does not leave SMs idle when there are many (4672 views of 2.4 MB: one CTA per view
  // ran at 6.9 TB/s, four at 7.3 TB/s)
  const int64_t vec_per_view = pixels_per_view * esize / 16;
  int64_t want = dc::ceil_div<int64_t>((int64_t)dc::sm_count() * 8, total_views);
  want = max(want, pixels_per_view * esize / (512 << 10));
  int64_t cap = dc::ceil_div<int64_t>(vec_per_view, (int64_t)kThreads * 4);
  unsigned gx = (unsigned)max((int64_t)1, min(want, max((int64_t)1, cap)));
  dim3 grid(gx, (unsigned)total_views);
  const size_t smem = sizeof(unsigned) * nbins;
  {  // same carve-out as the visibility filter these CTAs may share their SM with (two-stream step)
    const int carve = dc::stream_overlap() ? dc::kOverlapCarveoutPct : cudaSharedmemCarveoutDefault;
    static dc::FuncAttrCache c8, c32, c64;
    if (seg_dtype == DC_U8) DC_CUDA(c8.set(seg_histogram_kernel<uint8_t>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    else if (seg_dtype == DC_I32) DC_CUDA(c32.set(seg_histogram_kernel<int32_t>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    else DC_CUDA(c64.set(seg_histogram_kernel<long long>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
  }
  if (seg_dtype == DC_U8)
    seg_histogram_kernel<uint8_t><<<grid, kThreads, smem, st>>>((const uint8_t*)seg, pixels_per_view, nbins, counts, (unsigned long long*)outside);
  else if (seg_dtype == DC_I32)
    seg_histogram_kernel<int32_t><<<grid, kThreads, smem, st>>>((const int32_t*)seg, pixels_per_view, nbins, counts, (unsigned long long*)outside);
  else
    seg_histogram_kernel<long long><<<grid, kThreads, smem, st>>>((const long long*)seg, pixels_per_view, nbins, counts, (unsigned long long*)outside);
  DC_LAUNCH_CHECK();
  return DC_OK;
}

extern "C" int dc_view_table(const uint32_t* counts, const uint64_t* outside, const int64_t* feat_off,
                             const int32_t* view_scene, const int64_t* view_off, const int64_t* query_off,
                             const int64_t* wobj_off, int64_t total_views, int64_t total_rows, int64_t total_wobj,
                             int nbins, int32_t* row_object, int32_t* object_row, int32_t* view_status,
                             dc_stream_t stream) {
  DC_CHECK_ARG(counts && outside && feat_off && view_scene && view_off && query_off && wobj_off && row_object &&
                   object_row && view_status,
               "dc_view_table: null pointer argument");
  if (total_views <= 0) return DC_OK;
  cudaStream_t st = dc::as_stream(stream);
  if (total_wobj > 0) DC_CUDA(cudaMemsetAsync(object_row, 0xFF, sizeof(int32_t) * (size_t)total_wobj, st));
  (void)total_rows;
  const int threads = 128;  // four views per CTA, one warp each
  view_table_kernel<<<(unsigned)dc::ceil_div<int64_t>(total_views, threads / 32), threads, 0, st>>>(
      counts, (const unsigned long long*)outside, feat_off, view_scene, view_off, query_off, wobj_off, total_views, nbins, row_object,
      object_row, view_status);
  DC_LAUNCH_CHECK();
  return DC_OK;
}
