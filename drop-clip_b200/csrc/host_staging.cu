// Host-side staging helpers of the drop-in boundary (no device code).
//
// The reference hands MultiviewFeatureFusion.fuse() ~275 MB of pageable numpy arrays per MV-TOD
// scene (73 depth maps fp32, 73 instance maps int64, tools/preprocess_data.py:177-268). At that
// size the end-to-end rate of the GPU path is set by how fast the host can move those bytes into
// pinned memory, not by the kernels (0.1 ms/scene). Two things help:
//   * a list of equally sized arrays is copied into one pinned buffer by several threads in ONE
//     call (73 separate 1.2 MB tensor copies cost more in per-call overhead than in bandwidth);
//   * int64 instance maps are narrowed to uint8 on the fly (8x fewer bytes over PCIe and 8x less
//     HBM traffic in seg_histogram). Instance ids outside [0, 255] cannot be represented; the
//     helper reports them and the caller uploads the int64 maps unchanged, so the error behaviour
//     of the reference (IndexError for ids >= Q, quirk q7) is kept.
// These run on the caller's cores under ctypes (GIL released). They move and narrow bytes; nothing
// of the fusion arithmetic is evaluated here.
#include <emmintrin.h>  // SSE2 streaming stores (baseline x86-64)
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>

#include "common.cuh"

namespace {

// Copy into pinned staging memory with non-temporal stores: the destination is read next by the DMA engine,
// not by a core, so write-allocating it into the caches only adds a read-for-ownership of every line
// (a third of the DRAM traffic of a plain memcpy at these sizes).
inline void stream_copy(void* dst, const void* src, size_t len) {
  char* d = static_cast<char*>(dst);
  const char* s = static_cast<const char*>(src);
  const size_t head = ((16 - (reinterpret_cast<uintptr_t>(d) & 15)) & 15);
  if (len < 256 || head > len) {
    memcpy(d, s, len);
    return;
  }
  memcpy(d, s, head);
  d += head; s += head; len -= head;
  size_t n64 = len / 64;
  for (size_t i = 0; i < n64; ++i) {
    const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(s));
    const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(s + 16));
    const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(s + 32));
    const __m128i e = _mm_loadu_si128(reinterpret_cast<const __m128i*>(s + 48));
    _mm_stream_si128(reinterpret_cast<__m128i*>(d), a);
    _mm_stream_si128(reinterpret_cast<__m128i*>(d + 16), b);
    _mm_stream_si128(reinterpret_cast<__m128i*>(d + 32), c);
    _mm_stream_si128(reinterpret_cast<__m128i*>(d + 48), e);
    s += 64; d += 64;
  }
  memcpy(d, s, len - n64 * 64);
  _mm_sfence();
}

// A persistent worker pool: the helpers are called several times per scene, and spawning 16 threads per call
// costs 0.3-0.6 ms - as much as the copy itself at these sizes. Workers sleep on a condition variable between
// jobs; one job runs at a time (concurrent callers take turns); the caller works too. The pool is created on
// first use, grows to the largest thread count asked for, is never destroyed (threads are detached), and is
// rebuilt in a forked child (the parent's threads do not exist there).
class WorkerPool {
 public:
  static WorkerPool& instance() {
    static WorkerPool* pool = new WorkerPool();  // leaked on purpose: no destructor races at interpreter exit
    return *pool;
  }

  template <typename F>
  void run(int64_t n_items, int n_threads, F&& fn) {
    if (n_threads > n_items) n_threads = (int)n_items;
    if (n_threads <= 1) {
      for (int64_t i = 0; i < n_items; ++i) fn(i);
      return;
    }
    std::lock_guard<std::mutex> job(job_mutex_);
    std::function<void(int64_t)> f = fn;
    {
      std::unique_lock<std::mutex> lk(m_);
      if (owner_pid_ != getpid()) {  // forked: forget the parent's workers
        n_workers_ = 0;
        owner_pid_ = getpid();
      }
      while (n_workers_ < n_threads - 1) {
        const int id = n_workers_++;
        std::thread([this, id] { worker(id); }).detach();
      }
      fn_ = &f;
      n_items_ = n_items;
      next_.store(0, std::memory_order_relaxed);
      participants_ = n_threads - 1;
      pending_ = n_threads - 1;
      ++epoch_;
    }
    cv_start_.notify_all();
    drain(f, n_items);
    std::unique_lock<std::mutex> lk(m_);
    cv_done_.wait(lk, [this] { return pending_ == 0; });
    fn_ = nullptr;
  }

 private:
  void drain(const std::function<void(int64_t)>& f, int64_t n_items) {
    for (;;) {
      const int64_t i = next_.fetch_add(1, std::memory_order_relaxed);
      if (i >= n_items) return;
      f(i);
    }
  }

  void worker(int id) {
    uint64_t seen = 0;
    const pid_t pid = getpid();
    for (;;) {
      const std::function<void(int64_t)>* f;
      int64_t n;
      {
        std::unique_lock<std::mutex> lk(m_);
        cv_start_.wait(lk, [&] { return epoch_ != seen; });
        seen = epoch_;
        if (owner_pid_ != pid) return;
        if (id >= participants_) continue;
        f = fn_;
        n = n_items_;
      }
      drain(*f, n);
      std::unique_lock<std::mutex> lk(m_);
      if (--pending_ == 0) cv_done_.notify_all();
    }
  }

  std::mutex job_mutex_, m_;
  std::condition_variable cv_start_, cv_done_;
  const std::function<void(int64_t)>* fn_ = nullptr;
  std::atomic<int64_t> next_{0};
  int64_t n_items_ = 0;
  int n_workers_ = 0, participants_ = 0, pending_ = 0;
  uint64_t epoch_ = 0;
  pid_t owner_pid_ = getpid();
};

template <typename F>
void parallel_items(int64_t n_items, int n_threads, F&& fn) {
  WorkerPool::instance().run(n_items, n_threads, fn);
}

}  // namespace

extern "C" {

int dc_host_gather_copy(const void* const* srcs, int64_t n_items, int64_t item_bytes, void* dst, int n_threads) {
  DC_CHECK_ARG(srcs && dst && n_items >= 0 && item_bytes >= 0, "dc_host_gather_copy: bad argument");
  // split every item in slices so that a handful of large items still spreads over all threads
  const int64_t slice = 256 << 10;
  const int64_t per_item = item_bytes > 0 ? (item_bytes + slice - 1) / slice : 0;
  parallel_items(n_items * per_item, n_threads, [&](int64_t t) {
    const int64_t i = t / per_item, s = (t - i * per_item) * slice;
    const int64_t len = std::min(slice, item_bytes - s);
    stream_copy(static_cast<char*>(dst) + i * item_bytes + s, static_cast<const char*>(srcs[i]) + s, (size_t)len);
  });
  return DC_OK;
}

int dc_host_gather_narrow_i64_u8(const int64_t* const* srcs, int64_t n_items, int64_t item_elems, uint8_t* dst, int n_threads,
                                 int* out_of_range) {
  DC_CHECK_ARG(srcs && dst && out_of_range && n_items >= 0 && item_elems >= 0, "dc_host_gather_narrow_i64_u8: bad argument");
  const int64_t slice = 64 << 10;  // elements
  const int64_t per_item = item_elems > 0 ? (item_elems + slice - 1) / slice : 0;
  std::atomic<uint64_t> seen(0);
  parallel_items(n_items * per_item, n_threads, [&](int64_t t) {
    const int64_t i = t / per_item, s = (t - i * per_item) * slice;
    const int64_t len = std::min(slice, item_elems - s);
    const int64_t* __restrict__ a = srcs[i] + s;
    uint8_t* __restrict__ o = dst + i * item_elems + s;
    uint64_t acc = 0;
    for (int64_t j = 0; j < len; ++j) {
      const uint64_t v = (uint64_t)a[j];
      acc |= v;           // any bit above the low byte (negative values included) marks the map as not narrowable
      o[j] = (uint8_t)v;
    }
    if (acc & ~(uint64_t)0xff) seen.fetch_or(acc, std::memory_order_relaxed);
  });
  *out_of_range = (seen.load() & ~(uint64_t)0xff) ? 1 : 0;
  return DC_OK;
}

int dc_host_masks_to_seg(const uint8_t* const* masks, const int64_t* ids, const int64_t* mask_off, int n_views,
                         const int64_t* view_pixels, const int64_t* pix_off, int out_dtype, void* dst, int n_threads,
                         int* out_of_range) {
  DC_CHECK_ARG(masks && ids && mask_off && view_pixels && pix_off && dst && out_of_range && n_views >= 0,
               "dc_host_masks_to_seg: bad argument");
  DC_CHECK_ARG(out_dtype == DC_U8 || out_dtype == DC_I64, "dc_host_masks_to_seg: out_dtype must be DC_U8 or DC_I64");
  for (int v = 0; v < n_views; ++v)
    DC_CHECK_ARG(mask_off[v + 1] > mask_off[v] && view_pixels[v] >= 0, "dc_host_masks_to_seg: view %d has no mask", v);
  // work items: slices of a view's pixels, small enough that the running maxima stay in L1 across the K masks
  const int64_t slice = 4096;
  int64_t n_items = 0;
  for (int v = 0; v < n_views; ++v) n_items += (view_pixels[v] + slice - 1) / slice;
  std::atomic<int> bad(0);
  int64_t* item_view = static_cast<int64_t*>(malloc(sizeof(int64_t) * (size_t)(n_views + 1)));  // first item of each view
  if (!item_view) return ::dc::fail(DC_ERR_INVALID, "dc_host_masks_to_seg: out of host memory");
  item_view[0] = 0;
  for (int v = 0; v < n_views; ++v) item_view[v + 1] = item_view[v] + (view_pixels[v] + slice - 1) / slice;
  parallel_items(n_items, n_threads, [&](int64_t t) {
    const int v = (int)(std::upper_bound(item_view, item_view + n_views + 1, t) - item_view) - 1;
    const int64_t s = (t - item_view[v]) * slice;
    const int64_t len = std::min(slice, view_pixels[v] - s);
    int64_t acc[slice];
    for (int64_t k = mask_off[v]; k < mask_off[v + 1]; ++k) {
      const uint8_t* __restrict__ m = masks[k] + s;
      const uint64_t id = (uint64_t)ids[k];
      if (k == mask_off[v]) {
        for (int64_t j = 0; j < len; ++j) acc[j] = (int64_t)(m[j] * id);  // numpy's int64 product wraps
      } else {
        for (int64_t j = 0; j < len; ++j) acc[j] = std::max(acc[j], (int64_t)(m[j] * id));
      }
    }
    if (out_dtype == DC_U8) {
      uint8_t* __restrict__ o = static_cast<uint8_t*>(dst) + pix_off[v] + s;
      uint64_t seen = 0;
      for (int64_t j = 0; j < len; ++j) {
        seen |= (uint64_t)acc[j];
        o[j] = (uint8_t)acc[j];
      }
      if (seen & ~(uint64_t)0xff) bad.store(1, std::memory_order_relaxed);
    } else {
      memcpy(static_cast<int64_t*>(dst) + pix_off[v] + s, acc, sizeof(int64_t) * (size_t)len);
    }
  });
  free(item_view);
  *out_of_range = bad.load();
  return DC_OK;
}

}  // extern "C"
