// common.h -- shared host-side helpers for the kkx CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <stdexcept>
#include <atomic>
#include <mutex>
#include <stdlib.h>

namespace kkx {

struct CudaError : std::runtime_error {
  explicit CudaError(const std::string& s) : std::runtime_error(s) {}
};
struct ArgError : std::runtime_error {
  explicit ArgError(const std::string& s) : std::runtime_error(s) {}
};
struct IoError : std::runtime_error {
  explicit IoError(const std::string& s) : std::runtime_error(s) {}
};
struct StateError : std::runtime_error {   // call sequence error (nothing staged / nothing run yet) -> KKX_ERR_STATE
  explicit StateError(const std::string& s) : std::runtime_error(s) {}
};

#define KKX_CUDA(expr)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      char _b[512];                                                                         \
      snprintf(_b, sizeof _b, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                 \
               cudaGetErrorString(_e));                                                     \
      throw ::kkx::CudaError(_b);                                                           \
    }                                                                                       \
  } while (0)

// Diagnostic switches read from the environment (role cycle counters, perf-experiment masks) exist only in experiment
// builds (-DKKX_EXPERIMENTS, e.g. KKX_NVCC_EXTRA=-DKKX_EXPERIMENTS python -m kokorox_b200.build --force): in the
// production library no environment variable can change which kernel runs or what it computes.
#ifdef KKX_EXPERIMENTS
inline bool env_flag(const char* name, bool dflt) {
  const char* e = getenv(name);
  return e ? (e[0] != '0') : dflt;
}
inline int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}
#else
inline bool env_flag(const char*, bool dflt) { return dflt; }
inline int env_int(const char*, int dflt) { return dflt; }
#endif

// One-time per-device setup (a kernel's dynamic shared-memory limit, constant tables): two sessions on two
// threads may reach a launcher's first use together, so the flag is a std::once_flag per device, not a bool.
struct DevOnce {
  std::once_flag flag[64];
  template <class F> void run(int dev, F&& fn) {
    if (dev >= 0 && dev < 64) std::call_once(flag[dev], fn); else fn();
  }
};
// Call before launching `Kernel` with `bytes` of dynamic shared memory: raises the kernel's limit to `bytes` once per
// device and returns the current device; a failure throws CudaError.  The template argument is the kernel itself, not
// its type, so each kernel has its own once-state (conv_tc_kernel<128,3,1> and <64,4,1> share one function type).
template <auto Kernel>
int prepare_smem_launch(int bytes) {
  static DevOnce once;
  int dev = 0;
  KKX_CUDA(cudaGetDevice(&dev));
  once.run(dev, [bytes] { KKX_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)); });
  return dev;
}
inline int device_sm_count(int dev) {
  static std::atomic<int> cache[64];
  if (dev < 0 || dev >= 64) return 148;
  int n = cache[dev].load(std::memory_order_relaxed);
  if (n <= 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

// Launch-count bookkeeping ("gpu_launches" in bench.py) + optional per-launch error checks.
struct LaunchStats {
  int64_t launches = 0;
  bool check_each = false;  // KKX_DEBUG_SYNC=1: synchronize + check after every launch
  // per-kernel timing (kkx_profile_enable): one event after every launch on the in-order stream;
  // the gap between consecutive events is attributed to the launch in between
  bool profile = false;
  bool detail = false;                   // per-shape kernel names (KKX_PROFILE_DETAIL=1)
  std::vector<cudaEvent_t> events;       // pool, events[0] = start of run
  std::vector<std::string> names;        // names[i] = kernel launched before events[i+1]
  size_t n_events = 0;
  double conv_flops = 0;                 // algorithmic FLOPs issued through the shifted-GEMM kernels (all of them)
  double arb_flops = 0, arb_bytes = 0;   // share of the fused res-block conv (kernels_arb.cu) + its algorithmic HBM bytes
  cudaEvent_t next_event() {
    if (n_events == events.size()) {
      cudaEvent_t e; cudaEventCreate(&e); events.push_back(e);
    }
    return events[n_events++];
  }
};
extern thread_local LaunchStats* g_launch_stats;
extern thread_local bool g_dry_run;  // true while sizing arenas: launchers return immediately

inline void post_launch(const char* name, cudaStream_t st) {
  if (g_launch_stats) {
    g_launch_stats->launches++;
    if (g_launch_stats->profile) {
      cudaEventRecord(g_launch_stats->next_event(), st);
      g_launch_stats->names.push_back(name);
    }
  }
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && g_launch_stats && g_launch_stats->check_each) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    char b[512];
    snprintf(b, sizeof b, "kernel %s failed: %s", name, cudaGetErrorString(e));
    throw CudaError(b);
  }
}

// Bump allocator over one device allocation; reset per phase.  All returned pointers are
// 256-byte aligned.  Grow-only: a too-small arena is re-allocated (caller must have synced).
class Arena {
 public:
  ~Arena() { release(); }
  void release() {
    if (base_) cudaFree(base_);
    base_ = nullptr; cap_ = 0; used_ = 0;
  }
  void reserve(size_t bytes) {
    if (bytes <= cap_) return;
    release();
    KKX_CUDA(cudaMalloc(&base_, bytes));
    cap_ = bytes;
  }
  void reset() { used_ = 0; }
  // virtual mode: allocations only advance the counter (used to size the arena by a dry run)
  void set_virtual(bool v) { virtual_ = v; }
  size_t used() const { return used_; }
  size_t capacity() const { return cap_; }
  const void* base() const { return base_; }
  void* alloc_bytes(size_t bytes) {
    size_t a = (used_ + 255) & ~size_t(255);
    if (!virtual_ && a + bytes > cap_) {
      char b[256];
      snprintf(b, sizeof b, "arena overflow: need %zu + %zu > %zu", a, bytes, cap_);
      throw CudaError(b);
    }
    used_ = a + bytes;
    return static_cast<char*>(base_) + a;
  }
  template <class T> T* alloc(size_t n) { return static_cast<T*>(alloc_bytes(n * sizeof(T))); }

 private:
  void* base_ = nullptr;
  size_t cap_ = 0, used_ = 0;
  bool virtual_ = false;
};

// Pinned host staging memory for the small index tables a run uploads (level offsets, tile prefix sums, sample
// offsets).  A cudaMemcpyAsync from PAGEABLE memory synchronises the stream before it starts; from pinned memory
// it is a true asynchronous copy, so a B = 1 call no longer pays one stream drain per table.  Bump allocator,
// reset when the stream is known to be idle (start of a call); alloc() returns nullptr when full and the caller
// drains the stream and resets.
class PinnedArena {
 public:
  ~PinnedArena() { if (base_) cudaFreeHost(base_); }
  void reserve(size_t bytes) {
    if (bytes <= cap_) return;
    if (base_) cudaFreeHost(base_);
    base_ = nullptr; cap_ = 0; used_ = 0;
    KKX_CUDA(cudaMallocHost(&base_, bytes));
    cap_ = bytes;
  }
  void reset() { used_ = 0; }
  void* alloc_bytes(size_t bytes) {
    const size_t a = (used_ + 63) & ~size_t(63);
    if (a + bytes > cap_) return nullptr;
    used_ = a + bytes;
    return static_cast<char*>(base_) + a;
  }
 private:
  void* base_ = nullptr;
  size_t cap_ = 0, used_ = 0;
};

// A ragged "level": B items packed along the row axis with zero gaps between items.
// Item b owns rows [off[b], off[b] + len[b]).
struct Level {
  int B = 0;
  std::vector<int> off, len;
  int rows = 0;      // total rows incl. gaps
  int max_len = 0;
  long long sum_len = 0;
  int* d_off = nullptr;  // device copies
  int* d_len = nullptr;
  // prefix sums (B+1) of the per-item tile counts for 128- and 256-row tiles (persistent kernels)
  int* d_tiles128 = nullptr; int* d_tiles256 = nullptr;
  int ntiles128 = 0, ntiles256 = 0;
};

constexpr int kGapRows = 32;  // >= largest conv halo (k=11, dil=5 -> 25)

}  // namespace kkx
