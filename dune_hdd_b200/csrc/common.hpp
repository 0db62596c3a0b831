// Shared host-side plumbing of libhdd_b200: status codes, error string, CUDA checks, launch counter.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <ctime>
#include <sstream>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/hdd_b200.h"
#include "../../include/hdd_b200_testing.h"

namespace hdd {

// Exception carrying the hdd_status the C-ABI function will return.  The set mirrors the exception types the
// reference throws on this path (see include/hdd_b200.h).
struct Error : std::runtime_error {
  int status;
  Error(int s, const std::string& what) : std::runtime_error(what), status(s) {}
};

void set_last_error(const std::string& msg);

extern std::atomic<int64_t> g_kernel_launches;
inline void count_launch(int n = 1) { g_kernel_launches.fetch_add(n, std::memory_order_relaxed); }

#define HDD_THROW(status, msg)                     \
  do {                                             \
    std::ostringstream hdd_oss_;                   \
    hdd_oss_ << msg;                               \
    throw ::hdd::Error((status), hdd_oss_.str());  \
  } while (0)

#define HDD_CUDA(call)                                                                              \
  do {                                                                                              \
    cudaError_t hdd_err_ = (call);                                                                  \
    if (hdd_err_ != cudaSuccess)                                                                    \
      HDD_THROW(HDD_ERR_DEVICE, "CUDA error '" << cudaGetErrorString(hdd_err_) << "' at " << __FILE__ \
                                               << ":" << __LINE__ << " in " #call);                 \
  } while (0)

// Wraps the body of every extern "C" entry point.
template <class F>
int guarded(F&& f) noexcept {
  try {
    f();
    return HDD_OK;
  } catch (const Error& e) {
    set_last_error(e.what());
    return e.status;
  } catch (const std::bad_alloc&) {
    set_last_error("out of host memory");
    return HDD_ERR_INTERNAL;
  } catch (const std::exception& e) {
    set_last_error(e.what());
    return HDD_ERR_INTERNAL;
  } catch (...) {
    set_last_error("unknown error");
    return HDD_ERR_INTERNAL;
  }
}

// HDD_TIMING=1: wall-clock phases of the set-up entry points on stderr (diagnostics; synchronises the stream)
struct PhaseTimer {
  const char* scope;
  cudaStream_t stream;
  bool on;
  double last;
  static double now() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec + 1e-9 * ts.tv_nsec;
  }
  PhaseTimer(const char* sc, cudaStream_t s) : scope(sc), stream(s), last(0.0) {
    static const bool enabled = [] { const char* e = std::getenv("HDD_TIMING"); return e && e[0] == '1'; }();
    on = enabled;
    if (on) last = now();
  }
  void lap(const char* what) {
    if (!on) return;
    if (stream) cudaStreamSynchronize(stream);
    const double t = now();
    std::fprintf(stderr, "[hdd timing] %-18s %-28s %8.3f ms\n", scope, what, 1e3 * (t - last));
    last = t;
  }
};

// ---- host threading for the O(n_cells) passes over the caller's arrays -----------------------------------------
inline int worker_count(int64_t n) {
  const unsigned hw = std::thread::hardware_concurrency();
  int t = int(hw == 0 ? 4 : (hw > 32 ? 32 : hw));
  const int64_t by_size = n / 65536 + 1;  // do not spawn threads for small grids
  return int(by_size < t ? by_size : t);
}

template <class F>
void parallel_for_indexed(int64_t n, int nt, F&& f) {  // f(thread, begin, end), contiguous chunks in order
  if (n <= 0) return;
  if (nt <= 1) { f(0, int64_t(0), n); return; }
  std::vector<std::thread> th;
  const int64_t chunk = (n + nt - 1) / nt;
  for (int t = 0; t < nt; ++t) {
    const int64_t a = t * chunk, b = a + chunk < n ? a + chunk : n;
    if (a >= b) break;
    th.emplace_back([&f, t, a, b] { f(t, a, b); });
  }
  for (auto& x : th) x.join();
}

template <class F>
void parallel_for(int64_t n, F&& f) {  // f(begin, end)
  parallel_for_indexed(n, worker_count(n), [&f](int, int64_t a, int64_t b) { f(a, b); });
}

// bytes this library copied host -> device / device -> host since process start (bench.py's e2e.h2d_bytes_per_step)
extern std::atomic<int64_t> g_h2d_bytes, g_d2h_bytes;
inline cudaError_t h2d_async(void* dst, const void* src, size_t bytes, cudaStream_t s) {
  g_h2d_bytes.fetch_add(int64_t(bytes));
  return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s);
}

// HDD_CG_PHASES=1: the solver records a CUDA event after every phase of every iteration (halo exchange, SpMV, all-reduces,
// update, the multigrid stages, direction) - launched directly, not as a graph - and prints, at the end of the solve, the
// time per phase summed over the iterations (this rank's device timeline).  A diagnostic: the numbers of a normal run are
// taken without it.
struct SolvePhases {
  bool on = false;
  std::vector<std::pair<const char*, cudaEvent_t>> marks;
  void begin(cudaStream_t s) { if (on) mark("(start)", s); }
  void mark(const char* name, cudaStream_t s) {
    if (!on) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, s);
    marks.emplace_back(name, e);
  }
  void report(int rank, int iterations);  // mesh.cu
};
SolvePhases& phase_timer();

// Device memory of the library comes from a small caching allocator (mesh.cu): a freed block is kept and handed to the next
// request of the same size on the same device.  Discretizations are created and destroyed per solve in the reference's
// studies (test/linearelliptic.hh:150-160) with the same sizes every time, and cudaMalloc / cudaFree synchronise the device
// and - once peer access is enabled by NCCL or CUDA IPC - map / unmap the block on every peer, which costs milliseconds per
// call.  The cache holds at most kDevCacheFraction of the device memory (least recently freed blocks are released first) and
// is emptied when an allocation fails.  HDD_DEV_CACHE=0 turns it off.
void* dev_alloc(size_t bytes);
void dev_free(void* p, size_t bytes);
void dev_cache_release_all();

// RAII device buffer
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  void release() {
    if (p) dev_free(p, n * sizeof(T) + 32);
    p = nullptr;
    n = 0;
  }
  void alloc(size_t count) {
    release();
    if (count == 0) count = 1;
    // 32 bytes of slack: the bulk-copy SpMV rounds its 8-byte aligned row blocks out to 16-byte boundaries
    p = static_cast<T*>(dev_alloc(count * sizeof(T) + 32));
    n = count;
  }
  void upload(const T* host, size_t count, cudaStream_t s) {
    if (n < count || !p) alloc(count);
    if (count) HDD_CUDA(h2d_async(p, host, count * sizeof(T), s));
  }
  void zero(cudaStream_t s) {
    if (p) HDD_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s));
  }
};

}  // namespace hdd
