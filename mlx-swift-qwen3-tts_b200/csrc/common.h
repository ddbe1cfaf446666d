// Shared host-side plumbing for libqwen3tts_b200: status-carrying exception, CUDA error checks, device arena.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/qwen3tts_b200.h"

namespace q3 {

struct Error : std::runtime_error {
  q3tts_status status;
  Error(q3tts_status s, const std::string& m) : std::runtime_error(m), status(s) {}
};

[[noreturn]] inline void fail(q3tts_status s, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  throw Error(s, buf);
}

#define Q3_CUDA(expr)                                                                                  \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess)                                                                             \
      ::q3::fail(Q3TTS_ERR_CUDA, "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__, \
                 cudaGetErrorString(_e));                                                              \
  } while (0)

#define Q3_CHECK(cond, status, ...) \
  do {                              \
    if (!(cond)) ::q3::fail(status, __VA_ARGS__); \
  } while (0)

inline size_t dtype_size(int dt) { return dt == Q3TTS_F32 ? 4 : 2; }

// Programmatic dependent launch (PDL): a kernel launched with `pdl` may start (prologue, weight prefetch) while its
// predecessor in the stream is still draining; it calls pdl_wait() before touching anything the predecessor wrote.  Kernels
// call pdl_launch_dependents() early so their successor can be scheduled.  Both instructions are no-ops without the attribute.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline void launch_kernel_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  Q3_CUDA(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
}
inline bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("Q3TTS_PDL"); return !(e && atoi(e) == 0); }();
  return on;
}
#endif

// Counts every kernel this library launches (reported as q3tts_timing.kernel_launches / bench gpu_launches).
struct LaunchCounter {
  int64_t n = 0;
  bool capturing = false;   // while a CUDA graph is being captured launches are counted into `captured`
  int64_t captured = 0;
  inline void tick() { if (capturing) ++captured; else ++n; }
};

// Bump allocator over cudaMalloc'ed slabs: weights and state live for the handle's lifetime.
class DeviceArena {
 public:
  ~DeviceArena() { release(); }
  void* alloc(size_t bytes, size_t align = 256) {
    if (bytes == 0) bytes = align;
    size_t off = (used_ + align - 1) / align * align;
    if (slabs_.empty() || off + bytes > cap_) {
      size_t sz = bytes > kSlab ? bytes : kSlab;
      void* p = nullptr;
      Q3_CUDA(cudaMalloc(&p, sz));
      slabs_.push_back(p);
      cap_ = sz;
      used_ = 0;
      off = 0;
      total_ += sz;
    }
    used_ = off + bytes;
    return static_cast<char*>(slabs_.back()) + off;
  }
  template <typename T>
  T* alloc_n(size_t n) { return static_cast<T*>(alloc(n * sizeof(T))); }
  void release() {
    for (void* p : slabs_) cudaFree(p);
    slabs_.clear();
    cap_ = used_ = total_ = 0;
  }
  size_t total() const { return total_; }

 private:
  static constexpr size_t kSlab = size_t(256) << 20;
  std::vector<void*> slabs_;
  size_t cap_ = 0, used_ = 0, total_ = 0;
};

}  // namespace q3
