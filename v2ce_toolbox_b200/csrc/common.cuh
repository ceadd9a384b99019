// Shared helpers for libv2ce_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/v2ce_b200.h"

namespace v2ce {

// thread-local message of the last failing call (v2ce_last_error)
char* last_error_buffer();
int set_error(int code, const char* fmt, ...);

#define V2CE_CUDA_CHECK(expr)                                                                   \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return ::v2ce::set_error(V2CE_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                               __FILE__, __LINE__);                                             \
  } while (0)

#define V2CE_LAUNCH_CHECK(name)                                                                 \
  do {                                                                                          \
    cudaError_t _e = cudaGetLastError();                                                        \
    if (_e != cudaSuccess)                                                                      \
      return ::v2ce::set_error(V2CE_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(_e)); \
  } while (0)

#define V2CE_REQUIRE(cond, ...)                                                                 \
  do {                                                                                          \
    if (!(cond)) return ::v2ce::set_error(V2CE_ERR_INVALID, __VA_ARGS__);                       \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace.
struct Arena {
  char* base;
  size_t size;
  size_t off;
  Arena(void* p, size_t n) : base(static_cast<char*>(p)), size(n), off(0) {}
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 256);
    T* r = reinterpret_cast<T*>(base + off);
    off += count * sizeof(T);
    return r;
  }
  bool ok() const { return off <= size; }
};

// One packed 13-byte event record (timestamp <i8, x <i2, y <i2, polarity i1; any alignment), as the LDATI and baseline
// emitters write it.  Polarity -1 is folded into 0: the stage-2 metric (stage2_metrics.py:38-41) and the voxeliser
// both treat -1 like 0.  Other polarity values are returned as they are, for the caller to reject.
struct Rec { long long ts; int x, y, p; };

__device__ __forceinline__ Rec load_rec(const uint8_t* __restrict__ r) {
  unsigned long long t = 0ull;
#pragma unroll
  for (int b = 0; b < 8; ++b) t |= (unsigned long long)r[b] << (8 * b);
  Rec e;
  e.ts = (long long)t;
  e.x = (int)(short)((unsigned)r[8] | ((unsigned)r[9] << 8));
  e.y = (int)(short)((unsigned)r[10] | ((unsigned)r[11] << 8));
  e.p = (int)(signed char)r[12];
  if (e.p == -1) e.p = 0;
  return e;
}

int sm_count_cached();
// index (< 64) of the current CUDA device: function attributes and constant memory are per device, so the
// one-time-setup caches of the launchers are kept per device (one process may drive several GPUs)
int device_slot();

}  // namespace v2ce
