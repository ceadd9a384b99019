#include "common.cuh"

#include <string.h>

namespace v2ce {

char* last_error_buffer() {
  static thread_local char buf[1024] = {0};
  return buf;
}

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(last_error_buffer(), 1024, fmt, ap);
  va_end(ap);
  return code;
}

int device_slot() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  return dev & 63;
}

int sm_count_cached() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      return 148;
  }
  return cached;
}

}  // namespace v2ce

extern "C" const char* v2ce_last_error(void) { return v2ce::last_error_buffer(); }

extern "C" int v2ce_version(void) { return 100; }

extern "C" int v2ce_device_check(int device, int* sm_count, int* cc_major, int* cc_minor) {
  int n = 0;
  V2CE_CUDA_CHECK(cudaGetDeviceCount(&n));
  V2CE_REQUIRE(device >= 0 && device < n, "device %d out of range (%d visible)", device, n);
  int major = 0, minor = 0, sms = 0;
  V2CE_CUDA_CHECK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  V2CE_CUDA_CHECK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
  V2CE_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (sm_count) *sm_count = sms;
  if (cc_major) *cc_major = major;
  if (cc_minor) *cc_minor = minor;
  V2CE_REQUIRE(major == 10, "libv2ce_b200 is built for sm_100a only; device %d is sm_%d%d", device, major, minor);
  return V2CE_OK;
}

// ------------------------------------------------------------------------------------------
// Peer windows (include/v2ce_b200.h): CUDA IPC mappings of a destination buffer + copy-engine transfers
// ------------------------------------------------------------------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "V2CE_PEER_HANDLE_BYTES");

extern "C" int v2ce_peer_window_alloc(size_t bytes, void** window_dev, uint8_t* handle_out) {
  V2CE_REQUIRE(window_dev && handle_out && bytes > 0, "v2ce_peer_window_alloc: null argument or zero size");
  void* p = nullptr;
  V2CE_CUDA_CHECK(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return v2ce::set_error(V2CE_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
  }
  memcpy(handle_out, &h, sizeof(h));
  *window_dev = p;
  return V2CE_OK;
}

extern "C" int v2ce_peer_window_free(void* window_dev) {
  if (window_dev) V2CE_CUDA_CHECK(cudaFree(window_dev));
  return V2CE_OK;
}

extern "C" int v2ce_peer_window_open(const uint8_t* handle, void** window_dev) {
  V2CE_REQUIRE(handle && window_dev, "v2ce_peer_window_open: null argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void* p = nullptr;
  V2CE_CUDA_CHECK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  *window_dev = p;
  return V2CE_OK;
}

extern "C" int v2ce_peer_window_close(void* window_dev) {
  if (window_dev) V2CE_CUDA_CHECK(cudaIpcCloseMemHandle(window_dev));
  return V2CE_OK;
}

extern "C" int v2ce_peer_copy_async(void* dst_dev, const void* src_dev, size_t bytes, void* stream) {
  if (bytes == 0) return V2CE_OK;
  V2CE_REQUIRE(dst_dev && src_dev, "v2ce_peer_copy_async: null pointer");
  V2CE_CUDA_CHECK(cudaMemcpyAsync(dst_dev, src_dev, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
  return V2CE_OK;
}
