// Window assembly on sm_100a: writes the uint8 gray window tensor (n_windows, L+1, H, W_out) of one batch from frames
// that stay where the caller keeps them (include/v2ce_b200.h, v2ce_assemble_windows).
//
// One launch per batch, one thread per output pixel: the thread finds its source frame through the window's slot table,
// reads the pixel's C bytes at (row * pitch + (x0 + x) * C) and writes one gray byte.  Colour is converted as OpenCV's
// cvtColor(COLOR_{BGR,RGB,BGRA,RGBA}2GRAY) does for 8-bit input: 15-bit fixed point, rounded half up, alpha ignored.
// The coefficients were derived from cv2 itself and are pinned over all 2^24 colours by tests/test_frames_oracle.py.
#include "common.cuh"

namespace v2ce {
namespace frames {

constexpr int kThreads = 256;
constexpr int kB = 3735, kG = 19235, kR = 9798, kShift = 15;   // kB + kG + kR == 1 << kShift

__global__ void __launch_bounds__(kThreads) assemble_kernel(const long long* __restrict__ frames,
                                                            const int* __restrict__ slots, int H, int C, int rgb,
                                                            int x0, int W_out, uint8_t* __restrict__ out) {
  const int plane = H * W_out;
  const int p = blockIdx.x * kThreads + threadIdx.x;
  if (p >= plane) return;
  const int f = blockIdx.y;                                   // output frame: window * (L+1) + j
  const int s = __ldg(slots + f);
  const uint8_t* src = reinterpret_cast<const uint8_t*>(__ldg(frames + 2 * s));
  const long long pitch = __ldg(frames + 2 * s + 1);
  const int y = p / W_out, x = p - y * W_out;
  const uint8_t* px = src + y * pitch + (long long)(x0 + x) * C;
  int v;
  if (C == 1) {
    v = px[0];
  } else {
    const int c0 = px[0], c1 = px[1], c2 = px[2];
    const int b = rgb ? c2 : c0, r = rgb ? c0 : c2;
    v = (b * kB + c1 * kG + r * kR + (1 << (kShift - 1))) >> kShift;
  }
  out[(long long)f * plane + p] = (uint8_t)v;
}

}  // namespace frames
}  // namespace v2ce

using namespace v2ce;
using namespace v2ce::frames;

extern "C" int v2ce_assemble_windows(const int64_t* frames_dev, const int32_t* slots_dev, int32_t n_windows,
                                     int32_t frames_per_window, int32_t height, int32_t width, int32_t channels,
                                     int32_t rgb_order, int32_t x0, int32_t out_width, uint8_t* out_dev, void* stream) {
  V2CE_REQUIRE(frames_dev && slots_dev && out_dev, "NULL device pointer");
  V2CE_REQUIRE(channels == 1 || channels == 3 || channels == 4, "channels must be 1, 3 or 4, got %d", channels);
  V2CE_REQUIRE(rgb_order == 0 || rgb_order == 1, "rgb_order must be 0 (BGR) or 1 (RGB), got %d", rgb_order);
  V2CE_REQUIRE(n_windows >= 1 && frames_per_window >= 1, "bad window table (%d windows of %d frames)", n_windows,
               frames_per_window);
  V2CE_REQUIRE((int64_t)n_windows * frames_per_window <= 65535, "%d windows of %d frames are too many for one call",
               n_windows, frames_per_window);
  V2CE_REQUIRE(height >= 1 && width >= 1 && out_width >= 1, "bad frame geometry (%d x %d -> width %d)", height, width,
               out_width);
  V2CE_REQUIRE(x0 >= 0 && (int64_t)x0 + out_width <= width, "columns [%d, %d) are outside a frame of width %d", x0,
               x0 + out_width, width);
  V2CE_REQUIRE((int64_t)height * out_width < (1LL << 31), "a %d x %d output frame is too large", height, out_width);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const dim3 grid((unsigned)(((int64_t)height * out_width + kThreads - 1) / kThreads),
                  (unsigned)(n_windows * frames_per_window));
  assemble_kernel<<<grid, kThreads, 0, s>>>(reinterpret_cast<const long long*>(frames_dev), slots_dev, height, channels,
                                            rgb_order, x0, out_width, out_dev);
  V2CE_LAUNCH_CHECK("frames::assemble_kernel");
  return V2CE_OK;
}
