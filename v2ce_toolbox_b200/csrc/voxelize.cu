// Event stream -> voxel grid on sm_100a: counts packed 13-byte records into a float32 (F, 2, nbins, H, W) grid.
// The binning convention is the toolbox's own (include/v2ce_b200.h, v2ce_events_to_voxels); it is not a port of the
// reference's training voxeliser.
//
// One pass, no workspace: the grid and the four status counters are zeroed on the stream, then one thread per record
// decodes it, finds its frame by binary search over the edges (any record order), its bin in exact int64 arithmetic, and
// adds 1.0f to its cell with a fire-and-forget reduction.  The sums are integers, so the grid is bit-identical for
// every order of the additions while a cell stays below 2^24.
#include "common.cuh"

namespace v2ce {
namespace voxelize {

constexpr int kThreads = 256;

__device__ __forceinline__ void red_add_f32(float* p, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// f with e[f] <= t < e[f+1], given e[0] <= t < e[F]
__device__ __forceinline__ int find_frame(const long long* __restrict__ e, int F, long long t) {
  int lo = 0, hi = F;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(e + mid) <= t) lo = mid; else hi = mid;
  }
  return lo;
}

// One thread per record.  Measured on B200 and not kept (DESIGN.md §4.8): staging a block's records through shared
// memory with 16-byte loads, and warp aggregation of equal cells with __match_any_sync.
__global__ void __launch_bounds__(kThreads) voxelize_kernel(const uint8_t* __restrict__ rec, long long n,
                                                            const long long* __restrict__ edges, int F, int nbins,
                                                            int H, int W, float* __restrict__ vox,
                                                            unsigned long long* __restrict__ status) {
  const long long i = (long long)blockIdx.x * kThreads + threadIdx.x;
  int kind = -1;                                     // status slot of a skipped record
  long long cell = -1;
  if (i < n) {
    const Rec e = load_rec(rec + i * 13);
    if (e.x < 0 || e.x >= W || e.y < 0 || e.y >= H) {
      kind = 0;
    } else if (e.p != 0 && e.p != 1) {
      kind = 1;
    } else if (e.ts < __ldg(edges)) {
      kind = 2;
    } else if (e.ts >= __ldg(edges + F)) {
      kind = 3;
    } else {
      const int f = find_frame(edges, F, e.ts);
      const long long e0 = __ldg(edges + f);
      const long long len = __ldg(edges + f + 1) - e0;
      const long long c = ((e.ts - e0 + 1) * nbins - 1) / len;    // bin c starts at e0 + floor(c * len / nbins)
      const int plane = 1 - e.p;                                 // polarity 1 -> plane 0, 0 (and -1) -> plane 1
      cell = (((long long)(2 * f + plane) * nbins + c) * H + e.y) * W + e.x;
    }
  }
  if (cell >= 0) red_add_f32(vox + cell, 1.0f);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const unsigned m = __ballot_sync(0xffffffffu, kind == k);
    if (m && (threadIdx.x & 31) == 0) atomicAdd(status + k, (unsigned long long)__popc(m));
  }
}

}  // namespace voxelize
}  // namespace v2ce

using namespace v2ce;
using namespace v2ce::voxelize;

extern "C" int v2ce_events_to_voxels(const uint8_t* records_dev, int64_t n_events, const int64_t* frame_edges_us_dev,
                                     int32_t n_frames, int32_t nbins, int32_t height, int32_t width, float* voxels_dev,
                                     int64_t* status_dev, void* stream) {
  V2CE_REQUIRE(frame_edges_us_dev && voxels_dev && status_dev, "NULL device pointer");
  V2CE_REQUIRE(n_events >= 0 && (n_events == 0 || records_dev), "bad event array");
  V2CE_REQUIRE(n_frames >= 1 && nbins >= 1 && height >= 1 && width >= 1, "bad grid shape (F %d, nbins %d, %d x %d)",
               n_frames, nbins, height, width);
  const double cells = (double)n_frames * 2.0 * nbins * height * width;
  V2CE_REQUIRE(cells * 4.0 < 9.0e18, "grid of %.3g cells is too large", cells);
  V2CE_REQUIRE(n_events / kThreads < 0x7fffffffLL, "%lld events are too many for one call", (long long)n_events);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  V2CE_CUDA_CHECK(cudaMemsetAsync(voxels_dev, 0, (size_t)cells * sizeof(float), s));
  V2CE_CUDA_CHECK(cudaMemsetAsync(status_dev, 0, 4 * sizeof(int64_t), s));
  if (n_events == 0) return V2CE_OK;
  const unsigned blocks = (unsigned)((n_events + kThreads - 1) / kThreads);
  voxelize_kernel<<<blocks, kThreads, 0, s>>>(records_dev, n_events, reinterpret_cast<const long long*>(frame_edges_us_dev),
                                               n_frames, nbins, height, width, voxels_dev,
                                               reinterpret_cast<unsigned long long*>(status_dev));
  V2CE_LAUNCH_CHECK("voxelize::voxelize_kernel");
  return V2CE_OK;
}
