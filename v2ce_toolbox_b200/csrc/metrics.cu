// Stage-2 evaluation metric on sm_100a: nearest-timestamp distance between ground-truth and predicted events.
// Replaces /root/reference/train/scripts/stage2/stage2_metrics.py:22-88 (ts_diff_metric): for every ground-truth event
// the smallest |t_pred - t_gt| over the predicted events of the same polarity at the pixels within `search_range`
// (clamped to the sensor), capped at 1e6/fps/10*3 us (`overflow` counts the capped ones); the metric is the mean.
// The reference builds 346 x 260 x 2 Python lists and loops over events on the host (minutes per recording).
//
// Data layout: both event sets are the packed 13-byte records the pipeline produces (timestamp<i8, x<i2, y<i2,
// polarity i1).  Predicted timestamps are binned per (x, y, polarity) cell in CSR form -- count, exclusive scan, fill
// with an atomic cursor (the order inside a cell does not matter for a minimum) -- then one thread per ground-truth
// event scans the cells of its neighbourhood.  Integer distances are summed exactly in int64.
#include "common.cuh"

namespace v2ce {
namespace metrics {

__global__ void cell_count_kernel(const uint8_t* __restrict__ pred, long long n, int W, int H, int* __restrict__ count,
                                  int* __restrict__ bad) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Rec e = load_rec(pred + i * 13);
  if (e.x < 0 || e.x >= W || e.y < 0 || e.y >= H || (e.p != 0 && e.p != 1)) { atomicAdd(bad, 1); return; }
  atomicAdd(&count[(e.x * H + e.y) * 2 + e.p], 1);
}

// exclusive scan of `n` ints (one block; n ~ 180 k cells), start[n] = total; the cursors start at the cell starts
__global__ void cell_scan_kernel(const int* __restrict__ count, int n, int* __restrict__ start, int* __restrict__ cursor) {
  __shared__ int wsum[32];
  __shared__ int carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < n; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const int v = (i < n) ? count[i] : 0;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, inc, o);
      if ((threadIdx.x & 31) >= o) inc += t;
    }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
      const int w = (threadIdx.x < (blockDim.x >> 5)) ? wsum[threadIdx.x] : 0;
      int wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wi, o);
        if (threadIdx.x >= o) wi += t;
      }
      wsum[threadIdx.x] = wi - w;
    }
    __syncthreads();
    const int ex = carry_s + wsum[threadIdx.x >> 5] + inc - v;
    if (i < n) { start[i] = ex; cursor[i] = ex; }
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = ex + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) start[n] = carry_s;
}

__global__ void cell_fill_kernel(const uint8_t* __restrict__ pred, long long n, int W, int H, int* __restrict__ cursor,
                                 long long* __restrict__ cell_ts) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Rec e = load_rec(pred + i * 13);
  if (e.x < 0 || e.x >= W || e.y < 0 || e.y >= H || (e.p != 0 && e.p != 1)) return;
  cell_ts[atomicAdd(&cursor[(e.x * H + e.y) * 2 + e.p], 1)] = e.ts;
}

// result[0] += integer distances below the cap, result[1] += capped events, result[2] += events outside the sensor
__global__ void ts_diff_kernel(const uint8_t* __restrict__ gt, long long n, int W, int H, int range, double cap,
                               const int* __restrict__ start, const long long* __restrict__ cell_ts,
                               unsigned long long* __restrict__ result) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long sum = 0ull, over = 0ull, bad = 0ull;
  if (i < n) {
    const Rec e = load_rec(gt + i * 13);
    if (e.x < 0 || e.x >= W || e.y < 0 || e.y >= H || (e.p != 0 && e.p != 1)) {
      bad = 1ull;
    } else {
      long long best = LLONG_MAX;
      const int a0 = max(e.x - range, 0), a1 = min(e.x + range + 1, W), b0 = max(e.y - range, 0), b1 = min(e.y + range + 1, H);
      for (int a = a0; a < a1; ++a)
        for (int b = b0; b < b1; ++b) {
          const int cell = (a * H + b) * 2 + e.p;
          for (int k = start[cell]; k < start[cell + 1]; ++k) {
            const long long d = cell_ts[k] - e.ts;
            const long long ad = d < 0 ? -d : d;
            best = ad < best ? ad : best;
          }
        }
      // stage2_metrics.py:61,73-75: diff starts at 1e6 (no predicted event in the window, or none closer than 1e6 us)
      // and is capped when it exceeds 1e6/fps/10*3; at fps <= 0.3 the cap is >= 1e6, so the clamped value is what adds up
      const long long d = best > 1000000 ? 1000000 : best;
      if ((double)d > cap) over = 1ull; else sum = (unsigned long long)d;
    }
  }
  // block reduction, three atomics per block
  __shared__ unsigned long long red[3][8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    over += __shfl_xor_sync(0xffffffffu, over, o);
    bad += __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = sum; red[1][threadIdx.x >> 5] = over; red[2][threadIdx.x >> 5] = bad; }
  __syncthreads();
  if (threadIdx.x < 3) {
    unsigned long long t = 0ull;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[threadIdx.x][w];
    if (t) atomicAdd(result + threadIdx.x, t);
  }
}

}  // namespace metrics
}  // namespace v2ce

using namespace v2ce;
using namespace v2ce::metrics;

extern "C" int v2ce_ts_diff_workspace_bytes(int32_t width, int32_t height, int64_t n_pred, size_t* bytes) {
  V2CE_REQUIRE(bytes != nullptr && width > 0 && height > 0 && n_pred >= 0, "bad arguments");
  V2CE_REQUIRE((long long)width * height * 2 < (1LL << 30) && n_pred < (1LL << 31), "too large");
  const size_t cells = (size_t)width * height * 2;
  *bytes = align_up(4 * cells, 256) + align_up(4 * (cells + 1), 256) + align_up(4 * cells, 256) + align_up(8 * (size_t)(n_pred > 0 ? n_pred : 1), 256) + 256;
  return V2CE_OK;
}

extern "C" int v2ce_ts_diff_metric(const uint8_t* gt_records_dev, int64_t n_gt, const uint8_t* pred_records_dev, int64_t n_pred,
                                   int32_t width, int32_t height, int32_t search_range, double cap_us, void* ws_dev,
                                   size_t ws_bytes, int64_t* result_dev, void* stream) {
  V2CE_REQUIRE(ws_dev && result_dev, "NULL device pointer");
  V2CE_REQUIRE(n_gt >= 0 && n_pred >= 0 && (n_gt == 0 || gt_records_dev) && (n_pred == 0 || pred_records_dev), "bad event arrays");
  V2CE_REQUIRE(width > 0 && height > 0 && search_range >= 0 && search_range < 64, "bad geometry / search_range");
  size_t need = 0;
  if (int e = v2ce_ts_diff_workspace_bytes(width, height, n_pred, &need)) return e;
  if (need > ws_bytes) return set_error(V2CE_ERR_WORKSPACE, "ts_diff workspace too small: need %zu, got %zu", need, ws_bytes);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int cells = width * height * 2;
  Arena a(ws_dev, ws_bytes);
  int* count = a.take<int>(cells);
  int* start = a.take<int>(cells + 1);
  int* cursor = a.take<int>(cells);
  long long* cell_ts = a.take<long long>((size_t)(n_pred > 0 ? n_pred : 1));
  int* bad = a.take<int>(1);
  V2CE_CUDA_CHECK(cudaMemsetAsync(count, 0, sizeof(int) * cells, s));
  V2CE_CUDA_CHECK(cudaMemsetAsync(bad, 0, sizeof(int), s));
  V2CE_CUDA_CHECK(cudaMemsetAsync(result_dev, 0, 4 * sizeof(int64_t), s));
  if (n_pred > 0) {
    cell_count_kernel<<<(unsigned)((n_pred + 255) / 256), 256, 0, s>>>(pred_records_dev, n_pred, width, height, count, bad);
    V2CE_LAUNCH_CHECK("metrics::cell_count_kernel");
  }
  cell_scan_kernel<<<1, 1024, 0, s>>>(count, cells, start, cursor);
  V2CE_LAUNCH_CHECK("metrics::cell_scan_kernel");
  if (n_pred > 0) {
    cell_fill_kernel<<<(unsigned)((n_pred + 255) / 256), 256, 0, s>>>(pred_records_dev, n_pred, width, height, cursor, cell_ts);
    V2CE_LAUNCH_CHECK("metrics::cell_fill_kernel");
  }
  if (n_gt > 0) {
    ts_diff_kernel<<<(unsigned)((n_gt + 255) / 256), 256, 0, s>>>(gt_records_dev, n_gt, width, height, search_range, cap_us, start,
                                                                  cell_ts, reinterpret_cast<unsigned long long*>(result_dev));
    V2CE_LAUNCH_CHECK("metrics::ts_diff_kernel");
  }
  // result_dev[3] = predicted events outside the sensor (ignored, as they would raise IndexError upstream)
  V2CE_CUDA_CHECK(cudaMemcpyAsync(result_dev + 3, bad, sizeof(int), cudaMemcpyDeviceToDevice, s));
  return V2CE_OK;
}
