// Stage 1 on sm_100a: the V2ce3d 3D-UNet forward (eval mode) as a fixed schedule of fused
// conv launches.  Replaces /root/reference/scripts/v2ce_3d.py:12-30, scripts/unet_2layer.py:203-379,
// scripts/submodules.py:85-124,216-264 and scripts/spectral_norm.py:9-64.
//
// Activation layout in HBM: NDHWC bf16, (B, D=16, H, W, C), row m = ((b*D+d)*H+h)*W+w.
// Schedule per forward at depth % 8 == 0 (30 launches):
//   4  spectral-norm power-iteration kernels (fp32; 12 convs batched per launch), on a side stream
//   2  head: split-bf16 prep + the depth-merged halo kernel (2->32, LeakyReLU)
//   24 tcgen05 convs, per residual block
//        t = relu(bn1(conv1(x)))            x may be the virtual concat [nearest_up(prev), skip]
//        r = bn_d(conv_d(x) + bias_d)       1x1x1 shortcut, present on every block (SURVEY.md F4)
//        y = relu(bn2(conv2(t)) + r)
//      conv1 + shortcut in ONE launch of conv_halo_kdm.cuh for the 4 encoders (stride 2, parity views) and
//      decoders 2/3; conv1 on conv_halo.cuh and the shortcut on the gather kernel (conv_igemm.cuh, side stream) for the
//      2 resblocks and decoders 0/1; every conv2 on a halo kernel, writing its output nearest-upsampled where the
//      next decoder reads it that way; the prediction layer (32->20, ReLU, fp32 (B,L,20,H,W) output) rides in the
//      epilogue of decoders.3.conv2.
//   Otherwise: direct fp32 head kernel, gather kernel for the stride-2 convs and all shortcuts.
#include <map>
#include <string>
#include <vector>

#include <tuple>

#include "conv_halo_kdm.cuh"

namespace v2ce {
namespace unet {

using conv::ConvArgs;

constexpr float kBnEps = 1e-5f;
constexpr int kNumSn = 12;

// What a layer is in the network.  Its role decides its kernel, its channel split and its weight packings (layer_cfg,
// pack_layer) and where forward_impl runs it.  A block's layers follow each other: conv1, conv2, shortcut.
enum class Role { Head, EncConv1, EncShort, ResConv1, ResShort, DecConv1, DecShort, Conv2, Pred };

struct LayerSpec {
  const char* name;
  Role role;
  int block;        // index of the encoder / resblock / decoder the layer belongs to
  int cin, cout, k;
  bool sn, bias;
  const char* bn;   // BatchNorm prefix or nullptr
};

static const LayerSpec kLayers[] = {
    {"UNet.head.conv3d", Role::Head, 0, 2, 32, 3, false, true, nullptr},
    {"UNet.encoders.0.conv1", Role::EncConv1, 0, 32, 64, 3, false, false, "UNet.encoders.0.bn1"},
    {"UNet.encoders.0.conv2", Role::Conv2, 0, 64, 64, 3, false, false, "UNet.encoders.0.bn2"},
    {"UNet.encoders.0.downsample.0", Role::EncShort, 0, 32, 64, 1, false, true, "UNet.encoders.0.downsample.1"},
    {"UNet.encoders.1.conv1", Role::EncConv1, 1, 64, 128, 3, false, false, "UNet.encoders.1.bn1"},
    {"UNet.encoders.1.conv2", Role::Conv2, 1, 128, 128, 3, false, false, "UNet.encoders.1.bn2"},
    {"UNet.encoders.1.downsample.0", Role::EncShort, 1, 64, 128, 1, false, true, "UNet.encoders.1.downsample.1"},
    {"UNet.encoders.2.conv1", Role::EncConv1, 2, 128, 256, 3, false, false, "UNet.encoders.2.bn1"},
    {"UNet.encoders.2.conv2", Role::Conv2, 2, 256, 256, 3, false, false, "UNet.encoders.2.bn2"},
    {"UNet.encoders.2.downsample.0", Role::EncShort, 2, 128, 256, 1, false, true, "UNet.encoders.2.downsample.1"},
    {"UNet.encoders.3.conv1", Role::EncConv1, 3, 256, 512, 3, false, false, "UNet.encoders.3.bn1"},
    {"UNet.encoders.3.conv2", Role::Conv2, 3, 512, 512, 3, false, false, "UNet.encoders.3.bn2"},
    {"UNet.encoders.3.downsample.0", Role::EncShort, 3, 256, 512, 1, false, true, "UNet.encoders.3.downsample.1"},
    {"UNet.resblocks.0.conv1", Role::ResConv1, 0, 512, 512, 3, true, false, "UNet.resblocks.0.bn1"},
    {"UNet.resblocks.0.conv2", Role::Conv2, 0, 512, 512, 3, true, false, "UNet.resblocks.0.bn2"},
    {"UNet.resblocks.0.downsample.0", Role::ResShort, 0, 512, 512, 1, false, true, "UNet.resblocks.0.downsample.1"},
    {"UNet.resblocks.1.conv1", Role::ResConv1, 1, 512, 512, 3, true, false, "UNet.resblocks.1.bn1"},
    {"UNet.resblocks.1.conv2", Role::Conv2, 1, 512, 512, 3, true, false, "UNet.resblocks.1.bn2"},
    {"UNet.resblocks.1.downsample.0", Role::ResShort, 1, 512, 512, 1, false, true, "UNet.resblocks.1.downsample.1"},
    {"UNet.decoders.0.conv1", Role::DecConv1, 0, 768, 256, 3, true, false, "UNet.decoders.0.bn1"},
    {"UNet.decoders.0.conv2", Role::Conv2, 0, 256, 256, 3, true, false, "UNet.decoders.0.bn2"},
    {"UNet.decoders.0.downsample.0", Role::DecShort, 0, 768, 256, 1, false, true, "UNet.decoders.0.downsample.1"},
    {"UNet.decoders.1.conv1", Role::DecConv1, 1, 384, 128, 3, true, false, "UNet.decoders.1.bn1"},
    {"UNet.decoders.1.conv2", Role::Conv2, 1, 128, 128, 3, true, false, "UNet.decoders.1.bn2"},
    {"UNet.decoders.1.downsample.0", Role::DecShort, 1, 384, 128, 1, false, true, "UNet.decoders.1.downsample.1"},
    {"UNet.decoders.2.conv1", Role::DecConv1, 2, 192, 64, 3, true, false, "UNet.decoders.2.bn1"},
    {"UNet.decoders.2.conv2", Role::Conv2, 2, 64, 64, 3, true, false, "UNet.decoders.2.bn2"},
    {"UNet.decoders.2.downsample.0", Role::DecShort, 2, 192, 64, 1, false, true, "UNet.decoders.2.downsample.1"},
    {"UNet.decoders.3.conv1", Role::DecConv1, 3, 96, 32, 3, true, false, "UNet.decoders.3.bn1"},
    {"UNet.decoders.3.conv2", Role::Conv2, 3, 32, 32, 3, true, false, "UNet.decoders.3.bn2"},
    {"UNet.decoders.3.downsample.0", Role::DecShort, 3, 96, 32, 1, false, true, "UNet.decoders.3.downsample.1"},
    {"UNet.pred.conv3d", Role::Pred, 0, 32, 20, 1, false, true, nullptr},
};
constexpr int kNumLayers = sizeof(kLayers) / sizeof(kLayers[0]);

// ------------------------------------------------------------------------------------------
// head: Conv3d(2->32, k3, p1, bias) + LeakyReLU(0.01), fp32 in (B,L,2,H,W) -> bf16 NDHWC
// ------------------------------------------------------------------------------------------
// One thread = 4 consecutive output pixels of a row x 32 channels (128 accumulators).  The weights are FFMA
// constant-bank operands: with shared-memory weights the kernel ran at 36 % of its FP32 floor (two LDS.128 per
// 32 FMAs at 2 warps per scheduler).
__constant__ float c_head_w[27 * 2 * 32];     // [tap][cin][cout]
__constant__ float c_head_b[32];

__global__ void pack_head_kernel(const float* __restrict__ w, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 27 * 2 * 32) return;
  const int n = i % 32, ci = (i / 32) % 2, tap = i / 64;
  out[i] = w[((size_t)n * 2 + ci) * 27 + tap];
}

// U8 = true: x holds raw uint8 gray frames (B, D+1, H, W); image unit (b, l, c) is frame l + c (pair stacking) and
// every sample goes through the pre-processing of v2ce.py:45-64 -- float32 `/255`, Normalize(0.153, 0.165) as a
// float32 subtract and IEEE divide -- evaluated once per gray level into a 256-entry table (bit-identical to the
// host path; SURVEY.md N1).  The resize of image_pre_processing is the identity at the model's own resolution.
template <bool U8>
__global__ void __launch_bounds__(128) head_conv_kernel(const void* __restrict__ xin, int B, int D, int H, int W,
                                                         __nv_bfloat16* __restrict__ out) {
  __shared__ float lut[U8 ? 256 : 1];
  if (U8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
      lut[i] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)i, 255.f), 0.153f), 0.165f);
    __syncthreads();
  }
  const float* x = static_cast<const float*>(xin);
  const unsigned char* xu = static_cast<const unsigned char*>(xin);
  const int G = (W + 3) / 4;
  const long long total = (long long)B * D * H * G;
  const long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= total) return;
  const int w0 = (int)(gi % G) * 4;
  long long t = gi / G;
  const int ho = (int)(t % H);
  t /= H;
  const int d = (int)(t % D);
  const int b = (int)(t / D);
  float acc[4][32];
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int n = 0; n < 32; ++n) acc[p][n] = c_head_b[n];
  const size_t HW = (size_t)H * W;
#pragma unroll 1
  for (int kdh = 0; kdh < 9; ++kdh) {
    const int kd = kdh / 3, kh = kdh - kd * 3;
    const int di = d + kd - 1, hi = ho + kh - 1;
    if (di < 0 || di >= D || hi < 0 || hi >= H) continue;
    float xa[6], xb[6];
    if (U8) {
      const unsigned char* r0 = xu + (size_t)(b * (D + 1) + di) * HW + (size_t)hi * W;
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        const int wi = w0 - 1 + j;
        const bool ok = wi >= 0 && wi < W;
        xa[j] = ok ? lut[__ldg(r0 + wi)] : 0.f;
        xb[j] = ok ? lut[__ldg(r0 + HW + wi)] : 0.f;
      }
    } else {
      const float* r0 = x + ((size_t)(b * D + di) * 2) * HW + (size_t)hi * W;
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        const int wi = w0 - 1 + j;
        const bool ok = wi >= 0 && wi < W;
        xa[j] = ok ? __ldg(r0 + wi) : 0.f;
        xb[j] = ok ? __ldg(r0 + HW + wi) : 0.f;
      }
    }
    const float* wt = c_head_w + kdh * (3 * 64);
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
#pragma unroll
      for (int n = 0; n < 32; ++n) {
        const float wa = wt[kw * 64 + n], wb = wt[kw * 64 + 32 + n];
#pragma unroll
        for (int p = 0; p < 4; ++p) acc[p][n] = fmaf(xa[p + kw], wa, fmaf(xb[p + kw], wb, acc[p][n]));
      }
    }
  }
  const size_t m0 = ((size_t)(b * D + d) * H + ho) * W + w0;
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    if (w0 + p >= W) break;
    uint4 o[4];
    __nv_bfloat162* op = reinterpret_cast<__nv_bfloat162*>(o);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      float v0 = acc[p][2 * i], v1 = acc[p][2 * i + 1];
      v0 = v0 > 0.f ? v0 : 0.01f * v0;
      v1 = v1 > 0.f ? v1 : 0.01f * v1;
      op[i] = __floats2bfloat162_rn(v0, v1);
    }
    uint4* dst = reinterpret_cast<uint4*>(out + (m0 + p) * 32);
#pragma unroll
    for (int i = 0; i < 4; ++i) dst[i] = o[i];
  }
}

// ------------------------------------------------------------------------------------------
// head on the tensor pipe.  The 2-channel fp32 input becomes an 8-channel bf16 pixel
//     [x0h, x1h, x0l, x1l, x0h, x1h, 0, 0]        (xh = bf16(x), xl = bf16(x - xh))
// and the weights [w0h, w1h, w0h, w1h, w0l, w1l, 0, 0], so one K=16 MMA step per tap evaluates
// xh*wh + xl*wh + xh*wl: the fp32 product to ~2^-17, fp32 accumulation (the direct kernel above is pure fp32; both
// agree to ~1e-5 relative).  The 16-byte pixels are presented to conv_halo_kdm_kernel as overlapping 64-channel
// rows (make_patch_map); channels 8..15 of the single K step hold the next pixel and meet zero weights.
// ------------------------------------------------------------------------------------------
template <bool U8>
__global__ void __launch_bounds__(256) head_prep_kernel(const void* __restrict__ xin, int B, int D, int H, int W,
                                                         __nv_bfloat16* __restrict__ out) {
  __shared__ float lut[U8 ? 256 : 1];
  if (U8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
      lut[i] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)i, 255.f), 0.153f), 0.165f);
    __syncthreads();
  }
  const size_t HW = (size_t)H * W;
  const size_t total = (size_t)B * D * HW;
  // rows are stored with W+1 pixels, the last one zero: a patch row is [pixel p | pixel p+1], and the upper half carries
  // the kw = 2 tap of the pixel's right neighbour -- at the right image border that neighbour is the conv's zero padding
  const size_t rows = (size_t)B * D * H;
  // the K step of the last pixel reaches 16 bytes past the tensor: they meet zero weights but must be finite
  if (blockIdx.x == 0 && threadIdx.x < 8) reinterpret_cast<uint4*>(out)[rows * (W + 1) + threadIdx.x] = make_uint4(0u, 0u, 0u, 0u);
  for (size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (size_t)gridDim.x * blockDim.x)
    reinterpret_cast<uint4*>(out)[r * (W + 1) + W] = make_uint4(0u, 0u, 0u, 0u);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t pix = i % HW;
    const size_t pl = i / HW;                       // b*D + d
    float x0, x1;
    if (U8) {
      const unsigned char* xu = static_cast<const unsigned char*>(xin);
      const size_t b = pl / D, d = pl % D;
      const unsigned char* f0 = xu + (b * (D + 1) + d) * HW + pix;
      x0 = lut[__ldg(f0)];
      x1 = lut[__ldg(f0 + HW)];
    } else {
      const float* x = static_cast<const float*>(xin);
      x0 = __ldg(x + (pl * 2) * HW + pix);
      x1 = __ldg(x + (pl * 2 + 1) * HW + pix);
    }
    const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
    const __nv_bfloat16 l0 = __float2bfloat16_rn(x0 - __bfloat162float(h0)), l1 = __float2bfloat16_rn(x1 - __bfloat162float(h1));
    __nv_bfloat162 v[4];
    v[0] = __halves2bfloat162(h0, h1);
    v[1] = __halves2bfloat162(l0, l1);
    v[2] = __halves2bfloat162(h0, h1);
    v[3] = __floats2bfloat162_rn(0.f, 0.f);
    reinterpret_cast<uint4*>(out)[i + (pl * H + pix / W)] = *reinterpret_cast<const uint4*>(v);     // row pitch W+1
  }
}

// fp32 head weights (32, 2, 27) -> fp32 (32, 16, 27) holding exactly representable bf16 values.  Channels 0..7 of a
// tap are [w0h,w1h,w0h,w1h,w0l,w1l,0,0] of that tap.  A patch row is [pixel p | pixel p+1] (8 + 8 channels), so the
// K=16 step of tap (kh, kw=1) also carries tap (kh, kw=2) in channels 8..15: the kw = 2 taps become zero tiles that the
// kernel skips (HaloArgs::tap_mask) -- 6 MMA instructions per input slice instead of 9 for the warp that issues them.
// (Pairing kw = 1 with kw = 2, not kw = 0 with kw = 1: the row of tap kw = 0 of output column 0 lies left of the image and
// is zero-filled as a whole by TMA, upper half included; the right neighbour of the last column is the stored zero pixel.)
__global__ void head_split_weights_kernel(const float* __restrict__ w, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 32 * 16 * 27) return;
  const int tap = i % 27, c16 = (i / 27) % 16, n = i / (27 * 16);
  const int kw = tap % 3, c = c16 & 7;
  int src_tap = -1;
  if (c16 < 8) src_tap = (kw == 2) ? -1 : tap;              // kw = 0 and kw = 1 keep their own weights in the lower half
  else src_tap = (kw == 1) ? tap + 1 : -1;                  // upper half of kw = 1: the weights of kw = 2 (next pixel)
  float v = 0.f;
  if (src_tap >= 0 && c < 6) {
    const float wv = w[((size_t)n * 2 + (c & 1)) * 27 + src_tap];
    const float hi = __bfloat162float(__float2bfloat16_rn(wv));
    v = (c < 4) ? hi : __bfloat162float(__float2bfloat16_rn(wv - hi));
  }
  out[i] = v;
}

// The prediction layer (Conv3d 32->20, k1, bias, ReLU; v2ce_3d.py:29) is fused into the epilogue of
// decoders.3.conv2 (conv_halo.cuh / conv_halo_kdm.cuh, c_pred).

// ------------------------------------------------------------------------------------------
// Spectral norm: one power iteration per SN conv per forward (spectral_norm.py:19-31), fp32.
//   t = W^T u ; v = t/(|t|+eps) ; s = W v ; u = s/(|s|+eps) ; sigma = u . s
// ------------------------------------------------------------------------------------------
struct SnDesc {
  const float* W;   // (rows, K) row-major == weight_bar.view(height, -1)
  float* u;         // rows
  float* v;         // K
  float* t;         // K scratch
  float* s;         // rows scratch
  float* partial;   // ceil(K/32) partial sums of t^2
  int rows, K;
};

// Every sum below has a fixed order (no atomics): a rank that replays the steps of calls it does not own
// (v2ce_model_sn_advance) must reach bit-identical u, v and sigma.
// t = W^T u: one block per 32 columns, its 8 warps take the rows r = w, w+8, ... with eight loads in flight per lane
// (the first version walked all rows of a column in one thread: 151 MB of weights at 1.1 TB/s, 135 us per step, which
// is what a sharded clip's replay of the other ranks' calls costs per call).
constexpr int kSnCols = 32;
__global__ void __launch_bounds__(256) sn_wtu_kernel(const SnDesc* __restrict__ descs) {
  const SnDesc d = descs[blockIdx.y];
  if (blockIdx.x * kSnCols >= d.K) return;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int k = blockIdx.x * kSnCols + lane;
  __shared__ float part[8][kSnCols];
  float acc = 0.f;
  if (k < d.K) {
    const float* col = d.W + k;
    int r = w;
    for (; r + 56 < d.rows; r += 64) {
      float x[8], uu[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { x[j] = __ldg(col + (size_t)(r + 8 * j) * d.K); uu[j] = __ldg(d.u + r + 8 * j); }
#pragma unroll
      for (int j = 0; j < 8; ++j) acc = fmaf(x[j], uu[j], acc);
    }
    for (; r < d.rows; r += 8) acc = fmaf(__ldg(col + (size_t)r * d.K), __ldg(d.u + r), acc);
  }
  part[w][lane] = acc;
  __syncthreads();
  if (w == 0) {
    float tk = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) tk += part[j][lane];
    if (k < d.K) d.t[k] = tk;
    float sq = (k < d.K) ? tk * tk : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if (lane == 0) d.partial[blockIdx.x] = sq;
  }
}

__global__ void __launch_bounds__(256) sn_norm_v_kernel(const SnDesc* __restrict__ descs) {
  const SnDesc d = descs[blockIdx.x];
  __shared__ float red[256];
  const int nb = (d.K + kSnCols - 1) / kSnCols;
  float s = 0.f;
  for (int i = threadIdx.x; i < nb; i += 256) s += d.partial[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  const float nrm = sqrtf(red[0]) + 1e-12f;
  for (int k = threadIdx.x; k < d.K; k += 256) d.v[k] = d.t[k] / nrm;
}

// s = W v: one warp per row, 16-byte loads (K = Cin * 27 with Cin a multiple of 4), two of them in flight per lane
__global__ void __launch_bounds__(256) sn_wv_kernel(const SnDesc* __restrict__ descs) {
  const SnDesc d = descs[blockIdx.y];
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= d.rows) return;
  const int lane = threadIdx.x & 31;
  float acc = 0.f;
  if ((d.K & 3) == 0) {
    const float4* wr = reinterpret_cast<const float4*>(d.W + (size_t)row * d.K);
    const float4* vv = reinterpret_cast<const float4*>(d.v);
    const int n4 = d.K >> 2;
    float a0 = 0.f, a1 = 0.f;
    int q = lane;
    for (; q + 32 < n4; q += 64) {
      const float4 x0 = __ldg(wr + q), x1 = __ldg(wr + q + 32);
      const float4 y0 = vv[q], y1 = vv[q + 32];
      a0 = fmaf(x0.x, y0.x, a0); a0 = fmaf(x0.y, y0.y, a0); a0 = fmaf(x0.z, y0.z, a0); a0 = fmaf(x0.w, y0.w, a0);
      a1 = fmaf(x1.x, y1.x, a1); a1 = fmaf(x1.y, y1.y, a1); a1 = fmaf(x1.z, y1.z, a1); a1 = fmaf(x1.w, y1.w, a1);
    }
    if (q < n4) {
      const float4 x0 = __ldg(wr + q);
      const float4 y0 = vv[q];
      a0 = fmaf(x0.x, y0.x, a0); a0 = fmaf(x0.y, y0.y, a0); a0 = fmaf(x0.z, y0.z, a0); a0 = fmaf(x0.w, y0.w, a0);
    }
    acc = a0 + a1;
  } else {
    for (int k = lane; k < d.K; k += 32) acc = fmaf(__ldg(d.W + (size_t)row * d.K + k), d.v[k], acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) d.s[row] = acc;
}

__global__ void __launch_bounds__(256) sn_finish_kernel(const SnDesc* __restrict__ descs, float* __restrict__ sigma,
                                                         float* __restrict__ inv_sigma) {
  const SnDesc d = descs[blockIdx.x];
  __shared__ float red[256];
  float sq = 0.f;
  for (int r = threadIdx.x; r < d.rows; r += 256) sq += d.s[r] * d.s[r];
  red[threadIdx.x] = sq;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  const float nrm = sqrtf(red[0]) + 1e-12f;
  __syncthreads();
  float dot = 0.f;
  for (int r = threadIdx.x; r < d.rows; r += 256) {
    const float un = d.s[r] / nrm;
    d.u[r] = un;
    dot += un * d.s[r];
  }
  red[threadIdx.x] = dot;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    sigma[blockIdx.x] = red[0];
    inv_sigma[blockIdx.x] = 1.f / red[0];
  }
}

// ------------------------------------------------------------------------------------------
// model
// ------------------------------------------------------------------------------------------
// Which kernel runs a layer and how its (virtual-concat) input channels are laid out in memory.  Every activation
// is stored densely: its channel pitch is its channel count.  32-channel tensors (64 B per pixel) are presented by
// their TMA maps as 64-channel rows whose upper half is the NEXT pixel (conv_halo.cuh make_patch_map), which the
// kernels never multiply (K=16 steps beyond the real channels are skipped); the packed weights carry zeros there.
enum class Kernel {
  Direct,                   // fp32 on CUDA cores (head, pred)
  Gather,                   // gather implicit GEMM (conv_igemm.cuh)
  Halo,                     // halo tiles (conv_halo.cuh, or conv_halo_kdm.cuh when packed for it)
};

struct LayerCfg {
  Kernel kernel;
  int pad0, real0, pad1, real1;   // channels per source in the packed K dimension (pad) and how many are real
};

// K-chunk padding: the halo kernels multiply 64-channel chunks (one 128-byte swizzle row per pixel)
static inline int chunk_of(int c) { return c < 64 ? 64 : c; }

struct DevLayer {
  LayerCfg cfg{Kernel::Direct, 0, 0, 0, 0};
  __nv_bfloat16* wpack = nullptr;
  __nv_bfloat16* wpack_kdm = nullptr;   // depth-merged packing (conv_halo_kdm.cuh) for halo layers with Cout <= 64
  float* scale = nullptr;
  float* shift = nullptr;
  const float* inv_sigma = nullptr;     // spectral-norm layers: 1 / sigma on the device
  float* w32 = nullptr;     // head / pred fp32 weights, SN weight_bar
  float* bias = nullptr;    // head / pred bias
  int bn_tile = 0, num_kb = 0;
};

// The TMA views a halo launch reads its sources through: 64-channel patch rows (halo::make_patch_map), the head's
// split pixels as 16-channel rows (make_patch_map16) or one of the four parity views of a stride-2 input
// (make_parity_map).
enum class View { Patch64, Head16, Parity };

struct MapKey {
  View view;
  int q;                    // Parity: row parity * 2 + column parity
  const void* ptr;
  int B, D, H, W, cpitch;   // the tensor (B, D, H, W, cpitch)
  int PW, rows;             // the box: PW pixels by `rows` rows
  bool operator<(const MapKey& o) const {
    return std::tie(view, q, ptr, B, D, H, W, cpitch, PW, rows) <
           std::tie(o.view, o.q, o.ptr, o.B, o.D, o.H, o.W, o.cpitch, o.PW, o.rows);
  }
};

}  // namespace unet
}  // namespace v2ce

struct v2ce_model {
  int device = 0;
  unsigned long long uid = 0;           // unique per handle (constant-memory ownership)
  bool finalized = false;
  std::map<std::string, std::vector<float>> host;
  std::map<std::string, std::vector<int64_t>> shapes;
  v2ce::unet::DevLayer layers[v2ce::unet::kNumLayers];
  std::vector<void*> allocs;
  v2ce::unet::SnDesc* sn_descs_dev = nullptr;
  v2ce::unet::SnDesc sn_descs_host[v2ce::unet::kNumSn];
  float* sigma_dev = nullptr;
  float* inv_sigma_dev = nullptr;
  float* head_wpack = nullptr;          // head weights as [tap][cin][cout] (constant-memory image)
  int* error_flag_dev = nullptr;
  int max_rows = 0, max_k = 0;
  int64_t calls = 0;
  int last_launches = 0;
  int layer_timing = 0;                 // option "layer_timing": CUDA events around every launch of forward()
  int stop_after = -1;                  // option "stop_after" (per-layer tests): kLayers index, -1 = run the whole forward
  std::vector<std::pair<std::string, cudaEvent_t>> marks;
  cudaStream_t sn_stream = nullptr;     // the spectral-norm step overlaps the head / encoder convs
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev_side[16] = {nullptr};  // x-ready / shortcut-done pairs of the blocks whose shortcut runs on the side stream
  std::map<v2ce::unet::MapKey, CUtensorMap> tmaps;
};

namespace v2ce {
namespace unet {

template <typename T>
static int dev_alloc(v2ce_model* m, T** p, size_t count) {
  void* q = nullptr;
  V2CE_CUDA_CHECK(cudaMalloc(&q, count * sizeof(T)));
  m->allocs.push_back(q);
  *p = static_cast<T*>(q);
  return V2CE_OK;
}

static int upload(v2ce_model* m, float** dst, const std::vector<float>& v) {
  if (int e = dev_alloc(m, dst, v.size())) return e;
  V2CE_CUDA_CHECK(cudaMemcpy(*dst, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return V2CE_OK;
}

static const std::vector<float>* find(const v2ce_model* m, const std::string& key) {
  auto it = m->host.find(key);
  return it == m->host.end() ? nullptr : &it->second;
}

static bool known_name(const std::string& name) {
  for (int i = 0; i < kNumLayers; ++i) {
    const LayerSpec& L = kLayers[i];
    const std::string base = L.name;
    if (L.sn) {
      if (name == base + ".module.weight_bar" || name == base + ".module.weight_u" || name == base + ".module.weight_v")
        return true;
    } else {
      if (name == base + ".weight") return true;
      if (L.bias && name == base + ".bias") return true;
    }
    if (L.bn) {
      const std::string bn = L.bn;
      if (name == bn + ".weight" || name == bn + ".bias" || name == bn + ".running_mean" || name == bn + ".running_var")
        return true;
    }
  }
  return false;
}

constexpr int kSnLaunches = 4;   // kernels of one run_sn_step
static int run_sn_step(v2ce_model* m, cudaStream_t s) {
  dim3 g1((m->max_k + kSnCols - 1) / kSnCols, kNumSn);
  sn_wtu_kernel<<<g1, 256, 0, s>>>(m->sn_descs_dev);
  V2CE_LAUNCH_CHECK("sn_wtu_kernel");
  sn_norm_v_kernel<<<kNumSn, 256, 0, s>>>(m->sn_descs_dev);
  V2CE_LAUNCH_CHECK("sn_norm_v_kernel");
  dim3 g3((m->max_rows + 7) / 8, kNumSn);
  sn_wv_kernel<<<g3, 256, 0, s>>>(m->sn_descs_dev);
  V2CE_LAUNCH_CHECK("sn_wv_kernel");
  sn_finish_kernel<<<kNumSn, 256, 0, s>>>(m->sn_descs_dev, m->sigma_dev, m->inv_sigma_dev);
  V2CE_LAUNCH_CHECK("sn_finish_kernel");
  m->calls += 1;
  return V2CE_OK;
}

struct Dims {
  int H[5], W[5];
  long long M[5];
};

static Dims make_dims(int B, int D, int H, int W) {
  Dims d;
  d.H[0] = H; d.W[0] = W;
  for (int i = 1; i < 5; ++i) { d.H[i] = (d.H[i - 1] - 1) / 2 + 1; d.W[i] = (d.W[i - 1] - 1) / 2 + 1; }
  for (int i = 0; i < 5; ++i) d.M[i] = (long long)B * D * d.H[i] * d.W[i];
  return d;
}

struct Buffers {
  __nv_bfloat16 *head_in, *head, *enc[4], *res[2], *dec[4], *tmp_t, *tmp_r, *up, *up2;
  size_t bytes;
};

static Buffers carve(void* ws, const Dims& d) {
  Arena a(ws, (size_t)-1);
  Buffers b;
  static const int ch[5] = {32, 64, 128, 256, 512};
  b.head_in = a.take<__nv_bfloat16>(((size_t)d.M[0] + (size_t)d.M[0] / d.W[0] + 8) * 8 + 64);   // split-bf16 input pixels, rows of W+1 (last one zero)
  b.head = a.take<__nv_bfloat16>((size_t)d.M[0] * 32 + 64);  // 32 channels (+ the overlapped TMA view's reach)
  for (int i = 0; i < 4; ++i) b.enc[i] = a.take<__nv_bfloat16>((size_t)d.M[i + 1] * ch[i + 1]);
  for (int i = 0; i < 2; ++i) b.res[i] = a.take<__nv_bfloat16>((size_t)d.M[4] * 512);
  for (int i = 0; i < 4; ++i) b.dec[i] = a.take<__nv_bfloat16>((size_t)d.M[3 - i] * ch[3 - i]);
  size_t tmax = 0, umax = 0;
  for (int i = 0; i < 5; ++i) tmax = tmax > (size_t)d.M[i] * ch[i] ? tmax : (size_t)d.M[i] * ch[i];
  for (int i = 0; i < 4; ++i) umax = umax > (size_t)d.M[i] * ch[i + 1] ? umax : (size_t)d.M[i] * ch[i + 1];
  b.tmp_t = a.take<__nv_bfloat16>(tmax);
  b.tmp_r = a.take<__nv_bfloat16>(tmax);
  b.up = a.take<__nv_bfloat16>(umax);                                  // nearest-upsampled decoder inputs (written by the
  b.up2 = a.take<__nv_bfloat16>(umax);                                 // producing layer's epilogue), double-buffered
  b.bytes = align_up(a.off, 256);
  return b;
}

// kLayers index of the conv1 of block `block` with role r; the block's conv2 and shortcut follow it
static int conv1_of(Role r, int block) {
  for (int i = 0; i < kNumLayers; ++i)
    if (kLayers[i].role == r && kLayers[i].block == block) return i;
  return -1;
}

// kernel choice and channel padding per layer (see LayerCfg)
static LayerCfg layer_cfg(const LayerSpec& L) {
  if (L.role == Role::Head || L.role == Role::Pred) return LayerCfg{Kernel::Direct, 0, 0, 0, 0};
  // encoder conv1 (stride 2) and the shortcuts run on the gather kernel
  const bool halo = L.role == Role::Conv2 || L.role == Role::ResConv1 || L.role == Role::DecConv1;
  // conv1 / shortcut of a decoder read [up (2/3 of Cin) | skip (1/3)]
  const bool split = L.role == Role::DecConv1 || L.role == Role::DecShort;
  LayerCfg c{halo ? Kernel::Halo : Kernel::Gather, 0, split ? L.cin / 3 * 2 : L.cin, 0, split ? L.cin / 3 : 0};
  // the halo kernel multiplies whole 64-channel TMA rows (padding channels carry zero weights and are skipped
  // at K=16 granularity); the gather kernel addresses real channels through the pitch
  c.pad0 = halo ? chunk_of(c.real0) : c.real0;
  c.pad1 = halo && c.real1 ? chunk_of(c.real1) : c.real1;
  return c;
}

static int make_map(const MapKey& k, CUtensorMap* tm) {
  switch (k.view) {
    case View::Patch64: return halo::make_patch_map(tm, k.ptr, k.B, k.D, k.H, k.W, k.cpitch, k.PW, k.rows);
    case View::Head16: return halo::make_patch_map16(tm, k.ptr, k.B, k.D, k.H, k.W, k.PW, k.rows);
    case View::Parity:
      return halo::make_parity_map(tm, k.ptr, k.B, k.D, k.H, k.W, k.cpitch, k.q >> 1, k.q & 1, k.PW, k.rows);
  }
  return set_error(V2CE_ERR_STATE, "unknown tensor-map view %d", (int)k.view);
}

// make_map, cached per handle.  The map is returned by value: clearing the cache invalidates nothing a caller holds.
static int get_tmap(v2ce_model* m, const MapKey& key, CUtensorMap* out) {
  auto it = m->tmaps.find(key);
  if (it == m->tmaps.end()) {
    if (m->tmaps.size() > 512) m->tmaps.clear();      // callers that move their workspace every call must not grow the cache
    CUtensorMap tm;
    if (int e = make_map(key, &tm)) return e;
    it = m->tmaps.emplace(key, tm).first;
  }
  *out = it->second;
  return V2CE_OK;
}

// __constant__ memory is per device, not per handle: `load` (stream ordered) runs when another handle loaded this
// image on the device last
template <typename Load>
static int load_constants(unsigned long long (&owner)[64], const v2ce_model* m, Load load) {
  unsigned long long& o = owner[m->device & 63];
  if (o == m->uid) return V2CE_OK;
  if (int e = load()) return e;
  o = m->uid;
  return V2CE_OK;
}

// The one place that fills conv::ConvArgs: a gather implicit-GEMM launch (stride-2 convs, 1x1x1 shortcuts) of the
// k x k x k layer `dl` with cout outputs; p0 / p1 are the channel PITCHES of the sources
static ConvArgs conv_args(const DevLayer& dl, int k, int cout, const __nv_bfloat16* src0, int p0, int h0, int w0,
                          const __nv_bfloat16* src1, int p1, int B, int D, int hin, int win, int stride,
                          const __nv_bfloat16* residual, int act, __nv_bfloat16* out, int* error_flag) {
  ConvArgs a;
  a.src0 = src0; a.src1 = src1; a.C0 = dl.cfg.real0; a.C1 = dl.cfg.real1; a.Cin = a.C0 + a.C1;
  a.P0 = p0; a.P1 = p1;
  a.H0 = h0; a.W0 = w0; a.B = B; a.D = D; a.Hin = hin; a.Win = win;
  a.stride = stride; a.ksize = k; a.pad = k / 2;
  a.Hout = (hin + 2 * a.pad - k) / stride + 1;
  a.Wout = (win + 2 * a.pad - k) / stride + 1;
  a.taps = k * k * k;
  a.num_kb = dl.num_kb;
  a.M = B * D * a.Hout * a.Wout;
  a.Cout = cout;
  a.wpack = dl.wpack; a.scale = dl.scale; a.shift = dl.shift; a.inv_sigma = dl.inv_sigma;
  a.residual = residual; a.out = out; a.act = act;
  a.error_flag = error_flag;
  return a;
}

// The one place that fills halo::HaloArgs: a launch of layer `dl` over the output plane (B, D, H, W) with cout outputs,
// reading its sources through `view`.  With the depth-merged plan `kp` it runs conv_halo_kdm.cuh, otherwise
// conv_halo.cuh with the plan `hp`.  The Head16 view carries the head's 8-channel split pixels (head_prep_kernel).
static halo::HaloArgs halo_args(const DevLayer& dl, View view, const halo::HaloPlan* hp, const halo::KdmPlan* kp, int B,
                                int D, int H, int W, int cout, __nv_bfloat16* out, int out_pitch,
                                const __nv_bfloat16* residual, int res_pitch, int act, int* error_flag, int up_H = 0,
                                int up_W = 0, const DevLayer* pred = nullptr, float* pred_out = nullptr) {
  const bool head = view == View::Head16;
  const halo::TileShape ts = kp ? kp->ts : hp->ts;
  halo::HaloArgs a;
  // 64-channel SWIZZLE_128B patch rows, or the head's K-major SWIZZLE_32B rows (8-row groups 256 B apart) with the
  // taps (kh, 0) and (kh, 1) only: the kw = 2 weights ride in the upper half of kw = 1 (head_split_weights_kernel)
  a.a_row16 = head ? 2 : 8;
  a.a_desc_hi = head ? 0xC0004010u : 0x40004040u;
  a.tap_mask = head ? 0x0DB : 0x1FF;
  a.B = B; a.D = D; a.H = H; a.W = W;
  a.PW = ts.PW; a.TH = ts.TH; a.TW = kp ? kp->TW : ts.PW - 2;
  a.tiles_w = (W + a.TW - 1) / a.TW;
  a.tiles_h = (H + a.TH - 1) / a.TH;
  a.real0 = head ? 8 : dl.cfg.real0; a.real1 = dl.cfg.real1;
  a.ncc0 = chunk_of(a.real0) / 64; a.ncc1 = a.real1 ? chunk_of(a.real1) / 64 : 0;
  a.Cout = cout; a.out_pitch = out_pitch; a.res_pitch = res_pitch;
  a.T = kp ? halo::kKdmT : hp->T;
  a.SA = kp ? kp->SA : hp->SA;
  a.SB = kp ? 9 : hp->SB;
  a.a_stage_bytes = kp ? kp->a_stage_bytes : hp->a_stage_bytes;
  a.box_bytes = kp ? kp->box_bytes : hp->box_bytes;
  a.wpack = kp ? dl.wpack_kdm : dl.wpack; a.scale = dl.scale; a.shift = dl.shift; a.inv_sigma = dl.inv_sigma;
  a.residual = residual; a.out = out; a.act = act;
  a.up_H = up_H; a.up_W = up_W;
  a.pred_w = pred ? pred->w32 : nullptr;
  a.pred_b = pred ? pred->bias : nullptr;
  a.pred_out = pred_out;
  a.error_flag = error_flag;
  return a;
}

// gather implicit-GEMM launch of layer `li` (stride-2 convs, 1x1x1 shortcuts); c0/c1 are channel PITCHES
static int run_conv(v2ce_model* m, int li, const __nv_bfloat16* src0, int c0, int h0, int w0, const __nv_bfloat16* src1,
                    int c1, int B, int D, int hin, int win, int stride, const __nv_bfloat16* residual, int act,
                    __nv_bfloat16* out, cudaStream_t s) {
  const LayerSpec& L = kLayers[li];
  const DevLayer& dl = m->layers[li];
  if (dl.cfg.kernel != Kernel::Gather || c0 != dl.cfg.real0 || c1 != dl.cfg.real1)
    return set_error(V2CE_ERR_STATE, "layer %s: gather launch with pitches %d+%d, expected %d+%d", L.name, c0, c1,
                     dl.cfg.real0, dl.cfg.real1);
  return conv::launch_conv(conv_args(dl, L.k, L.cout, src0, c0, h0, w0, src1, c1, B, D, hin, win, stride, residual, act,
                                     out, m->error_flag_dev),
                           dl.bn_tile, s);
}

// halo-tile launch of layer `li` (3x3x3, stride 1); sources are full-resolution (B,D,H,W,pitch) tensors
static int run_halo(v2ce_model* m, int li, const __nv_bfloat16* src0, int p0, const __nv_bfloat16* src1, int p1, int B, int D,
                    int H, int W, const __nv_bfloat16* residual, int res_pitch, int act, __nv_bfloat16* out, int out_pitch,
                    cudaStream_t s, int up_H = 0, int up_W = 0, float* pred_out = nullptr, int short_li = -1,
                    __nv_bfloat16* short_out = nullptr, int short_pitch = 0, bool* short_done = nullptr) {
  const LayerSpec& L = kLayers[li];
  const DevLayer& dl = m->layers[li];
  if (dl.cfg.kernel != Kernel::Halo || p0 != dl.cfg.real0 || p1 != dl.cfg.real1)
    return set_error(V2CE_ERR_STATE, "layer %s: halo launch with pitches %d+%d, expected %d+%d", L.name, p0, p1,
                     dl.cfg.real0, dl.cfg.real1);
  const halo::HaloPlan plan = halo::plan_for(dl.bn_tile, D, H, W);
  // layers with few output channels: depth taps merged into the MMA N dimension (conv_halo_kdm.cuh)
  const halo::KdmPlan kplan = halo::plan_kdm(D, H, W);
  const bool kdm = dl.wpack_kdm != nullptr && kplan.ok;     // packed for Cout <= 64 (pack_layer)
  const DevLayer& pred = m->layers[kNumLayers - 1];
  const halo::HaloArgs a = halo_args(dl, View::Patch64, &plan, kdm ? &kplan : nullptr, B, D, H, W, L.cout, out, out_pitch,
                                     residual, res_pitch, act, m->error_flag_dev, up_H, up_W, pred_out ? &pred : nullptr,
                                     pred_out);
  if (pred_out) {
    static unsigned long long pred_owner[64] = {0};
    if (int e = load_constants(pred_owner, m, [&] { return halo::load_pred_constants(pred.w32, pred.bias, s); })) return e;
  }
  CUtensorMap tm0, tm1;
  if (int e = get_tmap(m, MapKey{View::Patch64, 0, src0, B, D, H, W, p0, a.PW, a.TH + 2}, &tm0)) return e;
  tm1 = tm0;
  if (src1)
    if (int e = get_tmap(m, MapKey{View::Patch64, 0, src1, B, D, H, W, p1, a.PW, a.TH + 2}, &tm1)) return e;
  if (short_done) *short_done = false;
  if (kdm) {
    // fuse the block's 1x1x1 shortcut conv (layer short_li) when asked for and packed
    if (short_li >= 0 && m->layers[short_li].wpack_kdm != nullptr) {
      const DevLayer& sl = m->layers[short_li];
      halo::KdmShort sc{sl.wpack_kdm, sl.scale, sl.shift, short_out, short_pitch};
      if (short_done) *short_done = true;
      return halo::launch_halo_kdm(tm0, tm1, a, &sc, kplan.smem_bytes, s);
    }
    return halo::launch_halo_kdm(tm0, tm1, a, nullptr, kplan.smem_bytes, s);
  }
  return halo::launch_halo(tm0, tm1, a, dl.bn_tile, plan.smem_bytes, s);
}

// stride-(1,2,2) first conv of encoder block `li` with the block's stride-2 1x1x1 shortcut (layer li+2) fused:
// x (B,D,Hin,Win,pin) -> out (B,D,Hout,Wout,Cout) [ReLU(bn1(conv1))] and short_out [bn_d(conv_d)].  Returns false in
// *done when the depth-merged kernel does not apply (the caller then runs the two gather launches).
static int run_enc_kdm(v2ce_model* m, int li, const __nv_bfloat16* x, int pin, int B, int D, int Hin, int Win,
                       __nv_bfloat16* out, __nv_bfloat16* short_out, cudaStream_t s, bool* done) {
  const LayerSpec& L = kLayers[li];
  const DevLayer& dl = m->layers[li];
  const DevLayer& sl = m->layers[li + 2];
  *done = false;
  const int Hout = (Hin - 1) / 2 + 1, Wout = (Win - 1) / 2 + 1;
  const halo::KdmPlan kp = halo::plan_kdm(D, Hout, Wout, 2);
  if (!kp.ok || dl.wpack_kdm == nullptr || sl.wpack_kdm == nullptr || Hin < 2 || Win < 2) return V2CE_OK;
  const halo::HaloArgs a = halo_args(dl, View::Parity, nullptr, &kp, B, D, Hout, Wout, L.cout, out, L.cout, nullptr, 0, 1,
                                     m->error_flag_dev);
  halo::ParityMaps pm;
  for (int q = 0; q < 4; ++q)
    if (int e = get_tmap(m, MapKey{View::Parity, q, x, B, D, Hin, Win, pin, a.PW, a.TH + 1}, &pm.m[q])) return e;
  halo::KdmShort sc{sl.wpack_kdm, sl.scale, sl.shift, short_out, L.cout};
  *done = true;
  return halo::launch_halo_kdm(pm.m[0], pm.m[0], a, &sc, kp.smem_bytes, s, &pm);
}

static int pack_layer(v2ce_model* m, int li, const float* w_dev, cudaStream_t s) {
  const LayerSpec& L = kLayers[li];
  DevLayer& dl = m->layers[li];
  const LayerCfg c = layer_cfg(L);
  dl.cfg = c;
  const int taps = L.k * L.k * L.k;
  const int cin_pad = c.pad0 + c.pad1;
  dl.bn_tile = conv::pick_bn(L.cout);
  if (c.kernel == Kernel::Halo && L.cout == 256) {
    // N tile of the 256- / 512-channel halo layers.  256-channel layers run as two N = 128 tiles: at 33 x 44 x 16 x 4
    // an N = 256 launch has 448 items = 3.03 waves of 148 CTAs (a quarter of the last wave's time is 4 items), the
    // N = 128 launch has 896 half-size items = 6.05 waves (3.5 full-item times) and a double-buffered accumulator, so
    // the epilogue overlaps the next item: encoders.2.conv2 0.326 -> 0.268 ms, decoders.0.conv1 0.823 -> 0.753,
    // decoders.0.conv2 0.381 -> 0.278 (profiles/layer_times_r2_l_*.txt).  512-channel layers (256 items = 1.73 waves
    // either way) gain nothing and stay at 256.
    dl.bn_tile = 128;
  }
  if (c.real0 + c.real1 != L.cin) return set_error(V2CE_ERR_STATE, "layer %s: channel split mismatch", L.name);
  if (c.kernel == Kernel::Halo) {
    const size_t n = (size_t)L.cout * 27 * cin_pad;
    dl.num_kb = 27 * cin_pad / conv::kBlockK;
    if (int e = dev_alloc(m, &dl.wpack, n)) return e;
    halo::pack_weights_halo_kernel<<<(int)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(
        w_dev, L.cout, L.cin, dl.bn_tile, c.pad0, c.real0, c.pad1, c.real1, dl.wpack);
    V2CE_LAUNCH_CHECK("pack_weights_halo_kernel");
    if (L.cout <= 64) {
      if (int e = dev_alloc(m, &dl.wpack_kdm, n)) return e;
      halo::pack_weights_kdm_kernel<<<(int)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(
          w_dev, L.cout, L.cin, c.pad0, c.real0, c.pad1, c.real1, dl.wpack_kdm);
      V2CE_LAUNCH_CHECK("pack_weights_kdm_kernel");
    }
    return V2CE_OK;
  }
  if (L.role == Role::EncConv1) {
    // stride-2 first conv of an encoder block: depth-merged packing for the parity-view kernel (conv_halo_kdm.cuh, S = 2)
    const size_t nk = (size_t)L.cout * 27 * chunk_of(c.real0);
    if (int e = dev_alloc(m, &dl.wpack_kdm, nk)) return e;
    halo::pack_weights_kdm_kernel<<<(int)((nk + 255) / 256 > 4096 ? 4096 : (nk + 255) / 256), 256, 0, s>>>(
        w_dev, L.cout, L.cin, chunk_of(c.real0), c.real0, 0, 0, dl.wpack_kdm);
    V2CE_LAUNCH_CHECK("pack_weights_kdm_kernel");
  }
  if (L.role == Role::EncShort || (L.role == Role::DecShort && L.cout <= 64)) {
    // the shortcut of an encoder or decoder block can ride in its conv1 launch (conv_halo_kdm.cuh): [Cout/32][cc][32][64]
    const int k0 = chunk_of(c.real0), k1 = c.real1 ? chunk_of(c.real1) : 0;
    const size_t ns = (size_t)L.cout * (k0 + k1);
    if (int e = dev_alloc(m, &dl.wpack_kdm, ns)) return e;
    halo::pack_weights_kdm_short_kernel<<<(int)((ns + 255) / 256), 256, 0, s>>>(w_dev, L.cout, L.cin, k0, c.real0, k1, c.real1,
                                                                                dl.wpack_kdm);
    V2CE_LAUNCH_CHECK("pack_weights_kdm_short_kernel");
  }
  dl.num_kb = (taps * cin_pad + conv::kBlockK - 1) / conv::kBlockK;
  const size_t n = (size_t)L.cout * dl.num_kb * conv::kBlockK;
  if (int e = dev_alloc(m, &dl.wpack, n)) return e;
  conv::pack_weights_kernel<<<(int)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(
      w_dev, L.cout, L.cin, taps, dl.bn_tile, dl.num_kb, c.pad0, c.real0, c.pad1, c.real1, dl.wpack);
  V2CE_LAUNCH_CHECK("pack_weights_kernel");
  return V2CE_OK;
}

}  // namespace unet
}  // namespace v2ce

using namespace v2ce;
using namespace v2ce::unet;

extern "C" int v2ce_model_create(v2ce_model** out, int device) {
  V2CE_REQUIRE(out != nullptr, "out is NULL");
  if (int e = v2ce_device_check(device, nullptr, nullptr, nullptr)) return e;
  static unsigned long long next_uid = 0;
  v2ce_model* m = new v2ce_model();
  m->device = device;
  m->uid = ++next_uid;
  *out = m;
  return V2CE_OK;
}

extern "C" int v2ce_model_destroy(v2ce_model* m) {
  if (!m) return V2CE_OK;
  for (void* p : m->allocs) cudaFree(p);
  for (auto& mk : m->marks) cudaEventDestroy(mk.second);
  if (m->ev_fork) cudaEventDestroy(m->ev_fork);
  if (m->ev_join) cudaEventDestroy(m->ev_join);
  for (auto ev : m->ev_side) if (ev) cudaEventDestroy(ev);
  if (m->sn_stream) cudaStreamDestroy(m->sn_stream);
  delete m;
  return V2CE_OK;
}

extern "C" int v2ce_model_set_tensor(v2ce_model* m, const char* name, const float* data_host, const int64_t* shape,
                                     int32_t ndim) {
  V2CE_REQUIRE(m && name && data_host && (shape || ndim == 0), "NULL argument");
  V2CE_REQUIRE(!m->finalized, "model already finalized");
  const std::string key = name;
  if (!known_name(key)) return set_error(V2CE_ERR_INVALID, "unknown state_dict entry '%s'", name);
  size_t n = 1;
  std::vector<int64_t> shp;
  for (int i = 0; i < ndim; ++i) { n *= (size_t)shape[i]; shp.push_back(shape[i]); }
  m->host[key] = std::vector<float>(data_host, data_host + n);
  m->shapes[key] = shp;
  return V2CE_OK;
}

extern "C" int v2ce_model_finalize(v2ce_model* m) {
  V2CE_REQUIRE(m != nullptr, "model is NULL");
  V2CE_REQUIRE(!m->finalized, "model already finalized");
  V2CE_CUDA_CHECK(cudaSetDevice(m->device));
  cudaStream_t s = 0;
  if (int e = dev_alloc(m, &m->sigma_dev, kNumSn)) return e;
  if (int e = dev_alloc(m, &m->inv_sigma_dev, kNumSn)) return e;
  if (int e = dev_alloc(m, &m->error_flag_dev, 1)) return e;
  V2CE_CUDA_CHECK(cudaMemset(m->error_flag_dev, 0, sizeof(int)));
  V2CE_CUDA_CHECK(cudaStreamCreateWithFlags(&m->sn_stream, cudaStreamNonBlocking));
  V2CE_CUDA_CHECK(cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming));
  V2CE_CUDA_CHECK(cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming));
  for (auto& ev : m->ev_side) V2CE_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  int sn_count = 0;
  for (int li = 0; li < kNumLayers; ++li) {
    const LayerSpec& L = kLayers[li];
    DevLayer& dl = m->layers[li];
    const std::string base = L.name;
    const int taps = L.k * L.k * L.k;
    const size_t wn = (size_t)L.cout * L.cin * taps;
    const std::vector<float>* w = find(m, base + (L.sn ? ".module.weight_bar" : ".weight"));
    if (!w || w->size() != wn) return set_error(V2CE_ERR_STATE, "missing or mis-sized weight for %s", L.name);
    if (int e = upload(m, &dl.w32, *w)) return e;
    const std::vector<float>* bias = L.bias ? find(m, base + ".bias") : nullptr;
    if (L.bias && (!bias || (int)bias->size() != L.cout)) return set_error(V2CE_ERR_STATE, "missing bias for %s", L.name);
    if (layer_cfg(L).kernel == Kernel::Direct) {   // head and pred run on CUDA cores in fp32
      if (int e = upload(m, &dl.bias, *bias)) return e;
      if (L.role == Role::Head) {
        if (int e = dev_alloc(m, &m->head_wpack, (size_t)27 * 2 * 32)) return e;
        pack_head_kernel<<<(27 * 2 * 32 + 255) / 256, 256, 0, s>>>(dl.w32, m->head_wpack);
        V2CE_LAUNCH_CHECK("pack_head_kernel");
        // tensor-pipe variant: split weights in the depth-merged packing, unit scale, bias as shift
        float* w8 = nullptr;
        if (int e = dev_alloc(m, &w8, (size_t)32 * 16 * 27)) return e;
        head_split_weights_kernel<<<(32 * 16 * 27 + 255) / 256, 256, 0, s>>>(dl.w32, w8);
        V2CE_LAUNCH_CHECK("head_split_weights_kernel");
        if (int e = dev_alloc(m, &dl.wpack_kdm, (size_t)32 * 27 * 64)) return e;
        halo::pack_weights_kdm_kernel<<<(32 * 27 * 64 + 255) / 256, 256, 0, s>>>(w8, 32, 16, 64, 16, 0, 0, dl.wpack_kdm);
        V2CE_LAUNCH_CHECK("pack_weights_kdm_kernel");
        if (int e = upload(m, &dl.scale, std::vector<float>(32, 1.f))) return e;
        dl.shift = dl.bias;
      }
      continue;
    }
    // eval-mode BatchNorm folded into y = acc*scale + shift (scale *= 1/sigma at run time for SN convs)
    std::vector<float> scale(L.cout, 1.f), shift(L.cout, 0.f);
    if (L.bn) {
      const std::string bn = L.bn;
      const std::vector<float>*g = find(m, bn + ".weight"), *b = find(m, bn + ".bias"), *mu = find(m, bn + ".running_mean"),
                              *var = find(m, bn + ".running_var");
      if (!g || !b || !mu || !var || (int)g->size() != L.cout || (int)b->size() != L.cout ||
          (int)mu->size() != L.cout || (int)var->size() != L.cout)
        return set_error(V2CE_ERR_STATE, "missing or mis-sized BatchNorm tensors %s.* (expected %d channels)", L.bn, L.cout);
      for (int c = 0; c < L.cout; ++c) {
        const float sc = (*g)[c] / sqrtf((*var)[c] + kBnEps);
        scale[c] = sc;
        shift[c] = (*b)[c] - (*mu)[c] * sc + (bias ? (*bias)[c] * sc : 0.f);
      }
    } else if (bias) {
      for (int c = 0; c < L.cout; ++c) shift[c] = (*bias)[c];
    }
    if (int e = upload(m, &dl.scale, scale)) return e;
    if (int e = upload(m, &dl.shift, shift)) return e;
    if (int e = pack_layer(m, li, dl.w32, s)) return e;
    if (L.sn) {
      V2CE_REQUIRE(sn_count < kNumSn, "too many spectral-norm layers");
      dl.inv_sigma = m->inv_sigma_dev + sn_count;
      SnDesc& d = m->sn_descs_host[sn_count];
      d.rows = L.cout;
      d.K = L.cin * taps;
      d.W = dl.w32;
      const std::vector<float>*u = find(m, base + ".module.weight_u"), *v = find(m, base + ".module.weight_v");
      if (!u || !v || (int)u->size() != d.rows || (int)v->size() != d.K)
        return set_error(V2CE_ERR_STATE, "missing weight_u / weight_v for %s", L.name);
      if (int e = upload(m, &d.u, *u)) return e;
      if (int e = upload(m, &d.v, *v)) return e;
      if (int e = dev_alloc(m, &d.t, (size_t)d.K)) return e;
      if (int e = dev_alloc(m, &d.s, (size_t)d.rows)) return e;
      if (int e = dev_alloc(m, &d.partial, (size_t)(d.K + kSnCols - 1) / kSnCols)) return e;
      m->max_rows = m->max_rows > d.rows ? m->max_rows : d.rows;
      m->max_k = m->max_k > d.K ? m->max_k : d.K;
      ++sn_count;
    }
  }
  V2CE_REQUIRE(sn_count == kNumSn, "expected %d spectral-norm convs, found %d", kNumSn, sn_count);
  if (int e = dev_alloc(m, &m->sn_descs_dev, kNumSn)) return e;
  V2CE_CUDA_CHECK(cudaMemcpy(m->sn_descs_dev, m->sn_descs_host, sizeof(SnDesc) * kNumSn, cudaMemcpyHostToDevice));
  V2CE_CUDA_CHECK(cudaDeviceSynchronize());
  // fp32 copies of the non-SN GEMM weights are no longer needed on the device side, but they are small
  // next to the activations; host staging copies are released.
  m->host.clear();
  m->finalized = true;
  return V2CE_OK;
}

extern "C" int v2ce_model_workspace_bytes(const v2ce_model* m, int32_t batch, int32_t depth, int32_t height,
                                          int32_t width, size_t* bytes) {
  V2CE_REQUIRE(m && bytes, "NULL argument");
  V2CE_REQUIRE(batch > 0 && depth > 0 && height > 0 && width > 0, "bad shape");
  V2CE_REQUIRE((long long)batch * depth * height * width < (1LL << 31), "batch*depth*H*W must be < 2^31");
  *bytes = carve(nullptr, make_dims(batch, depth, height, width)).bytes;
  return V2CE_OK;
}

extern "C" int v2ce_model_workspace_layout(const v2ce_model* m, int32_t batch, int32_t depth, int32_t height, int32_t width,
                                           int64_t* offsets, int32_t cap, int32_t* n) {
  V2CE_REQUIRE(m && offsets && n, "NULL argument");
  V2CE_REQUIRE(batch > 0 && depth > 0 && height > 0 && width > 0, "bad shape");
  V2CE_REQUIRE((long long)batch * depth * height * width < (1LL << 31), "batch*depth*H*W must be < 2^31");
  const Buffers b = carve(nullptr, make_dims(batch, depth, height, width));
  const __nv_bfloat16* p[] = {b.head_in, b.head, b.enc[0], b.enc[1], b.enc[2], b.enc[3], b.res[0], b.res[1],
                              b.dec[0], b.dec[1], b.dec[2], b.dec[3], b.tmp_t, b.tmp_r, b.up, b.up2};
  constexpr int kBufs = sizeof(p) / sizeof(p[0]);
  V2CE_REQUIRE(cap >= kBufs, "offsets holds %d entries, the layout has %d", cap, kBufs);
  for (int i = 0; i < kBufs; ++i) offsets[i] = (int64_t)reinterpret_cast<uintptr_t>(p[i]);
  *n = kBufs;
  return V2CE_OK;
}

static int forward_impl(v2ce_model* m, const void* x_dev, bool frames_u8, float* y_dev, int32_t B, int32_t D, int32_t H,
                        int32_t W, void* ws_dev, size_t ws_bytes, void* stream) {
  V2CE_REQUIRE(m && x_dev && y_dev && ws_dev, "NULL argument");
  V2CE_REQUIRE(m->finalized, "model not finalized");
  V2CE_REQUIRE(B > 0 && D > 0 && H > 0 && W > 0, "bad shape");
  V2CE_REQUIRE((long long)B * D * H * W < (1LL << 31), "batch*depth*H*W must be < 2^31");
  const Dims d = make_dims(B, D, H, W);
  const Buffers buf = carve(ws_dev, d);
  if (buf.bytes > ws_bytes) return set_error(V2CE_ERR_WORKSPACE, "workspace too small: need %zu, got %zu", buf.bytes, ws_bytes);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  size_t n_marks = 0;
  auto mark = [&](const char* what) {             // per-launch timing (tools/layer_times.py); off by default
    if (!m->layer_timing) return;
    if (n_marks == m->marks.size()) {
      cudaEvent_t ev;
      cudaEventCreate(&ev);
      m->marks.emplace_back(std::string(), ev);
    }
    m->marks[n_marks].first = what;
    cudaEventRecord(m->marks[n_marks].second, s);
    ++n_marks;
  };
  auto stop = [&]() -> int {
    V2CE_CUDA_CHECK(cudaEventRecord(m->ev_join, m->sn_stream));
    V2CE_CUDA_CHECK(cudaStreamWaitEvent(s, m->ev_join, 0));
    return V2CE_OK;
  };
  mark("start");
  // spectral-norm power iteration (input independent) on a side stream, joined before the first SN conv
  V2CE_CUDA_CHECK(cudaEventRecord(m->ev_fork, s));
  V2CE_CUDA_CHECK(cudaStreamWaitEvent(m->sn_stream, m->ev_fork, 0));
  if (int e = run_sn_step(m, m->sn_stream)) return e;
  V2CE_CUDA_CHECK(cudaEventRecord(m->ev_join, m->sn_stream));
  int launches = kSnLaunches;
  // After the launch that writes layer li's output: count it, record the layer's timing mark, and tell whether the
  // option "stop_after" ends the forward here -- at li, or at `also` (a block's shortcut fused into its conv1, pred in
  // decoders.3.conv2).  The caller then returns stop(), with the side stream joined into `s`.  Every launch writes out
  // of place, so the workspace then holds both the inputs of that layer and its output.
  auto launched = [&](int li, int also = -1) {
    ++launches;
    mark(kLayers[li].name);
    return m->stop_after >= 0 && (m->stop_after == li || m->stop_after == also);
  };

  const long long M0 = d.M[0];
  // 32-byte patch rows: 16-channel SWIZZLE_32B view of the 8-channel split pixels
  const halo::KdmPlan hplan = halo::plan_kdm(D, H, W, 1, 32);
  if (hplan.ok) {
    // head conv on the tensor pipe (see head_prep_kernel): split-bf16 pixels -> depth-merged halo kernel, LeakyReLU
    const size_t total = (size_t)M0;
    const int pgrid = (int)((total + 255) / 256 > 148 * 16 ? 148 * 16 : (total + 255) / 256);
    if (frames_u8) head_prep_kernel<true><<<pgrid, 256, 0, s>>>(x_dev, B, D, H, W, buf.head_in);
    else head_prep_kernel<false><<<pgrid, 256, 0, s>>>(x_dev, B, D, H, W, buf.head_in);
    V2CE_LAUNCH_CHECK("head_prep_kernel");
    ++launches;
    const halo::HaloArgs a = halo_args(m->layers[0], View::Head16, nullptr, &hplan, B, D, H, W, 32, buf.head, 32, nullptr,
                                       0, 2, m->error_flag_dev);
    CUtensorMap tm;
    if (int e = get_tmap(m, MapKey{View::Head16, 0, buf.head_in, B, D, H, W, 8, a.PW, a.TH + 2}, &tm)) return e;
    if (int e = halo::launch_halo_kdm(tm, tm, a, nullptr, hplan.smem_bytes, s)) return e;
  } else {
    const long long groups = (long long)B * D * H * ((W + 3) / 4);
    static unsigned long long head_owner[64] = {0};
    if (int e = load_constants(head_owner, m, [&]() -> int {
          V2CE_CUDA_CHECK(cudaMemcpyToSymbolAsync(c_head_w, m->head_wpack, sizeof(float) * 27 * 2 * 32, 0, cudaMemcpyDeviceToDevice, s));
          V2CE_CUDA_CHECK(cudaMemcpyToSymbolAsync(c_head_b, m->layers[0].bias, sizeof(float) * 32, 0, cudaMemcpyDeviceToDevice, s));
          return V2CE_OK;
        }))
      return e;
    if (frames_u8)
      head_conv_kernel<true><<<(int)((groups + 127) / 128), 128, 0, s>>>(x_dev, B, D, H, W, buf.head);
    else
      head_conv_kernel<false><<<(int)((groups + 127) / 128), 128, 0, s>>>(x_dev, B, D, H, W, buf.head);
    V2CE_LAUNCH_CHECK("head_conv_kernel");
  }
  if (launched(0)) return stop();

  static const int ch[5] = {32, 64, 128, 256, 512};
  const __nv_bfloat16* x = buf.head;
  // encoders: conv1 and the shortcut are stride (1,2,2) -> gather kernel; conv2 -> halo kernel
  for (int i = 0; i < 4; ++i) {
    const int l1 = conv1_of(Role::EncConv1, i);
    const int pin = ch[i], co = ch[i + 1];
    bool fused = false;
    if (int e = run_enc_kdm(m, l1, x, pin, B, D, d.H[i], d.W[i], buf.tmp_t, buf.tmp_r, s, &fused)) return e;
    if (fused) {
      if (launched(l1, l1 + 2)) return stop();
    } else {
      if (int e = run_conv(m, l1, x, pin, d.H[i], d.W[i], nullptr, 0, B, D, d.H[i], d.W[i], 2, nullptr, 1, buf.tmp_t, s)) return e;
      if (launched(l1)) return stop();
      if (int e = run_conv(m, l1 + 2, x, pin, d.H[i], d.W[i], nullptr, 0, B, D, d.H[i], d.W[i], 2, nullptr, 0, buf.tmp_r, s)) return e;
      if (launched(l1 + 2)) return stop();
    }
    if (int e = run_halo(m, l1 + 1, buf.tmp_t, co, nullptr, 0, B, D, d.H[i + 1], d.W[i + 1], buf.tmp_r, co, 1, buf.enc[i], co, s)) return e;
    if (launched(l1 + 1)) return stop();
    x = buf.enc[i];
  }
  // residual blocks at the bottleneck (first spectral-norm convs: join the side stream here)
  V2CE_CUDA_CHECK(cudaStreamWaitEvent(s, m->ev_join, 0));
  int side_ev = 0;
  for (int i = 0; i < 2; ++i) {
    const int l1 = conv1_of(Role::ResConv1, i);
    // conv1 (persistent CTAs, a partial last wave) and the block's shortcut both read x: the shortcut goes to the
    // side stream AFTER conv1 so that its CTAs fill the SMs conv1 frees in its tail; conv2 waits for it.
    // (With per-launch timing on, everything stays on one stream.)
    const bool side = !m->layer_timing;
    if (side) {
      V2CE_CUDA_CHECK(cudaEventRecord(m->ev_side[side_ev], s));
      V2CE_CUDA_CHECK(cudaStreamWaitEvent(m->sn_stream, m->ev_side[side_ev], 0));
    }
    if (int e = run_halo(m, l1, x, 512, nullptr, 0, B, D, d.H[4], d.W[4], nullptr, 0, 1, buf.tmp_t, 512, s)) return e;
    if (launched(l1)) return stop();
    if (int e = run_conv(m, l1 + 2, x, 512, d.H[4], d.W[4], nullptr, 0, B, D, d.H[4], d.W[4], 1, nullptr, 0, buf.tmp_r,
                         side ? m->sn_stream : s)) return e;
    if (side) {
      V2CE_CUDA_CHECK(cudaEventRecord(m->ev_side[side_ev + 1], m->sn_stream));
      V2CE_CUDA_CHECK(cudaStreamWaitEvent(s, m->ev_side[side_ev + 1], 0));
      side_ev += 2;
    }
    if (launched(l1 + 2)) return stop();
    // the last block's output is only ever read nearest-upsampled by decoders.0: write it that way
    if (i == 1) {
      if (int e = run_halo(m, l1 + 1, buf.tmp_t, 512, nullptr, 0, B, D, d.H[4], d.W[4], buf.tmp_r, 512, 1, buf.up, 512, s,
                           d.H[3], d.W[3])) return e;
    } else {
      if (int e = run_halo(m, l1 + 1, buf.tmp_t, 512, nullptr, 0, B, D, d.H[4], d.W[4], buf.tmp_r, 512, 1, buf.res[i], 512, s)) return e;
    }
    if (launched(l1 + 1)) return stop();
    x = buf.res[i];
  }
  // decoders: virtual concat [nearest_up(x), skip]; skips are enc2, enc1, enc0, head.  `up` is written directly by
  // the epilogue of the layer that produced x (upsample-on-store); two buffers alternate because a decoder reads
  // one while its conv2 writes the next.  The last decoder's conv2 also applies the prediction layer.
  int xc = 512;
  __nv_bfloat16* up_cur = buf.up;
  __nv_bfloat16* up_next = buf.up2;
  for (int i = 0; i < 4; ++i) {
    const int lvl = 3 - i;                       // output level
    const __nv_bfloat16* skip = lvl == 0 ? buf.head : buf.enc[lvl - 1];
    const int co = ch[lvl];                      // channels of the skip and of the outputs
    const int l1 = conv1_of(Role::DecConv1, i);
    bool short_done = false;
    const bool side = !m->layer_timing && side_ev + 2 <= 16;
    if (side) {
      V2CE_CUDA_CHECK(cudaEventRecord(m->ev_side[side_ev], s));
      V2CE_CUDA_CHECK(cudaStreamWaitEvent(m->sn_stream, m->ev_side[side_ev], 0));
    }
    if (int e = run_halo(m, l1, up_cur, xc, skip, co, B, D, d.H[lvl], d.W[lvl], nullptr, 0, 1, buf.tmp_t, co, s, 0, 0, nullptr,
                         l1 + 2, buf.tmp_r, co, &short_done)) return e;
    if (launched(l1, short_done ? l1 + 2 : -1)) return stop();
    if (!short_done) {
      if (int e = run_conv(m, l1 + 2, up_cur, xc, d.H[lvl], d.W[lvl], skip, co, B, D, d.H[lvl], d.W[lvl], 1, nullptr, 0, buf.tmp_r,
                           side ? m->sn_stream : s)) return e;
      if (side) {
        V2CE_CUDA_CHECK(cudaEventRecord(m->ev_side[side_ev + 1], m->sn_stream));
        V2CE_CUDA_CHECK(cudaStreamWaitEvent(s, m->ev_side[side_ev + 1], 0));
      }
      if (launched(l1 + 2)) return stop();
    }
    if (side) side_ev += 2;
    if (lvl > 0) {
      if (int e = run_halo(m, l1 + 1, buf.tmp_t, co, nullptr, 0, B, D, d.H[lvl], d.W[lvl], buf.tmp_r, co, 1, up_next, co, s,
                           d.H[lvl - 1], d.W[lvl - 1])) return e;
    } else {
      if (int e = run_halo(m, l1 + 1, buf.tmp_t, co, nullptr, 0, B, D, d.H[lvl], d.W[lvl], buf.tmp_r, co, 1, buf.dec[i], co, s,
                           0, 0, y_dev)) return e;
    }
    if (launched(l1 + 1, lvl == 0 ? kNumLayers - 1 : -1)) return stop();
    __nv_bfloat16* tsw = up_cur; up_cur = up_next; up_next = tsw;
    xc = co;
  }
  m->last_launches = launches;
  return V2CE_OK;
}

extern "C" int v2ce_model_forward(v2ce_model* m, const float* x_dev, float* y_dev, int32_t B, int32_t D, int32_t H,
                                  int32_t W, void* ws_dev, size_t ws_bytes, void* stream) {
  return forward_impl(m, x_dev, false, y_dev, B, D, H, W, ws_dev, ws_bytes, stream);
}

extern "C" int v2ce_model_forward_frames(v2ce_model* m, const uint8_t* frames_dev, float* y_dev, int32_t B, int32_t D,
                                         int32_t H, int32_t W, void* ws_dev, size_t ws_bytes, void* stream) {
  return forward_impl(m, frames_dev, true, y_dev, B, D, H, W, ws_dev, ws_bytes, stream);
}

extern "C" int v2ce_model_last_sigmas(const v2ce_model* m, float* sigma12_host) {
  V2CE_REQUIRE(m && sigma12_host && m->finalized, "bad argument");
  V2CE_CUDA_CHECK(cudaDeviceSynchronize());
  V2CE_CUDA_CHECK(cudaMemcpy(sigma12_host, m->sigma_dev, sizeof(float) * kNumSn, cudaMemcpyDeviceToHost));
  int flag = 0;
  V2CE_CUDA_CHECK(cudaMemcpy(&flag, m->error_flag_dev, sizeof(int), cudaMemcpyDeviceToHost));
  if (flag) return set_error(V2CE_ERR_CUDA, "conv pipeline watchdog fired");
  return V2CE_OK;
}

extern "C" int v2ce_model_call_count(const v2ce_model* m, int64_t* calls) {
  V2CE_REQUIRE(m && calls, "NULL argument");
  *calls = m->calls;
  return V2CE_OK;
}

extern "C" int v2ce_model_sn_advance(v2ce_model* m, int32_t n_calls, void* stream) {
  V2CE_REQUIRE(m && m->finalized && n_calls >= 0, "bad argument");
  for (int i = 0; i < n_calls; ++i)
    if (int e = run_sn_step(m, static_cast<cudaStream_t>(stream))) return e;
  return V2CE_OK;
}

extern "C" int v2ce_model_last_launches(const v2ce_model* m, int32_t* launches) {
  V2CE_REQUIRE(m && launches, "NULL argument");
  *launches = m->last_launches;
  return V2CE_OK;
}

extern "C" int v2ce_model_layer_times(v2ce_model* m, int32_t cap, float* ms_out, char* names_out, int32_t* count) {
  V2CE_REQUIRE(m && ms_out && names_out && count && cap > 0, "bad argument");
  V2CE_CUDA_CHECK(cudaDeviceSynchronize());
  int n = 0;
  for (size_t i = 1; i < m->marks.size() && n < cap; ++i) {
    if (m->marks[i].first == "start") break;     // marks of an earlier, longer forward
    float ms = 0.f;
    V2CE_CUDA_CHECK(cudaEventElapsedTime(&ms, m->marks[i - 1].second, m->marks[i].second));
    ms_out[n] = ms;
    snprintf(names_out + (size_t)n * 48, 48, "%s", m->marks[i].first.c_str());
    ++n;
  }
  *count = n;
  return V2CE_OK;
}

extern "C" int v2ce_model_set_option(v2ce_model* m, const char* key, int64_t value) {
  V2CE_REQUIRE(m && key, "NULL argument");
  if (std::string(key) == "layer_timing") { m->layer_timing = (int)value; return V2CE_OK; }
  if (std::string(key) == "stop_after") {
    V2CE_REQUIRE(value >= -1 && value < kNumLayers, "stop_after must be -1 or a layer index < %d", kNumLayers);
    m->stop_after = (int)value;
    return V2CE_OK;
  }
  return set_error(V2CE_ERR_INVALID, "unknown option '%s'", key);
}

extern "C" int v2ce_conv3d_bf16_ex(const void* src0_dev, int32_t c0, int32_t h0, int32_t w0, const void* src1_dev, int32_t c1,
                                   int32_t batch, int32_t depth, int32_t hin, int32_t win, int32_t ksize, int32_t stride_hw,
                                   const float* weight_host, int32_t cout, const float* scale_host, const float* shift_host,
                                   const void* residual_dev, int32_t act, void* out_dev, int32_t impl, void* stream) {
  V2CE_REQUIRE(src0_dev && weight_host && scale_host && shift_host && out_dev, "NULL argument");
  V2CE_REQUIRE(ksize == 1 || ksize == 3, "ksize must be 1 or 3");
  V2CE_REQUIRE(stride_hw == 1 || stride_hw == 2, "stride must be 1 or 2");
  V2CE_REQUIRE(c0 > 0 && c0 % 8 == 0 && c1 >= 0 && c1 % 8 == 0, "channel counts must be multiples of 8");
  V2CE_REQUIRE((src1_dev != nullptr) == (c1 > 0), "src1 and c1 must agree");
  const int bn = conv::pick_bn(cout);
  V2CE_REQUIRE(bn != 0, "cout must be a multiple of 32");
  if (impl >= 2)
    V2CE_REQUIRE(halo::plan_kdm(depth, stride_hw == 2 ? (hin - 1) / 2 + 1 : hin, stride_hw == 2 ? (win - 1) / 2 + 1 : win, stride_hw).ok,
                 "depth-merged halo kernel: depth % 8 == 0");
  if (impl == 3) V2CE_REQUIRE(residual_dev != nullptr, "impl 3: residual_dev receives the fused shortcut output");
  if (impl >= 1)
    V2CE_REQUIRE(ksize == 3 && (stride_hw == 1 || (impl >= 2 && c1 == 0)) && h0 == hin && w0 == win && c0 % 64 == 0 && c1 % 64 == 0,
                 "halo kernel: 3x3x3, stride 1 (depth-merged variant: also stride 2 with one source), no upsample, "
                 "channel pitches multiple of 64");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int cin = c0 + c1, taps = ksize * ksize * ksize;
  const int num_kb = (taps * cin + conv::kBlockK - 1) / conv::kBlockK;
  float *w_dev = nullptr, *scale_dev = nullptr, *shift_dev = nullptr;
  __nv_bfloat16 *wpack = nullptr, *wshort = nullptr;
  int* flag = nullptr;
  const size_t wn = (size_t)cout * cin * taps, pn = (size_t)cout * num_kb * conv::kBlockK;
  V2CE_CUDA_CHECK(cudaMalloc(&w_dev, wn * sizeof(float)));
  V2CE_CUDA_CHECK(cudaMalloc(&scale_dev, cout * sizeof(float)));
  V2CE_CUDA_CHECK(cudaMalloc(&shift_dev, cout * sizeof(float)));
  V2CE_CUDA_CHECK(cudaMalloc(&wpack, pn * sizeof(__nv_bfloat16)));
  V2CE_CUDA_CHECK(cudaMalloc(&flag, sizeof(int)));
  V2CE_CUDA_CHECK(cudaMemsetAsync(flag, 0, sizeof(int), s));
  V2CE_CUDA_CHECK(cudaMemcpyAsync(w_dev, weight_host, wn * sizeof(float), cudaMemcpyHostToDevice, s));
  V2CE_CUDA_CHECK(cudaMemcpyAsync(scale_dev, scale_host, cout * sizeof(float), cudaMemcpyHostToDevice, s));
  V2CE_CUDA_CHECK(cudaMemcpyAsync(shift_dev, shift_host, cout * sizeof(float), cudaMemcpyHostToDevice, s));
  const int pgrid = (int)((pn + 255) / 256 > 4096 ? 4096 : (pn + 255) / 256);
  if (impl == 1)
    halo::pack_weights_halo_kernel<<<pgrid, 256, 0, s>>>(w_dev, cout, cin, bn, c0, c0, c1, c1, wpack);
  else if (impl >= 2)
    halo::pack_weights_kdm_kernel<<<pgrid, 256, 0, s>>>(w_dev, cout, cin, c0, c0, c1, c1, wpack);
  else
    conv::pack_weights_kernel<<<pgrid, 256, 0, s>>>(w_dev, cout, cin, taps, bn, num_kb, c0, c0, c1, c1, wpack);
  int rc = V2CE_OK;
  if (cudaGetLastError() != cudaSuccess) rc = set_error(V2CE_ERR_CUDA, "weight pack launch failed");
  const int pad = ksize / 2;
  const int hout = (hin + 2 * pad - ksize) / stride_hw + 1, wout = (win + 2 * pad - ksize) / stride_hw + 1;
  // the hook's conv as a model layer whose channel pitches are its channel counts
  DevLayer dl;
  dl.cfg = LayerCfg{impl >= 1 ? Kernel::Halo : Kernel::Gather, c0, c0, c1, c1};
  dl.wpack = dl.wpack_kdm = wpack;
  dl.scale = scale_dev; dl.shift = shift_dev;
  dl.bn_tile = bn; dl.num_kb = num_kb;
  const __nv_bfloat16* src0 = static_cast<const __nv_bfloat16*>(src0_dev);
  const __nv_bfloat16* src1 = static_cast<const __nv_bfloat16*>(src1_dev);
  const __nv_bfloat16* residual = static_cast<const __nv_bfloat16*>(residual_dev);
  __nv_bfloat16* out = static_cast<__nv_bfloat16*>(out_dev);
  if (rc == V2CE_OK && impl >= 1) {
    const halo::HaloPlan plan = halo::plan_for(bn, depth, hin, win);
    const halo::KdmPlan kplan = halo::plan_kdm(depth, hout, wout, stride_hw);
    const bool s2 = stride_hw == 2;              // depth-merged variant only (checked above)
    const halo::HaloArgs a = halo_args(dl, s2 ? View::Parity : View::Patch64, &plan, impl >= 2 ? &kplan : nullptr, batch,
                                       depth, hout, wout, cout, out, cout, impl == 3 ? nullptr : residual, cout, act, flag);
    halo::ParityMaps pmaps;
    CUtensorMap tm0, tm1;
    if (s2) {
      for (int q = 0; q < 4 && rc == V2CE_OK; ++q)
        rc = make_map(MapKey{View::Parity, q, src0, batch, depth, hin, win, c0, a.PW, a.TH + 1}, &pmaps.m[q]);
      tm0 = pmaps.m[0];
    } else {
      rc = make_map(MapKey{View::Patch64, 0, src0, batch, depth, hin, win, c0, a.PW, a.TH + 2}, &tm0);
    }
    tm1 = tm0;
    if (rc == V2CE_OK && src1)
      rc = make_map(MapKey{View::Patch64, 0, src1, batch, depth, hin, win, c1, a.PW, a.TH + 2}, &tm1);
    if (rc == V2CE_OK && impl == 3) {
      // fused shortcut: 1x1x1 weights = centre tap of `weight`, same scale/shift, no activation -> residual_dev
      std::vector<float> wd((size_t)cout * cin);
      for (size_t i = 0; i < wd.size(); ++i) wd[i] = weight_host[i * 27 + 13];
      float* wd_dev = nullptr;
      if (cudaMalloc(&wd_dev, wd.size() * sizeof(float)) != cudaSuccess ||
          cudaMalloc(&wshort, wd.size() * sizeof(__nv_bfloat16)) != cudaSuccess)
        rc = set_error(V2CE_ERR_CUDA, "cudaMalloc failed");
      if (rc == V2CE_OK) {
        cudaMemcpyAsync(wd_dev, wd.data(), wd.size() * sizeof(float), cudaMemcpyHostToDevice, s);
        halo::pack_weights_kdm_short_kernel<<<(int)((wd.size() + 255) / 256), 256, 0, s>>>(wd_dev, cout, cin, c0, c0, c1, c1, wshort);
        cudaStreamSynchronize(s);
        halo::KdmShort sc{wshort, scale_dev, shift_dev, static_cast<__nv_bfloat16*>(const_cast<void*>(residual_dev)), cout};
        rc = halo::launch_halo_kdm(tm0, tm1, a, &sc, kplan.smem_bytes, s, s2 ? &pmaps : nullptr);
      }
      cudaStreamSynchronize(s);
      cudaFree(wd_dev);
    } else if (rc == V2CE_OK) {
      rc = impl == 2 ? halo::launch_halo_kdm(tm0, tm1, a, nullptr, kplan.smem_bytes, s, s2 ? &pmaps : nullptr)
                     : halo::launch_halo(tm0, tm1, a, bn, plan.smem_bytes, s);
    }
  } else if (rc == V2CE_OK) {
    rc = conv::launch_conv(conv_args(dl, ksize, cout, src0, c0, h0, w0, src1, c1, batch, depth, hin, win, stride_hw, residual,
                                     act, out, flag),
                           bn, s);
  }
  cudaError_t se = cudaStreamSynchronize(s);
  int hflag = 0;
  if (se == cudaSuccess) cudaMemcpy(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost);
  cudaFree(w_dev); cudaFree(scale_dev); cudaFree(shift_dev); cudaFree(wpack); cudaFree(wshort); cudaFree(flag);
  if (rc != V2CE_OK) return rc;
  if (se != cudaSuccess) return set_error(V2CE_ERR_CUDA, "conv3d_bf16 failed: %s", cudaGetErrorString(se));
  if (hflag) return set_error(V2CE_ERR_CUDA, "conv pipeline watchdog fired");
  return V2CE_OK;
}

// ------------------------------------------------------------------------------------------
// Bring-up microbenchmark: tensor-pipe rate of back-to-back tcgen05.mma (SS operands, M=128, K=16)
// on resident shared-memory tiles, no loads.  Gives the ceiling the conv kernels can reach with
// cta_group::1.  Not used by the product path.
// ------------------------------------------------------------------------------------------
namespace v2ce {
namespace unet {
template <int BN>
__global__ void __launch_bounds__(128) mma_rate_kernel(int iters, int naccs, long long* cycles_out) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = conv::smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(8) unsigned long long bar;
  const int warp = conv::uniform_warp_id();
  for (int i = threadIdx.x; i < (16384 + BN * 128) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem_raw + (base - raw))[i] = 0u;
  if (threadIdx.x == 0) {
    conv::mbar_init(conv::smem_u32(&bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(conv::smem_u32(&tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  conv::fence_proxy_async();
  conv::tcgen05_fence_before();
  __syncthreads();
  conv::tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  if (warp == 1) {
    const uint32_t idesc = conv::make_idesc(BN);
    const uint32_t a_addr = base, b_addr = base + 16384;
    long long t0 = clock64();
    for (int it = 0; it < iters; ++it) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        conv::tcgen05_mma_bf16_elect(tmem + (uint32_t)((it % naccs) * BN), conv::make_smem_desc(a_addr + k * 32),
                                     conv::make_smem_desc(b_addr + k * 32), idesc, 1u);
    }
    conv::tcgen05_commit_elect(conv::smem_u32(&bar));
    conv::mbar_wait(conv::smem_u32(&bar), 0, nullptr);
    long long t1 = clock64();
    if (threadIdx.x == 32 && blockIdx.x == 0) cycles_out[0] = t1 - t0;
  }
  conv::tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}
}  // namespace unet
}  // namespace v2ce

extern "C" int v2ce_debug_mma_rate(int32_t bn, int32_t iters, int32_t naccs, int32_t ctas, double* cycles_per_mma) {
  long long* d = nullptr;
  V2CE_CUDA_CHECK(cudaMalloc(&d, sizeof(long long)));
  const int smem = 16384 + 256 * 128 + 2048;
  #define RUN(N) { V2CE_CUDA_CHECK(cudaFuncSetAttribute(mma_rate_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
                   mma_rate_kernel<N><<<ctas, 128, smem>>>(iters, naccs, d); }
  if (bn == 32) RUN(32) else if (bn == 64) RUN(64) else if (bn == 96) RUN(96) else if (bn == 128) RUN(128)
  else if (bn == 192) RUN(192) else if (bn == 256) RUN(256)
  else { cudaFree(d); return set_error(V2CE_ERR_INVALID, "bn"); }
  #undef RUN
  V2CE_CUDA_CHECK(cudaDeviceSynchronize());
  long long c = 0;
  V2CE_CUDA_CHECK(cudaMemcpy(&c, d, sizeof(c), cudaMemcpyDeviceToHost));
  cudaFree(d);
  *cycles_per_mma = (double)c / ((double)iters * 4.0);
  return V2CE_OK;
}
