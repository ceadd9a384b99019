// Halo-tile Conv3d (3x3x3, stride 1, pad 1) for sm_100a: the A operand of all nine (kh,kw) taps of a
// depth slice comes from ONE shared-memory copy of the input patch.
//
// Why: with one gather per tap (conv_igemm.cuh) a 128xN tile needs 16 KB of activations per 64-wide
// k-block; for N <= 64 that is 128-256 B/clk/SM against ~40 B/clk/SM of L2->SM bandwidth, so the
// tensor pipe idles (measured: 5.6 % active on decoders.3.conv1).  Here TMA (cp.async.bulk.tensor.5d,
// 128B swizzle, zero fill outside the image = the conv padding) loads a (TH+2) x PW pixel patch of 64
// channels once per (kd, channel chunk); the tile's M index runs over the patch with pitch PW = TW+2,
// so tap (kh,kw) is the same buffer read from row kh*PW+kw on: a descriptor whose start address is
// shifted by whole 128-byte rows.  Rows whose column index falls in the 2 halo columns produce
// garbage accumulator rows that the epilogue skips (MMA rows are independent).
//
// Depth blocking: a CTA computes T consecutive depth slices of the same (h,w) tile (T accumulators of
// BN TMEM columns).  Slice d+t under tap kd reads input slice d+t+kd-1, so the T+2 patches d-1..d+T
// serve all 3*T (kd, t) pairs, and every weight tile (cc, kd, tap) fetched from L2 is used for T*128
// output rows instead of 128.  With M = 128 rows per weight tile the L2->SM weight stream alone needs
// 64 B/clk/SM (more than the fabric delivers: measured 12-25 % tensor-pipe activity); T = 4 cuts it to
// 16 B/clk and the patch traffic by a further (T+2)/(3T).
//
// Replaces the same reference calls as conv_igemm.cuh (submodules.py:249-263) for the 20 stride-1
// 3x3x3 convs, i.e. 91 % of the network's FLOPs.
//
// Persistent CTAs (one per SM) walk a strided tile sequence; the smem rings run on across tiles and, where
// 2*T*BN <= 512 TMEM columns, two accumulator sets let the epilogue of tile i overlap the MMAs of tile i+1.
// CTA = 224 threads: warp 0 TMA patch producer, warp 1 weight-tile producer (bulk copy), warp 2 TMEM
// allocator + MMA issuer (all three warp-converged, one elected lane issues), warps 3-6 epilogue (TMEM lane
// quarter = warp % 4).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "conv_igemm.cuh"

namespace v2ce {
namespace halo {

using namespace conv;

constexpr int kHaloThreads = 224;
constexpr int kMaxSA = 6, kMaxSB = 8;

struct HaloArgs {
  int B, D, H, W;
  int PW, TH, TW;              // patch pitch (TW + 2), output rows and valid columns of a tile; TH*PW <= 128
  int tiles_w, tiles_h;
  int ncc0, ncc1;              // 64-channel chunks taken from source 0 / source 1 (virtual concat)
  int real0, real1;            // real channels per source: a chunk with < 64 of them issues fewer K=16 MMA steps
  int Cout;                    // real output channels (multiple of BN)
  int out_pitch;               // channel pitch of `out`; columns [Cout, out_pitch) are zero-filled
  int res_pitch;               // channel pitch of `residual`
  int T;                       // depth slices per CTA (T accumulators); D % T == 0
  int SA, SB;                  // pipeline depths (patch ring / weight ring)
  int a_stage_bytes;           // bytes reserved per patch stage (multiple of 1024)
  int box_bytes;               // bytes one TMA box delivers: PW * (TH+2) * 128
  int a_row16;                 // conv_halo_kdm only: bytes of one patch pixel row / 16 -- 8 (64 channels, SWIZZLE_128B) or
                               // 2 (16 channels, SWIZZLE_32B: the head conv's 8-channel split pixels)
  uint32_t a_desc_hi;          // high word of the A operand's UMMA descriptor for that layout
  int tap_mask;                // conv_halo_kdm, stride 1: bit (kh*3+kw) set = the tap is multiplied (0x1FF; the head skips kw = 1)
  const __nv_bfloat16* wpack;  // [Cout/BN][ncc][3 kd][9 taps][BN][64], rows pre-swizzled
  const float* scale;
  const float* shift;
  const float* inv_sigma;
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;
  int act;
  int up_H, up_W;              // > 0: write the output nearest-upsampled to (up_H, up_W) (unet_2layer.py:359-362),
                               //      i.e. every source pixel is stored to all dst with (dst*H)//up_H == h
  const float* pred_w;         // != nullptr (BN == 32 only): fuse pred = relu(W[20][32] . y + b) and write the
  const float* pred_b;         //      float32 (B,L,20,H,W) network output instead of `out` (v2ce_3d.py:29)
  float* pred_out;
  int* error_flag;
};

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::
          "r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(bar)
      : "memory");
}

// Measured on B200 (tools/run_halo_cases.sh): the UMMA 128B swizzle is a function of the absolute shared-
// memory address, so a descriptor whose start is shifted by whole 128-byte rows reads a TMA-written patch
// correctly with base_offset = 0; setting base_offset = (addr >> 7) & 7 gives wrong results.

// NBUF = number of TMEM accumulator sets (T*BN columns each): 2 when 2*T*BN <= 512, so the epilogue of
// tile i overlaps the MMAs of tile i+1.
template <int BN, int T>
struct HaloCfg {
  static constexpr int kNBuf = (2 * T * BN <= 512) ? 2 : 1;
  static constexpr int kTmemCols = kNBuf * T * BN;
};

struct TileCoord { int n_tile, b, d0, h0, w0; };

// prediction layer (v2ce_3d.py:29, 32 -> 20 channels, 1x1x1, bias, ReLU) fused into the last decoder conv:
// [20][32] weights followed by [20] biases.  Loaded by load_pred_constants() before the launch that uses them.
__constant__ float c_pred[660];

__device__ __forceinline__ TileCoord decode_tile(int tile, const HaloArgs& a, int T, int n_tiles_unused) {
  // spatial tiles fastest, then depth group, batch, and the output-channel tile slowest: CTAs that run
  // at the same time read neighbouring patches and the same weights
  TileCoord c;
  const int tw_i = tile % a.tiles_w; tile /= a.tiles_w;
  const int th_i = tile % a.tiles_h; tile /= a.tiles_h;
  const int dgroups = a.D / T;
  c.d0 = (tile % dgroups) * T; tile /= dgroups;
  c.b = tile % a.B;
  c.n_tile = tile / a.B;
  c.h0 = th_i * a.TH;
  c.w0 = tw_i * a.TW;
  return c;
}

// Epilogue of one tile for the accumulator rows of one TMEM lane quarter: slices tt0, tt0+tt_step, ... < tt_end of
// the tile (accumulator of slice tt at TMEM columns `tmem_cols + tt*BN`, lane offset already in `tmem_cols`).
//   y = act(acc*scale(+1/sigma) + shift (+ residual)) -> bf16 NDHWC, optionally stored nearest-upsampled, or fed to
//   the fused prediction layer.  Chunks of 32 accumulator columns, flattened over (slice, column block); the residual
//   of chunk q+1 is requested before chunk q is processed: one exposed global-load latency per tile instead of one
//   per 16-byte piece (the epilogue was as long as the MMA phase -- ncu: 50 % of samples in long_scoreboard).
template <int BN>
__device__ __forceinline__ void halo_epilogue_slices(const HaloArgs& a, const TileCoord& tc, int n_tiles, uint32_t tmem_cols,
                                                     int tt0, int tt_step, int tt_end, int th, int tw,
                                                     const float* s_scale, const float* s_shift, const float* s_pred) {
  const int h = tc.h0 + th, w = tc.w0 + tw;
  const bool row_ok = (th < a.TH) && (tw < a.TW) && (h < a.H) && (w < a.W);
  // destination rows/columns of this source pixel when the output is written nearest-upsampled
  int uh0 = 0, uh1 = 0, uw0 = 0, uw1 = 0;
  if (a.up_H > 0 && row_ok) {
    uh0 = (h * a.up_H + a.H - 1) / a.H;  uh1 = ((h + 1) * a.up_H + a.H - 1) / a.H;
    uw0 = (w * a.up_W + a.W - 1) / a.W;  uw1 = ((w + 1) * a.up_W + a.W - 1) / a.W;
  }
  constexpr int kChunksPerSlice = BN / 32;
  const int n_slices = (tt_end - tt0 + tt_step - 1) / tt_step;
  const int n_chunks = n_slices * kChunksPerSlice;
  const size_t plane0 = (size_t)(tc.b * a.D + tc.d0);
  const size_t pix = (size_t)h * a.W + w;
  const size_t HWp = (size_t)a.H * a.W;
  uint4 rv[4] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
  auto res_ptr = [&](int q) {
    const int tt = tt0 + (q / kChunksPerSlice) * tt_step, c0 = (q % kChunksPerSlice) * 32;
    return reinterpret_cast<const uint4*>(a.residual + ((plane0 + tt) * HWp + pix) * a.res_pitch + tc.n_tile * BN + c0);
  };
  const bool has_res = (a.residual != nullptr) && row_ok;
  if (has_res && n_chunks > 0) {
    const uint4* rp = res_ptr(0);
#pragma unroll
    for (int g = 0; g < 4; ++g) rv[g] = __ldg(rp + g);
  }
#pragma unroll 1
  for (int q = 0; q < n_chunks; ++q) {
    const int tt = tt0 + (q / kChunksPerSlice) * tt_step, c0 = (q % kChunksPerSlice) * 32;
    const size_t plane = plane0 + tt;
    const size_t m = plane * HWp + pix;
    uint32_t v[32];
    tmem_ld_32x32b_x32(tmem_cols + (uint32_t)(tt * BN + c0), v);
    uint4 rn[4] = {rv[0], rv[1], rv[2], rv[3]};
    if (has_res && q + 1 < n_chunks) {
      const uint4* rp = res_ptr(q + 1);
#pragma unroll
      for (int g = 0; g < 4; ++g) rn[g] = __ldg(rp + g);
    }
    tmem_ld_wait();
    if (row_ok) {
      float yv[32];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const __nv_bfloat162* rp2 = reinterpret_cast<const __nv_bfloat162*>(&rv[g]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __bfloat1622float2(rp2[j]);      // zeros when there is no residual
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int n = c0 + g * 8 + 2 * j + hh;
            float tv = fmaf(__uint_as_float(v[g * 8 + 2 * j + hh]), s_scale[n], s_shift[n]) + (hh ? f.y : f.x);
            if (a.act == 1) tv = fmaxf(tv, 0.f);
            else if (a.act == 2) tv = tv > 0.f ? tv : 0.01f * tv;
            yv[g * 8 + 2 * j + hh] = tv;
          }
        }
      }
      if (BN == 32 && a.pred_w != nullptr) {
        // fused prediction layer: 20 dot products over the 32 channels of this pixel (four independent
        // accumulation chains at a time), ReLU, planar fp32 store.  The weights are FFMA constant-bank operands
        // (c_pred): no shared-memory loads in the loop.
        float* dst = a.pred_out + plane * 20 * HWp + pix;
#pragma unroll
        for (int n0 = 0; n0 < 20; n0 += 4) {
          float acc[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) acc[u] = c_pred[640 + n0 + u];
#pragma unroll
          for (int c = 0; c < 32; ++c) {
#pragma unroll
            for (int u = 0; u < 4; ++u) acc[u] = fmaf(yv[c], c_pred[(n0 + u) * 32 + c], acc[u]);
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) dst[(size_t)(n0 + u) * HWp] = fmaxf(acc[u], 0.f);
        }
      } else {
        uint4 ov[4];
        __nv_bfloat162* op = reinterpret_cast<__nv_bfloat162*>(ov);
#pragma unroll
        for (int j = 0; j < 16; ++j) op[j] = __floats2bfloat162_rn(yv[2 * j], yv[2 * j + 1]);
        if (a.up_H > 0) {
          for (int hh = uh0; hh < uh1; ++hh)
            for (int ww = uw0; ww < uw1; ++ww) {
              uint4* d4 = reinterpret_cast<uint4*>(a.out + ((plane * a.up_H + hh) * a.up_W + ww) * a.out_pitch +
                                                   tc.n_tile * BN + c0);
#pragma unroll
              for (int g = 0; g < 4; ++g) d4[g] = ov[g];
            }
        } else {
          uint4* d4 = reinterpret_cast<uint4*>(a.out + m * a.out_pitch + tc.n_tile * BN + c0);
#pragma unroll
          for (int g = 0; g < 4; ++g) d4[g] = ov[g];
        }
      }
      if (c0 + 32 == BN && tc.n_tile == n_tiles - 1 && a.up_H == 0 && a.pred_w == nullptr) {
        // zero the padding channels so later TMA reads see 0, not garbage
        for (int c = a.Cout; c < a.out_pitch; c += 8)
          *reinterpret_cast<uint4*>(a.out + m * a.out_pitch + c) = make_uint4(0u, 0u, 0u, 0u);
      }
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) rv[g] = rn[g];
  }
}


template <int BN, int T>
__global__ void __launch_bounds__(kHaloThreads) conv_halo_kernel(const __grid_constant__ CUtensorMap tm0,
                                                                  const __grid_constant__ CUtensorMap tm1,
                                                                  const HaloArgs a) {
  using Cfg = HaloCfg<BN, T>;
  constexpr int NBUF = Cfg::kNBuf;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  constexpr int kBStage = BN * kBlockK * 2;

  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31;
  const int n_tiles = a.Cout / BN;
  const int total_tiles = a.B * (a.D / T) * a.tiles_h * a.tiles_w * n_tiles;
  const int ncc = a.ncc0 + a.ncc1;

  const uint32_t a_base = base;
  const uint32_t b_base = base + (uint32_t)a.SA * a.a_stage_bytes;
  const uint32_t bar_base = b_base + (uint32_t)a.SB * kBStage;
  auto a_full = [&](int s) { return bar_base + 8u * s; };
  auto a_empty = [&](int s) { return bar_base + 8u * (kMaxSA + s); };
  auto b_full = [&](int s) { return bar_base + 8u * (2 * kMaxSA + s); };
  auto b_empty = [&](int s) { return bar_base + 8u * (2 * kMaxSA + kMaxSB + s); };
  auto tmem_full = [&](int s) { return bar_base + 8u * (2 * kMaxSA + 2 * kMaxSB + s); };
  auto tmem_empty = [&](int s) { return bar_base + 8u * (2 * kMaxSA + 2 * kMaxSB + 2 + s); };
  const int bar_bytes = (2 * kMaxSA + 2 * kMaxSB + 4) * 8;
  uint8_t* tail = smem + (bar_base - base) + bar_bytes;
  volatile uint32_t* tmem_ptr = reinterpret_cast<volatile uint32_t*>(tail);
  float* s_scale = reinterpret_cast<float*>(tail + 16);
  float* s_shift = s_scale + BN;
  float* s_pred = s_shift + BN;                   // [20][32] weights + [20] bias (used when a.pred_w != nullptr)

  if (tid == 0) {
    for (int s = 0; s < a.SA; ++s) { mbar_init(a_full(s), 1); mbar_init(a_empty(s), 1); }
    for (int s = 0; s < a.SB; ++s) { mbar_init(b_full(s), 1); mbar_init(b_empty(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tmem_full(s), 1); mbar_init(tmem_empty(s), 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(const_cast<uint32_t*>(tmem_ptr))),
                 "r"((uint32_t)Cfg::kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_acc = *tmem_ptr;

  // Persistent CTA: every role walks the same tile sequence; the smem rings and their phases run on
  // across tiles, so the producers prefetch the next tile while the current one is multiplied/stored.
  // The three feeding roles run warp-converged (uniform registers for addresses/descriptors); the single
  // issuing lane is chosen by elect.sync.
  if (warp == 0) {
    // ================= patch producer (TMA) =================
    int s = 0, ph = 1;                              // stage / parity of the empty barrier to wait on
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(tile, a, T, n_tiles);
      for (int cc = 0; cc < ncc; ++cc) {
        const bool first = cc < a.ncc0;
        const CUtensorMap* map = first ? &tm0 : &tm1;
        const int c0 = (first ? cc : cc - a.ncc0) * kBlockK;
        for (int z = 0; z < T + 2; ++z) {
          mbar_wait(a_empty(s), (uint32_t)ph, a.error_flag);
          if (elect_one()) {
            mbar_arrive_expect_tx(a_full(s), (uint32_t)a.box_bytes);
            tma_load_5d(a_base + (uint32_t)s * a.a_stage_bytes, map, c0, tc.w0 - 1, tc.h0 - 1, tc.d0 - 1 + z, tc.b, a_full(s));
          }
          __syncwarp();
          if (++s == a.SA) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= weight-tile producer (bulk copy) =================
    const int per_tile = ncc * 27;
    int s = 0, ph = 1;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(tile, a, T, n_tiles);
      const __nv_bfloat16* wt = a.wpack + (size_t)tc.n_tile * per_tile * (BN * kBlockK);
      for (int it = 0; it < per_tile; ++it) {
        mbar_wait(b_empty(s), (uint32_t)ph, a.error_flag);
        if (elect_one()) {
          mbar_arrive_expect_tx(b_full(s), (uint32_t)kBStage);
          bulk_copy_g2s(b_base + (uint32_t)s * kBStage, wt + (size_t)it * (BN * kBlockK), (uint32_t)kBStage, b_full(s));
        }
        __syncwarp();
        if (++s == a.SB) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 2) {
    // ================= MMA issuer =================
    constexpr uint32_t idesc = make_idesc(BN);
    int sb = 0, pb = 0;                             // weight ring position / parity
    int sw = 0, pw = 0;                             // next patch stage to wait for / its parity
    int arrived = 0, loads_base = 0;
    int s_first = 0;                                // stage of slice kd of the current chunk
    int iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
      const int ab = (NBUF == 2) ? (iter & 1) : 0;
      const int use = (NBUF == 2) ? (iter >> 1) : iter;
      mbar_wait(tmem_empty(ab), (uint32_t)((use & 1) ^ 1), a.error_flag);     // epilogue has drained this accumulator set
      tcgen05_fence_after();
      const uint32_t acc_base = tmem_acc + (uint32_t)(ab * T * BN);
      for (int cc = 0; cc < ncc; ++cc) {
        // channels beyond the real ones (the upper half of a 32-channel tensor's 64-channel rows) are not multiplied
        const int rem = (cc < a.ncc0) ? (a.real0 - cc * kBlockK) : (a.real1 - (cc - a.ncc0) * kBlockK);
        const int ks = rem >= kBlockK ? kBlockK / 16 : (rem + 15) / 16;
#pragma unroll 1
        for (int kd = 0; kd < 3; ++kd) {
          const int need = loads_base + cc * (T + 2) + kd + T;   // slices kd .. kd+T-1 of this chunk must have landed
          while (arrived < need) {
            mbar_wait(a_full(sw), (uint32_t)pw, a.error_flag);
            ++arrived;
            if (++sw == a.SA) { sw = 0; pw ^= 1; }
          }
          tcgen05_fence_after();
          uint32_t patch[T];
#pragma unroll
          for (int tt = 0; tt < T; ++tt) {
            int st = s_first + tt;
            if (st >= a.SA) st -= a.SA;
            patch[tt] = a_base + (uint32_t)st * a.a_stage_bytes;
          }
#pragma unroll 1
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(b_full(sb), (uint32_t)pb, a.error_flag);
            tcgen05_fence_after();
            const uint32_t b_addr = b_base + (uint32_t)sb * kBStage;
            const uint32_t shift = (uint32_t)((tap / 3) * a.PW + (tap % 3)) * 128u;
            const uint32_t acc0 = (cc | kd | tap) == 0 ? 0u : 1u;
#pragma unroll
            for (int tt = 0; tt < T; ++tt) {
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k) {
                if (k < ks)
                  tcgen05_mma_bf16_elect(acc_base + (uint32_t)(tt * BN), make_smem_desc(patch[tt] + shift + k * 32),
                                         make_smem_desc(b_addr + k * 32), idesc, k == 0 ? acc0 : 1u);
              }
            }
            tcgen05_commit_elect(b_empty(sb));
            if (++sb == a.SB) { sb = 0; pb ^= 1; }
          }
          // input slice kd is done after tap block kd; the last block frees the remaining T slices
          if (kd < 2) {
            tcgen05_commit_elect(a_empty(s_first));
            if (++s_first == a.SA) s_first = 0;
          } else {
#pragma unroll
            for (int z = 0; z < T; ++z) {
              tcgen05_commit_elect(a_empty(s_first));
              if (++s_first == a.SA) s_first = 0;
            }
          }
        }
      }
      tcgen05_commit_elect(tmem_full(ab));
      loads_base += ncc * (T + 2);
    }
  } else {
    // ================= epilogue (warps 3-6) =================
    const int quarter = warp & 3;
    const int i = quarter * 32 + lane;            // accumulator row == TMEM lane
    const int th = i / a.PW, tw = i % a.PW;
    const int etid = tid - 96;                    // 0..127 inside the epilogue group
    const float isg = a.inv_sigma ? __ldg(a.inv_sigma) : 1.f;
    if (a.pred_w != nullptr) {
      for (int j = etid; j < 660; j += 128) s_pred[j] = j < 640 ? __ldg(a.pred_w + j) : __ldg(a.pred_b + (j - 640));
    }
    int cur_n_tile = -1;
    int iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
      const TileCoord tc = decode_tile(tile, a, T, n_tiles);
      if (tc.n_tile != cur_n_tile) {              // (re)stage the folded BatchNorm scale/shift of this channel tile
        asm volatile("bar.sync 1, 128;" ::: "memory");
        for (int j = etid; j < BN; j += 128) {
          s_scale[j] = __ldg(a.scale + tc.n_tile * BN + j) * isg;
          s_shift[j] = __ldg(a.shift + tc.n_tile * BN + j);
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        cur_n_tile = tc.n_tile;
      }
      const int ab = (NBUF == 2) ? (iter & 1) : 0;
      const int use = (NBUF == 2) ? (iter >> 1) : iter;
      mbar_wait(tmem_full(ab), (uint32_t)(use & 1), a.error_flag);
      __syncwarp();
      tcgen05_fence_after();
      halo_epilogue_slices<BN>(a, tc, n_tiles, tmem_acc + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ab * T * BN), 0, 1, T,
                               th, tw, s_scale, s_shift, s_pred);
      // this accumulator set may be overwritten by the MMAs of a later tile
      tcgen05_fence_before();
      mbar_arrive(tmem_empty(ab));
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"((uint32_t)Cfg::kTmemCols) : "memory");
  }
}

// fp32 (Cout, Cin_real, 3,3,3) -> bf16 [Cout/BN][cc][kd][kh*3+kw][BN][64] (rows swizzled); padded input
// channel p maps to a real channel through two segments (pad0/real0 | pad1/real1), zero elsewhere.
__global__ void pack_weights_halo_kernel(const float* __restrict__ w, int Cout, int cin_real, int BN, int pad0, int real0,
                                         int pad1, int real1, __nv_bfloat16* __restrict__ out) {
  const int ncc = (pad0 + pad1) / kBlockK;
  const size_t total = (size_t)Cout * 27 * ncc * kBlockK;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int e = (int)(i % 8);
    const int qs = (int)((i / 8) % 8);
    const int r = (int)((i / 64) % BN);
    size_t tile = i / ((size_t)64 * BN);        // ((n_tile*ncc + cc)*3 + kd)*9 + tap9
    const int tap9 = (int)(tile % 9); tile /= 9;
    const int kd = (int)(tile % 3); tile /= 3;
    const int cc = (int)(tile % ncc);
    const int n_tile = (int)(tile / ncc);
    const int q = qs ^ (r & 7);
    const int p = cc * kBlockK + q * 8 + e;      // padded input channel
    int c = -1;
    if (p < pad0) { if (p < real0) c = p; }
    else { const int p1 = p - pad0; if (p1 < real1) c = real0 + p1; }
    const int n = n_tile * BN + r;
    float v = 0.f;
    if (c >= 0) v = w[((size_t)n * cin_real + c) * 27 + kd * 9 + tap9];
    out[i] = __float2bfloat16_rn(v);
  }
}

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// stream-ordered upload of the prediction layer into constant memory (device pointers, fp32)
inline int load_pred_constants(const float* w_dev, const float* b_dev, cudaStream_t s) {
  V2CE_CUDA_CHECK(cudaMemcpyToSymbolAsync(c_pred, w_dev, 640 * sizeof(float), 0, cudaMemcpyDeviceToDevice, s));
  V2CE_CUDA_CHECK(cudaMemcpyToSymbolAsync(c_pred, b_dev, 20 * sizeof(float), 640 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return V2CE_OK;
}

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// tensor map over a (B, D, H, W, Cpitch) bf16 activation: box = 64 channels x PW x (TH+2) pixels
inline int make_patch_map(CUtensorMap* map, const void* ptr, int B, int D, int H, int W, int cpitch, int PW, int rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return set_error(V2CE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  // a tensor stored with fewer than 64 channels per pixel is presented as overlapping 64-channel rows (the upper
  // part of a row is the next pixel): the box row stays a full 128-byte swizzle row, the kernels skip those K steps
  const int cview = cpitch < 64 ? 64 : cpitch;
  cuuint64_t dims[5] = {(cuuint64_t)cview, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[4] = {(cuuint64_t)cpitch * 2, (cuuint64_t)W * cpitch * 2, (cuuint64_t)H * W * cpitch * 2,
                           (cuuint64_t)D * H * W * cpitch * 2};
  cuuint32_t box[5] = {64u, (cuuint32_t)PW, (cuuint32_t)rows, 1u, 1u};
  cuuint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(V2CE_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return V2CE_OK;
}

// The head conv's input: 8-channel (16-byte) split-bf16 pixels.  Presented as overlapping 16-channel rows (the upper
// half is the next pixel and meets zero weights) in a SWIZZLE_32B box: one K=16 step per tap reads exactly one 32-byte
// row.  The 64-channel presentation of the same tensor moved 8x its bytes from L2 to shared memory (1.39 GB per
// forward, the TMA producer was what the head waited for: 0.39 ms, profiles/ncu_kdm_r2_c.txt).
inline int make_patch_map16(CUtensorMap* map, const void* ptr, int B, int D, int H, int W, int PW, int rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return set_error(V2CE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  const int cpitch = 8;
  const cuuint64_t Wp = (cuuint64_t)W + 1;          // rows are stored with one more (zero) pixel, see head_prep_kernel
  cuuint64_t dims[5] = {16u, Wp, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[4] = {(cuuint64_t)cpitch * 2, Wp * cpitch * 2, (cuuint64_t)H * Wp * cpitch * 2,
                           (cuuint64_t)D * H * Wp * cpitch * 2};
  cuuint32_t box[5] = {16u, (cuuint32_t)PW, (cuuint32_t)rows, 1u, 1u};
  cuuint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(V2CE_ERR_CUDA, "cuTensorMapEncodeTiled (16-channel view) failed with CUresult %d", (int)r);
  return V2CE_OK;
}

struct TileShape { int PW, TH; };
// pitch / rows per tile for an output plane of H x W (see file header); chosen to maximise the useful
// fraction of the 128 accumulator rows
inline TileShape pick_tile(int H, int W) {
  TileShape best{16, 8};
  double best_eff = 0.0;
  for (int pw = 10; pw <= 66; pw += 2) {
    const int tw = pw - 2, th = 128 / pw;
    if (th < 1) continue;
    const long tiles = (long)((W + tw - 1) / tw) * ((H + th - 1) / th);
    const double eff = (double)H * W / (tiles * 128.0);
    // prefer the smaller patch (less halo re-read) unless a wider one is clearly more efficient
    if (eff > best_eff + 0.01) { best_eff = eff; best = TileShape{pw, th}; }
  }
  return best;
}

struct HaloPlan {
  TileShape ts;
  int T, SA, SB, a_stage_bytes, box_bytes, smem_bytes;
};

inline HaloPlan plan_for(int bn, int D, int H, int W) {
  HaloPlan p;
  p.ts = pick_tile(H, W);
  const int rows = p.ts.PW * (p.ts.TH + 2);
  p.box_bytes = rows * 128;
  p.a_stage_bytes = ((rows + 2 + 7) / 8) * 1024;
  const int tail = (2 * kMaxSA + 2 * kMaxSB + 4) * 8 + 16 + 2 * bn * 4 + 660 * 4;
  const int budget = 227 * 1024 - 1024 - tail;
  const int b_stage = bn * kBlockK * 2;
  // depth blocking T and ring depths.  A chunk needs T patches before its first tap and holds T+2 over its
  // lifetime; the ring must be deep enough to prefetch the next chunk's first patches (SA >= T + 2 + T/2 would
  // be ideal), which T = 2 allows within 227 KB while T = 4 does not.
  p.T = bn <= 64 ? 4 : 2;   // measured: T=4 wins for N<=64, T=2 (double-buffered TMEM) for N=128
  while (p.T > 1 && (D % p.T != 0)) p.T /= 2;
  for (;; p.T /= 2) {
    p.SB = bn <= 32 ? 8 : bn <= 64 ? 6 : bn <= 128 ? 4 : 3;
    p.SA = kMaxSA;
    while (p.SA > p.T + 1 && p.SA * p.a_stage_bytes + p.SB * b_stage > budget) --p.SA;
    while (p.SB > 2 && p.SA * p.a_stage_bytes + p.SB * b_stage > budget) --p.SB;
    if (p.SA * p.a_stage_bytes + p.SB * b_stage <= budget || p.T == 1) break;
  }
  p.smem_bytes = p.SA * p.a_stage_bytes + p.SB * b_stage + tail + 1024;
  return p;
}

template <int BN, int T>
inline int launch_halo_one(const CUtensorMap& tm0, const CUtensorMap& tm1, const HaloArgs& a, int smem_bytes, cudaStream_t s) {
  static int configured[64] = {0};
  const int slot = device_slot();
  if (configured[slot] < smem_bytes) {
    V2CE_CUDA_CHECK(cudaFuncSetAttribute(conv_halo_kernel<BN, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    configured[slot] = smem_bytes;
  }
  const int total = a.B * (a.D / T) * a.tiles_h * a.tiles_w * (a.Cout / BN);
  int per_sm = 1;                                   // resident CTAs per SM (shared memory bound)
  if (2 * (smem_bytes + 1024) <= 227 * 1024 && 2 * HaloCfg<BN, T>::kTmemCols <= 512) per_sm = 2;
  const int grid = total < sm_count_cached() * per_sm ? total : sm_count_cached() * per_sm;
  conv_halo_kernel<BN, T><<<grid, kHaloThreads, smem_bytes, s>>>(tm0, tm1, a);
  V2CE_LAUNCH_CHECK("conv_halo_kernel");
  return V2CE_OK;
}

template <int BN>
inline int launch_halo_bn(const CUtensorMap& tm0, const CUtensorMap& tm1, const HaloArgs& a, int smem_bytes, cudaStream_t s) {
  if constexpr (BN <= 128) {
    if (a.T == 4) return launch_halo_one<BN, 4>(tm0, tm1, a, smem_bytes, s);
  }
  if (a.T == 2) return launch_halo_one<BN, 2>(tm0, tm1, a, smem_bytes, s);
  if (a.T == 1) return launch_halo_one<BN, 1>(tm0, tm1, a, smem_bytes, s);
  return set_error(V2CE_ERR_INVALID, "unsupported depth blocking T=%d for N tile %d", a.T, BN);
}

inline int launch_halo(const CUtensorMap& tm0, const CUtensorMap& tm1, const HaloArgs& a, int bn, int smem_bytes,
                       cudaStream_t s) {
  switch (bn) {
    case 32: return launch_halo_bn<32>(tm0, tm1, a, smem_bytes, s);
    case 64: return launch_halo_bn<64>(tm0, tm1, a, smem_bytes, s);
    case 128: return launch_halo_bn<128>(tm0, tm1, a, smem_bytes, s);
    case 256: return launch_halo_bn<256>(tm0, tm1, a, smem_bytes, s);
  }
  return set_error(V2CE_ERR_INVALID, "unsupported N tile %d", bn);
}

}  // namespace halo
}  // namespace v2ce
