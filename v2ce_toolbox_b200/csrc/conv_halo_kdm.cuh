// Halo-tile Conv3d (3x3x3, stride 1, pad 1) with the three depth taps merged into the MMA's N dimension, for
// layers with few output channels (N tile = 32), optionally with the block's 1x1x1 shortcut conv fused in.
//
// Why: tcgen05.mma with both operands in shared memory reads 128 rows of A and N rows of B (32 bytes each) per
// K=16 step; the shared-memory port moves 128 B/clk, so one step costs max(N/2, (128+N)/4) cycles
// (tools/mma_rate.py on B200: N=32 44.7, N=64 50.2, N=96 56.3, N=128 64, N=256 128).  At N=32 the tensor pipe is
// therefore busy 36 % of the time at best: the A operand is re-read for every 32 output channels.
//
// Input slice z under depth tap kd contributes to output slice z-kd+1 AT THE SAME accumulator rows.  With the
// accumulators of consecutive output slices in consecutive TMEM column blocks, ONE instruction of N = 3*32 = 96
//     D[:, (z-1 .. z+1) * 32 ..] += A_z(tap kh,kw) x [W(kd=2); W(kd=1); W(kd=0)]^T
// does the work of three, for one read of A: 56 cycles instead of 134.  Slices outside the CTA's depth block
// are dropped by shrinking N and offsetting the B descriptor by whole 32-row blocks; the first touch of an
// accumulator block (output slice z+1 at input slice z) is one extra N=32 instruction without the accumulate flag.
//
// Loop order per tile (spatial tile x T=8 output slices x 32 channels): channel chunk -> input slice -> 9 taps.
// The nine [3 kd][32][64] weight tiles of a chunk stay resident in shared memory (108 KB) while the T+2 input
// patches stream through a TMA ring; every patch is multiplied exactly once.  Depth slices -1 and D are zero
// padding and are skipped.
//
// Accumulator hand-off is per output slice: TMEM holds R slots of 32 columns, each with its own full/empty
// mbarrier.  Slice o is complete after input slice o+1 of the last chunk, so the epilogue (8 warps: two per TMEM
// lane quarter, alternate slices) drains it while later slices are still being multiplied, and frees the slot as
// soon as the values are in registers.  R = 16 (two tiles in flight) without the shortcut; with it, R = 8 and the
// other 256 columns hold the shortcut accumulators.
//
// Fused shortcut (SHORT): ResidualBlock3D's downsample branch bn_d(conv_d(x)) (submodules.py:244-247,259) is a
// 1x1x1 conv of the SAME input, i.e. the centre tap's A operand times a second weight tile: one extra N=32
// instruction per K step of the centre tap (+9 % tensor time) replaces a separate pass over the input
// (1.5 GB of reads at 346x260).  The epilogue writes both outputs.
//
// Layers with 64 output channels run as two N tiles of 32 (112 cycles per three taps instead of 150).
// Replaces the same reference calls as conv_halo.cuh (submodules.py:249-263).
#pragma once
#include "conv_halo.cuh"

namespace v2ce {
namespace halo {

constexpr int kKdmThreads = 384;      // warp 0 TMA patches, warp 1 weight tiles, warp 2 MMA issue, warp 3 idle, warps 4-11 epilogue
constexpr int kKdmBN = 32;
constexpr int kKdmT = 8;
constexpr int kKdmWTile = 3 * kKdmBN * kBlockK * 2;   // bytes of one (chunk, tap) weight tile: [3][32][64] bf16
constexpr int kKdmSTile = kKdmBN * kBlockK * 2;       // bytes of one (chunk) shortcut weight tile: [32][64] bf16
constexpr int kKdmWSlots = 10;                        // 9 taps + shortcut
constexpr int kKdmBars = 2 * kMaxSA + 2 * kKdmWSlots + 32;

// second output of the fused kernel (the block's shortcut branch)
struct KdmShort {
  const __nv_bfloat16* wpack;  // [Cout/32][ncc][32][64], rows pre-swizzled
  const float* scale;          // folded BatchNorm of the shortcut (bias included in shift)
  const float* shift;
  __nv_bfloat16* out;          // (B,D,H,W,out_pitch)
  int out_pitch;
};

// One 32-column accumulator chunk of one pixel row: y = act(acc*scale + shift (+ residual)) -> bf16 store (plain or
// nearest-upsampled) or the fused prediction layer.  `v` holds the raw accumulators.
struct KdmRow {
  size_t pix, HWp;
  int uh0, uh1, uw0, uw1;
  bool ok;
};

__device__ __forceinline__ void kdm_store_chunk(const HaloArgs& a, const KdmRow& r, const uint32_t (&v)[32], const uint4 (&rv)[4],
                                                const float* s_scale, const float* s_shift, int act, size_t plane, int n0,
                                                __nv_bfloat16* out, int out_pitch, int cout, bool main_out) {
  // scale / shift come in as 16-byte shared-memory loads (16 instead of 64 scalar ones): the epilogue warps are few
  // (two per scheduler) and issue-latency bound, every instruction saved shortens the slice (profiles/ncu_kdm_r2_c.txt)
  float yv[32];
  const float4* sc4 = reinterpret_cast<const float4*>(s_scale);
  const float4* sh4 = reinterpret_cast<const float4*>(s_shift);
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const __nv_bfloat162* rp2 = reinterpret_cast<const __nv_bfloat162*>(&rv[g]);
    const float4 sa = sc4[2 * g], sb = sc4[2 * g + 1], ta = sh4[2 * g], tb = sh4[2 * g + 1];
    const float sc[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
    const float sh[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __bfloat1622float2(rp2[j]);      // zeros when there is no residual
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int n = g * 8 + 2 * j + hh;
        float tv = fmaf(__uint_as_float(v[n]), sc[2 * j + hh], sh[2 * j + hh]) + (hh ? f.y : f.x);
        if (act == 1) tv = fmaxf(tv, 0.f);
        else if (act == 2) tv = fmaxf(tv, 0.01f * tv);  // LeakyReLU(0.01): max(x, 0.01 x)
        yv[n] = tv;
      }
    }
  }
  if (main_out && a.pred_w != nullptr) {
    // fused prediction layer (see conv_halo.cuh): weights are FFMA constant-bank operands
    float* dst = a.pred_out + plane * 20 * r.HWp + r.pix;
#pragma unroll
    for (int m0 = 0; m0 < 20; m0 += 4) {
      float acc[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[u] = c_pred[640 + m0 + u];
#pragma unroll
      for (int c = 0; c < 32; ++c) {
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[u] = fmaf(yv[c], c_pred[(m0 + u) * 32 + c], acc[u]);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) dst[(size_t)(m0 + u) * r.HWp] = fmaxf(acc[u], 0.f);
    }
    return;
  }
  uint4 ov[4];
  __nv_bfloat162* op = reinterpret_cast<__nv_bfloat162*>(ov);
#pragma unroll
  for (int j = 0; j < 16; ++j) op[j] = __floats2bfloat162_rn(yv[2 * j], yv[2 * j + 1]);
  if (main_out && a.up_H > 0) {
    for (int hh = r.uh0; hh < r.uh1; ++hh)
      for (int ww = r.uw0; ww < r.uw1; ++ww) {
        uint4* d4 = reinterpret_cast<uint4*>(out + ((plane * a.up_H + hh) * a.up_W + ww) * out_pitch + n0);
#pragma unroll
        for (int g = 0; g < 4; ++g) d4[g] = ov[g];
      }
    return;
  }
  __nv_bfloat16* row = out + (plane * r.HWp + r.pix) * out_pitch;
  uint4* d4 = reinterpret_cast<uint4*>(row + n0);
#pragma unroll
  for (int g = 0; g < 4; ++g) d4[g] = ov[g];
  if (n0 + 32 == cout) {
    // zero the padding channels so later TMA reads see 0, not garbage
    for (int c = cout; c < out_pitch; c += 8) *reinterpret_cast<uint4*>(row + c) = make_uint4(0u, 0u, 0u, 0u);
  }
}

// S = 2: stride (1,2,2).  A stride-2 3x3 conv is the sum of four stride-1 convs on the even/odd sub-images
// X_pq[i][j] = X[2i+p][2j+q] (2x2, 2x1, 1x2 and 1x1 taps), and TMA addresses each sub-image as a strided view of the
// same tensor (ParityMaps), zero fill at its borders = the conv padding.  Per input slice the CTA loads four parity
// patches of (TH+1) x PW pixels (PW = TW+1) and multiplies each by its taps through row-shifted descriptors:
//   q = 2p+q':  0 (even,even): tap (1,1)        1 (even row, odd col): (1,0), (1,2)+1
//               2 (odd row, even col): (0,1), (2,1)+PW     3 (odd,odd): (0,0), (0,2)+1, (2,0)+PW, (2,2)+PW+1
// so the input is read once (plus halo) instead of once per tap (the gather kernel moved 5.3 GB through L2 for
// encoders.0.conv1).  The block's stride-2 1x1x1 shortcut is the (1,1) tap, fused as in the stride-1 case.
struct ParityMaps { CUtensorMap m[4]; };

template <int N>
struct KdmInt { static constexpr int value = N; };

// taps in the order the stride-2 variant multiplies them
__device__ __constant__ int kS2TapOrder[9] = {4, 3, 5, 1, 7, 0, 2, 6, 8};

template <bool SHORT, int T, int S>
__global__ void __launch_bounds__(kKdmThreads) conv_halo_kdm_kernel(const __grid_constant__ CUtensorMap tm0,
                                                                     const __grid_constant__ CUtensorMap tm1,
                                                                     const __grid_constant__ ParityMaps pm,
                                                                     const HaloArgs a, const KdmShort sc) {
  // T output slices per tile: 8, or the whole depth of a 16-slice window (no depth halo: 16 patch loads per 16
  // output slices instead of 20, and fewer narrow edge instructions) when the shortcut does not need half of TMEM
  constexpr int BN = kKdmBN;
  static_assert(T == 8 || (T == 16 && !SHORT), "slots");
  constexpr int G = SHORT ? 1 : 16 / T;             // tiles whose accumulators fit in TMEM at once
  constexpr uint32_t kShortCols = 256;              // shortcut accumulator of slot s: column 256 + 32 s
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);

  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31;
  const int n_tiles = a.Cout / BN;
  const int total_tiles = a.B * (a.D / T) * a.tiles_h * a.tiles_w * n_tiles;
  const int ncc = a.ncc0 + a.ncc1;

  const uint32_t w_base = base;                                   // 9 resident tap tiles + the shortcut tile
  const uint32_t ws_base = base + 9u * kKdmWTile;
  const uint32_t a_base = ws_base + kKdmSTile;                    // patch ring
  const uint32_t bar_base = a_base + (uint32_t)a.SA * a.a_stage_bytes;
  auto a_full = [&](int s) { return bar_base + 8u * s; };
  auto a_empty = [&](int s) { return bar_base + 8u * (kMaxSA + s); };
  auto w_full = [&](int s) { return bar_base + 8u * (2 * kMaxSA + s); };
  auto w_empty = [&](int s) { return bar_base + 8u * (2 * kMaxSA + kKdmWSlots + s); };
  auto s_full = [&](int s) { return bar_base + 8u * (2 * kMaxSA + 2 * kKdmWSlots + s); };
  auto s_empty = [&](int s) { return bar_base + 8u * (2 * kMaxSA + 2 * kKdmWSlots + 16 + s); };
  uint8_t* tail = smem + (bar_base - base) + kKdmBars * 8;
  volatile uint32_t* tmem_ptr = reinterpret_cast<volatile uint32_t*>(tail);
  float* s_scale = reinterpret_cast<float*>(tail + 16);           // main scale | main shift | shortcut scale | shortcut shift
  float* s_shift = s_scale + BN;
  float* s_scale2 = s_shift + BN;
  float* s_shift2 = s_scale2 + BN;

  if (tid == 0) {
    for (int s = 0; s < a.SA; ++s) { mbar_init(a_full(s), 1); mbar_init(a_empty(s), 1); }
    for (int s = 0; s < kKdmWSlots; ++s) { mbar_init(w_full(s), 1); mbar_init(w_empty(s), 1); }
    for (int s = 0; s < 16; ++s) { mbar_init(s_full(s), 1); mbar_init(s_empty(s), 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(const_cast<uint32_t*>(tmem_ptr))),
                 "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_acc = *tmem_ptr;

  // input slices a tile multiplies: d0-1 .. d0+T, minus the zero-padding slices -1 and D
  auto z_lo = [&](int d0) { return d0 > 0 ? d0 - 1 : 0; };
  auto z_hi = [&](int d0) { return d0 + T < a.D ? d0 + T : a.D - 1; };

  if (warp == 0) {
    // ================= patch producer (TMA) =================
    int s = 0, ph = 1;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(tile, a, T, n_tiles);
      const int zl = z_lo(tc.d0), zh = z_hi(tc.d0);
      for (int cc = 0; cc < ncc; ++cc) {
        const bool first = cc < a.ncc0;
        const CUtensorMap* map = first ? &tm0 : &tm1;
        const int c0 = (first ? cc : cc - a.ncc0) * kBlockK;
        for (int z = zl; z <= zh; ++z) {
          if (S == 1) {
            mbar_wait(a_empty(s), (uint32_t)ph, a.error_flag);
            if (elect_one()) {
              mbar_arrive_expect_tx(a_full(s), (uint32_t)a.box_bytes);
              tma_load_5d(a_base + (uint32_t)s * a.a_stage_bytes, map, c0, tc.w0 - 1, tc.h0 - 1, z, tc.b, a_full(s));
            }
            __syncwarp();
            if (++s == a.SA) { s = 0; ph ^= 1; }
          } else {
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {           // parity patch q = 2*(row parity) + (column parity)
              mbar_wait(a_empty(s), (uint32_t)ph, a.error_flag);
              if (elect_one()) {
                mbar_arrive_expect_tx(a_full(s), (uint32_t)a.box_bytes);
                tma_load_5d(a_base + (uint32_t)s * a.a_stage_bytes, &pm.m[q], c0, tc.w0 - (q & 1), tc.h0 - (q >> 1), z, tc.b,
                            a_full(s));
              }
              __syncwarp();
              if (++s == a.SA) { s = 0; ph ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= weight-tile producer: slot = tap (9 = shortcut), refilled once per (tile, chunk) =================
    // With a single channel chunk the resident tiles only change with the N tile (the slowest tile coordinate):
    // they are then loaded once and reused by every following tile instead of being re-fetched per tile, which left
    // the MMA warp waiting for a 108 KB reload at every tile start.
    uint32_t ph = 1;
    int loaded_n_tile = -1;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(tile, a, T, n_tiles);
      for (int cc = 0; cc < ncc; ++cc) {
        if (ncc == 1 && tc.n_tile == loaded_n_tile) continue;
        loaded_n_tile = tc.n_tile;
        const __nv_bfloat16* wt = a.wpack + (size_t)(tc.n_tile * ncc + cc) * 9 * (kKdmWTile / 2);
        for (int ti = 0; ti < 9; ++ti) {
          const int tap = (S == 1) ? ti : kS2TapOrder[ti];      // refill in the order the slots are freed
          mbar_wait(w_empty(tap), ph, a.error_flag);
          if (elect_one()) {
            mbar_arrive_expect_tx(w_full(tap), (uint32_t)kKdmWTile);
            bulk_copy_g2s(w_base + (uint32_t)tap * kKdmWTile, wt + (size_t)tap * (kKdmWTile / 2), (uint32_t)kKdmWTile, w_full(tap));
          }
          __syncwarp();
        }
        if (SHORT) {
          mbar_wait(w_empty(9), ph, a.error_flag);
          if (elect_one()) {
            mbar_arrive_expect_tx(w_full(9), (uint32_t)kKdmSTile);
            bulk_copy_g2s(ws_base, sc.wpack + (size_t)(tc.n_tile * ncc + cc) * (kKdmSTile / 2), (uint32_t)kKdmSTile, w_full(9));
          }
          __syncwarp();
        }
        ph ^= 1u;
      }
    }
  } else if (warp == 2) {
    // ================= MMA issuer =================
    int sa = 0, pa = 0;                             // patch ring position / parity
    uint32_t pw = 0;                                // parity of the weight slots for the current load generation
    uint32_t pw_next = 0;
    int loaded_n_tile = -1;
    const uint32_t px16 = (uint32_t)a.a_row16;      // one patch pixel in descriptor units (16 B): 8, or 2 for the head's 32-byte rows
    const uint32_t pw8 = (uint32_t)a.PW * px16;     // one patch row of pixels
    const uint32_t a_hi = a.a_desc_hi;
    const uint32_t tap_mask = (uint32_t)a.tap_mask;
    const uint32_t idesc32 = make_idesc(BN);
    int iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
      const TileCoord tc = decode_tile(tile, a, T, n_tiles);
      const int zl = z_lo(tc.d0), zh = z_hi(tc.d0);
      const int slot0 = (iter % G) * T;
      const uint32_t par_empty = (uint32_t)(((iter / G) & 1) ^ 1);
      const uint32_t acc_base = tmem_acc + (uint32_t)(slot0 * BN);
      for (int cc = 0; cc < ncc; ++cc) {
        // channels beyond the real ones (the upper half of a 32-channel tensor's 64-channel rows) are not multiplied
        const int rem = (cc < a.ncc0) ? (a.real0 - cc * kBlockK) : (a.real1 - (cc - a.ncc0) * kBlockK);
        const int ks = rem >= kBlockK ? kBlockK / 16 : (rem + 15) / 16;
        const bool last_cc = (cc == ncc - 1);
        // weight generations (see the producer): does this (tile, chunk) start a new one, and will the next one?
        const bool w_new = !(ncc == 1 && tc.n_tile == loaded_n_tile);
        loaded_n_tile = tc.n_tile;
        if (w_new) { pw = pw_next; pw_next ^= 1u; }
        bool w_release = true;
        if (ncc == 1) {
          const int nxt = tile + (int)gridDim.x;
          w_release = nxt < total_tiles && decode_tile(nxt, a, T, n_tiles).n_tile != tc.n_tile;
        }
#pragma unroll 1
        for (int z = zl; z <= zh; ++z) {
          // output slices z-1+j, j = 0..2 (depth tap kd = 2-j), clipped to the block [d0, d0+T)
          const int jlo = (z - 1 >= tc.d0) ? 0 : (tc.d0 - z + 1);
          const int jhi = (z + 1 <= tc.d0 + T - 1) ? 2 : (tc.d0 + T - z);
          const int o_lo = z - 1 + jlo - tc.d0;     // first covered slice, relative to the block
          const bool first_z = (z == zl), last_z = (z == zh);
          if (cc == 0) {
            // slices this input touches first must have been drained by the epilogue (slot reuse)
            const int f_lo = first_z ? o_lo : o_lo + (jhi - jlo), f_hi = (first_z || jhi == 2) ? o_lo + (jhi - jlo) : -1;
            for (int o = f_lo; o <= f_hi; ++o) mbar_wait(s_empty(slot0 + o), par_empty, a.error_flag);
          }
          const uint32_t col = acc_base + (uint32_t)(o_lo * BN);
          const uint32_t n_all = (uint32_t)((jhi - jlo + 1) * BN);
          const uint32_t idesc_all = make_idesc((int)n_all);
          const uint32_t b_lo = smem_desc_lo(w_base + (uint32_t)jlo * (BN * 128));
          // one tap: all K=16 steps of A(rows shifted by a_t) x the tap's [kd-merged] weight tile; `lead` marks the
          // tile's very first instruction candidates (first tap in issue order)
          // KS = K=16 steps per tap as a compile-time constant: the MMA warp is what these kernels wait for (one warp
          // issues ~13 uniform-datapath instructions per tcgen05.mma at ~6.6 cycles each = 86 cycles against 56 on the
          // tensor pipe, profiles/ncu_kdm_r2_c.txt), and a per-step `k < ks` test was three of them.
          // EDGE = this input slice may be the first / last user of the chunk's weight tiles (waits for their arrival,
          // releases them); the slices in between carry neither test: two uniform compares and two branches per tap.
          auto issue_tap = [&](auto KS_, auto EDGE_, const int tap, const uint32_t a_t, const bool lead) {
            constexpr int KS = decltype(KS_)::value;
            constexpr bool EDGE = decltype(EDGE_)::value != 0;
            if (EDGE && first_z && w_new) {
              mbar_wait(w_full(tap), pw, a.error_flag);
              tcgen05_fence_after();
            }
            const uint32_t b_t = b_lo + (uint32_t)tap * (kKdmWTile >> 4);
#pragma unroll
            for (int k = 0; k < KS; ++k) {
              if (!lead || k != 0 || cc != 0) {
                tcgen05_mma_bf16_lo2(col, a_t + 2 * k, b_t + 2 * k, idesc_all, 1u, a_hi);
              } else if (first_z) {
                // first multiply into this tile's accumulators: nothing covered has been written yet
                tcgen05_mma_bf16_lo2(col, a_t, b_t, idesc_all, 0u, a_hi);
              } else {
                // slice z+1 (j = 2) is touched for the first time, the others accumulate
                const int j_old_hi = jhi < 1 ? jhi : 1;
                const uint32_t n_old = (uint32_t)((j_old_hi - jlo + 1) * BN);
                tcgen05_mma_bf16_lo2(col, a_t, b_t, make_idesc((int)n_old), 1u, a_hi);
                if (jhi == 2) tcgen05_mma_bf16_lo2(col + n_old, a_t, b_t + n_old * 8u, idesc32, 0u, a_hi);
              }
            }
            if (SHORT && tap == 4 && z >= tc.d0 && z < tc.d0 + T) {
              // shortcut conv of output slice z: centre tap of input slice z times the 1x1x1 weights
              if (EDGE && (first_z || z == tc.d0) && w_new) {   // first use of the shortcut tile in this chunk
                mbar_wait(w_full(9), pw, a.error_flag);
                tcgen05_fence_after();
              }
              const uint32_t scol = tmem_acc + kShortCols + (uint32_t)((slot0 + z - tc.d0) * BN);
              const uint32_t bs_lo = smem_desc_lo(ws_base);
#pragma unroll
              for (int k = 0; k < KS; ++k)
                tcgen05_mma_bf16_lo2(scol, a_t + 2 * k, bs_lo + 2 * k, idesc32, (cc != 0 || k != 0) ? 1u : 0u, a_hi);
            }
            if (EDGE && last_z && w_release) tcgen05_commit_elect(w_empty(tap));   // last use of this generation's tap tile
          };
          // all taps of one input slice (one patch, or the four parity patches of the stride-2 variant)
          auto issue_slice = [&](auto KS_, auto EDGE_) {
            constexpr int KS = decltype(KS_)::value;
            if (S == 1) {
              mbar_wait(a_full(sa), (uint32_t)pa, a.error_flag);
              tcgen05_fence_after();
              // descriptor low words of (tap 0, k 0); a tap adds (kh*PW + kw) pixel rows to A and one weight tile to
              // B, a K=16 step adds 32 B to both (fully unrolled: the issue loop must stay well under the 56 cycles
              // one N=96 instruction occupies the tensor pipe)
              const uint32_t a_lo = smem_desc_lo(a_base + (uint32_t)sa * a.a_stage_bytes);
#pragma unroll
              for (int tap = 0; tap < 9; ++tap)
                if (KS > 1 || ((tap_mask >> tap) & 1))          // only the head (one K step per tap) masks taps
                  issue_tap(KS_, EDGE_, tap, a_lo + (uint32_t)(tap / 3) * pw8 + (uint32_t)(tap % 3) * px16, tap == 0);
              tcgen05_commit_elect(a_empty(sa));
              if (++sa == a.SA) { sa = 0; pa ^= 1; }
            } else {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                mbar_wait(a_full(sa), (uint32_t)pa, a.error_flag);
                tcgen05_fence_after();
                const uint32_t a_lo = smem_desc_lo(a_base + (uint32_t)sa * a.a_stage_bytes);
                if (q == 0) {
                  issue_tap(KS_, EDGE_, 4, a_lo, true);
                } else if (q == 1) {
                  issue_tap(KS_, EDGE_, 3, a_lo, false);
                  issue_tap(KS_, EDGE_, 5, a_lo + px16, false);
                } else if (q == 2) {
                  issue_tap(KS_, EDGE_, 1, a_lo, false);
                  issue_tap(KS_, EDGE_, 7, a_lo + pw8, false);
                } else {
                  issue_tap(KS_, EDGE_, 0, a_lo, false);
                  issue_tap(KS_, EDGE_, 2, a_lo + px16, false);
                  issue_tap(KS_, EDGE_, 6, a_lo + pw8, false);
                  issue_tap(KS_, EDGE_, 8, a_lo + pw8 + px16, false);
                }
                tcgen05_commit_elect(a_empty(sa));
                if (++sa == a.SA) { sa = 0; pa ^= 1; }
              }
            }
          };
          const bool edge = first_z || last_z || (SHORT && z == tc.d0);
          if (edge) {
            if (ks == 4) issue_slice(KdmInt<4>{}, KdmInt<1>{});
            else if (ks == 2) issue_slice(KdmInt<2>{}, KdmInt<1>{});
            else if (ks == 1) issue_slice(KdmInt<1>{}, KdmInt<1>{});
            else issue_slice(KdmInt<3>{}, KdmInt<1>{});
          } else {
            if (ks == 4) issue_slice(KdmInt<4>{}, KdmInt<0>{});
            else if (ks == 2) issue_slice(KdmInt<2>{}, KdmInt<0>{});
            else if (ks == 1) issue_slice(KdmInt<1>{}, KdmInt<0>{});
            else issue_slice(KdmInt<3>{}, KdmInt<0>{});
          }
          if (SHORT && last_z && w_release) tcgen05_commit_elect(w_empty(9));
          if (last_cc) {
            // output slice z-1 has received its last contribution; at the end of the depth range so has slice z
            if (z - 1 >= tc.d0) tcgen05_commit_elect(s_full(slot0 + z - 1 - tc.d0));
            if (last_z && z < tc.d0 + T) tcgen05_commit_elect(s_full(slot0 + z - tc.d0));
          }
        }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue (warps 4-11) =================
    constexpr int kEpiThreads = kKdmThreads - 128;
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may read
    constexpr int kParts = kEpiThreads / 128;     // warps per lane quarter: they take the block's slices round robin
    const int half = (warp - 4) >> 2;             // which of them this warp is
    const int i = quarter * 32 + lane;            // accumulator row == TMEM lane
    const int th = i / a.PW, tw = i % a.PW;
    const int etid = tid - 128;                   // 0..255 inside the epilogue group
    const float isg = a.inv_sigma ? __ldg(a.inv_sigma) : 1.f;
    const uint32_t lane_base = tmem_acc + ((uint32_t)(quarter * 32) << 16);
    int cur_n_tile = -1;
    int iter = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
      const TileCoord tc = decode_tile(tile, a, T, n_tiles);
      if (tc.n_tile != cur_n_tile) {              // (re)stage the folded BatchNorm scale/shift of this channel tile
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        for (int j = etid; j < BN; j += kEpiThreads) {
          s_scale[j] = __ldg(a.scale + tc.n_tile * BN + j) * isg;
          s_shift[j] = __ldg(a.shift + tc.n_tile * BN + j);
          if (SHORT) {
            s_scale2[j] = __ldg(sc.scale + tc.n_tile * BN + j);
            s_shift2[j] = __ldg(sc.shift + tc.n_tile * BN + j);
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        cur_n_tile = tc.n_tile;
      }
      const int slot0 = (iter % G) * T;
      const uint32_t par_full = (uint32_t)((iter / G) & 1);
      const int h = tc.h0 + th, w = tc.w0 + tw;
      KdmRow r;
      r.ok = (th < a.TH) && (tw < a.TW) && (h < a.H) && (w < a.W);
      r.pix = (size_t)h * a.W + w;
      r.HWp = (size_t)a.H * a.W;
      r.uh0 = r.uh1 = r.uw0 = r.uw1 = 0;
      if (a.up_H > 0 && r.ok) {                   // destination rows/columns when the output is written nearest-upsampled
        r.uh0 = (h * a.up_H + a.H - 1) / a.H;  r.uh1 = ((h + 1) * a.up_H + a.H - 1) / a.H;
        r.uw0 = (w * a.up_W + a.W - 1) / a.W;  r.uw1 = ((w + 1) * a.up_W + a.W - 1) / a.W;
      }
      const size_t plane0 = (size_t)(tc.b * a.D + tc.d0);
      const int n0 = tc.n_tile * BN;
      const bool has_res = (a.residual != nullptr) && r.ok;
      auto res_ptr = [&](int tt) {
        return reinterpret_cast<const uint4*>(a.residual + ((plane0 + tt) * r.HWp + r.pix) * a.res_pitch + n0);
      };
      // the residual of the next slice is requested before the current one is processed
      uint4 rv[4] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
      if (has_res) {
        const uint4* rp = res_ptr(half);
#pragma unroll
        for (int g = 0; g < 4; ++g) rv[g] = __ldg(rp + g);
      }
#pragma unroll 1
      for (int tt = half; tt < T; tt += kParts) {
        const int slot = slot0 + tt;
        uint4 rn[4] = {rv[0], rv[1], rv[2], rv[3]};
        if (has_res && tt + kParts < T) {
          const uint4* rp = res_ptr(tt + kParts);
#pragma unroll
          for (int g = 0; g < 4; ++g) rn[g] = __ldg(rp + g);
        }
        mbar_wait(s_full(slot), par_full, a.error_flag);
        __syncwarp();
        tcgen05_fence_after();
        uint32_t v[32];
        tmem_ld_32x32b_x32(lane_base + (uint32_t)(slot * BN), v);
        tmem_ld_wait();
        if (!SHORT) {                              // values are in registers: the slot may be overwritten
          tcgen05_fence_before();
          mbar_arrive(s_empty(slot));
        }
        if (r.ok) kdm_store_chunk(a, r, v, rv, s_scale, s_shift, a.act, plane0 + tt, n0, a.out, a.out_pitch, a.Cout, true);
        if (SHORT) {
          tmem_ld_32x32b_x32(lane_base + kShortCols + (uint32_t)(slot * BN), v);
          tmem_ld_wait();
          tcgen05_fence_before();
          mbar_arrive(s_empty(slot));
          const uint4 zero[4] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
          if (r.ok) kdm_store_chunk(a, r, v, zero, s_scale2, s_shift2, 0, plane0 + tt, n0, sc.out, sc.out_pitch, a.Cout, false);
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) rv[g] = rn[g];
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(512u) : "memory");
  }
}

// fp32 (Cout, Cin_real, 3,3,3) -> bf16 [Cout/32][cc][kh*3+kw][j = 2-kd][32][64] (rows swizzled); channel padding as in
// pack_weights_halo_kernel
__global__ void pack_weights_kdm_kernel(const float* __restrict__ w, int Cout, int cin_real, int pad0, int real0, int pad1,
                                        int real1, __nv_bfloat16* __restrict__ out) {
  constexpr int BN = kKdmBN;
  const int ncc = (pad0 + pad1) / kBlockK;
  const size_t total = (size_t)Cout * 27 * ncc * kBlockK;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int e = (int)(i % 8);
    const int qs = (int)((i / 8) % 8);
    const int r = (int)((i / 64) % BN);
    size_t tile = i / ((size_t)64 * BN);        // ((n_tile*ncc + cc)*9 + tap9)*3 + j
    const int j = (int)(tile % 3); tile /= 3;
    const int tap9 = (int)(tile % 9); tile /= 9;
    const int cc = (int)(tile % ncc);
    const int n_tile = (int)(tile / ncc);
    const int kd = 2 - j;
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

// fp32 (Cout, Cin_real) 1x1x1 weights -> bf16 [Cout/32][cc][32][64] (rows swizzled), same channel padding
__global__ void pack_weights_kdm_short_kernel(const float* __restrict__ w, int Cout, int cin_real, int pad0, int real0, int pad1,
                                              int real1, __nv_bfloat16* __restrict__ out) {
  constexpr int BN = kKdmBN;
  const int ncc = (pad0 + pad1) / kBlockK;
  const size_t total = (size_t)Cout * ncc * kBlockK;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int e = (int)(i % 8);
    const int qs = (int)((i / 8) % 8);
    const int r = (int)((i / 64) % BN);
    const size_t tile = i / ((size_t)64 * BN);   // n_tile*ncc + cc
    const int cc = (int)(tile % ncc);
    const int n_tile = (int)(tile / ncc);
    const int q = qs ^ (r & 7);
    const int p = cc * kBlockK + q * 8 + e;      // padded input channel
    int c = -1;
    if (p < pad0) { if (p < real0) c = p; }
    else { const int p1 = p - pad0; if (p1 < real1) c = real0 + p1; }
    const int n = n_tile * BN + r;
    out[i] = __float2bfloat16_rn(c >= 0 ? w[(size_t)n * cin_real + c] : 0.f);
  }
}

struct KdmPlan {
  TileShape ts;          // PW (patch pitch) and TH (output rows per tile)
  int TW;                // valid output columns per tile: PW - 2 (stride 1) or PW - 1 (stride 2)
  int rows;              // rows of one TMA box: (TH+2)*PW or (TH+1)*PW
  int SA, a_stage_bytes, box_bytes, smem_bytes;
  bool ok;
};

// tile shape for the stride-2 variant over an OUTPUT plane of H x W: one halo column (PW = TW+1), TH*PW <= 128
inline TileShape pick_tile_s2(int H, int W) {
  TileShape best{16, 8};
  double best_eff = 0.0;
  for (int pw = 8; pw <= 64; pw += 1) {
    const int tw = pw - 1, th = 128 / pw;
    if (th < 1) continue;
    const long tiles = (long)((W + tw - 1) / tw) * ((H + th - 1) / th);
    const double eff = (double)H * W / (tiles * 128.0);
    if (eff > best_eff + 0.01) { best_eff = eff; best = TileShape{pw, th}; }
  }
  return best;
}

// the kernel applies to depth multiples of 8 and needs room for at least 3 patch stages beside the weights;
// H, W = output plane
inline KdmPlan plan_kdm(int D, int H, int W, int stride = 1, int row_bytes = 128) {
  KdmPlan p;
  if (stride == 2) {
    p.ts = pick_tile_s2(H, W);
    p.TW = p.ts.PW - 1;
    p.rows = p.ts.PW * (p.ts.TH + 1);
  } else {
    p.ts = pick_tile(H, W);
    p.TW = p.ts.PW - 2;
    p.rows = p.ts.PW * (p.ts.TH + 2);
  }
  p.box_bytes = p.rows * row_bytes;
  p.a_stage_bytes = ((p.rows + 2) * row_bytes + 1023) / 1024 * 1024;
  const int tail = kKdmBars * 8 + 16 + 4 * kKdmBN * 4;
  const int budget = 227 * 1024 - 1024 - tail - 9 * kKdmWTile - kKdmSTile;
  p.SA = budget / p.a_stage_bytes;
  if (p.SA > kMaxSA) p.SA = kMaxSA;
  p.ok = (D % kKdmT == 0) && p.SA >= (stride == 2 ? 4 : 3);
  p.smem_bytes = 9 * kKdmWTile + kKdmSTile + p.SA * p.a_stage_bytes + tail + 1024;
  return p;
}

// tensor map over the parity sub-image X[2i+ph][2j+pw] of a (B, D, H, W, Cpitch) bf16 activation: the same memory
// with doubled row / pixel strides; box = 64 channels x PW x rows pixels
inline int make_parity_map(CUtensorMap* map, const void* ptr, int B, int D, int H, int W, int cpitch, int ph, int pw, int PW,
                           int rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return set_error(V2CE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  const int Hp = (H - ph + 1) / 2, Wq = (W - pw + 1) / 2;
  if (Hp < 1 || Wq < 1) return set_error(V2CE_ERR_INVALID, "stride-2 conv needs at least 2x2 input pixels");
  const int cview = cpitch < 64 ? 64 : cpitch;   // overlapping 64-channel rows over a denser tensor, see make_patch_map
  cuuint64_t dims[5] = {(cuuint64_t)cview, (cuuint64_t)Wq, (cuuint64_t)Hp, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[4] = {(cuuint64_t)2 * cpitch * 2, (cuuint64_t)2 * W * cpitch * 2, (cuuint64_t)H * W * cpitch * 2,
                           (cuuint64_t)D * H * W * cpitch * 2};
  cuuint32_t box[5] = {64u, (cuuint32_t)PW, (cuuint32_t)rows, 1u, 1u};
  cuuint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
  void* base = const_cast<char*>(static_cast<const char*>(ptr)) + ((size_t)ph * W + pw) * cpitch * 2;
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(V2CE_ERR_CUDA, "cuTensorMapEncodeTiled (parity view) failed with CUresult %d", (int)r);
  return V2CE_OK;
}

template <bool SHORT, int T, int S>
inline int launch_kdm_one(const CUtensorMap& tm0, const CUtensorMap& tm1, const ParityMaps& pm, const HaloArgs& a,
                          const KdmShort& sc, int smem_bytes, cudaStream_t s) {
  static int configured[64] = {0};
  const int slot = device_slot();
  if (configured[slot] < smem_bytes) {
    V2CE_CUDA_CHECK(cudaFuncSetAttribute(conv_halo_kdm_kernel<SHORT, T, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    configured[slot] = smem_bytes;
  }
  const int total = a.B * (a.D / T) * a.tiles_h * a.tiles_w * (a.Cout / kKdmBN);
  const int grid = total < sm_count_cached() ? total : sm_count_cached();
  conv_halo_kdm_kernel<SHORT, T, S><<<grid, kKdmThreads, smem_bytes, s>>>(tm0, tm1, pm, a, sc);
  V2CE_LAUNCH_CHECK("conv_halo_kdm_kernel");
  return V2CE_OK;
}

// `sc` != nullptr: also compute the block's 1x1x1 shortcut conv of the same input (second output).
// `pm` != nullptr: stride (1,2,2); a.H / a.W are the OUTPUT plane and pm the four parity views of the single source.
inline int launch_halo_kdm(const CUtensorMap& tm0, const CUtensorMap& tm1, const HaloArgs& a, const KdmShort* sc, int smem_bytes,
                           cudaStream_t s, const ParityMaps* pm = nullptr) {
  if (a.D % kKdmT != 0 || a.Cout % kKdmBN != 0)
    return set_error(V2CE_ERR_INVALID, "depth-merged halo kernel: depth %d / Cout %d not supported", a.D, a.Cout);
  if (sc && (a.up_H > 0 || a.pred_w != nullptr || a.residual != nullptr))
    return set_error(V2CE_ERR_INVALID, "depth-merged halo kernel: the fused shortcut goes with a plain first conv");
  if (pm && a.ncc1 != 0) return set_error(V2CE_ERR_INVALID, "depth-merged halo kernel: stride 2 takes a single source");
  const bool t16 = !sc && a.D % 16 == 0;
  HaloArgs b = a;
  b.T = t16 ? 16 : 8;
  const KdmShort none{nullptr, nullptr, nullptr, nullptr, 0};
  static const ParityMaps no_pm{};
  if (pm) {
    if (sc) return launch_kdm_one<true, 8, 2>(tm0, tm1, *pm, b, *sc, smem_bytes, s);
    if (t16) return launch_kdm_one<false, 16, 2>(tm0, tm1, *pm, b, none, smem_bytes, s);
    return launch_kdm_one<false, 8, 2>(tm0, tm1, *pm, b, none, smem_bytes, s);
  }
  if (sc) return launch_kdm_one<true, 8, 1>(tm0, tm1, no_pm, b, *sc, smem_bytes, s);
  if (t16) return launch_kdm_one<false, 16, 1>(tm0, tm1, no_pm, b, none, smem_bytes, s);
  return launch_kdm_one<false, 8, 1>(tm0, tm1, no_pm, b, none, smem_bytes, s);
}

}  // namespace halo
}  // namespace v2ce
