// Implicit-GEMM Conv3d for sm_100a: tcgen05.mma (kind::f16, bf16 x bf16 -> fp32 in TMEM),
// weights streamed by the bulk-copy engine (cp.async.bulk, pre-swizzled tiles), activations
// gathered by cp.async into the 128B-swizzled K-major layout, epilogue fused:
//     y = act( acc * scale[n] (* 1/sigma) + shift[n] (+ residual[m][n]) )  -> bf16 NDHWC
//
// Replaces the cuDNN/ATen calls behind /root/reference/scripts/submodules.py:116-122 (ConvLayer3D)
// and :249-263 (ResidualBlock3D.forward), plus the upsample+concat copies of
// /root/reference/scripts/unet_2layer.py:358-364, which are folded into the A-operand gather.
//
// GEMM view:  D[m][n] = sum_k A[m][k] * Wt[n][k]
//   m = output position (b, d, ho, wo)            tile: 128 rows  (UMMA M = 128, cta_group::1)
//   n = output channel                            tile: BN in {32, 64, 128, 256}
//   k = (tap, input channel), tap = (kd*3+kh)*3+kw, k-block = 64 bf16 = one 128-byte swizzle row
//
// CTA = 320 threads:
//   warps 0-7  A producers (8 lanes per 128-byte row, 4 x 16-byte cp.async per thread per k-block; the gather is
//              instruction bound, hence 8 warps), then the epilogue (warps w and w+4 read TMEM lanes
//              32(w%4).. with tcgen05.ld 32x32b and alternate 32-column chunks)
//   warp 8     TMEM allocator + MMA issuer (warp converged, elect.sync)
//   warp 9     weight-tile bulk copies
// Synchronisation: full[s] (128 cp.async.mbarrier.arrive.noinc arrivals + 1 expect_tx arrival), empty[s] (tcgen05.commit),
// tmem_full (tcgen05.commit after the last k-block).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace v2ce {
namespace conv {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                 // bf16 elements = 128 bytes
constexpr int kThreads = 320;
constexpr int kProducerThreads = 256;
constexpr int kAStageBytes = kBlockM * kBlockK * 2;

struct ConvArgs {
  const __nv_bfloat16* src0;   // (B,D,H0,W0,C0); nearest-upsampled to (Hin,Win) when H0 != Hin or W0 != Win
  const __nv_bfloat16* src1;   // (B,D,Hin,Win,C1) or nullptr
  int C0, C1, Cin;             // real channels gathered from each source; Cin = C0 + C1
  int P0, P1;                  // channel pitch (elements per pixel) of each source, >= C0 / C1
  int H0, W0;
  int B, D, Hin, Win, Hout, Wout;
  int stride, ksize, pad;
  int taps, num_kb;
  int M, Cout;
  const __nv_bfloat16* wpack;  // [Cout/BN][num_kb][BN][64], rows pre-swizzled (128B pattern)
  const float* scale;          // [Cout]
  const float* shift;          // [Cout]
  const float* inv_sigma;      // device scalar (spectral norm) or nullptr
  const __nv_bfloat16* residual;  // [M][Cout] or nullptr
  __nv_bfloat16* out;          // [M][Cout]
  int act;                     // 0 none, 1 relu, 2 leaky_relu(0.01)
  int* error_flag;             // set to 1 by the pipeline watchdog
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a broken pipeline traps (the host sees a launch failure) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* error_flag) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) {
      if (error_flag) atomicExch(error_flag, 1);
      __threadfence_system();
      __trap();
    }
  }
}
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tcgen05_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Warp-converged issue helpers.  The loops that feed the tensor core run with all 32 lanes converged so
// that nvcc keeps addresses and descriptors in uniform registers; the instruction that must execute
// once is predicated on elect.sync inside the asm block.  (Running those loops under `if (lane == 0)`
// cost ~150 cycles per tcgen05.mma in R2UR/ELECT round trips -- measured with ncu source counters.)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, e;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tcgen05_mma_bf16_elect(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                       uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same with the descriptors given by their low words only (start address >> 4 | LBO field): the high word of a
// K-major SWIZZLE_128B descriptor is the constant 0x40004040 (SBO = 1024 B, version 1, layout type 2), so an issue
// loop advances a descriptor with one 32-bit add instead of rebuilding 64 bits (the MMA warp of the N=32 kernels was
// instruction bound: ~100 uniform-datapath instructions per tap, ncu source counters).
__device__ __forceinline__ uint32_t smem_desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ void tcgen05_mma_bf16_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                                    uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t.reg .b64 da, db;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(0x40004040u)
      : "memory");
}
// A and B operands in different shared-memory layouts: `a_hi` is the high word of A's descriptor
// (0x40004040 = K-major SWIZZLE_128B, SBO 1024 B; 0xC0004010 = K-major SWIZZLE_32B, SBO 256 B), B stays SWIZZLE_128B
__device__ __forceinline__ void tcgen05_mma_bf16_lo2(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                                     uint32_t accumulate, uint32_t a_hi) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t.reg .b64 da, db;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %6};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(0x40004040u), "r"(a_hi)
      : "memory");
}
__device__ __forceinline__ void tcgen05_commit_elect(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar)
      : "memory");
}
__device__ __forceinline__ int uniform_warp_id() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major, SWIZZLE_128B: rows of 128 bytes, 8-row groups 1024 bytes
// apart (SBO), LBO unused (1), descriptor version 1 (sm_100), layout type 2.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor: D=f32 (bit 4), A=B=bf16 (bits 7,10), both K-major, N>>3 at bit 17, M>>4 at bit 24.
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kBlockM >> 4) << 24);
}

template <int BN, int STAGES>
struct SmemLayout {
  static constexpr int kBStageBytes = BN * kBlockK * 2;
  static constexpr int kAOff = 0;
  static constexpr int kBOff = STAGES * kAStageBytes;
  static constexpr int kBarOff = kBOff + STAGES * kBStageBytes;      // full[STAGES], empty[STAGES], tmem_full
  static constexpr int kTmemPtrOff = kBarOff + (2 * STAGES + 1) * 8;
  static constexpr int kScaleOff = (kTmemPtrOff + 4 + 15) / 16 * 16;
  static constexpr int kShiftOff = kScaleOff + BN * 4;
  static constexpr int kRowsOff = kShiftOff + BN * 4;                // 3 x 128 ints: per-row gather descriptors
  static constexpr int kTotal = kRowsOff + 3 * 128 * 4;
  static constexpr int kDynamicBytes = kTotal + 1024;                // slack for the 1024-byte alignment
};

template <int BN, int STAGES>
__global__ void __launch_bounds__(kThreads) conv_igemm_kernel(const ConvArgs a) {
  using L = SmemLayout<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);

  const int tid = threadIdx.x;
  const int warp = uniform_warp_id(), lane = tid & 31;
  const int n_tiles = a.Cout / BN;
  const int n_tile = blockIdx.x % n_tiles;
  const int m_tile = blockIdx.x / n_tiles;

  const uint32_t a_base = base + L::kAOff;
  const uint32_t b_base = base + L::kBOff;
  const uint32_t bar_base = base + L::kBarOff;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * STAGES);
  volatile uint32_t* tmem_ptr = reinterpret_cast<volatile uint32_t*>(smem + L::kTmemPtrOff);
  float* s_scale = reinterpret_cast<float*>(smem + L::kScaleOff);
  float* s_shift = reinterpret_cast<float*>(smem + L::kShiftOff);
  int* s_rows = reinterpret_cast<int*>(smem + L::kRowsOff);

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), kProducerThreads + 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(const_cast<uint32_t*>(tmem_ptr))),
                 "r"((uint32_t)BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  {
    const float isg = a.inv_sigma ? __ldg(a.inv_sigma) : 1.f;
    for (int i = tid; i < BN; i += kThreads) {
      s_scale[i] = __ldg(a.scale + n_tile * BN + i) * isg;
      s_shift[i] = __ldg(a.shift + n_tile * BN + i);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_acc = *tmem_ptr;

  if (warp < 8) {
    // ================= A producer (8 warps) =================
    const int m = m_tile * kBlockM + (tid & 127);
    const bool row_ok = m < a.M;          // row owned by this thread in the epilogue (TMEM lane = tid)

    // Gather mapping: 8 consecutive lanes fetch the 8 x 16-byte chunks of one 128-byte k-block row, so a
    // warp instruction touches 4 full cache lines (not 32 partial ones); a thread serves the same chunk
    // q of rows  it*32 + (tid>>3), it = 0..3.  Per row it keeps two element offsets (centre tap, one per
    // source) and a 32-bit word: bits 0-26 = validity of the 27 taps, bits 27-30 = whether the nearest-
    // upsampled source moves by one pixel for kh/kw = 0 / 2 (always 1 when src0 is not upsampled).
    const int q = tid & 7, rg = tid >> 3;
    const bool ups = (a.H0 != a.Hin) || (a.W0 != a.Win);
    {
      // each producer thread derives the descriptor of ONE row (its epilogue row) and publishes it
      int o0 = 0, o1 = 0;
      uint32_t info = 0u;
      if (row_ok && tid < 128) {
        const int wo = m % a.Wout;
        int t = m / a.Wout;
        const int ho = t % a.Hout;
        t /= a.Hout;                       // t = b*D + d
        const int d = t % a.D;
        const int hc = ho * a.stride, wc = wo * a.stride;      // centre-tap input coordinates
        uint32_t vd = 0, vh = 0, vw = 0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          vd |= (uint32_t)((d + k - 1) >= 0 && (d + k - 1) < a.D) << k;
          vh |= (uint32_t)((hc + k - 1) >= 0 && (hc + k - 1) < a.Hin) << k;
          vw |= (uint32_t)((wc + k - 1) >= 0 && (wc + k - 1) < a.Win) << k;
        }
        uint32_t m9 = 0, mask = 0;
#pragma unroll
        for (int k = 0; k < 3; ++k) m9 |= ((vh >> k) & 1u) ? (vw << (3 * k)) : 0u;
#pragma unroll
        for (int k = 0; k < 3; ++k) mask |= ((vd >> k) & 1u) ? (m9 << (9 * k)) : 0u;
        if (a.ksize == 1) mask &= (1u << 13);
        int hs1 = hc, ws1 = wc;
        uint32_t bits = 0xFu;
        if (ups) {
          hs1 = (hc * a.H0) / a.Hin;
          ws1 = (wc * a.W0) / a.Win;
          bits = 0;
          if (hc - 1 >= 0 && ((hc - 1) * a.H0) / a.Hin != hs1) bits |= 1u;
          if (hc + 1 < a.Hin && ((hc + 1) * a.H0) / a.Hin != hs1) bits |= 2u;
          if (wc - 1 >= 0 && ((wc - 1) * a.W0) / a.Win != ws1) bits |= 4u;
          if (wc + 1 < a.Win && ((wc + 1) * a.W0) / a.Win != ws1) bits |= 8u;
        }
        info = mask | (bits << 27);
        o0 = ((t * a.H0 + hs1) * a.W0 + ws1) * a.P0;
        o1 = ((t * a.Hin + hc) * a.Win + wc) * a.P1;
      }
      if (tid < 128) {
        s_rows[tid] = o0;
        s_rows[128 + tid] = o1;
        s_rows[256 + tid] = (int)info;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");       // producer warps only
    }
    int off0[4], off1[4];
    uint32_t rinfo[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 32 + rg;
      off0[it] = s_rows[r];
      off1[it] = s_rows[128 + r];
      rinfo[it] = (uint32_t)s_rows[256 + r];
    }
    const uint32_t dst_thread = (uint32_t)rg * 128u + ((uint32_t)(q ^ (rg & 7)) << 4);
    const int plane0 = a.H0 * a.W0 * a.P0, row0 = a.W0 * a.P0;
    const int plane1 = a.Hin * a.Win * a.P1, row1 = a.Win * a.P1;

    int tap = 0, c = q * 8;             // this thread's (tap, channel) inside the current k-block
    while (c >= a.Cin) { c -= a.Cin; ++tap; }
    for (int kb = 0; kb < a.num_kb; ++kb) {
      const int s = kb % STAGES;
      mbar_wait(empty_bar(s), ((kb / STAGES) & 1) ^ 1, a.error_flag);
      const uint32_t dst = a_base + (uint32_t)s * kAStageBytes + dst_thread;
      const int tap27 = (a.ksize == 3) ? tap : 13;
      const int kd = tap27 / 9, kh = (tap27 / 3) % 3, kw = tap27 % 3;
      const bool k_ok = tap < a.taps;
      const bool from0 = c < a.C0;
      const __nv_bfloat16* sbase = from0 ? a.src0 + c : a.src1 + (c - a.C0);
      const int toff = from0 ? (kd - 1) * plane0 : ((kd - 1) * plane1 + (kh - 1) * row1 + (kw - 1) * a.P1);
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const uint32_t ri = rinfo[it];
        const bool ok = k_ok && ((ri >> tap27) & 1u);
        int off;
        if (from0) {
          const int dh = (kh == 0) ? -(int)((ri >> 27) & 1u) : (kh == 2) ? (int)((ri >> 28) & 1u) : 0;
          const int dw = (kw == 0) ? -(int)((ri >> 29) & 1u) : (kw == 2) ? (int)((ri >> 30) & 1u) : 0;
          off = off0[it] + toff + dh * row0 + dw * a.P0;
        } else {
          off = off1[it] + toff;
        }
        cp_async_16(dst + (uint32_t)it * 4096u, ok ? (const void*)(sbase + off) : (const void*)a.src0, ok ? 16u : 0u);
      }
      // The arrival on full[s] is performed by the copy unit when this thread's copies have landed
      // (no wait in the producer: a proxy fence here would drain every cp.async in flight and
      // serialise the pipeline -- measured: 2400 cycles per k-block).  The MMA thread orders the
      // generic-proxy writes before its async-proxy reads with one fence after the barrier wait.
      cp_async_mbar_arrive_noinc(full_bar(s));
      c += kBlockK;
      while (c >= a.Cin) { c -= a.Cin; ++tap; }
    }

    // ================= epilogue: TMEM -> registers -> bf16 global =================
    mbar_wait(tmem_full_bar, 0, a.error_flag);
    __syncwarp();                       // tcgen05.ld is .sync.aligned: the warp must be converged
    tcgen05_fence_after();
    const uint32_t lane_addr = tmem_acc + ((uint32_t)((warp & 3) * 32) << 16);   // warps w and w+4 share a lane quarter
    __nv_bfloat16* orow = a.out + (size_t)m * a.Cout + n_tile * BN;
    const __nv_bfloat16* rrow = a.residual ? a.residual + (size_t)m * a.Cout + n_tile * BN : nullptr;
#pragma unroll 1
    for (int c0 = (warp >> 2) * 32; c0 < BN; c0 += 64) {         // ... and alternate 32-column chunks
      uint32_t v[32];
      tmem_ld_32x32b_x32(lane_addr + (uint32_t)c0, v);
      tmem_ld_wait();
      if (row_ok) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float r[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) r[i] = 0.f;
          if (rrow) {
            const uint4 rv = __ldg(reinterpret_cast<const uint4*>(rrow + c0 + g * 8));
            const __nv_bfloat162* rp = reinterpret_cast<const __nv_bfloat162*>(&rv);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float2 f = __bfloat1622float2(rp[i]);
              r[2 * i] = f.x;
              r[2 * i + 1] = f.y;
            }
          }
          uint4 ov;
          __nv_bfloat162* op = reinterpret_cast<__nv_bfloat162*>(&ov);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float y[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int n = c0 + g * 8 + 2 * i + h;
              float t = fmaf(__uint_as_float(v[g * 8 + 2 * i + h]), s_scale[n], s_shift[n]) + r[2 * i + h];
              if (a.act == 1) t = fmaxf(t, 0.f);
              else if (a.act == 2) t = t > 0.f ? t : 0.01f * t;
              y[h] = t;
            }
            op[i] = __floats2bfloat162_rn(y[0], y[1]);
          }
          *reinterpret_cast<uint4*>(orow + c0 + g * 8) = ov;
        }
      }
    }
  } else if (warp == 8) {
    // ================= MMA issuer (warp converged, one elected lane issues) =================
    constexpr uint32_t idesc = make_idesc(BN);
    for (int kb = 0; kb < a.num_kb; ++kb) {
      const int s = kb % STAGES;
      mbar_wait(full_bar(s), (kb / STAGES) & 1, a.error_flag);
      fence_proxy_async();
      tcgen05_fence_after();
      const uint32_t a_addr = a_base + (uint32_t)s * kAStageBytes;
      const uint32_t b_addr = b_base + (uint32_t)s * L::kBStageBytes;
#pragma unroll
      for (int k = 0; k < kBlockK / 16; ++k) {
        tcgen05_mma_bf16_elect(tmem_acc, make_smem_desc(a_addr + k * 32), make_smem_desc(b_addr + k * 32), idesc,
                               (kb | k) != 0 ? 1u : 0u);
      }
      tcgen05_commit_elect(empty_bar(s));   // frees the stage once these MMAs have read it
    }
    tcgen05_commit_elect(tmem_full_bar);    // accumulator complete
    (void)lane;
  } else {
    // ================= weight-tile producer (bulk copy engine) =================
    const __nv_bfloat16* wt = a.wpack + (size_t)n_tile * a.num_kb * (BN * kBlockK);
    for (int kb = 0; kb < a.num_kb; ++kb) {
      const int s = kb % STAGES;
      mbar_wait(empty_bar(s), ((kb / STAGES) & 1) ^ 1, a.error_flag);
      if (elect_one()) {
        mbar_arrive_expect_tx(full_bar(s), (uint32_t)L::kBStageBytes);
        bulk_copy_g2s(b_base + (uint32_t)s * L::kBStageBytes, wt + (size_t)kb * (BN * kBlockK),
                      (uint32_t)L::kBStageBytes, full_bar(s));
      }
      __syncwarp();
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 8) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"((uint32_t)BN) : "memory");
  }
}

// Weight repack: fp32 (Cout, Cin_real, k,k,k) -> bf16 tiles [Cout/BN][num_kb][BN][64] with the 128B swizzle
// applied per row (16-byte chunk q of row r is stored at chunk q ^ (r & 7)); k = tap*Cin_pad + p, zero padded.
// Padded input channel p maps to a real channel through two segments (pad0/real0 | pad1/real1): the halo kernels
// read activations with fewer than 64 channels as 64-channel rows so every TMA box row is 128 bytes.
__global__ void pack_weights_kernel(const float* __restrict__ w, int Cout, int cin_real, int taps, int BN, int num_kb,
                                    int pad0, int real0, int pad1, int real1, __nv_bfloat16* __restrict__ out) {
  const int cin_pad = pad0 + pad1;
  const size_t total = (size_t)Cout * num_kb * kBlockK;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int e = (int)(i % 8);
    const int qs = (int)((i / 8) % 8);          // stored chunk
    const int r = (int)((i / 64) % BN);
    const size_t tile = i / ((size_t)64 * BN);  // n_tile*num_kb + kb
    const int kb = (int)(tile % num_kb);
    const int n_tile = (int)(tile / num_kb);
    const int q = qs ^ (r & 7);                 // logical chunk
    const int kk = kb * kBlockK + q * 8 + e;
    const int n = n_tile * BN + r;
    float v = 0.f;
    if (kk < taps * cin_pad) {
      const int tap = kk / cin_pad, p = kk % cin_pad;
      int c = -1;
      if (p < pad0) { if (p < real0) c = p; }
      else { const int p1 = p - pad0; if (p1 < real1) c = real0 + p1; }
      if (c >= 0) v = w[((size_t)n * cin_real + c) * taps + tap];
    }
    out[i] = __float2bfloat16_rn(v);
  }
}

inline int pick_bn(int cout) {
  if (cout % 256 == 0) return 256;
  if (cout % 128 == 0) return 128;
  if (cout % 64 == 0) return 64;
  if (cout % 32 == 0) return 32;
  return 0;
}

template <int BN, int STAGES>
inline int launch_one(const ConvArgs& a, cudaStream_t s) {
  using L = SmemLayout<BN, STAGES>;
  static bool configured[64] = {false};
  const int slot = device_slot();
  if (!configured[slot]) {
    V2CE_CUDA_CHECK(cudaFuncSetAttribute(conv_igemm_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         L::kDynamicBytes));
    configured[slot] = true;
  }
  const int m_tiles = (a.M + kBlockM - 1) / kBlockM;
  const int grid = m_tiles * (a.Cout / BN);
  conv_igemm_kernel<BN, STAGES><<<grid, kThreads, L::kDynamicBytes, s>>>(a);
  V2CE_LAUNCH_CHECK("conv_igemm_kernel");
  return V2CE_OK;
}

inline int launch_conv(const ConvArgs& a, int bn, cudaStream_t s) {
  // the gather uses 32-bit element offsets
  if ((long long)a.B * a.D * a.H0 * a.W0 * a.P0 >= (1LL << 31) || (long long)a.B * a.D * a.Hin * a.Win * a.P1 >= (1LL << 31) ||
      (long long)a.M * a.Cout >= (1LL << 40))
    return set_error(V2CE_ERR_RANGE, "activation tensor too large for 32-bit gather offsets; lower the batch size");
  switch (bn) {
    case 32: return launch_one<32, 4>(a, s);
    case 64: return launch_one<64, 4>(a, s);
    case 128: return launch_one<128, 3>(a, s);
    case 256: return launch_one<256, 4>(a, s);
  }
  return set_error(V2CE_ERR_INVALID, "unsupported N tile %d", bn);
}

}  // namespace conv
}  // namespace v2ce
