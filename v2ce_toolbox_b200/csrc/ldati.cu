// LDATI (stage 2) on sm_100a: event-count relocation, slot assignment in the reference's
// generation order, inverse-CDF timestamps, stable per-(frame,bin) radix sort and 13-byte
// record packing.  Replaces /root/reference/scripts/LDATI.py:13-51,80-106,126-310, plus the
// options the CLI leaves at their defaults: bidirectional relocation (:107-122) and the
// 'random' / 'none' strategies for multi-event pixel-bins (:173-174, :206-207, :241-244).
//
// Data layout in HBM
//   voxels   float32 (F,2,10,H,W): planes of H*W pixels; a thread owns V=4 consecutive
//            pixels (float4 loads, fully coalesced) of one polarity plane and walks the
//            10 bins (plane stride H*W).
//   elements one 32-bit (or 64-bit when H*W or the key range needs it) word per event:
//            [ sort key = ts - bin_base + BIAS | polarity | pixel ].  Everything a record
//            needs travels in the word, so the sort moves 4 bytes per event per pass.
//   records  13-byte packed AoS, written through shared memory with 16-byte stores.
//
// Order contract (SURVEY.md F5): per frame, bins ascending; inside a bin the events are
// sorted by (timestamp, g), g = position in the reference's pre-sort concatenation
// [neg singles][neg multis][pos singles][pos multis] (row-major pixels, j ascending).
// The emit kernel writes every event straight to slot g (prefix sums from the count
// pass), so a STABLE sort on the timestamp key alone yields the canonical order.
//
// Arithmetic contract (SURVEY.md F6, Appendix A): one IEEE rounding per reference torch
// op -- all float math below goes through __f*_rn / __d*_rn so nvcc cannot contract it.
#include "common.cuh"

#include <limits.h>
#include <string.h>

namespace v2ce {
namespace ldati {

constexpr int kBins = 9;          // event bins per frame pair (10 voxel bins -> 9)
constexpr int kQ = 18;            // scanned quantities per plane: singles[9], multis[9]
constexpr int kThreads = 256;
constexpr int kKeyBias = 8;       // slack below the bin origin (ts may undershoot it by 1 us)
// one-sweep sort (osw_*): 256 threads x 16 keys, <= 6-bit digits (64 digits = 32 counter lanes x 2 packed 16-bit counters)
constexpr int kOswKpt = 16;
constexpr int kOswTile = kThreads * kOswKpt;
constexpr int kOswRadixBits = 6;
constexpr int kOswRadix = 1 << kOswRadixBits;
constexpr int kOswMaxPasses = 6;
constexpr int kPackRecsPerWarpDecl = 128;      // records per pack chunk (pack_linear_kernel)
static inline int osw_passes(int key_bits) { return (key_bits + kOswRadixBits - 1) / kOswRadixBits; }

struct Geometry {
  int H, W, HW, F;
  int V;         // pixels per thread (4 when HW % 4 == 0, else 1)
  int NB;        // blocks per plane
  int pix_bits;  // bits of the pixel field
  int key_bits;  // bits of the sort key
  int wide;      // 1: 64-bit elements
  int pooling;   // != 0: the count workspace also holds every pixel-bin's count (the slope is fitted on pooled counts)
};

static Geometry make_geometry(const v2ce_ldati_params* p) {
  Geometry g;
  g.H = p->height;
  g.W = p->width;
  g.HW = p->height * p->width;
  g.F = p->n_frames;
  g.V = (g.HW % 4 == 0) ? 4 : 1;
  g.NB = (g.HW + kThreads * g.V - 1) / (kThreads * g.V);
  g.pix_bits = 1;
  while ((1LL << g.pix_bits) < g.HW) ++g.pix_bits;
  g.key_bits = 1;
  while ((1LL << g.key_bits) < (long long)p->key_span + 1) ++g.key_bits;
  g.wide = (g.pix_bits + 1 + g.key_bits > 32) ? 1 : 0;
  g.pooling = (p->pooling != 0 && p->multi_events == 1) ? 1 : 0;     // only the 'slope' strategy reads pooled counts
  return g;
}

// count workspace layout
struct CountWs {
  int32_t* partial;     // [F][2][NB][18]
  int32_t* warp_partial;  // [F][2][NB][8 warps][18]: the count pass's per-warp totals, reused by the emit pass
  int32_t* counts_all;    // pooling only: [F][2][9][HW] counts of every pixel-bin (neighbours feed the pooled slope)
  int32_t* block_base;  // [F][2][NB][18]
  int32_t* group_base;  // [F][9][4]
  int64_t* seg_start;   // [F*9+1]
  size_t bytes;
};

static CountWs carve_count_ws(void* ws, const Geometry& g) {
  Arena a(ws, (size_t)-1);
  CountWs w;
  size_t n = (size_t)g.F * 2 * g.NB * kQ;
  w.partial = a.take<int32_t>(n);
  w.block_base = a.take<int32_t>(n);
  w.group_base = a.take<int32_t>((size_t)g.F * kBins * 4);
  w.seg_start = a.take<int64_t>((size_t)g.F * kBins + 1);
  w.warp_partial = a.take<int32_t>(n * (kThreads / 32));
  w.counts_all = g.pooling ? a.take<int32_t>((size_t)g.F * 2 * kBins * g.HW) : nullptr;
  w.bytes = align_up(a.off, 256);
  return w;
}

// ---------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------
struct DevParams {
  int H, W, HW, F, NB;
  int true_div;
  long long frame_base;
  unsigned long long seed;
  double fps64, nbins64, r_fps64, r_nbins64;
  float fps32, nbins32, r_fps32, r_nbins32;
  float vs32, inv_vs32, vs2_32, r_vs2_32, six32, r6_32, eps6, eps8;
  float binstart[kBins];
  long long bin_base[kBins];
  int pix_bits, key_bits;
  int draws_m;
  int add_frame_offset;
  int multi_events;   // additional_events_strategy: 0 'none' (multi-event pixel-bins emit nothing), 1 'slope',
                      // 2 'random' (the raw draw is the time offset in seconds, LDATI.py:173-174)
  int pooling;        // 0 none, 1 'weighted' (3x3 binomial / 16), 2 'avg' (pool_k x pool_k box / pool_k^2); LDATI.py:176-183
  int pool_k;
  long long nan_ts;   // float NaN -> int64: INT64_MIN on x86 (cvttss2si) and on torch-CUDA (measured on B200)
  int segs_per_frame; // sort segments per frame: 9 (LDATI: one per bin) or 1 (baseline samplers: whole frames)
};

static DevParams make_dev_params(const v2ce_ldati_params* p, const Geometry& g) {
  DevParams d;
  d.H = g.H; d.W = g.W; d.HW = g.HW; d.F = g.F; d.NB = g.NB;
  d.true_div = p->true_div;
  d.frame_base = p->frame_base;
  d.seed = p->seed;
  d.fps64 = p->fps64; d.nbins64 = p->nbins64; d.r_fps64 = p->r_fps64; d.r_nbins64 = p->r_nbins64;
  d.fps32 = p->fps32; d.nbins32 = p->nbins32; d.r_fps32 = p->r_fps32; d.r_nbins32 = p->r_nbins32;
  d.vs32 = p->vs32; d.inv_vs32 = p->inv_vs32; d.vs2_32 = p->vs2_32; d.r_vs2_32 = p->r_vs2_32;
  d.six32 = p->six32; d.r6_32 = p->r6_32; d.eps6 = p->eps6; d.eps8 = p->eps8;
  for (int c = 0; c < kBins; ++c) { d.binstart[c] = p->binstart_t0_32[c]; d.bin_base[c] = p->bin_base_us[c]; }
  d.pix_bits = g.pix_bits; d.key_bits = g.key_bits;
  d.draws_m = 0;
  d.add_frame_offset = p->add_frame_offset;
  d.multi_events = p->multi_events;
  d.pooling = g.pooling ? p->pooling : 0;
  d.pool_k = p->pooling_kernel_size;
  d.nan_ts = LLONG_MIN;
  d.segs_per_frame = kBins;
  return d;
}

// y_relocate (LDATI.py:96-106) for one pixel: n[9] and the carried debts tend[9].
__device__ __forceinline__ void relocate_pixel(const float (&y)[10], float eps6, int (&n)[kBins], float (&tend)[kBins]) {
  float debt = 0.f;
#pragma unroll
  for (int c = 0; c < kBins; ++c) {
    float x = __fsub_rn(y[c], debt);
    float nc = ceilf(__fsub_rn(x, eps6));
    debt = __fsub_rn(nc, x);
    n[c] = __float2int_rz(nc);
    tend[c] = debt;
  }
  n[kBins - 1] += __float2int_rz(__fsub_rn(y[9], debt));   // `.int()` truncation, LDATI.py:106
}

// y_relocate(bidirectional=True) (LDATI.py:91-94,96-104,107-122) for one pixel: bins 0..3 carry the debt from
// the left, bins 8,7,6 carry `bless` from the right (seeded with the tenth voxel bin), bin 5 settles both, and
// bin 4 is never written by the reference (n = 0, tend = 0).
__device__ __forceinline__ void relocate_pixel_bidir(const float (&y)[10], float eps6, int (&n)[kBins], float (&tend)[kBins]) {
  float debt = 0.f;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float x = __fsub_rn(y[c], debt);
    float nc = ceilf(__fsub_rn(x, eps6));
    debt = __fsub_rn(nc, x);
    n[c] = __float2int_rz(nc);
    tend[c] = debt;
  }
  n[4] = 0;
  tend[4] = 0.f;
  float bless = y[9];
#pragma unroll
  for (int c = 8; c > 5; --c) {
    tend[c] = bless;
    const float fl = floorf(__fadd_rn(__fadd_rn(y[c], bless), eps6));
    bless = __fadd_rn(__fsub_rn(y[c], fl), bless);
    bless = (bless < 0.f) ? 0.f : bless;            // torch.clamp(min=0): NaN stays NaN
    n[c] = __float2int_rz(fl);
  }
  tend[5] = __fsub_rn(bless, debt);
  n[5] = __float2int_rz(ceilf(__fsub_rn(__fadd_rn(y[5], bless), debt)));
}

template <bool BIDIR>
__device__ __forceinline__ void relocate_any(const float (&y)[10], float eps6, int (&n)[kBins], float (&tend)[kBins]) {
  if (BIDIR) relocate_pixel_bidir(y, eps6, n, tend);
  else relocate_pixel(y, eps6, n, tend);
}

template <int V>
__device__ __forceinline__ void load_pixels(const float* __restrict__ plane0, int HW, int pix, float (&y)[V][10]) {
  if (V == 4) {
#pragma unroll
    for (int c = 0; c < 10; ++c) {
      float4 t = __ldg(reinterpret_cast<const float4*>(plane0 + (size_t)c * HW + pix));
      y[0][c] = t.x; y[1 % V][c] = t.y; y[2 % V][c] = t.z; y[3 % V][c] = t.w;
    }
  } else {
#pragma unroll
    for (int c = 0; c < 10; ++c) y[0][c] = __ldg(plane0 + (size_t)c * HW + pix);
  }
}

__device__ __forceinline__ int warp_incl_scan(int v) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) >= o) v += t;
  }
  return v;
}

// Philox4x32-10, counter (lo32(idx), hi32(idx), j>>2, 0), key = seed; see oracle/philox.py.
// One Philox block = the draws of four consecutive events of a pixel-bin: the emit loop evaluates it once per
// four events (philox_block) and picks word j & 3.
__device__ __forceinline__ void philox_block(unsigned long long idx, unsigned blk, unsigned long long seed, unsigned (&w)[4]) {
  unsigned c0 = (unsigned)idx, c1 = (unsigned)(idx >> 32), c2 = blk, c3 = 0u;
  unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  w[0] = c0; w[1] = c1; w[2] = c2; w[3] = c3;
}
// same generator with the fourth counter word as a stream id (baseline samplers: 0 integer-part uniforms, 1 fractional-part
// uniform, 2 Bernoulli uniform; oracle/baseline_oracle.py)
__device__ __forceinline__ float philox_uniform_stream(unsigned long long idx, unsigned j, unsigned long long seed, unsigned stream) {
  unsigned c0 = (unsigned)idx, c1 = (unsigned)(idx >> 32), c2 = j >> 2, c3 = stream;
  unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  const unsigned sel = j & 3u;
  const unsigned w = sel == 0 ? c0 : sel == 1 ? c1 : sel == 2 ? c2 : c3;
  return __fmul_rn((float)(w >> 8), 5.9604644775390625e-08f);   // 2^-24
}

__device__ __forceinline__ float philox_word_to_uniform(const unsigned (&w)[4], unsigned j) {
  const unsigned sel = j & 3u;
  const unsigned v = sel == 0 ? w[0] : sel == 1 ? w[1] : sel == 2 ? w[2] : w[3];
  return __fmul_rn((float)(v >> 8), 5.9604644775390625e-08f);   // 2^-24
}

__device__ __forceinline__ float philox_uniform(unsigned long long idx, unsigned j, unsigned long long seed) {
  unsigned c0 = (unsigned)idx, c1 = (unsigned)(idx >> 32), c2 = j >> 2, c3 = 0u;
  unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  unsigned sel = j & 3u;
  unsigned w = sel == 0 ? c0 : sel == 1 ? c1 : sel == 2 ? c2 : c3;
  return __fmul_rn((float)(w >> 8), 5.9604644775390625e-08f);   // 2^-24
}

// ---------------------------------------------------------------------------------------
// K3: count pass.  grid (NB, 2, F), 256 threads, V pixels per thread.
// ---------------------------------------------------------------------------------------
template <int V, bool BIDIR>
__global__ void __launch_bounds__(kThreads) count_kernel(const float* __restrict__ vox, DevParams P,
                                                          int32_t* __restrict__ partial,
                                                          int32_t* __restrict__ warp_partial,
                                                          float* __restrict__ ef_sums) {
  const int blk = blockIdx.x, p = blockIdx.y, f = blockIdx.z;
  const int pix = (blk * kThreads + threadIdx.x) * V;
  int tot[kQ];
#pragma unroll
  for (int q = 0; q < kQ; ++q) tot[q] = 0;
  if (pix < P.HW) {
    float y[V][10];
    load_pixels<V>(vox + ((size_t)(f * 2 + p) * 10) * P.HW, P.HW, pix, y);
    if (ef_sums != nullptr) {
      // event-frame sums (v2ce.py:255): s = y0; s += y1; ...; s += y9 -- sequential float32 adds, numpy's order
      float sum[V];
#pragma unroll
      for (int v = 0; v < V; ++v) {
        sum[v] = y[v][0];
#pragma unroll
        for (int c = 1; c < 10; ++c) sum[v] = __fadd_rn(sum[v], y[v][c]);
      }
      float* dst = ef_sums + (size_t)(f * 2 + p) * P.HW + pix;
      if (V == 4) *reinterpret_cast<float4*>(dst) = make_float4(sum[0], sum[1 % V], sum[2 % V], sum[3 % V]);
      else dst[0] = sum[0];
    }
#pragma unroll
    for (int v = 0; v < V; ++v) {
      int n[kBins];
      float tend[kBins];
      relocate_any<BIDIR>(y[v], P.eps6, n, tend);
#pragma unroll
      for (int c = 0; c < kBins; ++c) {
        tot[c] += (n[c] == 1);
        tot[kBins + c] += (n[c] >= 2 && P.multi_events) ? n[c] : 0;
      }
    }
  }
  __shared__ int red[kThreads / 32][kQ];
#pragma unroll
  for (int q = 0; q < kQ; ++q) {
    int v = tot[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][q] = v;
  }
  __syncthreads();
  if (threadIdx.x < kQ) {
    int s = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) s += red[w][threadIdx.x];
    partial[(((size_t)f * 2 + p) * P.NB + blk) * kQ + threadIdx.x] = s;
  }
  if (threadIdx.x < (kThreads / 32) * kQ)
    warp_partial[(((size_t)f * 2 + p) * P.NB + blk) * ((kThreads / 32) * kQ) + threadIdx.x] = (&red[0][0])[threadIdx.x];
}

// K4a: per frame, exclusive scan of the block partials over the plane; group bases; segment counts.
__global__ void scan_planes_kernel(const int32_t* __restrict__ partial, int32_t* __restrict__ block_base,
                                   int32_t* __restrict__ group_base, int64_t* __restrict__ seg_counts, int NB) {
  const int f = blockIdx.x;
  __shared__ int tot[2][kQ];
  const int t = threadIdx.x;
  if (t < 2 * kQ) {
    const int p = t / kQ, q = t % kQ;
    const size_t base = ((size_t)f * 2 + p) * NB * kQ + q;
    int run = 0;
    for (int b = 0; b < NB; ++b) {
      block_base[base + (size_t)b * kQ] = run;
      run += partial[base + (size_t)b * kQ];
    }
    tot[p][q] = run;
  }
  __syncthreads();
  if (t < kBins) {
    const int c = t;
    const int s_neg = tot[1][c], m_neg = tot[1][kBins + c], s_pos = tot[0][c], m_pos = tot[0][kBins + c];
    int32_t* gb = group_base + ((size_t)f * kBins + c) * 4;
    gb[0] = 0;                       // negative singles   (p-index 1 -> polarity 0, LDATI.py:290)
    gb[1] = s_neg;                   // negative multis
    gb[2] = s_neg + m_neg;           // positive singles
    gb[3] = s_neg + m_neg + s_pos;   // positive multis
    seg_counts[(size_t)f * kBins + c] = (int64_t)s_neg + m_neg + s_pos + m_pos;
  }
}

// K4b: exclusive scan of n int64 values into out[0..n] (out[n] = total); one block.
__global__ void scan_i64_kernel(const int64_t* __restrict__ in, int64_t* __restrict__ out, int n) {
  __shared__ long long wsum[32];
  __shared__ long long carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < n; base += blockDim.x) {
    int i = base + threadIdx.x;
    long long v = (i < n) ? in[i] : 0;
    long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      long long t = __shfl_up_sync(0xffffffffu, incl, o);
      if ((threadIdx.x & 31) >= o) incl += t;
    }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      long long w = (threadIdx.x < (blockDim.x >> 5)) ? wsum[threadIdx.x] : 0;
      long long wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        long long t = __shfl_up_sync(0xffffffffu, wi, o);
        if (threadIdx.x >= o) wi += t;
      }
      wsum[threadIdx.x] = wi - w;   // exclusive warp offsets
    }
    __syncthreads();
    long long carry = carry_s;
    long long excl = carry + wsum[threadIdx.x >> 5] + incl - v;
    if (i < n) out[i] = excl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) out[n] = carry_s;
}

// ---------------------------------------------------------------------------------------
// K5: emit pass.  Same grid as the count pass; recomputes the counts (the voxel chunk is
// L2-resident from the count pass), block-scans the 18 quantities and writes one element
// per event to its generation-order slot.
// ---------------------------------------------------------------------------------------
template <typename Elem>
__device__ __forceinline__ Elem make_elem(long long ts, bool is_nan, long long bin_base, int pol, int pix, int pix_bits,
                                          int key_bits, int32_t* status) {
  // key 0 is reserved for "NaN timestamp below the bin": it sorts first (its value,
  // INT64_MIN, is smaller than every real timestamp of the bin) and pack restores nan_ts.
  long long key = ts - bin_base + kKeyBias;
  if (is_nan) atomicAdd(status + 1, 1);
  const long long kmax = (1LL << key_bits) - 1;
  if (is_nan && (ts < bin_base - kKeyBias + 1)) {
    key = 0;
  } else if (key < 1 || key > kmax) {   // outside the representable key range: flagged, host raises
    atomicAdd(status + 0, 1);
    key = key < 1 ? 1 : kmax;
  }
  return (Elem)(((unsigned long long)key << (pix_bits + 1)) | ((unsigned long long)pol << pix_bits) |
                (unsigned long long)pix);
}

// y_relocate one bin at a time (same operations as relocate_pixel): the emit pass walks the bins with a
// three-bin window (the slope needs the counts of both neighbours) instead of holding all 9 x V counts and
// debts in registers.  Fully unrolled over bins the kernel was 18 k instructions at 190 registers: one block
// per SM, most stall samples on instruction fetch (ncu, profiles/).
__device__ __forceinline__ void relocate_step(float y, float y_last, bool last_bin, float eps6, float& debt, int& n, float& tend) {
  const float x = __fsub_rn(y, debt);
  const float nc = ceilf(__fsub_rn(x, eps6));
  debt = __fsub_rn(nc, x);
  n = __float2int_rz(nc);
  tend = debt;
  if (last_bin) n += __float2int_rz(__fsub_rn(y_last, debt));     // `.int()` truncation, LDATI.py:106
}

template <int V>
__device__ __forceinline__ void load_bin(const float* __restrict__ plane0, int HW, int pix, int c, float (&y)[V]) {
  if (V == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(plane0 + (size_t)c * HW + pix));
    y[0] = t.x; y[1 % V] = t.y; y[2 % V] = t.z; y[3 % V] = t.w;
  } else {
    y[0] = __ldg(plane0 + (size_t)c * HW + pix);
  }
}

// y_pooled (LDATI.py:176-183) of one pixel-bin from the stored counts of its plane `cp` = counts_all + ((f*2+p)*9+c)*HW:
// 'weighted' = 3x3 binomial kernel / 16 with zero padding (dyadic weights on small integers: every accumulation order
// gives the same float32); 'avg' = zero-padded k x k window sum (exact) divided by k*k in float32.
__device__ __noinline__ float pooled_count(const int32_t* __restrict__ cp, int H, int W, int pix, int pooling, int k) {
  const int h = pix / W, w = pix - h * W;
  if (pooling == 1) {
    float acc = 0.f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
#pragma unroll
      for (int dx = -1; dx <= 1; ++dx) {
        const int hh = h + dy, ww = w + dx;
        const float wt = ((dy == 0) ? 2.f : 1.f) * ((dx == 0) ? 2.f : 1.f) * 0.0625f;
        const float x = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? (float)__ldg(cp + (size_t)hh * W + ww) : 0.f;
        acc = __fadd_rn(acc, __fmul_rn(wt, x));
      }
    }
    return acc;
  }
  const int r = k >> 1;
  long long sum = 0;
  for (int hh = max(h - r, 0); hh <= min(h + r, H - 1); ++hh)
    for (int ww = max(w - r, 0); ww <= min(w + r, W - 1); ++ww) sum += __ldg(cp + (size_t)hh * W + ww);
  return __fdiv_rn((float)sum, (float)(k * k));
}

template <int V, typename Elem, bool BIDIR, bool POOL>
__global__ void __launch_bounds__(kThreads) emit_kernel(const float* __restrict__ vox, DevParams P,
                                                         const int32_t* __restrict__ block_base,
                                                         const int32_t* __restrict__ group_base,
                                                         const int64_t* __restrict__ seg_start,
                                                         const int32_t* __restrict__ warp_partial,
                                                         const int32_t* __restrict__ counts_all,
                                                         const float* __restrict__ draws, Elem* __restrict__ elems,
                                                         int32_t* __restrict__ status) {
  const int blk = blockIdx.x, p = blockIdx.y, f = blockIdx.z;
  const int pix0 = (blk * kThreads + threadIdx.x) * V;
  const bool active = pix0 < P.HW;
  const float* plane0 = vox + ((size_t)(f * 2 + p) * 10) * P.HW;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // ---- per-warp totals of the 18 quantities (singles / multi-event totals per bin), left by the count pass ----
  __shared__ int wtot[kThreads / 32][kQ];
  __shared__ float2 s_par[kThreads / 32][32][V];      // (k, b) of every pixel of the block for the current bin
  if (threadIdx.x < (kThreads / 32) * kQ)
    (&wtot[0][0])[threadIdx.x] = warp_partial[(((size_t)f * 2 + p) * P.NB + blk) * ((kThreads / 32) * kQ) + threadIdx.x];
  __syncthreads();
  // ---- bins in order, three-bin window of counts; voxels re-read (L1/L2 hits) ----
  const int pol = 1 - p;                         // p-index 0 = positive plane -> polarity 1
  const int grp = (p == 1) ? 0 : 2;              // negative plane is emitted first
  const size_t bb = (((size_t)f * 2 + p) * P.NB + blk) * kQ;
  const unsigned long long frame = (unsigned long long)(P.frame_base + f);
  // slots: [segment start] + [group base] + [blocks before] + [warps before] + [lanes before].  The first three do not
  // depend on the lane and the fourth only on the warp: 18 threads fetch them once per block instead of every thread
  // loading five words and summing up to seven per-warp totals in every bin iteration.
  __shared__ long long s_base[kQ];               // q < 9: singles of bin q, q >= 9: multi-events of bin q - 9
  __shared__ int s_wpre[kThreads / 32][kQ];      // events of the warps before this one
  if (threadIdx.x < kQ) {
    const int q = threadIdx.x, c = q % kBins;
    const int32_t* gb = group_base + ((size_t)f * kBins + c) * 4;
    s_base[q] = seg_start[(size_t)f * kBins + c] + gb[grp + (q >= kBins ? 1 : 0)] + block_base[bb + q];
    int run = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) { s_wpre[w][q] = run; run += wtot[w][q]; }
  }
  __syncthreads();
  __shared__ int4 s_lane[kThreads / 32][32];     // per lane and bin: {quads before, events before, counts of pixels 0..2, count of pixel 3}
  float debt[V], tend_cur[V], tend_next[V], y9[V];
  int n_prev[V], n_cur[V], n_next[V];
#pragma unroll
  for (int v = 0; v < V; ++v) { debt[v] = 0.f; n_prev[v] = n_cur[v] = n_next[v] = 0; tend_cur[v] = tend_next[v] = 0.f; y9[v] = 0.f; }
  // BIDIR: the right-to-left chain of bins 8..5 cannot be walked with the sliding window, so this (cold, off-CLI)
  // instantiation keeps the nine counts and tendencies of its pixels in local arrays and feeds the window from them.
  int n_all[BIDIR ? V : 1][kBins];
  float tend_all[BIDIR ? V : 1][kBins];
  if (BIDIR) {
#pragma unroll
    for (int v = 0; v < V; ++v)
#pragma unroll
      for (int c = 0; c < kBins; ++c) { n_all[v][c] = 0; tend_all[v][c] = 0.f; }
    if (active) {
      float y[V][10];
      load_pixels<V>(plane0, P.HW, pix0, y);
#pragma unroll
      for (int v = 0; v < V; ++v) relocate_pixel_bidir(y[v], P.eps6, n_all[v], tend_all[v]);
    }
#pragma unroll
    for (int v = 0; v < V; ++v) {
      n_cur[v] = n_all[v][0]; tend_cur[v] = tend_all[v][0];
      n_next[v] = n_all[v][1]; tend_next[v] = tend_all[v][1];
    }
  } else if (active) {
    float y0[V], y1[V];
    load_bin<V>(plane0, P.HW, pix0, 0, y0);
    load_bin<V>(plane0, P.HW, pix0, 1, y1);
    load_bin<V>(plane0, P.HW, pix0, 9, y9);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      relocate_step(y0[v], 0.f, false, P.eps6, debt[v], n_cur[v], tend_cur[v]);
      relocate_step(y1[v], 0.f, false, P.eps6, debt[v], n_next[v], tend_next[v]);
    }
  }
#pragma unroll 1
  for (int c = 0; c < kBins; ++c) {
    int ts1 = 0, tsm = 0;
#pragma unroll
    for (int v = 0; v < V; ++v) { ts1 += (n_cur[v] == 1); tsm += (n_cur[v] >= 2 && P.multi_events) ? n_cur[v] : 0; }
    // one scan for both quantities while the multi-event total of a lane stays below 2^16 (singles: <= 4 per lane)
    const bool small = tsm < 65536;
    int ex1, exm;
    if (__all_sync(0xffffffffu, small)) {
      const int both = warp_incl_scan(ts1 | (tsm << 8));
      ex1 = (both & 255) - ts1;
      exm = (both >> 8) - tsm;
    } else {
      ex1 = warp_incl_scan(ts1) - ts1;
      exm = warp_incl_scan(tsm) - tsm;
    }
    // Single events: one lane per pixel group (cheap, float64 path).
    // Multi-event pixel-bins: WARP-COOPERATIVE.  A lane looping over its own pixels' events runs to the warp's
    // maximum count (~15 on dense inputs) while the mean is 4.5: 5.3 active lanes per warp instruction (ncu).  The
    // warp's events of this bin are instead cut into QUADS -- four consecutive events j = 4q .. 4q+3 of one pixel-bin,
    // i.e. the four words of ONE Philox block -- numbered in generation order and dealt out 32 at a time: a lane finds
    // its quad's source lane by binary search over the shuffled exclusive scan, reads that pixel's slope parameters
    // and counts from shared memory, evaluates one Philox block and writes up to four consecutive slots.
    const long long bin_base = P.bin_base[c];
    const float bstart = P.binstart[c];
    if (active) {
      long long slot_s = s_base[c] + s_wpre[warp][c] + ex1;
#pragma unroll
      for (int v = 0; v < V; ++v) {
        if (n_cur[v] == 1) {
          // single event (LDATI.py:156-165): float64 path
          double t = (double)tend_cur[v];
          t = P.true_div ? __ddiv_rn(__ddiv_rn(t, P.fps64), P.nbins64)
                         : __dmul_rn(__dmul_rn(t, P.r_fps64), P.r_nbins64);
          t = __dadd_rn(t, (double)bstart);
          t = __dmul_rn(t, 1e6);
          const long long ts = (long long)t;
          elems[slot_s++] = make_elem<Elem>(ts, false, bin_base, pol, pix0 + v, P.pix_bits, P.key_bits, status);
        }
      }
    }
    // per-pixel slope parameters (LDATI.py:184-192) of this lane's multi-event pixels -> shared memory
    int cnt[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int nc = n_cur[v];
      cnt[v] = (active && nc >= 2 && P.multi_events) ? nc : 0;
      float kk = 0.f, b = 0.f;
      if (cnt[v]) {
        float S = 0.f;
        float y_fit = (float)nc;                 // the counts the slope is fitted on: pooled (LDATI.py:176-186) or raw
        if (POOL) {
          const int32_t* cp = counts_all + (((size_t)f * 2 + p) * kBins + c) * P.HW;
          y_fit = pooled_count(cp, P.H, P.W, pix0 + v, P.pooling, P.pool_k);
          if (c > 0 && c < kBins - 1)
            S = __fsub_rn(pooled_count(cp + P.HW, P.H, P.W, pix0 + v, P.pooling, P.pool_k),
                          pooled_count(cp - P.HW, P.H, P.W, pix0 + v, P.pooling, P.pool_k));
        } else if (c > 0 && c < kBins - 1) {
          S = __fsub_rn((float)n_next[v], (float)n_prev[v]);
        }
        const float num = __fsub_rn(__fmul_rn(3.f, S), 0.f);
        kk = P.true_div ? __fdiv_rn(__fdiv_rn(num, P.six32), P.vs2_32)
                        : __fmul_rn(__fmul_rn(num, P.r6_32), P.r_vs2_32);
        kk = __fdiv_rn(kk, __fadd_rn(y_fit, P.eps8));
        b = __fsub_rn(P.inv_vs32, __fmul_rn(__fmul_rn(P.vs32, kk), 0.5f));
      }
      s_par[warp][lane][v] = make_float2(kk, b);
    }
    // quads of this lane's pixels; the fast path holds while every pixel-bin has < 1024 events (three counts pack
    // into one word) -- beyond that (out-of-contract voxel values) the per-lane loop below takes over
    const int q0 = (cnt[0] + 3) >> 2, q1 = (cnt[1 % V] * (V > 1) + 3) >> 2, q2 = (cnt[2 % V] * (V > 2) + 3) >> 2,
              q3 = (cnt[3 % V] * (V > 3) + 3) >> 2;
    const int tq = q0 + q1 + q2 + q3;
    const bool fits = (cnt[0] | cnt[1 % V] | cnt[2 % V] | cnt[3 % V]) < 1024;
    const int incq = warp_incl_scan(tq);
    const int exq = incq - tq;
    const int TQ_warp = __shfl_sync(0xffffffffu, incq, 31);
    s_lane[warp][lane] = make_int4(exq, exm, cnt[0] | ((cnt[1 % V] * (V > 1)) << 10) | ((cnt[2 % V] * (V > 2)) << 20),
                                   cnt[3 % V] * (V > 3));
    __syncwarp();
    if (__all_sync(0xffffffffu, fits)) {
      const long long warp_slot = s_base[kBins + c] + s_wpre[warp][kBins + c];
      for (int e0 = 0; e0 < TQ_warp; e0 += 32) {
        const int e = e0 + lane;
        // source lane: the last one whose exclusive quad offset is <= e
        int src = 0;
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
          const int probe = src + step;
          const int off = __shfl_sync(0xffffffffu, exq, probe & 31);
          if (probe < 32 && off <= e) src = probe;
        }
        if (e < TQ_warp) {
          const int4 sl = s_lane[warp][src];
          const int c0 = sl.z & 1023, c1 = (sl.z >> 10) & 1023, c2 = (sl.z >> 20) & 1023, c3 = sl.w;
          const int t0 = (c0 + 3) >> 2, t1 = t0 + ((c1 + 3) >> 2), t2 = t1 + ((c2 + 3) >> 2);
          const int le = e - sl.x;
          const int v = (le >= t0) + (le >= t1) + (le >= t2);
          const int qi = le - (v == 0 ? 0 : v == 1 ? t0 : v == 2 ? t1 : t2);        // quad index inside the pixel-bin
          const int nv = v == 0 ? c0 : v == 1 ? c1 : v == 2 ? c2 : c3;              // events of the pixel-bin
          const int ebefore = sl.y + (v == 0 ? 0 : v == 1 ? c0 : v == 2 ? c0 + c1 : c0 + c1 + c2) + 4 * qi;
          const int nev = min(4, nv - 4 * qi);
          const float2 par = s_par[warp][src][v];
          const float kk = par.x, b = par.y;
          const float bb2 = __fmul_rn(b, b);
          const float k2 = __fmul_rn(2.f, kk);
          const int pix = (blk * kThreads + warp * 32 + src) * V + v;
          const unsigned long long idx = ((frame * 2ull + (unsigned)p) * 9ull + (unsigned)c) * (unsigned long long)P.HW + (unsigned)pix;
          unsigned w4[4] = {0u, 0u, 0u, 0u};
          if (draws == nullptr) philox_block(idx, (unsigned)qi, P.seed, w4);
          const size_t di = ((((size_t)f * 2 + p) * kBins + c) * P.HW + pix) * (size_t)P.draws_m + 4 * qi;
          Elem* dst = elems + warp_slot + ebefore;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (i < nev) {
              float u;
              if (draws != nullptr) u = (4 * qi + i < P.draws_m) ? __ldg(draws + di + i) : 0.f;
              else u = __fmul_rn((float)(w4[i] >> 8), 5.9604644775390625e-08f);   // 2^-24
              float t;
              if (P.multi_events == 2) {
                t = u;                                   // 'random': additional_ts = raw draw (LDATI.py:173-174)
              } else if (kk == 0.f) {
                t = P.true_div ? __fdiv_rn(__fdiv_rn(u, P.fps32), P.nbins32)
                               : __fmul_rn(__fmul_rn(u, P.r_fps32), P.r_nbins32);
              } else {
                const float disc = __fadd_rn(bb2, __fmul_rn(k2, u));
                t = __fdiv_rn(__fadd_rn(-b, __fsqrt_rn(disc)), kk);
              }
              t = __fadd_rn(t, bstart);
              t = __fmul_rn(t, 1e6f);
              const bool is_nan = (t != t);
              const long long ts = is_nan ? P.nan_ts : (long long)t;
              dst[i] = make_elem<Elem>(ts, is_nan, bin_base, pol, pix, P.pix_bits, P.key_bits, status);
            }
          }
        }
      }
    } else if (active) {
      // a pixel-bin with >= 1024 events (out-of-contract voxel values): per-lane loop
      long long slot_m = s_base[kBins + c] + s_wpre[warp][kBins + c] + exm;
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int nc = cnt[v];
        const int pix = pix0 + v;
        const float2 par = s_par[warp][lane][v];
        const float kk = par.x, b = par.y;
        const float bb2 = __fmul_rn(b, b);
        const float k2 = __fmul_rn(2.f, kk);
        const unsigned long long idx = ((frame * 2ull + (unsigned)p) * 9ull + (unsigned)c) * (unsigned long long)P.HW + (unsigned)pix;
#pragma unroll 1
        for (int j = 0; j < nc; ++j) {
          float u;
          if (draws != nullptr) {
            const size_t di = ((((size_t)f * 2 + p) * kBins + c) * P.HW + pix) * (size_t)P.draws_m + j;
            u = (j < P.draws_m) ? __ldg(draws + di) : 0.f;
          } else {
            u = philox_uniform(idx, (unsigned)j, P.seed);
          }
          float t;
          if (P.multi_events == 2) {
            t = u;                                   // 'random': additional_ts = raw draw (LDATI.py:173-174)
          } else if (kk == 0.f) {
            t = P.true_div ? __fdiv_rn(__fdiv_rn(u, P.fps32), P.nbins32)
                           : __fmul_rn(__fmul_rn(u, P.r_fps32), P.r_nbins32);
          } else {
            const float disc = __fadd_rn(bb2, __fmul_rn(k2, u));
            t = __fdiv_rn(__fadd_rn(-b, __fsqrt_rn(disc)), kk);
          }
          t = __fadd_rn(t, bstart);
          t = __fmul_rn(t, 1e6f);
          const bool is_nan = (t != t);
          const long long ts = is_nan ? P.nan_ts : (long long)t;
          elems[slot_m++] = make_elem<Elem>(ts, is_nan, bin_base, pol, pix, P.pix_bits, P.key_bits, status);
        }
      }
    }
    __syncwarp();
    // advance the window: bin c+2 becomes `next`
#pragma unroll
    for (int v = 0; v < V; ++v) { n_prev[v] = n_cur[v]; n_cur[v] = n_next[v]; tend_cur[v] = tend_next[v]; n_next[v] = 0; }
    if (BIDIR) {
      if (c + 2 < kBins) {
#pragma unroll
        for (int v = 0; v < V; ++v) { n_next[v] = n_all[v][c + 2]; tend_next[v] = tend_all[v][c + 2]; }
      }
    } else if (active && c + 2 < kBins) {
      float yn[V];
      load_bin<V>(plane0, P.HW, pix0, c + 2, yn);
#pragma unroll
      for (int v = 0; v < V; ++v)
        relocate_step(yn[v], y9[v], c + 2 == kBins - 1, P.eps6, debt[v], n_next[v], tend_next[v]);
    }
  }
}

// ---------------------------------------------------------------------------------------
// K6: segmented stable LSD radix sort on the key field (one-sweep passes, osw_*).  Tiles never straddle segments.
// ---------------------------------------------------------------------------------------
struct SortWs {
  void* elem_a;
  void* elem_b;
  int32_t* tile_first;   // [NS+1] first 4096-key tile of each segment (exclusive scan of tiles per segment)
  int32_t* tile_seg;     // [NT_max]
  char* osw_zero;        // start of the region cleared before every call: tickets, histograms, look-back state
  size_t osw_zero_bytes;
  int32_t* tickets;      // [kOswMaxPasses]
  int32_t* seg_hist;     // [kOswMaxPasses][NS][64]
  unsigned long long* tstate;   // [kOswMaxPasses][NT_max][64]
  int32_t* chunk_seg;    // [ceil(total / 128)] segment of the first record of every 128-record pack chunk
  size_t bytes;
  int nt_max;
};

static SortWs carve_sort_ws(void* ws, const Geometry& g, int64_t total, int elem_bytes) {
  Arena a(ws, (size_t)-1);
  SortWs s;
  const int ns = g.F * kBins;
  s.elem_a = a.take<char>((size_t)(total > 0 ? total : 1) * elem_bytes);
  s.elem_b = a.take<char>((size_t)(total > 0 ? total : 1) * elem_bytes);
  s.nt_max = (int)((total + kOswTile - 1) / kOswTile) + ns;
  s.tile_first = a.take<int32_t>((size_t)ns + 1);
  s.tile_seg = a.take<int32_t>((size_t)s.nt_max);
  const int passes = osw_passes(g.key_bits);
  s.tickets = a.take<int32_t>(kOswMaxPasses);
  s.osw_zero = reinterpret_cast<char*>(s.tickets);
  s.seg_hist = a.take<int32_t>((size_t)passes * ns * kOswRadix);
  s.tstate = a.take<unsigned long long>((size_t)passes * s.nt_max * kOswRadix);
  s.osw_zero_bytes = (size_t)((a.base + a.off) - s.osw_zero);
  s.chunk_seg = a.take<int32_t>((size_t)(total / kPackRecsPerWarpDecl) + 2);
  s.bytes = align_up(a.off, 256);
  return s;
}

// one block: tiles per segment -> tile_first (exclusive scan) and tile_seg
__global__ void build_tiles_kernel(const int64_t* __restrict__ seg_start, int ns, int tile, int32_t* __restrict__ tile_first) {
  __shared__ int carry_s;
  __shared__ int wsum[32];
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < ns; base += blockDim.x) {
    const int s = base + threadIdx.x;
    int nt = 0;
    if (s < ns) nt = (int)((seg_start[s + 1] - seg_start[s] + tile - 1) / tile);
    int inc = warp_incl_scan(nt);
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
      int w = (threadIdx.x < (blockDim.x >> 5)) ? wsum[threadIdx.x] : 0;
      int wi = warp_incl_scan(w);
      wsum[threadIdx.x] = wi - w;
    }
    __syncthreads();
    const int first = carry_s + wsum[threadIdx.x >> 5] + inc - nt;
    if (s < ns) tile_first[s] = first;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = first + nt;
    __syncthreads();
  }
  if (threadIdx.x == 0) tile_first[ns] = carry_s;
}

// tile -> segment: one thread per tile, binary search over tile_first (a dense segment owns hundreds of tiles; one
// thread per SEGMENT writing them serially cost 53 us on the dense microbench)
__global__ void fill_tile_seg_kernel(const int32_t* __restrict__ tile_first, int ns, int32_t* __restrict__ tile_seg) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= tile_first[ns]) return;
  int lo = 0, hi = ns - 1;                       // last segment s with tile_first[s] <= t (empty segments repeat values)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (tile_first[mid] <= t) lo = mid; else hi = mid - 1;
  }
  tile_seg[t] = lo;
}

// ---------------------------------------------------------------------------------------
// K6 passes.  A histogram / scan / scatter sort on 2048-key tiles spent 140 us per pass for 21.6 M keys in its
// scatter alone (88 % of the ADU pipe: eight dependent __match_any_sync rounds per thread rank the keys;
// profiles/ncu_ldati_r2_a.txt), plus a histogram kernel, three scan kernels and a second read of every key per pass.
// Here a pass is ONE kernel over 4096-key tiles:
//   * the tile's digit counts are chained to the tiles before it IN ITS SEGMENT by decoupled look-back (one 64-bit
//     status word per (tile, digit): flag | count); tiles take tickets from an atomic counter, so a tile only ever
//     waits for tiles that already run;
//   * the digit bases inside a segment come from a per-segment histogram: of the first pass from one read of the keys
//     (osw_hist_kernel), of every later pass from the scatter pass before it, which has the keys in registers;
//   * the tile is ordered by digit in shared memory and leaves as runs of consecutive addresses.
// ---------------------------------------------------------------------------------------
constexpr unsigned long long kOswFlagAgg = 1ull << 62, kOswFlagIncl = 2ull << 62, kOswValMask = (1ull << 62) - 1ull;

// digit histograms of ALL passes per segment, from one read of the keys
template <typename Elem>
__global__ void __launch_bounds__(kThreads) osw_hist_kernel(const Elem* __restrict__ in, const int64_t* __restrict__ seg_start,
                                                             const int32_t* __restrict__ tile_first,
                                                             const int32_t* __restrict__ tile_seg, int ns, int shift0, int rb,
                                                             int passes, int32_t* __restrict__ seg_hist) {
  const int tile = blockIdx.x;
  if (tile >= tile_first[ns]) return;
  const int seg = tile_seg[tile];
  const int tin = tile - tile_first[seg];
  const long long start = seg_start[seg] + (long long)tin * kOswTile;
  const int cnt = (int)min((long long)kOswTile, seg_start[seg + 1] - start);
  __shared__ int h[kOswMaxPasses][kOswRadix];
  for (int i = threadIdx.x; i < kOswMaxPasses * kOswRadix; i += kThreads) (&h[0][0])[i] = 0;
  __syncthreads();
  const unsigned mask = (1u << rb) - 1u;
  const int lane = threadIdx.x & 31;
  Elem key[kOswKpt];
#pragma unroll
  for (int k = 0; k < kOswKpt; ++k) {                       // all loads in flight before the first use
    const int i = k * kThreads + threadIdx.x;
    key[k] = (i < cnt) ? in[start + i] : (Elem)0;
  }
#pragma unroll
  for (int k = 0; k < kOswKpt; ++k) {
    const bool valid = k * kThreads + (int)threadIdx.x < cnt;
    const unsigned vm = __ballot_sync(0xffffffffu, valid);
    if (vm == 0u) continue;
    const int first = __ffs(vm) - 1;
    for (int p = 0; p < passes; ++p) {
      const unsigned d = (unsigned)(key[k] >> (shift0 + p * rb)) & mask;
      // massive ties (a sparse clip: thousands of events share one timestamp) would serialise on one counter
      const unsigned d0 = __shfl_sync(0xffffffffu, d, first);
      if (__all_sync(0xffffffffu, !valid || d == d0)) {
        if (lane == first) atomicAdd(&h[p][d0], __popc(vm));
      } else if (valid) {
        atomicAdd(&h[p][d], 1);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < passes * kOswRadix; i += kThreads) {
    const int c = (&h[0][0])[i];
    if (c) atomicAdd(&seg_hist[((size_t)(i / kOswRadix) * ns + seg) * kOswRadix + (i % kOswRadix)], c);
  }
}

__device__ __forceinline__ int osw_pad(int i) { return i + (i >> 5); }        // counters: one pad word per 32
__device__ __forceinline__ int osw_pad16(int i) { return i + (i >> 4); }      // key transpose: one pad slot per 16
constexpr int kOswCounterWords = 32 * kThreads + (32 * kThreads >> 5);         // 8448
constexpr int kOswStageSlots = kOswTile + (kOswTile >> 4);                     // 4352

// One pass.  Ranking without match / atomics: every thread counts the digits of its 16 CONSECUTIVE keys in private
// packed 16-bit counters in shared memory ([32 lanes][256 threads] words, two digits per word); one padded raking
// scan over (digit, thread) turns the counters into tile-local stable positions.  Keys are loaded coalesced and
// transposed to the blocked arrangement through (padded) shared memory.  103 us per pass for 21.6 M keys (1.7 TB/s of
// key traffic, 73 % of the shared-memory wavefront peak).  Measured and not adopted: ranking with one ballot per
// digit bit in warp-private counters (CUB's match-by-bits): fewer shared-memory wavefronts (41 %) but 72 % of the ALU
// pipe, 119-129 us per pass (profiles/ncu_ldati_r2_c.txt).
template <typename Elem>
__global__ void __launch_bounds__(kThreads, 4) osw_scatter_kernel(const Elem* __restrict__ in, Elem* __restrict__ out,
                                                                const int64_t* __restrict__ seg_start,
                                                                const int32_t* __restrict__ tile_first,
                                                                const int32_t* __restrict__ tile_seg, int ns, int shift, int rb,
                                                                const int32_t* __restrict__ seg_hist,      // [ns][64], this pass
                                                                unsigned long long* tstate,               // [nt][64], this pass
                                                                int32_t* __restrict__ ticket) {
  extern __shared__ __align__(16) unsigned char osw_smem[];
  uint32_t* cntw = reinterpret_cast<uint32_t*>(osw_smem);      // packed digit counters, later their exclusive scan
  Elem* stage = reinterpret_cast<Elem*>(osw_smem);             // aliases the counters (used before and after them)
  __shared__ int s_tile;
  __shared__ int lbase[kOswRadix + 1];                         // tile-local position of each digit's first key
  __shared__ int delta[kOswRadix];                             // (position in the segment) - (position in the tile) per digit
  __shared__ uint32_t wsum[kThreads / 32];
  __shared__ uint32_t s_total;
  __shared__ int hsum[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1);
  __syncthreads();
  const int tile = s_tile;
  if (tile >= tile_first[ns]) return;
  const int seg = tile_seg[tile];
  const int tfirst = tile_first[seg];
  const int tin = tile - tfirst;
  const long long sstart = seg_start[seg];
  const long long start = sstart + (long long)tin * kOswTile;
  const int cnt = (int)min((long long)kOswTile, seg_start[seg + 1] - start);
  const unsigned mask = (1u << rb) - 1u;

  // ---- coalesced load, transpose to blocked: thread t owns keys [16t, 16t+16) of the tile ----
#pragma unroll
  for (int k = 0; k < kOswKpt; ++k) {
    const int i = k * kThreads + tid;
    stage[osw_pad16(i)] = (i < cnt) ? in[start + i] : (Elem)0;
  }
  __syncthreads();
  Elem key[kOswKpt];
#pragma unroll
  for (int j = 0; j < kOswKpt; ++j) key[j] = stage[osw_pad16(kOswKpt * tid + j)];
  __syncthreads();

  // ---- private packed counters: digit d -> word (d & 31, tid), half (d >> 5) ----
#pragma unroll
  for (int l = 0; l < 32; ++l) cntw[osw_pad(l * kThreads + tid)] = 0u;
  // (own column only: no barrier needed before the thread's own increments)
  int lpos[kOswKpt];                                           // first the rank among the thread's own keys
  const int nvalid = min(max(cnt - kOswKpt * tid, 0), kOswKpt);
#pragma unroll
  for (int j = 0; j < kOswKpt; ++j) {
    lpos[j] = 0;
    if (j < nvalid) {
      const unsigned d = (unsigned)(key[j] >> shift) & mask;
      unsigned short* c = reinterpret_cast<unsigned short*>(cntw + osw_pad((int)(d & 31u) * kThreads + tid)) + (d >> 5);
      const unsigned short r = *c;
      lpos[j] = r;
      *c = (unsigned short)(r + 1);
    }
  }
  __syncthreads();
  // ---- raking exclusive scan over the flat (lane-major, thread-minor) counter array; both halves at once ----
  {
    uint32_t sum = 0u;
#pragma unroll
    for (int j = 0; j < 32; ++j) sum += cntw[33 * tid + j];                        // osw_pad(32*tid + j) == 33*tid + j
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t woff = 0u, total = 0u;
#pragma unroll
    for (int wv = 0; wv < kThreads / 32; ++wv) { const uint32_t t = wsum[wv]; if (wv < warp) woff += t; total += t; }
    if (tid == 0) s_total = total;
    uint32_t run = woff + inc - sum;
#pragma unroll
    for (int j = 0; j < 32; ++j) { const uint32_t wv = cntw[33 * tid + j]; cntw[33 * tid + j] = run; run += wv; }
  }
  __syncthreads();
  const int total_lo = (int)(s_total & 0xffffu);                // keys whose digit is < 32
  // ---- tile-local stable positions; digit starts ----
#pragma unroll
  for (int j = 0; j < kOswKpt; ++j) {
    const unsigned d = (unsigned)(key[j] >> shift) & mask;
    const uint32_t wv = cntw[osw_pad((int)(d & 31u) * kThreads + tid)];
    lpos[j] += (d >> 5) ? total_lo + (int)(wv >> 16) : (int)(wv & 0xffffu);
  }
  int my_start = 0;
  if (tid < kOswRadix) {
    const uint32_t wv = cntw[osw_pad((tid & 31) * kThreads)];
    my_start = (tid >> 5) ? total_lo + (int)(wv >> 16) : (int)(wv & 0xffffu);
    lbase[tid] = my_start;
  }
  if (tid == 0) lbase[kOswRadix] = cnt;
  // digit bases inside the segment: exclusive scan of the segment's histogram of this pass (64 values, two warps)
  int hcount = 0, hinc = 0;
  if (tid < kOswRadix) {
    hcount = seg_hist[(size_t)seg * kOswRadix + tid];
    hinc = hcount;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, hinc, o);
      if (lane >= o) hinc += t;
    }
    if (lane == 31) hsum[warp] = hinc;
  }
  __syncthreads();                                             // counters are dead from here: `stage` may be written
  // ---- decoupled look-back over the earlier tiles of this segment, one thread per digit ----
  if (tid < kOswRadix) {
    const long long digit_base = (long long)(hinc - hcount) + (warp == 1 ? hsum[0] : 0);
    const unsigned long long mine = (unsigned long long)(lbase[tid + 1] - my_start);
    volatile unsigned long long* st = tstate + (size_t)tile * kOswRadix + tid;
    unsigned long long excl = 0ull;
    if (tin == 0) {
      *st = kOswFlagIncl | mine;
    } else {
      *st = kOswFlagAgg | mine;
      int look = tile - 1;
      while (true) {
        const unsigned long long v = *(volatile unsigned long long*)(tstate + (size_t)look * kOswRadix + tid);
        if ((v >> 62) == 0ull) continue;                       // not published yet: that tile holds an earlier ticket
        excl += v & kOswValMask;
        if ((v >> 62) == 2ull) break;
        --look;
      }
      *st = kOswFlagIncl | (excl + mine);
    }
    delta[tid] = (int)(digit_base + (long long)excl) - my_start;
  }
  // ---- order the tile by digit in shared memory, then write every digit's run to consecutive addresses ----
#pragma unroll
  for (int j = 0; j < kOswKpt; ++j)
    if (j < nvalid) stage[lpos[j]] = key[j];
  __syncthreads();
  Elem* dst = out + sstart;
#pragma unroll 4
  for (int k = 0; k < kOswKpt; ++k) {
    const int i = k * kThreads + tid;
    if (i < cnt) {
      const Elem e = stage[i];
      const unsigned d = (unsigned)(e >> shift) & mask;
      dst[delta[d] + i] = e;
    }
  }
}

// ---------------------------------------------------------------------------------------
// K7: 13-byte records, linear over the whole sorted stream.  FOUR consecutive records are exactly 13 aligned 32-bit
// words, so a thread loads four elements with one 16-byte load, builds their 13 words in registers with fixed byte
// permutes, and the warp transposes its 32 x 13 words through shared memory (stride 13: conflict free) into 416
// consecutive words that leave as 16-byte coalesced stores.  No byte stores anywhere.  Staging bytes through shared
// memory with 13 one-byte stores per record reached 92 % of the LSU wavefront peak and took 103 us for 21.6 M
// events; assembling the words with 5 shuffles each was worse (230 us, 311 instructions per 32 records --
// profiles/ncu_ldati_r2_c.txt).  A record's segment (bin origin, frame offset) is found from a per-128-record table.
// ---------------------------------------------------------------------------------------
constexpr int kPackRecsPerWarp = kPackRecsPerWarpDecl;

// segment of the first record of every 128-record chunk: one thread per chunk, binary search over seg_start
__global__ void pack_chunk_seg_kernel(const int64_t* __restrict__ seg_start, int ns, long long total,
                                      int32_t* __restrict__ chunk_seg) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long r = c * kPackRecsPerWarp;
  if (r >= total) return;
  int lo = 0, hi = ns - 1;                       // last segment s with seg_start[s] <= r (empty segments repeat values)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (seg_start[mid] <= r) lo = mid; else hi = mid - 1;
  }
  chunk_seg[c] = lo;
}

template <typename Elem>
__global__ void __launch_bounds__(kThreads) pack_linear_kernel(const Elem* __restrict__ in, const int64_t* __restrict__ seg_start,
                                                                const int32_t* __restrict__ chunk_seg, int ns, long long total,
                                                                DevParams P, const int64_t* __restrict__ frame_offset_us,
                                                                uint8_t* __restrict__ out) {
  __shared__ __align__(16) unsigned sm[kThreads / 32][32 * 13];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long chunk = (long long)blockIdx.x * (kThreads / 32) + warp;
  const long long r0 = chunk * kPackRecsPerWarp;
  if (r0 >= total) return;                                   // whole warp
  const int nrec = (int)min((long long)kPackRecsPerWarp, total - r0);
  const long long mine = r0 + 4 * lane;                      // this lane's four records
  const unsigned long long pix_mask = (1ull << P.pix_bits) - 1ull;
  // elements: the sort buffers are 256-byte aligned and `mine` is a multiple of 4 -> one 16-byte (32-byte) load
  Elem e[4] = {0, 0, 0, 0};
  if (4 * lane + 3 < nrec) {
    if (sizeof(Elem) == 4) {
      const uint4 t = __ldg(reinterpret_cast<const uint4*>(in + mine));
      e[0] = (Elem)t.x; e[1] = (Elem)t.y; e[2] = (Elem)t.z; e[3] = (Elem)t.w;
    } else {
      const ulonglong2 t0 = __ldg(reinterpret_cast<const ulonglong2*>(in + mine));
      const ulonglong2 t1 = __ldg(reinterpret_cast<const ulonglong2*>(in + mine + 2));
      e[0] = (Elem)t0.x; e[1] = (Elem)t0.y; e[2] = (Elem)t1.x; e[3] = (Elem)t1.y;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * lane + j < nrec) e[j] = in[mine + j];
  }
  int seg = chunk_seg[chunk];
  unsigned w[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const long long idx = mine + j;
    if (4 * lane + j < nrec) {
      while (seg + 1 < ns && idx >= seg_start[seg + 1]) ++seg;     // rarely more than zero steps (L1 hits)
    }
    const int f = seg / P.segs_per_frame, c = seg - f * P.segs_per_frame;
    const long long base_ts = P.bin_base[c] - kKeyBias;
    long long off = 0;
    if (P.add_frame_offset && frame_offset_us != nullptr) off = frame_offset_us[f];
    const unsigned long long ev = (unsigned long long)e[j];
    const unsigned pix = (unsigned)(ev & pix_mask);
    const long long key = (long long)(ev >> (P.pix_bits + 1));
    long long ts = (key == 0) ? P.nan_ts : (base_ts + key);
    ts = (long long)((unsigned long long)ts + (unsigned long long)off);
    const unsigned y = pix / (unsigned)P.W, x = pix - y * (unsigned)P.W;
    w[4 * j + 0] = (unsigned)((unsigned long long)ts);
    w[4 * j + 1] = (unsigned)((unsigned long long)ts >> 32);
    w[4 * j + 2] = (x & 0xffffu) | (y << 16);
    w[4 * j + 3] = (unsigned)((ev >> P.pix_bits) & 1ull);          // polarity byte
  }
  // 4 x 13 bytes -> 13 words: record j starts at byte 13 j, i.e. at byte (j) of word 3 j + ... (fixed permutes)
  unsigned o[13];
  o[0] = w[0];  o[1] = w[1];  o[2] = w[2];
  o[3] = (w[3] & 0xffu) | (w[4] << 8);
  o[4] = __funnelshift_r(w[4], w[5], 24);
  o[5] = __funnelshift_r(w[5], w[6], 24);
  o[6] = (w[6] >> 24) | ((w[7] & 0xffu) << 8) | (w[8] << 16);
  o[7] = __funnelshift_r(w[8], w[9], 16);
  o[8] = __funnelshift_r(w[9], w[10], 16);
  o[9] = (w[10] >> 16) | ((w[11] & 0xffu) << 16) | (w[12] << 24);
  o[10] = __funnelshift_r(w[12], w[13], 8);
  o[11] = __funnelshift_r(w[13], w[14], 8);
  o[12] = (w[14] >> 8) | (w[15] << 24);
  unsigned* row = sm[warp];
#pragma unroll
  for (int k = 0; k < 13; ++k) row[13 * lane + k] = o[k];
  __syncwarp();
  unsigned char* gdst = out + (unsigned long long)r0 * 13ull;   // 128 records * 13 B = 1664 B per chunk: 16-byte aligned
  const int nbytes = nrec * 13;
  const unsigned long long galign = (unsigned long long)(uintptr_t)gdst;
  if (nrec == kPackRecsPerWarp && (galign & 15ull) == 0ull) {
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const int v = lane + 32 * m;                            // 104 vectors of 16 bytes
      if (v < 104) reinterpret_cast<uint4*>(gdst)[v] = reinterpret_cast<const uint4*>(row)[v];
    }
  } else {                                                    // the stream's last chunk, or a caller buffer that is not 16-byte aligned
    for (int k = lane; 4 * k < nbytes; k += 32) {
      if (4 * k + 4 <= nbytes && (galign & 3ull) == 0ull) {
        reinterpret_cast<unsigned*>(gdst)[k] = row[k];
      } else {
        for (int t = 0; t < 4 && 4 * k + t < nbytes; ++t) gdst[4 * k + t] = (unsigned char)(row[k] >> (8 * t));
      }
    }
  }
}

template <int V>
__global__ void relocate_debug_kernel(const float* __restrict__ vox, int HW, float eps6, int bidirectional,
                                      int32_t* __restrict__ counts, float* __restrict__ tend_out) {
  const int plane = blockIdx.y;   // f*2+p
  const int pix = (blockIdx.x * blockDim.x + threadIdx.x) * V;
  if (pix >= HW) return;
  float y[V][10];
  load_pixels<V>(vox + (size_t)plane * 10 * HW, HW, pix, y);
#pragma unroll
  for (int v = 0; v < V; ++v) {
    int n[kBins];
    float tend[kBins];
    if (bidirectional) relocate_pixel_bidir(y[v], eps6, n, tend);
    else relocate_pixel(y[v], eps6, n, tend);
#pragma unroll
    for (int c = 0; c < kBins; ++c) {
      counts[((size_t)plane * kBins + c) * HW + pix + v] = n[c];
      if (tend_out != nullptr) tend_out[((size_t)plane * kBins + c) * HW + pix + v] = tend[c];
    }
  }
}

// ---------------------------------------------------------------------------------------
// Baseline samplers 'random' / 'even' (stage-2 comparison methods; SURVEY.md 8f N4;
// /root/reference/train/scripts/stage2/sample_methods/random_even_sample.py:118-170).  No count relocation: every voxel
// value y of the TEN bins yields floor(y) events -- at u * delta ('random') or j / (floor(y) + 1) * delta ('even') into its
// bin -- plus one more with probability frac(y) at u * delta / floor(y) / (floor(y) + 1) * delta; a frame's events are
// sorted by timestamp.  Same structure as LDATI: count pass -> scans -> emit to generation-order slots -> one-sweep sort
// (one segment per FRAME, 16-bit keys at 30 fps: three passes over 64-bit elements) -> records.
// Generation order g: [bin c][negative plane, positive plane][integer-part events (pixel, j), fractional-part events].
// ---------------------------------------------------------------------------------------
constexpr int kBaseBins = 10;
constexpr int kBaseQ = 2 * kBaseBins;      // per plane: (bin, kind) with kind 0 = integer-part events, 1 = fractional-part events

struct BaseDev {
  int H, W, HW, F, NB;
  int mode;                 // 1 random, 2 even
  long long frame_base;
  unsigned long long seed;
  float delta32;
  float start[kBaseBins];
  long long key_base;       // timestamps are stored as key = ts - key_base + kKeyBias
  int pix_bits, key_bits;
};

struct BaseWs {
  int32_t* partial;       // [F][2][NB][20]
  int32_t* block_base;    // [F][2][NB][20]
  int32_t* group_base;    // [F][10][4]: neg int, neg frac, pos int, pos frac
  int64_t* seg_start;     // [F+1]
  size_t bytes;
};

static BaseWs carve_base_ws(void* ws, int F, int NB) {
  Arena a(ws, (size_t)-1);
  BaseWs w;
  const size_t n = (size_t)F * 2 * NB * kBaseQ;
  w.partial = a.take<int32_t>(n);
  w.block_base = a.take<int32_t>(n);
  w.group_base = a.take<int32_t>((size_t)F * kBaseBins * 4);
  w.seg_start = a.take<int64_t>((size_t)F + 1);
  w.bytes = align_up(a.off, 256);
  return w;
}

// events of one pixel-bin: floor(y) integer-part events and the Bernoulli(frac) one
__device__ __forceinline__ void base_counts(float y, unsigned long long idx, unsigned long long seed, int& n_int, int& n_frac,
                                            float& ip) {
  ip = floorf(y);
  n_int = ip > 0.f ? __float2int_rz(ip) : 0;
  const float frac = __fsub_rn(y, ip);
  n_frac = philox_uniform_stream(idx, 0u, seed, 2u) < frac ? 1 : 0;       // torch.bernoulli(p): u < p
}

template <int V>
__global__ void __launch_bounds__(kThreads) base_count_kernel(const float* __restrict__ vox, BaseDev P, int32_t* __restrict__ partial) {
  const int blk = blockIdx.x, p = blockIdx.y, f = blockIdx.z;
  const int pix = (blk * kThreads + threadIdx.x) * V;
  int tot[kBaseQ];
#pragma unroll
  for (int q = 0; q < kBaseQ; ++q) tot[q] = 0;
  if (pix < P.HW) {
    float y[V][10];
    load_pixels<V>(vox + ((size_t)(f * 2 + p) * 10) * P.HW, P.HW, pix, y);
    const unsigned long long plane = ((unsigned long long)(P.frame_base + f) * 2ull + (unsigned)p) * (unsigned long long)kBaseBins;
#pragma unroll
    for (int v = 0; v < V; ++v)
#pragma unroll
      for (int c = 0; c < kBaseBins; ++c) {
        int ni, nf;
        float ip;
        base_counts(y[v][c], (plane + (unsigned)c) * (unsigned long long)P.HW + (unsigned)(pix + v), P.seed, ni, nf, ip);
        tot[2 * c] += ni;
        tot[2 * c + 1] += nf;
      }
  }
  __shared__ int red[kThreads / 32][kBaseQ];
#pragma unroll
  for (int q = 0; q < kBaseQ; ++q) {
    int v = tot[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][q] = v;
  }
  __syncthreads();
  if (threadIdx.x < kBaseQ) {
    int sum = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) sum += red[w][threadIdx.x];
    partial[(((size_t)f * 2 + p) * P.NB + blk) * kBaseQ + threadIdx.x] = sum;
  }
}

// per frame: exclusive scan of the block partials over each plane, the 40 group bases, the frame total
__global__ void base_scan_kernel(const int32_t* __restrict__ partial, int32_t* __restrict__ block_base,
                                 int32_t* __restrict__ group_base, int64_t* __restrict__ frame_counts, int NB) {
  const int f = blockIdx.x;
  __shared__ int tot[2][kBaseQ];
  const int t = threadIdx.x;
  if (t < 2 * kBaseQ) {
    const int p = t / kBaseQ, q = t % kBaseQ;
    const size_t base = ((size_t)f * 2 + p) * NB * kBaseQ + q;
    int run = 0;
    for (int b = 0; b < NB; ++b) {
      block_base[base + (size_t)b * kBaseQ] = run;
      run += partial[base + (size_t)b * kBaseQ];
    }
    tot[p][q] = run;
  }
  __syncthreads();
  if (t == 0) {
    long long run = 0;
    for (int c = 0; c < kBaseBins; ++c) {
      int32_t* gb = group_base + ((size_t)f * kBaseBins + c) * 4;
      // negative plane (p-index 1) first, inside a plane integer-part events before fractional-part events
      gb[0] = (int32_t)run; run += tot[1][2 * c];
      gb[1] = (int32_t)run; run += tot[1][2 * c + 1];
      gb[2] = (int32_t)run; run += tot[0][2 * c];
      gb[3] = (int32_t)run; run += tot[0][2 * c + 1];
    }
    frame_counts[f] = run;
  }
}

template <int V>
__global__ void __launch_bounds__(kThreads) base_emit_kernel(const float* __restrict__ vox, BaseDev P,
                                                              const int32_t* __restrict__ block_base,
                                                              const int32_t* __restrict__ group_base,
                                                              const int64_t* __restrict__ seg_start,
                                                              unsigned long long* __restrict__ elems, int32_t* __restrict__ status) {
  const int blk = blockIdx.x, p = blockIdx.y, f = blockIdx.z;
  const int pix0 = (blk * kThreads + threadIdx.x) * V;
  const bool active = pix0 < P.HW;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int pol = 1 - p;
  const size_t bb = (((size_t)f * 2 + p) * P.NB + blk) * kBaseQ;
  const long long frame_start = seg_start[f];
  const unsigned long long plane = ((unsigned long long)(P.frame_base + f) * 2ull + (unsigned)p) * (unsigned long long)kBaseBins;
  __shared__ int wsum[kThreads / 32][2];
  float y[V][10];
#pragma unroll
  for (int v = 0; v < V; ++v)
#pragma unroll
    for (int c = 0; c < 10; ++c) y[v][c] = 0.f;
  if (active) load_pixels<V>(vox + ((size_t)(f * 2 + p) * 10) * P.HW, P.HW, pix0, y);
#pragma unroll 1
  for (int c = 0; c < kBaseBins; ++c) {
    int ni[V], nf[V];
    float ip[V];
    int ti = 0, tf = 0;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      ni[v] = nf[v] = 0; ip[v] = 0.f;
      if (active) {
        float yc = y[0][0];
#pragma unroll
        for (int cc = 0; cc < 10; ++cc) if (cc == c) yc = y[v][cc];            // register select (c is a runtime index)
        base_counts(yc, (plane + (unsigned)c) * (unsigned long long)P.HW + (unsigned)(pix0 + v), P.seed, ni[v], nf[v], ip[v]);
      }
      ti += ni[v]; tf += nf[v];
    }
    const int inc_i = warp_incl_scan(ti), inc_f = warp_incl_scan(tf);
    if (lane == 31) { wsum[warp][0] = inc_i; wsum[warp][1] = inc_f; }
    __syncthreads();
    int wi = 0, wf = 0;
    for (int w = 0; w < warp; ++w) { wi += wsum[w][0]; wf += wsum[w][1]; }
    __syncthreads();
    const int32_t* gb = group_base + ((size_t)f * kBaseBins + c) * 4;
    const int grp = (p == 1) ? 0 : 2;
    long long slot_i = frame_start + gb[grp] + block_base[bb + 2 * c] + wi + (inc_i - ti);
    long long slot_f = frame_start + gb[grp + 1] + block_base[bb + 2 * c + 1] + wf + (inc_f - tf);
    const float st = P.start[c];
    auto put = [&](long long slot, float t, int pix) {
      t = __fmul_rn(__fadd_rn(t, st), 1e6f);
      const bool bad = !(t == t) || fabsf(t) > 9.0e18f;
      const long long ts = bad ? LLONG_MIN : (long long)t;
      long long key = ts - P.key_base + kKeyBias;
      const long long kmax = (1LL << P.key_bits) - 1;
      if (bad || key < 1 || key > kmax) {               // non-finite or far outside the frame: flagged, the host raises
        atomicAdd(status + 0, 1);
        key = key < 1 ? 1 : kmax;
      }
      elems[slot] = ((unsigned long long)key << (P.pix_bits + 1)) | ((unsigned long long)pol << P.pix_bits) |
                    (unsigned long long)pix;
    };
    if (active) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const unsigned long long idx = (plane + (unsigned)c) * (unsigned long long)P.HW + (unsigned)(pix0 + v);
        const float den = __fadd_rn(ip[v], 1.f);
        for (int j = 0; j < ni[v]; ++j) {
          const float t = P.mode == 1 ? __fmul_rn(philox_uniform_stream(idx, (unsigned)j, P.seed, 0u), P.delta32)
                                      : __fmul_rn(__fdiv_rn((float)j, den), P.delta32);
          put(slot_i++, t, pix0 + v);
        }
        if (nf[v]) {
          const float t = P.mode == 1 ? __fmul_rn(philox_uniform_stream(idx, 0u, P.seed, 1u), P.delta32)
                                      : __fmul_rn(__fdiv_rn(ip[v], den), P.delta32);
          put(slot_f++, t, pix0 + v);
        }
      }
    }
  }
}

static int validate_base(const v2ce_baseline_params* p) {
  V2CE_REQUIRE(p != nullptr, "params is NULL");
  V2CE_REQUIRE(p->height > 0 && p->width > 0 && p->n_frames > 0, "bad geometry %dx%d x %d frames", p->height, p->width,
               p->n_frames);
  V2CE_REQUIRE(p->width < 32768 && p->height < 32768, "x/y are int16 fields: H,W must be < 32768");
  V2CE_REQUIRE((long long)p->height * p->width < (1LL << 30), "plane too large");
  V2CE_REQUIRE(p->n_frames <= 65535, "at most 65535 frames per call (grid.z)");
  V2CE_REQUIRE(p->mode == 1 || p->mode == 2, "mode must be 1 ('random') or 2 ('even')");
  V2CE_REQUIRE(p->key_span > 0 && p->key_span < (1 << 30), "bad key_span %d", p->key_span);
  return V2CE_OK;
}

struct BaseGeom { int HW, V, NB, pix_bits, key_bits; };
static BaseGeom base_geom(const v2ce_baseline_params* p) {
  BaseGeom g;
  g.HW = p->height * p->width;
  g.V = (g.HW % 4 == 0) ? 4 : 1;
  g.NB = (g.HW + kThreads * g.V - 1) / (kThreads * g.V);
  g.pix_bits = 1;
  while ((1LL << g.pix_bits) < g.HW) ++g.pix_bits;
  g.key_bits = 1;
  while ((1LL << g.key_bits) < (long long)p->key_span + 1) ++g.key_bits;
  return g;
}
static BaseDev base_dev(const v2ce_baseline_params* p, const BaseGeom& g) {
  BaseDev d;
  d.H = p->height; d.W = p->width; d.HW = g.HW; d.F = p->n_frames; d.NB = g.NB;
  d.mode = p->mode; d.frame_base = p->frame_base; d.seed = p->seed; d.delta32 = p->delta32;
  for (int c = 0; c < kBaseBins; ++c) d.start[c] = p->binstart_t0_32[c];
  d.key_base = p->key_base_us; d.pix_bits = g.pix_bits; d.key_bits = g.key_bits;
  return d;
}

static int validate(const v2ce_ldati_params* p) {
  V2CE_REQUIRE(p != nullptr, "params is NULL");
  V2CE_REQUIRE(p->height > 0 && p->width > 0 && p->n_frames > 0, "bad geometry %dx%d x %d frames", p->height,
               p->width, p->n_frames);
  V2CE_REQUIRE(p->width < 32768 && p->height < 32768, "x/y are int16 fields: H,W must be < 32768");
  V2CE_REQUIRE((long long)p->height * p->width < (1LL << 30), "plane too large");
  V2CE_REQUIRE(p->n_frames <= 65535, "at most 65535 frames per call (grid.z)");
  V2CE_REQUIRE(p->key_span > 0 && p->key_span < (1 << 30), "bad key_span %d", p->key_span);
  V2CE_REQUIRE(p->multi_events >= 0 && p->multi_events <= 2, "multi_events must be 0 ('none'), 1 ('slope') or 2 ('random')");
  V2CE_REQUIRE(p->bidirectional == 0 || p->bidirectional == 1, "bidirectional must be 0 or 1");
  V2CE_REQUIRE(p->pooling >= 0 && p->pooling <= 2, "pooling must be 0 ('none'), 1 ('weighted') or 2 ('avg')");
  V2CE_REQUIRE(p->pooling != 2 || (p->pooling_kernel_size >= 1 && (p->pooling_kernel_size & 1) && p->pooling_kernel_size <= 255),
               "pooling_kernel_size must be odd (an even AvgPool2d kernel changes the plane size; the reference fails too)");
  V2CE_REQUIRE(p->pooling == 0 || p->n_frames * 2 <= 65535, "pooling: at most 32767 frames per call");
  return V2CE_OK;
}

}  // namespace ldati
}  // namespace v2ce

using namespace v2ce;
using namespace v2ce::ldati;

extern "C" size_t v2ce_ldati_params_size(void) { return sizeof(v2ce_ldati_params); }

extern "C" int v2ce_ldati_params_validate(const v2ce_ldati_params* p) { return validate(p); }

extern "C" int v2ce_ldati_count_workspace_bytes(const v2ce_ldati_params* p, size_t* bytes) {
  if (int e = validate(p)) return e;
  V2CE_REQUIRE(bytes != nullptr, "bytes is NULL");
  Geometry g = make_geometry(p);
  *bytes = carve_count_ws(nullptr, g).bytes;
  return V2CE_OK;
}

extern "C" int v2ce_ldati_emit_workspace_bytes(const v2ce_ldati_params* p, int64_t total_events, size_t* bytes) {
  if (int e = validate(p)) return e;
  V2CE_REQUIRE(bytes != nullptr && total_events >= 0, "bad arguments");
  V2CE_REQUIRE(total_events < (1LL << 31) - (1LL << 20), "more than 2^31 events in one call; split the frames");
  Geometry g = make_geometry(p);
  *bytes = carve_sort_ws(nullptr, g, total_events, g.wide ? 8 : 4).bytes;
  return V2CE_OK;
}

extern "C" int v2ce_ldati_count(const float* voxels_dev, const v2ce_ldati_params* p, void* count_ws_dev,
                                size_t count_ws_bytes, int64_t* seg_counts_dev, void* stream) {
  return v2ce_ldati_count_ef(voxels_dev, p, count_ws_dev, count_ws_bytes, seg_counts_dev, nullptr, stream);
}

extern "C" int v2ce_ldati_count_ef(const float* voxels_dev, const v2ce_ldati_params* p, void* count_ws_dev,
                                   size_t count_ws_bytes, int64_t* seg_counts_dev, float* ef_sums_dev, void* stream) {
  if (int e = validate(p)) return e;
  V2CE_REQUIRE(voxels_dev && count_ws_dev && seg_counts_dev, "NULL device pointer");
  Geometry g = make_geometry(p);
  CountWs w = carve_count_ws(count_ws_dev, g);
  if (w.bytes > count_ws_bytes)
    return set_error(V2CE_ERR_WORKSPACE, "count workspace too small: need %zu, got %zu", w.bytes, count_ws_bytes);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DevParams P = make_dev_params(p, g);
  dim3 grid(g.NB, 2, g.F);
  if (p->bidirectional) {
    if (g.V == 4) count_kernel<4, true><<<grid, kThreads, 0, s>>>(voxels_dev, P, w.partial, w.warp_partial, ef_sums_dev);
    else count_kernel<1, true><<<grid, kThreads, 0, s>>>(voxels_dev, P, w.partial, w.warp_partial, ef_sums_dev);
  } else {
    if (g.V == 4) count_kernel<4, false><<<grid, kThreads, 0, s>>>(voxels_dev, P, w.partial, w.warp_partial, ef_sums_dev);
    else count_kernel<1, false><<<grid, kThreads, 0, s>>>(voxels_dev, P, w.partial, w.warp_partial, ef_sums_dev);
  }
  V2CE_LAUNCH_CHECK("ldati::count_kernel");
  if (g.pooling) {
    // the slope of a multi-event pixel-bin is fitted on spatially pooled counts: keep every pixel-bin's count
    if (g.V == 4) {
      dim3 rgrid((g.HW / 4 + 255) / 256, g.F * 2);
      relocate_debug_kernel<4><<<rgrid, 256, 0, s>>>(voxels_dev, g.HW, p->eps6, p->bidirectional, w.counts_all, nullptr);
    } else {
      dim3 rgrid((g.HW + 255) / 256, g.F * 2);
      relocate_debug_kernel<1><<<rgrid, 256, 0, s>>>(voxels_dev, g.HW, p->eps6, p->bidirectional, w.counts_all, nullptr);
    }
    V2CE_LAUNCH_CHECK("ldati::relocate_debug_kernel");
  }
  scan_planes_kernel<<<g.F, 64, 0, s>>>(w.partial, w.block_base, w.group_base, seg_counts_dev, g.NB);
  V2CE_LAUNCH_CHECK("ldati::scan_planes_kernel");
  scan_i64_kernel<<<1, 1024, 0, s>>>(seg_counts_dev, w.seg_start, g.F * kBins);
  V2CE_LAUNCH_CHECK("ldati::scan_i64_kernel");
  return V2CE_OK;
}

// Sorts the `total` elements in sw.elem_a stably by their key field inside each of the `ns` segments
// [seg_start[i], seg_start[i+1]) and writes their 13-byte records to `out`.  P supplies the field widths and the
// timestamp origin of every segment (see pack_linear_kernel).
template <typename Elem>
static int sort_and_pack(const SortWs& sw, const int64_t* seg_start, int ns, int64_t total, const DevParams& P,
                         const int64_t* frame_off, uint8_t* out, cudaStream_t s) {
  // one-sweep LSD passes over the key field, <= 6 bits each
  const int passes = osw_passes(P.key_bits);
  const int rb = (P.key_bits + passes - 1) / passes;
  build_tiles_kernel<<<1, 1024, 0, s>>>(seg_start, ns, kOswTile, sw.tile_first);
  V2CE_LAUNCH_CHECK("ldati::build_tiles_kernel");
  fill_tile_seg_kernel<<<(sw.nt_max + 255) / 256, 256, 0, s>>>(sw.tile_first, ns, sw.tile_seg);
  V2CE_LAUNCH_CHECK("ldati::fill_tile_seg_kernel");
  V2CE_CUDA_CHECK(cudaMemsetAsync(sw.osw_zero, 0, sw.osw_zero_bytes, s));
  Elem* src = static_cast<Elem*>(sw.elem_a);
  Elem* dst = static_cast<Elem*>(sw.elem_b);
  osw_hist_kernel<Elem><<<sw.nt_max, kThreads, 0, s>>>(src, seg_start, sw.tile_first, sw.tile_seg, ns, P.pix_bits + 1, rb,
                                                       passes, sw.seg_hist);
  V2CE_LAUNCH_CHECK("ldati::osw_hist_kernel");
  const size_t smem = (size_t)kOswCounterWords * 4 > (size_t)kOswStageSlots * sizeof(Elem)
                          ? (size_t)kOswCounterWords * 4 : (size_t)kOswStageSlots * sizeof(Elem);
  for (int pass = 0; pass < passes; ++pass) {
    osw_scatter_kernel<Elem><<<sw.nt_max, kThreads, smem, s>>>(
        src, dst, seg_start, sw.tile_first, sw.tile_seg, ns, P.pix_bits + 1 + pass * rb, rb,
        sw.seg_hist + (size_t)pass * ns * kOswRadix, sw.tstate + (size_t)pass * sw.nt_max * kOswRadix, sw.tickets + pass);
    V2CE_LAUNCH_CHECK("ldati::osw_scatter_kernel");
    Elem* t = src; src = dst; dst = t;
  }
  const long long nchunks = (total + kPackRecsPerWarp - 1) / kPackRecsPerWarp;
  pack_chunk_seg_kernel<<<(int)((nchunks + 255) / 256), 256, 0, s>>>(seg_start, ns, total, sw.chunk_seg);
  V2CE_LAUNCH_CHECK("ldati::pack_chunk_seg_kernel");
  pack_linear_kernel<Elem><<<(int)((nchunks + kThreads / 32 - 1) / (kThreads / 32)), kThreads, 0, s>>>(
      src, seg_start, sw.chunk_seg, ns, total, P, frame_off, out);
  V2CE_LAUNCH_CHECK("ldati::pack_linear_kernel");
  return V2CE_OK;
}

template <typename Elem>
static int emit_impl(const float* vox, const v2ce_ldati_params* p, const Geometry& g, const CountWs& cw, void* emit_ws,
                     size_t emit_ws_bytes, const float* draws, int draws_m, const int64_t* frame_off, int64_t total,
                     uint8_t* out, int32_t* status, cudaStream_t s) {
  SortWs sw = carve_sort_ws(emit_ws, g, total, sizeof(Elem));
  if (sw.bytes > emit_ws_bytes)
    return set_error(V2CE_ERR_WORKSPACE, "emit workspace too small: need %zu, got %zu", sw.bytes, emit_ws_bytes);
  DevParams P = make_dev_params(p, g);
  P.draws_m = draws_m;
  Elem* ea = static_cast<Elem*>(sw.elem_a);
  V2CE_CUDA_CHECK(cudaMemsetAsync(status, 0, 4 * sizeof(int32_t), s));
  dim3 grid(g.NB, 2, g.F);
#define V2CE_LAUNCH_EMIT(V_, BIDIR_, POOL_)                                                                      \
  emit_kernel<V_, Elem, BIDIR_, POOL_><<<grid, kThreads, 0, s>>>(vox, P, cw.block_base, cw.group_base, cw.seg_start, \
                                                                  cw.warp_partial, cw.counts_all, draws, ea, status)
  const bool bidir = p->bidirectional != 0, pool = g.pooling != 0;
  if (g.V == 4) {
    if (bidir) { if (pool) V2CE_LAUNCH_EMIT(4, true, true); else V2CE_LAUNCH_EMIT(4, true, false); }
    else { if (pool) V2CE_LAUNCH_EMIT(4, false, true); else V2CE_LAUNCH_EMIT(4, false, false); }
  } else {
    if (bidir) { if (pool) V2CE_LAUNCH_EMIT(1, true, true); else V2CE_LAUNCH_EMIT(1, true, false); }
    else { if (pool) V2CE_LAUNCH_EMIT(1, false, true); else V2CE_LAUNCH_EMIT(1, false, false); }
  }
#undef V2CE_LAUNCH_EMIT
  V2CE_LAUNCH_CHECK("ldati::emit_kernel");
  if (total == 0) return V2CE_OK;
  return sort_and_pack<Elem>(sw, cw.seg_start, g.F * kBins, total, P, frame_off, out, s);
}

extern "C" int v2ce_ldati_emit(const float* voxels_dev, const v2ce_ldati_params* p, const void* count_ws_dev,
                               void* emit_ws_dev, size_t emit_ws_bytes, const float* draws_dev, int32_t draws_m,
                               const int64_t* frame_offset_us_dev, int64_t total_events, uint8_t* events_out_dev,
                               int32_t* status_dev, void* stream) {
  if (int e = validate(p)) return e;
  V2CE_REQUIRE(voxels_dev && count_ws_dev && emit_ws_dev && status_dev, "NULL device pointer");
  V2CE_REQUIRE(total_events >= 0 && total_events < (1LL << 31) - (1LL << 20), "total_events out of range");
  V2CE_REQUIRE(total_events == 0 || events_out_dev != nullptr, "events_out_dev is NULL");
  V2CE_REQUIRE(draws_dev == nullptr || draws_m >= 0, "bad draws_m");
  Geometry g = make_geometry(p);
  CountWs cw = carve_count_ws(const_cast<void*>(count_ws_dev), g);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (g.wide)
    return emit_impl<unsigned long long>(voxels_dev, p, g, cw, emit_ws_dev, emit_ws_bytes, draws_dev, draws_m,
                                         frame_offset_us_dev, total_events, events_out_dev, status_dev, s);
  return emit_impl<unsigned int>(voxels_dev, p, g, cw, emit_ws_dev, emit_ws_bytes, draws_dev, draws_m,
                                 frame_offset_us_dev, total_events, events_out_dev, status_dev, s);
}

extern "C" int v2ce_ldati_relocate(const float* voxels_dev, int32_t n_frames, int32_t height, int32_t width,
                                   int32_t bidirectional, int32_t* counts_dev, float* tend_dev, void* stream) {
  V2CE_REQUIRE(voxels_dev && counts_dev && tend_dev, "NULL device pointer");
  V2CE_REQUIRE(n_frames > 0 && height > 0 && width > 0 && n_frames * 2 <= 65535, "bad geometry");
  const int HW = height * width;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (HW % 4 == 0) {
    dim3 grid((HW / 4 + 255) / 256, n_frames * 2);
    relocate_debug_kernel<4><<<grid, 256, 0, s>>>(voxels_dev, HW, 1e-6f, bidirectional, counts_dev, tend_dev);
  } else {
    dim3 grid((HW + 255) / 256, n_frames * 2);
    relocate_debug_kernel<1><<<grid, 256, 0, s>>>(voxels_dev, HW, 1e-6f, bidirectional, counts_dev, tend_dev);
  }
  V2CE_LAUNCH_CHECK("ldati::relocate_debug_kernel");
  return V2CE_OK;
}

// ---------------------------------------------------------------------------------------
// Baseline samplers: C ABI
// ---------------------------------------------------------------------------------------
extern "C" size_t v2ce_baseline_params_size(void) { return sizeof(v2ce_baseline_params); }

extern "C" int v2ce_baseline_count_workspace_bytes(const v2ce_baseline_params* p, size_t* bytes) {
  if (int e = validate_base(p)) return e;
  V2CE_REQUIRE(bytes != nullptr, "bytes is NULL");
  *bytes = carve_base_ws(nullptr, p->n_frames, base_geom(p).NB).bytes;
  return V2CE_OK;
}

static Geometry base_sort_geometry(const v2ce_baseline_params* p, const BaseGeom& bg) {
  Geometry g;
  g.H = p->height; g.W = p->width; g.HW = bg.HW; g.F = p->n_frames; g.V = bg.V; g.NB = bg.NB;
  g.pix_bits = bg.pix_bits; g.key_bits = bg.key_bits; g.wide = 1; g.pooling = 0;
  return g;
}

// the sort workspace is carved for F * 9 segments (LDATI's layout); the baseline sort uses F of them
extern "C" int v2ce_baseline_emit_workspace_bytes(const v2ce_baseline_params* p, int64_t total_events, size_t* bytes) {
  if (int e = validate_base(p)) return e;
  V2CE_REQUIRE(bytes != nullptr && total_events >= 0, "bad arguments");
  V2CE_REQUIRE(total_events < (1LL << 31) - (1LL << 20), "more than 2^31 events in one call; split the frames");
  *bytes = carve_sort_ws(nullptr, base_sort_geometry(p, base_geom(p)), total_events, 8).bytes;
  return V2CE_OK;
}

extern "C" int v2ce_baseline_count(const float* voxels_dev, const v2ce_baseline_params* p, void* count_ws_dev,
                                   size_t count_ws_bytes, int64_t* frame_counts_dev, void* stream) {
  if (int e = validate_base(p)) return e;
  V2CE_REQUIRE(voxels_dev && count_ws_dev && frame_counts_dev, "NULL device pointer");
  const BaseGeom g = base_geom(p);
  BaseWs w = carve_base_ws(count_ws_dev, p->n_frames, g.NB);
  if (w.bytes > count_ws_bytes)
    return set_error(V2CE_ERR_WORKSPACE, "count workspace too small: need %zu, got %zu", w.bytes, count_ws_bytes);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const BaseDev P = base_dev(p, g);
  dim3 grid(g.NB, 2, p->n_frames);
  if (g.V == 4) base_count_kernel<4><<<grid, kThreads, 0, s>>>(voxels_dev, P, w.partial);
  else base_count_kernel<1><<<grid, kThreads, 0, s>>>(voxels_dev, P, w.partial);
  V2CE_LAUNCH_CHECK("ldati::base_count_kernel");
  base_scan_kernel<<<p->n_frames, 64, 0, s>>>(w.partial, w.block_base, w.group_base, frame_counts_dev, g.NB);
  V2CE_LAUNCH_CHECK("ldati::base_scan_kernel");
  scan_i64_kernel<<<1, 1024, 0, s>>>(frame_counts_dev, w.seg_start, p->n_frames);
  V2CE_LAUNCH_CHECK("ldati::scan_i64_kernel");
  return V2CE_OK;
}

extern "C" int v2ce_baseline_emit(const float* voxels_dev, const v2ce_baseline_params* p, const void* count_ws_dev,
                                  void* emit_ws_dev, size_t emit_ws_bytes, const int64_t* frame_offset_us_dev,
                                  int64_t total_events, uint8_t* events_out_dev, int32_t* status_dev, void* stream) {
  if (int e = validate_base(p)) return e;
  V2CE_REQUIRE(voxels_dev && count_ws_dev && emit_ws_dev && status_dev, "NULL device pointer");
  V2CE_REQUIRE(total_events >= 0 && total_events < (1LL << 31) - (1LL << 20), "total_events out of range");
  V2CE_REQUIRE(total_events == 0 || events_out_dev != nullptr, "events_out_dev is NULL");
  typedef unsigned long long Elem;
  const BaseGeom bg = base_geom(p);
  const Geometry g = base_sort_geometry(p, bg);
  BaseWs cw = carve_base_ws(const_cast<void*>(count_ws_dev), p->n_frames, bg.NB);
  SortWs sw = carve_sort_ws(emit_ws_dev, g, total_events, sizeof(Elem));
  if (sw.bytes > emit_ws_bytes)
    return set_error(V2CE_ERR_WORKSPACE, "emit workspace too small: need %zu, got %zu", sw.bytes, emit_ws_bytes);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const BaseDev P = base_dev(p, bg);
  V2CE_CUDA_CHECK(cudaMemsetAsync(status_dev, 0, 4 * sizeof(int32_t), s));
  if (total_events == 0) return V2CE_OK;
  Elem* elems = static_cast<Elem*>(sw.elem_a);
  dim3 grid(bg.NB, 2, p->n_frames);
  if (bg.V == 4) base_emit_kernel<4><<<grid, kThreads, 0, s>>>(voxels_dev, P, cw.block_base, cw.group_base, cw.seg_start, elems, status_dev);
  else base_emit_kernel<1><<<grid, kThreads, 0, s>>>(voxels_dev, P, cw.block_base, cw.group_base, cw.seg_start, elems, status_dev);
  V2CE_LAUNCH_CHECK("ldati::base_emit_kernel");
  // records: the LDATI record writer with one segment per frame whose key origin is the frame's
  DevParams D;
  memset(&D, 0, sizeof(D));
  D.H = p->height; D.W = p->width; D.HW = bg.HW; D.F = p->n_frames; D.NB = bg.NB;
  D.pix_bits = bg.pix_bits; D.key_bits = bg.key_bits;
  D.add_frame_offset = p->add_frame_offset;
  D.nan_ts = LLONG_MIN;
  D.segs_per_frame = 1;
  D.bin_base[0] = p->key_base_us;
  return sort_and_pack<Elem>(sw, cw.seg_start, p->n_frames, total_events, D, frame_offset_us_dev, events_out_dev, s);
}
