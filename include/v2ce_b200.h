/*
 * v2ce_b200.h -- C ABI of libv2ce_b200.so: the B200 (sm_100a) implementation of the
 * V2CE video->continuous-events hot path.
 *
 * The reference (ucsd-hdsi-dvs/V2CE-Toolbox) has no FFI layer: its hot path is three
 * Python callables imported by v2ce.py:15-17.  Each entry point below replaces the
 * device work of one of them; the Python shims in v2ce_toolbox_b200/ (same names and
 * signatures as the reference modules) are the only callers.  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C types only; every pointer named *_dev is a CUDA device pointer owned by
 *     the caller (in practice: torch's caching allocator), every `stream` is a
 *     cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *   - all work is enqueued on `stream`; no call synchronises the device unless it
 *     says so; the library never frees caller memory;
 *   - return value 0 = success, negative = error; v2ce_last_error() gives the message
 *     of the last failing call on this thread;
 *   - there is NO CPU fallback: without a usable sm_100 device every compute call fails.
 */
#ifndef V2CE_B200_H
#define V2CE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define V2CE_OK 0
#define V2CE_ERR_INVALID (-1)
#define V2CE_ERR_CUDA (-2)
#define V2CE_ERR_WORKSPACE (-3)
#define V2CE_ERR_STATE (-4)
#define V2CE_ERR_RANGE (-5)

const char* v2ce_last_error(void);
int v2ce_version(void);
/* Fills sm count / compute capability of `device`; fails if it is not sm_100. */
int v2ce_device_check(int device, int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * Stage 2 -- LDATI.  Replaces scripts/LDATI.py:126-214 (sample_voxel_statistical) with its
 * helpers y_relocate (:80-106), calculate_statistical_linear_params_for_stage2 (:13-51),
 * pick_elements (:217-245) and pick_and_sort (:248-310).  The configuration v2ce.py:356 uses
 * (bidirectional=False, additional_events_strategy='slope', pooling_type='none') is the tuned path;
 * bidirectional=True and the 'random' / 'none' strategies are implemented as options of the same
 * kernels, and so is pooling_type 'avg' / 'weighted' (the slope is fitted on pooled counts; the Python
 * shim accepts every pooling_type the reference does).
 *
 * The scalar constants are computed by the host with the reference's own Python
 * expressions (SURVEY.md Appendix A) so the kernel reproduces torch's rounding.
 * ------------------------------------------------------------------------------------------ */
typedef struct v2ce_ldati_params {
  int32_t height, width;     /* H, W of one voxel plane                                      */
  int32_t n_frames;          /* F frame pairs in this call; voxels are (F,2,10,H,W) float32  */
  int32_t true_div;          /* 0: torch-CUDA scalar semantics (x * (1/s)); 1: torch-CPU (x / s) */
  int64_t frame_base;        /* global index of frame 0 (Philox counter, SURVEY.md F7)       */
  uint64_t seed;             /* Philox key                                                   */
  double fps64, nbins64;     /* divisors of the single-event path when true_div              */
  double r_fps64, r_nbins64; /* 1.0/fps, 1.0/9 in double (LDATI.py:156 on CUDA)              */
  float fps32, nbins32;      /* divisors of the k==0 path when true_div                      */
  float r_fps32, r_nbins32;  /* float32(1.0/fps), float32(1.0/9)                             */
  float vs32;                /* float32(voxel_step)                                          */
  float inv_vs32;            /* float32(1/voxel_step)                                        */
  float vs2_32;              /* float32(voxel_step**2)        (divisor when true_div)        */
  float r_vs2_32;            /* float32(1.0/voxel_step**2)                                   */
  float six32, r6_32;        /* 6.0f and float32(1.0/6)                                      */
  float eps6, eps8;          /* float32(1e-6), float32(1e-8)                                 */
  float binstart_t0_32[16];  /* torch.arange(0,1/fps,voxel_step)[c] + t0, float32, 9 used    */
  int64_t bin_base_us[16];   /* sort-key origin per bin: trunc(binstart_t0_32[c]*1e6)        */
  int32_t key_span;          /* max (ts - bin_base_us) expected + slack; key bits derive from it */
  int32_t add_frame_offset;  /* 1: add frame_offset_us[f] to every timestamp (fused CLI path, v2ce.py:365) */
  int32_t multi_events;      /* additional_events_strategy for pixel-bins holding more than one event:
                              * 1 = 'slope' (inverse CDF of the linear density, LDATI.py:184-196; the CLI's setting),
                              * 2 = 'random' (the raw uniform draw is the offset in SECONDS, LDATI.py:173-174),
                              * 0 = 'none' (such pixel-bins emit nothing, LDATI.py:206-207,241-244)             */
  int32_t bidirectional;     /* 1: y_relocate(bidirectional=True), LDATI.py:107-122 (bin_base_us / key_span must
                              * then cover tendencies in (-1, y[9]] bins; see v2ce_toolbox_b200/ldati.py)        */
  int32_t pooling;           /* pooling_type: 0 = 'none', 1 = 'weighted' (3x3 binomial / 16), 2 = 'avg' (box of
                              * pooling_kernel_size^2, zero padded, count_include_pad) -- LDATI.py:176-183; only read when
                              * multi_events == 1.                                                                 */
  int32_t pooling_kernel_size; /* odd; 'avg' only                                                                  */
} v2ce_ldati_params;

/* Host-only guards for bindings that mirror the struct (ctypes, cgo, JNI): its size in this build, and the argument
 * checks every LDATI entry point applies (0 or a negative error code; message in v2ce_last_error()). */
size_t v2ce_ldati_params_size(void);
int v2ce_ldati_params_validate(const v2ce_ldati_params* p);

/* Workspace needed by v2ce_ldati_count (also holds the scan results v2ce_ldati_emit reads). */
int v2ce_ldati_count_workspace_bytes(const v2ce_ldati_params* p, size_t* bytes);
/* Additional workspace needed by v2ce_ldati_emit for `total_events` events. */
int v2ce_ldati_emit_workspace_bytes(const v2ce_ldati_params* p, int64_t total_events, size_t* bytes);

/* Pass 1 (LDATI.py:80-106 + the bookkeeping of :217-245): integer event counts per pixel-bin,
 * per-(frame,bin) segment totals and the prefix sums that give every event its slot in the
 * reference's pre-sort concatenation order.  seg_counts_dev: int64 [F][9]. */
int v2ce_ldati_count(const float* voxels_dev, const v2ce_ldati_params* p, void* count_ws_dev, size_t count_ws_bytes,
                     int64_t* seg_counts_dev, void* stream);

/* v2ce_ldati_count that also writes the per-polarity event-frame sums of v2ce_ef_accumulate(keep_polarity = 1)
 * (v2ce.py:255: float32 [F][2][H][W], the 10 bins added left to right) from the SAME read of the voxels: in the CLI
 * pipeline both stages consume the network output of a batch, 7.2 MB per frame pair each.  ef_sums_dev may be NULL. */
int v2ce_ldati_count_ef(const float* voxels_dev, const v2ce_ldati_params* p, void* count_ws_dev, size_t count_ws_bytes,
                        int64_t* seg_counts_dev, float* ef_sums_dev, void* stream);

/* Pass 2 (LDATI.py:156-212, :248-310): timestamps, stable per-segment sort by timestamp,
 * 13-byte packed records {int64 timestamp; int16 x; int16 y; int8 polarity}.
 * draws_dev: NULL -> counter-based Philox draws keyed by p->seed; else a dense float32
 * (F,2,9,H,W,draws_m) tensor of injected uniforms (the reference's torch.rand layout).
 * frame_offset_us_dev: int64 [F] or NULL.  total_events must equal the sum of seg_counts.
 * status_dev: int32[4] = {clamped keys, NaN timestamps, slot overruns, reserved}. */
int v2ce_ldati_emit(const float* voxels_dev, const v2ce_ldati_params* p, const void* count_ws_dev,
                    void* emit_ws_dev, size_t emit_ws_bytes, const float* draws_dev, int32_t draws_m,
                    const int64_t* frame_offset_us_dev, int64_t total_events, uint8_t* events_out_dev,
                    int32_t* status_dev, void* stream);

/* Debug/parity hook for LDATI.py:80-123 alone (y_relocate): int32 counts (F,2,9,H,W) and float32 tendencies. */
int v2ce_ldati_relocate(const float* voxels_dev, int32_t n_frames, int32_t height, int32_t width, int32_t bidirectional,
                        int32_t* counts_dev, float* tend_dev, void* stream);

/* ---- baseline samplers 'random' / 'even' (SURVEY.md 8f N4) -------------------------------------------------------
 * Replaces /root/reference/train/scripts/stage2/sample_methods/random_even_sample.py:118-170 (sample_voxel_baseline and
 * its pick_and_sort): every value y of the TEN voxel bins yields floor(y) events plus one more with probability frac(y);
 * a frame's events are sorted by timestamp.  Same two-phase protocol and record format as LDATI. */
typedef struct v2ce_baseline_params {
  int32_t height, width;     /* H, W of one voxel plane                                                  */
  int32_t n_frames;          /* F frame pairs in this call; voxels are (F,2,10,H,W) float32              */
  int32_t mode;              /* 1 = 'random' (uniform draw per event), 2 = 'even' (j / (floor(y)+1))      */
  int64_t frame_base;        /* global index of frame 0 (Philox counter)                                  */
  uint64_t seed;             /* Philox key; streams 0 / 1 / 2 = integer-part, fractional-part, Bernoulli  */
  float delta32;             /* float32(1 / (fps * 10)): the multiplier of `ts * delta`                   */
  float binstart_t0_32[10];  /* torch.arange(0, 1/fps, 1/fps/10) + t0 as float32, evaluated like the reference's device */
  int64_t key_base_us;       /* timestamps are sorted as ts - key_base_us + 8; <= the frame's first timestamp */
  int32_t key_span;          /* largest ts - key_base_us accepted (status counts events outside)          */
  int32_t add_frame_offset;  /* 1: add frame_offset_us_dev[f] to the records' timestamps                  */
} v2ce_baseline_params;

size_t v2ce_baseline_params_size(void);
int v2ce_baseline_count_workspace_bytes(const v2ce_baseline_params* p, size_t* bytes);
int v2ce_baseline_emit_workspace_bytes(const v2ce_baseline_params* p, int64_t total_events, size_t* bytes);
/* frame_counts_dev: int64 [F] events per frame */
int v2ce_baseline_count(const float* voxels_dev, const v2ce_baseline_params* p, void* count_ws_dev, size_t count_ws_bytes,
                        int64_t* frame_counts_dev, void* stream);
/* status_dev: int32[4] = {timestamps outside the key range (non-finite or negative voxels in 'even' mode), 0, 0, 0} */
int v2ce_baseline_emit(const float* voxels_dev, const v2ce_baseline_params* p, const void* count_ws_dev, void* emit_ws_dev,
                       size_t emit_ws_bytes, const int64_t* frame_offset_us_dev, int64_t total_events,
                       uint8_t* events_out_dev, int32_t* status_dev, void* stream);

/* ---- stage-2 evaluation metric (SURVEY.md 8f N4) ------------------------------------------------------------------
 * Replaces /root/reference/train/scripts/stage2/stage2_metrics.py:22-88 (ts_diff_metric): for every ground-truth event the
 * smallest |t_pred - t_gt| over the predicted events of the same polarity at the pixels within search_range (clamped to
 * the width x height sensor; 0 <= search_range < 64), clamped to 1e6 (also when the window is empty) and capped at
 * cap_us = 1e6/fps/10*3.  Both event sets are packed 13-byte records on the device (ground-truth polarity -1 counts as
 * 0, :38-41).  result_dev: int64[4] = {sum of the clamped integer distances that are not capped, number
 * of capped ground-truth events ("overflow"), ground-truth events outside the sensor, predicted events outside the
 * sensor}; the metric is (result[0] + result[1] * cap_us) / n_gt. */
int v2ce_ts_diff_workspace_bytes(int32_t width, int32_t height, int64_t n_pred, size_t* bytes);
int v2ce_ts_diff_metric(const uint8_t* gt_records_dev, int64_t n_gt, const uint8_t* pred_records_dev, int64_t n_pred,
                        int32_t width, int32_t height, int32_t search_range, double cap_us, void* ws_dev, size_t ws_bytes,
                        int64_t* result_dev, void* stream);



/* ------------------------------------------------------------------------------------------
 * Event frames.  Replaces v2ce.py:241-280 (write_event_frame_video) up to the cv2 encoder.
 * ------------------------------------------------------------------------------------------ */
/* v2ce.py:255 / :259-260 -- sums (N,2,H,W) [keep_polarity] or (N,1,H,W) float32. */
int v2ce_ef_accumulate(const float* voxels_dev, int32_t n_pairs, int32_t height, int32_t width,
                       int32_t keep_polarity, float* sums_dev, void* stream);
/* v2ce.py:262-264 -- exact order statistics of the positive sums by radix select.
 * result_dev: int64[4] = {n_positive, rank_lo, bits(value[rank_lo]), bits(value[rank_lo+1 clamped])};
 * the host applies numpy's float64 lerp and min(., ceil).  multiplicity = 3 in gray mode
 * (np.repeat of the channel, v2ce.py:260), 1 otherwise.  ws: v2ce_ef_select_workspace_bytes(). */
int v2ce_ef_select_workspace_bytes(size_t* bytes);
int v2ce_ef_select(const float* sums_dev, int64_t n_values, double percentile, int32_t multiplicity,
                   void* ws_dev, size_t ws_bytes, int64_t* result_dev, void* stream);
/* v2ce.py:267-277 -- clip / normalise in float64 -> uint8 BGR frames (N,H,W,3). */
int v2ce_ef_normalize(const float* sums_dev, int32_t n_pairs, int32_t height, int32_t width,
                      int32_t keep_polarity, double upper_bound, uint8_t* frames_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Image pre-processing for frames that are NOT at the model's resolution.  Replaces v2ce.py:45-64
 * (image_pre_processing): /255, cv2.resize(INTER_LINEAR) to the model's height, pair stacking,
 * Normalize(0.153, 0.165) -- bit-identical to the host path (oracle/resize_oracle.py).
 * frames_dev: uint8 gray (n_windows, frames_per_window, src_h, src_w); units_dev: float32
 * (n_windows, frames_per_window - 1, 2, dst_h, dst_w), the input layout of v2ce_model_forward.
 * (Frames already at the model's height go to v2ce_model_forward_frames instead.)
 * ------------------------------------------------------------------------------------------ */
int v2ce_image_units(const uint8_t* frames_dev, int32_t n_windows, int32_t frames_per_window, int32_t src_h,
                     int32_t src_w, int32_t dst_h, int32_t dst_w, float* units_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage 1 -- V2ce3d.  Replaces scripts/v2ce_3d.py:12-30 (V2ce3d), scripts/unet_2layer.py:203-379
 * (UNet3D), scripts/submodules.py:85-124,216-264 (ConvLayer3D, ResidualBlock3D) and
 * scripts/spectral_norm.py:9-64 (SpectralNorm) in eval mode.
 * ------------------------------------------------------------------------------------------ */
typedef struct v2ce_model v2ce_model;

int v2ce_model_create(v2ce_model** out, int device);
int v2ce_model_destroy(v2ce_model* m);
/* One call per state_dict entry, reference key names ("UNet.encoders.0.conv1.weight", ...,
 * "UNet.decoders.0.conv1.module.weight_bar").  data_host: float32, C-contiguous, host memory.
 * Unknown names (e.g. num_batches_tracked) return V2CE_ERR_INVALID. */
int v2ce_model_set_tensor(v2ce_model* m, const char* name, const float* data_host, const int64_t* shape,
                          int32_t ndim);
/* Folds BatchNorm (eval) into per-channel scale/shift, packs bf16 weight tiles. */
int v2ce_model_finalize(v2ce_model* m);
int v2ce_model_workspace_bytes(const v2ce_model* m, int32_t batch, int32_t depth, int32_t height,
                               int32_t width, size_t* bytes);
/* Byte offsets into the workspace of its bf16 activation buffers at this shape (per-layer tests), in this order:
 * head_in, head, enc0..3, res0..1, dec0..3, tmp_t, tmp_r, up, up2 (16 entries; cap must be >= 16, *n receives 16). */
int v2ce_model_workspace_layout(const v2ce_model* m, int32_t batch, int32_t depth, int32_t height, int32_t width,
                                int64_t* offsets, int32_t cap, int32_t* n);
/* x_dev (B,L,2,H,W) float32 -> y_dev (B,L,20,H,W) float32 (v2ce_3d.py:26-30).  Advances the
 * spectral-norm power iteration by one step, as the reference does on every forward. */
int v2ce_model_forward(v2ce_model* m, const float* x_dev, float* y_dev, int32_t batch, int32_t depth,
                       int32_t height, int32_t width, void* ws_dev, size_t ws_bytes, void* stream);
/* Same forward fed with raw frames: frames_dev (B, L+1, H, W) uint8 gray, window b = L+1 consecutive frames.  The
 * pre-processing of v2ce.py:45-64 at the model's own resolution (float32 /255, pair stacking, Normalize(0.153, 0.165);
 * the resize is the identity there) is evaluated inside the head conv, bit-identically to the host path. */
int v2ce_model_forward_frames(v2ce_model* m, const uint8_t* frames_dev, float* y_dev, int32_t batch, int32_t depth,
                              int32_t height, int32_t width, void* ws_dev, size_t ws_bytes, void* stream);
/* Spectral-norm state access (parity tests, multi-GPU replay): 12 sigmas of the last forward;
 * number of forwards so far; advance the iteration n calls without running the network. */
int v2ce_model_last_sigmas(const v2ce_model* m, float* sigma12_host);
int v2ce_model_call_count(const v2ce_model* m, int64_t* calls);
int v2ce_model_sn_advance(v2ce_model* m, int32_t n_calls, void* stream);
/* Number of kernels the last complete forward launched (bench.py's gpu_launches). */
int v2ce_model_last_launches(const v2ce_model* m, int32_t* launches);

/* Layer-level hook used by the parity tests: one fused conv launch.
 *  src0 (B,D,H0,W0,C0) bf16 [nearest-upsampled to (Hin,Win) when H0!=Hin], src1 (B,D,Hin,Win,C1) bf16 or NULL,
 *  weight_host (Cout, C0+C1, k,k,k) float32, scale/shift float32[Cout] (host), residual (M,Cout) bf16 or NULL,
 *  act: 0 none, 1 relu, 2 leaky_relu(0.01).  out (B,D,Hout,Wout,Cout) bf16. */
int v2ce_conv3d_bf16(const void* src0_dev, int32_t c0, int32_t h0, int32_t w0, const void* src1_dev, int32_t c1,
                     int32_t batch, int32_t depth, int32_t hin, int32_t win, int32_t ksize, int32_t stride_hw,
                     const float* weight_host, int32_t cout, const float* scale_host, const float* shift_host,
                     const void* residual_dev, int32_t act, void* out_dev, void* stream);

/* Same hook with the kernel made explicit: impl 0 = gather implicit GEMM (csrc/conv_igemm.cuh), 1 = halo-tile
 * kernel (csrc/conv_halo.cuh; 3x3x3, stride 1, h0==hin, channel pitches multiple of 64), 2 = its depth-merged
 * variant (csrc/conv_halo_kdm.cuh; additionally Cout <= 64, depth % 8 == 0), 3 = the same with the fused 1x1x1
 * shortcut: residual_dev is then an OUTPUT (B,D,H,W,Cout) bf16 receiving scale*conv1x1(x, weight[:,:,1,1,1])+shift.
 * desc_mode is a bring-up switch of the shifted shared-memory descriptor (0 or 1). */
int v2ce_conv3d_bf16_ex(const void* src0_dev, int32_t c0, int32_t h0, int32_t w0, const void* src1_dev, int32_t c1,
                        int32_t batch, int32_t depth, int32_t hin, int32_t win, int32_t ksize, int32_t stride_hw,
                        const float* weight_host, int32_t cout, const float* scale_host, const float* shift_host,
                        const void* residual_dev, int32_t act, void* out_dev, int32_t impl, int32_t desc_mode,
                        void* stream);
/* Bring-up microbenchmark: cycles per back-to-back tcgen05.mma (M=128, N=bn, K=16, both operands in shared
 * memory) with `naccs` accumulators in rotation on `ctas` CTAs. */
int v2ce_debug_mma_rate(int32_t bn, int32_t iters, int32_t naccs, int32_t ctas, double* cycles_per_mma);
/* Per-launch device times of the last forward, measured with CUDA events on the launch stream when the option
 * "layer_timing" is 1: ms_out[i] and the layer name (48 bytes each, NUL terminated) of launch i. */
int v2ce_model_layer_times(v2ce_model* m, int32_t cap, float* ms_out, char* names_out, int32_t* count);
/* Tuning / bring-up options of a model handle: "desc_mode", "layer_timing", and "stop_after" (per-layer tests; default
 * -1 = off): a layer index in state-dict order (head 0 .. pred 31); the forward returns right after the launch that
 * writes that layer's output, with every stream it used joined into `stream`.  A block's shortcut fused into its conv1
 * stops after that launch, pred after decoders.3.conv2.  The workspace then holds the layer's inputs and its output. */
int v2ce_model_set_option(v2ce_model* m, const char* key, int64_t value);

/* ------------------------------------------------------------------------------------------
 * Peer windows -- the shard merge of the multi-GPU clip driver (v2ce_toolbox_b200/dist.py; the reference is
 * single-process: this replaces the concatenation of v2ce.py:226 across ranks).  One process per GPU; the
 * destination rank allocates a window, ships its 64-byte handle to the other ranks (any host channel), and every
 * rank copies its shard straight into place with the copy engines over NVLink: no SM, no collective kernel
 * competing with the persistent conv CTAs.
 *   v2ce_peer_window_alloc : cudaMalloc on the current device + cudaIpcGetMemHandle
 *   v2ce_peer_window_open  : map another process's window (peer access enabled lazily); _close unmaps it
 *   v2ce_peer_copy_async   : cudaMemcpyAsync(dst, src, bytes) on `stream`; dst / src may be opened windows
 * ------------------------------------------------------------------------------------------ */
#define V2CE_PEER_HANDLE_BYTES 64
int v2ce_peer_window_alloc(size_t bytes, void** window_dev, uint8_t handle_out[V2CE_PEER_HANDLE_BYTES]);
int v2ce_peer_window_free(void* window_dev);
int v2ce_peer_window_open(const uint8_t handle[V2CE_PEER_HANDLE_BYTES], void** window_dev);
int v2ce_peer_window_close(void* window_dev);
int v2ce_peer_copy_async(void* dst_dev, const void* src_dev, size_t bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* V2CE_B200_H */
