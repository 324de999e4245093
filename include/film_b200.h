/*
 * film_b200.h -- C ABI of the B200-native FILM inference engine (libfilm_b200.so).
 *
 * Drop-in boundary: every entry point replaces one piece of the reference's Python
 * inference wrapper, `eval/interpolator.py` (google-research/frame-interpolation):
 *
 *   film_create            <- Interpolator.__init__  (eval/interpolator.py:135-150,
 *                             tf.saved_model.load at :148)
 *   film_interpolate       <- Interpolator.interpolate (eval/interpolator.py:152-176):
 *                             _pad_to_align (:30-63) -> self._model(inputs) (:170-172,
 *                             i.e. models/film_net/interpolator.py:89-207) -> crop (:175)
 *   film_interpolate_tiled <- Interpolator.__call__ tiled branch
 *                             (eval/interpolator.py:192-206; image_to_patches :66-99,
 *                             patches_to_image :102-126)
 *   film_interpolate_device<- same as film_interpolate with device-resident frames; no
 *                             reference counterpart (the reference pays H2D + D2H + sync
 *                             per call at :171,:176); used by the recursive scheduler
 *                             (eval/util.py:62-91) and the multi-GPU shards.
 *
 * Plain C: pointers and sizes only, no torch / CUDA types in the signatures (a CUDA
 * stream is passed as void*). All frames are float32, NHWC, C-contiguous, 3 channels,
 * nominally in [0,1]; `dt` (B floats) is accepted and ignored exactly like the
 * reference ignores `time` (models/film_net/interpolator.py:102,163). Outputs are
 * NOT clipped (clipping happens in eval/util.py:51 on the reference side).
 *
 * Status codes: 0 ok; 1 bad argument (shape / alignment / divisibility);
 * 2 CUDA error; 3 weight-file mismatch; 4 not supported. film_last_error() returns
 * a human-readable message for the last non-zero status on that handle (or on
 * creation, when handle is NULL).
 *
 * There is no CPU fallback: every entry point fails with status 2 if no sm_100
 * device is present.
 *
 * Threading: a handle owns one CUDA stream, its per-shape plans (activation arenas, CUDA
 * graphs) and its staging buffers, so calls on ONE handle must be serialised by the caller;
 * different handles (one per GPU, or several per GPU when memory allows: ~20 GB per cached
 * 1080p shape) are independent and may be driven from different threads or processes.
 */
#ifndef FILM_B200_H_
#define FILM_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define FILM_API __attribute__((visibility("default")))
#else
#define FILM_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct film_handle film_handle;

enum {
  FILM_OK = 0,
  FILM_ERR_ARG = 1,
  FILM_ERR_CUDA = 2,
  FILM_ERR_WEIGHTS = 3,
  FILM_ERR_UNSUPPORTED = 4
};

/* Per-call engine statistics (all times are device times from CUDA events). */
typedef struct film_profile_t {
  double last_call_ms;        /* event time of the last network call (excl. H2D/D2H)      */
  double last_h2d_ms;         /* host->device copy time of the last host-pointer call     */
  double last_d2h_ms;         /* device->host copy time of the last host-pointer call     */
  double conv_flops;          /* reference-graph conv FLOPs of the last call (2*MAC)      */
  double mma_flops;           /* tensor-core FLOPs actually issued (1 or 3 passes per stage, padded K) */
  double warp_bytes;          /* algorithmic bytes of the warp-gather kernels (rd+wr)      */
  int64_t kernel_launches;    /* kernels launched (or graph nodes replayed) by the last call */
  int64_t arena_bytes;        /* device memory held by the plan used by the last call     */
  int32_t padded_h, padded_w; /* network resolution of the last call                       */
  int32_t used_graph;         /* 1 if the last call replayed a CUDA graph                  */
  int32_t reserved;
} film_profile_t;

/* Loads a FILMW1 weight file (see frame_interpolation_b200/weights.py), repacks the
 * HWIO kernels into the engine's split-bf16 K-major layout on `device_ordinal`,
 * creates the stream.  Replaces tf.saved_model.load (eval/interpolator.py:148). */
FILM_API int film_create(film_handle** out, const char* weights_path, int device_ordinal);

FILM_API void film_destroy(film_handle* h);

/* Host pointers. x0/x1/out: B*H*W*3 floats. align <= 0 disables padding
 * (eval/interpolator.py:149: `align or None`). A padded size that is not a multiple of 64 needs
 * option "any_size" (status 4 otherwise); at least 64 rows and columns (status 1 otherwise).
 * Blocks until `out` is written. */
FILM_API int film_interpolate(film_handle* h, const float* x0, const float* x1, const float* dt,
                     int B, int H, int W, int align, float* out);

/* Host pointers, B == 1. Splits the frame into block_h x block_w non-overlapping tiles
 * (row-major tile order), pads every tile independently to `align`, runs the network
 * per tile, stitches. H % block_h == 0 and W % block_w == 0 or status 1. */
FILM_API int film_interpolate_tiled(film_handle* h, const float* x0, const float* x1, const float* dt,
                           int H, int W, int align, int block_h, int block_w, float* out);

/* Device pointers (same layout), row pitches in floats (pitch >= W*3) so a tile of a
 * larger frame can be passed as a strided view. Asynchronous on `cuda_stream`
 * (a cudaStream_t; NULL = the handle's own stream, in which case the call returns after
 * enqueueing; use film_synchronize). */
FILM_API int film_interpolate_device(film_handle* h, const float* d_x0, const float* d_x1,
                            int B, int H, int W, int64_t in_pitch, int align,
                            float* d_out, int64_t out_pitch, void* cuda_stream);

/* Recursive mid-point interpolation between two (H, W, 3) host frames, the whole binary tree of
 * eval/util.py:62-91 (`_recursive_generator`) evaluated with every intermediate frame resident in
 * HBM: 2 uploads, 2^times - 1 network calls, 1 download.  `out` receives 2^times + 1 frames in
 * display order INCLUDING both end points (what interpolate_recursively_from_memory yields for one
 * pair, eval/util.py:125-153).  Results are bit-identical to calling film_interpolate recursively. */
FILM_API int film_interpolate_recursive(film_handle* h, const float* frame0, const float* frame1, int H, int W,
                                        int align, int times_to_interpolate, float* out);

/* 8-bit front / back end (SURVEY 8f row 3): the frames cross PCIe as uint8 (4x fewer bytes) and the reference's
 * conversions run on the device, bit-identical to the host versions:
 *   in : float32 = uint8 / 255                         (eval/util.py:38-41, read_image)
 *   out: uint8   = trunc(clip(x * 255, 0, 255) + 0.5)  (eval/util.py:51-52, write_image)
 * film_interpolate_u8 == to_uint8(film_interpolate(x0 / 255, x1 / 255)).  film_interpolate_recursive_u8 keeps the
 * recursion on the unquantised float32 mid-frames (like eval/util.py:85-91) and quantises only what it returns. */
FILM_API int film_interpolate_u8(film_handle* h, const uint8_t* x0, const uint8_t* x1, int B, int H, int W, int align,
                                 uint8_t* out);
FILM_API int film_interpolate_recursive_u8(film_handle* h, const uint8_t* frame0, const uint8_t* frame1, int H, int W,
                                           int align, int times_to_interpolate, uint8_t* out);

/* Page-locked host memory for frames (cudaHostAlloc): uploads / downloads of pinned buffers run at
 * PCIe speed instead of through the driver's pageable staging path. The Python wrapper returns its
 * results in pooled buffers allocated here. NULL on failure. */
FILM_API void* film_host_alloc(size_t bytes);
FILM_API void film_host_free(void* p);

FILM_API int film_synchronize(film_handle* h);

/* Fills *out with statistics of the last call on this handle. */
FILM_API int film_profile(film_handle* h, film_profile_t* out);

/* Engine options, set before the first call of a given shape.
 *   "conv_impl"   : 0 = tcgen05 implicit-GEMM kernels (default, the product path),
 *                   1 = fp32 CUDA-core validation kernels (debug only; used by the
 *                       tests to cross-check the tensor-core path on the device)
 *   "use_graph"   : 1 = capture each shape's schedule in a CUDA graph (default), 0 = eager
 *   "keep_debug"  : 1 = keep every intermediate tensor alive (no arena reuse) so that film_debug_read can
 *                   return it after the call; 0 (default) = activation buffers are recycled inside a plan
 *   "time_ops"    : 1 = run eagerly with one CUDA-event pair per kernel (see film_op_table)
 *   "conv3x3_v2"  : 1 = persistent tap-reuse kernel for 3x3 convs (default), 0 = generic kernel
 *   "conv3x3_2cta": 1 = CTA-pair (tcgen05 cta_group::2, M = 256) kernel for the streamed-weight 3x3
 *                   convs of the large pyramid levels (default), 0 = off, 2 = every eligible layer
 *   "conv3x3_halo": wide halo boxes -- one (64 ch, 10 px, 18 rows) TMA box per chunk serves all nine taps
 *                   (UMMA descriptors at pixel offsets): 3 = both persistent kernels, 64- and 32-channel chunks
 *                   (default: validated on hardware in round 2, -0.6 % / -2.0 % step time in two same-box A/Bs),
 *                   2 = 64-channel chunks only, 1 = CTA-pair kernel only, 0 = three dx-shifted 8-px boxes
 *   "fe_conv0_tc" : cfeat_conv_0 (3 -> 64, K = 27): 0 = register-tiled fp32 FMA kernel reading the fp32 image directly
 *                   (default: exact fp32 arithmetic, no widened image tensor), 1 = tensor-core kernel over a 32-channel-
 *                   padded split image (0.78 ms against 0.87 ms over the seven levels in per-op timing)
 *   "conv3x3_dual": 1 = the CTA-pair kernel serves TWO spatial work items per streamed weight tap (both items' halo boxes
 *                   resident, two accumulator sets in TMEM): halves the weight bytes pulled from L2 per item on the
 *                   layers that are L2->SM ingest bound (default); 0 = one item per weight pass
 *   "plane_skip"  : 1 = lo planes that no consumer reads (destinations of single-pass convs) are neither gathered nor
 *                   written (default), 0 = always both planes
 *   "mma_straight": 1 = with resident weights one elected lane issues a whole activation stage as straight-line code
 *                   (default), 0 = per-tap issue loop
 *   "arena_reuse" : 1 = activation buffers are recycled inside a plan by liveness (default), 0 = one buffer per tensor
 *   "fuse_flow_head": 1 = on flow level 0 (32-filter predictor) conv_3, conv_4 and the residual add run in the epilogue of
 *                   conv_2 (default), 2 = also on level 1 (64 filters: measured epilogue-bound, slower), 0 = separate launch
 *   "fuse_rgb_head": 1 = the linear 1x1 RGB head and the crop run in the epilogue of the decoder's last 3x3 conv (default;
 *                   the 64-channel activation is never stored), 0 = separate kernel
 *   "use_lanes"   : 1 = enqueue independent branches on separate streams (default 0)
 *   "clear_plans" : (any value) drop every cached (H, W, align) plan -- CUDA graph and activation arena --
 *                   after draining the handle's stream.  Plans are cached per shape and never evicted
 *                   otherwise, except that a shape whose arena cannot be allocated triggers one
 *                   drop-and-retry before FILM_ERR_CUDA is returned. */
/*   "any_size"    : 1 = padded frame sizes that are not multiples of 64 are computed like the reference graph does
 *                   (VALID pooling floors; flows and the decoder resize to each level's size), from 64 rows / columns
 *                   up; 0 (default) = they are refused with status 4.  Checked on every call, before the plan cache:
 *                   turning it off refuses such a size again even when its plan is cached.  It never changes how a
 *                   64-aligned size is computed.
 *   "onepass_mask": precision plan -- bit s selects the single-pass product (A_hi x W_hi, fp16 operands, fp32
 *                   accumulate) for stage s (film_stage_count / film_stage_name); every other conv runs the
 *                   three-pass split product.  The default is the measured plan of DESIGN.md section 3;
 *                   0 = every conv three-pass (fp32-grade).  "onepass_default" (any value) restores it. */
FILM_API int film_set_option(film_handle* h, const char* name, int value);
/* Reads back an integer option ("onepass_mask", "onepass_default", "conv3x3_halo", "conv3x3_2cta", "keep_debug",
 * "any_size"). */
FILM_API int film_get_option(film_handle* h, const char* name, int* value);

/* Stages of the precision plan: film_stage_count() names ("fe_i0_k01", "flow_L3", "fus2_c1", ...), index =
 * bit position in "onepass_mask".  film_stage_name copies the NUL-terminated name into buf. */
FILM_API int film_stage_count(void);
FILM_API int film_stage_name(int stage, char* buf, int buf_size);

/* Debug/parity hook: copies an intermediate tensor of the LAST call to host as float32
 * NHWC. `name` is e.g. "feat0/3" (feature pyramid of image 0, level 3), "flow_fwd/0",
 * "flow_bwd/2", "image". Returns the element count through *count when dst == NULL. */
FILM_API int film_debug_read(film_handle* h, const char* name, float* dst, int64_t* count);

/* Per-op table of the plan used by the last call, as CSV text
 * "idx,category,name,ms,ref_flops,alg_bytes" (category 0 = tcgen05 conv, 1 = warp gather,
 * 2 = other bandwidth kernels). `ms` is filled by calls made with option "time_ops" = 1
 * (eager run, one CUDA event pair per kernel on the launching stream), else -1.
 * *needed receives the buffer size required. */
FILM_API int film_op_table(film_handle* h, char* buf, int64_t buf_size, int64_t* needed);

FILM_API const char* film_last_error(film_handle* h);

/* Version / build info string: "film_b200 <ver> sm_100a split=fp16x2 mma=...". */
FILM_API const char* film_version(void);

#ifdef __cplusplus
}
#endif
#endif /* FILM_B200_H_ */
