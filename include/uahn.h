/*
 * uahn.h — C ABI of the B200-native UAHN forward (the CUAHN-VIO per-frame hot path).
 *
 * Drop-in boundary: these entry points are what a binding of the reference's
 * `pytorch::HomographyNet` (cuahn_ros/homography_network/src/HomographyNet.h:23-67) would call
 * instead of `torch::jit::Module::forward` (HomographyNet.cpp:42,183,211).  Plain pointers and sizes
 * only; no torch / Eigen / OpenCV types.  All functions return UAHN_OK (0) or a negative error code
 * and record a message retrievable with uahn_last_error() — the reference swallows errors
 * (HomographyNet.cpp:87-93,155-158); the C++ shim in include/HomographyNet.h restores its
 * print-and-continue behaviour on top of these codes.
 *
 * Units / conventions (SURVEY §8b): corner order UL, BL, BR, UR as (u, v) pixels of the 320x224
 * image; `mean` = displacement of the previous-image corners into the current image;
 * `cov` = 8x8 row-major, px², symmetric (block-diagonal 2x2 per corner).
 */
#ifndef UAHN_H_
#define UAHN_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define UAHN_API __attribute__((visibility("default")))
#else
#define UAHN_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define UAHN_IMG_H 224
#define UAHN_IMG_W 320
#define UAHN_IMG_PIXELS (UAHN_IMG_H * UAHN_IMG_W)
#define UAHN_MC_SAMPLES 16
#define UAHN_FC_IN 5120
#define UAHN_FC_HIDDEN 256
/* bytes of explicit MC-dropout keep-masks per pair: 2 heads x 16 samples x (5120 + 256) */
#define UAHN_MASK_BYTES_PER_PAIR (2 * UAHN_MC_SAMPLES * (UAHN_FC_IN + UAHN_FC_HIDDEN))

enum {
  UAHN_OK = 0,
  UAHN_ERR_INVALID = -1,   /* bad argument */
  UAHN_ERR_CUDA = -2,      /* CUDA runtime failure (message has the cudaError string) */
  UAHN_ERR_WEIGHTS = -3,   /* weight file missing / malformed / wrong schema */
  UAHN_ERR_STATE = -4,     /* e.g. uahn_infer before two images were loaded (HomographyNet.cpp:155-158) */
  UAHN_ERR_UNSUPPORTED = -5
};

/* Which traced graph of trace_model.py:36-46 the handle reproduces. */
enum {
  UAHN_VARIANT_AUTO = -1,   /* whatever graph the weights file was exported from (weights.export_torchscript records
                               it): the reference's iterative slot runs "whatever the file holds", HomographyNet.cpp:104-124 */
  UAHN_VARIANT_FULL = 0,    /* traced_full_model: blocks 1+2+3+4, no prior            */
  UAHN_VARIANT_PRIOR3 = 1,  /* traced_model_3_blocks_using_prior: prior + blocks 2,3,4 */
  UAHN_VARIANT_PRIOR2 = 2,  /* blocks_to_run = 2 (model_to_trace.py:72): prior + blocks 3,4 */
  UAHN_VARIANT_PRIOR1 = 3   /* blocks_to_run = 1: prior + block 4 only                 */
};

enum {
  UAHN_PRECISION_FP32 = 0,  /* validation mode: true fp32 FFMA convolutions           */
  UAHN_PRECISION_BF16 = 1   /* tcgen05 bf16 implicit-GEMM convolutions, fp32 accumulate */
};

#define UAHN_SHOW_ERROR_AUTO (-1) /* uahn_config.show_error: take the `_showError` flag recorded in the weights file */

typedef struct uahn_handle uahn_handle;

typedef struct uahn_config {
  const char* weights_path; /* flat file written by cuahn_vio_b200.weights.export_state_dict()    */
  int variant;              /* UAHN_VARIANT_*                                                     */
  int show_error;           /* 1 = also produce the photometric error map (`_showError` graphs)   */
  int precision;            /* UAHN_PRECISION_*                                                   */
  int device;               /* CUDA device ordinal                                                */
  int max_batch;            /* largest n accepted by uahn_infer_batch* (activations are preallocated) */
  void* stream;             /* cudaStream_t to run on; NULL = the handle creates its own          */
} uahn_config;

/* MC-dropout randomness (model_to_trace.py:222-235, 266-273).
 * keep_masks == NULL: masks are drawn in-kernel from Philox4x32-7 keyed by (seed, first_pair_index + i).
 * keep_masks != NULL: explicit replay; HOST (or device, for the *_device call) bytes, 1 = kept, 0 = dropped,
 *   laid out [pair][head(0=mean,1=uncertainty)][sample 0..15][5120 inputs, then 256 hidden], the 5120 axis
 *   in the reference's NCHW flatten order c*20 + h*5 + w.  Kept values are scaled by 1/0.95.
 * A NULL uahn_rng* means seed 0; uahn_infer then numbers its calls itself (a per-handle counter is the pair index), so
 * consecutive frames and IEKF iterations draw different masks, as the reference's forward does.  The batch entry
 * points use pair index first_pair_index + i; passing the same (seed, first_pair_index) twice REPLAYS the same masks —
 * advance first_pair_index by n per call for fresh ones. */
typedef struct uahn_rng {
  uint64_t seed;
  uint64_t first_pair_index;
  const uint8_t* keep_masks;
} uahn_rng;

UAHN_API int uahn_create(const uahn_config* cfg, uahn_handle** out);
UAHN_API void uahn_destroy(uahn_handle* h);
UAHN_API const char* uahn_last_error(const uahn_handle* h); /* h may be NULL: error of the last failed uahn_create */

/* Replaces HomographyNet::load_current_img (HomographyNet.cpp:127-151): gray is CV_8UC1 rows x cols with
 * `stride` bytes per row, borrowed only for the duration of the call.  prev <- curr, curr <- gray. */
UAHN_API int uahn_load_image(uahn_handle* h, const uint8_t* gray, int rows, int cols, size_t stride, double time_stamp);

/* Replaces HomographyNet::network_inference (HomographyNet.cpp:153-252) on the (prev, curr) pair.
 * prior_px: 8 doubles (required for PRIOR* variants, ignored for FULL).  err_map: 224*320 bytes
 * (error clamped to [0,255] and truncated like HomographyNet.cpp:201) or NULL. */
UAHN_API int uahn_infer(uahn_handle* h, const double* prior_px, const uahn_rng* rng, double* mean8, double* cov64,
               uint8_t* err_map);

/* n independent pairs, HOST buffers; copies in/out are part of the call.
 * prev, curr: n x 224 x 320 u8.  prior: n x 8 float (NULL for FULL).  mean: n x 8, cov: n x 64,
 * err: n x 224 x 320 float (|warp(curr) - prev| * 255, unclamped like model_to_trace.py:325-327) or NULL. */
UAHN_API int uahn_infer_batch(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const float* prior,
                     const uahn_rng* rng, float* mean, float* cov, float* err);

/* Same, but every pointer is DEVICE memory on cfg.device; asynchronous on the handle's stream. */
UAHN_API int uahn_infer_batch_device(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const float* prior,
                            const uahn_rng* rng, float* mean, float* cov, float* err);

/* Pipelined form of uahn_infer_batch for streams of batches: returns as soon as the work is enqueued.  The H2D copy of
 * submission i+1 (on an internal copy stream, double-buffered device staging) overlaps the forward of submission i;
 * results land in `mean` / `cov` (HOST, should be pinned) when uahn_wait() returns.  Philox masks only, no error map.
 * At most two submissions are in flight: a third call blocks the copy stream until the first has finished. */
UAHN_API int uahn_submit_batch(uahn_handle* h, int n, const uint8_t* prev, const uint8_t* curr, const float* prior,
                      const uahn_rng* rng, float* mean, float* cov);
/* The streaming pattern of HomographyNet::load_current_img (HomographyNet.cpp:143: prev <- curr), batched and
 * pipelined like uahn_submit_batch: `frames` holds n_frames consecutive frames of ONE sequence (n_frames x 224 x 320
 * u8, HOST), pair i = (frames[i], frames[i+1]); prior / mean / cov have n_frames - 1 rows.  Every frame crosses PCIe
 * once (71 680 B per pair instead of 143 360 B).  n_frames - 1 <= max_batch. */
UAHN_API int uahn_submit_sequence(uahn_handle* h, int n_frames, const uint8_t* frames, const float* prior,
                         const uahn_rng* rng, float* mean, float* cov);
UAHN_API int uahn_wait(uahn_handle* h);

UAHN_API int uahn_synchronize(uahn_handle* h);
UAHN_API void* uahn_stream(uahn_handle* h);
/* Kernel launches issued by this handle since creation (bench.py's gpu_launches). */
UAHN_API uint64_t uahn_launch_count(const uahn_handle* h);
UAHN_API double uahn_latest_inference_time(const uahn_handle* h); /* HomographyNet::get_latest_inference_time */
UAHN_API int uahn_image_count(const uahn_handle* h);               /* HomographyNet::img_counter */
UAHN_API int uahn_variant(const uahn_handle* h);    /* the resolved UAHN_VARIANT_* (after UAHN_VARIANT_AUTO) */
UAHN_API int uahn_show_error(const uahn_handle* h); /* the resolved show_error flag */

/* Per-stage device timing (bench.py's roofline): when enabled, every forward brackets each kernel group with
 * CUDA events on the handle's stream.  Categories: 0 = warp/concat/pool + error map + the remap of raw
 * sequence submissions (HBM-bound),
 * 1 = conv stacks (tensor-bound), 2 = MC-head 5120->256 GEMMs (tensor-bound), 3 = FC8+DLT / MC expand / final.
 * uahn_profile_read synchronises, adds the elapsed ms of all finished groups into ms[4] / launches[4]
 * (accumulating since the last uahn_profile_enable(h, 1)) and returns UAHN_OK. */
UAHN_API int uahn_profile_enable(uahn_handle* h, int on);
UAHN_API int uahn_profile_read(uahn_handle* h, double* ms4, uint64_t* launches4);

/* Host replica of the in-kernel Philox mask generator: fills UAHN_MASK_BYTES_PER_PAIR bytes for one pair. */
UAHN_API int uahn_philox_keep_masks(uint64_t seed, uint64_t pair_index, uint8_t* out);

/* ---- stage entry points (parity tests; HOST buffers, synchronous) -------------------------------------- */
/* model_to_trace.py:42-61 on the fixed source corners: offsets n x 8 -> H n x 9 (row-major 3x3). */
UAHN_API int uahn_stage_dlt(uahn_handle* h, int n, const float* offsets, float* H);
/* warp.py:60-79: img n x 224 x 320 u8, H n x 9 -> out n x 224 x 320 float; optional NW tap indices. */
UAHN_API int uahn_stage_warp(uahn_handle* h, int n, const uint8_t* img, const float* H, float* out, int16_t* ix_nw,
                    int16_t* iy_nw);
/* model_to_trace.py:18-38 (transfer_mean_var_single) + the output packing of :311-317: var n x 8 (sigma^2 per corner
 * coordinate), Hp n x 9 (part-1 homography), pts_w n x 8 (corners + mu) -> flow n x 8, cov n x 64. */
UAHN_API int uahn_stage_transfer(uahn_handle* h, int n, const float* var, const float* Hp, const float* pts_w, float* flow,
                        float* cov);
/* One Conv2d+LeakyReLU layer of the handle's precision path: `layer` e.g. "block_3_1"; in: n x Cin x Hin x Win
 * float (NCHW); the result is read back with uahn_debug_read("act:<layer>") as n x Cout x Ho x Wo. */
UAHN_API int uahn_stage_conv(uahn_handle* h, const char* layer, int n, const float* in_nchw);
/* Values captured during the LAST uahn_infer_batch* call.  what: "H<b>" (n x 9, cumulative after block b;
 * "H0" = prior), "d<b>" (n x 8), "feat<b>" (n x 5120 in NCHW flatten order), "x<b>" (block input,
 * n x 2 x h x w), "mcmean"/"mclogvar" (n x 16 x 8).  Returns number of floats written or <0. */
UAHN_API long uahn_debug_read(uahn_handle* h, const char* what, float* out, size_t capacity_floats);

#ifdef __cplusplus
}
#endif
#endif /* UAHN_H_ */
