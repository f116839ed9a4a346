/*
 * uahn_filter.h — filter bank: the EKF states of n sequences kept on the GPU next to one uahn_handle, propagated and
 * updated by sm_100a kernels around one batched forward per IEKF iteration.  Plain C ABI, Eigen-free.
 *
 * Replaces, over n sequences at once, the per-frame filter loop of VioManager (cuahn_ros/cuahn/src/core/VioManager.cpp:
 * 181-275): Propagator::propagate_with_imu for every sequence (uahn_imu_propagate), then the IEKF loop around the
 * network (uahn_ekf_iekf_frame).  Per slot the result is what uahn_imu_propagate / uahn_ekf_iekf_frame leave in that
 * slot's uahn_ekf_state (fp64 on both sides; see DESIGN §11 for how close).
 *
 * Asynchronous calls: uahn_filter_propagate, uahn_filter_frame and uahn_filter_frame_raw only enqueue work on the stream
 * of the bank's handle (and, for raw frames, on the bank's copy stream).
 * Their HOST inputs are borrowed until uahn_filter_wait returns, and their HOST outputs land there (the contract of
 * uahn_submit_batch / uahn_wait; pinned buffers are recommended).  Messages of failed calls: uahn_last_error(h).
 */
#ifndef UAHN_FILTER_H_
#define UAHN_FILTER_H_

#include "uahn.h"
#include "uahn_ekf.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct uahn_filter uahn_filter;

/* n slots (1 <= n <= max_batch of h) with one propagator configuration.  The bank owns its states, its two n-frame
 * buffers (previous / current frame of every slot) and its prior / mean / cov buffers: uahn_infer_batch* on h stays
 * usable between frames.  States start zeroed; set them with uahn_filter_set_states. */
UAHN_API int uahn_filter_create(uahn_handle* h, int n, const uahn_propagator_config* cfg, uahn_filter** out);
UAHN_API void uahn_filter_destroy(uahn_filter* f);

/* slots [first, first + count): copy HOST states in and zero their frame counters (a new sequence); synchronous. */
UAHN_API int uahn_filter_set_states(uahn_filter* f, int first, int count, const uahn_ekf_state* states);
/* slots [first, first + count) -> HOST states, after all enqueued work; synchronous. */
UAHN_API int uahn_filter_get_states(uahn_filter* f, int first, int count, uahn_ekf_state* states);

/* uahn_imu_propagate for every slot: slot i's raw readings are imu[offsets[i] .. offsets[i+1]) (HOST), integrated
 * between t0[i] and t1[i].  t1[i] <= t0[i]: slot i reports UAHN_ERR_STATE at uahn_filter_wait and keeps its state. */
UAHN_API int uahn_filter_propagate(uahn_filter* f, const uahn_imu_sample* imu, const int* offsets, const double* t0,
                                   const double* t1);

/* uahn_ekf_iekf_frame for every slot.  frames: n new 224x320 u8 frames (HOST, one per slot; the slot's previous frame
 * is its prev).  Iteration it runs uahn_infer_batch_device over the n pairs on h (it == 0) or h_iter (it > 0; NULL = h)
 * with MC-dropout pair index first_pair_index + it * n + slot; rng NULL = seed 0 and a bank counter that advances by
 * max_iter * n per frame (fresh masks every frame).  Explicit keep-masks: UAHN_ERR_UNSUPPORTED.  h_iter must be on h's
 * device with max_batch >= n; its forward is ordered against the bank's stream with events.
 * use_measurement: n bytes (0 = skip the updates of that slot this frame, the reference's timestamp gate) or NULL = all.
 * A slot updates when its frame count (frames since its set_states) is > min_images; with fewer than 2 frames it skips
 * the updates ("Only has one image") and still resets its offsets.  A singular (or NaN) innovation covariance stops the
 * slot where uahn_ekf_iekf_frame returns: no further updates, no reset, UAHN_ERR_INVALID at uahn_filter_wait.
 * Optional HOST outputs, max_iter x n rows each (row it * n + slot): prior_out (x8 float, the prior the forward got),
 * mean_out (x8), cov_out (x64) (rows of a slot with fewer than 2 frames are not meaningful); imu_out: n x 16 IMU values
 * after the frame (the trajectory). */
UAHN_API int uahn_filter_frame(uahn_filter* f, uahn_handle* h_iter, const uint8_t* frames, int max_iter, double K_net_Cov,
                               int min_images, const uint8_t* use_measurement, const uahn_rng* rng, float* prior_out,
                               float* mean_out, float* cov_out, double* imu_out);

/* Raw camera frames (undistort + resize on the device, as uahn_set_undistort_maps / uahn_load_raw_image do for one
 * handle).  One camera per bank (the bank already has one propagator config, i.e. one rig).  map1 / map2: HOST, 224*320
 * floats each (uahn_undistort_init_maps' output); raw frames are raw_rows x raw_cols u8 (2 ... 32767 each).  Allocates the
 * raw staging (2 x n raw frames on the device) and the bank's copy stream on first use; synchronous. */
UAHN_API int uahn_filter_set_undistort_maps(uahn_filter* f, int raw_rows, int raw_cols, const float* map1, const float* map2);

/* uahn_filter_frame with raw frames: raw holds n HOST frames [n][raw_rows][stride] (stride >= raw_cols bytes, slot i's
 * frame at raw + i * raw_rows * stride).  Slot i's current frame becomes remap(raw_i) (cv::remap INTER_LINEAR,
 * constant-0 border, bit for bit); everything after that (ring flip, priors, forwards, updates, outputs, rng numbering,
 * status) is exactly uahn_filter_frame's, and the two calls may alternate on one bank.  The upload runs on the bank's copy
 * stream into one of two staging buffers, so with pinned frames the upload of the next call overlaps this call's
 * forward.  UAHN_ERR_STATE without maps. */
UAHN_API int uahn_filter_frame_raw(uahn_filter* f, uahn_handle* h_iter, const uint8_t* raw, size_t stride, int max_iter,
                                   double K_net_Cov, int min_images, const uint8_t* use_measurement, const uahn_rng* rng,
                                   float* prior_out, float* mean_out, float* cov_out, double* imu_out);

/* Parity entry, in the manner of uahn_stage_undistort: remap n raw frames (laid out as for uahn_filter_frame_raw) with
 * the bank's maps into out (HOST, n x 224 x 320 u8) without touching the bank's ring or states; synchronous. */
UAHN_API int uahn_filter_stage_undistort(uahn_filter* f, const uint8_t* raw, size_t stride, uint8_t* out);

/* Waits for everything enqueued on the bank; status (optional): n per-slot codes since the previous wait (UAHN_OK,
 * UAHN_ERR_STATE, UAHN_ERR_INVALID).  Returns the first nonzero slot code, else UAHN_OK (or a CUDA error). */
UAHN_API int uahn_filter_wait(uahn_filter* f, int* status);

#ifdef __cplusplus
}
#endif
#endif /* UAHN_FILTER_H_ */
