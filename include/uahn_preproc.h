/*
 * uahn_preproc.h — the step immediately in front of the UAHN path (SURVEY §8f, "next" row 2): undistort + resize of the
 * raw camera frame to the network's 224x320, 90-degree-FoV pinhole image.
 *
 * Replaces, in the reference,
 *   CamBase::initialize_undist_map / initialize_undist_map_fisheye   cuahn_ros/ov_core/src/cam/CamBase.h:165-180
 *   CamBase::undistort_and_resize_img (cv::remap, INTER_LINEAR)      cuahn_ros/ov_core/src/cam/CamBase.h:182-186
 *   and its call site                                                 cuahn_ros/cuahn/src/core/VioManager.cpp:181-188
 * so that raw frames can be handed to the library directly (one H2D of the raw frame, a gather kernel, no host OpenCV).
 * The arithmetic is OpenCV's, reproduced bit for bit: maps in double like cv::[fisheye::]initUndistortRectifyMap,
 * sampling like cv::remap on CV_8UC1 with CV_32FC1 maps (1/32-pixel fixed-point coordinates, integer bilinear table,
 * constant-0 border).
 */
#ifndef UAHN_PREPROC_H_
#define UAHN_PREPROC_H_

#include "uahn.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Host only.  k = (fx, fy, cx, cy) and d = 4 distortion coefficients of the RAW camera (fisheye != 0: equidistant
 * k1..k4, cv::fisheye; else radtan k1, k2, p1, p2).  map1 / map2: 224*320 floats each — the raw-image x / y sampled by
 * every output pixel; the target camera is fixed: f = 159.5, c = (159.5, 111.5) (CamBase.h:166-169). */
UAHN_API int uahn_undistort_init_maps(int fisheye, const double* k4, const double* d4, float* map1, float* map2);

/* Upload the maps (HOST pointers) and declare the raw frame size; enables uahn_load_raw_image and
 * uahn_submit_sequence_raw.  Waits for the handle's enqueued work first: a submission already made keeps the old maps. */
UAHN_API int uahn_set_undistort_maps(uahn_handle* h, int raw_rows, int raw_cols, const float* map1, const float* map2);

/* uahn_submit_sequence with raw frames: raw holds n_frames HOST frames [n_frames][raw_rows][stride] of ONE sequence
 * (stride >= raw_cols bytes).  Pair i = (remap(raw_i), remap(raw_{i+1})), cv::remap-exact with the handle's maps.
 * Everything after the remap (priors, rng numbering, outputs, the uahn_wait contract, at most two in flight) is
 * exactly uahn_submit_sequence's.  UAHN_ERR_STATE without maps.  The upload of submission i+1 runs on the copy
 * stream under the remap and forward of submission i; raw should be pinned for the copy to overlap.  Device memory:
 * two staging buffers of (max_batch + 1) raw frames, allocated by the first call. */
UAHN_API int uahn_submit_sequence_raw(uahn_handle* h, int n_frames, const uint8_t* raw, size_t stride,
                                      const float* prior, const uahn_rng* rng, float* mean, float* cov);

/* undistort_and_resize_img + load_current_img (VioManager.cpp:181-188) in one call: raw is CV_8UC1 raw_rows x raw_cols
 * with `stride` bytes per row, borrowed for the duration of the call.  prev <- curr, curr <- remap(raw). */
UAHN_API int uahn_load_raw_image(uahn_handle* h, const uint8_t* raw, int rows, int cols, size_t stride, double time_stamp);

/* Parity-test entry: remap one raw frame and return the 224x320 u8 image (HOST buffers, synchronous). */
UAHN_API int uahn_stage_undistort(uahn_handle* h, const uint8_t* raw, int rows, int cols, size_t stride, uint8_t* out);

#ifdef __cplusplus
}
#endif
#endif /* UAHN_PREPROC_H_ */
