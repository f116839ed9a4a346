// Host-side consumer of the UAHN outputs (SURVEY §8f row 1): the EKF measurement update of CUAHN-VIO and the IEKF loop
// around the network call, Eigen-free.  Reference: cuahn_ros/cuahn/src/update/UpdaterHNet.cpp:28-61,
// cuahn_ros/cuahn/src/update/UpdaterHNet.h:56-66, cuahn_ros/cuahn/src/state/State.cpp:101-111,
// cuahn_ros/cuahn/src/core/VioManager.cpp:227-275, ov_core/src/utils/quat_ops.h:141-145,479-484,526-538.
#include <cmath>
#include <cstring>

#include "../../include/uahn_ekf.h"
#include "ekf_math.h"

using namespace uahn_ekf;

extern "C" {

int uahn_ekf_prior_px(const uahn_ekf_state* s, double* prior_px8, double* propagated8) {
  if (!s || !prior_px8) return UAHN_ERR_INVALID;
  for (int c = 0; c < 4; ++c)
    for (int k = 0; k < 2; ++k) {
      const double v = s->offset[c][k];                        // VioManager.cpp:230-233
      if (propagated8) propagated8[2 * c + k] = v;
      prior_px8[2 * c + k] = v * UAHN_FOCAL_PX;                // :234
    }
  return UAHN_OK;
}

int uahn_ekf_update(uahn_ekf_state* s, const double* mean_px8, const double* cov_px64, const double* propagated8,
                    int update_offset, double K_net_Cov) {
  if (!s || !mean_px8 || !cov_px64 || !propagated8) return UAHN_ERR_INVALID;
  double* P = s->cov;
  double Sinv[64], work[64];
  for (int i = 0; i < 8; ++i)
    for (int j = 0; j < 8; ++j) Sinv[i * 8 + j] = innovation_cov_element(P, cov_px64, K_net_Cov, i, j);
  if (!invert8(Sinv, work)) return UAHN_ERR_INVALID;
  double K[D * 8];
  for (int r = 0; r < D; ++r)
    for (int j = 0; j < 8; ++j) K[r * 8 + j] = gain_element(P, Sinv, r, j);
  double inno[8];
  for (int i = 0; i < 8; ++i) inno[i] = innovation_element(mean_px8, propagated8, i);
  double HP[8 * D];
  for (int i = 0; i < 8; ++i) std::memcpy(HP + i * D, P + meas_row(i) * D, D * sizeof(double));
  for (int r = 0; r < D; ++r)
    for (int c = 0; c < D; ++c) P[r * D + c] -= cov_update_element(K, HP, r, c);
  // without update_offset only the 15 IMU rows of the increment are used
  double dx[D];
  const int rows = update_offset ? D : 15;
  for (int r = 0; r < rows; ++r) dx[r] = increment_element(K, inno, r);
  apply_increment(s, dx, update_offset);
  return UAHN_OK;
}

int uahn_ekf_reset_offsets(uahn_ekf_state* s) {
  if (!s) return UAHN_ERR_INVALID;
  std::memset(s->offset, 0, sizeof(s->offset));
  for (int r = 0; r < D; ++r)
    for (int c = 0; c < D; ++c)
      if (!reset_keeps(r, c)) s->cov[r * D + c] = 0.0;
  return UAHN_OK;
}

int uahn_ekf_iekf_frame(uahn_handle* h, uahn_handle* h_iter, uahn_ekf_state* s, int max_iter, double K_net_Cov,
                        int min_images, int use_measurement, const uahn_rng* rng, double* mean_px8, double* cov_px64) {
  if (!h || !s || max_iter < 1) return UAHN_ERR_INVALID;
  double mean[8] = {0}, cov[64] = {0};
  for (int it = 0; it < max_iter; ++it) {                                                          // VioManager.cpp:227
    double prior_px[8], propagated[8];
    uahn_ekf_prior_px(s, prior_px, propagated);                                                    // :230-234
    uahn_handle* net = (it > 0 && h_iter) ? h_iter : h;                                            // HomographyNet.cpp:209
    // fresh MC-dropout masks for every forward (model_to_trace.py:266-273): iteration `it` of this frame uses pair index
    // first_pair_index + it (the caller advances first_pair_index by max_iter per frame); a NULL rng lets each handle
    // number its own calls
    uahn_rng it_rng{};
    if (rng) { it_rng = *rng; it_rng.first_pair_index += (uint64_t)it; }
    int rc = uahn_infer(net, prior_px, rng ? &it_rng : nullptr, mean, cov, nullptr);               // :236
    if (rc == UAHN_ERR_STATE) continue;        // "Only has one image": outputs untouched, loop goes on (HomographyNet.cpp:155-158)
    if (rc) return rc;
    if (use_measurement && uahn_image_count(h) > min_images) {                                     // :257
      rc = uahn_ekf_update(s, mean, cov, propagated, it != max_iter - 1, K_net_Cov);               // :260-264
      if (rc) return rc;
    }
  }
  uahn_ekf_reset_offsets(s);                                                                       // :275
  if (mean_px8) std::memcpy(mean_px8, mean, sizeof(mean));
  if (cov_px64) std::memcpy(cov_px64, cov, sizeof(cov));
  return UAHN_OK;
}

}  // extern "C"
