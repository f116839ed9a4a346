// IMU propagation of the CUAHN-VIO filter state (SURVEY §8f row 3), Eigen-free fp64 host code.
// Reference: cuahn_ros/cuahn/src/state/Propagator.cpp:28-79 (propagate_with_imu), :80-180 (select_imu_readings),
// :183-339 (predict_and_compute), :342-363 (predict_mean_discrete); Propagator.h:50-103,179-195;
// cuahn_ros/cuahn/src/state/StateHelper.cpp:28-32; State.h:110-113; ov_core/src/utils/quat_ops.h:141-145,479-484,
// 526-550,573-588.  Products are evaluated left to right like the Eigen expressions they restate.
#include <cmath>
#include <cstring>
#include <vector>

#include "../../include/uahn_ekf.h"
#include "ekf_math.h"

namespace {

using namespace uahn_ekf;

uahn_imu_sample interpolate(const uahn_imu_sample& a, const uahn_imu_sample& b, double t) {   // Propagator.h:179-189
  const double lambda = (t - a.t) / (b.t - a.t);
  uahn_imu_sample d;
  d.t = t;
  for (int i = 0; i < 3; ++i) {
    d.am[i] = (1 - lambda) * a.am[i] + lambda * b.am[i];
    d.wm[i] = (1 - lambda) * a.wm[i] + lambda * b.wm[i];
  }
  return d;
}

std::vector<uahn_imu_sample> select(const uahn_imu_sample* imu, int n, double time0, double time1) {   // Propagator.cpp:80-180
  std::vector<uahn_imu_sample> prop;
  if (n <= 0) return prop;
  for (int i = 0; i < n - 1; ++i) {
    if (imu[i + 1].t > time0 && imu[i].t < time0) {            // start of the integration period: split
      prop.push_back(interpolate(imu[i], imu[i + 1], time0));
      continue;
    }
    if (imu[i].t >= time0 && imu[i + 1].t <= time1) {          // middle
      prop.push_back(imu[i]);
      continue;
    }
    if (imu[i + 1].t > time1) {                                // end: split the next measurement at time1
      if (imu[i].t > time1 && i == 0) {
        break;
      } else if (imu[i].t > time1) {
        prop.push_back(interpolate(imu[i - 1], imu[i], time1));
      } else {
        prop.push_back(imu[i]);
      }
      if (prop.back().t != time1) prop.push_back(interpolate(imu[i], imu[i + 1], time1));
      break;
    }
  }
  if (prop.empty()) return prop;
  for (size_t i = 0; i + 1 < prop.size(); ++i)                  // no zero-dt intervals
    if (std::fabs(prop[i + 1].t - prop[i].t) < 1e-12) {
      prop.erase(prop.begin() + i);
      --i;
    }
  return prop;
}

// predict_and_compute (ekf_math.h) on zeroed F / Fw
void predict_and_compute_dense(const Cfg& c, uahn_ekf_state* s, const uahn_imu_sample& dm, const uahn_imu_sample& dp, double* F,
                               double* Fw) {
  std::memset(F, 0, sizeof(double) * D * D);
  std::memset(Fw, 0, sizeof(double) * D * 15);
  predict_and_compute(c, s, dm, dp, interval_trig(c, s, dm, dp), F, Fw);
}

// StateHelper.cpp:28-32: P <- F P F^T + Fw Q Fw^T (Q diagonal)
void propagate_cov(const Cfg& c, uahn_ekf_state* s, const double* F, const double* Fw) {
  std::vector<double> FP(D * D);
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < D; ++j) FP[i * D + j] = fp_element(F, s->cov, i, j, ALL_BLOCKS);
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < D; ++j) s->cov[i * D + j] = pn_element(c, FP.data(), F, Fw, i, j, ALL_BLOCKS);
}

}  // namespace

extern "C" {

int uahn_imu_select_readings(const uahn_imu_sample* imu, int n, double time0, double time1, uahn_imu_sample* out, int capacity,
                             int* n_out) {
  if (!imu || !out || !n_out || n < 0) return UAHN_ERR_INVALID;
  const std::vector<uahn_imu_sample> p = select(imu, n, time0, time1);
  if ((int)p.size() > capacity) return UAHN_ERR_INVALID;
  for (size_t i = 0; i < p.size(); ++i) out[i] = p[i];
  *n_out = (int)p.size();
  return UAHN_OK;
}

int uahn_imu_predict_and_compute(const uahn_propagator_config* cfg, uahn_ekf_state* s, const uahn_imu_sample* minus,
                                 const uahn_imu_sample* plus, double* F, double* Fw) {
  if (!cfg || !s || !minus || !plus || !F || !Fw) return UAHN_ERR_INVALID;
  predict_and_compute_dense(resolve_config(cfg), s, *minus, *plus, F, Fw);
  return UAHN_OK;
}

int uahn_imu_propagate(const uahn_propagator_config* cfg, uahn_ekf_state* s, const uahn_imu_sample* imu, int n, double time0,
                       double time1, int* n_intervals) {
  if (!cfg || !s || !imu) return UAHN_ERR_INVALID;
  if (!(time1 > time0)) return UAHN_ERR_STATE;   // Propagator.cpp:32-42: same instant / backwards (the reference exits)
  const Cfg c = resolve_config(cfg);
  const std::vector<uahn_imu_sample> p = select(imu, n, time0, time1);
  std::vector<double> F(D * D), Fw(D * 15);   // zeroed once: predict_and_compute writes the same nonzero blocks every time
  int count = 0;
  if (p.size() > 1)                                                                            // :64-71
    for (size_t i = 0; i + 1 < p.size(); ++i, ++count) {
      predict_and_compute(c, s, p[i], p[i + 1], interval_trig(c, s, p[i], p[i + 1]), F.data(), Fw.data());
      propagate_cov(c, s, F.data(), Fw.data());
    }
  if (n_intervals) *n_intervals = count;
  return UAHN_OK;
}

}  // extern "C"
