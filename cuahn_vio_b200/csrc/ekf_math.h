// fp64 per-element math of the CUAHN-VIO filter, shared by the host consumer (imu_propagate.cpp, ekf_update.cpp,
// compiled with -ffp-contract=off) and the filter-bank kernels (filter_bank.cu, compiled with -fmad=false): one
// transcription of the reference, two compilations.  Every expression is evaluated left to right like the Eigen
// expression it restates, and every sum runs over its index in ascending order, so both compilations round alike (the
// device's sin / cos may differ from the host's libm in the last bit).
// References: see the headers of imu_propagate.cpp and ekf_update.cpp.
#pragma once
#include <math.h>
#include <string.h>

#include "../../include/uahn_ekf.h"

#ifdef __CUDACC__
#define UAHN_HD __host__ __device__
#else
#define UAHN_HD
#endif

namespace uahn_ekf {

constexpr int D = UAHN_EKF_DIM;
struct V3 { double v[3]; };
struct M3 { double m[9]; };

// ---- 3x3 helpers (quat_ops.h) ---------------------------------------------------------------------------------
UAHN_HD inline M3 skew(const V3& w) { return {{0, -w.v[2], w.v[1], w.v[2], 0, -w.v[0], -w.v[1], w.v[0], 0}}; }   // quat_ops.h:141-145
UAHN_HD inline M3 eye() { return {{1, 0, 0, 0, 1, 0, 0, 0, 1}}; }
UAHN_HD inline M3 mul(const M3& a, const M3& b) {
  M3 c;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double acc = 0;
      for (int k = 0; k < 3; ++k) acc += a.m[i * 3 + k] * b.m[k * 3 + j];
      c.m[i * 3 + j] = acc;
    }
  return c;
}
UAHN_HD inline V3 mul(const M3& a, const V3& b) {
  V3 c;
  for (int i = 0; i < 3; ++i) c.v[i] = a.m[i * 3] * b.v[0] + a.m[i * 3 + 1] * b.v[1] + a.m[i * 3 + 2] * b.v[2];
  return c;
}
UAHN_HD inline M3 tr(const M3& a) { return {{a.m[0], a.m[3], a.m[6], a.m[1], a.m[4], a.m[7], a.m[2], a.m[5], a.m[8]}}; }
UAHN_HD inline M3 add(const M3& a, const M3& b) { M3 c; for (int i = 0; i < 9; ++i) c.m[i] = a.m[i] + b.m[i]; return c; }
UAHN_HD inline M3 sub(const M3& a, const M3& b) { M3 c; for (int i = 0; i < 9; ++i) c.m[i] = a.m[i] - b.m[i]; return c; }
UAHN_HD inline M3 scale(double s, const M3& a) { M3 c; for (int i = 0; i < 9; ++i) c.m[i] = s * a.m[i]; return c; }
UAHN_HD inline V3 add(const V3& a, const V3& b) { return {{a.v[0] + b.v[0], a.v[1] + b.v[1], a.v[2] + b.v[2]}}; }
UAHN_HD inline V3 sub(const V3& a, const V3& b) { return {{a.v[0] - b.v[0], a.v[1] - b.v[1], a.v[2] - b.v[2]}}; }
UAHN_HD inline V3 scale(double s, const V3& a) { return {{s * a.v[0], s * a.v[1], s * a.v[2]}}; }
UAHN_HD inline double dot(const V3& a, const V3& b) { return a.v[0] * b.v[0] + a.v[1] * b.v[1] + a.v[2] * b.v[2]; }
UAHN_HD inline M3 outer(const V3& a, const V3& b) {
  M3 c;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) c.m[i * 3 + j] = a.v[i] * b.v[j];
  return c;
}
UAHN_HD inline double norm(const V3& a) { return sqrt(dot(a, a)); }

// quat_ops.h:546-550 (Hamilton, scalar first): R = (q0^2 - |qv|^2) I + 2 qv qv^T + 2 q0 [qv]x
UAHN_HD inline M3 ham_quat_2_rot(const double* q) {
  const V3 qv{{q[1], q[2], q[3]}};
  return add(add(scale(q[0] * q[0] - (q[1] * q[1] + q[2] * q[2] + q[3] * q[3]), eye()), scale(2.0, outer(qv, qv))),
             scale(2.0 * q[0], skew(qv)));
}
// The trigonometry of a rotation vector of norm n, evaluated once: sin / cos of n / 2 and of n.  predict_and_compute takes
// it precomputed, so that the device's out-of-line slow-path reduction of sin / cos is called where little is live.
struct Trig { double n, sh, ch, s, c; };
UAHN_HD inline Trig trig_of(const V3& rv) {
  const double n = norm(rv);
  return {n, sin(n * 0.5), cos(n * 0.5), sin(n), cos(n)};
}
// quat_ops.h:582-588
UAHN_HD inline void rotvec_2_ham_quat(const V3& rv, const Trig& g, double* q) {
  const double k = g.n > 0.0 ? g.sh / g.n : 0.5;                // (the reference divides by the norm unconditionally)
  q[0] = g.ch;
  for (int i = 0; i < 3; ++i) q[1 + i] = k * rv.v[i];
}
// quat_ops.h:573-580
UAHN_HD inline M3 jr_theta(const V3& th, const Trig& g) {
  const double n = g.n;
  if (!(n > 0.0)) return eye();                                 // limit of the reference's expression
  const M3 S = skew(th);
  return add(sub(eye(), scale((1 - g.c) / (n * n), S)), scale((n - g.s) / (n * n * n), mul(S, S)));
}
// quat_ops.h:526-538 then :479-484: out <- quatnorm(Ham_quat_update(rot_vec) * q).  The reference divides by the angle
// unconditionally and would produce NaN for an exactly zero increment; the limit sin(a/2)/a -> 1/2 is used instead.
UAHN_HD inline void quat_update(const V3& rot_vec, const Trig& g, const double* q, double* out) {
  const double angle = g.n;
  const double k = angle > 0.0 ? g.sh / angle : 0.5;
  const double d0 = k * rot_vec.v[0], d1 = k * rot_vec.v[1], d2 = k * rot_vec.v[2], c = g.ch;
  // qR = [[c, -d^T], [d, c I + skew_x(-d)]]  (quat_ops.h:532-535)
  const double M[16] = {c, -d0, -d1, -d2, d0, c, d2, -d1, d1, -d2, c, d0, d2, d1, -d0, c};
  double qn[4];
  for (int r = 0; r < 4; ++r) qn[r] = M[r * 4] * q[0] + M[r * 4 + 1] * q[1] + M[r * 4 + 2] * q[2] + M[r * 4 + 3] * q[3];
  if (qn[3] < 0) for (int r = 0; r < 4; ++r) qn[r] = -qn[r];    // quat_ops.h:480-482 (sic: index 3)
  const double n = sqrt(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2] + qn[3] * qn[3]);
  for (int r = 0; r < 4; ++r) out[r] = qn[r] / n;
}

UAHN_HD inline void put(double* F, int ld, int r0, int c0, const M3& b) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) F[(r0 + i) * ld + c0 + j] = b.m[i * 3 + j];
}
UAHN_HD inline M3 get(const double* F, int ld, int r0, int c0) {
  M3 b;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) b.m[i * 3 + j] = F[(r0 + i) * ld + c0 + j];
  return b;
}

// ---- IMU propagation (Propagator.cpp:183-363, StateHelper.cpp:28-32) ------------------------------------------------
struct Cfg {   // uahn_propagator_config with the reference defaults resolved (resolve_config)
  M3 cRi;
  V3 it;
  double q_diag[15];
  V3 gravity;
  int imu_avg;
};

// host only: the configuration with the reference defaults filled in
inline Cfg resolve_config(const uahn_propagator_config* c) {
  Cfg r;
  memcpy(r.cRi.m, c->c_R_i, sizeof(r.cRi.m));
  memcpy(r.it.v, c->i_t_i2c, sizeof(r.it.v));
  const double sw = c->sigma_w > 0 ? c->sigma_w : 1.6968e-04, sa = c->sigma_a > 0 ? c->sigma_a : 2.0000e-3;   // Propagator.h:50-71
  const double swb = c->sigma_wb > 0 ? c->sigma_wb : 1.9393e-05, sab = c->sigma_ab > 0 ? c->sigma_ab : 3.0000e-03;
  for (int i = 0; i < 3; ++i) {                                                                                // Propagator.h:93-97
    r.q_diag[i] = pow(sw, 2);
    r.q_diag[3 + i] = pow(sa, 2);
    r.q_diag[6 + i] = pow(sab, 2);
    r.q_diag[9 + i] = pow(swb, 2);
    r.q_diag[12 + i] = 1.0e-04;
  }
  r.gravity = {{0.0, 0.0, -(c->gravity_mag > 0 ? c->gravity_mag : 9.81)}};                                     // Propagator.h:100
  r.imu_avg = c->imu_avg != 0 ? 1 : 0;
  return r;
}

// F's nonzero 3x3 blocks: bit c of f_row_blocks(b) is set when block row b has a block in block column c (the put()s
// of predict_and_compute).  Block rows: p, theta, v, ba, bg, then the four offsets.
UAHN_HD inline unsigned f_row_blocks(int b) {
  switch (b) {
    case 0: return 1u << 0 | 1u << 2 | 1u << 4;              // p: p, v, bg
    case 1: return 1u << 1 | 1u << 4;                        // theta: theta, bg
    case 2: return 1u << 1 | 1u << 2 | 1u << 3 | 1u << 4;    // v: theta, v, ba, bg
    case 3: return 1u << 3;                                  // ba
    case 4: return 1u << 4;                                  // bg
    default: return 1u << 0 | 1u << 1 | 1u << 2 | 1u << 4 | 1u << b;   // offset k: p, theta, v, bg, itself
  }
}
constexpr unsigned ALL_BLOCKS = 0x1FFu;

// the bias-corrected rates of one interval (:198-204)
UAHN_HD inline void interval_rates(const Cfg& c, const uahn_ekf_state* s, const uahn_imu_sample& dm, const uahn_imu_sample& dp,
                                   V3* w_hat, V3* a_hat) {
  const V3 ba{{s->imu[10], s->imu[11], s->imu[12]}}, bg{{s->imu[13], s->imu[14], s->imu[15]}};
  const V3 w1 = sub({{dm.wm[0], dm.wm[1], dm.wm[2]}}, bg), a1 = sub({{dm.am[0], dm.am[1], dm.am[2]}}, ba);
  const V3 w2 = sub({{dp.wm[0], dp.wm[1], dp.wm[2]}}, bg), a2 = sub({{dp.am[0], dp.am[1], dp.am[2]}}, ba);
  *w_hat = c.imu_avg ? scale(.5, add(w1, w2)) : w2;
  *a_hat = c.imu_avg ? scale(.5, add(a1, a2)) : a2;
}
// the trigonometry of the interval's rotation dt * w_hat (quat_update, rotvec_2_ham_quat and jr_theta all take it)
UAHN_HD inline Trig interval_trig(const Cfg& c, const uahn_ekf_state* s, const uahn_imu_sample& dm, const uahn_imu_sample& dp) {
  V3 w_hat, a_hat;
  interval_rates(c, s, dm, dp, &w_hat, &a_hat);
  return trig_of(scale(dp.t - dm.t, w_hat));
}

// predict_and_compute for one interval, g = interval_trig(c, s, dm, dp): advances the mean of *s (IMU value, offsets)
// and writes the nonzero blocks of F (27x27) and Fw (27x15), row-major.  The caller provides F and Fw with zeros
// everywhere else (the pattern is fixed, so a caller that keeps the arrays across intervals zeroes them once).
UAHN_HD inline void predict_and_compute(const Cfg& c, uahn_ekf_state* s, const uahn_imu_sample& dm, const uahn_imu_sample& dp,
                                        const Trig& g, double* F, double* Fw) {
  const double dt = dp.t - dm.t;
  const V3 pos{{s->imu[0], s->imu[1], s->imu[2]}}, vel{{s->imu[7], s->imu[8], s->imu[9]}};
  V3 w_hat, a_hat;
  interval_rates(c, s, dm, dp, &w_hat, &a_hat);
  const M3 Rot = ham_quat_2_rot(s->imu + 3), RotT = tr(Rot);
  const V3 muw{{0.0, 0.0, -1.0}}, ez{{0.0, 0.0, 1.0}};
  const M3 I = eye();
  // :213-216
  const V3 wc = mul(c.cRi, w_hat);
  const V3 vc = mul(c.cRi, add(vel, mul(skew(w_hat), c.it)));
  const V3 muc = mul(mul(c.cRi, RotT), muw);
  const double dc = mul(Rot, add(pos, c.it)).v[2];
  const double CAM[4][2] = {{-1.0, -0.69906}, {-1.0, 0.69906}, {1.0, 0.69906}, {1.0, -0.69906}};   // State.h:110-113 (z = 1)
  V3 pt[4];
  for (int k = 0; k < 4; ++k) pt[k] = {{CAM[k][0] + s->offset[k][0], CAM[k][1] + s->offset[k][1], 1.0 + s->offset[k][2]}};

  // ---- predict_mean_discrete (:342-363)
  double new_q[4];
  quat_update(scale(dt, w_hat), g, s->imu + 3, new_q);
  const V3 new_v = add(vel, scale(dt, add(add(scale(-1.0, mul(skew(w_hat), vel)), a_hat), mul(RotT, c.gravity))));
  const V3 new_p = add(pos, scale(dt, add(scale(-1.0, mul(skew(w_hat), pos)), vel)));
  const M3 H = add(skew(wc), scale(1.0 / dc, outer(vc, muc)));
  V3 new_off[4];
  for (int k = 0; k < 4; ++k) {
    const M3 common = sub(I, outer(pt[k], ez));
    const V3 cur{{s->offset[k][0], s->offset[k][1], s->offset[k][2]}};
    new_off[k] = add(cur, scale(dt, mul(scale(-1.0, common), mul(H, pt[k]))));
  }

  // ---- Jacobians (:224-325)
  const int P = 0, Q = 3, V = 6, BA = 9, BG = 12;
  put(F, D, P, P, sub(I, scale(dt, skew(w_hat))));
  put(F, D, P, V, scale(dt, I));
  put(F, D, P, BG, scale(-dt, skew(pos)));
  double dq[4];
  rotvec_2_ham_quat(scale(dt, w_hat), g, dq);
  put(F, D, Q, Q, tr(ham_quat_2_rot(dq)));
  put(F, D, Q, BG, scale(-dt, jr_theta(scale(dt, w_hat), g)));
  put(F, D, V, Q, scale(dt, skew(mul(RotT, c.gravity))));
  put(F, D, V, V, sub(I, scale(dt, skew(w_hat))));
  put(F, D, V, BA, scale(-dt, I));
  put(F, D, V, BG, scale(-dt, skew(vel)));
  put(F, D, BA, BA, I);
  put(F, D, BG, BG, I);

  const double scalar = dot(ez, vc) / dc;                                                      // :240-241
  const M3 J_f_df = scale(-dt, I);                                                             // :288
  const V3 J_dc_p = mul(tr(Rot), ez);                        // (ezT * Rot)^T                    :289
  const V3 J_dc_q = mul(tr(scale(-1.0, mul(Rot, skew(add(pos, c.it))))), ez);                  // :290
  const M3 J_muc_q = mul(c.cRi, skew(mul(RotT, muw)));                                         // :291
  const M3 J_vc_v = c.cRi, J_vc_bw = mul(c.cRi, skew(c.it)), J_wc_bw = scale(-1.0, c.cRi);     // Propagator.h:192-194
  const M3 Swc = skew(wc);
  const V3 ezSwc = mul(tr(Swc), ez);                         // (ezT * skew_x(wc))^T
  for (int k = 0; k < 4; ++k) {
    const V3& p = pt[k];
    const double ez_swc_p = dot(ezSwc, p), muc_p = dot(muc, p);
    // J_df_pt = [wc]x + vc muc^T / dc - (ezT [wc]x pt) I - pt (ezT [wc]x) - scalar ((muc^T pt) I + pt muc^T)   (:244-246)
    M3 J_df_pt = add(Swc, scale(1.0 / dc, outer(vc, muc)));
    J_df_pt = sub(J_df_pt, scale(ez_swc_p, I));
    J_df_pt = sub(J_df_pt, outer(p, ezSwc));
    J_df_pt = sub(J_df_pt, scale(scalar, add(scale(muc_p, I), outer(p, muc))));
    const M3 common = sub(I, outer(p, ez));                                                    // :247
    const V3 J_df_dc = mul(scale(1.0 / dc / dc * muc_p, scale(-1.0, common)), vc);             // :248
    const M3 J_df_vc = scale(1.0 / dc * muc_p, common);                                        // :249
    const M3 J_df_muc = scale(1.0 / dc, outer(mul(common, vc), p));                            // :250
    const M3 J_df_wc = scale(-1.0, mul(common, skew(p)));                                      // :251
    const int R = 15 + 3 * k;
    put(F, D, R, P, outer(mul(J_f_df, J_df_dc), J_dc_p));                                      // :294
    put(F, D, R, Q, mul(J_f_df, add(outer(J_df_dc, J_dc_q), mul(J_df_muc, J_muc_q))));         // :295
    put(F, D, R, V, mul(mul(J_f_df, J_df_vc), J_vc_v));                                        // :296
    put(F, D, R, BG, mul(J_f_df, add(mul(J_df_vc, J_vc_bw), mul(J_df_wc, J_wc_bw))));          // :297
    put(F, D, R, R, add(I, mul(J_f_df, J_df_pt)));                                             // :298
  }
  // Fw (:319-332)
  const M3 dtI = get(F, D, P, V);
  put(Fw, 15, P, 0, scale(-1.0, get(F, D, P, BG)));
  put(Fw, 15, P, 12, dtI);
  put(Fw, 15, Q, 0, scale(-1.0, get(F, D, Q, BG)));
  put(Fw, 15, V, 0, scale(-1.0, get(F, D, V, BG)));
  put(Fw, 15, V, 3, dtI);
  put(Fw, 15, BA, 6, dtI);
  put(Fw, 15, BG, 9, dtI);
  for (int k = 0; k < 4; ++k) put(Fw, 15, 15 + 3 * k, 0, scale(-1.0, get(F, D, 15 + 3 * k, BG)));

  // new mean (:335-345)
  for (int i = 0; i < 3; ++i) { s->imu[i] = new_p.v[i]; s->imu[7 + i] = new_v.v[i]; }
  for (int i = 0; i < 4; ++i) s->imu[3 + i] = new_q[i];
  for (int k = 0; k < 4; ++k)
    for (int i = 0; i < 3; ++i) s->offset[k][i] = new_off[k].v[i];
}

// P <- F P F^T + Fw Q Fw^T (Q diagonal), element by element in two passes: FP = F P, then P'[i][j] = (FP F^T)[i][j] +
// (Fw Q Fw^T)[i][j].  `blocks` restricts the sum over k to F's nonzero block columns of the row that multiplies (the
// host passes ALL_BLOCKS, the reference's dense sum); skipped terms are exact zeros for finite P.
UAHN_HD inline double fp_element(const double* F, const double* P, int i, int j, unsigned blocks) {
  double acc = 0;
  for (int b = 0; b < 9; ++b)
    if (blocks >> b & 1u)
      for (int k = 3 * b; k < 3 * b + 3; ++k) acc += F[i * D + k] * P[k * D + j];
  return acc;
}
UAHN_HD inline double pn_element(const Cfg& c, const double* FP, const double* F, const double* Fw, int i, int j,
                                 unsigned blocks) {
  double acc = 0;
  for (int b = 0; b < 9; ++b)
    if (blocks >> b & 1u)
      for (int k = 3 * b; k < 3 * b + 3; ++k) acc += FP[i * D + k] * F[j * D + k];
  double nq = 0;
  for (int k = 0; k < 15; ++k) nq += Fw[i * 15 + k] * c.q_diag[k] * Fw[j * 15 + k];
  return acc + nq;
}

// ---- EKF measurement update (UpdaterHNet.cpp:28-61) --------------------------------------------------------------
// rows of the measurement Jacobian H (UpdaterHNet.h:58-62): the (u, v) components of the four offsets
UAHN_HD inline int meas_row(int i) { return 15 + 3 * (i >> 1) + (i & 1); }   // 15, 16, 18, 19, 21, 22, 24, 25

// In-place inverse of an 8x8 matrix by Gauss-Jordan elimination with partial pivoting; inv: 64 doubles of workspace.
UAHN_HD inline bool invert8(double* a, double* inv) {
  for (int i = 0; i < 64; ++i) inv[i] = (i / 8 == i % 8) ? 1.0 : 0.0;
  for (int c = 0; c < 8; ++c) {
    int piv = c;
    for (int r = c + 1; r < 8; ++r)
      if (fabs(a[r * 8 + c]) > fabs(a[piv * 8 + c])) piv = r;
    if (!(fabs(a[piv * 8 + c]) > 0.0)) return false;   // singular (or NaN)
    if (piv != c)
      for (int k = 0; k < 8; ++k) {
        const double t = a[c * 8 + k]; a[c * 8 + k] = a[piv * 8 + k]; a[piv * 8 + k] = t;
        const double u = inv[c * 8 + k]; inv[c * 8 + k] = inv[piv * 8 + k]; inv[piv * 8 + k] = u;
      }
    const double d = 1.0 / a[c * 8 + c];
    for (int k = 0; k < 8; ++k) { a[c * 8 + k] *= d; inv[c * 8 + k] *= d; }
    for (int r = 0; r < 8; ++r) {
      if (r == c) continue;
      const double f = a[r * 8 + c];
      if (f == 0.0) continue;
      for (int k = 0; k < 8; ++k) { a[r * 8 + k] -= f * a[c * 8 + k]; inv[r * 8 + k] -= f * inv[c * 8 + k]; }
    }
  }
  for (int i = 0; i < 64; ++i) a[i] = inv[i];
  return true;
}

// S[i][j] = H P H^T + Hn (K_net_Cov * Cov / 25440.25) Hn^T, Hn = I (UpdaterHNet.cpp:31, UpdaterHNet.h:64)
UAHN_HD inline double innovation_cov_element(const double* P, const double* cov_px64, double K_net_Cov, int i, int j) {
  return P[meas_row(i) * D + meas_row(j)] + K_net_Cov * cov_px64[i * 8 + j] / 25440.25;
}
// K = P H^T S^-1  (27 x 8)
UAHN_HD inline double gain_element(const double* P, const double* Sinv, int r, int j) {
  double acc = 0.0;
  for (int i = 0; i < 8; ++i) acc += P[r * D + meas_row(i)] * Sinv[i * 8 + j];
  return acc;
}
// innovation = mean / 159.5 - propagated (:33)
UAHN_HD inline double innovation_element(const double* mean_px8, const double* propagated8, int i) {
  return mean_px8[i] / UAHN_FOCAL_PX - propagated8[i];
}
// P <- (I - K H) P = P - K (H P)  (:36): the subtrahend of P[r][c]; HP holds the rows meas_row(0..7) of the old P
UAHN_HD inline double cov_update_element(const double* K, const double* HP, int r, int c) {
  double acc = 0.0;
  for (int i = 0; i < 8; ++i) acc += K[r * 8 + i] * HP[i * D + c];
  return acc;
}
// state increment dx = K * innovation (:39-44)
UAHN_HD inline double increment_element(const double* K, const double* inno, int r) {
  double acc = 0.0;
  for (int i = 0; i < 8; ++i) acc += K[r * 8 + i] * inno[i];
  return acc;
}
// state += dx (:47-60); without update_offset only the 15 IMU rows of dx are read and the offsets stay
UAHN_HD inline void apply_increment(uahn_ekf_state* s, const double* dx, int update_offset) {
  double* x = s->imu;
  for (int k = 0; k < 3; ++k) x[k] += dx[k];                                                       // :47
  {   // :48  q <- quatnorm(Ham_quat_update(dtheta) * q)
    double q[4];
    for (int r = 0; r < 4; ++r) q[r] = x[3 + r];
    const V3 dtheta{{dx[3], dx[4], dx[5]}};
    quat_update(dtheta, trig_of(dtheta), q, x + 3);
  }
  for (int k = 0; k < 3; ++k) x[7 + k] += dx[6 + k];                                               // :49
  for (int k = 0; k < 3; ++k) x[10 + k] += dx[9 + k];                                              // :50
  for (int k = 0; k < 3; ++k) x[13 + k] += dx[12 + k];                                             // :51
  if (update_offset)                                                                               // :55-60
    for (int c = 0; c < 4; ++c)
      for (int k = 0; k < 3; ++k) s->offset[c][k] += dx[15 + 3 * c + k];
}

// State::reset_4pt_offset (State.cpp:101-111): the covariance keeps only its IMU 15x15 block
UAHN_HD inline bool reset_keeps(int r, int c) { return r < 15 && c < 15; }

}  // namespace uahn_ekf
