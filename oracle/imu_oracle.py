"""TEST INFRASTRUCTURE — numpy restatement of the CUAHN-VIO IMU propagation (SURVEY §8f row 3).

Only tests/ may import this.  Follows, expression by expression (products left to right, like Eigen):
  Propagator::select_imu_readings / interpolate_data   /root/reference/cuahn_ros/cuahn/src/state/Propagator.cpp:80-180,
                                                       Propagator.h:179-189
  Propagator::predict_and_compute                      Propagator.cpp:183-339
  Propagator::predict_mean_discrete                    Propagator.cpp:342-363
  constants / noise                                    Propagator.h:50-103,192-194 ; State.h:110-113
  StateHelper::propagate_Cov                           cuahn/src/state/StateHelper.cpp:28-32
  quaternion helpers                                   ov_core/src/utils/quat_ops.h:141-145,479-484,526-550,573-588

Zero rotations: rotvec_2_ham_quat and jr_theta take the limits sin(a/2)/a -> 1/2 and J_r -> I at an exactly zero angle
(n == 0 only), as csrc/ekf_math.h does.  The reference divides by the angle unconditionally (NaN there); the limit is
the library's documented deviation.

Parity pinning: none available from the reference (no tests, Eigen absent) — "parity unpinned"; tests/test_imu.py
checks this restatement against finite differences of its own mean propagation and the C++ against this restatement.
"""
from __future__ import annotations

import numpy as np

from oracle.ekf_oracle import ham_quat_update, quatnorm, skew_x

CAM_PTS = np.array([[-1.0, -0.69906, 1.0], [-1.0, 0.69906, 1.0], [1.0, 0.69906, 1.0], [1.0, -0.69906, 1.0]])   # State.h:110-113
I33 = np.eye(3)
EZT = np.array([[0.0, 0.0, 1.0]])
MUW = np.array([[0.0], [0.0], [-1.0]])


def ham_quat_2_rot(q):                              # quat_ops.h:546-550
    qv = q[1:4].reshape(3, 1)
    return np.eye(3) * (q[0] * q[0] - (q[1] * q[1] + q[2] * q[2] + q[3] * q[3])) + 2 * qv @ qv.T + 2 * q[0] * skew_x(qv[:, 0])


def rotvec_2_ham_quat(rv):                          # quat_ops.h:582-588
    n = np.linalg.norm(rv)
    q = np.empty(4)
    q[0] = np.cos(n * 0.5)
    q[1:4] = (np.sin(n * 0.5) / n if n != 0 else 0.5) * rv
    return q


def jr_theta(th):                                   # quat_ops.h:573-580
    n = np.linalg.norm(th)
    if n == 0:
        return np.eye(3)
    S = skew_x(th)
    return np.eye(3) - (1 - np.cos(n)) / (n * n) * S + (n - np.sin(n)) / (n * n * n) * S @ S


SIGMA_DEFAULTS = {"sigma_w": 1.6968e-04, "sigma_a": 2.0000e-3, "sigma_wb": 1.9393e-05, "sigma_ab": 3.0000e-03}  # Propagator.h:50-71
GRAVITY_DEFAULT = 9.81                                                                                          # Propagator.h:100


def noise_Q(sw=1.6968e-04, sa=2.0000e-3, swb=1.9393e-05, sab=3.0000e-03):     # Propagator.h:50-97
    Q = np.zeros((15, 15))
    Q[0:3, 0:3] = sw ** 2 * I33
    Q[3:6, 3:6] = sa ** 2 * I33
    Q[6:9, 6:9] = sab ** 2 * I33
    Q[9:12, 9:12] = swb ** 2 * I33
    Q[12:15, 12:15] = 1.0e-04 * I33
    return Q


def interpolate(a, b, t):                           # Propagator.h:179-189 ; samples are (t, wm[3], am[3])
    lam = (t - a[0]) / (b[0] - a[0])
    return (t, (1 - lam) * a[1] + lam * b[1], (1 - lam) * a[2] + lam * b[2])


def select_imu_readings(imu, time0, time1):         # Propagator.cpp:80-180
    prop = []
    if not imu:
        return prop
    for i in range(len(imu) - 1):
        if imu[i + 1][0] > time0 and imu[i][0] < time0:
            prop.append(interpolate(imu[i], imu[i + 1], time0))
            continue
        if imu[i][0] >= time0 and imu[i + 1][0] <= time1:
            prop.append(imu[i])
            continue
        if imu[i + 1][0] > time1:
            if imu[i][0] > time1 and i == 0:
                break
            elif imu[i][0] > time1:
                prop.append(interpolate(imu[i - 1], imu[i], time1))
            else:
                prop.append(imu[i])
            if prop[-1][0] != time1:
                prop.append(interpolate(imu[i], imu[i + 1], time1))
            break
    if not prop:
        return prop
    i = 0
    while i < len(prop) - 1:
        if abs(prop[i + 1][0] - prop[i][0]) < 1e-12:
            prop.pop(i)
        else:
            i += 1
    return prop


def predict_mean_discrete(imu, offsets, cRi, it, dt, w_hat, a_hat, gravity):
    """Propagator.cpp:342-363 (+ the shared quantities of :213-221).  Returns (new imu[16], new offsets[4,3])."""
    pos, q, vel = imu[0:3], imu[3:7], imu[7:10]
    Rot = ham_quat_2_rot(q)
    wc = cRi @ w_hat
    vc = cRi @ (vel + skew_x(w_hat) @ it)
    muc = (cRi @ Rot.T @ MUW)[:, 0]
    dc = (Rot @ (pos + it))[2]
    new = imu.copy()
    new[3:7] = quatnorm(ham_quat_update(w_hat * dt) @ q)
    new[7:10] = vel + dt * (-skew_x(w_hat) @ vel + a_hat + Rot.T @ gravity)
    new[0:3] = pos + dt * (-skew_x(w_hat) @ pos + vel)
    H = skew_x(wc) + vc.reshape(3, 1) @ muc.reshape(1, 3) / dc
    noff = np.empty((4, 3))
    for k in range(4):
        pt = (CAM_PTS[k] + offsets[k]).reshape(3, 1)
        noff[k] = offsets[k] + dt * (-(I33 - pt @ EZT) @ H @ pt)[:, 0]
    return new, noff


def predict_and_compute(imu, offsets, cRi, it, minus, plus, imu_avg=True, gravity_mag=9.81):
    """Propagator.cpp:183-339.  Returns (new imu, new offsets, F[27,27], Fw[27,15])."""
    imu, offsets = imu.astype(np.float64), offsets.astype(np.float64)
    dt = plus[0] - minus[0]
    ba, bg = imu[10:13], imu[13:16]
    w1, a1, w2, a2 = minus[1] - bg, minus[2] - ba, plus[1] - bg, plus[2] - ba
    w_hat, a_hat = (.5 * (w1 + w2), .5 * (a1 + a2)) if imu_avg else (w2, a2)
    gravity = np.array([0.0, 0.0, -gravity_mag])
    pos, q, vel = imu[0:3], imu[3:7], imu[7:10]
    Rot = ham_quat_2_rot(q)
    wc = (cRi @ w_hat).reshape(3, 1)
    vc = (cRi @ (vel + skew_x(w_hat) @ it)).reshape(3, 1)
    muc = cRi @ Rot.T @ MUW
    dc = (Rot @ (pos + it))[2]
    new_imu, new_off = predict_mean_discrete(imu, offsets, cRi, it, dt, w_hat, a_hat, gravity)

    P, Qi, V, BA, BG = 0, 3, 6, 9, 12
    F = np.zeros((27, 27))
    Fw = np.zeros((27, 15))
    F[P:P + 3, P:P + 3] = I33 - dt * skew_x(w_hat)
    F[P:P + 3, V:V + 3] = dt * I33
    F[P:P + 3, BG:BG + 3] = -dt * skew_x(pos)
    F[Qi:Qi + 3, Qi:Qi + 3] = ham_quat_2_rot(rotvec_2_ham_quat(w_hat * dt)).T
    F[Qi:Qi + 3, BG:BG + 3] = -dt * jr_theta(w_hat * dt)
    F[V:V + 3, Qi:Qi + 3] = dt * skew_x(Rot.T @ gravity)
    F[V:V + 3, V:V + 3] = I33 - dt * skew_x(w_hat)
    F[V:V + 3, BA:BA + 3] = -dt * I33
    F[V:V + 3, BG:BG + 3] = -dt * skew_x(vel)
    F[BA:BA + 3, BA:BA + 3] = I33
    F[BG:BG + 3, BG:BG + 3] = I33

    scalar = (EZT @ vc).item() / dc
    Swc = skew_x(wc[:, 0])
    J_f_df = -dt * I33
    J_dc_p = EZT @ Rot
    J_dc_q = EZT @ (-Rot @ skew_x(pos + it))
    J_muc_q = cRi @ skew_x((Rot.T @ MUW)[:, 0])
    J_vc_v, J_vc_bw, J_wc_bw = cRi, cRi @ skew_x(it), -cRi                                  # Propagator.h:192-194
    for k in range(4):
        pt = (CAM_PTS[k] + offsets[k]).reshape(3, 1)
        J_df_pt = (Swc + vc @ muc.T / dc - (EZT @ Swc @ pt).item() * I33 - pt @ EZT @ Swc
                   - scalar * ((muc.T @ pt).item() * I33 + pt @ muc.T))
        common = I33 - pt @ EZT
        J_df_dc = 1.0 / dc / dc * (muc.T @ pt).item() * (-common) @ vc
        J_df_vc = 1.0 / dc * (muc.T @ pt).item() * common
        J_df_muc = 1.0 / dc * common @ vc @ pt.T
        J_df_wc = -common @ skew_x(pt[:, 0])
        R = 15 + 3 * k
        F[R:R + 3, P:P + 3] = J_f_df @ J_df_dc @ J_dc_p
        F[R:R + 3, Qi:Qi + 3] = J_f_df @ (J_df_dc @ J_dc_q + J_df_muc @ J_muc_q)
        F[R:R + 3, V:V + 3] = J_f_df @ J_df_vc @ J_vc_v
        F[R:R + 3, BG:BG + 3] = J_f_df @ (J_df_vc @ J_vc_bw + J_df_wc @ J_wc_bw)
        F[R:R + 3, R:R + 3] = I33 + J_f_df @ J_df_pt
    Fw[P:P + 3, 0:3] = -F[P:P + 3, BG:BG + 3]
    Fw[P:P + 3, 12:15] = F[P:P + 3, V:V + 3]
    Fw[Qi:Qi + 3, 0:3] = -F[Qi:Qi + 3, BG:BG + 3]
    Fw[V:V + 3, 0:3] = -F[V:V + 3, BG:BG + 3]
    Fw[V:V + 3, 3:6] = Fw[P:P + 3, 12:15]
    Fw[BA:BA + 3, 6:9] = Fw[P:P + 3, 12:15]
    Fw[BG:BG + 3, 9:12] = Fw[P:P + 3, 12:15]
    for k in range(4):
        R = 15 + 3 * k
        Fw[R:R + 3, 0:3] = -F[R:R + 3, BG:BG + 3]
    return new_imu, new_off, F, Fw


def plane_distance(imu, it):
    """dc of predict_and_compute (Propagator.cpp:216): the camera's distance to the ground plane, which the corner
    dynamics divide by."""
    return (ham_quat_2_rot(imu[3:7]) @ (imu[0:3] + it))[2]


def propagate(imu, offsets, P, cRi, it, readings, time0, time1, imu_avg=True, sigma_w=0.0, sigma_a=0.0, sigma_wb=0.0,
              sigma_ab=0.0, gravity_mag=0.0, dc_trace=None):
    """Propagator.cpp:28-79 + StateHelper.cpp:28-32.  The sigmas and gravity_mag resolve like uahn_propagator_config's
    (resolve_config): a value <= 0 selects the reference default.  dc_trace (a list) receives plane_distance() of the
    state entering every interval."""
    prop = select_imu_readings(readings, time0, time1)
    given = {"sigma_w": sigma_w, "sigma_a": sigma_a, "sigma_wb": sigma_wb, "sigma_ab": sigma_ab}
    sig = {k: v if v > 0 else SIGMA_DEFAULTS[k] for k, v in given.items()}
    Q = noise_Q(sig["sigma_w"], sig["sigma_a"], sig["sigma_wb"], sig["sigma_ab"])
    g = gravity_mag if gravity_mag > 0 else GRAVITY_DEFAULT
    P = P.astype(np.float64).copy()
    n = 0
    if len(prop) > 1:
        for i in range(len(prop) - 1):
            if dc_trace is not None:
                dc_trace.append(plane_distance(imu, it))
            imu, offsets, F, Fw = predict_and_compute(imu, offsets, cRi, it, prop[i], prop[i + 1], imu_avg, g)
            P = F @ P @ F.T + Fw @ Q @ Fw.T
            n += 1
    return imu, offsets, P, n
