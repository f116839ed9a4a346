"""TEST INFRASTRUCTURE — numpy restatement of the CUAHN-VIO EKF measurement update (SURVEY §8f row 1).

Only tests/ may import this.  Follows, line by line:
  UpdaterHNet::update      /root/reference/cuahn_ros/cuahn/src/update/UpdaterHNet.cpp:28-61
  H / Hn                   /root/reference/cuahn_ros/cuahn/src/update/UpdaterHNet.h:56-66
  State::reset_4pt_offset  /root/reference/cuahn_ros/cuahn/src/state/State.cpp:101-111
  skew_x / quatnorm / Ham_quat_update   /root/reference/cuahn_ros/ov_core/src/utils/quat_ops.h:141-145, 479-484, 526-538

Parity pinning: the reference ships no tests or vectors for this function and its C++ needs Eigen (absent here), so
this restatement is pinned only by the analytic known-answer tests in tests/test_ekf.py — "parity unpinned" in the
sense of the task contract; the formulas are a dozen lines of dense linear algebra transcribed from the cited lines.
"""
from __future__ import annotations

import numpy as np

FOCAL = 159.5


def measurement_jacobian() -> np.ndarray:
    H = np.zeros((8, 27))                       # UpdaterHNet.h:58-62
    for i, col in enumerate((15, 18, 21, 24)):
        H[2 * i:2 * i + 2, col:col + 2] = np.eye(2)
    return H


def skew_x(w):                                   # quat_ops.h:141-145
    return np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]], dtype=np.float64)


def ham_quat_update(rot_vec):                    # quat_ops.h:526-538
    """The reference divides by the angle unconditionally (NaN at zero); an exactly zero angle takes the limit
    sin(a/2)/a -> 1/2 instead, the library's documented deviation (csrc/ekf_math.h quat_update)."""
    ang = np.linalg.norm(rot_vec)
    dqv = (np.sin(ang * 0.5) / ang if ang != 0 else 0.5) * rot_vec
    M = np.eye(4) * np.cos(ang * 0.5)
    M[1:4, 1:4] += skew_x(-dqv)
    M[0, 1:4] = -dqv
    M[1:4, 0] = dqv
    return M


def quatnorm(q):                                 # quat_ops.h:479-484 (tests index 3, as the reference does)
    q = q.copy()
    if q[3] < 0:
        q *= -1
    return q / np.linalg.norm(q)


def update(imu, offsets, P, mean_px, cov_px, propagated, update_offset: bool, K_net_Cov: float = 10.0):
    """Returns (imu[16], offsets[4,3], P[27,27]) after UpdaterHNet::update."""
    imu, offsets, P = imu.astype(np.float64).copy(), offsets.astype(np.float64).copy(), P.astype(np.float64).copy()
    H, Hn = measurement_jacobian(), np.eye(8)
    K = P @ H.T @ np.linalg.inv(H @ P @ H.T + Hn @ (K_net_Cov * cov_px / 25440.25) @ Hn.T)     # :31
    inno = mean_px / FOCAL - propagated                                                       # :33
    P = (np.eye(27) - K @ H) @ P                                                              # :36
    d = K @ inno if update_offset else np.concatenate([K[:15] @ inno, np.zeros(12)])          # :39-44
    imu[0:3] += d[0:3]                                                                        # :47
    imu[3:7] = quatnorm(ham_quat_update(d[3:6]) @ imu[3:7])                                   # :48
    imu[7:10] += d[6:9]
    imu[10:13] += d[9:12]
    imu[13:16] += d[12:15]
    if update_offset:                                                                         # :55-60
        offsets += d[15:27].reshape(4, 3)
    return imu, offsets, P


def reset_4pt_offset(offsets, P):                # State.cpp:101-111
    Pn = np.zeros_like(P)
    Pn[:15, :15] = P[:15, :15]
    return np.zeros_like(offsets), Pn
