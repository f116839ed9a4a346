"""TEST INFRASTRUCTURE — per-slot replay of the filter bank (include/uahn_filter.h, DESIGN §11 "Per-slot semantics") on
the numpy restatements of imu_oracle.py and ekf_oracle.py.

Only tests/ may import this.  It shares no code with csrc/ekf_math.h, so the bank's kernels can be held to it directly.
A slot's state is a tuple (imu[16], offsets[4, 3], P[27, 27]) of float64 arrays; a propagator configuration is a dict
with the fields of uahn_propagator_config (c_R_i, i_t_i2c, imu_avg, sigma_w, sigma_a, sigma_wb, sigma_ab, gravity_mag),
where a sigma or gravity_mag <= 0 selects the reference default.

  propagate()       uahn_filter_propagate for one slot: t1 <= t0 (NaN included) reports ERR_STATE, state untouched
  frame()           uahn_filter_frame for one slot, fed the network rows the bank reported
  edge_schedules()  IMU schedules at the edges of select_imu_readings and of the rotation math
  propagate_slot(), replay_slot()   the same, as picklable jobs for a process pool (workers import numpy and oracle only)
"""
from __future__ import annotations

import numpy as np

from oracle import ekf_oracle as E, imu_oracle as I

OK, ERR_INVALID, ERR_STATE = 0, -1, -4      # include/uahn.h
HZ_IMU, HZ_CAM = 500.0, 30.0                # tools/filter_bench.py
PLANE_MIN = 0.05                            # |dc| below this: the corner dynamics' 1 / dc is ill-posed (ekf_math.h:185)
COND_MAX = 1e12                             # cond(S) above this: the update is ill-posed in fp64
_H = E.measurement_jacobian()


def _propagate_kw(cfg):
    """imu_propagate's keywords: imu_avg is required (uahn_propagator_config has no default for it); a sigma or
    gravity_mag left out is 0, the reference default."""
    return {"imu_avg": bool(cfg["imu_avg"]),
            **{k: cfg.get(k, 0.0) for k in ("sigma_w", "sigma_a", "sigma_wb", "sigma_ab", "gravity_mag")}}


def propagate(state, readings, t0, t1, cfg):
    """→ (status, state, intervals, min |dc| over the intervals (inf if none))."""
    if not t1 > t0:
        return ERR_STATE, state, 0, np.inf
    dcs = []
    with np.errstate(all="ignore"):
        imu, off, P, n = I.propagate(*state, np.asarray(cfg["c_R_i"], np.float64).reshape(3, 3),
                                     np.asarray(cfg["i_t_i2c"], np.float64), readings, t0, t1, dc_trace=dcs,
                                     **_propagate_kw(cfg))
    return OK, (imu, off, P), n, min((abs(d) for d in dcs), default=np.inf)


def innovation_cov(P, cov_px, K_net_Cov):
    """S = H P H^T + Hn (K_net_Cov * Cov / 25440.25) Hn^T (UpdaterHNet.cpp:31), as ekf_oracle.update forms it."""
    return _H @ P @ _H.T + K_net_Cov * cov_px / 25440.25


def frame(state, count, mean_rows, cov_rows, max_iter, K_net_Cov, min_images, use=True):
    """One frame of one slot whose frame counter was `count` before it.  mean_rows [max_iter, 8] / cov_rows
    [max_iter, 8, 8]: the float rows the network produced for this slot, widened to float64.

    → dict(status, state, count, prior [max_iter, 8] float32, cond [cond(S) of every update], amp, prior_amp).  A
    non-finite S or a singular one (np.linalg.inv raises) is ERR_INVALID: the slot stops for the frame and is not reset.

    amp is the first-order amplification of a relative rounding error through the frame's updates:
    prod_it cond(S_it) * max|S_0| / max|S_it|.  With one update it is cond(S).  A later update's S is the difference of
    the earlier P and K H P, so it carries an error of eps * max|S_0| / max|S_it| relative to itself before its inverse
    amplifies that by cond(S_it).  When max|S_0| / max|S_1| is large (a measurement noise far below H P H^T) the second
    update is ill-posed whatever cond(S_1) is, and amp says so.  prior_amp[it] is the same product over the updates
    before iteration `it` only: what prior[it] inherits (1 for it = 0)."""
    imu, off, P = state
    count = count + 1
    prior = np.empty((max_iter, 8), np.float32)
    conds, amp, s0, prior_amp = [], 1.0, None, []
    status = OK
    with np.errstate(all="ignore"):
        for it in range(max_iter):
            prior[it] = (off[:, :2].reshape(8) * E.FOCAL).astype(np.float32)
            prior_amp.append(amp)
            if status or not (count >= 2 and count > min_images and use):
                continue
            cov = np.asarray(cov_rows[it], np.float64).reshape(8, 8)
            S = innovation_cov(P, cov, K_net_Cov)
            if not np.isfinite(S).all():
                status = ERR_INVALID
                continue
            conds.append(float(np.linalg.cond(S)))
            s0 = np.abs(S).max() if s0 is None else s0
            amp *= conds[-1] * s0 / np.abs(S).max()
            try:
                imu, off, P = E.update(imu, off, P, np.asarray(mean_rows[it], np.float64), cov, off[:, :2].reshape(8),
                                       it != max_iter - 1, K_net_Cov)
            except np.linalg.LinAlgError:
                status = ERR_INVALID
        if not status:
            off, P = E.reset_4pt_offset(off, P)
    return {"status": status, "state": (imu, off, P), "count": count, "prior": prior, "cond": conds, "amp": amp,
            "prior_amp": prior_amp}


# ---- configurations and states ----------------------------------------------------------------------------------------

def rotation(rng, tilt):
    q = np.concatenate([[1.0], tilt * rng.standard_normal(3)])
    q /= np.linalg.norm(q)
    return I.ham_quat_2_rot(q), q


def configs(rng):
    """The two propagator configurations the parity tests run, with P0 scales:
      A  the reference defaults, imu_avg on, a slightly tilted extrinsic; P0 ~ 1e-4
      B  imu_avg off, each sigma a different 10-100x its default (so a swap of two is visible), gravity_mag 9.80665, a
         strongly rotated extrinsic; P0 ~ 1e-8, so that the Fw Q Fw^T terms are a visible share of P."""
    cRi_a, _ = rotation(rng, 0.1)
    cRi_b, _ = rotation(rng, 1.0)
    d = I.SIGMA_DEFAULTS
    return {
        "A": ({"c_R_i": cRi_a, "i_t_i2c": 0.05 * rng.standard_normal(3), "imu_avg": 1}, 1e-4),
        "B": ({"c_R_i": cRi_b, "i_t_i2c": 0.1 * rng.standard_normal(3), "imu_avg": 0, "sigma_w": 20 * d["sigma_w"],
               "sigma_a": 50 * d["sigma_a"], "sigma_wb": 100 * d["sigma_wb"], "sigma_ab": 10 * d["sigma_ab"],
               "gravity_mag": 9.80665}, 1e-8),
    }


def initial_state(rng, p_scale=1e-4):
    """A camera ~1.5 m above the plane looking down (the corner dynamics divide by the height), P0 ~ p_scale.  The
    quaternion has q[3] >= 0, the sign every quaternion update leaves (quatnorm)."""
    _, q = rotation(rng, 0.1)
    q = q if q[3] >= 0 else -q
    imu = np.concatenate([[0.3, -0.2, 1.5] + 0.1 * rng.standard_normal(3), q, 0.5 * rng.standard_normal(3),
                          0.02 * rng.standard_normal(3), 0.005 * rng.standard_normal(3)])
    off = 0.02 * rng.standard_normal((4, 3))
    A = rng.standard_normal((27, 27))
    P = p_scale * ((A @ A.T) / 27 + 1e-2 * np.eye(27))
    return imu, off, P


# ---- IMU schedules ------------------------------------------------------------------------------------------------

def reading(rng, t, w_scale=0.3, w_mean=(0.0, 0.0, 0.0)):
    return (t, np.asarray(w_mean) + w_scale * rng.standard_normal(3), np.array([0, 0, 9.81]) + 0.5 * rng.standard_normal(3))


def bench_step(rng, t0, phase, dt=1.0 / HZ_CAM):
    """tools/filter_bench.py's imu_steps for one slot: 500 Hz readings at phase + k / 500 from just before t0 to just after
    t0 + dt.  → (readings, t0, t1)."""
    k0 = int(np.floor((t0 - phase) * HZ_IMU)) - 1
    cnt = int(np.ceil(dt * HZ_IMU)) + 3
    return [reading(rng, phase + (k0 + j) / HZ_IMU) for j in range(cnt)], t0, t0 + dt


def edge_schedules(rng):
    """→ list of dict(name, readings, t0, t1, zero_bg).  zero_bg: the slot's gyro bias must be exactly zero (with wm = 0
    exactly the bias-corrected rate is exactly zero, so every interval takes the zero-angle limits)."""
    t0 = 10.0 + 0.01 * rng.random()
    out = []

    def add(name, readings, a, b, zero_bg=False):
        out.append({"name": name, "readings": readings, "t0": a, "t1": b, "zero_bg": zero_bg})

    add("bench", *bench_step(rng, t0, 0.002 * rng.random()))
    add("gap_0.5s", *bench_step(rng, t0, 0.002 * rng.random(), 0.5))
    # a < t0 < t1 < b < c: interpolated at t0 and at t1 and nothing between
    t1 = t0 + 1.0 / HZ_CAM
    add("one_interval", [reading(rng, t0 - 0.001), reading(rng, t1 + 0.001), reading(rng, t1 + 0.003)], t0, t1)
    r = [reading(rng, 10.0 + k / HZ_IMU) for k in range(24)]
    add("on_readings", r, r[2][0], r[19][0])
    add("late_start", [reading(rng, t0 + 0.005 + k / HZ_IMU) for k in range(20)], t0, t1)
    add("early_end", [reading(rng, t0 - 0.001 + k / HZ_IMU) for k in range(10)], t0, t1)
    r, _, _ = bench_step(rng, t0, 0.0)
    r.insert(8, reading(rng, r[7][0] + 5e-13))                    # < 1e-12 s after its neighbour: de-duplicated
    add("near_duplicate", r, t0, t1)
    add("empty", [], t0, t1)
    add("single", [reading(rng, t0 + 0.01)], t0, t1)
    r, _, _ = bench_step(rng, t0, 0.001)
    add("t1_eq_t0", r, t0, t0)
    add("t1_lt_t0", r, t0, t0 - 0.01)
    add("t1_nan", r, t0, float("nan"))
    add("stationary", [(t, np.zeros(3), am) for t, _, am in bench_step(rng, t0, 0.0015)[0]], t0, t1, zero_bg=True)
    r, _, _ = bench_step(rng, t0, 0.0005)
    add("spin_20rad_s", [reading(rng, t, 0.5, (3.0, -4.0, 19.4)) for t, _, _ in r], t0, t1)
    return out


# ---- process-pool jobs ----------------------------------------------------------------------------------------------

def propagate_slot(job):
    """job = (state, readings, t0, t1, cfg) → propagate()'s result."""
    return propagate(*job)


def replay_slot(job):
    """A slot's closed loop, frame by frame.  job = dict(state, cfg, steps, mean, cov, max_iter, K_net_Cov, min_images,
    use): steps[k] = (readings, t0, t1) propagated before frame k (None: no propagation), mean [frames, max_iter, 8] and
    cov [frames, max_iter, 8, 8] the slot's network rows.  The replay stops after the first failing frame.

    → list per frame of dict(status, prior, cond, min_dc, state)."""
    state, count, out = job["state"], 0, []
    for k in range(len(job["steps"])):
        min_dc, status = np.inf, OK
        if job["steps"][k] is not None:
            status, state, _, min_dc = propagate(state, *job["steps"][k], job["cfg"])
        r = frame(state, count, job["mean"][k], job["cov"][k], job["max_iter"], job["K_net_Cov"], job["min_images"],
                  job["use"])
        state, count = r["state"], r["count"]
        out.append({"status": r["status"] or status, "prior": r["prior"], "cond": r["cond"], "min_dc": min_dc,
                    "state": state})
        if r["status"]:
            break
    return out
