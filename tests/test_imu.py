"""SURVEY §8f row 3 — IMU propagation (Propagator.cpp:28-363) behind the C ABI vs the numpy restatement, and the
restatement's Jacobians vs finite differences of its own mean propagation.  CPU only."""
import numpy as np
import pytest

from oracle import filter_oracle as F, imu_oracle as I


@pytest.fixture(scope="module")
def api():
    from cuahn_vio_b200 import build
    build.build()
    from cuahn_vio_b200 import api as a
    a.load_library()
    return a


def _rot(rng):
    q = rng.standard_normal(4)
    q /= np.linalg.norm(q)
    return I.ham_quat_2_rot(q), q


def _state(rng):
    _, q = _rot(rng)
    if q[3] < 0:
        q = -q
    imu = np.concatenate([[0.3, -0.2, 1.5] + 0.1 * rng.standard_normal(3), q, 0.5 * rng.standard_normal(3),
                          0.02 * rng.standard_normal(3), 0.005 * rng.standard_normal(3)])
    # keep the camera looking at the ground plane from above: height dc well away from zero
    off = 0.02 * rng.standard_normal((4, 3))
    A = rng.standard_normal((27, 27))
    P = 1e-4 * (A @ A.T) / 27 + 1e-6 * np.eye(27)
    return imu, off, P


def _readings(rng, t0=10.0, n=30, hz=200.0):
    return [(t0 + k / hz, 0.3 * rng.standard_normal(3), np.array([0, 0, 9.81]) + 0.5 * rng.standard_normal(3)) for k in range(n)]


def _extrinsics(rng):
    cRi, _ = _rot(rng)
    return cRi, 0.05 * rng.standard_normal(3)


def test_select_readings_matches_restatement(api):
    rng = np.random.default_rng(3)
    r = _readings(rng)
    for t0, t1 in ((10.012, 10.071), (10.0, 10.05), (10.0025, 10.1449), (9.0, 10.02), (10.01, 10.01 + 1e-13), (11.0, 12.0)):
        got = api.imu_select_readings(r, t0, t1)
        exp = I.select_imu_readings(r, t0, t1)
        assert len(got) == len(exp)
        for g, e in zip(got, exp):
            assert g[0] == e[0] and np.array_equal(g[1], e[1]) and np.array_equal(g[2], e[2])
    inner = api.imu_select_readings(r, 10.012, 10.071)
    assert inner[0][0] == 10.012 and inner[-1][0] == 10.071 and all(b[0] > a[0] for a, b in zip(inner, inner[1:]))
    assert api.imu_select_readings([], 0.0, 1.0) == []


@pytest.mark.parametrize("imu_avg", [True, False])
def test_predict_and_compute_matches_restatement(api, imu_avg):
    rng = np.random.default_rng(8)
    for trial in range(10):
        imu, off, P = _state(rng)
        cRi, it = _extrinsics(rng)
        r = _readings(rng, n=2)
        cfg = api.PropagatorConfig.make(cRi, it, imu_avg)
        st = api.EkfState.from_arrays(imu, off, P)
        F, Fw = api.imu_predict_and_compute(cfg, st, r[0], r[1])
        imu2, off2, P2 = st.arrays()
        ei, eo, eF, eFw = I.predict_and_compute(imu, off, cRi, it, r[0], r[1], imu_avg)
        assert np.abs(imu2 - ei).max() < 1e-13 and np.abs(off2 - eo).max() < 1e-13
        assert np.abs(F - eF).max() < 1e-12 and np.abs(Fw - eFw).max() < 1e-12
        assert np.array_equal(P2, P)                       # the covariance is propagate_Cov's job


def test_jacobians_match_finite_differences():
    """F's additive blocks = d(new state)/d(state) of predict_mean_discrete (checks the transcription of :224-325)."""
    rng = np.random.default_rng(21)
    imu, off, _ = _state(rng)
    cRi, it = _extrinsics(rng)
    r = _readings(rng, n=2)
    dt = r[1][0] - r[0][0]
    _, _, F, _ = I.predict_and_compute(imu, off, cRi, it, r[0], r[1], True)
    g = np.array([0, 0, -9.81])

    def mean(imu_, off_):
        w_hat = .5 * ((r[0][1] - imu_[13:16]) + (r[1][1] - imu_[13:16]))
        a_hat = .5 * ((r[0][2] - imu_[10:13]) + (r[1][2] - imu_[10:13]))
        ni, no = I.predict_mean_discrete(imu_, off_, cRi, it, dt, w_hat, a_hat, g)
        return np.concatenate([ni[0:3], ni[7:10], ni[10:13], ni[13:16], no.ravel()])   # p, v, ba, bg, offsets

    rows = [0, 1, 2, 6, 7, 8, 9, 10, 11, 12, 13, 14] + list(range(15, 27))          # error-state rows of those outputs
    eps = 1e-6
    # columns: p (0-2), v (6-8), ba (9-11), bg (12-14) live in imu[0:3], imu[7:10], imu[10:13], imu[13:16]
    for col, idx in [(0, 0), (1, 1), (2, 2), (6, 7), (7, 8), (8, 9), (9, 10), (10, 11), (11, 12), (12, 13), (13, 14), (14, 15)]:
        d = np.zeros(16); d[idx] = eps
        num = (mean(imu + d, off) - mean(imu - d, off)) / (2 * eps)
        assert np.abs(num - F[rows, col]).max() < 2e-7, (col, np.abs(num - F[rows, col]).max())
    for k in range(4):
        for j in range(3):
            d = np.zeros((4, 3)); d[k, j] = eps
            num = (mean(imu, off + d) - mean(imu, off - d)) / (2 * eps)
            assert np.abs(num - F[rows, 15 + 3 * k + j]).max() < 2e-7


def _propagate_both(api, c, state, readings, t0, t1):
    """uahn_imu_propagate and filter_oracle.propagate from the same state → (host status, intervals, state arrays),
    (oracle status, intervals, state)."""
    st = api.EkfState.from_arrays(*state)
    try:
        rc, n = 0, api.imu_propagate(api.PropagatorConfig.make(**c), st, readings, t0, t1)
    except api.UahnError as e:
        rc, n = int(str(e).rsplit(" ", 1)[1]), 0
    status, est, en, _ = F.propagate(state, readings, t0, t1, c)
    return (rc, n, st.arrays()), (status, en, est)


def test_propagate_matches_restatement_and_keeps_cov_psd(api):
    rng = np.random.default_rng(13)
    imu, off, P = _state(rng)
    cRi, it = _extrinsics(rng)
    r = _readings(rng, n=40)
    (_, n, (imu2, off2, P2)), (_, en, (ei, eo, eP)) = _propagate_both(
        api, {"c_R_i": cRi, "i_t_i2c": it, "imu_avg": 1}, (imu, off, P), r, 10.012, 10.1333)
    assert n == en and n >= 20
    assert np.abs(imu2 - ei).max() < 1e-12 and np.abs(off2 - eo).max() < 1e-12
    assert np.abs(P2 - eP).max() < 1e-12 * max(1.0, np.abs(eP).max())
    st = api.EkfState.from_arrays(imu2, off2, P2)
    cfg = api.PropagatorConfig.make(cRi, it, True)
    assert np.linalg.eigvalsh(0.5 * (P2 + P2.T)).min() > 0 and np.trace(P2) > np.trace(P)
    # the prior the network gets after propagation: offsets x 159.5 (VioManager.cpp:230-234)
    prior_px, prop = api.ekf_prior_px(st)
    assert np.allclose(prior_px, off2[:, :2].reshape(8) * 159.5) and np.abs(prior_px).max() > 1e-3
    with pytest.raises(api.UahnError):
        api.imu_propagate(cfg, st, r, 10.1, 10.1)          # same instant: the reference exits (Propagator.cpp:32-35)


SCHEDULES = F.edge_schedules(np.random.default_rng(5))


@pytest.mark.parametrize("config", ["A", "B"])
@pytest.mark.parametrize("schedule", range(len(SCHEDULES)), ids=[s["name"] for s in SCHEDULES])
def test_propagate_edge_schedules_match_restatement(api, config, schedule):
    """uahn_imu_propagate (ekf_math.h on the host) against the numpy restatement over the schedules the filter-bank
    tests give their slots: long gaps, no interpolation, de-duplication, empty and single-reading lists, t1 <= t0, an
    exactly zero rate (the zero-angle limits) and a fast spin.  Configuration B sets every field of
    uahn_propagator_config away from its default."""
    rng = np.random.default_rng(100 + schedule)
    c, p_scale = F.configs(rng)[config]
    s = SCHEDULES[schedule]
    imu, off, P = F.initial_state(rng, p_scale)
    if s["zero_bg"]:
        imu[13:16] = 0.0
    (rc, n, (hi, ho, hP)), (status, en, (ei, eo, eP)) = _propagate_both(api, c, (imu, off, P), s["readings"], s["t0"], s["t1"])
    assert rc == status and n == en
    if status or n == 0:                       # t1 <= t0, or fewer than two selected readings: the state stays
        assert np.array_equal(hi, imu) and np.array_equal(ho, off) and np.array_equal(hP, P)
        assert s["name"] in ("empty", "single", "t1_eq_t0", "t1_lt_t0", "t1_nan")
        return
    assert np.isfinite(hi).all() and np.isfinite(hP).all() and np.isfinite(eP).all()
    e_imu = (np.abs(hi - ei) / np.maximum(1.0, np.abs(ei))).max()
    e_off = (np.abs(ho - eo) / np.maximum(1.0, np.abs(eo))).max()
    e_P = np.abs(hP - eP).max() / np.abs(eP).max()
    print(f"{s['name']} {config}: {n} intervals, imu {e_imu:.1e}, offsets {e_off:.1e}, P {e_P:.1e} (relative)")
    assert e_imu <= 1e-13 and e_off <= 1e-13 and e_P <= 1e-13        # worst seen: 9e-16
