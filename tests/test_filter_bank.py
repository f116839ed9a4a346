"""Filter bank (include/uahn_filter.h): n EKF states propagated and updated on the GPU around one batched forward, held
to the batch-1 host path (uahn_imu_propagate, uahn_ekf_update, uahn_ekf_reset_offsets) replayed slot by slot."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from cuahn_vio_b200 import synthetic as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HZ_IMU, HZ_CAM = 500.0, 30.0


@pytest.fixture(scope="module")
def api():
    from cuahn_vio_b200 import build
    build.build()
    from cuahn_vio_b200 import api as a
    a.load_library()
    return a


# ---- CPU --------------------------------------------------------------------------------------------------

def test_filter_header_matches_binding_and_exports(api):
    src = open(os.path.join(ROOT, "include", "uahn_filter.h")).read()
    declared = sorted(set(re.findall(r"\b(uahn_filter_\w+)\s*\(", src)))
    assert declared == sorted(api.FILTER_SYMBOLS)
    lib = api.load_library()
    for name in api.FILTER_SYMBOLS:
        assert hasattr(lib, name), name


def test_filter_kernels_do_not_spill(api):
    from cuahn_vio_b200 import build
    src = os.path.join(build.CSRC, "filter_bank.cu")
    out = subprocess.run([build.NVCC, *build.FLAGS, "-fmad=false", "-Xptxas=-v", "-c", src, "-o", os.devnull],
                         capture_output=True, text=True, check=True).stderr
    kernels = re.findall(r"Compiling entry function '(\w+)'", out)
    assert len([k for k in kernels if "filter_" in k]) == 3
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", out)
    assert spills and all(a == "0" and b == "0" for a, b in spills), out


# ---- helpers ------------------------------------------------------------------------------------------------

def _rot(rng, tilt):
    q = np.concatenate([[1.0], tilt * rng.standard_normal(3)])
    q /= np.linalg.norm(q)
    from oracle import imu_oracle as I
    return I.ham_quat_2_rot(q), q


def _state(rng):
    """test_imu._state with a camera that looks down at the plane from ~1.5 m (the corner dynamics divide by the
    height) so that the states stay finite over a few frames."""
    _, q = _rot(rng, 0.1)
    imu = np.concatenate([[0.3, -0.2, 1.5] + 0.1 * rng.standard_normal(3), q, 0.5 * rng.standard_normal(3),
                          0.02 * rng.standard_normal(3), 0.005 * rng.standard_normal(3)])
    off = 0.02 * rng.standard_normal((4, 3))
    A = rng.standard_normal((27, 27))
    P = 1e-4 * (A @ A.T) / 27 + 1e-6 * np.eye(27)
    return imu, off, P


def _extrinsics(rng):
    cRi, _ = _rot(rng, 0.1)
    return cRi, 0.05 * rng.standard_normal(3)


def _readings(rng, t0, t1, phase):
    """500 Hz readings from just before t0 to just after t1, offset by a per-slot phase."""
    k0, k1 = int(np.floor((t0 - phase) * HZ_IMU)) - 1, int(np.ceil((t1 - phase) * HZ_IMU)) + 1
    return [(phase + k / HZ_IMU, 0.3 * rng.standard_normal(3), np.array([0, 0, 9.81]) + 0.5 * rng.standard_normal(3))
            for k in range(k0, k1 + 1)]


def _host_state(api, imu, off, P):
    return api.EkfState.from_arrays(imu, off, P)


def _assert_state_close(api, got, host, tol):
    gi, go, gP = got
    hi, ho, hP = host.arrays()
    assert np.isfinite(hi).all() and np.isfinite(hP).all()
    assert np.abs(gi - hi).max() <= tol and np.abs(go - ho).max() <= tol, (np.abs(gi - hi).max(), np.abs(go - ho).max())
    assert np.abs(gP - hP).max() <= tol * max(1.0, np.abs(hP).max()), np.abs(gP - hP).max()


# ---- GPU -----------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def wfile(api):
    from cuahn_vio_b200 import weights
    return weights.synthetic_weights_file(0)


@pytest.mark.gpu
def test_propagation_matches_host_per_slot(api, wfile):
    n = 37
    rng = np.random.default_rng(37)
    states = [_state(rng) for _ in range(n)]
    cRi, it = _extrinsics(rng)
    cfg = api.PropagatorConfig.make(cRi, it, True)
    t0 = 10.0 + 0.01 * rng.random(n)
    t1 = t0 + 1.0 / HZ_CAM + 0.01 * rng.random(n)
    t1[5] = t0[5]                                               # same instant: UAHN_ERR_STATE, state untouched
    readings = [_readings(rng, t0[i], t1[i], 0.002 * rng.random()) for i in range(n)]
    readings[9] = [r for r in readings[9] if r[0] < t0[9]][-1:]  # fewer than two readings in range: no interval
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net, api.FilterBank(net, n, cfg) as bank:
        bank.set_states(0, [s[0] for s in states], [s[1] for s in states], [s[2] for s in states])
        bank.propagate(readings, t0, t1)
        status = bank.wait()
        got = bank.get_states()
    assert status[5] == api.ERR_STATE and (np.delete(status, 5) == 0).all()
    for i in range(n):
        host = _host_state(api, *states[i])
        if i == 5:
            gi, go, gP = (g[i] for g in got)
            assert np.array_equal(gi, states[i][0]) and np.array_equal(go, states[i][1]) and np.array_equal(gP, states[i][2])
            continue
        api.imu_propagate(cfg, host, readings[i], t0[i], t1[i])
        _assert_state_close(api, tuple(g[i] for g in got), host, 1e-12)
    assert np.array_equal(got[2][9], states[9][2])              # no interval: P untouched


def _host_frame(api, host, it_outputs, count, max_iter, K_net_Cov, min_images, use):
    """uahn_ekf_iekf_frame's loop with the network outputs the device reported (float -> double)."""
    lib = api.load_library()
    for it in range(max_iter):
        _, propagated = api.ekf_prior_px(host)
        if count < 2:
            continue
        if use and count > min_images:
            mean, cov = (np.asarray(a, np.float64) for a in it_outputs[it])
            rc = lib.uahn_ekf_update(C.byref(host), api._ptr(mean), api._ptr(np.ascontiguousarray(cov.reshape(64))),
                                     api._ptr(propagated), int(it != max_iter - 1), float(K_net_Cov))
            if rc:
                return rc
    lib.uahn_ekf_reset_offsets(C.byref(host))
    return 0


def _sequences(n, n_frames):
    seqs = [S.synthetic_sequence(n_frames, seed=4000 + i)[0] for i in range(n)]
    return np.stack(seqs, 1)                                    # [frame][slot]


@pytest.fixture(scope="module")
def frames16():
    return _sequences(16, 6)


@pytest.mark.gpu
@pytest.mark.parametrize("precision,max_iter", [("fp32", 1), ("fp32", 2), ("bf16", 1), ("bf16", 2)])
def test_closed_loop_matches_host_replay(api, wfile, frames16, precision, max_iter):
    n, n_frames = 16, frames16.shape[0]
    K_net_Cov, min_images, seed = 10.0, 2, 7
    rng = np.random.default_rng(16 + max_iter)
    states = [_state(rng) for _ in range(n)]
    cRi, it = _extrinsics(rng)
    cfg = api.PropagatorConfig.make(cRi, it, True)
    use = np.ones(n, np.uint8)
    use[3] = 0                                                  # the reference's timestamp gate closed for slot 3
    restart_slot, restart_frame = 5, 3
    new_state = _state(rng)
    phase = 0.002 * rng.random(n)
    net = api.Uahn(wfile, "prior3", precision=precision, max_batch=n)
    net_iter = api.Uahn(wfile, "prior2", precision=precision, max_batch=n) if max_iter > 1 else None
    hosts = [_host_state(api, *s) for s in states]
    counts = np.zeros(n, int)
    prev = np.zeros_like(frames16[0])
    with net, api.FilterBank(net, n, cfg) as bank:
        bank.set_states(0, [s[0] for s in states], [s[1] for s in states], [s[2] for s in states])
        for k in range(n_frames):
            if k == restart_frame:                             # a new sequence in one slot
                bank.set_states(restart_slot, new_state[0][None], new_state[1][None], new_state[2][None])
                hosts[restart_slot] = _host_state(api, *new_state)
                counts[restart_slot] = 0
            if k > 0:
                t0 = 10.0 + (k - 1) / HZ_CAM + phase
                t1 = t0 + 1.0 / HZ_CAM
                readings = [_readings(rng, t0[i], t1[i], phase[i]) for i in range(n)]
                bank.propagate(readings, t0, t1)
                for i in range(n):
                    api.imu_propagate(cfg, hosts[i], readings[i], t0[i], t1[i])
            first = 1000 + k * max_iter * n
            out = bank.frame(frames16[k], max_iter, K_net_Cov, min_images, use, seed=seed, first_pair=first,
                             iterative=net_iter)
            assert (bank.wait() == 0).all()
            counts += 1
            for it_ in range(max_iter):
                h = net if it_ == 0 or net_iter is None else net_iter
                m, c, _ = h.infer_batch(prev, frames16[k], out["prior"][it_], seed=seed, first_pair=first + it_ * n)
                assert np.array_equal(m, out["mean"][it_]) and np.array_equal(c, out["cov"][it_]), (k, it_)
            for i in range(n):
                rows = [(out["mean"][it_, i], out["cov"][it_, i]) for it_ in range(max_iter)]
                # prior of every iteration: (float)(host offsets x 159.5), replayed step by step
                lib = api.load_library()
                for it_ in range(max_iter):
                    px, _ = api.ekf_prior_px(hosts[i])
                    exp = px.astype(np.float32)
                    assert (np.abs(out["prior"][it_, i] - exp) <= np.spacing(np.abs(exp))).all(), (k, i, it_)
                    if counts[i] >= 2 and use[i] and counts[i] > min_images:
                        mean, cov = (np.asarray(a, np.float64) for a in rows[it_])
                        _, propagated = api.ekf_prior_px(hosts[i])
                        assert lib.uahn_ekf_update(C.byref(hosts[i]), api._ptr(mean),
                                                   api._ptr(np.ascontiguousarray(cov.reshape(64))), api._ptr(propagated),
                                                   int(it_ != max_iter - 1), float(K_net_Cov)) == 0
                lib.uahn_ekf_reset_offsets(C.byref(hosts[i]))
                assert np.abs(out["imu"][i] - hosts[i].arrays()[0]).max() <= 1e-10
            prev = frames16[k]
        got = bank.get_states()
    if net_iter is not None:
        net_iter.close()
    assert counts.max() > min_images                           # the update gate opened mid-sequence
    for i in range(n):
        _assert_state_close(api, tuple(g[i] for g in got), hosts[i], 1e-10)
    # slot 3 never updated: its IMU value is the host propagation alone; updated slots moved away from it
    assert not np.array_equal(got[0][0], got[0][3])


@pytest.mark.gpu
def test_null_rng_draws_fresh_masks(api, wfile, frames16):
    n = 16
    cfg = api.PropagatorConfig.make(np.eye(3), np.zeros(3), True)
    rng = np.random.default_rng(3)
    states = [_state(rng) for _ in range(n)]
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net, api.FilterBank(net, n, cfg) as bank:
        bank.set_states(0, [s[0] for s in states], [s[1] for s in states], [s[2] for s in states])
        off = np.zeros(n, np.uint8)
        outs = []
        for _ in range(3):                                     # same frames, no updates: only the masks can change
            outs.append(bank.frame(frames16[0], 1, use_measurement=off))
            bank.wait()
    assert np.array_equal(outs[1]["prior"], outs[2]["prior"])
    assert not np.array_equal(outs[1]["mean"], outs[2]["mean"])


@pytest.mark.gpu
def test_singular_slot_stops_alone(api, wfile, frames16):
    n, K_net_Cov, min_images, max_iter = 4, 10.0, 0, 2
    rng = np.random.default_rng(44)
    states = [_state(rng) for _ in range(n)]
    bad = 2
    states[bad] = (states[bad][0], states[bad][1], np.full((27, 27), np.nan))
    cRi, it = _extrinsics(rng)
    cfg = api.PropagatorConfig.make(cRi, it, True)
    hosts = [_host_state(api, *s) for s in states]
    rcs = np.zeros(n, int)
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net, api.FilterBank(net, n, cfg) as bank:
        bank.set_states(0, [s[0] for s in states], [s[1] for s in states], [s[2] for s in states])
        for k in range(2):
            if k:
                t0 = np.full(n, 10.0)
                t1 = t0 + 1.0 / HZ_CAM
                readings = [_readings(rng, t0[i], t1[i], 0.0) for i in range(n)]
                bank.propagate(readings, t0, t1)
                for i in range(n):
                    api.imu_propagate(cfg, hosts[i], readings[i], t0[i], t1[i])
            out = bank.frame(frames16[k, :n], max_iter, K_net_Cov, min_images, seed=1, first_pair=50 * k)
            status = bank.wait()
            for i in range(n):
                if rcs[i]:
                    continue
                rows = [(out["mean"][it_, i], out["cov"][it_, i]) for it_ in range(max_iter)]
                rcs[i] = _host_frame(api, hosts[i], rows, k + 1, max_iter, K_net_Cov, min_images, True)
        got = bank.get_states()
    assert rcs[bad] == api.ERR_INVALID and status[bad] == api.ERR_INVALID
    assert (np.delete(status, bad) == 0).all() and (np.delete(rcs, bad) == 0).all()
    hi, ho, hP = hosts[bad].arrays()
    assert np.abs(got[0][bad] - hi).max() <= 1e-10 and np.abs(got[1][bad] - ho).max() <= 1e-10
    assert np.isnan(got[2][bad]).all() and np.isnan(hP).all()
    for i in range(n):
        if i != bad:
            _assert_state_close(api, tuple(g[i] for g in got), hosts[i], 1e-10)


@pytest.mark.gpu
def test_argument_checks_enqueue_nothing(api, wfile, frames16):
    n = 8
    cfg = api.PropagatorConfig.make(np.eye(3), np.zeros(3), True)
    lib = api.load_library()
    rng = np.random.default_rng(8)
    states = [_state(rng) for _ in range(n)]
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net, \
            api.Uahn(wfile, "prior2", precision="fp32", max_batch=n - 1) as small:
        with pytest.raises(api.UahnError, match="max_batch"):
            api.FilterBank(net, n + 1, cfg)
        with api.FilterBank(net, n, cfg) as bank:
            bank.set_states(0, [s[0] for s in states], [s[1] for s in states], [s[2] for s in states])
            before, launches = bank.get_states(), net.launch_count
            with pytest.raises(api.UahnError, match="max_batch"):
                bank.frame(frames16[0, :n], 2, iterative=small)
            assert lib.uahn_filter_frame(bank._f, None, None, 1, 10.0, 2, None, None, None, None, None, None) == api.ERR_INVALID
            assert "null frames" in lib.uahn_last_error(net._h).decode()
            masks = np.ones((n, api.MASK_BYTES_PER_PAIR), np.uint8)
            with pytest.raises(api.UahnError, match="explicit masks"):
                bank.frame(frames16[0, :n], 1, keep_masks=masks)
            assert (bank.wait() == 0).all()
            after = bank.get_states()
            assert net.launch_count == launches
            assert all(np.array_equal(a, b) for a, b in zip(before, after))
