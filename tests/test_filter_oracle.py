"""Filter bank (include/uahn_filter.h) against the numpy oracle (oracle/filter_oracle.py), which shares no code with
csrc/ekf_math.h: propagation of 1000 slots over edge schedules under two configurations, staging growth between two
propagations, updates whose innovation covariance runs up to cond 1e12, and the benchmark's 64-frame closed loop
replayed slot by slot.  The host consumer compiles the same header as the kernels, so tests/test_filter_bank.py cannot
see a mistake in it; these tests can."""
import concurrent.futures as cf
import importlib.util
import multiprocessing as mp
import os

import numpy as np
import pytest

from cuahn_vio_b200 import synthetic as Syn
from oracle import filter_oracle as F
from oracle import imu_oracle as I

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 2.0 ** -52
# bounds, about 100x the worst error seen on one B200 (the run prints the worst of each on every run)
PROP_TOL = 1e-12           # propagation: IMU / offsets x max(1, |x|), P x max|P|; worst seen 1.0e-14
LOOP_TOL = 1e-11           # closed loop on its well-posed frames, same scales; worst seen 9.4e-14
UPDATE_ULPS = 100          # updates: UPDATE_ULPS x amp x 2^-52 (amp = cond(S) for one update, filter_oracle.frame),
                           # same scales (P: the larger max|P| before and after the update); worst seen 19 (host, cond 1e12)


@pytest.fixture(scope="module")
def api():
    from cuahn_vio_b200 import build
    build.build()
    from cuahn_vio_b200 import api as a
    a.load_library()
    return a


@pytest.fixture(scope="module")
def wfile(api):
    from cuahn_vio_b200 import weights
    return weights.synthetic_weights_file(0)


def _pool_map(fn, jobs):
    """fn over jobs in spawned worker processes (numpy and the oracle only); none outlives the call."""
    workers = max(1, min(32, os.cpu_count() or 1, len(jobs)))
    with cf.ProcessPoolExecutor(max_workers=workers, mp_context=mp.get_context("spawn")) as ex:
        return list(ex.map(fn, jobs, chunksize=max(1, len(jobs) // (4 * workers))))


def _errors(got, exp, p_scale=None):
    """Worst relative errors (imu, offsets, P) of a bank state against an oracle state: IMU value and offsets per
    component against max(1, |x|), P against max|P| (or p_scale)."""
    (gi, go, gP), (ei, eo, eP) = got, exp
    rel = lambda a, b: float((np.abs(a - b) / np.maximum(1.0, np.abs(b))).max())
    scale = p_scale if p_scale is not None else max(np.abs(eP).max(), np.finfo(float).tiny)
    return rel(gi, ei), rel(go, eo), float(np.abs(gP - eP).max() / scale)


def _ulp_ok(got, exp, rel=0.0):
    """Within one float ulp, plus rel x max(1, |x|) (priors of later iterations inherit the update's error)."""
    exp = np.asarray(exp, np.float32)
    err = np.abs(np.asarray(got, np.float64) - exp)
    return bool((err <= np.spacing(np.abs(exp)) + rel * np.maximum(1.0, np.abs(exp))).all())


def _set_all(bank, states):
    bank.set_states(0, [s[0] for s in states], [s[1] for s in states], [s[2] for s in states])


def _slot(got, i):
    return tuple(g[i] for g in got)


# ---- CPU: the oracle's frame() against the host update it replays ------------------------------------------------

def _designed_block(rng, cond, scale=1e-3):
    """A random SPD 8x8 matrix of norm `scale` and condition number `cond`."""
    Q, _ = np.linalg.qr(rng.standard_normal((8, 8)))
    return scale * Q @ np.diag(np.logspace(0, -np.log10(cond), 8)) @ Q.T


MEAS_ROWS = [15, 16, 18, 19, 21, 22, 24, 25]        # ekf_math.h meas_row(): the (u, v) rows of the four offsets
ITERATED_TOL_MAX = 1e-6                             # every tolerance of a max_iter 2 comparison must be at most this


def _tolerance_report(label, stats):
    """stats[max_iter] = [worst error / (amp x 2^-52), largest tolerance, largest cond(S), comparisons]."""
    for mi, (w, tol, cond, k) in sorted(stats.items()):
        print(f"[{label}] max_iter {mi}: {k} states compared, worst error / (amp x 2^-52) = {w:.2e}, "
              f"largest tolerance {tol:.1e}, largest cond(S) {cond:.1e}")


def _record(stats, max_iter, err, tol, cond):
    s = stats.setdefault(max_iter, [0.0, 0.0, 0.0, 0])
    s[0], s[1], s[2], s[3] = max(s[0], err / tol * UPDATE_ULPS), max(s[1], tol), max(s[2], cond), s[3] + 1
    if max_iter > 1:                       # a looser bound would accept a skipped or wrong second update
        assert tol <= ITERATED_TOL_MAX, (tol, cond)


def test_frame_oracle_matches_host_update(api):
    """filter_oracle.frame against uahn_ekf_update / uahn_ekf_reset_offsets (the loop of uahn_ekf_iekf_frame), across
    the gates.  max_iter 1 with K_net_Cov 0, so S = H P H^T exactly: cond(S) 1e2 ... 1e12 (invert8 against LAPACK), and
    an exactly zero block (singular S).  max_iter 2 with Cov designed proportional to H P H^T, so that the second
    update's S stays within 4/3 of the first's: cond(S) 1e2 ... 3e3, every tolerance at most ITERATED_TOL_MAX."""
    rng = np.random.default_rng(77)
    cases = [(1, 10.0 ** k, 2 + k % 2) for k in range(2, 13)] + [(1, None, 2), (1, 1e6, 1)]
    cases += [(2, c, count) for c in (1e2, 1e3, 3e3) for count in (2, 3)] + [(2, 1e3, 1)]
    stats = {}
    lib = api.load_library()
    for max_iter, cond, count in cases:
        imu, off, P = F.initial_state(rng)
        min_images = 2                                            # count 1 -> frame 2: the gate stays closed
        T = _designed_block(rng, cond if cond else 10.0)
        # congruence on the measurement rows: P stays SPD and its measurement block becomes T
        G = np.eye(27)
        G[np.ix_(MEAS_ROWS, MEAS_ROWS)] = np.linalg.cholesky(T) @ np.linalg.inv(
            np.linalg.cholesky(P[np.ix_(MEAS_ROWS, MEAS_ROWS)]))
        P = G @ P @ G.T
        if cond is None:
            P[MEAS_ROWS, :] = 0.0
            P[:, MEAS_ROWS] = 0.0
        mean = rng.standard_normal((max_iter, 8)).astype(np.float32)
        if max_iter == 1:
            K_net_Cov = 0.0
            A = rng.standard_normal((1, 8, 8))
            cov = (A @ A.transpose(0, 2, 1)).astype(np.float32)   # multiplied by 0: S = H P H^T
        else:
            K_net_Cov = 1.0
            cov = np.stack([(25440.25 * T).astype(np.float32)] * 2)   # K_net_Cov Cov / 25440.25 = T
        r = F.frame((imu, off, P), count, mean, cov, max_iter, K_net_Cov, min_images)
        host = api.EkfState.from_arrays(imu, off, P)
        rc = 0
        for it in range(max_iter):
            px, propagated = api.ekf_prior_px(host)
            assert _ulp_ok(r["prior"][it], px, UPDATE_ULPS * r["prior_amp"][it] * EPS if it else 0.0), (cond, it)
            if count + 1 < 2 or count + 1 <= min_images:
                continue
            try:
                api.ekf_update(host, mean[it].astype(np.float64), cov[it].astype(np.float64).reshape(64), propagated,
                               it != max_iter - 1, K_net_Cov)
            except api.UahnError:
                rc = api.ERR_INVALID
                break
        if not rc:
            lib.uahn_ekf_reset_offsets(host)
        assert r["status"] == rc, (max_iter, cond, count)
        if rc:
            assert cond is None
            continue
        if not r["cond"]:
            assert count + 1 <= min_images and all(np.array_equal(a, b) for a, b in zip(host.arrays(), r["state"]))
            continue
        tol = UPDATE_ULPS * r["amp"] * EPS
        e = _errors(host.arrays(), r["state"], max(np.abs(P).max(), np.abs(r["state"][2]).max()))
        _record(stats, max_iter, max(e), tol, max(r["cond"]))
        assert max(e) <= tol, (max_iter, cond, e, tol)
    assert stats[1][2] > 1e11 and stats[2][3] >= 6           # the designed conditioning was reached; both depths ran
    _tolerance_report("frame oracle vs host", stats)


# ---- GPU -------------------------------------------------------------------------------------------------------------

def _prop_schedules(rng, n):
    """Every third slot takes the next edge schedule, the others a random bench step (500 Hz / 30 Hz)."""
    edges = F.edge_schedules(rng)
    out = []
    for i in range(n):
        if i % 3 == 0:
            out.append(edges[(i // 3) % len(edges)])
        else:
            t0 = 10.0 + 0.01 * rng.random()
            r, t0, t1 = F.bench_step(rng, t0, 0.002 * rng.random())
            out.append({"name": "random", "readings": r, "t0": t0, "t1": t1, "zero_bg": False})
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["A", "B"])
def test_propagation_matches_oracle_n1000(api, wfile, config):
    """1000 slots (several waves of one CTA per slot, not a multiple of 128): status, IMU value, offsets and P of every
    slot against the oracle; slots that must stay untouched, bit for bit."""
    n = 1000
    rng = np.random.default_rng({"A": 1000, "B": 1001}[config])
    c, p_scale = F.configs(rng)[config]
    sched = _prop_schedules(rng, n)
    states = []
    for s in sched:
        imu, off, P = F.initial_state(rng, p_scale)
        if s["zero_bg"]:
            imu[13:16] = 0.0
        states.append((imu, off, P))
    t0 = np.array([s["t0"] for s in sched])
    t1 = np.array([s["t1"] for s in sched])
    cfg = api.PropagatorConfig.make(**c)
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net, api.FilterBank(net, n, cfg) as bank:
        _set_all(bank, states)
        bank.propagate([s["readings"] for s in sched], t0, t1)
        status = bank.wait()
        got = bank.get_states()
    exp = _pool_map(F.propagate_slot, [(states[i], sched[i]["readings"], t0[i], t1[i], c) for i in range(n)])
    worst = np.zeros(3)
    for i in range(n):
        st, est, intervals, _ = exp[i]
        assert status[i] == st, (i, sched[i]["name"], status[i], st)
        if st or intervals == 0:
            assert all(np.array_equal(a, b) for a, b in zip(_slot(got, i), states[i])), (i, sched[i]["name"])
            continue
        e = np.array(_errors(_slot(got, i), est))
        worst = np.maximum(worst, e)
        assert (e <= PROP_TOL).all(), (i, sched[i]["name"], e)
    assert (status == F.ERR_STATE).sum() == sum(s["name"] in ("t1_eq_t0", "t1_lt_t0", "t1_nan") for s in sched) > 0
    print(f"[propagation n=1000 {config}] worst relative error: imu {worst[0]:.1e}, offsets {worst[1]:.1e}, P {worst[2]:.1e}")


@pytest.mark.gpu
def test_staging_growth_between_propagations(api, wfile):
    """Two propagations enqueued without a wait; the second selects more than 1.5x the first's readings, so
    ensure_samples reallocates the staging while the first may still be in flight.  Equal to two oracle propagations."""
    n = 64
    rng = np.random.default_rng(64)
    c, p_scale = F.configs(rng)["A"]
    states = [F.initial_state(rng, p_scale) for _ in range(n)]
    phase = 0.002 * rng.random(n)
    first = [F.bench_step(rng, 10.0 + phase[i], phase[i]) for i in range(n)]
    second = [F.bench_step(rng, first[i][2], phase[i], 0.5) for i in range(n)]
    bound = lambda steps: sum(len(s[0]) + 2 for s in steps)         # uahn_filter_propagate's staging bound
    assert bound(second) > bound(first) + bound(first) // 2 + 64      # ensure_samples' capacity after the first call
    cfg = api.PropagatorConfig.make(**c)
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net, api.FilterBank(net, n, cfg) as bank:
        _set_all(bank, states)
        for steps in (first, second):
            bank.propagate([s[0] for s in steps], [s[1] for s in steps], [s[2] for s in steps])
        status = bank.wait()
        got = bank.get_states()
    assert (status == 0).all()
    mid = _pool_map(F.propagate_slot, [(states[i], *first[i], c) for i in range(n)])
    exp = _pool_map(F.propagate_slot, [(mid[i][1], *second[i], c) for i in range(n)])
    worst = 0.0
    for i in range(n):
        e = _errors(_slot(got, i), exp[i][1])
        worst = max(worst, max(e))
        assert max(e) <= PROP_TOL, (i, e)
    print(f"[staging growth] worst relative error {worst:.1e}")


def _designed_state(rng, c, readings, t0, t1, cond):
    """A state whose measurement block of P, after frame 0's offset reset and one propagation interval over
    `readings`, is a random SPD matrix of condition number `cond` (None: exactly zero, the readings then being empty).
    After the reset P keeps only its IMU block P15, and one interval maps it to A P15 A^T with A = H F[:, :15]; P15 =
    A^+ T A^+T gives T (the process noise of the offset rows is made negligible by the configuration's sigma_w)."""
    imu, off, _ = F.initial_state(rng)
    P = np.zeros((27, 27))
    if cond is not None:
        prop = I.select_imu_readings(readings, t0, t1)
        assert len(prop) == 2
        _, _, Fm, _ = I.predict_and_compute(imu, np.zeros((4, 3)), np.asarray(c["c_R_i"]).reshape(3, 3),
                                            np.asarray(c["i_t_i2c"]), prop[0], prop[1], bool(c["imu_avg"]))
        A = F.E.measurement_jacobian() @ Fm[:, :15]
        T = _designed_block(rng, cond)
        Ap = np.linalg.pinv(A)
        P15 = Ap @ T @ Ap.T
        P[:15, :15] = 0.5 * (P15 + P15.T)
    return imu, off, P


@pytest.mark.gpu
def test_updates_at_the_conditioning_edges(api, wfile):
    """One update (max_iter 1) with cond(H P H^T) designed from 1e2 to 1e12: K_net_Cov = 1e-9 (S ~ H P H^T) and 0 (S =
    H P H^T; one slot's block is exactly zero, so ERR_INVALID exactly where LAPACK finds S singular), each within
    UPDATE_ULPS x cond(S) x 2^-52; K_net_Cov = 1e18, where nothing may move.  Two updates (max_iter 2, a prior2 h_iter)
    at K_net_Cov = 1000, where the network's Cov term dominates S and the second update is as well posed as the first:
    every tolerance at most ITERATED_TOL_MAX.  (With a measurement noise far below H P H^T the second update's S is the
    cancellation remnant of the first's, and no bound can hold it; the test_filter_bank / closed-loop tests run max_iter
    2 at working conditions.)  Each against ekf_oracle.update fed the bank's own state and network rows."""
    conds = [10.0 ** k for k in range(2, 13)]
    slot_conds = conds + conds + [None]                               # the last slot: an exactly zero block
    n = len(slot_conds)
    rng = np.random.default_rng(12)
    c = {"c_R_i": F.rotation(rng, 0.1)[0], "i_t_i2c": 0.05 * rng.standard_normal(3), "imu_avg": 1, "sigma_w": 1e-12}
    t0, t1 = 10.0, 10.0 + 1.0 / F.HZ_CAM
    one = [F.reading(rng, t0 - 0.001), F.reading(rng, t1 + 0.001), F.reading(rng, t1 + 0.003)]   # one interval
    readings = [one if sc is not None else [] for sc in slot_conds]
    states = [_designed_state(rng, c, one, t0, t1, sc) for sc in slot_conds]
    prev, curr, _, _ = Syn.tiled_batch(n, unique=8)
    stats = {}
    cfg = api.PropagatorConfig.make(**c)
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net, \
            api.Uahn(wfile, "prior2", precision="fp32", max_batch=n) as net2, api.FilterBank(net, n, cfg) as bank:
        for K_net_Cov, max_iter in ((1e-9, 1), (0.0, 1), (1e18, 1), (1000.0, 2)):
            _set_all(bank, states)
            bank.frame(prev, 1, K_net_Cov, 0, seed=3, first_pair=0)   # frame 1 of every slot: no update, offsets reset
            assert (bank.wait() == 0).all()
            bank.propagate(readings, np.full(n, t0), np.full(n, t1))
            assert (bank.wait() == 0).all()
            pre = bank.get_states()
            out = bank.frame(curr, max_iter, K_net_Cov, 0, seed=3, first_pair=n, iterative=net2)
            status = bank.wait()
            post = bank.get_states()
            for i in range(n):
                r = F.frame(_slot(pre, i), 1, out["mean"][:, i], out["cov"][:, i], max_iter, K_net_Cov, 0)
                assert status[i] == r["status"], (K_net_Cov, max_iter, i, status[i], r["status"])
                for it in range(max_iter):                           # prior[it] inherits the updates before it only
                    assert _ulp_ok(out["prior"][it, i], r["prior"][it], UPDATE_ULPS * r["prior_amp"][it] * EPS if it else 0.0), \
                        (K_net_Cov, max_iter, i, it)
                if r["status"]:
                    assert slot_conds[i] is None and K_net_Cov == 0.0
                    assert all(np.array_equal(a, b) for a, b in zip(_slot(post, i), _slot(pre, i)))   # stopped, no reset
                    continue
                tol = UPDATE_ULPS * r["amp"] * EPS
                e = _errors(_slot(post, i), r["state"], max(np.abs(pre[2][i]).max(), np.abs(r["state"][2]).max()))
                if K_net_Cov < 1 or max_iter > 1:
                    _record(stats, max_iter, max(e), tol, max(r["cond"]))
                assert max(e) <= tol, (K_net_Cov, max_iter, i, slot_conds[i], r["cond"], e, tol)
                if K_net_Cov == 1e18:                                 # K ~ 1e-14: the IMU value and P15 stay
                    assert np.abs(post[0][i] - pre[0][i]).max() <= 1e-12
                    assert np.abs(post[2][i][:15, :15] - pre[2][i][:15, :15]).max() <= 1e-12 * np.abs(pre[2][i]).max()
            if K_net_Cov == 0.0:
                assert status[n - 1] == api.ERR_INVALID and (status[:n - 1] == 0).all()
    assert stats[1][2] > 1e11 and stats[2][3] == n                   # the designed conditioning was reached; both depths ran
    _tolerance_report("updates", stats)


def _bench_module():
    spec = importlib.util.spec_from_file_location("filter_bench", os.path.join(ROOT, "tools", "filter_bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _closed_loop(api, wfile, n, n_frames, max_iter):
    """tools/filter_bench.py's closed loop (same seeds, states, IMU steps, frames, configuration, K_net_Cov and
    min_images) over n slots; after every frame the status, priors, network rows and full states are recorded, then
    every slot is replayed through filter_oracle with the bank's network rows.  → (records, replays)."""
    fb = _bench_module()
    lib = api.load_library()
    rng = np.random.default_rng(n)
    prev_u, curr_u, _, _ = Syn.tiled_batch(n, unique=64)
    frames = [prev_u, curr_u]
    steps = fb.imu_steps(n, n_frames, rng)
    imu0, off0, P0 = fb.initial_states(api, n, rng)
    c = {"c_R_i": np.eye(3), "i_t_i2c": np.array([0.0, 0.0, 0.05]), "imu_avg": 1}
    rec = {"status": [], "prior": [], "mean": [], "cov": [], "states": []}
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net, \
            api.Uahn(wfile, "prior2", precision="bf16", max_batch=n) as net2, \
            api.FilterBank(net, n, api.PropagatorConfig.make(**c)) as bank:
        bank.set_states(0, imu0, off0, P0)
        for k in range(n_frames):
            r, offsets, t0, t1 = steps[k]
            if k:
                assert lib.uahn_filter_propagate(bank._f, r.ctypes.data, offsets.ctypes.data, t0.ctypes.data,
                                                 t1.ctypes.data) == 0
            out = bank.frame(frames[k % 2], max_iter, fb.K_NET_COV, 2, iterative=net2 if max_iter > 1 else None)
            rec["status"].append(bank.wait())
            for key in ("prior", "mean", "cov"):
                rec[key].append(out[key])
            rec["states"].append(bank.get_states())

    def slot_steps(i):
        out = [None]
        for r, offsets, t0, t1 in steps[1:]:
            out.append(([(float(x["t"]), x["wm"].copy(), x["am"].copy()) for x in r[offsets[i]:offsets[i + 1]]],
                        float(t0[i]), float(t1[i])))
        return out

    jobs = [{"state": (imu0[i], off0[i], P0[i]), "cfg": c, "steps": slot_steps(i),
             "mean": [rec["mean"][k][:, i] for k in range(n_frames)], "cov": [rec["cov"][k][:, i] for k in range(n_frames)],
             "max_iter": max_iter, "K_net_Cov": fb.K_NET_COV, "min_images": 2, "use": True} for i in range(n)]
    return rec, _pool_map(F.replay_slot, jobs)


def _check_closed_loop(rec, replays, label):
    """Per slot: priors within one float ulp and states within LOOP_TOL on every frame before the oracle's first
    ill-posed one (|dc| < PLANE_MIN or cond(S) > COND_MAX); the bank's failure frame equal to the oracle's, or, where
    the error amplification near divergence makes it unstable, between the first ill-posed frame and the oracle's
    failure frame (each such case printed).  → per-slot (bank failure frame, oracle failure frame)."""
    n_frames, n = len(rec["status"]), len(replays)
    worst, fails, compared = np.zeros(3), [], 0
    for i, rp in enumerate(replays):
        ill = next((k for k, f in enumerate(rp) if f["min_dc"] < F.PLANE_MIN or max(f["cond"], default=0.0) > F.COND_MAX),
                   n_frames)
        o_fail = next((k for k, f in enumerate(rp) if f["status"]), None)
        b_fail = next((k for k in range(n_frames) if rec["status"][k][i]), None)
        for k in range(min(ill, len(rp) if o_fail is None else o_fail)):
            assert _ulp_ok(rec["prior"][k][:, i], rp[k]["prior"]), (label, i, k)
            e = np.array(_errors(_slot(rec["states"][k], i), rp[k]["state"]))
            worst = np.maximum(worst, e)
            compared += 1
            assert (e <= LOOP_TOL).all(), (label, i, k, e)
        if b_fail is not None:
            assert rec["status"][b_fail][i] == F.ERR_INVALID
        if b_fail != o_fail:
            lo, hi = ill, n_frames if o_fail is None else o_fail
            print(f"[{label}] slot {i}: bank fails at frame {b_fail}, oracle at {o_fail}, first ill-posed frame {ill}")
            assert b_fail is not None and lo <= b_fail <= hi, (label, i, b_fail, o_fail, ill)
        if b_fail is not None or o_fail is not None:
            last = len(rp) if o_fail is None else o_fail + 1
            fails.append((i, b_fail, o_fail, ill, min(f["min_dc"] for f in rp[:last]),
                          max((c for f in rp[:last] for c in f["cond"]), default=0.0)))
    print(f"[{label}] {compared} well-posed slot-frames compared; worst relative error: imu {worst[0]:.1e}, "
          f"offsets {worst[1]:.1e}, P {worst[2]:.1e}")
    print(f"[{label}] {len(fails)} of {n} slots fail (slot, bank frame, oracle frame, first ill-posed frame, "
          f"min |dc| up to the failure, max cond(S)): " + ", ".join(f"({a}, {b}, {c}, {d}, {e:.1e}, {g:.1e})"
                                                                    for a, b, c, d, e, g in fails))
    return fails


@pytest.mark.gpu
def test_bench_closed_loop_matches_oracle_replay(api, wfile):
    """The benchmark's loop: bf16 prior3, 136 slots (a partial second begin-kernel CTA), 64 frames, max_iter 1,
    K_net_Cov 1000, min_images 2."""
    rec, replays = _closed_loop(api, wfile, 136, 64, 1)
    fails = _check_closed_loop(rec, replays, "bench loop n=136")
    # every slot that fails, in the bank and in the oracle alike, first becomes ill-posed by its plane distance
    assert all(ill <= o and dc < F.PLANE_MIN for _, _, o, ill, dc, _ in fails if o is not None)


@pytest.mark.gpu
def test_iterated_closed_loop_matches_oracle_replay(api, wfile):
    """max_iter 2 with a prior2 h_iter, 40 slots, 24 frames."""
    rec, replays = _closed_loop(api, wfile, 40, 24, 2)
    _check_closed_loop(rec, replays, "iterated loop n=40")
