"""Filter bank with raw camera frames (uahn_filter_set_undistort_maps / _frame_raw / _stage_undistort): n frames undistorted
by one batched remap kernel, bit for bit cv::remap, feeding the same closed loop as pre-undistorted frames."""
import os
import re
import subprocess

import numpy as np
import pytest

from cuahn_vio_b200 import synthetic as S
from oracle import preproc_oracle as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAMS = ["uzhfpv_indoor_fwd", "uzhfpv_outdoor_45", "radtan_test"]
HZ_IMU, HZ_CAM = 500.0, 30.0


@pytest.fixture(scope="module")
def api():
    from cuahn_vio_b200 import build
    build.build()
    from cuahn_vio_b200 import api as a
    a.load_library()
    return a


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "preproc.npz"))


@pytest.fixture(scope="module")
def raw(golden):
    f = S.synthetic_raw_frame(int(golden["raw_seed"]))
    assert int(f.astype(np.int64).sum()) == int(golden["raw_checksum"])
    return f


def _maps(api, golden, name):
    """The library's host maps, patched where the fixture recorded a difference from OpenCV's."""
    m = api.undistort_init_maps(bool(golden[f"{name}_fisheye"]), golden[f"{name}_k"], golden[f"{name}_d"])
    out = []
    for tag, a in zip(("m1", "m2"), m):
        a = a.copy().ravel()
        a[golden[f"{name}_{tag}_diff_idx"]] = golden[f"{name}_{tag}_diff_val"]
        out.append(a.reshape(224, 320))
    return out


# ---- CPU --------------------------------------------------------------------------------------------------------

def test_remap_kernel_does_not_spill(api):
    from cuahn_vio_b200 import build
    src = os.path.join(build.CSRC, "image_kernels.cu")
    out = subprocess.run([build.NVCC, *build.FLAGS, "-Xptxas=-v", "-c", src, "-o", os.devnull],
                         capture_output=True, text=True, check=True).stderr
    blocks = re.split(r"Compiling entry function '", out)
    remap = [b for b in blocks if "remap_bilinear_u8_kernel" in b.split("'")[0]]
    assert len(remap) == 1, out                                 # one remap kernel serves every frame count
    m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", remap[0])
    assert m and m.groups() == ("0", "0"), remap[0]


# ---- GPU --------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def wfile(api):
    from cuahn_vio_b200 import weights
    return weights.synthetic_weights_file(0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CAMS)
def test_bank_undistort_bit_exact(api, wfile, golden, raw, name):
    n = 37
    c1, c2 = _maps(api, golden, name)
    cfg = api.PropagatorConfig.make(np.eye(3), np.zeros(3), True)
    same = np.broadcast_to(raw, (n,) + raw.shape)
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net, api.FilterBank(net, n, cfg) as bank:
        bank.set_undistort_maps(480, 640, c1, c2)
        assert (bank.stage_undistort(same) == golden[f"{name}_remap"][None]).all()
        bank.set_undistort_maps(480, 640, c1 + np.float32(200.0), c2 - np.float32(150.0))
        assert (bank.stage_undistort(same) == golden[f"{name}_remap_shifted"][None]).all()
        padded = np.zeros((n, 480, 700), np.uint8)
        padded[:, :, :640] = raw
        view = padded[:, :, :640]
        assert view.strides[1] == 700                           # passed as is: row stride > cols
        assert (bank.stage_undistort(view) == golden[f"{name}_remap_shifted"][None]).all()
        # a different frame in every slot: slot / row-stride indexing errors show up here and not with identical frames
        rolled = np.stack([np.roll(raw, (5 * i, 11 * i), axis=(0, 1)) for i in range(n)])
        padded[:, :, :640] = rolled
        bank.set_undistort_maps(480, 640, c1, c2)
        got = bank.stage_undistort(view)
        for i in range(n):
            assert np.array_equal(got[i], P.remap_bilinear_u8(rolled[i], c1, c2)), i


def _state(rng):
    q = np.concatenate([[1.0], 0.1 * rng.standard_normal(3)])
    q /= np.linalg.norm(q)
    imu = np.concatenate([[0.3, -0.2, 1.5] + 0.1 * rng.standard_normal(3), q, 0.5 * rng.standard_normal(3),
                          0.02 * rng.standard_normal(3), 0.005 * rng.standard_normal(3)])
    A = rng.standard_normal((27, 27))
    return imu, 0.02 * rng.standard_normal((4, 3)), 1e-4 * (A @ A.T) / 27 + 1e-6 * np.eye(27)


def _readings(rng, t0, t1, phase):
    k0, k1 = int(np.floor((t0 - phase) * HZ_IMU)) - 1, int(np.ceil((t1 - phase) * HZ_IMU)) + 1
    return [(phase + k / HZ_IMU, 0.3 * rng.standard_normal(3), np.array([0, 0, 9.81]) + 0.5 * rng.standard_normal(3))
            for k in range(k0, k1 + 1)]


N_SLOTS, N_FRAMES, MID_FRAME = 16, 6, 3


@pytest.fixture(scope="module")
def sequence(api, golden, raw):
    """Raw frames [frame][slot] (each slot a shifted copy of the fixture frame, moving from frame to frame), their
    host remaps, the maps, and the IMU readings between frames."""
    c1, c2 = _maps(api, golden, CAMS[0])
    raws = np.stack([np.stack([np.roll(raw, (3 * i + 2 * k, 7 * i + 5 * k), axis=(0, 1)) for i in range(N_SLOTS)])
                     for k in range(N_FRAMES)])
    und = np.stack([np.stack([P.remap_bilinear_u8(f, c1, c2) for f in fk]) for fk in raws])
    rng = np.random.default_rng(61)
    states = [_state(rng) for _ in range(N_SLOTS)]
    q = np.concatenate([[1.0], 0.1 * rng.standard_normal(3)])
    from oracle import imu_oracle as I
    cfg_args = (I.ham_quat_2_rot(q / np.linalg.norm(q)), 0.05 * rng.standard_normal(3))
    phase = 0.002 * rng.random(N_SLOTS)
    steps = []
    for k in range(1, N_FRAMES):
        t0 = 10.0 + (k - 1) / HZ_CAM + phase
        t1 = t0 + 1.0 / HZ_CAM
        steps.append(([_readings(rng, t0[i], t1[i], phase[i]) for i in range(N_SLOTS)], t0, t1))
    return {"maps": (c1, c2), "raw": raws, "und": und, "states": states, "cfg": cfg_args, "steps": steps}


def _run(api, wfile, seq, precision, max_iter, mode):
    """The closed loop over the sequence.  mode: "frame" (pre-undistorted frames, wait per frame), "raw" (frame_raw, one
    frame through frame() in the middle, wait per frame), "raw_nowait" (frame_raw from pinned buffers, one wait at the end).
    → per-frame outputs, final states."""
    import torch
    n = N_SLOTS
    K_net_Cov, min_images, seed = 10.0, 2, 7
    use = np.ones(n, np.uint8)
    use[3] = 0
    cfg = api.PropagatorConfig.make(*seq["cfg"], True)
    net = api.Uahn(wfile, "prior3", precision=precision, max_batch=n)
    net_iter = api.Uahn(wfile, "prior2", precision=precision, max_batch=n) if max_iter > 1 else None
    outs = []
    with net, api.FilterBank(net, n, cfg) as bank:
        st = seq["states"]
        bank.set_states(0, [s[0] for s in st], [s[1] for s in st], [s[2] for s in st])
        if mode != "frame":
            bank.set_undistort_maps(480, 640, *seq["maps"])
        for k in range(N_FRAMES):
            if k > 0:
                bank.propagate(*seq["steps"][k - 1])
            kw = dict(max_iter=max_iter, K_net_Cov=K_net_Cov, min_images=min_images, use_measurement=use, seed=seed,
                      first_pair=1000 + k * max_iter * n, iterative=net_iter)
            if mode == "frame" or (mode == "raw" and k == MID_FRAME):
                outs.append(bank.frame(seq["und"][k], **kw))
            elif mode == "raw":
                outs.append(bank.frame_raw(seq["raw"][k], **kw))
            else:
                buf = torch.empty(seq["raw"][k].shape, dtype=torch.uint8, pin_memory=True).numpy()
                buf[:] = seq["raw"][k]
                outs.append(bank.frame_raw(buf, **kw))      # the bank keeps buf alive until wait()
            if mode != "raw_nowait":
                assert (bank.wait() == 0).all()
        if mode == "raw_nowait":
            assert (bank.wait() == 0).all()
        got = bank.get_states()
    if net_iter is not None:
        net_iter.close()
    return outs, got


def _assert_runs_equal(a, b):
    (oa, sa), (ob, sb) = a, b
    for k, (x, y) in enumerate(zip(oa, ob)):
        for key in ("prior", "mean", "cov", "imu"):
            np.testing.assert_array_equal(x[key], y[key], err_msg=f"frame {k} {key}")
    for x, y in zip(sa, sb):
        np.testing.assert_array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("precision,max_iter", [("fp32", 1), ("fp32", 2), ("bf16", 1), ("bf16", 2)])
def test_raw_closed_loop_matches_undistorted_bank(api, wfile, sequence, precision, max_iter):
    ref = _run(api, wfile, sequence, precision, max_iter, "frame")
    raw_run = _run(api, wfile, sequence, precision, max_iter, "raw")
    _assert_runs_equal(raw_run, ref)
    assert not np.array_equal(ref[0][1]["mean"], ref[0][2]["mean"])   # the frames move: the outputs do too


@pytest.mark.gpu
def test_raw_frames_overlap_safely(api, wfile, sequence):
    """Six frame_raw calls enqueued back to back: the uploads of frames k and k + 2 share a staging buffer."""
    ref = _run(api, wfile, sequence, "bf16", 2, "frame")
    _assert_runs_equal(_run(api, wfile, sequence, "bf16", 2, "raw_nowait"), ref)


@pytest.mark.gpu
def test_raw_argument_checks_enqueue_nothing(api, wfile, golden, raw):
    n = 8
    lib = api.load_library()
    c1, c2 = _maps(api, golden, CAMS[2])
    cfg = api.PropagatorConfig.make(np.eye(3), np.zeros(3), True)
    rng = np.random.default_rng(9)
    states = [_state(rng) for _ in range(n)]
    frames = np.ascontiguousarray(np.broadcast_to(raw, (n,) + raw.shape))
    out = np.empty((n, 224, 320), np.uint8)

    def frame_raw(ptr, stride):
        return lib.uahn_filter_frame_raw(bank._f, None, ptr, stride, 1, 10.0, 2, None, None, None, None, None, None)

    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net, api.FilterBank(net, n, cfg) as bank:
        bank.set_states(0, [s[0] for s in states], [s[1] for s in states], [s[2] for s in states])
        before, launches = bank.get_states(), net.launch_count

        def error():
            return lib.uahn_last_error(net._h).decode()
        assert frame_raw(api._ptr(frames), 640) == api.ERR_STATE and "set_undistort_maps" in error()
        assert lib.uahn_filter_stage_undistort(bank._f, api._ptr(frames), 640, api._ptr(out)) == api.ERR_STATE
        for rows, cols in ((0, 640), (480, 40000), (40000, 640), (480, 0)):
            assert lib.uahn_filter_set_undistort_maps(bank._f, rows, cols, api._ptr(c1), api._ptr(c2)) == api.ERR_INVALID
            assert f"raw size {rows}x{cols}" in error()
        assert frame_raw(api._ptr(frames), 640) == api.ERR_STATE  # failed set_undistort_maps calls set no maps
        bank.set_undistort_maps(480, 640, c1, c2)
        assert frame_raw(None, 640) == api.ERR_INVALID and "null raw" in error()
        assert frame_raw(api._ptr(frames), 639) == api.ERR_INVALID and "stride 639" in error()
        assert lib.uahn_filter_stage_undistort(bank._f, api._ptr(frames), 639, api._ptr(out)) == api.ERR_INVALID
        assert lib.uahn_filter_set_undistort_maps(bank._f, 480, 40000, api._ptr(c1), api._ptr(c2)) == api.ERR_INVALID
        assert (bank.wait() == 0).all()
        assert net.launch_count == launches
        assert all(np.array_equal(a, b) for a, b in zip(before, bank.get_states()))
        # the maps set before the failed call are still in place
        assert (bank.stage_undistort(frames) == P.remap_bilinear_u8(raw, c1, c2)[None]).all()
