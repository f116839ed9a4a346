"""uahn_submit_sequence_raw: the pipelined sequence entry point fed raw camera frames, undistorted on the device by the
batched remap kernel, bit for bit what uahn_submit_sequence computes from the same frames remapped on the host."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from cuahn_vio_b200 import synthetic as S
from oracle import preproc_oracle as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAMS = ["uzhfpv_indoor_fwd", "uzhfpv_outdoor_45", "radtan_test"]
# both sides of every batch-size kernel switch (latency path <= 8, texture warp > 8, fused MC GEMM >= 64) and max_batch;
# the remap kernel takes 8 frames per CTA row, so n + 1 frames is a multiple of 8 only at 63
PAIRS = [1, 8, 9, 63, 64, 300, 1024]
PADDED = {9, 300}                # pair counts submitted with a 700-byte row stride
MAX_BATCH = max(PAIRS)


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


def _shifted(frame, count, start=0):
    """count shifted copies of one raw frame: the scene moves by (2, 3) px per frame."""
    return np.stack([np.roll(frame, (2 * k, 3 * k), axis=(0, 1)) for k in range(start, start + count)])


def _remap(frames, maps):
    return np.stack([P.remap_bilinear_u8(f, *maps) for f in frames])


def _priors(n, seed):
    return (2.0 * np.random.default_rng(seed).standard_normal((n, 8))).astype(np.float32)


def _pinned(a):
    import torch
    t = torch.empty(a.shape, dtype=torch.uint8 if a.dtype == np.uint8 else torch.float32, pin_memory=True)
    out = t.numpy()
    out[:] = a
    return out


def _submit_undistorted(net, frames, prior, seed, first_pair):
    """uahn_submit_sequence on host frames → (mean, cov) once the handle has been waited on."""
    n = frames.shape[0] - 1
    frames, prior = np.ascontiguousarray(frames), np.ascontiguousarray(prior, np.float32)
    mean, cov = np.empty((n, 8), np.float32), np.empty((n, 8, 8), np.float32)
    net.submit_sequence_ptrs(n + 1, frames.ctypes.data, prior.ctypes.data, mean.ctypes.data, cov.ctypes.data, seed=seed,
                             first_pair=first_pair)
    return mean, cov, (frames, prior)


# ---- CPU --------------------------------------------------------------------------------------------------------

def test_symbol_exported_and_binding_matches_header(api):
    lib = api.load_library()
    assert "uahn_submit_sequence_raw" in api.PREPROC_SYMBOLS and hasattr(lib, "uahn_submit_sequence_raw")
    hdr = open(os.path.join(ROOT, "include", "uahn_preproc.h")).read()
    m = re.search(r"UAHN_API int uahn_submit_sequence_raw\(([^)]*)\);", hdr)
    assert m, "prototype not found"
    ctype = {"uahn_handle*": C.c_void_p, "int": C.c_int, "const uint8_t*": C.c_void_p, "size_t": C.c_size_t,
             "const float*": C.c_void_p, "const uahn_rng*": C.POINTER(api._Rng), "float*": C.c_void_p}
    params = [" ".join(p.split()).rsplit(" ", 1)[0] for p in m.group(1).split(",")]
    assert list(lib.uahn_submit_sequence_raw.argtypes) == [ctype[p] for p in params], params
    assert lib.uahn_submit_sequence_raw.restype is C.c_int


# ---- GPU --------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def wfile(api):
    from cuahn_vio_b200 import weights
    return weights.synthetic_weights_file(0)


@pytest.fixture(scope="module")
def sequence(raw):
    return _shifted(raw, MAX_BATCH + 1)


@pytest.fixture(scope="module")
def remapped(api, golden, sequence):
    """Per camera: the maps and the host remap of the whole sequence (computed once)."""
    cache = {}

    def get(name):
        if name not in cache:
            maps = _maps(api, golden, name)
            cache[name] = (maps, _remap(sequence, maps))
        return cache[name]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("cam", CAMS)
def test_raw_sequence_matches_host_remapped(api, wfile, sequence, remapped, precision, cam):
    maps, und = remapped(cam)
    prior = _priors(MAX_BATCH, 5)
    with api.Uahn(wfile, "prior3", precision=precision, max_batch=MAX_BATCH) as net, \
            api.Uahn(wfile, "prior3", precision=precision, max_batch=MAX_BATCH) as ref:
        net.set_undistort_maps(480, 640, *maps)
        for n in PAIRS:
            frames = sequence[:n + 1]
            if n in PADDED:
                padded = np.zeros((n + 1, 480, 700), np.uint8)
                padded[:, :, :640] = frames
                frames = padded[:, :, :640]
                assert frames.strides[1] == 700                 # passed as is: row stride > cols
            m, c = net.submit_sequence_raw(frames, prior[:n], seed=3, first_pair=17 + n)
            rm, rc, _ = _submit_undistorted(ref, und[:n + 1], prior[:n], 3, 17 + n)
            net.wait()
            ref.wait()
            np.testing.assert_array_equal(m, rm, err_msg=f"{n} pairs: mean")
            np.testing.assert_array_equal(c, rc, err_msg=f"{n} pairs: cov")
            assert np.isfinite(m).all() and np.abs(m).max() > 0
            if n > 1:
                assert not np.array_equal(m[0], m[1])           # the frames move: so do the outputs


N_OVERLAP, K_OVERLAP = 64, 6


@pytest.mark.gpu
def test_unwaited_raw_submissions_overlap_safely(api, wfile, raw, remapped):
    """Six raw submissions from six pinned buffers without a wait (submissions k and k + 2 share a staging set) ==
    the same six with a wait after each; so do raw and pre-undistorted submissions alternating on one handle."""
    maps, _ = remapped(CAMS[0])
    n = N_OVERLAP
    raws = [_pinned(_shifted(raw, n + 1, start=40 * i)) for i in range(K_OVERLAP)]
    unds = [_pinned(_remap(r, maps)) for r in raws]
    priors = [_pinned(_priors(n, 20 + i)) for i in range(K_OVERLAP)]

    def run(net, wait_each, alternate):
        outs = []
        for i in range(K_OVERLAP):
            m, c = _pinned(np.zeros((n, 8), np.float32)), _pinned(np.zeros((n, 64), np.float32))
            if alternate and i % 2:
                net.submit_sequence_ptrs(n + 1, unds[i].ctypes.data, priors[i].ctypes.data, m.ctypes.data, c.ctypes.data,
                                         seed=9, first_pair=1000 * i)
            else:
                net.submit_sequence_raw_ptrs(n + 1, raws[i].ctypes.data, 640, priors[i].ctypes.data, m.ctypes.data,
                                             c.ctypes.data, seed=9, first_pair=1000 * i)
            if wait_each:
                net.wait()
            outs.append((m, c))
        net.wait()
        return outs

    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net:
        net.set_undistort_maps(480, 640, *maps)
        ref = run(net, True, False)
        for alternate in (False, True):
            got = run(net, False, alternate)
            for i, ((m, c), (rm, rc)) in enumerate(zip(got, ref)):
                np.testing.assert_array_equal(m, rm, err_msg=f"alternate={alternate} submission {i}: mean")
                np.testing.assert_array_equal(c, rc, err_msg=f"alternate={alternate} submission {i}: cov")
    assert not np.array_equal(ref[0][0], ref[1][0])


@pytest.mark.gpu
def test_map_replacement_waits_for_submissions_in_flight(api, wfile, golden, raw, remapped):
    """uahn_set_undistort_maps right after an unwaited raw submission: that submission keeps the old maps, the next one
    uses the new maps; a larger raw size after that reallocates the staging between submissions."""
    n = 20
    maps_a, _ = remapped(CAMS[0])
    maps_b = _maps(api, golden, CAMS[2])
    big = S.synthetic_raw_frame(int(golden["raw_seed"]) + 1, rows=512, cols=704)
    steps = [((480, 640), maps_a, _pinned(_shifted(raw, n + 1))),
             ((480, 640), maps_b, _pinned(_shifted(raw, n + 1, start=7))),
             ((512, 704), maps_a, _pinned(_shifted(big, n + 1, start=3)))]
    prior = _pinned(_priors(n, 31))
    with api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as net, \
            api.Uahn(wfile, "prior3", precision="bf16", max_batch=n) as ref:
        outs = []
        for i, ((rows, cols), maps, frames) in enumerate(steps):
            net.set_undistort_maps(rows, cols, *maps)           # no wait since the previous submission
            m, c = _pinned(np.zeros((n, 8), np.float32)), _pinned(np.zeros((n, 64), np.float32))
            net.submit_sequence_raw_ptrs(n + 1, frames.ctypes.data, cols, prior.ctypes.data, m.ctypes.data, c.ctypes.data,
                                         seed=2, first_pair=50 * i)
            outs.append((m, c))
        net.wait()
        for i, ((_, maps, frames), (m, c)) in enumerate(zip(steps, outs)):
            rm, rc, _ = _submit_undistorted(ref, _remap(frames, maps), prior, 2, 50 * i)
            ref.wait()
            np.testing.assert_array_equal(m, rm, err_msg=f"submission {i}: mean")
            np.testing.assert_array_equal(c.reshape(n, 8, 8), rc, err_msg=f"submission {i}: cov")
        wrong, _, _ = _submit_undistorted(ref, _remap(steps[0][2], maps_b), prior, 2, 0)
        ref.wait()
        assert not np.array_equal(outs[0][0], wrong)            # the maps matter


@pytest.mark.gpu
def test_argument_checks_enqueue_nothing(api, wfile, raw, remapped):
    n = 9
    lib = api.load_library()
    maps, _ = remapped(CAMS[2])
    frames = _pinned(_shifted(raw, n + 2))                      # one frame more than max_batch + 1
    prior = _pinned(_priors(n + 1, 4))
    mean, cov = np.zeros((n + 1, 8), np.float32), np.zeros((n + 1, 64), np.float32)
    masks = np.zeros(api.MASK_BYTES_PER_PAIR, np.uint8)

    def call(net, n_frames=n + 1, raw_p=frames.ctypes.data, stride=640, prior_p=prior.ctypes.data, mean_p=mean.ctypes.data,
             cov_p=cov.ctypes.data, keep=None):
        rng = api._Rng(6, 70, None if keep is None else keep.ctypes.data)
        return lib.uahn_submit_sequence_raw(net._h, n_frames, api._ptr(raw_p), stride, api._ptr(prior_p), C.byref(rng),
                                            api._ptr(mean_p), api._ptr(cov_p))

    def valid(net):
        m, c = _pinned(np.zeros((n, 8), np.float32)), _pinned(np.zeros((n, 64), np.float32))
        assert call(net, mean_p=m.ctypes.data, cov_p=c.ctypes.data) == 0
        net.wait()
        return m, c

    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as net:
        launches = net.launch_count

        def check(rc, expected, words):
            assert rc == expected, (rc, expected, words)
            assert words in lib.uahn_last_error(net._h).decode(), (words, lib.uahn_last_error(net._h))
        check(call(net), api.ERR_STATE, "set_undistort_maps")
        net.set_undistort_maps(480, 640, *maps)
        check(call(net, raw_p=None), api.ERR_INVALID, "null buffer")
        check(call(net, mean_p=None), api.ERR_INVALID, "null buffer")
        check(call(net, cov_p=None), api.ERR_INVALID, "null buffer")
        check(call(net, n_frames=1), api.ERR_STATE, "Only has one image")
        check(call(net, n_frames=0), api.ERR_STATE, "Only has one image")
        check(call(net, n_frames=n + 2), api.ERR_INVALID, f"max_batch={n}")
        check(call(net, keep=masks), api.ERR_UNSUPPORTED, "explicit masks")
        check(call(net, prior_p=None), api.ERR_INVALID, "needs a prior")
        check(call(net, stride=639), api.ERR_INVALID, "stride 639")
        check(call(net, stride=2 ** 31), api.ERR_INVALID, f"stride {2 ** 31}")
        net.wait()
        assert net.launch_count == launches
        got = valid(net)
    with api.Uahn(wfile, "prior3", precision="fp32", max_batch=n) as fresh:
        fresh.set_undistort_maps(480, 640, *maps)
        want = valid(fresh)
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a, b)
