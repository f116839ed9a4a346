"""ctypes binding of libuahn.so (include/uahn.h) and a Python mirror of `pytorch::HomographyNet`.

This is the host-side surface for tests and bench.py.  There is no CPU fallback: if the CUDA
library cannot be loaded or no sm_100 device is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

IMG_H, IMG_W = 224, 320
MASK_BYTES_PER_PAIR = 2 * 16 * (5120 + 256)
VARIANTS = {"auto": -1, "full": 0, "prior3": 1, "prior2": 2, "prior1": 3}
PRECISIONS = {"fp32": 0, "bf16": 1}
_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libuahn.so")
EXPORTED_SYMBOLS = [
    "uahn_create", "uahn_destroy", "uahn_last_error", "uahn_load_image", "uahn_infer", "uahn_infer_batch",
    "uahn_infer_batch_device", "uahn_synchronize", "uahn_stream", "uahn_launch_count",
    "uahn_latest_inference_time", "uahn_image_count", "uahn_philox_keep_masks", "uahn_stage_dlt",
    "uahn_stage_warp", "uahn_debug_read", "uahn_profile_enable", "uahn_profile_read", "uahn_stage_conv", "uahn_submit_batch", "uahn_submit_sequence",
    "uahn_wait", "uahn_stage_transfer", "uahn_variant", "uahn_show_error",
]
PREPROC_SYMBOLS = ["uahn_undistort_init_maps", "uahn_set_undistort_maps", "uahn_load_raw_image", "uahn_stage_undistort"]
EKF_SYMBOLS = ["uahn_ekf_prior_px", "uahn_ekf_update", "uahn_ekf_reset_offsets", "uahn_ekf_iekf_frame",
               "uahn_imu_select_readings", "uahn_imu_predict_and_compute", "uahn_imu_propagate"]
FILTER_SYMBOLS = ["uahn_filter_create", "uahn_filter_destroy", "uahn_filter_set_states", "uahn_filter_get_states",
                  "uahn_filter_propagate", "uahn_filter_frame", "uahn_filter_wait", "uahn_filter_set_undistort_maps",
                  "uahn_filter_frame_raw", "uahn_filter_stage_undistort"]
ERR_INVALID, ERR_STATE, ERR_UNSUPPORTED = -1, -4, -5


class UahnError(RuntimeError):
    pass


class _Config(C.Structure):
    _fields_ = [("weights_path", C.c_char_p), ("variant", C.c_int), ("show_error", C.c_int), ("precision", C.c_int),
                ("device", C.c_int), ("max_batch", C.c_int), ("stream", C.c_void_p)]


class EkfState(C.Structure):
    """uahn_ekf_state (include/uahn_ekf.h): IMU value, the four 4-point offsets, the 27x27 covariance."""
    _fields_ = [("imu", C.c_double * 16), ("offset", (C.c_double * 3) * 4), ("cov", C.c_double * (27 * 27))]

    @classmethod
    def from_arrays(cls, imu, offsets, P):
        s = cls()
        s.imu[:] = [float(v) for v in np.asarray(imu, np.float64).reshape(16)]
        for c in range(4):
            s.offset[c][:] = [float(v) for v in np.asarray(offsets, np.float64).reshape(4, 3)[c]]
        s.cov[:] = [float(v) for v in np.asarray(P, np.float64).reshape(27 * 27)]
        return s

    def arrays(self):
        return (np.array(self.imu[:], np.float64), np.array([list(self.offset[c]) for c in range(4)], np.float64),
                np.array(self.cov[:], np.float64).reshape(27, 27))


class ImuSample(C.Structure):
    _fields_ = [("t", C.c_double), ("wm", C.c_double * 3), ("am", C.c_double * 3)]


class PropagatorConfig(C.Structure):
    """uahn_propagator_config: camera extrinsics of the planar-homography corner dynamics + IMU noise."""
    _fields_ = [("c_R_i", C.c_double * 9), ("i_t_i2c", C.c_double * 3), ("sigma_w", C.c_double), ("sigma_a", C.c_double),
                ("sigma_wb", C.c_double), ("sigma_ab", C.c_double), ("gravity_mag", C.c_double), ("imu_avg", C.c_int)]

    @classmethod
    def make(cls, c_R_i, i_t_i2c, imu_avg: bool = True):
        c = cls()
        c.c_R_i[:] = [float(v) for v in np.asarray(c_R_i, np.float64).reshape(9)]
        c.i_t_i2c[:] = [float(v) for v in np.asarray(i_t_i2c, np.float64).reshape(3)]
        c.imu_avg = int(imu_avg)
        return c


def _imu_array(readings):
    arr = (ImuSample * len(readings))()
    for a, (t, wm, am) in zip(arr, readings):
        a.t = float(t)
        a.wm[:] = [float(v) for v in wm]
        a.am[:] = [float(v) for v in am]
    return arr


def imu_select_readings(readings, time0: float, time1: float):
    lib = load_library()
    arr = _imu_array(readings)
    out = (ImuSample * (len(readings) + 4))()
    n = C.c_int(0)
    rc = lib.uahn_imu_select_readings(arr, len(readings), float(time0), float(time1), out, len(out), C.byref(n))
    if rc:
        raise UahnError(f"uahn_imu_select_readings: error {rc}")
    return [(o.t, np.array(o.wm[:]), np.array(o.am[:])) for o in out[:n.value]]


def imu_predict_and_compute(cfg: "PropagatorConfig", state: "EkfState", minus, plus):
    lib = load_library()
    a = _imu_array([minus, plus])
    F, Fw = np.empty((27, 27), np.float64), np.empty((27, 15), np.float64)
    rc = lib.uahn_imu_predict_and_compute(C.byref(cfg), C.byref(state), C.byref(a[0]), C.byref(a[1]), _ptr(F), _ptr(Fw))
    if rc:
        raise UahnError(f"uahn_imu_predict_and_compute: error {rc}")
    return F, Fw


def imu_propagate(cfg: "PropagatorConfig", state: "EkfState", readings, time0: float, time1: float) -> int:
    lib = load_library()
    arr = _imu_array(readings)
    n = C.c_int(0)
    rc = lib.uahn_imu_propagate(C.byref(cfg), C.byref(state), arr, len(readings), float(time0), float(time1), C.byref(n))
    if rc:
        raise UahnError(f"uahn_imu_propagate: error {rc}")
    return n.value


class _Rng(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("first_pair_index", C.c_uint64), ("keep_masks", C.c_void_p)]


_lib = None


def load_library(path: str | None = None):
    """Load libuahn.so (building is `python -m cuahn_vio_b200.build` / `__graft_entry__.build()`)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("UAHN_LIB_PATH") or _LIB_PATH     # UAHN_LIB_PATH: A/B runs against another build
    if not os.path.exists(p):
        raise UahnError(f"{p} not found: build it first (python cuahn_vio_b200/build.py); there is no CPU fallback")
    lib = C.CDLL(p)
    vp, i, u64, dbl = C.c_void_p, C.c_int, C.c_uint64, C.c_double
    lib.uahn_create.argtypes = [C.POINTER(_Config), C.POINTER(vp)]
    lib.uahn_create.restype = i
    lib.uahn_destroy.argtypes = [vp]
    lib.uahn_destroy.restype = None
    lib.uahn_last_error.argtypes = [vp]
    lib.uahn_last_error.restype = C.c_char_p
    lib.uahn_load_image.argtypes = [vp, vp, i, i, C.c_size_t, dbl]
    lib.uahn_load_image.restype = i
    lib.uahn_infer.argtypes = [vp, vp, C.POINTER(_Rng), vp, vp, vp]
    lib.uahn_infer.restype = i
    for f in (lib.uahn_infer_batch, lib.uahn_infer_batch_device):
        f.argtypes = [vp, i, vp, vp, vp, C.POINTER(_Rng), vp, vp, vp]
        f.restype = i
    lib.uahn_submit_batch.argtypes = [vp, i, vp, vp, vp, C.POINTER(_Rng), vp, vp]
    lib.uahn_submit_batch.restype = i
    lib.uahn_submit_sequence.argtypes = [vp, i, vp, vp, C.POINTER(_Rng), vp, vp]
    lib.uahn_submit_sequence.restype = i
    lib.uahn_wait.argtypes = [vp]
    lib.uahn_wait.restype = i
    lib.uahn_synchronize.argtypes = [vp]
    lib.uahn_synchronize.restype = i
    lib.uahn_stream.argtypes = [vp]
    lib.uahn_stream.restype = vp
    lib.uahn_launch_count.argtypes = [vp]
    lib.uahn_launch_count.restype = u64
    lib.uahn_latest_inference_time.argtypes = [vp]
    lib.uahn_latest_inference_time.restype = dbl
    lib.uahn_image_count.argtypes = [vp]
    lib.uahn_image_count.restype = i
    lib.uahn_philox_keep_masks.argtypes = [u64, u64, vp]
    lib.uahn_philox_keep_masks.restype = i
    lib.uahn_stage_dlt.argtypes = [vp, i, vp, vp]
    lib.uahn_stage_dlt.restype = i
    lib.uahn_stage_warp.argtypes = [vp, i, vp, vp, vp, vp, vp]
    lib.uahn_stage_warp.restype = i
    lib.uahn_stage_transfer.argtypes = [vp, i, vp, vp, vp, vp, vp]
    lib.uahn_stage_transfer.restype = i
    lib.uahn_variant.argtypes = [vp]
    lib.uahn_variant.restype = i
    lib.uahn_show_error.argtypes = [vp]
    lib.uahn_show_error.restype = i
    lib.uahn_profile_enable.argtypes = [vp, i]
    lib.uahn_profile_enable.restype = i
    lib.uahn_profile_read.argtypes = [vp, vp, vp]
    lib.uahn_profile_read.restype = i
    lib.uahn_stage_conv.argtypes = [vp, C.c_char_p, i, vp]
    lib.uahn_stage_conv.restype = i
    lib.uahn_debug_read.argtypes = [vp, C.c_char_p, vp, C.c_size_t]
    lib.uahn_debug_read.restype = C.c_long
    lib.uahn_undistort_init_maps.argtypes = [i, vp, vp, vp, vp]
    lib.uahn_undistort_init_maps.restype = i
    lib.uahn_set_undistort_maps.argtypes = [vp, i, i, vp, vp]
    lib.uahn_set_undistort_maps.restype = i
    lib.uahn_load_raw_image.argtypes = [vp, vp, i, i, C.c_size_t, dbl]
    lib.uahn_load_raw_image.restype = i
    lib.uahn_stage_undistort.argtypes = [vp, vp, i, i, C.c_size_t, vp]
    lib.uahn_stage_undistort.restype = i
    ekf = C.POINTER(EkfState)
    lib.uahn_ekf_prior_px.argtypes = [ekf, vp, vp]
    lib.uahn_ekf_prior_px.restype = i
    lib.uahn_ekf_update.argtypes = [ekf, vp, vp, vp, i, dbl]
    lib.uahn_ekf_update.restype = i
    lib.uahn_ekf_reset_offsets.argtypes = [ekf]
    lib.uahn_ekf_reset_offsets.restype = i
    lib.uahn_ekf_iekf_frame.argtypes = [vp, vp, ekf, i, dbl, i, i, C.POINTER(_Rng), vp, vp]
    lib.uahn_ekf_iekf_frame.restype = i
    lib.uahn_imu_select_readings.argtypes = [vp, i, dbl, dbl, vp, i, vp]
    lib.uahn_imu_select_readings.restype = i
    lib.uahn_imu_predict_and_compute.argtypes = [vp, ekf, vp, vp, vp, vp]
    lib.uahn_imu_predict_and_compute.restype = i
    lib.uahn_imu_propagate.argtypes = [vp, ekf, vp, i, dbl, dbl, vp]
    lib.uahn_imu_propagate.restype = i
    lib.uahn_filter_create.argtypes = [vp, i, vp, C.POINTER(vp)]
    lib.uahn_filter_create.restype = i
    lib.uahn_filter_destroy.argtypes = [vp]
    lib.uahn_filter_destroy.restype = None
    for f in (lib.uahn_filter_set_states, lib.uahn_filter_get_states):
        f.argtypes = [vp, i, i, vp]
        f.restype = i
    lib.uahn_filter_propagate.argtypes = [vp, vp, vp, vp, vp]
    lib.uahn_filter_propagate.restype = i
    lib.uahn_filter_frame.argtypes = [vp, vp, vp, i, dbl, i, vp, C.POINTER(_Rng), vp, vp, vp, vp]
    lib.uahn_filter_frame.restype = i
    lib.uahn_filter_wait.argtypes = [vp, vp]
    lib.uahn_filter_wait.restype = i
    lib.uahn_filter_set_undistort_maps.argtypes = [vp, i, i, vp, vp]
    lib.uahn_filter_set_undistort_maps.restype = i
    lib.uahn_filter_frame_raw.argtypes = [vp, vp, vp, C.c_size_t, i, dbl, i, vp, C.POINTER(_Rng), vp, vp, vp, vp]
    lib.uahn_filter_frame_raw.restype = i
    lib.uahn_filter_stage_undistort.argtypes = [vp, vp, C.c_size_t, vp]
    lib.uahn_filter_stage_undistort.restype = i
    if path is None:
        _lib = lib
    return lib


def undistort_init_maps(fisheye: bool, k, d):
    """CamBase::initialize_undist_map[_fisheye] through the C ABI (host only): map1, map2 float32 [224, 320]."""
    lib = load_library()
    k, d = np.ascontiguousarray(k, np.float64).reshape(4), np.ascontiguousarray(d, np.float64).reshape(4)
    m1, m2 = np.empty((IMG_H, IMG_W), np.float32), np.empty((IMG_H, IMG_W), np.float32)
    rc = lib.uahn_undistort_init_maps(int(fisheye), _ptr(k), _ptr(d), _ptr(m1), _ptr(m2))
    if rc:
        raise UahnError(f"uahn_undistort_init_maps: error {rc}")
    return m1, m2


def ekf_update(state: "EkfState", mean_px, cov_px, propagated, update_offset: bool, K_net_Cov: float = 10.0):
    """UpdaterHNet::update through the C ABI (host only)."""
    lib = load_library()
    m, c, p = (np.ascontiguousarray(a, np.float64) for a in (mean_px, cov_px, propagated))
    rc = lib.uahn_ekf_update(C.byref(state), _ptr(m), _ptr(c), _ptr(p), int(update_offset), float(K_net_Cov))
    if rc:
        raise UahnError(f"uahn_ekf_update: error {rc}")


def ekf_prior_px(state: "EkfState"):
    lib = load_library()
    a, b = np.empty(8, np.float64), np.empty(8, np.float64)
    lib.uahn_ekf_prior_px(C.byref(state), _ptr(a), _ptr(b))
    return a, b


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.c_void_p(int(a))   # raw address (e.g. torch tensor.data_ptr())


def philox_keep_masks(seed: int, pair_index: int) -> np.ndarray:
    """Host replica of the in-kernel mask generator → uint8 [2, 16, 5376] (1 = kept)."""
    out = np.empty((2, 16, 5120 + 256), np.uint8)
    rc = load_library().uahn_philox_keep_masks(seed, pair_index, _ptr(out))
    if rc:
        raise UahnError(f"uahn_philox_keep_masks rc={rc}")
    return out


def pack_keep_masks(masks) -> np.ndarray:
    """(m1[16,5120], m2[16,256], u1, u2) float {0,1/0.95} tensors → explicit keep-mask bytes [2,16,5376]."""
    m1, m2, u1, u2 = [np.asarray(m) != 0 for m in masks]
    return np.ascontiguousarray(np.stack([np.concatenate([m1, m2], 1), np.concatenate([u1, u2], 1)]).astype(np.uint8))


class Uahn:
    """Thin RAII wrapper over a uahn_handle."""

    def __init__(self, weights_path: str, variant: str = "prior3", show_error: bool = False, precision: str = "fp32",
                 device: int = 0, max_batch: int = 1, stream: int | None = None):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.variant, self.show_error, self.precision, self.max_batch = variant, show_error, precision, max_batch
        cfg = _Config(os.fsencode(weights_path), VARIANTS[variant], -1 if show_error is None else int(show_error),
                      PRECISIONS[precision], device, max_batch, stream)
        rc = self._lib.uahn_create(C.byref(cfg), C.byref(self._h))
        if rc:
            msg = self._lib.uahn_last_error(None).decode()
            self._h = None
            raise UahnError(f"uahn_create failed ({rc}): {msg}")
        # "auto" / None: resolved from the records weights.export_torchscript wrote into the file
        self.variant = {v: k for k, v in VARIANTS.items()}[self._lib.uahn_variant(self._h)]
        self.show_error = bool(self._lib.uahn_show_error(self._h))

    def close(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.uahn_destroy(h)
            self._h = None        # (no ctypes call here: this also runs at interpreter shutdown)

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc < 0:
            raise UahnError(f"rc={rc}: {self._lib.uahn_last_error(self._h).decode()}")
        return rc

    @staticmethod
    def _rng(seed, first_pair, masks):
        return _Rng(seed, first_pair, _ptr(masks).value if masks is not None else None)

    # -- reference call surface ----------------------------------------------------------------------
    def load_image(self, img: np.ndarray, time_stamp: float = 0.0):
        img = np.ascontiguousarray(img, np.uint8)
        self._check(self._lib.uahn_load_image(self._h, _ptr(img), img.shape[0], img.shape[1], img.strides[0], time_stamp))

    def set_undistort_maps(self, raw_rows: int, raw_cols: int, map1: np.ndarray, map2: np.ndarray):
        m1, m2 = np.ascontiguousarray(map1, np.float32), np.ascontiguousarray(map2, np.float32)
        self._check(self._lib.uahn_set_undistort_maps(self._h, raw_rows, raw_cols, _ptr(m1), _ptr(m2)))

    def load_raw_image(self, raw: np.ndarray, time_stamp: float = 0.0):
        raw = np.ascontiguousarray(raw, np.uint8)
        self._check(self._lib.uahn_load_raw_image(self._h, _ptr(raw), raw.shape[0], raw.shape[1], raw.strides[0], time_stamp))

    def stage_undistort(self, raw: np.ndarray) -> np.ndarray:
        raw = np.ascontiguousarray(raw, np.uint8)
        out = np.empty((IMG_H, IMG_W), np.uint8)
        self._check(self._lib.uahn_stage_undistort(self._h, _ptr(raw), raw.shape[0], raw.shape[1], raw.strides[0], _ptr(out)))
        return out

    def infer(self, prior_px=None, seed: int = 0, pair_index: int | None = None, keep_masks: np.ndarray | None = None,
              want_error: bool = False):
        """pair_index None (default): the handle numbers its calls itself, so every forward draws fresh MC-dropout
        masks like the reference (model_to_trace.py:266-273); an explicit (seed, pair_index) replays a given draw."""
        prior = None if prior_px is None else np.ascontiguousarray(prior_px, np.float64).reshape(8)
        mean, cov = np.empty(8, np.float64), np.empty((8, 8), np.float64)
        err = np.empty((IMG_H, IMG_W), np.uint8) if want_error else None
        if pair_index is None and keep_masks is None and seed == 0:
            rng_ref = None
        else:
            rng = self._rng(seed, pair_index or 0, keep_masks)
            rng_ref = C.byref(rng)
        self._check(self._lib.uahn_infer(self._h, _ptr(prior), rng_ref, _ptr(mean), _ptr(cov), _ptr(err)))
        return mean, cov, err

    def infer_batch(self, prev: np.ndarray, curr: np.ndarray, prior: np.ndarray | None = None, seed: int = 0,
                    first_pair: int = 0, keep_masks: np.ndarray | None = None, want_error: bool = False):
        n = prev.shape[0]
        prev, curr = np.ascontiguousarray(prev, np.uint8), np.ascontiguousarray(curr, np.uint8)
        prior = None if prior is None else np.ascontiguousarray(prior, np.float32).reshape(n, 8)
        if keep_masks is not None:
            keep_masks = np.ascontiguousarray(keep_masks, np.uint8)
            assert keep_masks.size == n * MASK_BYTES_PER_PAIR
        mean, cov = np.empty((n, 8), np.float32), np.empty((n, 8, 8), np.float32)
        err = np.empty((n, IMG_H, IMG_W), np.float32) if want_error else None
        rng = self._rng(seed, first_pair, keep_masks)
        self._check(self._lib.uahn_infer_batch(self._h, n, _ptr(prev), _ptr(curr), _ptr(prior), C.byref(rng), _ptr(mean),
                                               _ptr(cov), _ptr(err)))
        return mean, cov, err

    def infer_batch_ptrs(self, n, prev, curr, prior, mean, cov, err=None, seed=0, first_pair=0, device=True):
        """Raw-address form (device pointers by default): asynchronous on the handle's stream."""
        rng = _Rng(seed, first_pair, None)
        f = self._lib.uahn_infer_batch_device if device else self._lib.uahn_infer_batch
        self._check(f(self._h, n, _ptr(prev), _ptr(curr), _ptr(prior), C.byref(rng), _ptr(mean), _ptr(cov), _ptr(err)))

    def submit_batch_ptrs(self, n, prev, curr, prior, mean, cov, seed=0, first_pair=0):
        """Pipelined host-buffer submission (raw addresses of pinned host memory); pair with wait()."""
        rng = _Rng(seed, first_pair, None)
        self._check(self._lib.uahn_submit_batch(self._h, n, _ptr(prev), _ptr(curr), _ptr(prior), C.byref(rng), _ptr(mean),
                                                _ptr(cov)))

    def submit_sequence_ptrs(self, n_frames, frames, prior, mean, cov, seed=0, first_pair=0):
        """Pipelined submission of one sequence: pair i = (frames[i], frames[i+1]); raw pinned-host addresses."""
        rng = _Rng(seed, first_pair, None)
        self._check(self._lib.uahn_submit_sequence(self._h, n_frames, _ptr(frames), _ptr(prior), C.byref(rng), _ptr(mean),
                                                   _ptr(cov)))

    def iekf_frame(self, state: "EkfState", max_iter: int = 1, K_net_Cov: float = 10.0, min_images: int = 10,
                   use_measurement: bool = True, seed: int = 0, pair_index: int | None = None,
                   iterative: "Uahn | None" = None):
        """One camera frame of the IEKF loop (VioManager.cpp:227-275); returns the last network (mean, cov) in px.
        pair_index None: fresh masks on every forward (per-handle counters); explicit: iteration `it` uses pair_index + it."""
        mean, cov = np.empty(8, np.float64), np.empty((8, 8), np.float64)
        rng = None if pair_index is None and seed == 0 else C.byref(_Rng(seed, pair_index or 0, None))
        self._check(self._lib.uahn_ekf_iekf_frame(self._h, iterative._h if iterative else None, C.byref(state), max_iter,
                                                  float(K_net_Cov), min_images, int(use_measurement), rng,
                                                  _ptr(mean), _ptr(cov)))
        return mean, cov

    def wait(self):
        self._check(self._lib.uahn_wait(self._h))

    def synchronize(self):
        self._check(self._lib.uahn_synchronize(self._h))

    @property
    def stream(self) -> int:
        return int(self._lib.uahn_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self._lib.uahn_launch_count(self._h))

    @property
    def img_counter(self) -> int:
        return int(self._lib.uahn_image_count(self._h))

    @property
    def latest_inference_time(self) -> float:
        return float(self._lib.uahn_latest_inference_time(self._h))

    def profile_enable(self, on: bool = True):
        self._check(self._lib.uahn_profile_enable(self._h, int(on)))

    def profile_read(self):
        """→ (ms[4], launches[4]) per category: 0 warp/error-map, 1 conv stacks, 2 MC-head GEMMs, 3 small head kernels."""
        ms, cnt = np.zeros(4, np.float64), np.zeros(4, np.uint64)
        self._check(self._lib.uahn_profile_read(self._h, _ptr(ms), _ptr(cnt)))
        return ms, cnt

    # -- stage entry points --------------------------------------------------------------------------
    def stage_dlt(self, offsets: np.ndarray) -> np.ndarray:
        off = np.ascontiguousarray(offsets, np.float32).reshape(-1, 8)
        out = np.empty((off.shape[0], 3, 3), np.float32)
        self._check(self._lib.uahn_stage_dlt(self._h, off.shape[0], _ptr(off), _ptr(out)))
        return out

    def stage_warp(self, img: np.ndarray, H: np.ndarray):
        img = np.ascontiguousarray(img, np.uint8).reshape(-1, IMG_H, IMG_W)
        H = np.ascontiguousarray(H, np.float32).reshape(-1, 9)
        n = img.shape[0]
        out = np.empty((n, IMG_H, IMG_W), np.float32)
        ix, iy = np.empty((n, IMG_H, IMG_W), np.int16), np.empty((n, IMG_H, IMG_W), np.int16)
        self._check(self._lib.uahn_stage_warp(self._h, n, _ptr(img), _ptr(H), _ptr(out), _ptr(ix), _ptr(iy)))
        return out, ix, iy

    def stage_transfer(self, var: np.ndarray, Hp: np.ndarray, pts_w: np.ndarray):
        """transfer_mean_var_single + packing (model_to_trace.py:18-38, 311-317) → flow [n, 8], cov [n, 8, 8]."""
        var = np.ascontiguousarray(var, np.float32).reshape(-1, 8)
        n = var.shape[0]
        Hp = np.ascontiguousarray(Hp, np.float32).reshape(n, 9)
        pts_w = np.ascontiguousarray(pts_w, np.float32).reshape(n, 8)
        flow, cov = np.empty((n, 8), np.float32), np.empty((n, 8, 8), np.float32)
        self._check(self._lib.uahn_stage_transfer(self._h, n, _ptr(var), _ptr(Hp), _ptr(pts_w), _ptr(flow), _ptr(cov)))
        return flow, cov

    def stage_conv(self, layer: str, x: np.ndarray, out_shape) -> np.ndarray:
        """Run one Conv2d+LeakyReLU layer (x: n x Cin x H x W float32) → n x Cout x Ho x Wo."""
        x = np.ascontiguousarray(x, np.float32)
        self._check(self._lib.uahn_stage_conv(self._h, layer.encode(), x.shape[0], _ptr(x)))
        return self.debug_read("act:" + layer, (x.shape[0],) + tuple(out_shape))

    def debug_read(self, what: str, shape) -> np.ndarray:
        out = np.empty(shape, np.float32)
        got = self._check(self._lib.uahn_debug_read(self._h, what.encode(), _ptr(out), out.size))
        if got != out.size:
            raise UahnError(f"debug_read({what}): got {got} floats, expected {out.size}")
        return out


class HomographyNet:
    """Python mirror of `pytorch::HomographyNet` (HomographyNet.h:23-67) over the C ABI.

    Same members and argument meaning: ctor(model path → weights file, iterative model path, use_prior,
    num_of_iteration, show_imgs); load_current_img; network_inference(prior_4pt_offset_vec, iteration);
    get_pred_mean / get_pred_Cov / get_latest_inference_time; img_counter.  Variant selection follows the
    reference's file-name convention (`_showError` substring, HomographyNet.cpp:96-100).
    """

    def __init__(self, network_model_path: str, network_model_iterative_path: str = "", use_prior: bool = True,
                 num_of_iteration: int = 1, show_imgs: bool = False, precision: str = "bf16", device: int = 0,
                 iterative_variant: str = "auto"):
        self.use_prior = use_prior
        self.show_error = "_showError" in network_model_path
        self.show_imgs = show_imgs
        self._main = Uahn(network_model_path, "prior3" if use_prior else "full", self.show_error, precision, device, 1)
        self._iter = None
        if num_of_iteration > 1:
            # the reference's second slot runs whatever graph the file holds (HomographyNet.cpp:104-124): "auto" takes the
            # variant weights.export_torchscript recorded; files without a record fall back to the 2-block schedule
            ipath = network_model_iterative_path or network_model_path
            ishow = "_showError" in ipath
            try:
                self._iter = Uahn(ipath, iterative_variant, ishow, precision, device, 1)
            except UahnError:
                if iterative_variant != "auto":
                    raise
                self._iter = Uahn(ipath, "prior2", ishow, precision, device, 1)
        self._mean = np.zeros(8)
        self._cov = np.zeros((8, 8))
        self.error_map = None
        self.seed = 0
        self._calls = 0

    @property
    def img_counter(self) -> int:
        return self._main.img_counter

    def load_current_img(self, img: np.ndarray, time_stamp: float):
        self._main.load_image(img, time_stamp)
        if self._iter is not None:
            self._iter.load_image(img, time_stamp)

    def network_inference(self, prior_4pt_offset_vec, iteration: int = 0):
        if self.img_counter < 2:                       # HomographyNet.cpp:155-158: message, outputs untouched
            print("HNet cannot inference! Only has one image!")
            return
        net = self._main if iteration == 0 or self._iter is None else self._iter
        self._calls += 1
        mean, cov, err = net.infer(prior_4pt_offset_vec if self.use_prior else None, seed=self.seed,
                                   pair_index=self._calls, want_error=self.show_imgs and net.show_error)
        self._mean, self._cov, self.error_map = mean, cov, err

    def get_pred_mean(self):
        return self._mean.copy()

    def get_pred_Cov(self):
        return self._cov.copy()

    def get_latest_inference_time(self) -> float:
        return self._main.latest_inference_time


class FilterBank:
    """n EKF states on the device next to one Uahn handle (include/uahn_filter.h).

    States are numpy arrays: imu [k, 16], offsets [k, 4, 3], cov [k, 27, 27] (float64).  propagate() and frame() only
    enqueue work; their inputs must stay alive and their outputs are valid once wait() has returned."""

    def __init__(self, net: "Uahn", n: int, cfg: "PropagatorConfig"):
        self._lib, self.net, self.n = net._lib, net, n
        self._f = C.c_void_p()
        self._cfg = cfg
        self._keep = []
        self._raw_shape = None       # (raw_rows, raw_cols) of the maps set last
        net._check(self._lib.uahn_filter_create(net._h, n, C.byref(cfg), C.byref(self._f)))

    def close(self):
        f = getattr(self, "_f", None)
        if f is not None and f.value:
            self._lib.uahn_filter_destroy(f)
            self._f = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        return self.net._check(rc)

    def set_states(self, first: int, imu, offsets, cov):
        imu = np.asarray(imu, np.float64).reshape(-1, 16)
        k = imu.shape[0]
        raw = np.empty((k, 16 + 12 + 27 * 27), np.float64)      # uahn_ekf_state rows
        raw[:, :16] = imu
        raw[:, 16:28] = np.asarray(offsets, np.float64).reshape(k, 12)
        raw[:, 28:] = np.asarray(cov, np.float64).reshape(k, 27 * 27)
        self._check(self._lib.uahn_filter_set_states(self._f, first, k, _ptr(raw)))

    def get_states(self, first: int = 0, count: int | None = None):
        """→ (imu [k, 16], offsets [k, 4, 3], cov [k, 27, 27])"""
        count = self.n - first if count is None else count
        raw = np.empty((count, 16 + 12 + 27 * 27), np.float64)
        self._check(self._lib.uahn_filter_get_states(self._f, first, count, _ptr(raw)))
        return raw[:, :16].copy(), raw[:, 16:28].reshape(count, 4, 3).copy(), raw[:, 28:].reshape(count, 27, 27).copy()

    def propagate(self, readings, t0, t1):
        """readings: one list of (t, wm[3], am[3]) per slot; t0 / t1: per-slot interval ends."""
        flat = [r for slot in readings for r in slot]
        offsets = np.zeros(self.n + 1, np.int32)
        offsets[1:] = np.cumsum([len(slot) for slot in readings])
        imu = _imu_array(flat) if flat else (ImuSample * 1)()
        t0, t1 = np.ascontiguousarray(t0, np.float64), np.ascontiguousarray(t1, np.float64)
        self._keep += [imu, offsets, t0, t1]
        self._check(self._lib.uahn_filter_propagate(self._f, imu, _ptr(offsets), _ptr(t0), _ptr(t1)))

    def frame(self, frames, max_iter: int = 1, K_net_Cov: float = 10.0, min_images: int = 10, use_measurement=None,
              seed: int = 0, first_pair: int | None = None, iterative: "Uahn | None" = None, keep_masks=None):
        """One IEKF frame for every slot → dict of numpy outputs (prior/mean [max_iter, n, 8], cov [max_iter, n, 8, 8],
        imu [n, 16]), filled when wait() returns.  first_pair None: the bank numbers its frames itself."""
        frames = np.ascontiguousarray(frames, np.uint8)
        assert frames.shape == (self.n, IMG_H, IMG_W)
        return self._frame(self._lib.uahn_filter_frame, (_ptr(frames),), frames, max_iter, K_net_Cov, min_images,
                           use_measurement, seed, first_pair, iterative, keep_masks)

    def frame_raw(self, raw, max_iter: int = 1, K_net_Cov: float = 10.0, min_images: int = 10, use_measurement=None,
                  seed: int = 0, first_pair: int | None = None, iterative: "Uahn | None" = None, keep_masks=None):
        """frame() with raw camera frames [n, raw_rows, raw_cols] u8 (any row stride), undistorted on the device with the
        maps of set_undistort_maps(); same arguments and outputs as frame()."""
        raw, stride = self._raw_frames(raw)
        return self._frame(self._lib.uahn_filter_frame_raw, (_ptr(raw), stride), raw, max_iter, K_net_Cov, min_images,
                           use_measurement, seed, first_pair, iterative, keep_masks)

    def _frame(self, fn, frame_args, frames, max_iter, K_net_Cov, min_images, use_measurement, seed, first_pair, iterative,
               keep_masks):
        use = None if use_measurement is None else np.ascontiguousarray(use_measurement, np.uint8)
        out = {"prior": np.empty((max_iter, self.n, 8), np.float32), "mean": np.empty((max_iter, self.n, 8), np.float32),
               "cov": np.empty((max_iter, self.n, 8, 8), np.float32), "imu": np.empty((self.n, 16), np.float64)}
        rng = None
        if first_pair is not None or seed or keep_masks is not None:
            rng = C.byref(_Rng(seed, first_pair or 0, _ptr(keep_masks).value if keep_masks is not None else None))
        self._keep += [frames, use, out]
        self._check(fn(self._f, iterative._h if iterative else None, *frame_args, max_iter, float(K_net_Cov), min_images,
                       _ptr(use), rng, _ptr(out["prior"]), _ptr(out["mean"]), _ptr(out["cov"]), _ptr(out["imu"])))
        return out

    def set_undistort_maps(self, raw_rows: int, raw_cols: int, map1: np.ndarray, map2: np.ndarray):
        """One camera for every slot: map1 / map2 float32 [224, 320] (undistort_init_maps), raw frames raw_rows x raw_cols."""
        m1, m2 = np.ascontiguousarray(map1, np.float32), np.ascontiguousarray(map2, np.float32)
        assert m1.shape == (IMG_H, IMG_W) and m2.shape == (IMG_H, IMG_W)
        self._raw_shape = None
        self._check(self._lib.uahn_filter_set_undistort_maps(self._f, raw_rows, raw_cols, _ptr(m1), _ptr(m2)))
        self._raw_shape = (raw_rows, raw_cols)

    def stage_undistort(self, raw) -> np.ndarray:
        """The n raw frames [n, raw_rows, raw_cols] remapped with the bank's maps → [n, 224, 320] u8 (synchronous)."""
        raw, stride = self._raw_frames(raw)
        out = np.empty((self.n, IMG_H, IMG_W), np.uint8)
        self._check(self._lib.uahn_filter_stage_undistort(self._f, _ptr(raw), stride, _ptr(out)))
        return out

    def _raw_frames(self, raw):
        """→ (array, row stride): [n, rows, cols] u8 whose frames sit rows * stride bytes apart, copied only if they do not."""
        raw = np.asarray(raw)
        assert raw.dtype == np.uint8 and raw.ndim == 3 and raw.shape[0] == self.n, (raw.dtype, raw.shape)
        rows, cols = raw.shape[1:]
        # the library reads rows x cols of the maps' raw size: a smaller array would be read past its end
        assert self._raw_shape is None or (rows, cols) == self._raw_shape, ((rows, cols), self._raw_shape)
        s0, s1, s2 = raw.strides
        if not (s2 == 1 and s1 >= cols and (self.n == 1 or s0 == rows * s1)):
            raw = np.ascontiguousarray(raw)
            s1 = cols
        return raw, s1

    def wait(self):
        """→ per-slot codes since the previous wait (0, ERR_STATE, ERR_INVALID)."""
        status = np.zeros(self.n, np.int32)
        rc = self._lib.uahn_filter_wait(self._f, _ptr(status))
        self._keep = []
        if rc not in (0, ERR_STATE, ERR_INVALID):
            self._check(rc)
        return status
