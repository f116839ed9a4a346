"""Closed-loop frames/s of the filter bank (include/uahn_filter.h) against the host filter loop around one batched forward.

S sequences x F frames of a bf16 prior3 handle, a 500 Hz synthetic IMU and a 30 Hz camera, at S = 128 and 1024.  Three
arms, timed in the same process and alternated:
  bank     uahn_filter_propagate + uahn_filter_frame per step (max_iter 1), one uahn_filter_wait at the end
  host     per step: S x uahn_imu_propagate, one uahn_infer_batch with those priors, S x uahn_ekf_update (fewer steps)
  network  uahn_infer_batch_device at n = S with fixed priors (device buffers)
The bank's filter-kernel time per step comes from CUDA kernel records of torch.profiler in a separate pass.  Frames and
IMU readings are generated from seeds before timing.  Prints one JSON line; --out FILE also writes it to FILE.

--raw adds, per size, two arms alternated with the bank arm, and a "raw" record:
  raw bank  uahn_filter_propagate + uahn_filter_frame_raw per step: pinned 640x480 frames (synthetic_raw_frame, a few
            unique ones tiled to S) undistorted on the device with the uahn_undistort_init_maps maps of one fixture camera
  ceiling   a bare pinned cudaMemcpyAsync of the same raw bytes per step
A profiled raw-bank pass of its own gives the remap kernel's and the filter kernels' time per step, the device time of the
host-to-device copies and how much of it ran while a kernel was running.  raw_step_over_bound = raw-bank step /
max(ceiling copy time, network step + filter kernels + remap), every term from the same run.

  python tools/filter_bench.py [--sizes 128 1024] [--frames 64] [--host-steps 4] [--raw] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HZ_IMU, HZ_CAM = 500.0, 30.0
# the synthetic weights' outputs are not measurements of the synthetic IMU motion: a large measurement noise keeps the
# filters from diverging over the timed frames (the work per update does not depend on it)
K_NET_COV = 1000.0
IMU_DTYPE = np.dtype([("t", np.float64), ("wm", np.float64, 3), ("am", np.float64, 3)])   # uahn_imu_sample
RAW_ROWS, RAW_COLS, RAW_UNIQUE = 480, 640, 8
RAW_CAMERA = "uzhfpv_indoor_fwd"                 # a fisheye camera of tests/golden/preproc.npz
HBM_BYTES_PER_S = 7.7e12                         # B200 data sheet (one GPU): the bound the remap kernel is held to


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in q.split(",")]
    return name, power


def initial_states(api, S, rng):
    imu = np.zeros((S, 16))
    imu[:, 0:3] = [0.3, -0.2, 1.5] + 0.1 * rng.standard_normal((S, 3))
    q = np.concatenate([np.ones((S, 1)), 0.1 * rng.standard_normal((S, 3))], 1)
    imu[:, 3:7] = q / np.linalg.norm(q, axis=1, keepdims=True)
    imu[:, 7:10] = 0.5 * rng.standard_normal((S, 3))
    off = 0.02 * rng.standard_normal((S, 4, 3))
    A = rng.standard_normal((27, 27))
    P = np.broadcast_to(1e-4 * (A @ A.T) / 27 + 1e-6 * np.eye(27), (S, 27, 27)).copy()
    return imu, off, P


def imu_steps(S, steps, rng):
    """Per step: readings [S x k] of every slot covering [t0, t1] (offsets into one flat array), t0, t1."""
    out = []
    phase = 0.002 * rng.random(S)
    for k in range(steps):
        t0 = 10.0 + k / HZ_CAM + phase
        t1 = t0 + 1.0 / HZ_CAM
        k0 = np.floor((t0 - phase) * HZ_IMU).astype(int) - 1
        cnt = int(np.ceil((1.0 / HZ_CAM) * HZ_IMU)) + 3
        r = np.zeros((S, cnt), IMU_DTYPE)
        r["t"] = phase[:, None] + (k0[:, None] + np.arange(cnt)[None]) / HZ_IMU
        r["wm"] = 0.3 * rng.standard_normal((S, cnt, 3))
        r["am"] = np.array([0, 0, 9.81]) + 0.5 * rng.standard_normal((S, cnt, 3))
        offsets = (np.arange(S + 1) * cnt).astype(np.int32)
        out.append((np.ascontiguousarray(r.reshape(-1)), offsets, t0, t1))
    return out


def pinned(shape, dtype):
    import torch
    return torch.empty(shape, dtype=dtype, pin_memory=True).numpy()


def run_size(api, wfile, S, n_frames, host_steps, rounds, raw_arms=False):
    import torch
    lib = api.load_library()
    rng = np.random.default_rng(S)
    from cuahn_vio_b200 import synthetic as Syn
    prev_u, curr_u, _, prior_u = Syn.tiled_batch(S, unique=64)
    frames = [pinned(prev_u.shape, torch.uint8), pinned(prev_u.shape, torch.uint8)]
    frames[0][:], frames[1][:] = prev_u, curr_u                 # frame k of every slot: frames[k % 2]
    steps = imu_steps(S, n_frames, rng)
    imu0, off0, P0 = initial_states(api, S, rng)
    cfg = api.PropagatorConfig.make(np.eye(3), [0.0, 0.0, 0.05], True)
    net = api.Uahn(wfile, "prior3", precision="bf16", max_batch=S)
    bank = api.FilterBank(net, S, cfg)
    st = torch.cuda.ExternalStream(net.stream)

    failed = []   # slots whose filter diverged in a pass (they skip their updates from then on)

    def bank_pass(frames_n):
        bank.set_states(0, imu0, off0, P0)
        torch.cuda.synchronize()
        t = time.perf_counter()
        for k in range(frames_n):
            r, offsets, t0, t1 = steps[k]
            if k:
                assert lib.uahn_filter_propagate(bank._f, r.ctypes.data, offsets.ctypes.data, t0.ctypes.data, t1.ctypes.data) == 0
            assert lib.uahn_filter_frame(bank._f, None, frames[k % 2].ctypes.data, 1, K_NET_COV, 2, None, None, None, None, None,
                                         None) == 0
        status = bank.wait()
        dt = time.perf_counter() - t
        failed.append(int((status != 0).sum()))
        return dt / frames_n

    # network alone: device frames and fixed priors
    d_prev = torch.from_numpy(prev_u).cuda()
    d_curr = torch.from_numpy(curr_u).cuda()
    d_prior = torch.from_numpy(prior_u.reshape(S, 8)).cuda()
    d_mean = torch.empty((S, 8), device="cuda")
    d_cov = torch.empty((S, 64), device="cuda")

    def net_pass(k_steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record()
            for k in range(k_steps):
                net.infer_batch_ptrs(S, d_prev.data_ptr(), d_curr.data_ptr(), d_prior.data_ptr(), d_mean.data_ptr(),
                                     d_cov.data_ptr(), first_pair=k * S)
            e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3 / k_steps

    def host_pass(k_steps):
        states = (api.EkfState * S)()
        for i in range(S):
            src = api.EkfState.from_arrays(imu0[i], off0[i], P0[i])
            C.memmove(C.addressof(states[i]), C.addressof(src), C.sizeof(api.EkfState))
        prior = np.empty((S, 8), np.float32)
        propagated = np.empty((S, 8))
        px = np.empty(8)
        m64, c64 = np.empty(8), np.empty(64)
        n_int = C.c_int(0)
        t_prop = 0.0
        t = time.perf_counter()
        for k in range(k_steps):
            r, offsets, t0, t1 = steps[k + 1]
            tp = time.perf_counter()
            for i in range(S):
                lib.uahn_imu_propagate(C.byref(cfg), C.byref(states[i]), r[offsets[i]:].ctypes.data, int(offsets[i + 1] - offsets[i]),
                                       float(t0[i]), float(t1[i]), C.byref(n_int))
            t_prop += time.perf_counter() - tp
            for i in range(S):
                lib.uahn_ekf_prior_px(C.byref(states[i]), api._ptr(px), api._ptr(propagated[i]))
                prior[i] = px
            mean, cov, _ = net.infer_batch(frames[k % 2], frames[(k + 1) % 2], prior, first_pair=k * S)
            cov = cov.reshape(S, 64)
            for i in range(S):
                m64[:], c64[:] = mean[i], cov[i]
                lib.uahn_ekf_update(C.byref(states[i]), api._ptr(m64), api._ptr(c64), api._ptr(propagated[i]), 0, K_NET_COV)
                lib.uahn_ekf_reset_offsets(C.byref(states[i]))
        dt = time.perf_counter() - t
        return dt / k_steps, t_prop / (k_steps * S)

    raw = RawArms(api, bank, S, steps, imu0, off0, P0) if raw_arms else None

    # warm-up of every shape
    bank_pass(4)
    net_pass(3)
    host_pass(1)
    if raw:
        raw.bank_pass(4)
        raw.ceiling_pass(3)
    res = {"bank_step_s": [], "net_step_s": [], "host_step_s": [], "host_prop_per_seq_s": []}
    for _ in range(rounds):
        res["bank_step_s"].append(bank_pass(n_frames))
        res["net_step_s"].append(net_pass(n_frames))
        if raw:
            raw.timed_round(n_frames)
    hs, hp = host_pass(host_steps)
    res["host_step_s"].append(hs)
    res["host_prop_per_seq_s"].append(hp)
    for _ in range(rounds):
        res["bank_step_s"].append(bank_pass(n_frames))
        res["net_step_s"].append(net_pass(n_frames))
        if raw:
            raw.timed_round(n_frames)

    # filter-kernel time per step: CUDA kernel records of a profiled bank pass of its own
    from torch.profiler import ProfilerActivity, profile
    prof_frames = 16
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        bank_pass(prof_frames)
    kern = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "filter_" in ev.name:
            name = ev.name.split("filter_")[1].split("_kernel")[0]
            kern[name] = kern.get(name, 0.0) + ev.device_time / 1e6
    kern = {k: v / prof_frames for k, v in kern.items()}
    bank_s, net_s, host_s = (float(np.median(res[k])) for k in ("bank_step_s", "net_step_s", "host_step_s"))
    raw_row = raw.result(prof_frames, net_s) if raw else None
    bank.close()
    net.close()
    filt = sum(kern.values())
    row = {
        "S": S, "frames": n_frames, "host_steps": host_steps,
        "bank_frames_per_s": S / bank_s, "host_loop_frames_per_s": S / host_s, "network_frames_per_s": S / net_s,
        "bank_over_host": host_s / bank_s,
        "bank_step_ms": bank_s * 1e3, "network_step_ms": net_s * 1e3, "host_step_ms": host_s * 1e3,
        "filter_kernel_ms_per_step": filt * 1e3, "filter_kernel_ms_per_step_by_kernel": {k: v * 1e3 for k, v in kern.items()},
        "filter_kernel_share_of_network_step": filt / net_s,
        "bank_slots_failed_per_pass": failed, "K_net_Cov": K_NET_COV,
        "host_propagate_ms_per_sequence": float(np.median(res["host_prop_per_seq_s"])) * 1e3,
        "bank_step_ms_all": [v * 1e3 for v in res["bank_step_s"]], "network_step_ms_all": [v * 1e3 for v in res["net_step_s"]],
    }
    if raw_row:
        row["raw"] = raw_row
    return row


def _union(intervals):
    out = []
    for a, b in sorted(intervals):
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return out


def _overlap(intervals, union):
    """Total length of `intervals` that lies inside the (sorted, disjoint) `union`."""
    tot = 0.0
    for a, b in intervals:
        for c, d in union:
            if c >= b:
                break
            tot += max(0.0, min(b, d) - max(a, c))
    return tot


class RawArms:
    """The --raw arms on the bank of run_size: frame_raw from pinned raw frames, and the bare copy of the same bytes."""

    def __init__(self, api, bank, S, steps, imu0, off0, P0):
        import torch
        from cuahn_vio_b200 import synthetic as Syn
        self.api, self.lib, self.bank, self.S, self.steps = api, api.load_library(), bank, S, steps
        self.state0, self.failed = (imu0, off0, P0), []     # slots whose filter diverged, per raw-bank pass
        golden = np.load(os.path.join(ROOT, "tests", "golden", "preproc.npz"))
        m1, m2 = api.undistort_init_maps(bool(golden[f"{RAW_CAMERA}_fisheye"]), golden[f"{RAW_CAMERA}_k"],
                                         golden[f"{RAW_CAMERA}_d"])
        bank.set_undistort_maps(RAW_ROWS, RAW_COLS, m1, m2)
        uniq = np.stack([Syn.synthetic_raw_frame(900 + i, RAW_ROWS, RAW_COLS) for i in range(RAW_UNIQUE)])
        # frame k of every slot: host[k % 2]; slot i shows unique frame (i + k) % RAW_UNIQUE
        self.host = [torch.empty((S, RAW_ROWS, RAW_COLS), dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        for j, t in enumerate(self.host):
            t.numpy()[:] = uniq[(np.arange(S) + j) % RAW_UNIQUE]
        self.dev = torch.empty((S, RAW_ROWS, RAW_COLS), dtype=torch.uint8, device="cuda")
        self.copy_stream = torch.cuda.Stream()
        self.res = {"raw_step_s": [], "ceiling_step_s": []}

    def bank_pass(self, frames_n):
        import torch
        bank, lib = self.bank, self.lib
        bank.set_states(0, *self.state0)
        torch.cuda.synchronize()
        t = time.perf_counter()
        for k in range(frames_n):
            r, offsets, t0, t1 = self.steps[k]
            if k:
                assert lib.uahn_filter_propagate(bank._f, r.ctypes.data, offsets.ctypes.data, t0.ctypes.data, t1.ctypes.data) == 0
            assert lib.uahn_filter_frame_raw(bank._f, None, self.host[k % 2].data_ptr(), RAW_COLS, 1, K_NET_COV, 2, None, None,
                                             None, None, None, None) == 0
        status = bank.wait()
        dt = time.perf_counter() - t
        self.failed.append(int((status != 0).sum()))
        return dt / frames_n

    def ceiling_pass(self, frames_n):
        import torch
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(self.copy_stream):
            e0.record()
            for k in range(frames_n):
                self.dev.copy_(self.host[k % 2], non_blocking=True)      # cudaMemcpyAsync from pinned memory
            e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3 / frames_n

    def timed_round(self, frames_n):
        self.res["raw_step_s"].append(self.bank_pass(frames_n))
        self.res["ceiling_step_s"].append(self.ceiling_pass(frames_n))

    def result(self, prof_frames, net_s):
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            self.bank_pass(prof_frames)
        remap = filt = h2d = 0.0
        kernels, copies = [], []
        for ev in prof.events():
            if ev.device_type.name != "CUDA":
                continue
            span = (ev.time_range.start, ev.time_range.end)
            if ev.name.startswith("Memcpy HtoD"):
                h2d += ev.device_time / 1e6
                copies.append(span)
                continue
            if ev.name.startswith("Memcpy") or ev.name.startswith("Memset"):
                continue
            kernels.append(span)
            if "remap_bilinear_u8" in ev.name:
                remap += ev.device_time / 1e6
            elif "filter_" in ev.name:
                filt += ev.device_time / 1e6
        remap, filt, h2d = remap / prof_frames, filt / prof_frames, h2d / prof_frames
        copy_total = sum(b - a for a, b in copies)
        overlap = _overlap(copies, _union(kernels)) / copy_total if copy_total else 0.0
        raw_s, ceil_s = (float(np.median(self.res[k])) for k in ("raw_step_s", "ceiling_step_s"))
        raw_bytes = self.S * RAW_ROWS * RAW_COLS
        remap_bytes = self.S * (RAW_ROWS * RAW_COLS + 224 * 320)      # raw frames read + undistorted frames written
        bound = max(ceil_s, net_s + filt + remap)
        return {
            "raw_rows": RAW_ROWS, "raw_cols": RAW_COLS, "camera": RAW_CAMERA,
            "raw_bank_frames_per_s": self.S / raw_s, "raw_bank_step_ms": raw_s * 1e3,
            "raw_h2d_ceiling_ms_per_step": ceil_s * 1e3, "raw_h2d_ceiling_GB_per_s": raw_bytes / ceil_s / 1e9,
            "h2d_device_ms_per_step_in_raw_bank": h2d * 1e3, "h2d_share_under_kernels": overlap,
            "remap_kernel_ms_per_step": remap * 1e3, "remap_bytes_per_step": remap_bytes,
            "remap_GB_per_s": remap_bytes / remap / 1e9 if remap else None,
            "remap_hbm_bound_ms": remap_bytes / HBM_BYTES_PER_S * 1e3,
            "remap_share_of_hbm_bound": (remap_bytes / HBM_BYTES_PER_S) / remap if remap else None,
            "filter_kernel_ms_per_step": filt * 1e3, "network_step_ms": net_s * 1e3,
            "compute_ms_per_step": (net_s + filt + remap) * 1e3, "raw_bound_ms": bound * 1e3,
            "raw_step_over_bound": raw_s / bound,
            "raw_bank_slots_failed_per_pass": self.failed,
            "raw_bank_step_ms_all": [v * 1e3 for v in self.res["raw_step_s"]],
            "raw_h2d_ceiling_ms_all": [v * 1e3 for v in self.res["ceiling_step_s"]],
        }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[128, 1024])
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--host-steps", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--raw", action="store_true", help="add the raw-frame arms (uahn_filter_frame_raw, bare raw copy)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    from cuahn_vio_b200 import api, build, weights
    build.build()
    wfile = weights.synthetic_weights_file(0)
    name, power = gpu_info()
    rows = [run_size(api, wfile, S, a.frames, a.host_steps, a.rounds, a.raw) for S in a.sizes]
    line = json.dumps({"tool": "filter_bench", "gpu": name, "power_limit": power, "imu_hz": HZ_IMU, "camera_hz": HZ_CAM,
                       "precision": "bf16", "variant": "prior3", "max_iter": 1, "results": rows})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
