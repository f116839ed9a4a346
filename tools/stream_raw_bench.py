"""Pairs/s of the pipelined sequence entry point fed raw camera frames (uahn_submit_sequence_raw) against its ceiling.

A bf16 prior3 handle with max_batch 1024 and the uahn_undistort_init_maps maps of one fixture camera; every call
submits one sequence of 1025 frames (1024 pairs) from pinned host memory, two buffers used in turn.  One timed step is
--calls back-to-back submissions and one uahn_wait (>= 8192 pairs); the arms alternate step by step, --steps timed
steps each after --warmup untimed ones:
  raw       uahn_submit_sequence_raw: 640x480 u8 raw frames (synthetic_raw_frame, a few unique ones tiled), each
            call's upload + batched remap + forward
  undist    uahn_submit_sequence on the same frames undistorted beforehand (73.5 MB per call instead of 315 MB)
  copy      a bare pinned cudaMemcpyAsync of the same raw bytes per call: the ceiling of the raw arm
  forward   the forward alone on device-resident frames (uahn_infer_batch_device), CUDA events on the handle's stream
The remap kernel's time per call comes from the handle's CUDA-event profile (uahn_profile_*, category 0 holds the
warps and the remap): category 0 of raw calls minus that of undistorted calls on the same frames.
raw_over_bound = raw call time / max(copy time, forward + remap), every term from the same run: 1.0 means the raw
call takes no longer than the slower of its upload and its compute.  A step ends with its last call's remap and forward,
which no further upload hides: (forward + remap) / --calls of each raw call.  Prints one JSON line; --out FILE also
writes it to FILE.

  python tools/stream_raw_bench.py [--steps 20] [--warmup 3] [--calls 8] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from filter_bench import gpu_info                # noqa: E402  (device name and power limit from nvidia-smi)
PAIRS = 1024                                     # pairs per call = max_batch
RAW_ROWS, RAW_COLS, RAW_UNIQUE = 480, 640, 8
RAW_CAMERA = "uzhfpv_indoor_fwd"                 # a fisheye camera of tests/golden/preproc.npz
IMG = 224 * 320
PROFILE_CALLS = 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps per arm first")
    ap.add_argument("--calls", type=int, default=8, help="submissions of 1024 pairs per step")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if a.calls * PAIRS < 8192:
        ap.error("a step must hold at least 8192 pairs")
    import torch
    from cuahn_vio_b200 import api, build, weights
    from cuahn_vio_b200 import synthetic as Syn
    build.build()
    name, power = gpu_info()
    golden = np.load(os.path.join(ROOT, "tests", "golden", "preproc.npz"))
    maps = api.undistort_init_maps(bool(golden[f"{RAW_CAMERA}_fisheye"]), golden[f"{RAW_CAMERA}_k"],
                                   golden[f"{RAW_CAMERA}_d"])
    net = api.Uahn(weights.synthetic_weights_file(0), "prior3", precision="bf16", max_batch=PAIRS)
    net.set_undistort_maps(RAW_ROWS, RAW_COLS, *maps)
    uniq = np.stack([Syn.synthetic_raw_frame(900 + i, RAW_ROWS, RAW_COLS) for i in range(RAW_UNIQUE)])
    uniq_und = np.stack([net.stage_undistort(f) for f in uniq])
    nf = PAIRS + 1

    def pinned(shape, dtype):
        return torch.empty(shape, dtype=dtype, pin_memory=True)

    # buffer j, frame k shows unique frame (k + j) % RAW_UNIQUE: consecutive frames differ
    raw = [pinned((nf, RAW_ROWS, RAW_COLS), torch.uint8) for _ in range(2)]
    und = [pinned((nf, 224, 320), torch.uint8) for _ in range(2)]
    for j in range(2):
        idx = (np.arange(nf) + j) % RAW_UNIQUE
        raw[j].numpy()[:] = uniq[idx]
        und[j].numpy()[:] = uniq_und[idx]
    prior = pinned((PAIRS, 8), torch.float32)
    prior.numpy()[:] = Syn.tiled_batch(PAIRS, unique=64)[3].reshape(PAIRS, 8)
    mean = [pinned((PAIRS, 8), torch.float32) for _ in range(2)]
    cov = [pinned((PAIRS, 64), torch.float32) for _ in range(2)]
    d_frames = und[0].cuda()
    d_prior, d_mean, d_cov = prior.cuda(), torch.empty((PAIRS, 8), device="cuda"), torch.empty((PAIRS, 64), device="cuda")
    d_raw = torch.empty((nf, RAW_ROWS, RAW_COLS), dtype=torch.uint8, device="cuda")
    copy_stream = torch.cuda.Stream()
    net_stream = torch.cuda.ExternalStream(net.stream)
    pair = [0]

    def submit_raw(i):
        net.submit_sequence_raw_ptrs(nf, raw[i % 2].data_ptr(), RAW_COLS, prior.data_ptr(), mean[i % 2].data_ptr(),
                                     cov[i % 2].data_ptr(), seed=1, first_pair=pair[0])
        pair[0] += PAIRS

    def submit_und(i):
        net.submit_sequence_ptrs(nf, und[i % 2].data_ptr(), prior.data_ptr(), mean[i % 2].data_ptr(), cov[i % 2].data_ptr(),
                                 seed=1, first_pair=pair[0])
        pair[0] += PAIRS

    def host_step(submit):
        net.wait()
        t = time.perf_counter()
        for i in range(a.calls):
            submit(i)
        net.wait()
        return (time.perf_counter() - t) / a.calls

    def event_step(stream, body):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record()
            for i in range(a.calls):
                body(i)
            e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3 / a.calls

    def copy_body(i):
        d_raw.copy_(raw[i % 2], non_blocking=True)             # cudaMemcpyAsync from pinned memory

    def forward_body(i):
        net.infer_batch_ptrs(PAIRS, d_frames.data_ptr(), d_frames.data_ptr() + IMG, d_prior.data_ptr(), d_mean.data_ptr(),
                             d_cov.data_ptr(), seed=1, first_pair=i * PAIRS)

    arms = {"raw": lambda: host_step(submit_raw), "undist": lambda: host_step(submit_und),
            "copy": lambda: event_step(copy_stream, copy_body), "forward": lambda: event_step(net_stream, forward_body)}
    for _ in range(a.warmup):
        for f in arms.values():
            f()
    res = {k: [] for k in arms}
    for _ in range(a.steps):
        for k, f in arms.items():
            res[k].append(f())

    # remap kernel time per call: category 0 (warps + remap) of raw calls minus that of undistorted calls, alternated
    cat0 = {"raw": [], "undist": []}
    launches = {"raw": [], "undist": []}
    for _ in range(2):
        for k, submit in (("raw", submit_raw), ("undist", submit_und)):
            net.profile_enable(True)
            for i in range(PROFILE_CALLS):
                submit(i)
                net.wait()
            ms, cnt = net.profile_read()
            net.profile_enable(False)
            cat0[k].append(ms[0] / PROFILE_CALLS)
            launches[k].append(int(cnt[0]) / PROFILE_CALLS)
    remap_ms = (np.mean(cat0["raw"]) - np.mean(cat0["undist"]))
    net.close()

    med = {k: float(np.median(v)) for k, v in res.items()}
    remap_s = remap_ms / 1e3
    bound = max(med["copy"], med["forward"] + remap_s)
    raw_bytes = nf * RAW_ROWS * RAW_COLS
    remap_bytes = nf * (RAW_ROWS * RAW_COLS + IMG)              # raw frames read + undistorted frames written
    line = json.dumps({
        "tool": "stream_raw_bench", "gpu": name, "power_limit": power, "precision": "bf16", "variant": "prior3",
        "max_batch": PAIRS, "pairs_per_call": PAIRS, "calls_per_step": a.calls, "steps": a.steps, "warmup": a.warmup,
        "raw_rows": RAW_ROWS, "raw_cols": RAW_COLS, "camera": RAW_CAMERA, "raw_bytes_per_call": raw_bytes,
        "raw_pairs_per_s": PAIRS / med["raw"], "undistorted_pairs_per_s": PAIRS / med["undist"],
        "copy_ceiling_pairs_per_s": PAIRS / med["copy"], "forward_pairs_per_s": PAIRS / med["forward"],
        "raw_ms_per_call": med["raw"] * 1e3, "undistorted_ms_per_call": med["undist"] * 1e3,
        "copy_ms_per_call": med["copy"] * 1e3, "copy_GB_per_s": raw_bytes / med["copy"] / 1e9,
        "forward_ms_per_call": med["forward"] * 1e3, "remap_kernel_ms_per_call": remap_ms,
        "remap_GB_per_s": remap_bytes / remap_s / 1e9 if remap_s > 0 else None,
        "warp_stage_ms_per_call": {k: [float(x) for x in v] for k, v in cat0.items()},
        "warp_stage_launches_per_call": {k: v for k, v in launches.items()},
        "bound_ms_per_call": bound * 1e3, "serialised_ms_per_call": (med["copy"] + med["forward"] + remap_s) * 1e3,
        "raw_over_bound": med["raw"] / bound,
        "all_ms": {k: [v * 1e3 for v in vs] for k, vs in res.items()},
    })
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
