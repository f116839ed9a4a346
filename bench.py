#!/usr/bin/env python
"""bench.py — UAHN image-pair inferences/sec on N B200 (BASELINE.json metric) + p50 batch-1 latency.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|fp32] [--dump-outputs DIR]

A "step" is one pass of the hot path (3-block UAHN with EKF prior: prior DLT, blocks 2,3 and the
uncertainty block 4, covariance transfer) over the workload of BASELINE.json configs[3]: 8192 synthetic pairs,
sharded by sequence over the N ranks (`sharding.shard_range`; strong scaling, the default) and run in
`uahn_infer_batch` calls of `--batch` (1024) pairs.  `--scaling weak` keeps `--batch` pairs per GPU per step instead.
N > 1 is launched by torchrun (one rank per GPU); pairs are independent, so ranks never exchange data on
the timed path — NCCL is used only for the start/stop barrier and the max-over-ranks of the device time.

The pairs are consecutive frames of synthetic sequences (AR(1) corner walk), each rank's shard one run of B + 1 frames.
Printed JSON (one line, rank 0): value = whole-job pairs/s with inputs resident in HBM, timed WITHOUT the per-stage
profiling events; roofline / stage split = a second pass with them; e2e = the same workload through the host-buffer
C-ABI call (pinned host inputs, H2D + D2H inside the timed region) with the bare-copy ceiling beside it;
config3_256_pairs = BASELINE.json configs[2] (256 pairs in one infer_batch) with its own roofline;
latency_batch1 = configs[1] in bf16 AND fp32; streaming_show_error = configs[4];
cpu_baseline = the reference's own TorchScript graphs (oracle/_ref) on the host cores (all threads, 1 thread, twins).

Every timed pass (value, the profiled pass, config3_256_pairs, e2e, its copy ceiling, e2e_independent_pairs) runs
exactly K = --steps steps; the JSON reports K with each.  A run with a few steps rests on a few calls (config3_256_pairs
on K calls of about 0.7 ms), so compare only runs with the same --steps; the default is 20.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "UAHN image-pair inferences/sec"
UNIT = "pairs/s"
# algorithmic work per pair, 3-block variant (SURVEY §8d / BASELINE.md §4)
CONV_MACS = 463_892_480
MC_GEMM_MACS = 2 * 16 * 5120 * 256
TOTAL_MACS = 505_982_976
WARP_BYTES = 573_440


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("UAHN_BENCH_PRECISION", "bf16"), choices=["bf16", "fp32"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): --total-pairs per step sharded by sequence over the ranks (BASELINE.json "
                         "configs[3]: 8192 pairs over 1/2/4/8 GPUs); weak: --batch pairs per GPU per step")
    ap.add_argument("--total-pairs", type=int, default=8192, help="pairs per step over ALL ranks (strong scaling)")
    ap.add_argument("--batch", type=int, default=1024, help="pairs per uahn_infer_batch call (and per GPU per step with --scaling weak)")
    ap.add_argument("--chunk", type=int, default=0, help="pairs per infer_batch call (0 = --batch)")
    ap.add_argument("--seq-pairs", type=int, default=64, help="pairs per synthetic sequence (the sharding unit)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (mean [pairs, 8], cov [pairs, 8, 8], float32, all ranks "
                         "in rank order) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


DUMP_BYTES = 60 << 20      # one dump stays below 64 MB


def dump_outputs(directory: str, arrays: dict):
    """Write {name: array with one row per pair} as directory/<name>.npy.  Above DUMP_BYTES every array keeps the same
    rows, a seeded sample in pair order, so two runs with the same arguments write the same pairs."""
    import numpy as np
    n = len(next(iter(arrays.values())))
    per_pair = sum(a[:1].nbytes for a in arrays.values())
    if n * per_pair > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // per_pair, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.dev = device_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------------------
REF_FILES = {("prior3", False): "traced_model_3_blocks_using_prior.pt", ("full", False): "traced_full_model.pt",
             ("prior3", True): "traced_model_3_blocks_using_prior_showError.pt", ("full", True): "traced_full_model_showError.pt"}


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def reference_runner(variant: str = "prior3", show_error: bool = False, threads: int | None = None):
    """Callable running ONE pair through the reference's CPU implementation + its description.

    kind "reference": the TorchScript trace of the unmodified reference model (oracle/_ref, built in the
    container by oracle/build_ref.py exactly as trace_model.py:36-46 does) executed by libtorch on the host cores, with
    the call protocol of HomographyNet.cpp:167-197 (inputs [1,1,224,320] x2 (+ [1,1,4,2] prior), forward, tuple unpack
    to float[8] / float[64]).  kind "port": the oracle restatement (same ATen ops) when the prebuilt trace is absent.
    """
    import torch
    from cuahn_vio_b200 import synthetic as S
    # all the host threads this process may use (torchrun exports OMP_NUM_THREADS=1 to its ranks)
    torch.set_num_threads(threads or host_threads())
    path = os.path.join(ROOT, "oracle", "_ref", REF_FILES[(variant, show_error)])
    prev, curr, _, prior = S.synthetic_batch(16)
    i1 = [torch.from_numpy(p).float().div(255.0).view(1, 1, 224, 320) for p in prev]
    i2 = [torch.from_numpy(c).float().div(255.0).view(1, 1, 224, 320) for c in curr]
    pr = [torch.from_numpy(p).view(1, 1, 4, 2) for p in prior]
    if os.path.exists(path):
        mod = torch.jit.load(path, map_location="cpu")
        mod.eval()

        def run(i):
            j = i % 16
            with torch.no_grad():
                out = mod(i1[j], i2[j], pr[j]) if variant == "prior3" else mod(i1[j], i2[j])
                return out[0].reshape(8).tolist(), out[1].reshape(64).tolist()      # HomographyNet.cpp:190-197
        kind = "reference"
    else:
        from oracle import uahn_oracle as O
        sd = S.synthetic_state_dict(0)
        masks = S.torch_dropout_masks(0)

        def run(i):
            j = i % 16
            return O.forward(i1[j], i2[j], sd, masks, pr[j] if variant == "prior3" else None, show_error)
        kind = "port"
    return run, kind, torch.get_num_threads()


def time_reference(seconds: float, variant: str = "prior3", show_error: bool = False, threads: int | None = None,
                   max_calls: int = 4000, warm: int = 20):
    run, kind, threads = reference_runner(variant, show_error, threads)
    for i in range(warm):
        run(i)
    lat = []
    t_end = time.perf_counter() + seconds
    i = 0
    while time.perf_counter() < t_end and i < max_calls:
        t0 = time.perf_counter()
        run(i)
        lat.append(time.perf_counter() - t0)
        i += 1
    total = sum(lat)
    name = REF_FILES[(variant, show_error)][:-3]
    return {"value": len(lat) / total, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{len(lat)} sequential batch-1 forwards of {name} after {warm} warm-up "
                      f"(libtorch CPU, {threads} threads, {os.cpu_count()} host cpus)",
            "mean_ms": 1e3 * total / len(lat), "p50_ms": 1e3 * statistics.median(lat),
            "p90_ms": 1e3 * sorted(lat)[int(0.9 * (len(lat) - 1))]}


def cpu_baseline_block(seconds: float):
    """BASELINE.md §3: the 3-block graph on all host threads (the headline cpu_baseline) + a 1-thread figure, the full
    cascade and the `_showError` twins (config 5), each a bounded sample."""
    import torch
    base = time_reference(seconds, "prior3")
    side = max(2.0, seconds / 4)
    detail = {"prior3_1_thread": time_reference(side, "prior3", threads=1, warm=3),
              "full": time_reference(side, "full", warm=5),
              "prior3_showError": time_reference(side, "prior3", True, warm=5),
              "full_showError": time_reference(side, "full", True, warm=5)}
    base["detail"] = {k: {kk: v[kk] for kk in ("value", "cores", "kind", "mean_ms", "p50_ms", "p90_ms", "sample")} for k, v in detail.items()}
    base["host"] = {"nproc": os.cpu_count(), "usable_threads": host_threads(), "torch": torch.__version__,
                    "cpu_model": next((l.split(":", 1)[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")), None)}
    torch.set_num_threads(host_threads())
    return base


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    K, W = args.steps, max(args.warmup, 1)
    run, kind, threads = reference_runner("prior3")
    per_step = 32          # bounded sample of the workload per step (the reference cannot batch)
    for i in range(W * 4):
        run(i)
    t0 = time.perf_counter()
    for s in range(K):
        for i in range(per_step):
            run(s * per_step + i)
    dt = time.perf_counter() - t0
    v = K * per_step / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * dt / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"3-block UAHN (traced_model_3_blocks_using_prior), {per_step} sequential batch-1 "
                                   f"pairs per step on host CPU: a bounded sample of the {args.total_pairs}-pair workload "
                                   "(the reference cannot batch)", "pairs_per_step": per_step, "variant": "prior3",
                       "torch": torch.__version__},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind,
                             "sample": f"{K} steps x {per_step} sequential batch-1 forwards, libtorch CPU, {threads} threads"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(device_index: int):
    """Pin this rank's CPU threads (and therefore its pinned host buffers, first-touch) to the NUMA node its GPU hangs off.
    With 8 ranks streaming 73 MB per step each, H2D copies that cross the socket interconnect cost end-to-end rate.
    Tries sysfs (PCI device -> numa_node) and then NVML's CPU affinity of the device.  Returns a record saying which
    source worked, or why none did (a VM without NUMA information reports node -1 everywhere)."""
    rec = {"node": None, "cpus": None, "source": None, "why": None}
    why = []
    try:
        import torch
        pr = torch.cuda.get_device_properties(device_index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node >= 0:
            cpus = set()
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
            cpus &= os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
                rec.update(node=node, cpus=len(cpus), source="sysfs")
                return rec
            why.append(f"sysfs node {node} has no usable cpus")
        else:
            why.append(f"sysfs numa_node of {bdf} is {node}")
    except Exception as e:   # noqa: BLE001
        why.append(f"sysfs: {type(e).__name__}: {e}")
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1} & os.sched_getaffinity(0)
        if cpus and len(cpus) < len(os.sched_getaffinity(0)):
            os.sched_setaffinity(0, cpus)
            rec.update(cpus=len(cpus), source="nvml cpu affinity")
            try:
                rec["node"] = int(pynvml.nvmlDeviceGetNumaNodeId(h))
            except Exception:   # noqa: BLE001
                pass
            return rec
        why.append(f"nvml affinity covers {len(cpus)} of {len(os.sched_getaffinity(0))} usable cpus (no restriction)")
    except Exception as e:   # noqa: BLE001
        why.append(f"nvml: {type(e).__name__}: {e}")
    rec["why"] = "; ".join(why)
    return rec


# ---------------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from cuahn_vio_b200 import api, build, synthetic as S, weights
    from cuahn_vio_b200.sharding import reduce_max_ms, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else {"node": None, "source": None, "why": "single rank: not bound"}
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()
    wfile = weights.synthetic_weights_file(0)

    K, W = args.steps, max(args.warmup, 3)
    # ---- the shard of this rank (SURVEY §8e): contiguous blocks of whole sequences -----------------------------
    if args.scaling == "strong":
        n_seq = max(1, args.total_pairs // args.seq_pairs)
        lo, hi = shard_range(n_seq, rank, world)
        B = (hi - lo) * args.seq_pairs
        total_pairs = n_seq * args.seq_pairs
        if B == 0:
            raise SystemExit(f"bench.py: rank {rank} got an empty shard ({n_seq} sequences over {world} ranks)")
    else:
        B = args.batch
        total_pairs = world * B
    chunk = min(args.chunk or args.batch, B)
    FR = 224 * 320
    n_sets = 3 if B <= 2048 else 2                # rotate input sets: each (B+1) x 71 680 B of u8 frames; with the activations >> 126 MB L2
    # The workload (BASELINE.json configs[3], SURVEY §8d): pairs are consecutive frames of synthetic sequences whose
    # corner displacements follow a smooth AR(1) walk; this rank's shard is one run of B + 1 frames (a 65-frame sequence
    # replayed there and back, so consecutive frames always stay close), pair i = (frame i, frame i + 1).
    seq_frames, _, seq_prior = S.synthetic_sequence(65, seed=20240 + 1000 * rank)
    reps = (B + 64) // 65 + 1
    hf = np.ascontiguousarray(np.concatenate([seq_frames, seq_frames[::-1]] * reps, 0)[:B + 1])
    hprior = np.ascontiguousarray(np.concatenate([seq_prior, -seq_prior[::-1]] * reps, 0)[:B].reshape(B, 8))
    stream = torch.cuda.Stream(dev)      # non-default stream shared by torch events and the library's launches
    torch.cuda.set_stream(stream)
    net = api.Uahn(wfile, "prior3", show_error=False, precision=args.precision, device=local, max_batch=chunk,
                   stream=stream.cuda_stream)
    sets = []
    for s in range(n_sets):
        roll = s * 7
        sets.append((torch.from_numpy(np.roll(hf, roll, 0)).to(dev), torch.from_numpy(np.roll(hprior, roll, 0)).to(dev)))
    mean = torch.empty(B, 8, device=dev)
    cov = torch.empty(B, 64, device=dev)
    first0 = rank * B if args.scaling == "weak" else lo * args.seq_pairs      # global index of this shard's first pair

    def run_resident(f, pr, n_pairs=B, call=chunk, base=0):
        for o in range(0, n_pairs, call):
            n = min(call, n_pairs - o)
            # prev = frames[o : o+n], curr = frames[o+1 : o+n+1]: the same buffer, one frame apart
            net.infer_batch_ptrs(n, f.data_ptr() + (base + o) * FR, f.data_ptr() + (base + o + 1) * FR, pr[base + o:].data_ptr(),
                                 mean[base + o:].data_ptr(), cov[base + o:].data_ptr(), seed=1, first_pair=first0 + base + o)

    def step(i):
        run_resident(*sets[i % n_sets])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed_device(fn, steps):
        """K steps between events on the launching stream, barrier + synchronize on both sides, max over ranks (ms)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for i in range(steps):
            fn(i)
        e1.record(stream)
        barrier()
        return reduce_max_ms(e0.elapsed_time(e1), dev)

    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.start()
    for i in range(W):
        step(i)
    # keep the GPU under the same load for ~0.6 s before the timed region so the 200 ms clock sampler sees it
    t_load = time.perf_counter()
    j = 0
    while time.perf_counter() - t_load < 0.6:
        step(j)
        j += 1
        torch.cuda.synchronize()
    # ---- pass 1: the headline value, no profiling events inside the timed region --------------------------------
    l0 = net.launch_count
    ms_max = timed_device(lambda i: step(W + i), K)
    launches = net.launch_count - l0
    # the last timed step's results, before the passes below overwrite them
    last = {"mean": mean.cpu().numpy(), "cov": cov.view(B, 8, 8).cpu().numpy()} if args.dump_outputs else None
    value = total_pairs * K / (ms_max * 1e-3)
    clk = clocks.stop() if clocks else None
    # ---- pass 2: per-stage CUDA events (uahn_profile_*) for the roofline and the stage split ----------------------
    net.profile_enable(True)
    ms_prof = timed_device(lambda i: step(W + i), K)
    prof_ms, prof_cnt = net.profile_read()
    net.profile_enable(False)

    # ---- BASELINE.json configs[2]: 256 pairs in ONE infer_batch on one GPU, with its own roofline ------------------
    cfg3 = None
    if world == 1 and B >= 256 + 7 * 16:
        n3 = 256
        f0, p0 = sets[0]
        for i in range(W + 5):
            run_resident(f0, p0, n3, n3, base=(i % 8) * 16)
        ms3 = timed_device(lambda i: run_resident(*sets[i % n_sets], n3, n3, base=(i % 8) * 16), K)
        net.profile_enable(True)
        timed_device(lambda i: run_resident(*sets[i % n_sets], n3, n3, base=(i % 8) * 16), K)
        p3, c3 = net.profile_read()
        net.profile_enable(False)
        cfg3 = {"pairs_per_call": n3, "ms_per_call": ms3 / K, "value": n3 * K / (ms3 * 1e-3), "unit": UNIT,
                "stage_ms_per_call": {"warp_concat_pool": p3[0] / K, "conv_stacks": p3[1] / K, "mc_head_gemm": p3[2] / K,
                                      "fc_dlt_mc_small": p3[3] / K},
                "launches_per_call": int(sum(int(v) for v in c3) // K)}

    # ---- e2e: host buffers through the C ABI, copies inside the timed region ---------------------------
    # The call a streaming user makes for a sequence: uahn_submit_sequence from pinned host memory — every frame crosses
    # PCIe once, the H2D of step i+1 overlaps the forward of step i on an internal copy stream, results come back to
    # pinned host memory.  Every step's inputs and results cross PCIe inside the timed region.
    pfr = torch.from_numpy(hf).pin_memory()
    ppr = torch.from_numpy(hprior).pin_memory()
    hmean = torch.empty(B, 8).pin_memory()
    hcov = torch.empty(B, 64).pin_memory()

    def step_e2e(i):
        for o in range(0, B, chunk):
            n = min(chunk, B - o)
            net.submit_sequence_ptrs(n + 1, pfr.data_ptr() + o * FR, ppr[o:].data_ptr(), hmean[o:].data_ptr(),
                                     hcov[o:].data_ptr(), seed=1, first_pair=first0 + o)

    def timed(fn, steps):
        for i in range(2):
            fn(i)
        net.wait()
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            fn(i)
        net.wait()
        torch.cuda.synchronize()
        return total_pairs * steps / (reduce_max_ms(1e3 * (time.perf_counter() - t0), dev) * 1e-3)

    e2e_value = timed(step_e2e, K)      # the last forward (not hidden behind a following copy) is part of the timed region
    # results of the two paths must agree (same frames, priors, seed and pair indices)
    run_resident(torch.from_numpy(hf).to(dev), torch.from_numpy(hprior).to(dev))
    torch.cuda.synchronize()
    same = bool(torch.equal(hmean.to(dev), mean))
    calls_per_step = (B + chunk - 1) // chunk
    h2d_step = (B + calls_per_step) * 71680 + B * 32

    # ---- the bare-copy ceiling of the same H2D stream: all ranks at once, nothing but cudaMemcpyAsync of the step's frames
    # from the same pinned buffer (what bounds e2e when the host side is the limit) -------------------------------------
    dstage = torch.empty((B + 1) * FR, dtype=torch.uint8, device=dev)
    copy_stream = torch.cuda.Stream(dev)

    def copy_step(i):
        with torch.cuda.stream(copy_stream):
            dstage.copy_(pfr.view(-1), non_blocking=True)

    def timed_copy(steps):
        for i in range(2):
            copy_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            copy_step(i)
        copy_stream.synchronize()
        return reduce_max_ms(1e3 * (time.perf_counter() - t0), dev) * 1e-3
    t_copy = timed_copy(K)
    h2d_gbs_all = world * (B + 1) * FR * K / t_copy / 1e9
    ceiling_pairs = total_pairs * K / t_copy
    del dstage

    # ---- the same pairs submitted as INDEPENDENT pairs (uahn_submit_batch): prev and curr arrays are separate host
    # buffers, so every frame crosses PCIe twice ------------------------------------------------------------------------
    php = torch.from_numpy(np.ascontiguousarray(hf[:-1])).pin_memory()
    phc = torch.from_numpy(np.ascontiguousarray(hf[1:])).pin_memory()

    def step_pairs(i):
        for o in range(0, B, chunk):
            n = min(chunk, B - o)
            net.submit_batch_ptrs(n, php[o:].data_ptr(), phc[o:].data_ptr(), ppr[o:].data_ptr(), hmean[o:].data_ptr(),
                                  hcov[o:].data_ptr(), seed=1, first_pair=first0 + o)
    e2e_pairs_value = timed(step_pairs, K)

    if last is not None:
        parts = [last]
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, last)
        if rank == 0:
            dump_outputs(args.dump_outputs, {k: np.concatenate([p[k] for p in parts]) for k in last})

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    # DRAM traffic of the conv group from the committed ncu --set full capture of this workload (per pair)
    traffic, traffic_src = None, None
    for name in ("r02_conv_traffic.json", "r01_conv_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath) and args.precision == "bf16":
            tj = json.load(open(tpath))
            traffic = tj["conv_group_dram_bytes_per_step"] / tj["pairs"] * chunk
            traffic_src = f"committed ncu capture profiles/{name} ({tj['pairs']} pairs per call), not measured in this run"
            break
    peak = peaks["bf16_tflops_sustained"]

    def tensor_roofline(conv_ms_per_call, pairs_per_call, calls):
        flops = 2.0 * CONV_MACS * pairs_per_call
        ach = flops / (conv_ms_per_call * 1e-3) / 1e12 if conv_ms_per_call > 0 else 0.0
        return {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if peak else None,
                "kernel": "conv implicit-GEMM group (15 launches per call: blocks 2,3,4; fused 7x7+5x5 fronts of blocks 3,4)",
                "algorithmic_flops_per_launch_group": flops, "ms_per_launch_group": conv_ms_per_call,
                "launch_groups_per_step": calls,
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']})"}

    conv_ms_per_call = prof_ms[1] / K / calls_per_step
    warp_ms_per_step = prof_ms[0] / K
    roof = tensor_roofline(conv_ms_per_call, chunk, calls_per_step)
    roof.update({"traffic": traffic, "traffic_source": traffic_src,
                 "hbm_frac_conv_group": (traffic / (conv_ms_per_call * 1e-3) / 1e9 / peaks["hbm_gbs"]) if traffic and conv_ms_per_call > 0 else None,
                 "ms_per_step": prof_ms[1] / K, "timed_in": f"second pass of {K} steps with per-stage CUDA events on the launching stream"})
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": f"3-block UAHN (traced_model_3_blocks_using_prior) over {total_pairs} synthetic pairs per step, "
                               f"sharded by sequence ({args.seq_pairs} pairs each) over {world} GPU: {B} pairs per GPU per step "
                               f"in infer_batch calls of {chunk} (pairs = consecutive frames of synthetic AR(1) sequences)",
                   "variant": "prior3", "total_pairs_per_step": total_pairs, "pairs_per_gpu_per_step": B, "pairs_per_call": chunk,
                   "precision": args.precision,
                   "weights": "synthetic seed 0 (reference checkpoint not shipped; bf16 tolerances are validated on these weights only)",
                   "l2": f"inputs rotate over {n_sets} resident sets of {(B + 1) * 71680 / 1e6:.0f} MB; with the "
                         f"{2.0 * chunk:.0f} MB of activations per call the working set is far beyond the 126 MB L2",
                   "parallelism": f"independent pairs, {world} shard(s) from sharding.shard_range, no data-path collective",
                   "host_numa_binding_rank0": numa},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_step,
                "d2h_bytes_per_step": B * 72 * 4, "steps": K, "matches_device_path": same,
                "what": "uahn_submit_sequence + uahn_wait from pinned host buffers: the shard's consecutive frames, each "
                        "uploaded once per step (per-GPU byte counts)",
                "h2d_ceiling": {"pairs_per_s": ceiling_pairs, "h2d_gbs_all_ranks": h2d_gbs_all,
                                "what": "bare cudaMemcpyAsync of the same frames from the same pinned buffers, all ranks "
                                        "concurrently, no kernels"},
                "h2d_ceiling_frac": e2e_value / ceiling_pairs if ceiling_pairs else None,
                "bound": "device (resident rate)" if value <= ceiling_pairs else "host-to-device copy"},
        "e2e_independent_pairs": {"value": e2e_pairs_value, "unit": UNIT, "h2d_bytes_per_step": B * (2 * 71680 + 32),
                                  "d2h_bytes_per_step": B * 72 * 4, "steps": K,
                                  "what": "the same pairs through uahn_submit_batch with separate prev / curr host arrays "
                                          "(every frame crosses PCIe twice)"},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": roof,
        "profiled_pass": {"steps": K, "ms_per_step": ms_prof / K, "note": "the pass the stage split and the roofline come from; "
                          "`value` is from the pass without profiling events"},
        "stage_ms_per_step": {"warp_concat_pool": warp_ms_per_step, "conv_stacks": prof_ms[1] / K,
                              "mc_head_gemm": prof_ms[2] / K, "fc_dlt_mc_small": prof_ms[3] / K},
        "stage_launches_per_step": {k: int(v // K) for k, v in zip(("warp", "conv", "mc_gemm", "small"), prof_cnt)},
        "hbm": {"kernel": f"warp+concat+pool (3 texture-gather launches + the cell-array fill per call, {calls_per_step} call(s) per step; "
                          "the fill's time is inside, only the 3 warps are credited)",
                "algorithmic_bytes_per_step": 3 * WARP_BYTES * B,
                "achieved_gbs": (3 * WARP_BYTES * B / (warp_ms_per_step * 1e-3) / 1e9) if warp_ms_per_step > 0 else None,
                "peak_gbs": peaks["hbm_gbs"], "layout": "fp32 in/out as in the reference (573 440 B per warp)"},
    }
    if line["hbm"]["achieved_gbs"]:
        line["hbm"]["frac"] = line["hbm"]["achieved_gbs"] / peaks["hbm_gbs"]
    if cfg3:
        r3 = tensor_roofline(cfg3["stage_ms_per_call"]["conv_stacks"], cfg3["pairs_per_call"], 1)
        w3 = cfg3["stage_ms_per_call"]["warp_concat_pool"]
        cfg3["roofline"] = r3
        cfg3["hbm"] = {"achieved_gbs": 3 * WARP_BYTES * cfg3["pairs_per_call"] / (w3 * 1e-3) / 1e9 if w3 > 0 else None,
                       "peak_gbs": peaks["hbm_gbs"]}
        if cfg3["hbm"]["achieved_gbs"]:
            cfg3["hbm"]["frac"] = cfg3["hbm"]["achieved_gbs"] / peaks["hbm_gbs"]
        cfg3["what"] = "BASELINE.json configs[2]: 3-block UAHN, 256 synthetic pairs in ONE uahn_infer_batch_device call, inputs resident"
        line["config3_256_pairs"] = cfg3

    # ---- p50 batch-1 latency (BASELINE.json configs[1]: full cascade, no prior; fp32 validation and bf16 modes) ----
    if not args.no_latency and world == 1:
        lat = {}
        for precision in ("bf16", "fp32"):
            for variant in ("full", "prior3"):
                with api.Uahn(wfile, variant, precision=precision, device=local, max_batch=1) as n1:
                    n1.load_image(hf[0], 0.0)
                    n1.load_image(hf[1], 1.0)
                    pr = hprior[0].reshape(8).astype(np.float64) if variant == "prior3" else None
                    for i in range(100):
                        n1.infer(pr, seed=1, pair_index=i)
                    ts = []
                    for i in range(2000 if precision == "bf16" else 500):
                        t0 = time.perf_counter()
                        n1.infer(pr, seed=1, pair_index=i)
                        ts.append(time.perf_counter() - t0)
                    ts.sort()
                    lat[f"{variant}_{precision}"] = {
                        "p50_ms": 1e3 * ts[len(ts) // 2], "p90_ms": 1e3 * ts[int(len(ts) * 0.9)],
                        "p99_ms": 1e3 * ts[int(len(ts) * 0.99)], "calls": len(ts), "kernels_per_call": None,
                        "what": "uahn_infer wall clock: prior H2D + forward (one CUDA graph) + 72-float D2H, frames resident"}
                    l1 = n1.launch_count
                    n1.infer(pr, seed=1, pair_index=0)
                    lat[f"{variant}_{precision}"]["kernels_per_call"] = int(n1.launch_count - l1)
        lat["full"], lat["prior3"] = lat["full_bf16"], lat["prior3_bf16"]        # (round-1 key names)
        line["latency_batch1"] = lat
        # ---- BASELINE.json configs[4]: showError variant streamed frame by frame (full cascade + covariance +
        # photometric-error map), frame k's `curr` reused as frame k+1's `prev` on the device ---------------------
        n_stream = 2000
        sf, _, _ = S.synthetic_sequence(64, seed=777)
        with api.Uahn(wfile, "full", show_error=True, precision=args.precision, device=local, max_batch=1) as ns:
            ns.load_image(sf[0], 0.0)
            for i in range(1, 40):
                ns.load_image(sf[i % 64], float(i))
                ns.infer(None, seed=1, pair_index=i, want_error=True)
            ts = []
            t_all = time.perf_counter()
            for i in range(n_stream):
                j = i % 126
                f = sf[j] if j < 64 else sf[126 - j]                    # there-and-back over the 64 frames
                t0 = time.perf_counter()
                ns.load_image(f, float(i))                              # 71 680 B H2D
                ns.infer(None, seed=1, pair_index=i, want_error=True)    # forward + 72 floats + 71 680 B u8 map D2H
                ts.append(time.perf_counter() - t0)
            t_all = time.perf_counter() - t_all
            ts.sort()
            line["streaming_show_error"] = {
                "frames": n_stream, "frames_per_s": n_stream / t_all, "p50_ms": 1e3 * ts[len(ts) // 2],
                "p90_ms": 1e3 * ts[int(len(ts) * 0.9)], "p99_ms": 1e3 * ts[int(len(ts) * 0.99)],
                "h2d_bytes_per_frame": 71680, "d2h_bytes_per_frame": 72 * 4 + 71680,
                "what": "full cascade + covariance + photometric-error map per frame through uahn_load_image + uahn_infer "
                        "(CUDA-graph replay), synthetic AR(1) sequence"}

    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline_block(args.cpu_seconds)
    else:
        line["cpu_baseline"] = None
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
