#!/usr/bin/env python
"""bench.py -- candidate windows/s of the PICO cascade scan (RunCascade, core/pigo.go:212-258) on 1080p frames.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` (N>1 under torchrun, one rank per GPU) prints ONE JSON
line on rank 0.  A "step" = one pass of the hot path (scan of every (scale,row,col) window + emission-order finalize,
then for N>1 the single NCCL gather of the detection slices) over one batch of synthetic frames.

Workload = BASELINE.json configs[2]: batch of 256 x 1920x1080 uint8 frames PER GPU (weak scaling), facefinder cascade,
reference test parameters MinSize 20 / MaxSize 1000 / ShiftFactor 0.2 / ScaleFactor 1.1 (core/pigo_test.go:44-50),
894,448 windows per frame.  configs[1] (one 1080p frame) is a pure latency case (one frame is ~6 us of issue work);
it is measured too and reported under "single_frame", but the metric -- a throughput -- is quoted on the batch.
Inputs (530 MB per GPU) exceed the 126 MB L2, so no L2 flush is needed between iterations.

  value     : windows/s, frames already resident in HBM, timed with CUDA events on the launching stream, max over ranks
  e2e       : same metric through the public host API (pigo_run_cascade_batch with HOST buffers): pinned H2D of the
              frames and D2H of counts+detections inside the timed region
  roofline  : the scan kernel's ALGORITHMIC bytes (frames*rows*dim + 16*n_det + cascade bytes; SURVEY.md section 8d)
              over its CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs.  This path is issue/latency bound,
              NOT HBM bound (2.3 B/window): the fraction is reported as it is.
  cpu_baseline / --impl reference : the CPU restatement of the reference (oracle/, kind "port" -- the reference is Go
              and no Go toolchain exists here) on the host cores, frame-parallel, bounded sample.

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0's frame-ordered result) as float32 .npy
files, so that two builds can be compared output for output: the frames are seeded, identical from run to run.
  counts.npy       [frames]             detections found per frame (may exceed the 1024 slots of a frame)
  detections.npy   [frames, 1024, 4]    (row, col, scale, score) per slot, zero past the frame's count
  frame_index.npy  [frames]             which frames of the step these are (a seeded sample when all would exceed 64 MB)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

ROWS, COLS = 1080, 1920
PARAMS = (20, 1000, 0.2, 1.1)
CASCADE_BYTES = 241488  # codes 119,808 + leaves 119,808 + thresholds 1,872 (SURVEY.md section 7.2)


def make_frames(nframes: int, seed0: int) -> np.ndarray:
    """Deterministic content classes U/S/F (SURVEY.md section 8d): 24 base frames, the rest are circular shifts."""
    from pigo_b200 import synth
    nbase = min(nframes, 24)
    base = synth.make_batch(nbase, ROWS, COLS, "USF", seed0=seed0)
    out = np.empty((nframes, ROWS, COLS), dtype=np.uint8)
    for i in range(nframes):
        b = base[i % nbase]
        k = i // nbase
        out[i] = b if k == 0 else np.roll(b, (17 * k, 29 * k), axis=(0, 1))
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_run(frames: np.ndarray, steps: int, warmup: int, nthreads: int):
    """Times the CPU restatement (oracle) frame-parallel on `nthreads` host threads; returns (windows/s, ms/step)."""
    import oracle_lib as O
    import pigo_b200
    face = O.OracleFace(pigo_b200.load_cascade("facefinder"))
    W = O.count_windows(ROWS, COLS, *PARAMS)
    for _ in range(warmup):
        face.run_cascade_batch(frames, ROWS, COLS, COLS, *PARAMS, 0.0, cap_per_frame=2048, nthreads=nthreads)
    t0 = time.perf_counter()
    for _ in range(steps):
        face.run_cascade_batch(frames, ROWS, COLS, COLS, *PARAMS, 0.0, cap_per_frame=2048, nthreads=nthreads)
    dt = time.perf_counter() - t0
    return W * frames.shape[0] * steps / dt, dt / steps * 1e3


def host_info() -> dict:
    """CPU model / thread count of this box and whether a Go toolchain exists (it decides `kind`: "reference" needs Go)."""
    model = None
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    try:
        gov = subprocess.run(["go", "version"], capture_output=True, text=True, timeout=10).stdout.strip() or None
    except Exception:
        gov = None
    try:
        load = os.getloadavg()[0]
    except OSError:
        load = None
    return {"cpu_model": model, "logical_cpus": os.cpu_count(), "go_version": gov, "loadavg_1m": load}


def cpu_sample_frames(nthreads: int, requested: int) -> int:
    """Frames per CPU step: at least 4 per thread so that every core works and the dynamic frame queue evens out the
    class-dependent cost (round 1 fed 64 frames to 128 threads: half the cores idle)."""
    return requested or max(16, min(512, 4 * nthreads))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname: str, dets: np.ndarray, counts: np.ndarray):
    """dets: [frames, cap, 4] int32 (row, col, scale, float32 bits of the score), counts: [frames] int32; see --dump-outputs."""
    nf, cap = dets.shape[:2]
    keep = max(1, DUMP_LIMIT_BYTES // (cap * 16 + 8))
    idx = np.arange(nf) if nf <= keep else np.sort(np.random.default_rng(0).choice(nf, keep, replace=False))
    d, c = dets[idx], counts[idx]
    out = np.empty(d.shape, dtype=np.float32)
    out[..., :3] = d[..., :3]
    out[..., 3] = d.view(np.float32)[..., 3]
    out[np.arange(cap)[None, :] >= np.minimum(c, cap)[:, None]] = 0   # slots past the count hold nothing a caller may read
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "detections.npy"), out)
    np.save(os.path.join(dirname, "counts.npy"), c.astype(np.float32))
    np.save(os.path.join(dirname, "frame_index.npy"), idx.astype(np.float32))


def _claim_stdout():
    """The contract is ONE JSON line on stdout: everything else any library writes to fd 1 (NCCL prints its version
    banner there at WARN level, torchrun children inherit the fd) is sent to stderr; the line itself goes to the saved fd."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _emit(fd, obj):
    sys.stdout.flush()
    os.write(fd, (json.dumps(obj) + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=256, help="frames per GPU per step")
    ap.add_argument("--cpu-sample-frames", type=int, default=0, help="frames in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[3] / configs[4] blocks (developer runs)")
    ap.add_argument("--pipeline-frames", type=int, default=64, help="frames per GPU per step of the configs[4] pipeline block")
    ap.add_argument("--opts", default="", help="developer sweeps: library options as name=value,... (default: none)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's detections to DIR/*.npy (see the module doc)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    out_fd = _claim_stdout()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    config = {"workload": "configs[2]: batch 256 x 1920x1080 synthetic grayscale frames per GPU (classes U/S/F), facefinder, "
                          "MinSize 20 MaxSize 1000 ShiftFactor 0.2 ScaleFactor 1.1, angle 0",
              "frames_per_gpu": args.frames, "windows_per_frame": 894448, "l2": "inputs (530 MB/GPU) larger than L2, no flush",
              "parallelism": f"frame-sharded dp{world}"}

    # ------------------------------------------------------------------ reference arm: the CPU path on host cores
    if args.impl == "reference":
        if rank != 0:
            return
        nthreads = ncores
        sample = cpu_sample_frames(nthreads, args.cpu_sample_frames)
        frames = make_frames(sample, 0)
        v1, _ = cpu_reference_run(frames[:min(sample, 3)], 1, 0, 1)
        v, ms = cpu_reference_run(frames, args.steps, max(args.warmup, 1), nthreads)
        config = dict(config, frames_per_step_cpu=sample, note="reference arm: `frames_per_step_cpu` frames of the same workload per "
                      "step on the host cores (the metric is a rate); frames_per_gpu is the GPU arm's batch")
        _emit(out_fd, {
            "impl": "reference", "metric": "candidate windows/s on 1080p frames", "value": v, "unit": "windows/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": "windows/s", "cores": nthreads, "kind": "port",
                             "sample": f"{sample} of the workload's 1080p frames per step, frame-parallel (dynamic queue) on {nthreads} "
                                       "threads (C -O2 restatement of core/pigo.go RunCascade; the Go reference cannot be built here)",
                             "single_thread_value": v1, "host": host_info()},
            "e2e": {"value": v, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0})
        return

    # ------------------------------------------------------------------ our arm
    import torch
    import pigo_b200
    from pigo_b200 import dist as pdist

    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "WARN"   # errors only (they land on stderr, see _claim_stdout)
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = local_rank if world > 1 else 0
    torch.cuda.set_device(dev)
    pigo_b200.init(dev)
    for kv in filter(None, args.opts.split(",")):
        pigo_b200.set_option(kv.split("=")[0], int(kv.split("=")[1]))
    clf = pigo_b200.NewPigo().Unpack(pigo_b200.load_cascade("facefinder"))
    W = pigo_b200.count_windows(ROWS, COLS, *PARAMS)
    nf = args.frames
    cap = 1024

    frames_host = make_frames(nf, seed0=1000 * rank)
    pinned = torch.from_numpy(frames_host).pin_memory()
    d_frames = pinned.to(f"cuda:{dev}", non_blocking=False)
    d_out = torch.zeros((nf, cap, 4), dtype=torch.int32, device=f"cuda:{dev}")
    d_cnt = torch.zeros(nf, dtype=torch.int32, device=f"cuda:{dev}")
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    st = stream.cuda_stream

    def step_device():
        """Returns what the step hands its caller: this rank's (dets, counts), or for N>1 the gathered lists on rank 0."""
        clf.run_cascade_batch_device(d_frames.data_ptr(), nf, ROWS * COLS, ROWS, COLS, COLS, *PARAMS, 0.0,
                                     d_out.data_ptr(), cap, d_cnt.data_ptr(), st)
        if world > 1:
            return pdist.gather_detections(d_out, d_cnt, dst=0)
        return [d_out], [d_cnt]

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{dev}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput ("value")
    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()   # nvidia-smi samples every 100 ms: started before the warm-up so the short timed region is covered
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    launches0 = pigo_b200.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        last = step_device()
    e1.record(stream)
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = pigo_b200.launch_count() - launches0
    dumped = None
    if args.dump_outputs and rank == 0:   # copied now: the passes below overwrite d_out / d_cnt
        dets_last, cnt_last = pdist.merge_gathered(*last, nf * world)
        dumped = (dets_last.cpu().numpy(), cnt_last.cpu().numpy())
    for _ in range(args.steps):   # keep the GPU under the same load while the sampler collects a few more points
        step_device()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms_step = ms_total / args.steps
    value = W * nf * world / (ms_step * 1e-3)
    ndet = int(d_cnt.clamp(max=cap).sum().item())

    # ---- roofline pass: per-kernel CUDA events inside the library (separate pass so the events do not perturb `value`)
    pigo_b200.set_option("timing", 1)
    for _ in range(args.steps):
        step_device()
    torch.cuda.synchronize()
    kt = {}
    for name in ("tiled", "gather", "deep", "finalize"):
        n = pigo_b200.get_option(f"t_{name}_n")
        ns = pigo_b200.get_option(f"t_{name}_ns")
        if n > 0:
            kt[name] = {"launches": int(n), "avg_us": ns / n / 1e3, "total_ms": ns / 1e6}
    pigo_b200.set_option("timing", 0)
    # useful-lane metric of the tile role: live lanes per walk iteration (dead lanes walk a dummy tree), one extra step
    pigo_b200.set_option("walk_stats", 1)
    step_device()
    torch.cuda.synchronize()
    wu, wi = pigo_b200.get_option("walk_useful"), pigo_b200.get_option("walk_iters")
    pigo_b200.set_option("walk_stats", 0)
    lanes = {"live_lanes_per_tile_walk_iteration": (wu / wi) if wi > 0 else None, "tile_role_tree_walks_per_step": int(wu),
             "tile_role_walk_iterations_per_step": int(wi)}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
    dom = max(kt.items(), key=lambda kv: kv[1]["total_ms"]) if kt else None
    roofline = None
    if dom:
        # One launch of the dominant kernel (the fused scan kernel, "tiled") covers one pipeline group of `sub_batch`
        # frames: algorithmic bytes per launch = its frames once + its share of the detections + the cascade once.
        launches_per_step = dom[1]["launches"] / args.steps
        frames_per_launch = nf / launches_per_step
        alg_bytes = frames_per_launch * ROWS * COLS + 16 * ndet / launches_per_step + CASCADE_BYTES
        scan_ms = sum(v["total_ms"] for k, v in kt.items() if k != "finalize") / args.steps
        launch_ms = dom[1]["avg_us"] / 1e3
        achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
        traffic = None
        traffic_src = None
        for name in ("traffic_r02.json", "traffic_r01.json"):
            try:   # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from the committed ncu --set full capture
                tr = json.load(open(os.path.join(ROOT, "profiles", name)))
                if tr.get("kernel") == dom[0]:
                    same = tr["frames_per_launch"] == frames_per_launch
                    traffic = tr["dram_bytes_per_launch"] * (1.0 if same else frames_per_launch / tr["frames_per_launch"])
                    traffic_src = f"profiles/{name}: ncu dram bytes of one captured launch of {tr['frames_per_launch']} frames" + \
                        ("" if same else ", scaled by frames per launch")
                    break
            except Exception:
                pass
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "kernel": dom[0], "kernel_launch_ms": launch_ms, "frames_per_launch": frames_per_launch,
                    "scan_kernels_ms_per_step": scan_ms, "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                    "traffic_note": traffic_src,
                    "kernels": kt, "tile_role_lanes": lanes, "note": "path is issue/latency/L2-transaction bound (2.3 algorithmic B/window), not HBM "
                    "bound; see DESIGN.md"}

    # ---- end to end through the host API: pinned H2D of the frames + D2H of counts and detections every step
    out_h = np.zeros((nf, cap), dtype=pigo_b200.DET_DTYPE)
    cnt_h = np.zeros(nf, dtype=np.int32)
    L = pigo_b200.lib()

    def step_host():
        rc = L.pigo_run_cascade_batch(clf._h, pinned.data_ptr(), nf, ROWS * COLS, ROWS, COLS, COLS, PARAMS[0], PARAMS[1],
                                      PARAMS[2], PARAMS[3], 0.0, out_h.ctypes.data, cap, cnt_h.ctypes.data, 0, None)
        if rc != 0:
            raise RuntimeError(L.pigo_last_error().decode())
    e2e_steps = max(2, min(args.steps, 5))
    step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_host()
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / e2e_steps
    e2e_value = W * nf * world / (e2e_ms * 1e-3)
    d2h = nf * 4 + int(min(int(cnt_h.max()), cap)) * 16 * nf

    # ---- configs[1]: single 1080p frame (latency case), device resident
    single = None
    if rank == 0:
        one_out = torch.zeros((1, cap, 4), dtype=torch.int32, device=f"cuda:{dev}")
        one_cnt = torch.zeros(1, dtype=torch.int32, device=f"cuda:{dev}")
        lat = {}
        for label, idx in (("U", 0), ("S", 1), ("F", 2)):
            fr = d_frames[idx:idx + 1]
            ts = []
            for it in range(13):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                clf.run_cascade_batch_device(fr.data_ptr(), 1, ROWS * COLS, ROWS, COLS, COLS, *PARAMS, 0.0,
                                             one_out.data_ptr(), cap, one_cnt.data_ptr(), st)
                b.record(stream)
                torch.cuda.synchronize()
                if it >= 3:
                    ts.append(a.elapsed_time(b))
            lat[label] = float(np.median(ts))
        med = float(np.mean(list(lat.values())))
        single = {"workload": "configs[1]: one 1920x1080 frame, device resident", "ms_per_frame_by_class": lat,
                  "windows_per_s": W / (med * 1e-3)}
        # the same call captured once into a CUDA graph and replayed (launch overhead off the critical path)
        try:
            glat = {}
            for label, idx in (("U", 0), ("S", 1), ("F", 2)):
                fr = d_frames[idx:idx + 1]
                # un-captured call first: it plans + allocates the workspace the capture then takes out of the pool for good
                clf.run_cascade_batch_device(fr.data_ptr(), 1, ROWS * COLS, ROWS, COLS, COLS, *PARAMS, 0.0,
                                             one_out.data_ptr(), cap, one_cnt.data_ptr(), st)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream, capture_error_mode="relaxed"):
                    clf.run_cascade_batch_device(fr.data_ptr(), 1, ROWS * COLS, ROWS, COLS, COLS, *PARAMS, 0.0,
                                                 one_out.data_ptr(), cap, one_cnt.data_ptr(), stream.cuda_stream)
                ts = []
                for it in range(13):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(stream)
                    g.replay()
                    b.record(stream)
                    torch.cuda.synchronize()
                    if it >= 3:
                        ts.append(a.elapsed_time(b))
                glat[label] = float(np.median(ts))
            single["cuda_graph_ms_per_frame_by_class"] = glat
        except Exception as e:   # noqa: BLE001 -- the graph leg is informative, never fatal
            single["cuda_graph_error"] = repr(e)[:200]
        # host API: pigo_run_cascade on one host frame (H2D, scan, D2H, sync), wall clock
        hts = []
        one_h = np.zeros(cap, dtype=pigo_b200.DET_DTYPE)
        n_h = C.c_int()
        for it in range(23):
            t0 = time.perf_counter()
            rc = L.pigo_run_cascade(clf._h, pinned[2].data_ptr(), ROWS, COLS, COLS, PARAMS[0], PARAMS[1], PARAMS[2], PARAMS[3], 0.0,
                                    one_h.ctypes.data, cap, C.byref(n_h))
            if it >= 3:
                hts.append((time.perf_counter() - t0) * 1e3)
            assert rc == 0
        single["host_api_ms_per_frame"] = float(np.median(hts))

    # ---- configs[1]/[2] at the reference's documented parameters (README: ShiftFactor 0.1 -> 4.1 M windows per 1080p frame):
    #      64 device-resident frames of the same workload, rank 0, N=1 only
    doc_params = None
    if rank == 0 and world == 1 and not args.no_extra:
        nd = min(64, nf)
        Wd = pigo_b200.count_windows(ROWS, COLS, PARAMS[0], PARAMS[1], 0.1, PARAMS[3])
        capd = 4096
        d_out_d = torch.zeros((nd, capd, 4), dtype=torch.int32, device=f"cuda:{dev}")
        d_cnt_d = torch.zeros(nd, dtype=torch.int32, device=f"cuda:{dev}")
        ts = []
        for it in range(7):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            clf.run_cascade_batch_device(d_frames.data_ptr(), nd, ROWS * COLS, ROWS, COLS, COLS, PARAMS[0], PARAMS[1], 0.1, PARAMS[3], 0.0,
                                         d_out_d.data_ptr(), capd, d_cnt_d.data_ptr(), st)
            b.record(stream)
            torch.cuda.synchronize()
            if it >= 2:
                ts.append(a.elapsed_time(b))
        md = float(np.median(ts))
        doc_params = {"workload": f"{nd} x 1920x1080 frames of the bench batch, MinSize 20 MaxSize 1000 ShiftFactor 0.1 ScaleFactor 1.1 (README parameters), "
                                  "device resident, CUDA events, median of 5 after 2 warm-ups",
                      "windows_per_frame": int(Wd), "ms_per_step": md, "windows_per_s": Wd * nd / (md * 1e-3),
                      "detections_per_step": int(torch.minimum(d_cnt_d, torch.tensor(capd, device=d_cnt_d.device)).sum())}
        del d_out_d, d_cnt_d

    # ---- configs[3]: 3840x2160 frames, rotated scan at EVERY table slot a = k/32 (rank 0, N=1 only: a sweep, not a scaling case)
    config4 = None
    if rank == 0 and world == 1 and not args.no_extra:
        from pigo_b200 import synth
        R4, C4, n4 = 2160, 3840, 8
        fr4 = np.stack([synth.frame_faces(None, R4, C4, shift=(31 * i, 17 * i), noise_seed=i) for i in range(n4)])
        d4 = torch.from_numpy(fr4).to(f"cuda:{dev}")
        o4 = torch.zeros((n4, 4096, 4), dtype=torch.int32, device=f"cuda:{dev}")
        c4 = torch.zeros(n4, dtype=torch.int32, device=f"cuda:{dev}")
        W4 = pigo_b200.count_windows(R4, C4, *PARAMS)
        per_slot = {}
        for k in range(0, 33):
            ts = []
            for it in range(5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                clf.run_cascade_batch_device(d4.data_ptr(), n4, R4 * C4, R4, C4, C4, *PARAMS, k / 32.0, o4.data_ptr(), 4096, c4.data_ptr(), st)
                b.record(stream)
                torch.cuda.synchronize()
                if it >= 2:
                    ts.append(a.elapsed_time(b))
            per_slot[k] = n4 * W4 / (float(np.median(ts)) * 1e-3)
        rot = [per_slot[k] for k in range(1, 33)]
        config4 = {"workload": f"configs[3]: {n4} x 3840x2160 frames (class F), test parameters, angle k/32 for k = 1..32 (classifyRotatedRegion), "
                               "device resident, CUDA events, median of 3 after 2 warm-ups per slot",
                   "windows_per_frame": W4, "unit": "windows/s", "rotated_min": min(rot), "rotated_median": float(np.median(rot)),
                   "rotated_max": max(rot), "unrotated_angle0": per_slot[0], "per_slot": {str(k): per_slot[k] for k in range(1, 33)}}
        del d4, o4, c4

    # ---- configs[4]: face -> cluster -> 2 pupils -> 15 landmarks on 1080p class-F frames, frames sharded over the ranks,
    #      one gather of faces + eyes + landmarks to rank 0 inside the timed step
    config5 = None
    if not args.no_extra:
        from pigo_b200 import pipeline, synth
        nf5, cap5 = args.pipeline_frames, 32
        plc = pigo_b200.NewPuplocCascade().UnpackCascade(pigo_b200.load_cascade("puploc"))
        names = sorted(set(pipeline.EYE_CASCADES + pipeline.MOUTH_CASCADES))
        flp = {n: pigo_b200.NewPuplocCascade().UnpackCascade(pigo_b200.load_cascade("lps/" + n)) for n in names}
        hs, fl = pipeline.landmark_call_arrays(flp)
        ncalls = len(fl)
        f5 = np.stack([synth.frame_faces(None, ROWS, COLS, shift=(37 * (i + nf5 * rank), 53 * (i + nf5 * rank)), noise_seed=100 + i + nf5 * rank)
                       for i in range(nf5)])
        p5 = torch.from_numpy(f5).pin_memory()
        d5 = p5.to(f"cuda:{dev}")
        faces5 = torch.zeros((nf5, cap5, 4), dtype=torch.int32, device=f"cuda:{dev}")
        nfaces5 = torch.zeros(nf5, dtype=torch.int32, device=f"cuda:{dev}")
        points5 = torch.zeros((nf5, cap5, 2 + ncalls, 4), dtype=torch.int32, device=f"cuda:{dev}")
        prm = pigo_b200.PipelineParams(PARAMS[0], PARAMS[1], PARAMS[2], PARAMS[3], 0.0, 0.1, 50, 63, 63, 0)

        def step_pipeline():
            rc = L.pigo_detect_batch(clf._h, plc._h, hs, fl.ctypes.data, ncalls, d5.data_ptr(), nf5, ROWS * COLS, ROWS, COLS, COLS, C.byref(prm), None, 7,
                                     faces5.data_ptr(), cap5, nfaces5.data_ptr(), points5.data_ptr(), 3, st)
            if rc != 0:
                raise RuntimeError(L.pigo_last_error().decode())
            if world > 1:
                pdist.gather_pipeline(faces5, nfaces5, points5, dst=0)

        for _ in range(3):
            step_pipeline()
        barrier()
        k5 = max(3, min(args.steps, 10))
        l5 = pigo_b200.launch_count()
        a5, b5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a5.record(stream)
        for _ in range(k5):
            step_pipeline()
        b5.record(stream)
        barrier()
        ms5 = max_over_ranks(a5.elapsed_time(b5)) / k5
        l5 = (pigo_b200.launch_count() - l5) // k5
        nref = int(((faces5[:, :, 2] > 50).sum()).item())
        # per-kernel device time of one step (separate pass)
        pigo_b200.set_option("timing", 1)
        step_pipeline()
        torch.cuda.synchronize()
        kt5 = {n: pigo_b200.get_option(f"t_{n}_ns") / 1e6 for n in ("tiled", "gather", "deep", "finalize", "cluster", "seeds", "puploc")}
        pigo_b200.set_option("timing", 0)
        # end to end through the host API: pinned frames in, faces + points out, every step
        fh = np.zeros((nf5, cap5), dtype=pigo_b200.DET_DTYPE)
        nh = np.zeros(nf5, dtype=np.int32)
        ph = np.zeros((nf5, cap5, 2 + ncalls), dtype=pigo_b200.POINT_DTYPE)

        def step_pipeline_host():
            rc = L.pigo_detect_batch(clf._h, plc._h, hs, fl.ctypes.data, ncalls, p5.data_ptr(), nf5, ROWS * COLS, ROWS, COLS, COLS, C.byref(prm), None, 7,
                                     fh.ctypes.data, cap5, nh.ctypes.data, ph.ctypes.data, 0, None)
            if rc != 0:
                raise RuntimeError(L.pigo_last_error().decode())
        step_pipeline_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            step_pipeline_host()
        barrier()
        e5 = max_over_ranks((time.perf_counter() - t0) * 1e3) / 3
        same = bool(np.array_equal(fh.view(np.int32).reshape(nf5, cap5, 4), faces5.cpu().numpy()) and
                    np.array_equal(ph.view(np.int32).reshape(nf5, cap5, 2 + ncalls, 4), points5.cpu().numpy()))
        if rank == 0:
            config5 = {"workload": f"configs[4]: {nf5} x 1920x1080 class-F frames per GPU -> RunCascade -> ClusterDetections(0.1) -> 2 x RunDetector "
                                   "(63 perturbations) -> 15 x GetLandmarkPoint (63) per face with Scale > 50, sequenced on the device "
                                   "(pigo_detect_batch); frames sharded over the ranks, faces + eyes + landmarks gathered to rank 0 inside the step",
                       "frames_per_gpu": nf5, "n_gpus": world, "value": nf5 * world / (ms5 * 1e-3), "unit": "frames/s", "ms_per_step": ms5,
                       "faces_refined_rank0": nref, "landmark_points_rank0": nref * ncalls, "launches_per_step": int(l5),
                       "kernel_ms_rank0": kt5,
                       "e2e": {"value": nf5 * world / (e5 * 1e-3), "unit": "frames/s", "ms_per_step": e5, "h2d_bytes_per_step": nf5 * ROWS * COLS,
                               "d2h_bytes_per_step": int(fh.nbytes + nh.nbytes + ph.nbytes), "matches_device_path": same},
                       "gathered_bytes_per_rank": int(faces5.numel() * 4 + nfaces5.numel() * 4 + points5.numel() * 4)}
        del d5

    # ---- CPU baseline (rank 0, N=1 only)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample = min(cpu_sample_frames(ncores, args.cpu_sample_frames), nf)
        v, ms = cpu_reference_run(frames_host[:sample], 2, 1, ncores)
        v1, ms1 = cpu_reference_run(frames_host[:3], 1, 0, 1)
        cpu_baseline = {"value": v, "unit": "windows/s", "cores": ncores, "kind": "port",
                        "sample": f"first {sample} frames of this workload x 2 passes, frame-parallel (dynamic queue) on {ncores} threads",
                        "single_thread_value": v1, "host": host_info(), "note": "C -O2 restatement of core/pigo.go (oracle/); the Go "
                        "reference cannot be built in this image (no Go toolchain)"}

    if dumped is not None:
        dump_outputs(args.dump_outputs, *dumped)
    if rank == 0:
        _emit(out_fd, {
            "metric": "candidate windows/s on 1080p frames", "value": value, "unit": "windows/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": "windows/s", "h2d_bytes_per_step": nf * ROWS * COLS, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "single_frame": single, "doc_params": doc_params, "config4": config4, "config5": config5,
            "detections_per_step": ndet})
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
