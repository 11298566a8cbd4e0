#!/usr/bin/env python
"""bench.py — 1080p frames/sec of the Motion (Laplace, 6-level) hot path on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  (N>1: launched by torchrun, one rank per GPU, NCCL; weak scaling — every rank serves its own
   `lanes` independent streams; the only collective on the data path is a one-time broadcast of the
   parameter block.)

A *step* = one frame for each of `lanes` independent 1920x1080x3 streams (one launch set of the
lane-batched kernels).  `value` = frames/s with frames resident in HBM; `e2e` = the same metric
through the public host API (pinned host frames in, pinned host frames out, copies inside the
timed region).  `--impl reference` times the reference's own CPU implementation of the path (its sources
compiled in place into oracle/_ref, OpenCV kernels through cv2, all host threads; the oracle restatement if that
module is absent) on the same workload.

`--dump-outputs DIR` writes, after the timed steps, a fixed seeded sample of the frames the last device-resident step
produced (DIR/output.npy, float32) with their flat indices into the [lanes, H, W, 3] output (DIR/output_index.npy,
float64) and that shape (DIR/output_shape.npy).  The clip is synthetic and the sample's seed fixed, so two builds run
with the same arguments can be compared value for value.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, CH, LEVELS = 1920, 1080, 3, 6
UI = dict(amplification=20, wavelength=50.0, low=0.4, high=3.0, chroma=0, levels=LEVELS, fps=30.0)
METRIC = "1080p frames/sec (Laplace, 6-level)"
WORKLOAD = "Motion (Laplace) 1920x1080x3 BGR, 6 levels, IIR 0.4-3 Hz @30fps, alpha=20 (BASELINE.json configs[1])"


def level_pixels(w, h, levels):
    out = []
    for _ in range(levels + 1):
        out.append(w * h)
        w, h = (w + 1) // 2, (h + 1) // 2
    return out


def a_min_bytes(w, h, c, levels):
    """SURVEY.md §8d: 2*C*P0 (u8 in+out) + 16*C*sum_{l=1}^{L-1} P_l (two f32 states, read+write)."""
    p = level_pixels(w, h, levels)
    return 2 * c * p[0] + 16 * c * sum(p[1:levels])


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons for one GPU; started before the warm-up (nvidia-smi takes
    ~0.2 s to emit its first row) and filtered to the rows that fall inside the timed regions."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.windows = index, [], None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if not any(t0 - 0.02 <= ts <= t1 + 0.02 for t0, t1 in self.windows):
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons),
                "note": "nvidia-smi rows inside the device-resident and e2e timed regions"}


def make_clip(t_frames, lanes):
    """[T][lanes][H][W][3] u8: lane k is the base clip rolled by 37*k px (distinct content per stream)."""
    from lvm_b200.synth import synth_frame
    base = [synth_frame(t, W, H, CH) for t in range(t_frames)]
    clip = np.empty((t_frames, lanes, H, W, CH), np.uint8)
    for t in range(t_frames):
        for k in range(lanes):
            clip[t, k] = np.roll(base[t], (11 * k, 37 * k), axis=(0, 1))
    return clip


DUMP_SAMPLES, DUMP_SEED = 1 << 22, 20240611   # <= 48 MB of float32 values + float64 indices


def dump_outputs(out_d, out_dir):
    """Writes a seeded sample of the device output tensor out_d (uint8, any shape) to out_dir as float32 / float64 .npy."""
    import torch
    total = out_d.numel()
    if total <= DUMP_SAMPLES:
        idx = np.arange(total, dtype=np.int64)
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(total, DUMP_SAMPLES, replace=False, shuffle=False))
    vals = out_d.reshape(-1)[torch.from_numpy(idx).to(out_d.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "output.npy"), vals.astype(np.float32))
    np.save(os.path.join(out_dir, "output_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "output_shape.npy"), np.array(out_d.shape, np.float64))


def oracle_cfg():
    from oracle import livim_oracle as O
    return O, O.ProcessorConfig(magnification=O.to_params(O.MODE_LAPLACE, UI["amplification"], UI["wavelength"],
                                                          UI["low"], UI["high"], UI["chroma"], UI["levels"], UI["fps"]))


def cpu_arm():
    """The CPU arm: the reference's own sources compiled in place (oracle/_ref/_livim_ref, OpenCV kernels through
    cv2) when that module is present — kind "reference" — else the oracle restatement — kind "port".
    -> (process(frame) callable, kind, description)."""
    import cv2
    O, ocfg = oracle_cfg()
    from oracle import livim_ref
    R = livim_ref.load()
    if R is not None:
        rcfg = livim_ref.to_ref_config(R, ocfg)
        proc = R.Processor()
        return (lambda f: proc.process(f, rcfg)), "reference", \
            f"reference src/processing compiled in place (oracle/_ref), OpenCV {cv2.__version__} kernels via cv2"
    proc = O.MagnificationProcessor()
    return (lambda f: proc.process(f, ocfg)), "port", f"cv2 {cv2.__version__} oracle restatement"


def cpu_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    import cv2
    build = [l.strip() for l in cv2.getBuildInformation().splitlines() if l.strip()][:6]
    return {"model": model, "logical_cpus": os.cpu_count() or 1, "cv2": cv2.__version__, "cv2_build_head": build}


def time_cpu_single(threads, n_warm, n_frames):
    """BASELINE.md section 3 protocol: one stream, cv2.setNumThreads(threads), n_warm untimed frames, then n_frames timed
    one by one -> median ms/frame.  -> dict"""
    import cv2
    from lvm_b200.synth import synth_frame
    process, kind, what = cpu_arm()
    cv2.setNumThreads(threads)
    frames = [synth_frame(t, W, H, CH) for t in range(8)]
    for t in range(n_warm):
        process(frames[t % 8])
    ms = []
    for t in range(n_frames):
        t0 = time.perf_counter()
        process(frames[(n_warm + t) % 8])
        ms.append((time.perf_counter() - t0) * 1e3)
    med = statistics.median(ms)
    return {"threads": threads, "warmup_frames": n_warm, "frames": n_frames, "median_ms_per_frame": med, "fps": 1e3 / med,
            "mean_fps": n_frames / (sum(ms) * 1e-3), "kind": kind, "what": what}


def _cpu_worker(idx, threads, n_warm, n_frames, ready_q, start_evt, out_q):
    """One independent stream of the CPU arm in its own process (throughput mode, the like-for-like of the GPU arm's lanes)."""
    try:
        import cv2
        from lvm_b200.synth import synth_frame
        process, kind, what = cpu_arm()
        cv2.setNumThreads(threads)
        frames = [np.roll(synth_frame(t, W, H, CH), (11 * idx, 37 * idx), axis=(0, 1)) for t in range(4)]
        for t in range(n_warm):
            process(frames[t % 4])
        ready_q.put(idx)
        start_evt.wait()
        t0 = time.perf_counter()               # CLOCK_MONOTONIC: comparable across processes
        for t in range(n_frames):
            process(frames[(n_warm + t) % 4])
        out_q.put((idx, n_frames, t0, time.perf_counter(), kind, what))
    except Exception as e:                      # a worker that dies must not hang the parent
        ready_q.put(idx)
        out_q.put((idx, 0, 0.0, 0.0, "failed", repr(e)))


def time_cpu_multiprocess(procs, threads, n_warm, n_frames):
    """procs independent streams x threads OpenCV threads each: aggregate frames / (last end - first start)."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    ready_q, out_q, start_evt = ctx.Queue(), ctx.Queue(), ctx.Event()
    ws = [ctx.Process(target=_cpu_worker, args=(i, threads, n_warm, n_frames, ready_q, start_evt, out_q)) for i in range(procs)]
    for w in ws:
        w.start()
    for _ in ws:
        ready_q.get(timeout=600)
    start_evt.set()
    res = [out_q.get(timeout=600) for _ in ws]
    for w in ws:
        w.join(timeout=30)
    ok = [r for r in res if r[1] > 0]
    if not ok:
        return {"processes": procs, "threads_each": threads, "failed": [r[5] for r in res][:2]}
    span = max(r[3] for r in ok) - min(r[2] for r in ok)
    total = sum(r[1] for r in ok)
    return {"processes": len(ok), "threads_each": threads, "warmup_frames": n_warm, "frames_each": n_frames, "fps": total / span,
            "seconds": span, "kind": ok[0][4], "what": ok[0][5]}


def mp_shape(cores):
    """Throughput mode of the CPU arm: OpenCV barely scales past a handful of threads on one 1080p frame, so the host's
    cores are used as cores/4 independent streams of 4 threads each."""
    threads = 4 if cores >= 8 else 1
    return max(1, cores // threads), threads


def run_reference(args, rank, world):
    if rank != 0:
        return None
    per_step = args.ref_frames_per_step
    cores = os.cpu_count() or 1
    procs, threads = mp_shape(cores)
    # throughput mode (the like-for-like of the GPU arm's lanes): every step = per_step frames on each of procs streams
    mpr = time_cpu_multiprocess(procs, threads, args.warmup * per_step, args.steps * per_step)
    # latency mode (one stream, all threads) beside it
    one = time_cpu_single(cores, min(8, args.warmup * per_step), min(64, args.steps * per_step))
    fps = max(mpr.get("fps", 0.0), one["fps"])
    dt = (mpr["seconds"] if mpr.get("fps", 0.0) >= one["fps"] else one["frames"] / one["mean_fps"])
    kind, what = one["kind"], one["what"]
    sample = (f"{args.steps} steps x {per_step} frames of the 1080p workload on each of {procs} independent streams x {threads} "
              f"OpenCV threads ({what}); single stream on {cores} threads beside it")
    return json.dumps({
        "impl": "reference", "metric": "1080p frames/sec (Laplace, 6-level)", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step": per_step * (procs if mpr.get("fps", 0.0) >= one["fps"] else 1),
                   "mode": "throughput: independent streams over all host cores (the GPU arm steps `lanes` independent streams)"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample,
                         "multi_process": mpr, "single_stream_all_threads": one, "host": cpu_info()},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def kernel_table(prof, lanes, band_from_state=False):
    """prof: {(kernel name, level): (launches, total ms)} from mc_profile_read -> (per-kernel table sorted by time share,
    {kernel: ncu DRAM bytes per launch scaled to `lanes`} from profiles/traffic.json for captures that still apply)."""
    px = level_pixels(W, H, LEVELS)
    total_ms = sum(v[1] for v in prof.values())
    table = []
    for (name, lvl), (n, tms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
        # alg = this kernel's share of A_min (SURVEY 8d); io = bytes its interface forces through HBM
        if name == "level" and lvl >= 1:
            alg = 16 * CH * px[lvl] * lanes                       # two f32 state planes, read + write
            # + G_l read, G_{l+1} write, and the band M_l write unless the synthesis rebuilds it from hi/lo
            io = alg + 4 * CH * (px[lvl] * (1 if band_from_state else 2) + px[lvl + 1]) * lanes
        elif name in ("level", "down"):                           # level 0: Lab16 -> pyrDown -> G1
            alg = 0
            io = (2 * CH * px[0] + 4 * CH * px[1]) * lanes
        elif name == "ingest_lab":                                # u8 -> Lab16 planes + G1
            alg = CH * px[0] * lanes
            io = alg + 2 * CH * px[0] * lanes + 4 * CH * px[1] * lanes
        elif name == "lab16":
            alg = CH * px[0] * lanes                              # u8 frame read
            io = alg + 2 * CH * px[0] * lanes                     # + Lab16 write
        elif name == "egress":
            alg = CH * px[0] * lanes                              # u8 frame write
            if band_from_state:   # + Lab16 read, hi_1/lo_1 read (band 1 rebuilt from state), cur_2 read
                io = alg + (2 * CH * px[0] + 8 * CH * px[1] + (8 if LEVELS == 3 else 4) * CH * px[2]) * lanes
            else:                 # + Lab16 read, M_1 read, cur_2 read
                io = alg + (2 * CH * px[0] + 4 * CH * px[1] + 4 * CH * px[2]) * lanes
        else:                                                     # collapse
            alg = 0
            if band_from_state:   # hi_l/lo_l read, cur_l write, cur_{l+1} read (from state when it is the top band)
                io = (12 * px[lvl] + (8 if lvl + 1 == LEVELS - 1 else 4) * px[lvl + 1]) * CH * lanes
            else:                 # M_l read + write, M_{l+1} read
                io = (8 * px[lvl] + 4 * px[lvl + 1]) * CH * lanes
        us = tms / n * 1e3
        table.append({"kernel": f"{name}[{lvl}]", "us_per_launch": us, "share": tms / total_ms,
                      "algorithmic_GBps": alg / (us * 1e-6) / 1e9, "interface_GBps": io / (us * 1e-6) / 1e9,
                      "interface_bytes": io})
    # DRAM bytes per launch from the committed `ncu --set full` captures (profiles/traffic.json).  A capture only
    # speaks for the kernel it was taken on: entries whose recorded interface model no longer matches the current
    # kernel (e.g. after the band stopped being stored) are dropped -> traffic null until re-captured.
    traffic = {}
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        model = {t["kernel"]: t["interface_bytes"] / lanes for t in table}
        traffic = {k: (v["dram_read_bytes"] + v["dram_write_bytes"]) * lanes / v["lanes"] for k, v in tj.items()
                   if k in model and abs(v.get("interface_bytes_per_lane", 0) - model[k]) <= 0.01 * model[k]}
    except Exception:
        pass
    return table, traffic


def run_ours(args, rank, world, local_rank):
    import torch
    import lvm_b200 as L
    from lvm_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the magnification core has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # one-time broadcast of the parameter block from rank 0 (the path's only collective)
    from lvm_b200.shard import broadcast_params, max_over_ranks as _max_over_ranks
    p = None
    if rank == 0:
        p = capi.McParams()
        capi.lib().mc_params_from_ui(C.byref(p), capi.MODE_LAPLACE, UI["amplification"], UI["wavelength"], UI["low"],
                                     UI["high"], UI["chroma"], UI["levels"], UI["fps"])
    p = broadcast_params(p, dist, device="cuda")

    lanes, T = args.lanes, args.clip_frames
    clip_h = make_clip(T, lanes)
    row = W * CH
    frame_bytes = H * row * lanes

    proc = L.MagnificationProcessor(device=local_rank, lanes=lanes)
    for kv in args.opt:                       # A/B knobs of the library (mc_set_option), e.g. --opt lane_groups=1
        k, v = kv.split("=")
        proc.set_option(k, int(v))
    stream = torch.cuda.ExternalStream(proc.stream, device=local_rank)
    clip_d = torch.from_numpy(clip_h).cuda()
    out_d = torch.empty((lanes, H, W, CH), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    in_ptrs = [clip_d[t].data_ptr() for t in range(T)]
    out_ptr = out_d.data_ptr()

    def step_dev(i):
        ok = proc.process_device(in_ptrs[i % T], W, H, CH, row, p, out_ptr, row)
        assert ok

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return _max_over_ranks(x, dist, device="cuda")

    # ---- device-resident throughput ----------------------------------------------------------
    vis = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v]
    sampler = ClockSampler(vis[local_rank] if local_rank < len(vis) else local_rank)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        step_dev(i)
    barrier()
    t_w0 = time.time()
    l0 = proc.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(args.steps):
        step_dev(args.warmup + i)
    e1.record(stream)
    barrier()
    sampler.window(t_w0, time.time())
    ms = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs and rank == 0:      # out_d holds the last timed step's frames
        dump_outputs(out_d, args.dump_outputs)
    from lvm_b200.shard import sum_over_ranks
    launches = int(sum_over_ranks(float(proc.launch_count - l0), dist, device="cuda"))
    fps = world * lanes * args.steps / (ms * 1e-3)

    # ---- end to end through the host API (pinned frames in / out, copies inside the region) ----
    # the pinned staging buffers are allocated (first touched) on the NUMA node of this rank's GPU
    from lvm_b200.shard import bind_to_gpu_numa_node
    prev_affinity, numa = bind_to_gpu_numa_node(local_rank)
    clip_p = torch.from_numpy(clip_h).pin_memory()
    depth = 3
    outs_p = [torch.empty((lanes, H, W, CH), dtype=torch.uint8).pin_memory() for _ in range(depth)]
    proc.reset()

    def run_e2e(n, start):
        done = 0
        for i in range(n):
            if i - done >= depth:
                assert proc.collect(); done += 1
            proc.submit(clip_p[(start + i) % T].data_ptr(), W, H, CH, row, p, outs_p[i % depth].data_ptr(), row)
        while done < n:
            assert proc.collect(); done += 1

    run_e2e(max(args.warmup, 3), 0)
    barrier()
    t0 = time.perf_counter()
    t_w0 = time.time()
    run_e2e(args.steps, args.warmup)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    sampler.window(t_w0, time.time())
    clocks = sampler.stop() if rank == 0 else None
    e2e_fps = world * lanes * args.steps / e2e_s
    barrier()

    # ---- the call the drop-in adapter makes: ONE stream, blocking mc_process, host frame in / host frame out ----
    single = None
    if rank == 0:
        from lvm_b200.synth import synth_frame
        sp = L.MagnificationProcessor(device=local_rank, lanes=1)
        fr = [synth_frame(t, W, H, CH) for t in range(4)]
        pin_in = [torch.from_numpy(f).pin_memory() for f in fr]
        pin_out = torch.empty((H, W, CH), dtype=torch.uint8).pin_memory()
        cfg1 = L.ProcessorConfig(magnification=L.toParams(L.MagUiValues(L.MagnificationMode.Laplace, UI["amplification"], UI["wavelength"],
                                                                         UI["low"], UI["high"], UI["chroma"], UI["levels"], UI["fps"])))
        for i in range(6):
            sp.process_image(fr[i % 4], cfg1)
        lat_pg, lat_pin = [], []
        for i in range(40):
            t0 = time.perf_counter()
            sp.process_image(fr[i % 4], cfg1)                      # pageable numpy in, numpy out (what a cv::Mat frame is)
            lat_pg.append(time.perf_counter() - t0)
        for i in range(40):
            t0 = time.perf_counter()
            sp.process_host(pin_in[i % 4].data_ptr(), W, H, CH, row, p, pin_out.data_ptr(), row)   # pinned (mc_host_alloc-style) frames
            lat_pin.append(time.perf_counter() - t0)
        sp.close()
        # (still bound to the GPU's NUMA node: the pinned frames above were first-touched next to the GPU's PCIe root)
        single = {"lanes": 1, "pageable_ms_median": statistics.median(lat_pg) * 1e3, "pinned_ms_median": statistics.median(lat_pin) * 1e3,
                  "pageable_fps": 1.0 / statistics.median(lat_pg), "pinned_fps": 1.0 / statistics.median(lat_pin),
                  "note": "blocking call per frame, copies included; what MagnificationProcessorB200::process does per cv::Mat"}

    if prev_affinity is not None:
        os.sched_setaffinity(0, prev_affinity)   # the CPU baseline below uses every host core again

    # ---- per-kernel device time (roofline of the dominant kernel) -------------------------------
    roof = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        proc.reset()
        for i in range(3):
            step_dev(i)
        proc.sync()
        proc.set_option("profile_kernels", 1)
        n_prof = min(args.steps, 20)
        for i in range(n_prof):
            step_dev(3 + i)
        prof = proc.profile_read()
        proc.set_option("profile_kernels", 0)
        table, traffic = kernel_table(prof, lanes, band_from_state=True)   # the library default
        dom = table[0]
        fused = next(t for t in table if t["kernel"] == "level[1]")   # the fused Laplace-pyramid + IIR kernel
        roof = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["algorithmic_GBps"], "peak": peak,
                "unit": "GB/s", "frac": dom["algorithmic_GBps"] / peak, "traffic": traffic.get(dom["kernel"]),
                "peak_source": peak_src, "interface_frac": dom["interface_GBps"] / peak,
                "bound_note": ("the step's largest kernels are the exact OpenCV colour conversions: BGR->Lab ingest is bound by "
                               "the L1 data pipe (two divergent 32-byte LUT gathers per pixel; ncu: l1tex 82 %, dram 16 %), "
                               "Lab->BGR egress by issue slots; their HBM fraction is low by construction.  The HBM-bound "
                               "kernel of the path is the fused per-level pyramid+IIR kernel reported under fused_level_kernel "
                               "(interface_frac = bytes its interface moves / time / peak)"),
                "fused_level_kernel": {"kernel": "level[1]", "achieved": fused["algorithmic_GBps"],
                                       "frac": fused["algorithmic_GBps"] / peak,
                                       "interface_frac": fused["interface_GBps"] / peak,
                                       "us_per_launch": fused["us_per_launch"], "traffic": traffic.get("level[1]")},
                "frame": {"a_min_bytes": a_min_bytes(W, H, CH, LEVELS),
                          "achieved": a_min_bytes(W, H, CH, LEVELS) * (fps / world) / 1e9,
                          "frac": a_min_bytes(W, H, CH, LEVELS) * (fps / world) / 1e9 / peak},
                "kernels": table}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # BASELINE.md section 3: 8 warm-up + >= 64 timed frames, median, at 1 thread and at all threads; plus the
        # throughput mode (independent streams over all cores) that corresponds to what the GPU arm measures
        cores = os.cpu_count() or 1
        allt = time_cpu_single(cores, 8, args.cpu_frames)
        onet = time_cpu_single(1, 4, max(16, args.cpu_frames // 4))
        procs, threads = mp_shape(cores)
        mpr = time_cpu_multiprocess(procs, threads, 4, 16)
        best = max(allt["fps"], mpr.get("fps", 0.0))
        cpu = {"value": best, "unit": "frames/s", "cores": cores, "kind": allt["kind"],
               "sample": (f"{allt['what']}: best of one stream on {cores} threads ({args.cpu_frames} frames, median) and "
                          f"{procs} independent streams x {threads} threads (16 frames each)"),
               "single_stream_all_threads": allt, "single_stream_1_thread": onet, "multi_process": mpr, "host": cpu_info()}

    line = None
    if rank == 0:
        line = json.dumps({
            "metric": METRIC if args.workload == "1080p6" else "4K frames/sec (Laplace, 8-level)", "value": fps, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "lanes_per_gpu": lanes, "frames_per_step": lanes * world,
                       "clip_frames": T, "options": args.opt,
                       "device_io": "`value` is device-in / device-out (frames resident in HBM, the ceiling a decoder/encoder hand-off would see)",
                       "l2": f"inputs {T * frame_bytes / 1e6:.0f} MB + per-lane state cycle through > L2 (126 MB); no flush needed"},
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": frame_bytes,
                    "d2h_bytes_per_step": frame_bytes, "pipeline_depth": depth, "numa": numa,
                    "single_stream_blocking": single},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        })
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return line


class StdoutToStderr:
    """Everything but the final JSON line goes to stderr — NCCL (NCCL_DEBUG=VERSION/INFO), torch and cuFFT log
    to fd 1, and the contract is ONE JSON line on stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--lanes", type=int, default=64, help="independent 1080p streams per GPU, stepped in lock-step")
    ap.add_argument("--clip-frames", type=int, default=8)
    ap.add_argument("--cpu-frames", type=int, default=64)
    ap.add_argument("--ref-frames-per-step", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--opt", action="append", default=[], help="library option key=value (mc_set_option), repeatable")
    ap.add_argument("--workload", default="1080p6", choices=["1080p6", "4k8"],
                    help="1080p6 = BASELINE.json configs[1] (the headline, default); 4k8 = configs[4]: 3840x2160, 8 levels")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's output frames to DIR as .npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.workload == "4k8":       # BASELINE.json configs[4]: a parity-test case, reported as an extra line on request
        global W, H, LEVELS, WORKLOAD
        W, H, LEVELS = 3840, 2160, 8
        UI["levels"] = 8
        WORKLOAD = "Motion (Laplace) 3840x2160x3 BGR, 8 levels, IIR 0.4-3 Hz @30fps, alpha=20 (BASELINE.json configs[4])"
        if args.lanes == 64:
            args.lanes = 16          # 4 x the pixels per stream: the same bytes per step as 64 lanes of 1080p
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    with StdoutToStderr():
        if args.impl == "reference":
            line = run_reference(args, rank, world)
        else:
            if args.warmup < 3:
                args.warmup = 3
            line = run_ours(args, rank, world, local_rank)
    if line is not None:
        print(line, flush=True)


if __name__ == "__main__":
    main()
