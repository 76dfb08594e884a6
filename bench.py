#!/usr/bin/env python
"""Benchmark of the SIFT hot path on B200 (contract in the task description / SURVEY.md 8d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...          (one rank per GPU, no data-path collective)

--dump-outputs DIR writes the features and descriptors the `value` path returned in its last timed step as .npy files
(dump_outputs), so that two builds can be compared output for output on the same seeded frames.

Workload ("step") = one pass of the hot path over a batch of FRAMES_PER_STEP synthetic 3840x2160
8-bit frames per GPU, popsift::Config defaults with octaves=5, levels=3 (BASELINE.json configs[2]:
octave 0 is the 2x up-scaled 7680x4320 plane).  Frames are independent, so ranks shard them with
no collective ("weak" scaling: per-GPU batch fixed).

Printed JSON (rank 0, one line):
  value     Mpixels/s of input pixels, whole job, inputs resident in HBM before the timed region
            (ps_submit_dev_u8 -> ps_counts -> ps_download: all kernels + result download).
  e2e       same metric through the C++ drop-in API (PopSift::enqueue -> SiftJob::get, popsift_b200/bin/api_bench)
            from PAGEABLE host frames, driven exactly like the reference arm drives the reference
            (oracle/ref_driver.cpp --bench): host->device copy of every frame and device->host copy of every
            result inside the timed region.  `e2e.pinned_ctypes` keeps the round-1 number (Python mirror,
            page-locked frames) for comparison.
  roofline  pyramid stage: algorithmic bytes per frame (68 B per octave-pixel, SURVEY 8d) / CUDA-event
            time of the pyramid launches of one frame, against the measured HBM peak
            (MEASURED_PEAKS.json); `dominant_kernel` = the octave-0 fused blur+DoG launches alone.
  cpu_baseline  the CPU oracle port (oracle/sift_oracle.c, OpenMP) timed on the first four frames of the workload;
  opencv_cpu    cv2.SIFT on the same frame, all host cores (the CPU baseline north_star names).
`--impl reference` times the UNMODIFIED reference PopSift (oracle/_ref, CUDA, built from
/root/reference) on the same frames through its own public API (host buffers in, host features out); with
--gpus N rank 0 starts one reference process per GPU (each on its own per-GPU batch: weak scaling, like our arm) and reports the aggregate.
Every rank (and every child process it starts) is bound to the CPUs of its GPU's NUMA node before any
page-locked allocation.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 3840, 2160
OCTAVES, LEVELS = 5, 3
FRAMES_PER_STEP = 32     # long enough that the 4-slot pipeline spends most of a step in steady state
SLOTS = int(os.environ.get("POPSIFT_BENCH_SLOTS", "4"))     # images in flight per GPU
BYTES_PER_OCTAVE_PIXEL = 4 * (3 * LEVELS + 8)     # 68 B (SURVEY.md 8d)
METRIC = "Mpixels/s SIFT extract @ 3840x2160 gray"
WORKLOAD = ("3840x2160 u8 gray, octaves=5 levels=3, default Config (upscale 2x: octave 0 = 7680x4320), RootSift, desc loop; "
            "%d frames per step per GPU" % FRAMES_PER_STEP)


def gpu_numa_cpus(index):
    """CPUs of the NUMA node GPU `index` hangs off (sysfs), or None when that cannot be determined."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        dom, rest = bus.split(":", 1)
        node = int(open("/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:], rest)).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        return sorted(cpus) or None
    except Exception:
        return None


def bind_to_gpu_node(index):
    """pin this process (its threads and children inherit it) to the GPU's NUMA node; returns what was done"""
    cpus = gpu_numa_cpus(index)
    if not cpus:
        return {"bound": False}
    try:
        os.sched_setaffinity(0, cpus)
        return {"bound": True, "cpus": len(cpus), "first_cpu": cpus[0]}
    except Exception as e:
        return {"bound": False, "error": str(e)}


def write_frames(frames, td):
    from popsift_b200.synth import write_pgm
    paths = []
    for i, f in enumerate(frames):
        p = os.path.join(td, "f%d.pgm" % i)
        write_pgm(p, f)
        paths.append(p)
    return paths


def run_children(cmds, barrier=None, cpus=None, timeout=1500):
    """start one benchmark child per command; wait until every child has printed `ready` (warm-up done), release
    them together through their --go-file, return their JSON lines"""
    import tempfile as _tf
    procs = []
    for i, (cmd, go) in enumerate(cmds):
        pre = None
        if cpus and cpus[i]:
            c = cpus[i]
            pre = (lambda c=c: os.sched_setaffinity(0, c))
        procs.append(subprocess.Popen(cmd + ["--go-file", go], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, preexec_fn=pre))
    for pr in procs:
        ln = pr.stdout.readline()
        if ln.strip() != "ready":
            err = pr.stderr.read()[-300:]
            for q in procs:
                q.kill()
            raise RuntimeError("benchmark child failed before the timed region: %s %s" % (ln.strip(), err))
    if barrier:
        barrier()
    for _cmd, go in cmds:
        open(go, "w").close()
    outs = []
    for pr in procs:
        out, err = pr.communicate(timeout=timeout)
        line = [l for l in out.splitlines() if l.startswith("{")]
        if pr.returncode != 0 or not line:
            raise RuntimeError("benchmark child failed: %s" % err.strip()[-300:])
        outs.append(json.loads(line[-1]))
    return outs


def synth_frames(n, rank):
    """n distinct 4K frames: one generated frame (seed 7 + rank) and shifted/flipped variants."""
    from popsift_b200.synth import make_frame
    base = make_frame(W, H, 7 + rank)
    out = [base]
    for i in range(1, n):
        f = np.roll(base, (37 * i, 91 * i), axis=(0, 1))
        if i & 1:
            f = f[:, ::-1]
        if i & 2:
            f = f[::-1, :]
        out.append(np.ascontiguousarray(f))
    return out


def octave_pixels():
    from popsift_b200 import api
    c = api.Config()
    c.setOctaves(OCTAVES)
    return [(w, h) for (w, h) in c.geometry(W, H)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).
    The sampler is started ahead of the region; only samples stamped inside [t0, t1] are used."""

    FIELDS = ["timestamp", "clocks.sm", "clocks.max.sm", "power.draw", "clocks_event_reasons.hw_slowdown",
              "clocks_event_reasons.hw_thermal_slowdown", "clocks_event_reasons.sw_thermal_slowdown",
              "clocks_event_reasons.sw_power_cap"]

    def __init__(self, device):
        self.device, self.proc, self.rows = device, None, []

    def start(self):
        for fields in (self.FIELDS, [f.replace("clocks_event_reasons", "clocks_throttle_reasons") for f in self.FIELDS]):
            try:
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + ",".join(fields),
                                              "--format=csv,noheader,nounits", "-lms", "20"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except Exception:
                self.proc = None
                return
            time.sleep(0.3)
            if self.proc.poll() is None:
                break
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, n_all = [], [], set(), 0
        for ts, ln in self.rows:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 8:
                continue
            n_all += 1
            if t0 is not None and not (t0 - 0.02 <= ts <= t1 + 0.02):
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_total": n_all}


# one `ncu --set full --clock-control none` capture of tools/one_frame.py 3840 2160 5 1 (round 1, after the
# last kernel change); per frame / per octave-0 level launch
NCU_SOURCE = "profiles/r02_ncu_full_frame_4k.csv"
NCU_PYRAMID_DRAM_BYTES = 2222500352
NCU_LEVEL_DRAM_BYTES = 368350822


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def run_ours(args, rank, world, local_rank):
    import torch
    from popsift_b200 import api

    torch.cuda.set_device(local_rank)
    L = api.load_library()
    cfg = api.Config()
    cfg.setOctaves(OCTAVES)
    cfg.setLevels(LEVELS)
    frames = synth_frames(FRAMES_PER_STEP, rank)
    npix_step = FRAMES_PER_STEP * W * H

    # ---------------- device-resident path (`value`) ----------------
    ctx = L.ps_create(local_rank, C.byref(cfg._c), W, H, SLOTS)
    if not ctx:
        raise SystemExit("ps_create failed: " + L.ps_last_error(None).decode())
    dev_frames = [torch.from_numpy(f).cuda() for f in frames]
    # page-locked result buffers (ps_host_alloc): ps_download DMA-copies straight into them
    res = api._PinnedBlock(L, 200000, 200000)
    feat_buf, desc_buf = res.feat, res.desc
    nf, nd = C.c_int32(), C.c_int32()

    def chk(rc):
        if rc != 0:
            raise SystemExit("popsift_b200 error %d: %s" % (rc, L.ps_last_error(ctx).decode()))

    def step_dev(keep=None):
        """FRAMES_PER_STEP frames, SLOTS in flight; every job's features + descriptors land on the host.
        `keep`: a _PinnedBlock with room for the whole step; each frame's results then land in a region of their own,
        appended to keep.frames as (first feature, features, first descriptor, descriptors)."""
        tot_f = tot_d = 0
        inflight = []

        def fetch(s0):
            chk(L.ps_counts(ctx, s0, C.byref(nf), C.byref(nd)))
            if keep is None:
                chk(L.ps_download(ctx, s0, feat_buf.ctypes.data, desc_buf.ctypes.data))
            else:
                if tot_f + nf.value > keep.n_feat or tot_d + nd.value > keep.n_desc:
                    raise SystemExit("bench.py: the last timed step returned more results than the warm-up step")
                chk(L.ps_download(ctx, s0, keep.pf + 72 * tot_f, keep.pd + 512 * tot_d))
                keep.frames.append((tot_f, nf.value, tot_d, nd.value))
            return nf.value, nd.value

        for i, df in enumerate(dev_frames):
            s = i % SLOTS
            if len(inflight) == SLOTS:
                f, d = fetch(inflight.pop(0))
                tot_f += f; tot_d += d
            chk(L.ps_submit_dev_u8(ctx, s, df.data_ptr(), W, W, H))
            inflight.append(s)
        for s0 in inflight:
            f, d = fetch(s0)
            tot_f += f; tot_d += d
        return tot_f, tot_d

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        warm = step_dev()
    last_step = None
    if args.dump_outputs and rank == 0:
        # the last timed step downloads into a block allocated here, one region per frame, so that keeping its results
        # changes only where ps_download writes; sized from the warm-up step, which ran the same frames
        last_step = api._PinnedBlock(L, warm[0] + warm[0] // 8 + 1, warm[1] + warm[1] // 8 + 1)
        last_step.frames = []
    barrier()
    launches0 = L.ps_launch_count(ctx)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    slot_streams = [torch.cuda.ExternalStream(L.ps_slot_stream(ctx, s)) for s in range(SLOTS)]
    tstream = torch.cuda.Stream()
    with torch.cuda.stream(tstream):
        ev0.record(tstream)
    for st in slot_streams:        # the slots' work is ordered after ev0
        st.wait_event(ev0)
    t0 = time.perf_counter()
    wall0 = time.time()
    counts = (0, 0)
    for k in range(args.steps):
        counts = step_dev(last_step if k == args.steps - 1 else None)
    for st in slot_streams:        # ev1 after everything the slots did
        e = torch.cuda.Event()
        e.record(st)
        tstream.wait_event(e)
    ev1.record(tstream)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    dev_ms = ev0.elapsed_time(ev1)
    launches = L.ps_launch_count(ctx) - launches0
    clocks = sampler.stop(wall0, time.time()) if rank == 0 else None
    if last_step is not None:
        dump_outputs(args.dump_outputs, [(last_step.feat[f0:f0 + n], last_step.desc[d0:d0 + m], last_step.pd + 512 * d0)
                                         for f0, n, d0, m in last_step.frames])
        last_step.free()

    # ---------------- roofline of the pyramid stage (same context, slot 0 holds the last frame) ----
    chk(L.ps_submit_dev_u8(ctx, 0, dev_frames[0].data_ptr(), W, W, H))
    chk(L.ps_counts(ctx, 0, C.byref(nf), C.byref(nd)))
    s0 = slot_streams[0]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > L2 (126 MB)
    pyr_ms, dom_ms = [], []
    geo = octave_pixels()
    for it in range(3 + 10):
        with torch.cuda.stream(s0):
            flush.fill_(it & 0xff)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(s0)
        chk(L.ps_run_pyramid_only(ctx, 0))
        b.record(s0)
        b.synchronize()
        if it >= 3:
            pyr_ms.append(a.elapsed_time(b))
    for it in range(3 + 10):
        with torch.cuda.stream(s0):
            flush.fill_(it & 0xff)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(s0)
        for lvl in range(1, LEVELS + 3):
            chk(L.ps_run_level_only(ctx, 0, 0, lvl))
        b.record(s0)
        b.synchronize()
        if it >= 3:
            dom_ms.append(a.elapsed_time(b) / (LEVELS + 2))
    L.ps_destroy(ctx)
    res.free()
    del dev_frames, flush
    torch.cuda.empty_cache()

    # ---------------- end-to-end path, Python mirror + page-locked frames (round-1 definition, kept as an extra) ----
    pinned = [torch.from_numpy(f).pin_memory().numpy() for f in frames]
    ps = api.PopSift(cfg, device=local_rank, max_width=W, max_height=H, slots=SLOTS)

    def step_e2e():
        jobs, tf, td = [], 0, 0
        for f in pinned:
            jobs.append(ps.enqueue(W, H, f))
            if len(jobs) == SLOTS:
                r = jobs.pop(0).get(); tf += r.getFeatureCount(); td += r.getDescriptorCount()
        for j in jobs:
            r = j.get(); tf += r.getFeatureCount(); td += r.getDescriptorCount()
        return tf, td

    for _ in range(args.warmup):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    pinned_wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    ps.uninit()
    del pinned

    # ---------------- end-to-end path: the C++ drop-in API from pageable frames (the headline e2e) ----------------
    exe = os.path.join(ROOT, "popsift_b200", "bin", "api_bench")
    if not os.path.exists(exe):
        raise SystemExit("bench.py: %s is missing - build the product first (python -m popsift_b200.build)" % exe)
    with tempfile.TemporaryDirectory() as td:
        cmd = [exe, "--octaves", str(OCTAVES), "--levels", str(LEVELS), "--device", str(local_rank), "--slots", str(SLOTS),
               "--bench", str(args.steps), str(args.warmup)]
        for pth in write_frames(frames, td):
            cmd += ["-i", pth]
        torch.cuda.synchronize()
        j = run_children([(cmd, os.path.join(td, "go"))], barrier=barrier)[0]
    e2e_wall_ms = j["total_ms"]
    ecounts = (j["features_last_step"], j["descriptors_last_step"])
    if ecounts != counts:
        raise SystemExit("bench.py: the C++ API leg found %s features/descriptors, the C-ABI leg %s" % (ecounts, counts))

    # whole-job aggregate: SUM of pixels, MAX over ranks of the elapsed time (device-timed for `value`;
    # wall clock for e2e, which includes host work by definition)
    from popsift_b200 import shard
    total_pix, dev_ms = shard.aggregate(npix_step * args.steps, dev_ms, device="cuda")
    _, wall_ms = shard.aggregate(0, wall_ms, device="cuda")
    _, e2e_wall_ms = shard.aggregate(0, e2e_wall_ms, device="cuda")
    _, pinned_wall_ms = shard.aggregate(0, pinned_wall_ms, device="cuda")
    if rank != 0:
        return None

    peak, peak_src = measured_peak()
    sum_wh = sum(w * h for w, h in geo)
    alg_bytes_frame = BYTES_PER_OCTAVE_PIXEL * sum_wh
    pyr = statistics.median(pyr_ms)
    dom = statistics.median(dom_ms)
    dom_bytes = 12 * geo[0][0] * geo[0][1]       # read G[l-1], write G[l], write DoG[l-1]
    out = {
        "metric": METRIC, "value": total_pix / (dev_ms * 1e-3) / 1e6, "unit": "Mpixels/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": FRAMES_PER_STEP, "slots": SLOTS,
                   "sharding": "frames across ranks, no collective",
                   "l2": "working set per frame 3.0 GB of planes >> 126 MB L2; L2 flushed (256 MB fill) before each roofline sample"},
        "wall_ms_per_step": wall_ms / args.steps,
        "features_per_step": counts[0], "descriptors_per_step": counts[1],
        "gpu_launches": int(launches),
        "e2e": {"value": total_pix / (e2e_wall_ms * 1e-3) / 1e6, "unit": "Mpixels/s",
                "h2d_bytes_per_step": FRAMES_PER_STEP * W * H,
                "d2h_bytes_per_step": int(ecounts[0] * 72 + ecounts[1] * 512 + FRAMES_PER_STEP * 128),
                "api": "C++ drop-in API: PopSift::enqueue -> SiftJob::get -> delete (popsift_b200/bin/api_bench), PAGEABLE std::vector "
                       "frames, one process per GPU -- the same driver loop as the reference arm's (oracle/ref_driver.cpp --bench)",
                "pinned_ctypes": {"value": npix_step * world / (pinned_wall_ms * 1e-3) / 1e6, "unit": "Mpixels/s",
                                  "api": "popsift_b200.api.PopSift.enqueue -> SiftJob.get (Python mirror of the C ABI), page-locked frames"}},
        "roofline": {"bound": "hbm", "stage": "pyramid (all launches of one frame)", "achieved": alg_bytes_frame / (pyr * 1e-3) / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": alg_bytes_frame / (pyr * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                     "algorithmic_bytes": alg_bytes_frame, "ms": pyr,
                     # dram__bytes_read.sum + dram__bytes_write.sum of the 26 pyramid launches of one frame, one
                     # `ncu --set full` capture (profiles/r02_ncu_full_frame_4k.csv); below the algorithmic bytes
                     # because part of every plane is still dirty in the 126 MB L2 when its consumer starts
                     "traffic": NCU_PYRAMID_DRAM_BYTES, "traffic_source": NCU_SOURCE,
                     "dominant_kernel": {"name": "march_level_kernel (octave 0, levels 1..5: blur + DoG, avg per launch)",
                                         "algorithmic_bytes": dom_bytes, "ms": dom,
                                         "achieved": dom_bytes / (dom * 1e-3) / 1e9, "frac": dom_bytes / (dom * 1e-3) / 1e9 / peak,
                                         "traffic": NCU_LEVEL_DRAM_BYTES}},
        "clocks": clocks,
        "numa": NUMA_INFO,
    }
    if world == 1:      # reported baselines: rank 0 at N=1 only (torchrun pins OMP_NUM_THREADS=1)
        out.update(cpu_baselines(frames))
    return out


DUMP_BYTES = 64 << 20
DUMP_DESC_SAMPLE = 65536


def dump_outputs(out_dir, per_frame, seed=0):
    """What the timed (device-resident) path handed back for each frame of its last step, as .npy files in `out_dir`.
    The library emits features in no fixed order, so each frame's features are sorted (octave, y, x, sigma, num_ori,
    orientations) and orientation slots beyond num_ori are written as 0:
      counts.npy           float64 [frames, 2]   features, descriptors per frame
      features.npy         float32 [n, 10]       frame, octave, x, y, sigma, num_ori, ori[4]
      descriptors.npy      float32 [s, 128]      a seeded sample of the descriptors (all of them if they fit 64 MB)
      descriptor_rows.npy  float64 [s, 2]        row in features.npy and orientation index of each sampled descriptor
    Descriptor j of the full list is the one of feature row r, orientation k, enumerated in row order, then k.
    `per_frame`: (features, descriptors, host address of descriptor 0 that the features' desc_ptr refer to) per frame."""
    os.makedirs(out_dir, exist_ok=True)
    counts, feats, rows, idx = [], [], [], []
    for i, (feat, desc, desc_base) in enumerate(per_frame):
        n = feat["num_ori"].astype(np.int64)
        ori = np.where(np.arange(4)[None, :] < n[:, None], feat["ori"], np.float32(0))
        order = np.lexsort(tuple(ori[:, k] for k in range(3, -1, -1)) + (n, feat["sigma"], feat["x"], feat["y"], feat["octave"]))
        t = np.zeros((len(feat), 10), np.float32)
        t[:, 0] = i
        t[:, 1:6] = np.stack([feat["octave"], feat["x"], feat["y"], feat["sigma"], n], 1)[order]
        t[:, 6:] = ori[order]
        base = sum(len(f) for f in feats)
        nk = n[order]
        k = np.arange(nk.sum()) - np.repeat(np.cumsum(nk) - nk, nk)
        f_in = np.repeat(order, nk)
        rows.append(np.stack([base + np.repeat(np.arange(len(order)), nk), k], 1))
        idx.append(np.stack([np.full(len(k), i), (feat["desc_ptr"][f_in, k].astype(np.int64) - desc_base) // 512], 1))
        counts.append((len(feat), len(desc)))
        feats.append(t)
    features = np.concatenate(feats) if feats else np.zeros((0, 10), np.float32)
    rows, idx = np.concatenate(rows), np.concatenate(idx)
    room = max(0, (DUMP_BYTES - features.nbytes - 16 * len(counts)) // (512 + 16))
    pick = np.arange(len(rows))
    if len(rows) > min(room, DUMP_DESC_SAMPLE):
        pick = np.sort(np.random.default_rng(seed).choice(len(rows), min(room, DUMP_DESC_SAMPLE), replace=False))
    desc = np.stack([per_frame[f][1][d] for f, d in idx[pick]]) if len(pick) else np.zeros((0, 128), np.float32)
    np.save(os.path.join(out_dir, "counts.npy"), np.array(counts, np.float64).reshape(-1, 2))
    np.save(os.path.join(out_dir, "features.npy"), features)
    np.save(os.path.join(out_dir, "descriptors.npy"), desc.astype(np.float32))
    np.save(os.path.join(out_dir, "descriptor_rows.npy"), rows[pick].astype(np.float64))


def cpu_baselines(frames, n_oracle=4):
    """CPU oracle port on the first `n_oracle` frames of the workload (about 10 s on the box's host cores) and
    OpenCV SIFT on the first frame: bounded samples, reported baselines."""
    res = {}
    frame = frames[0]
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as ol
        cores = ol.lib().orc_set_threads(0)
        o = ol.Oracle(ol.make_config(octaves=OCTAVES), W, H)
        sample = frames[:n_oracle]
        nf = 0
        t = time.perf_counter()
        for f in sample:
            o.run(f)
            nf += o.features()[0].shape[0]
        dt = time.perf_counter() - t
        res["cpu_baseline"] = {"value": len(sample) * W * H / dt / 1e6, "unit": "Mpixels/s", "cores": cores, "kind": "port",
                               "sample": "%d frames 3840x2160 of the same workload, oracle/sift_oracle.c (OpenMP), %.2f s, %d features"
                                         % (len(sample), dt, nf)}
        o.close()
    except Exception as e:  # the oracle is test infrastructure; its absence must not hide the GPU numbers
        res["cpu_baseline"] = {"value": None, "unit": "Mpixels/s", "cores": 0, "kind": "port", "sample": "unavailable: %s" % e}
    try:
        import cv2
        n = os.cpu_count() or 1
        cv2.setNumThreads(n)
        sift = cv2.SIFT_create(nOctaveLayers=3, contrastThreshold=0.04, edgeThreshold=10, sigma=1.6)
        sift.detectAndCompute(frame, None)
        ts = []
        kp = []
        for _ in range(3):
            t = time.perf_counter(); kp, _d = sift.detectAndCompute(frame, None); ts.append(time.perf_counter() - t)
        dt = statistics.median(ts)
        res["opencv_cpu"] = {"value": W * H / dt / 1e6, "unit": "Mpixels/s", "cores": n,
                             "sample": "cv2 %s SIFT_create(3,0.04,10,1.6).detectAndCompute, 1 frame 3840x2160, median of 3, %d keypoints" % (cv2.__version__, len(kp))}
    except Exception as e:
        res["opencv_cpu"] = {"value": None, "unit": "Mpixels/s", "cores": 0, "sample": "unavailable: %s" % e}
    return res


def run_reference(args, rank, world, local_rank):
    """The unmodified reference (CUDA) through its own API.  Rank 0 alone runs it: one reference process per GPU
    (`--gpus N`), each on its own batch of frames (weak scaling, like our arm), released together."""
    if rank != 0:
        return None
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_dump")
    if not os.path.exists(exe):
        return {"impl": "reference", "unavailable": "oracle/_ref/ref_dump not built (needs /root/reference at build time)"}
    n = max(1, args.gpus)
    try:
        with tempfile.TemporaryDirectory() as td:
            cmds, cpus = [], []
            for g in range(n):
                sub = os.path.join(td, "g%d" % g)
                os.makedirs(sub)
                cmd = [exe, "--octaves", str(OCTAVES), "--levels", str(LEVELS), "--device", str(g), "--bench", str(args.steps), str(args.warmup)]
                for pth in write_frames(synth_frames(FRAMES_PER_STEP, g), sub):
                    cmd += ["-i", pth]
                cmds.append((cmd, os.path.join(sub, "go")))
                cpus.append(gpu_numa_cpus(g))
            outs = run_children(cmds, cpus=cpus)
    except Exception as e:
        return {"impl": "reference", "unavailable": "ref_dump failed: %s" % str(e)[-200:]}
    total_ms = max(j["total_ms"] for j in outs)
    px = sum(j["pixels_per_step"] for j in outs) * args.steps
    v = px / (total_ms * 1e-3) / 1e6
    return {"impl": "reference", "metric": METRIC, "value": v, "unit": "Mpixels/s", "n_gpus": n, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": FRAMES_PER_STEP,
                       "note": "reference PopSift is CUDA-only (no CPU implementation exists); one reference process per GPU through "
                               "PopSift::enqueue/SiftJob::get with pageable host buffers, started together"},
            "features_per_step": sum(j["features_last_step"] for j in outs), "descriptors_per_step": sum(j["descriptors_last_step"] for j in outs),
            "per_gpu_mpix_per_s": [j["mpix_per_s"] for j in outs],
            "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": 2 * n, "kind": "reference",
                             "sample": "%d frames 3840x2160 per step per GPU, unmodified reference libpopsift (oracle/_ref) on %d B200, "
                                       "2 host threads per GPU" % (FRAMES_PER_STEP, n)},
            "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


NUMA_INFO = {"bound": False}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path computed in its last step (rank 0's frames) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    global NUMA_INFO
    if args.impl == "ours":        # before torch / any page-locked allocation
        NUMA_INFO = bind_to_gpu_node(local_rank)
    if args.impl == "reference":
        out = run_reference(args, rank, world, local_rank)
        if out is not None:
            print(json.dumps(out), flush=True)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product has no CPU path")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    out = run_ours(args, rank, world, local_rank)
    if out is not None:
        print(json.dumps(out), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
