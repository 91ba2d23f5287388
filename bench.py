#!/usr/bin/env python
"""Benchmark of the two hot paths named by BASELINE.json (one JSON line on stdout, rank 0).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU algorithm (oracle port)
    python bench.py --steps K --dump-outputs DIR             # + the outputs of the last timed step of every leg as DIR/*.npy

Primary line  = ORB keypoints/s, BASELINE configs[1]: 640x480, 8 levels, 1000 kps/frame, batch of 64 frames / GPU.
`secondary`   = LM iterations/s, BASELINE configs[3]: 50 KF / 5000 landmarks / ~29k edges, Huber, 10 LM iterations.
A "step" is one pass of the hot path over one batch (ORB: one 64-frame batch; BA: one optimize(10) of the window).

value : device-resident throughput (inputs already in HBM, CUDA events on the launching stream)
e2e   : the same metric through the host-buffer C-ABI call (H2D of inputs + D2H of results inside the timed region)
roofline / cpu_baseline : see DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

_OUT = sys.stdout
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from tools import synth  # noqa: E402

ORB_METRIC = "ORB keypoints/sec at 640x480 (8-level pyramid, 1000 kps/frame)"
BA_METRIC = "LM iterations/sec on 50-KF/5k-point local BA"
W, H, NFEAT, NLEV, BATCH = 640, 480, 1000, 8, 64
BA_ITERS = 10
C5_METRIC = "LM iterations/sec on 2000-KF/50k-point global-scale BA (BASELINE configs[4])"
C5_ITERS = 5
MATCH_METRIC = "MatchByWindow frame pairs/sec at 1000 x 1000 keypoints (win 20, ratio 0.9)"
MATCH_PAIRS = 8
ORB_WORKLOAD = "ORB extraction 640x480, 8-level pyramid (scale 1.2), FAST 20/7, 1000 kps/frame, batch of 64 frames per GPU"


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture of this round (None if not captured)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_traffic.json")))
    if not files:
        return None
    try:
        return json.load(open(files[-1])).get(kernel)
    except Exception:
        return None


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.samples, self.stop, self.index = [], False, index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) > 2 + i and s[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


def matcher_frames():
    """MATCH_PAIRS (frame, shifted frame) pairs of the ORB benchmark texture: what Track hands to MatchByWindow."""
    imgs = []
    for k in range(MATCH_PAIRS):
        a = synth.orb_frame(2000 + k)
        imgs += [a, np.roll(a, (3 + k % 3, -5 + k % 4), axis=(0, 1))]
    return np.stack(imgs)


DUMP_LIMIT_BYTES = 64 << 20


def kp_columns(kps):
    """[..., 7] float32 columns (x, y, size, angle, response, octave, class_id) of KP_DTYPE records; exact for the int fields."""
    return np.stack([kps[f].astype(np.float32) for f in kps.dtype.names], axis=-1)


def write_dump(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, float32 or float64 only."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# =================================================================================================
# reference arm: the reference's CPU algorithm (oracle port; the reference itself needs OpenCV/g2o/ROS, absent here)
# =================================================================================================
def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle
    cores = os.cpu_count() or 1
    nframes = max(cores, 8)
    imgs = synth.orb_batch(min(nframes, BATCH))
    exts = [pyoracle.OrbOracle(NFEAT, 1.2, NLEV, 20) for _ in range(cores)]

    def work(k):
        kps, _ = exts[k % cores].extract(imgs[k % len(imgs)])
        return len(kps)
    pool = ThreadPoolExecutor(cores)
    for _ in range(args.warmup):
        list(pool.map(work, range(nframes)))
    t0 = time.perf_counter()
    tot = 0
    for _ in range(args.steps):
        tot += sum(pool.map(work, range(nframes)))
    dt = time.perf_counter() - t0
    orb_v = tot / dt
    # BA: g2o is single-threaded -> 1 core
    prob = synth.ba_config("C4")
    t_ba, it_ba = 0.0, 0
    for k in range(args.warmup + args.steps):
        o = pyoracle.BAOracle(prob)
        t1 = time.perf_counter()
        n, _ = o.optimize(BA_ITERS)
        if k >= args.warmup:
            t_ba += time.perf_counter() - t1; it_ba += n
    ba_v = it_ba / t_ba
    # matcher: oracle restatement of ORBmatcher::MatchByWindow on one core over (frame, shifted frame) pairs
    from se2lam_b200.matcher import FrameView
    mimgs = matcher_frames()[:4]
    ex = [exts[0].extract(im) for im in mimgs]
    pairs = [(FrameView(*ex[0]), FrameView(*ex[1])), (FrameView(*ex[2]), FrameView(*ex[3]))]
    match_cpu = cpu_match(pairs)
    line = {
        "impl": "reference", "metric": ORB_METRIC, "value": orb_v, "unit": "keypoints/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": ORB_WORKLOAD, "sample": f"{nframes} frames per step (bounded sample of the same workload)"},
        "cpu_baseline": {"value": orb_v, "unit": "keypoints/s", "cores": cores, "kind": "port",
                         "sample": f"{nframes} frames/step x {args.steps} steps, one extractor per thread"},
        "e2e": {"value": orb_v, "unit": "keypoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "secondary": {"metric": BA_METRIC, "value": ba_v, "unit": "LM iterations/s", "higher_is_better": True, "dtype": "f64",
                      "config": {"workload": f"local BA {prob.P} KF / {prob.L} landmarks / {prob.E} EdgeSE2XYZ + {prob.O} PreEdgeSE2, Huber, {BA_ITERS} LM iterations"},
                      "cpu_baseline": {"value": ba_v, "unit": "LM iterations/s", "cores": 1, "kind": "port",
                                       "sample": f"{args.steps} x optimize({BA_ITERS})"},
                      "e2e": {"value": ba_v, "unit": "LM iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
        "matcher": {"metric": MATCH_METRIC, "value": match_cpu["value"], "unit": "frame pairs/s", "higher_is_better": True,
                    "cpu_baseline": match_cpu, "e2e": {"value": match_cpu["value"], "unit": "frame pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
    }
    _OUT.write(json.dumps(line) + "\n"); _OUT.flush()


# =================================================================================================
# this repo's arm
# =================================================================================================
def run_ours(args):
    import torch
    import torch.distributed as dist
    from se2lam_b200 import _capi
    from se2lam_b200.ba import LocalBA
    from se2lam_b200.orb import ORBextractor

    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _capi.lib()
    hbm_peak, peak_src = peaks()
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ------------------------------------------------------------------------------------------ ORB
    NROT = 8   # distinct 64-frame input batches: 8 x 19.7 MB = 157 MB > 126 MB L2
    base = synth.orb_batch(BATCH, first_seed=1000 + 64 * rank)
    host_batches = []
    for r in range(NROT):
        b = np.roll(base, r * 7, axis=2) if r else base          # cheap distinct content, same statistics
        host_batches.append(torch.from_numpy(np.ascontiguousarray(b)).pin_memory())
    dev_batches = [hb.to(dev, non_blocking=True) for hb in host_batches]
    ext = ORBextractor(NFEAT, 1.2, NLEV, fastTh=20, max_width=W, max_height=H, max_batch=BATCH, device=local_rank)
    d_kps = torch.empty(BATCH * NFEAT * 28, dtype=torch.uint8, device=dev)
    d_desc = torch.empty(BATCH * NFEAT * 32, dtype=torch.uint8, device=dev)
    d_counts = torch.zeros((max(args.steps, args.warmup) + 1, BATCH), dtype=torch.int32, device=dev)   # one row per step
    sptr = stream.cuda_stream
    # Two batches in flight (--orb-inflight 2; default 1): consecutive steps alternate between two extractor contexts on two
    # streams, exactly what se2gpu_orb_submit / _wait does for host buffers; the kernels of batch k+1 fill the issue slots the
    # latency-bound tails of batch k leave idle. Every step is still one complete pass over one 64-frame batch and all K steps
    # finish inside the timed region (the closing event waits for both streams).
    inflight = max(1, min(2, args.orb_inflight))
    exts2 = [ext] + [ORBextractor(NFEAT, 1.2, NLEV, fastTh=20, max_width=W, max_height=H, max_batch=BATCH, device=local_rank) for _ in range(inflight - 1)]
    streams2 = [stream] + [torch.cuda.Stream(device=dev) for _ in range(inflight - 1)]
    outs2 = [(d_kps, d_desc)] + [(torch.empty_like(d_kps), torch.empty_like(d_desc)) for _ in range(inflight - 1)]

    def orb_step(k, lanes=inflight):
        q = k % lanes
        exts2[q].extract_device(dev_batches[k % NROT], BATCH, H, W, outs2[q][0], outs2[q][1], d_counts[k], stream=streams2[q].cuda_stream)

    def orb_join():     # the primary stream waits for the work of the other one
        for q in range(1, inflight):
            ev = torch.cuda.Event()
            ev.record(streams2[q])
            stream.wait_event(ev)

    def orb_fork():     # ... and the other stream starts after what is on the primary stream
        for q in range(1, inflight):
            ev = torch.cuda.Event()
            ev.record(stream)
            streams2[q].wait_event(ev)

    for k in range(args.warmup):
        orb_step(k)
    barrier()
    launches0 = lib.se2gpu_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        e0.record(stream)
        orb_fork()
        for k in range(args.steps):
            orb_step(k)
        orb_join()
        e1.record(stream)
        barrier()
    dump = {}
    if args.dump_outputs:
        # what the last timed step handed its caller: per-frame counts, keypoints and descriptors of the 64-frame batch; the
        # slots past a frame's count are not written by the extractor and are zeroed here
        last = args.steps - 1
        kq, dq = outs2[last % inflight]
        n = d_counts[last].cpu().numpy()
        valid = (np.arange(NFEAT)[None, :] < n[:, None])[..., None]
        kp = kq.cpu().numpy().view(_capi.KP_DTYPE).reshape(BATCH, NFEAT)
        dump["orb_counts"] = n.astype(np.float32)
        dump["orb_keypoints"] = np.where(valid, kp_columns(kp), 0).astype(np.float32)
        dump["orb_descriptors"] = np.where(valid, dq.cpu().numpy().reshape(BATCH, NFEAT, 32), 0).astype(np.float32)
    kp_total = d_counts[:args.steps].sum()
    orb_ms = max_over_ranks(e0.elapsed_time(e1))
    # the same K steps strictly one after the other on one context / stream (what a single se2gpu_orb handle delivers)
    orb_ms_serial = orb_ms
    if inflight > 1:
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for k in range(args.steps):
            orb_step(k, 1)
        f1.record(stream)
        barrier()
        orb_ms_serial = max_over_ranks(f0.elapsed_time(f1))
    orb_launches = lib.se2gpu_launch_count() - launches0
    # per-kernel times: an identical second pass with a CUDA-event pair around every kernel (this serialises the blur,
    # which the timed pass overlaps with FAST+selection on a side stream, so the per-kernel sum exceeds ms_per_step)
    ext.profile(True)
    for k in range(args.steps):
        orb_step(k, 1)
    torch.cuda.synchronize()
    prof = ext.profile_read()
    ext.profile(False)
    kps_done = sum_over_ranks(float(kp_total.item()))
    orb_value = kps_done / (orb_ms * 1e-3)
    # algorithmic bytes per frame (SURVEY.md section 8d): pyramid pixels P_pyr, 60 B per returned keypoint
    P_pyr = 0
    for l in range(NLEV):
        wl, hl, _ = C.c_int(), C.c_int(), C.c_int()
        lib.se2gpu_orb_level_dims(ext.h, l, C.byref(wl), C.byref(hl), C.byref(_))
        P_pyr += wl.value * hl.value
    kp_per_frame = kps_done / (world * args.steps * BATCH)
    alg = {"pyramid": P_pyr, "orb_fast_cells": P_pyr, "orb_blur": P_pyr, "orb_orient_describe": 60 * kp_per_frame, "orb_select": 8 * kp_per_frame}
    single = {g: v for g, v in prof.items() if v[1] > 0}
    dom = max(single, key=lambda g: single[g][0])
    dom_ms = single[dom][0] / single[dom][1]
    achieved = alg[dom] * BATCH / (dom_ms * 1e-3) / 1e9
    step_alg_bytes = (3 * P_pyr + 60 * kp_per_frame) * BATCH
    roof = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
            "traffic": ncu_traffic(dom), "algorithmic_bytes_per_launch": alg[dom] * BATCH, "peak_source": peak_src, "kernel_ms": dom_ms,
            "kernel_share_of_step": single[dom][0] / sum(v[0] for v in single.values()),
            "per_kernel_ms": {g: v[0] / v[1] for g, v in single.items()},
            "per_kernel_note": "second, event-instrumented pass (kernels serialised); the timed pass runs orb_blur on a side stream (levels 0-1 behind the pyramid tail, the rest next to orb_fast_cells+orb_select)",
            "whole_path_GBps": step_alg_bytes / (orb_ms / args.steps * 1e-3) / 1e9,
            # the path is instruction-issue bound (DESIGN.md section 2): issue-slot utilisation and lane efficiency of the
            # dominant kernel from the committed ncu capture of this round
            "issue": ncu_traffic("issue:" + dom)}
    clocks = clk.summary()

    # e2e: host buffers through the C ABI (H2D of the frames + D2H of keypoints / descriptors / counts inside the timed region).
    #   e2e.value        se2gpu_orb_submit / _wait, two batches in flight: the H2D copy of batch k+1 and the D2H copy of batch
    #                    k-1 overlap the kernels of batch k (page-locked caller buffers)
    #   e2e.sync         se2gpu_orb_extract, one synchronous call per batch (page-locked caller buffers)
    #   e2e.pageable     se2gpu_orb_extract with ordinary pageable caller buffers (what Frame.cpp:25 hands over: a cv::Mat)
    def pinned_out():
        return (torch.empty(BATCH * NFEAT * 28, dtype=torch.uint8).pin_memory().numpy().view(_capi.KP_DTYPE),
                torch.empty(BATCH * NFEAT * 32, dtype=torch.uint8).pin_memory().numpy(), torch.zeros(BATCH, dtype=torch.int32).pin_memory().numpy())
    outs = [pinned_out(), pinned_out()]
    kps_h, desc_h, counts_h = outs[0]

    def orb_e2e(k):
        hb = host_batches[k % NROT].numpy()
        _capi.check(lib.se2gpu_orb_extract(ext.h, hb.ctypes.data, BATCH, W, H, W, W * H, kps_h.ctypes.data, desc_h.ctypes.data,
                                           counts_h.ctypes.data), "se2gpu_orb_extract")
        return int(counts_h.sum())
    e2e_steps = 0 if args.quick else args.steps
    for k in range(0 if args.quick else max(args.warmup, 1)):
        orb_e2e(k)
    barrier()
    t0 = time.perf_counter()
    tot = 0
    for k in range(e2e_steps):
        tot += orb_e2e(k)
    torch.cuda.synchronize()
    e2e_sync_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    orb_e2e_sync_value = sum_over_ranks(float(tot)) / (e2e_sync_ms * 1e-3) if e2e_steps else None
    # pipelined
    def submit(k):
        hb = host_batches[k % NROT].numpy()
        o = outs[k & 1]
        _capi.check(lib.se2gpu_orb_submit(ext.h, hb.ctypes.data, BATCH, W, H, W, W * H, o[0].ctypes.data, o[1].ctypes.data, o[2].ctypes.data),
                    "se2gpu_orb_submit")
    def wait(k):
        _capi.check(lib.se2gpu_orb_wait(ext.h), "se2gpu_orb_wait")
        return int(outs[k & 1][2].sum())
    for k in range(0 if args.quick else 2):        # creates the second context, warms both
        submit(k)
    for k in range(0 if args.quick else 2):
        wait(k)
    barrier()
    t0 = time.perf_counter()
    tot = 0
    for k in range(e2e_steps):
        submit(k)
        if k >= 1:
            tot += wait(k - 1)
    if e2e_steps:
        tot += wait(e2e_steps - 1)
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    orb_e2e_value = sum_over_ranks(float(tot)) / (e2e_ms * 1e-3) if e2e_steps else 0.0
    # pageable caller buffers (input and outputs): staged through the library's page-locked buffers
    page_in = [np.array(host_batches[r].numpy(), copy=True) for r in range(min(NROT, 3))]
    kps_p = np.zeros(BATCH * NFEAT, _capi.KP_DTYPE); desc_p = np.zeros(BATCH * NFEAT * 32, np.uint8); counts_p = np.zeros(BATCH, np.int32)
    pg_steps = e2e_steps
    t0 = time.perf_counter()
    totp = 0
    for k in range(pg_steps):
        hb = page_in[k % len(page_in)]
        _capi.check(lib.se2gpu_orb_extract(ext.h, hb.ctypes.data, BATCH, W, H, W, W * H, kps_p.ctypes.data, desc_p.ctypes.data, counts_p.ctypes.data),
                    "se2gpu_orb_extract")
        totp += int(counts_p.sum())
    e2e_page_ms = (time.perf_counter() - t0) * 1e3
    orb_e2e_page_value = (totp / (e2e_page_ms * 1e-3)) if pg_steps else None
    # single-frame latency of the same host call (the reference extracts one frame per Frame constructor, Frame.cpp:25)
    single_ms = single_page_ms = None
    if e2e_steps:
        one = host_batches[0].numpy()[:1]
        for _ in range(3):
            _capi.check(lib.se2gpu_orb_extract(ext.h, one.ctypes.data, 1, W, H, W, W * H, kps_h.ctypes.data, desc_h.ctypes.data, counts_h.ctypes.data), "se2gpu_orb_extract")
        t0 = time.perf_counter()
        for _ in range(50):
            _capi.check(lib.se2gpu_orb_extract(ext.h, one.ctypes.data, 1, W, H, W, W * H, kps_h.ctypes.data, desc_h.ctypes.data, counts_h.ctypes.data), "se2gpu_orb_extract")
        single_ms = (time.perf_counter() - t0) * 1e3 / 50
        onep = np.array(one, copy=True)                 # pageable frame + pageable outputs: the reference's call pattern (Frame.cpp:25)
        t0 = time.perf_counter()
        for _ in range(50):
            _capi.check(lib.se2gpu_orb_extract(ext.h, onep.ctypes.data, 1, W, H, W, W * H, kps_p.ctypes.data, desc_p.ctypes.data, counts_p.ctypes.data), "se2gpu_orb_extract")
        single_page_ms = (time.perf_counter() - t0) * 1e3 / 50

    # ------------------------------------------------------------------------------------------ matcher
    from se2lam_b200.matcher import FrameView, ORBmatcher
    mimgs = matcher_frames()
    d_mimgs = torch.from_numpy(mimgs).to(dev)
    NP2 = 2 * MATCH_PAIRS
    m_kps = torch.zeros(NP2 * NFEAT * 28, dtype=torch.uint8, device=dev)
    m_desc = torch.zeros(NP2 * NFEAT * 32, dtype=torch.uint8, device=dev)
    m_counts = torch.zeros(NP2, dtype=torch.int32, device=dev)
    ext.extract_device(d_mimgs, NP2, H, W, m_kps, m_desc, m_counts, stream=sptr)
    torch.cuda.synchronize()
    mt = ORBmatcher(0.9, device=local_rank, max_queries=NFEAT, max_db=NFEAT)
    m_prev = torch.zeros(2 * NFEAT, dtype=torch.float32, device=dev)
    m_out = torch.zeros((MATCH_PAIRS, NFEAT), dtype=torch.int32, device=dev)
    m_nm = torch.zeros(MATCH_PAIRS, dtype=torch.int32, device=dev)
    mgrid = FrameView(None, None).grid()

    def match_step(k):
        pi = k % MATCH_PAIRS
        a, b = 2 * pi, 2 * pi + 1
        ORBmatcher.KeypointsToPointsDevice(m_kps.data_ptr() + a * NFEAT * 28, NFEAT, m_prev, d_n=m_counts.data_ptr() + 4 * a, stream=sptr)
        mt.MatchByWindowDevice(m_kps.data_ptr() + a * NFEAT * 28, m_desc.data_ptr() + a * NFEAT * 32, NFEAT,
                               m_kps.data_ptr() + b * NFEAT * 28, m_desc.data_ptr() + b * NFEAT * 32, NFEAT, m_prev, mgrid, 20,
                               m_out[pi], m_nm.data_ptr() + 4 * pi, d_n1=m_counts.data_ptr() + 4 * a, d_n2=m_counts.data_ptr() + 4 * b,
                               stream=sptr)
    msteps = max(args.steps, 1) * MATCH_PAIRS
    for k in range(MATCH_PAIRS):
        match_step(k)
    barrier()
    ml0 = lib.se2gpu_launch_count()
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0.record(stream)
    for k in range(msteps):
        match_step(k)
    m1.record(stream)
    barrier()
    if args.dump_outputs:       # the last timed pair: vnMatches12, the updated vbPrevMatched and the number of matches
        pi = (msteps - 1) % MATCH_PAIRS
        n1 = int(m_counts[2 * pi].item())
        dump["matcher_matches12"] = m_out[pi, :n1].cpu().numpy().astype(np.float32)
        dump["matcher_prev_matched"] = m_prev[:2 * n1].cpu().numpy().reshape(n1, 2)
        dump["matcher_nmatches"] = m_nm[pi:pi + 1].cpu().numpy().astype(np.float32)
    match_ms = max_over_ranks(m0.elapsed_time(m1))
    match_launches = lib.se2gpu_launch_count() - ml0
    match_value = sum_over_ranks(float(msteps)) / (match_ms * 1e-3)
    mt.profile(True)
    for k in range(MATCH_PAIRS):
        match_step(k)
    torch.cuda.synchronize()
    mprof = {g: v for g, v in mt.profile_read().items() if v[1] > 0}
    mt.profile(False)
    mrounds, mfallback = mt.last_rounds()
    mdom = max(mprof, key=lambda g: mprof[g][0])
    mdom_ms = mprof[mdom][0] / mprof[mdom][1]
    # algorithmic bytes per pair: both keypoint sets and descriptor sets read once (60 B per keypoint), vbPrevMatched in/out,
    # vnMatches12 out; the candidate table between k_candidates and k_resolve is an implementation detail and not counted
    match_alg = 2 * NFEAT * 60 + NFEAT * (16 + 4)
    c_h = m_counts.cpu().numpy()
    kps_h2 = m_kps.cpu().numpy().view(_capi.KP_DTYPE).reshape(NP2, NFEAT)
    desc_h2 = m_desc.cpu().numpy().reshape(NP2, NFEAT, 32)
    # e2e: host buffers through the handle's host entry point (upload of both frames + download of matches / vbPrevMatched)
    host_pairs = []
    for pi in range(MATCH_PAIRS):
        a, b = 2 * pi, 2 * pi + 1
        host_pairs.append((FrameView(kps_h2[a, :c_h[a]].copy(), desc_h2[a, :c_h[a]].copy()), FrameView(kps_h2[b, :c_h[b]].copy(), desc_h2[b, :c_h[b]].copy())))
    me2e_steps = 0 if args.quick else msteps
    nm_tot = 0
    t0 = time.perf_counter()
    for k in range(me2e_steps):
        f1, f2 = host_pairs[k % MATCH_PAIRS]
        pv = np.stack([f1.keyPointsUn["x"], f1.keyPointsUn["y"]], axis=1).astype(np.float32)
        n_, _ = mt.MatchByWindow(f1, f2, pv, 20)
        nm_tot += n_
    match_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    match_info = {
        "metric": MATCH_METRIC, "value": match_value, "unit": "frame pairs/s", "higher_is_better": True, "dtype": "u32 popcount",
        "ms_per_pair": match_ms / msteps, "pairs_timed": msteps, "matches_per_pair": float(m_nm.float().mean().item()),
        "config": {"workload": f"MatchByWindow on {MATCH_PAIRS} (frame, shifted frame) pairs of the ORB benchmark texture, {NFEAT} keypoints each, "
                               "device-resident extractor outputs, window 20 px, level offset 1, ratio 0.9",
                   "l2": "inputs are 120 KB per pair: L2 resident by nature of the workload (latency bound)"},
        "e2e": {"value": (sum_over_ranks(float(me2e_steps)) / (match_e2e_ms * 1e-3)) if me2e_steps else None, "unit": "frame pairs/s",
                "h2d_bytes_per_step": 2 * NFEAT * 60 + NFEAT * 8, "d2h_bytes_per_step": NFEAT * 12 + 4},
        "gpu_launches": int(match_launches), "speculative_rounds": mrounds, "sequential_fallback": bool(mfallback),
        "roofline": {"bound": "hbm", "kernel": mdom, "achieved": match_alg / (mdom_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                     "frac": match_alg / (mdom_ms * 1e-3) / 1e9 / hbm_peak, "traffic": ncu_traffic(mdom), "algorithmic_bytes_per_launch": match_alg,
                     "kernel_ms": mdom_ms, "per_kernel_ms": {g: v[0] / v[1] for g, v in mprof.items()},
                     "note": "120 KB per pair: the ceiling is launch + dependency latency (3 launches, a handful of resolve rounds), not HBM"},
    }

    # ------------------------------------------------------------------------------------------ BA
    prob = synth.ba_config("C4")
    ar_bufs = {}

    def allreduce(ptr_, count, op, strm):
        # wrap the library's device buffer as a torch tensor (no copy) and reduce it in place on `strm`
        key = (ptr_, count)
        if key not in ar_bufs:
            class _A:  # __cuda_array_interface__ holder
                pass
            a = _A()
            a.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8", "data": (ptr_, False), "version": 2}
            ar_bufs[key] = torch.as_tensor(a, device=dev)
        t = ar_bufs[key]
        dist.all_reduce(t, op=dist.ReduceOp.SUM if op == 0 else dist.ReduceOp.MAX)
    ba = LocalBA.from_problem(prob, device=local_rank, rank=rank, world=world, allreduce=allreduce if world > 1 else None,
                              stream=sptr)
    exchange = "none (single GPU)"
    if world > 1:
        # one persistent cooperative kernel per rank and optimize(): the kernels sum the envelope of [S|b] and the [chi2, scale, abort]
        # scalars over NVLink peer mappings (CUDA IPC) themselves, handshaking through epoch flags in peer memory; no NCCL on the path.
        # All ranks must agree on the mode: fall back to the NCCL all-reduce everywhere if any rank cannot map its peers.
        def _gather(b):
            out = [None] * world
            dist.all_gather_object(out, b)
            return out
        ok = 1
        try:
            ba.enable_peer_exchange(_gather)
        except Exception as e:      # noqa: BLE001 - e.g. IPC not permitted in this container
            print(f"[bench] rank {rank}: fused peer exchange unavailable ({e}); using the NCCL all-reduce", file=sys.stderr)
            ok = 0
        flag = torch.tensor([ok], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 1:
            exchange = "in-kernel: each rank runs ONE persistent cooperative kernel per optimize(); the kernels sum the envelope of [S|b] and [chi2, scale, abort] over NVLink peer mappings (epoch flags in peer memory), no NCCL call on the path"
        else:
            exchange = "NCCL all-reduce of [S|b] + [chi2,scale] per trial"
            ba = LocalBA.from_problem(prob, device=local_rank, rank=rank, world=world, allreduce=allreduce, stream=sptr)
    for _ in range(max(args.warmup, 1)):
        ba.reset(); ba.optimize(BA_ITERS)
    barrier()
    ba.profile(True)
    bl0 = lib.se2gpu_launch_count()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 0
    barrier()
    b0.record(stream)
    for _ in range(args.steps):
        ba.reset()
        n, st = ba.optimize(BA_ITERS)
        iters += n
    b1.record(stream)
    barrier()
    if args.dump_outputs:       # the last optimize(): estimates and the chi2 after each iteration
        dump["ba_poses"], dump["ba_points"] = ba.get()
        dump["ba_chi2"] = np.ascontiguousarray(st["chi2_after"], np.float64)
    ba_ms = max_over_ranks(b0.elapsed_time(b1))
    ba_launches = lib.se2gpu_launch_count() - bl0
    bprof = ba.profile_read()
    ba.profile(False)
    trials = int(st["trials"].sum())
    ba_value = iters / (ba_ms * 1e-3)
    E, L, P, O = prob.E, prob.L, prob.P, prob.O
    nS = (3 * (P - 1)) * (3 * (P - 1) + 1) // 2
    # algorithmic bytes per kernel per launch (SURVEY.md section 8d terms)
    balg = {"ba_linearize": E * (56 + 48 + 72) + L * 72, "ba_pose_reduce": P * 72 + E * 72, "ba_lm_prep": L * 72 + E * 72,
            "ba_schur": E * 72 + L * 72 + nS * 8, "ba_chol_solve": nS * 8 * 2, "ba_backsub_update": E * 72 + L * (72 + 24) + (P + L) * 48,
            "ba_lm_control": 0, "ba_persistent": 0, "ba_stage_S": nS * 8}
    iter_alg = E * 424 + L * 288 + P * 120 + O * 112 + nS * 8
    balg["ba_persistent"] = iter_alg * iters / max(args.steps, 1)      # one launch = one optimize() = `iters/steps` LM iterations
    bs = {g: v for g, v in bprof.items() if v[1] > 0}
    persistent = "ba_persistent" in bs
    if persistent:   # one launch per optimize(): the roofline kernel is the whole persistent kernel, phases are reported beside it
        phases = {g: v for g, v in bs.items() if g != "ba_persistent"}   # incl. ba_stage_S (TMA bulk copy of S)
        bs = {"ba_persistent": bs["ba_persistent"]}
    bdom = max(bs, key=lambda g: bs[g][0])
    bdom_ms = bs[bdom][0] / bs[bdom][1]
    bach = balg[bdom] / (bdom_ms * 1e-3) / 1e9
    ba_roof = {"bound": "hbm", "kernel": bdom, "achieved": bach, "peak": hbm_peak, "unit": "GB/s", "frac": bach / hbm_peak,
               "traffic": ncu_traffic(bdom), "algorithmic_bytes_per_launch": balg[bdom],
               "peak_source": peak_src, "kernel_ms": bdom_ms, "kernel_share_of_step": bs[bdom][0] / sum(v[0] for v in bs.values()),
               "per_kernel_ms": {g: v[0] / v[1] for g, v in bs.items()},
               "per_phase_ms_per_optimize": ({g: v[0] / v[1] for g, v in phases.items()} if persistent else None),
               "whole_path_GBps": iter_alg / (ba_ms / max(iters, 1) * 1e-3) / 1e9,
               "note": "the window (14 MB/iteration) is L2-resident and launch/latency bound; see DESIGN.md"}
    # e2e: upload the window, optimise, read the estimates back, every step
    t0 = time.perf_counter()
    it2 = 0
    for _ in range(e2e_steps):
        ba.set_problem(prob)
        n, _ = ba.optimize(BA_ITERS)
        ba.get()
        it2 += n
    ba_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    h2d = sum(a.nbytes for a in (prob.poses, prob.points, prob.uv, prob.info, prob.odo_meas, prob.odo_info)) + 4 * (2 * E + 2 * O) + P
    d2h = 8 * 3 * (P + L)

    # ------------------------------------------------------------------------------------------ BA, config 5 (2000 KF / 50k landmarks)
    c5_info = None
    if not args.no_c5:
        prob5 = synth.ba_config("C5")
        ba5 = LocalBA.from_problem(prob5, device=local_rank, rank=rank, world=world, allreduce=allreduce if world > 1 else None, stream=sptr)
        ba5.optimize(C5_ITERS)
        c5_steps = args.steps
        barrier()
        ba5.profile(True)
        c5l0 = lib.se2gpu_launch_count()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        it5 = 0
        barrier()
        c0.record(stream)
        for _ in range(c5_steps):
            ba5.reset()
            n5, st5 = ba5.optimize(C5_ITERS)
            it5 += n5
        c1.record(stream)
        barrier()
        if args.dump_outputs:
            dump["c5_poses"], dump["c5_points"] = ba5.get()
            dump["c5_chi2"] = np.ascontiguousarray(st5["chi2_after"], np.float64)
        c5_ms = max_over_ranks(c0.elapsed_time(c1))
        c5_launches = lib.se2gpu_launch_count() - c5l0
        c5prof = {g: v for g, v in ba5.profile_read().items() if v[1] > 0}
        ba5.profile(False)
        E5, L5, P5, O5 = prob5.E, prob5.L, prob5.P, prob5.O
        n5u = 3 * (P5 - 1)
        band5 = n5u * 18                                          # stored doubles of the reduced system: block half-bandwidth 5
        iter_alg5 = E5 * 424 + L5 * 288 + P5 * 120 + O5 * 112 + band5 * 8
        c5alg = {"ba_linearize": E5 * (56 + 48 + 72) + L5 * 72, "ba_pose_reduce": P5 * 72 + E5 * 72, "ba_lm_prep": L5 * 72 + E5 * 72,
                 "ba_schur": E5 * 72 + L5 * 72 + band5 * 8, "ba_chol_solve": band5 * 8 * 2, "ba_backsub_update": E5 * 72 + L5 * (72 + 24) + (P5 + L5) * 48,
                 "ba_lm_control": 0}
        c5dom = max(c5prof, key=lambda g: c5prof[g][0])
        c5dom_ms = c5prof[c5dom][0] / c5prof[c5dom][1]
        c5ach = c5alg.get(c5dom, 0) / (c5dom_ms * 1e-3) / 1e9 / max(world, 1)
        t0 = time.perf_counter()
        ba5.set_problem(prob5); n5e, _ = ba5.optimize(C5_ITERS); ba5.get()
        c5_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        c5_info = {
            "metric": C5_METRIC, "value": it5 / (c5_ms * 1e-3), "unit": "LM iterations/s", "higher_is_better": True, "dtype": "f64", "scaling": "strong",
            "ms_per_iteration": c5_ms / max(it5, 1), "iterations_timed": it5, "lambda_trials_last_optimize": int(st5["trials"].sum()),
            "config": {"workload": f"BA {P5} KF / {L5} landmarks / {E5} EdgeSE2XYZ + {O5} PreEdgeSE2, Huber, {C5_ITERS} LM iterations per optimize",
                       "parallelism": ("single GPU" if world == 1 else f"landmark-sharded over {world} GPUs, one NCCL all-reduce of the band-stored reduced system ({band5 * 8 / 1e6:.2f} MB) + one of [chi2, scale, stop] per trial") +
                                      "; reduced solve = partitioned block-band LDL^T (ba_band.cu)"},
            "e2e": {"value": n5e / (c5_e2e_ms * 1e-3), "unit": "LM iterations/s", "h2d_bytes_per_step": int(E5 * 48 + (P5 + L5) * 24 + O5 * 80), "d2h_bytes_per_step": int(24 * (P5 + L5)),
                    "note": "set_problem (host re-index of 297k edges) + optimize + get"},
            "gpu_launches": int(c5_launches),
            "roofline": {"bound": "hbm", "kernel": c5dom, "achieved": c5ach, "peak": hbm_peak, "unit": "GB/s", "frac": c5ach / hbm_peak,
                         "traffic": ncu_traffic("c5:" + c5dom), "algorithmic_bytes_per_launch": c5alg.get(c5dom, 0) / max(world, 1), "kernel_ms": c5dom_ms,
                         "per_kernel_ms": {g: v[0] / v[1] for g, v in c5prof.items()},
                         "whole_path_GBps": iter_alg5 / (c5_ms / max(it5, 1) * 1e-3) / 1e9},
        }

    if rank == 0:
        cpu_orb, cpu_ba = cpu_baselines() if (world == 1 and not args.quick) else (None, None)
        line = {
            "metric": ORB_METRIC, "value": orb_value, "unit": "keypoints/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": orb_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": ORB_WORKLOAD,
                       "frames_per_step_per_gpu": BATCH, "parallelism": f"frames sharded over {world} GPU(s), no collective",
                       "l2": f"inputs rotate over {NROT} distinct batches = {NROT * BATCH * W * H / 1e6:.0f} MB > 126 MB L2",
                       "batches_in_flight": inflight,
                       "ms_per_step_one_batch_in_flight": orb_ms_serial / args.steps,
                       "keypoints_per_frame": kp_per_frame},
            "e2e": {"value": orb_e2e_value, "unit": "keypoints/s", "h2d_bytes_per_step": BATCH * W * H,
                    "d2h_bytes_per_step": BATCH * NFEAT * 60 + BATCH * 4, "ms_per_step": e2e_ms / max(args.steps, 1),
                    "api": "se2gpu_orb_submit / se2gpu_orb_wait, two 64-frame batches in flight, page-locked caller buffers",
                    "sync": {"value": orb_e2e_sync_value, "ms_per_step": e2e_sync_ms / max(args.steps, 1), "api": "se2gpu_orb_extract, one synchronous call per batch, page-locked caller buffers"},
                    "pageable": {"value": orb_e2e_page_value, "ms_per_step": (e2e_page_ms / pg_steps) if pg_steps else None,
                                 "api": "se2gpu_orb_extract with pageable caller buffers (staged through the library's page-locked buffers)"},
                    "single_frame_ms": single_ms, "single_frame_pageable_ms": single_page_ms},
            "gpu_launches": int(orb_launches + ba_launches),
            "roofline": roof, "clocks": clocks,
            "secondary": {
                "metric": BA_METRIC, "value": ba_value, "unit": "LM iterations/s", "higher_is_better": True, "dtype": "f64",
                "scaling": "strong", "ms_per_step": ba_ms / args.steps, "iterations_per_step": iters / args.steps,
                "lambda_trials_per_step": trials,
                "config": {"workload": f"local BA {P} KF / {L} landmarks / {E} EdgeSE2XYZ + {O} PreEdgeSE2, Huber, {BA_ITERS} LM iterations",
                           "parallelism": "single GPU, one persistent cooperative kernel per optimize()" if world == 1 else f"landmark-sharded over {world} GPUs; exchange: {exchange}"},
                "e2e": {"value": it2 / (ba_e2e_ms * 1e-3), "unit": "LM iterations/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
                "gpu_launches": int(ba_launches), "roofline": ba_roof},
        }
        line["matcher"] = match_info
        if c5_info:
            line["tertiary"] = c5_info
        line["gpu_launches"] = int(orb_launches + ba_launches + match_launches)
        if cpu_orb:
            line["cpu_baseline"] = cpu_orb
            line["secondary"]["cpu_baseline"] = cpu_ba
            line["matcher"]["cpu_baseline"] = cpu_match(host_pairs)
            if c5_info:
                from oracle import pyoracle
                o5 = pyoracle.BAOracle(prob5)
                t1 = time.perf_counter(); n5c, _ = o5.optimize(3); dt5 = time.perf_counter() - t1
                line["tertiary"]["cpu_baseline"] = {"value": n5c / dt5, "unit": "LM iterations/s", "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
                                                    "sample": "1 x optimize(3) of the same window, single thread (skyline Cholesky)"}
        if args.dump_outputs:       # rank 0's outputs
            write_dump(args.dump_outputs, dump)
        _OUT.write(json.dumps(line) + "\n"); _OUT.flush()
    if world > 1:
        dist.destroy_process_group()


def cpu_baselines():
    """The oracle port timed on this box's host cores on a bounded sample (reported baseline, not the target)."""
    from oracle import pyoracle
    imgs = synth.orb_batch(4)
    o = pyoracle.OrbOracle(NFEAT, 1.2, NLEV, 20)
    o.extract(imgs[0])
    t0 = time.perf_counter()
    tot = 0
    reps = 0
    while time.perf_counter() - t0 < 8.0:
        for im in imgs:
            tot += len(o.extract(im)[0])
        reps += 1
    dt = time.perf_counter() - t0
    cpu_orb = {"value": tot / dt, "unit": "keypoints/s", "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
               "sample": f"{reps * len(imgs)} frames (seeds 1000-1003 repeated), single thread, oracle -O2 no -march"}
    # second, labelled figure (SURVEY 8d): the same sources with -O3 -march=native (FMA contraction still off: the arithmetic,
    # and therefore the keypoints, are the same)
    try:
        import ctypes as C
        # built for this host's CPU at run time, in a temporary directory: the benchmark writes nothing into the tree
        with tempfile.TemporaryDirectory() as tmp:
            native = os.path.join(tmp, "liboracle_native.so")
            subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "native", "CXX=g++", f"NATIVE_LIB={native}"], check=True,
                           timeout=300, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            N = C.CDLL(native)
        N.orb_oracle_create.restype = C.c_void_p
        N.orb_oracle_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int]
        N.orb_oracle_extract.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        N.orb_oracle_destroy.argtypes = [C.c_void_p]
        hn = N.orb_oracle_create(NFEAT, 1.2, NLEV, 20)
        kp = np.zeros(NFEAT, pyoracle.KP_DTYPE); ds = np.zeros((NFEAT, 32), np.uint8)
        t0 = time.perf_counter(); totn = 0
        while time.perf_counter() - t0 < 3.0:
            for im in imgs:
                totn += N.orb_oracle_extract(hn, im.ctypes.data, im.shape[1], im.shape[0], im.strides[0], kp.ctypes.data, ds.ctypes.data)
        cpu_orb["native"] = {"value": totn / (time.perf_counter() - t0), "flags": "-O3 -march=native -ffp-contract=off", "cores": 1}
        N.orb_oracle_destroy(hn)
    except Exception as e:      # noqa: BLE001 - the labelled extra is optional
        cpu_orb["native"] = {"unavailable": str(e)[:120]}
    prob = synth.ba_config("C4")
    t_ba, it_ba, reps = 0.0, 0, 0
    while t_ba < 4.0:
        ob = pyoracle.BAOracle(prob)
        t1 = time.perf_counter()
        n, _ = ob.optimize(BA_ITERS)
        t_ba += time.perf_counter() - t1; it_ba += n; reps += 1
    cpu_ba = {"value": it_ba / t_ba, "unit": "LM iterations/s", "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
              "sample": f"{reps} x optimize({BA_ITERS}) of the same window, single thread"}
    return cpu_orb, cpu_ba


def cpu_match(host_pairs):
    """The matcher oracle (restatement of ORBmatcher::MatchByWindow + the Frame grid) on one host core, bounded sample."""
    from oracle import pyoracle
    from tests.matcher_cases import GRID
    t0 = time.perf_counter(); n = 0
    while time.perf_counter() - t0 < 2.0:
        f1, f2 = host_pairs[n % len(host_pairs)]
        pv = np.stack([f1.keyPointsUn["x"], f1.keyPointsUn["y"]], axis=1).astype(np.float32)
        pyoracle.match_by_window(f1.keyPointsUn, f1.descriptors, f2.keyPointsUn, f2.descriptors, pv, GRID, 20, 1, 0, 8, 0.9)
        n += 1
    return {"value": n / (time.perf_counter() - t0), "unit": "frame pairs/s", "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
            "sample": f"{n} pairs, single thread"}


def _reserve_stdout():
    """Only the final JSON line may reach stdout (NCCL / torch print banners there): point fd 1 at stderr for the
    duration of the run and return a writer bound to the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    global _OUT
    _OUT = _reserve_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every leg (the matcher leg times one pass over its pairs per step)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quick", action="store_true", help="profiling runs: skip the CPU baseline and the e2e legs")
    ap.add_argument("--orb-inflight", type=int, default=1, help="64-frame batches in flight in the device-resident ORB leg (2 = two extractor contexts / streams; measured +1.7 %: the kernels already fill the machine)")
    ap.add_argument("--no-c5", action="store_true", help="skip the BASELINE configs[4] leg (2000 KF / 50k landmarks; ~20 s of host-side synthesis)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of every leg as DIR/<name>.npy "
                                                          "(float32 / float64; inputs are seeded, so two builds can be compared file by file)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this repo's CUDA path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
