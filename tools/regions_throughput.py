"""Throughput and latency of the region calls (CNNAccelerator.detect_regions), with the centre-crop path beside them.

One process, one GPU.  Three workloads over 640x480 BGR frames:
  grid    (a) 63 regions per frame: side 128, stride 64 (grid_regions)
  pyramid (b) 80 regions per frame: sides 480 / 240 / 128, stride side / 2
  centre  (c) one region per frame: the centre crop, i.e. what detect_frames computes
and, host-fed only, grid (a) on every other frame: the staging plan then copies each referenced frame on its own.
For each: host-fed frames/s and regions/s from pinned frames far larger than L2 (host wall clock around calls that return with
the predictions on the host), and device-resident frames/s and regions/s (CUDA events) with the time split into pre-processing
(preprocess_regions) and conv + tail (infer_batch on the same number of 128x128 images).  Beside them from the same run:
detect_frames frames/s host-fed and device-resident, device-resident infer_batch images/s, and batch-1 p50 / p99 of one VGA
frame with grid (a) against detect_frames of one frame.  The card's name and power limit are read in the same run.

    python tools/regions_throughput.py [--frames 2048] [--dev-frames 1024] [--seconds 2] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import fpga_cnn_b200 as fc  # noqa: E402
import inputs  # noqa: E402

H, W = 480, 640


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return [l.strip() for l in r.stdout.splitlines() if l.strip()] or [r.stderr.strip()]


def wall_rate(fn, seconds):
    """calls / s over back-to-back calls of fn for at least `seconds` (after one warm-up call)."""
    fn()
    calls, t0 = 0, time.perf_counter()
    while True:
        fn()
        calls += 1
        dt = time.perf_counter() - t0
        if calls >= 3 and dt >= seconds:
            return calls / dt


def event_ms(fn, seconds):
    """Mean CUDA-event milliseconds of fn on torch's current stream (after one warm-up call)."""
    import torch
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, total, t0 = 0, 0.0, time.perf_counter()
    while reps < 3 or time.perf_counter() - t0 < seconds:
        a.record()
        fn()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
        reps += 1
    return total / reps


def workloads(n):
    centre = np.array([(f, (W - H) // 2, 0, H) for f in range(n)], np.int32)
    return {"grid": fc.grid_regions(n, H, W, 128, 64),
            "pyramid": fc.grid_regions(n, H, W, [480, 240, 128], [240, 120, 64]),
            "centre": centre}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=2048, help="pinned host frames (1.8 GiB at 2048)")
    ap.add_argument("--dev-frames", type=int, default=1024, help="device-resident frames (0.9 GiB at 1024)")
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    dev = torch.device("cuda", 0)
    meta = {"card": card(), "frame": [H, W], "host_frames": a.frames, "dev_frames": a.dev_frames}
    lines = []

    def emit(d):
        d = {**meta, **d}
        lines.append(d)
        print(json.dumps(d), flush=True)

    acc = fc.CNNAccelerator()
    acc.load_weights(os.path.join(ROOT, "tests", "golden", "weights.bin"))
    acc.set_shifts(7, 10, 11)
    acc.load_classifier(*inputs.make_fc())

    host = fc.alloc_host((a.frames, H, W, 3))
    block = inputs.make_frames(("smooth", 1), 16, H, W)
    for i in range(0, a.frames, 16):
        host[i:i + 16] = block[:a.frames - i]

    # host-fed
    per_s = wall_rate(lambda: acc.detect_frames(host), a.seconds)
    emit({"what": "host_fed", "path": "detect_frames", "frames_per_s": per_s * a.frames})
    for name, reg in workloads(a.frames).items():
        per_s = wall_rate(lambda: acc.detect_regions(host, reg), a.seconds)
        emit({"what": "host_fed", "path": "detect_regions", "workload": name, "regions_per_frame": len(reg) / a.frames,
              "frames_per_s": per_s * a.frames, "regions_per_s": per_s * len(reg)})
    # the staging plan's worst case: regions on every other frame, so every referenced frame is a chunk of its own
    sparse = workloads(a.frames)["grid"]
    sparse = sparse[sparse[:, 0] % 2 == 0]
    per_s = wall_rate(lambda: acc.detect_regions(host, sparse), a.seconds)
    emit({"what": "host_fed", "path": "detect_regions", "workload": "grid_every_other_frame", "frames_referenced": a.frames // 2,
          "referenced_frames_per_s": per_s * (a.frames // 2), "regions_per_s": per_s * len(sparse)})

    # device-resident (frames 0.9 GiB, far larger than the 126 MB L2)
    t = torch.from_numpy(host[:a.dev_frames]).to(dev)
    nd = a.dev_frames
    probs = torch.empty((nd, 6), dtype=torch.float32, device=dev)
    cls = torch.empty((nd,), dtype=torch.int32, device=dev)
    box = torch.empty((nd, 4), dtype=torch.int32, device=dev)
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    detect_dev = lambda: acc._check(acc._libc.cnnacc_detect_frames(acc._h, p(t), nd, H, W, None, p(probs), p(cls), p(box),
                                                                   fc._lib.FLAG_DEVICE_PTRS))
    with acc._on_stream_of(t):
        ms = event_ms(detect_dev, a.seconds)
    pre_ms = event_ms(lambda: acc.preprocess(t), a.seconds)
    emit({"what": "device_resident", "path": "detect_frames", "frames_per_s": nd / ms * 1e3, "ms": ms, "preprocess_ms": pre_ms})
    for name, reg in workloads(nd).items():
        ms = event_ms(lambda: acc.detect_regions(t, reg), a.seconds)
        pre_ms = event_ms(lambda: acc.preprocess_regions(t, reg), a.seconds)
        gray = acc.preprocess_regions(t, reg)
        conv_ms = event_ms(lambda: acc.infer_batch(gray), a.seconds)
        del gray
        emit({"what": "device_resident", "path": "detect_regions", "workload": name, "regions": len(reg),
              "frames_per_s": nd / ms * 1e3, "regions_per_s": len(reg) / ms * 1e3, "ms": ms,
              "preprocess_ms": pre_ms, "conv_tail_ms": conv_ms})
    imgs = torch.from_numpy(inputs.make_images(("rng", 5), 16384)).to(dev)     # 256 MiB
    ms = event_ms(lambda: acc.infer_batch(imgs), a.seconds)
    emit({"what": "device_resident", "path": "infer_batch", "images": 16384, "images_per_s": 16384 / ms * 1e3, "ms": ms})
    del t, imgs
    torch.cuda.synchronize()

    # batch 1: one VGA frame (pageable, as a camera loop has it)
    one = np.ascontiguousarray(block[:1])
    grid1 = fc.grid_regions(1, H, W, 128, 64)
    for path, fn in (("detect_regions_grid63", lambda: acc.detect_regions(one, grid1)), ("detect_frames", lambda: acc.detect_frames(one))):
        for _ in range(50):
            fn()
        ts = []
        for _ in range(2000):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e6
        emit({"what": "batch1", "path": path, "p50_us": float(np.percentile(ts, 50)), "p99_us": float(np.percentile(ts, 99))})

    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
