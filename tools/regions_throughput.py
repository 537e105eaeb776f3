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
--objects adds the merging calls: detect_objects (detect_regions + per-frame greedy NMS on the GPU) host-fed and
device-resident beside detect_regions for grid (a) and pyramid (b), merge_regions alone on device tensors at 63 and at
2925 regions per frame (side 128, stride 8), and batch-1 p50 / p99 of detect_objects on one VGA frame with grid (a).
--rects measures rectangle regions (frame, x, y, w, h) instead: detect_regions and detect_objects host-fed and
device-resident on
  aspect  (d) 157 rectangles per frame: 128x128, 256x128 and 128x256 at stride 64 (grid_rects)
  random  (e) 48 seeded random rectangles per frame, 128..640 wide and 128..480 tall
beside grid (a) as squares in the same run, and batch-1 p50 / p99 of one VGA frame with aspect (d).
--scan measures the scanning calls (one conv pass per frame, every 128x128 window at a stride): scan_frames at strides 64,
32, 16 and 8 host-fed and device-resident, alternated with detect_regions on the same grid_regions windows at 64 and 32;
scan_objects at 64 and 8 with score_min 0 and with the 97th percentile of the window scores; batch-1 p50 / p99 of one pageable
frame through scan_frames and scan_objects; the device-time split of scan_frames at stride 8 into gray, conv and window tail
(torch.profiler kernel times, in a pass of its own); how often scan and detect_regions agree on the class of the same window.
--pyramid measures the pyramid calls: scan_pyramid on the VGA four-level set (640x480, 512x384, 320x240, 256x192) at strides
8, 16 and 32 and on 1920x1080 frames with the six-level set (1536x864 .. 256x144) at stride 16, device-resident us per frame
and host-fed frames/s, alternated twice with detect_regions on the same frame rectangles (VGA stride 32 and 16); the
device-time split of scan_pyramid_objects into gray, level resize, conv, window tail and merge (torch.profiler, a pass of its
own) and the conv time of each level alone (run_batch on its gray); batch-1 p50 / p99 of one pageable frame.
--scan-rates --vs-lib LIB compares scan_frames (device-resident us per frame and host-fed frames/s at strides 64 and 8) with
this tree's library and with another build of it, LIB (for example the parent commit's, built in a worktree:
`git worktree add /tmp/parent HEAD~1 && make -C /tmp/parent/fpga-cnn-object-detection-accelerator_b200/csrc`), in
subprocesses alternated --runs times, so both see the same card in the same command.

    python tools/regions_throughput.py [--frames 2048] [--dev-frames 1024] [--seconds 2] [--objects | --rects | --scan | --pyramid |
                                        --scan-rates [--vs-lib LIB --runs 2]]
                                       [--out FILE]
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
    ap.add_argument("--objects", action="store_true", help="measure the merging calls (detect_objects / merge_regions)")
    ap.add_argument("--rects", action="store_true", help="measure rectangle regions (detect_regions / detect_objects)")
    ap.add_argument("--scan", action="store_true", help="measure the scanning calls (scan_frames / scan_objects)")
    ap.add_argument("--pyramid", action="store_true", help="measure the pyramid calls (scan_pyramid / scan_pyramid_objects)")
    ap.add_argument("--scan-rates", action="store_true", help="scan_frames rates at strides 64 and 8 only")
    ap.add_argument("--vs-lib", default=None, help="with --scan-rates: alternate with this other libcnnacc.so")
    ap.add_argument("--runs", type=int, default=2)
    a = ap.parse_args()
    if a.scan_rates:
        return scan_rates(a)
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

    if a.objects:
        objects(a, acc, host, emit)
        return write(a, lines)
    if a.rects:
        rects(a, acc, host, emit)
        return write(a, lines)
    if a.scan:
        scan(a, acc, host, emit)
        return write(a, lines)
    if a.pyramid:
        pyramid(a, acc, host, emit)
        return write(a, lines)

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

    write(a, lines)


def write(a, lines):
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


def objects(a, acc, host, emit):
    """detect_objects beside detect_regions (host-fed and device-resident, alternated in one run), merge_regions alone, batch 1."""
    import torch
    dev = torch.device("cuda", 0)
    kw = dict(score_min=0.0, iou_max=0.5, max_det=100)
    for name in ("grid", "pyramid"):
        reg = workloads(a.frames)[name]
        rates = {}
        for rep in range(2):                                 # alternate the two calls to see the spread
            for path, fn in (("detect_regions", lambda: acc.detect_regions(host, reg)),
                             ("detect_objects", lambda: acc.detect_objects(host, reg, **kw))):
                rates.setdefault(path, []).append(wall_rate(fn, a.seconds) * a.frames)
        for path, r in rates.items():
            emit({"what": "host_fed", "path": path, "workload": name, "regions_per_frame": len(reg) / a.frames,
                  "frames_per_s": max(r), "frames_per_s_runs": r})
        emit({"what": "host_fed", "ratio": "detect_objects/detect_regions", "workload": name,
              "value": max(rates["detect_objects"]) / max(rates["detect_regions"])})
    t = torch.from_numpy(host[:a.dev_frames]).to(dev)
    nd = a.dev_frames
    for name in ("grid", "pyramid"):
        reg = workloads(nd)[name]
        ms = {}
        for rep in range(2):
            for path, fn in (("detect_regions", lambda: acc.detect_regions(t, reg)),
                             ("detect_objects", lambda: acc.detect_objects(t, reg, **kw))):
                ms.setdefault(path, []).append(event_ms(fn, a.seconds))
        for path, m in ms.items():
            emit({"what": "device_resident", "path": path, "workload": name, "regions": len(reg), "ms": min(m), "ms_runs": m,
                  "frames_per_s": nd / min(m) * 1e3})
        emit({"what": "device_resident", "ratio": "detect_objects/detect_regions (frames/s)", "workload": name,
              "value": min(ms["detect_regions"]) / min(ms["detect_objects"])})
    del t
    # the merge alone on device predictions: 63 regions per frame (stride 64) and 2925 (stride 8)
    for stride, frames in ((64, 16384), (8, 1024)):
        reg = fc.grid_regions(frames, H, W, 128, stride)
        n = len(reg)
        rng = np.random.default_rng(stride)
        cls = torch.from_numpy(rng.integers(0, 6, n).astype(np.int32)).to(dev)
        scores = torch.from_numpy(rng.random(n, np.float32)).to(dev)
        b1 = rng.integers(0, 64, (n, 2))
        bbox = torch.from_numpy(np.concatenate([b1, b1 + rng.integers(8, 64, (n, 2))], 1).astype(np.int32)).to(dev)
        ms = event_ms(lambda: acc.merge_regions(reg, cls, scores, bbox, frames, **kw), a.seconds)
        emit({"what": "device_resident", "path": "merge_regions", "regions_per_frame": n // frames, "frames": frames, "ms": ms,
              "frames_per_s": frames / ms * 1e3, "regions_per_s": n / ms * 1e3, "us_per_frame": ms * 1e3 / frames})
    # batch 1: one VGA frame (pageable, as a camera loop has it)
    one = np.ascontiguousarray(host[:1])
    grid1 = fc.grid_regions(1, H, W, 128, 64)
    for path, fn in (("detect_objects_grid63", lambda: acc.detect_objects(one, grid1, **kw)),
                     ("detect_regions_grid63", lambda: acc.detect_regions(one, grid1))):
        for _ in range(50):
            fn()
        ts = []
        for _ in range(2000):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e6
        emit({"what": "batch1", "path": path, "p50_us": float(np.percentile(ts, 50)), "p99_us": float(np.percentile(ts, 99))})


def rect_workloads(n):
    rng = np.random.default_rng(6)
    k = 48
    w, h = rng.integers(128, W + 1, n * k), rng.integers(128, H + 1, n * k)
    rnd = np.stack([np.repeat(np.arange(n), k), rng.integers(0, W + 1 - w), rng.integers(0, H + 1 - h), w, h], 1).astype(np.int32)
    return {"aspect": fc.grid_rects(n, H, W, [(128, 128), (256, 128), (128, 256)], 64), "random": rnd,
            "grid_squares": workloads(n)["grid"]}


def rects(a, acc, host, emit):
    """detect_regions and detect_objects on rectangles, host-fed and device-resident, with grid (a) as squares beside them."""
    import torch
    dev = torch.device("cuda", 0)
    kw = dict(score_min=0.0, iou_max=0.5, max_det=100)
    for name, reg in rect_workloads(a.frames).items():
        for path, fn in (("detect_regions", lambda: acc.detect_regions(host, reg)),
                         ("detect_objects", lambda: acc.detect_objects(host, reg, **kw))):
            per_s = wall_rate(fn, a.seconds)
            emit({"what": "host_fed", "path": path, "workload": name, "regions_per_frame": len(reg) / a.frames,
                  "frames_per_s": per_s * a.frames, "regions_per_s": per_s * len(reg)})
    t = torch.from_numpy(host[:a.dev_frames]).to(dev)
    nd = a.dev_frames
    for name, reg in rect_workloads(nd).items():
        for path, fn in (("detect_regions", lambda: acc.detect_regions(t, reg)),
                         ("detect_objects", lambda: acc.detect_objects(t, reg, **kw))):
            ms = event_ms(fn, a.seconds)
            emit({"what": "device_resident", "path": path, "workload": name, "regions": len(reg), "ms": ms,
                  "frames_per_s": nd / ms * 1e3, "regions_per_s": len(reg) / ms * 1e3})
        pre_ms = event_ms(lambda: acc.preprocess_regions(t, reg), a.seconds)
        emit({"what": "device_resident", "path": "preprocess_regions", "workload": name, "regions": len(reg), "ms": pre_ms,
              "regions_per_s": len(reg) / pre_ms * 1e3})
    del t
    torch.cuda.synchronize()
    one = np.ascontiguousarray(host[:1])
    aspect1 = rect_workloads(1)["aspect"]
    for path, fn in (("detect_regions_aspect157", lambda: acc.detect_regions(one, aspect1)),
                     ("detect_objects_aspect157", lambda: acc.detect_objects(one, aspect1, **kw))):
        for _ in range(50):
            fn()
        ts = []
        for _ in range(2000):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e6
        emit({"what": "batch1", "path": path, "p50_us": float(np.percentile(ts, 50)), "p99_us": float(np.percentile(ts, 99))})


def batch1(emit, path, fn):
    """p50 / p99 wall time of fn over 2000 calls after 50 warm-up calls."""
    for _ in range(50):
        fn()
    ts = []
    for _ in range(2000):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    ts = np.array(ts) * 1e6
    emit({"what": "batch1", "path": path, "p50_us": float(np.percentile(ts, 50)), "p99_us": float(np.percentile(ts, 99))})


def scan(a, acc, host, emit):
    """scan_frames / scan_objects beside detect_regions on the same windows, host-fed and device-resident, each comparison
    alternated twice in this run; batch 1; the stride-8 device-time split; class agreement with detect_regions."""
    import torch
    dev = torch.device("cuda", 0)
    t = torch.from_numpy(host[:a.dev_frames]).to(dev)
    nd = a.dev_frames
    strides = (64, 32, 16, 8)
    for where, frames, n, measure, unit in (("host_fed", host, a.frames, lambda fn: 1.0 / wall_rate(fn, a.seconds), "s"),
                                            ("device_resident", t, nd, lambda fn: event_ms(fn, a.seconds) / 1e3, "s")):
        secs = {}
        for rep in range(2):
            for stride in strides:
                secs.setdefault(("scan_frames", stride), []).append(measure(lambda: acc.scan_frames(frames, stride)))
                if stride in (64, 32):
                    reg = fc.grid_regions(n, H, W, 128, stride)
                    secs.setdefault(("detect_regions", stride), []).append(measure(lambda: acc.detect_regions(frames, reg)))
        for (path, stride), v in secs.items():
            windows = n * len(fc.grid_regions(1, H, W, 128, stride))
            emit({"what": where, "path": path, "stride": stride, "windows_per_frame": windows // n, "s_runs": v,
                  "frames_per_s": n / min(v), "windows_per_s": windows / min(v), "us_per_frame": min(v) / n * 1e6})
        for stride in (64, 32):
            emit({"what": where, "ratio": "scan_frames/detect_regions (frames/s)", "stride": stride,
                  "value": min(secs[("detect_regions", stride)]) / min(secs[("scan_frames", stride)])})
        if where == "device_resident":
            ok = min(secs[("scan_frames", 64)]) <= min(secs[("detect_regions", 64)])
            emit({"what": where, "gate": "scan_frames stride 64 not slower than detect_regions on the same 63 windows",
                  "pass": bool(ok)})
        # scan_objects at 64 and 8: every window a candidate, and only the top 3 % of window scores
        secs = {}
        for stride in (64, 8):
            cls, probs, _ = acc.scan_frames(t[:64], stride)
            sc = probs[torch.arange(len(cls), device=dev), cls.long()].cpu().numpy()
            thr = float(np.percentile(sc, 97))
            for rep in range(2):
                for score_min in (0.0, thr):
                    kw = dict(score_min=score_min, iou_max=0.5, max_det=100)
                    secs.setdefault((stride, score_min), []).append(measure(lambda: acc.scan_objects(frames, stride, **kw)))
                    secs.setdefault((stride, "scan_frames"), []).append(measure(lambda: acc.scan_frames(frames, stride)))
        for (stride, what), v in secs.items():
            emit({"what": where, "path": "scan_frames" if what == "scan_frames" else "scan_objects", "stride": stride,
                  **({} if what == "scan_frames" else {"score_min": what, "candidates": "all" if what == 0.0 else "top 3 %"}),
                  "s_runs": v, "frames_per_s": n / min(v), "us_per_frame": min(v) / n * 1e6})
    # how often a scan window and the detect_regions region on the same square agree on the class (information only)
    for stride in (64, 32):
        reg = fc.grid_regions(64, H, W, 128, stride)
        c_scan = acc.scan_frames(t[:64], stride)[0].cpu().numpy()
        c_reg = acc.detect_regions(t[:64], reg)[0].cpu().numpy()
        emit({"what": "agreement", "stride": stride, "windows": len(reg), "same_class": float((c_scan == c_reg).mean())})
    # device-time split at stride 8 (kernel times from torch.profiler, a pass of its own)
    from torch.profiler import ProfilerActivity, profile
    acc.scan_frames(t, 8)
    torch.cuda.synchronize()
    reps = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            acc.scan_frames(t, 8)
        torch.cuda.synchronize()
    split = {}
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if us <= 0:
            continue
        name = e.key
        part = ("gray" if "gray_full_kernel" in name else "window_tail" if "ScanWindows" in name
                else "conv" if "fused" in name else "other")
        split[part] = split.get(part, 0.0) + us / reps / nd
    emit({"what": "device_split", "path": "scan_frames", "stride": 8, "frames": nd, "us_per_frame": split,
          "kernels": sorted({e.key for e in prof.key_averages()})})
    del t
    torch.cuda.synchronize()
    one = np.ascontiguousarray(host[:1])
    batch1(emit, "scan_frames_stride64", lambda: acc.scan_frames(one, 64))
    batch1(emit, "scan_objects_stride64", lambda: acc.scan_objects(one, 64))
    batch1(emit, "scan_frames_stride8", lambda: acc.scan_frames(one, 8))
    batch1(emit, "scan_objects_stride8", lambda: acc.scan_objects(one, 8))
    batch1(emit, "detect_regions_grid63", lambda: acc.detect_regions(one, fc.grid_regions(1, H, W, 128, 64)))


def scan_rates(a):
    """scan_frames device-resident us per frame and host-fed frames/s at strides 64 and 8 over --frames VGA frames, with the
    library CNNACC_LIB_PATH names (this tree's when unset); with --vs-lib, subprocesses alternate this tree's library and
    that one --runs times."""
    if a.vs_lib:
        lines = []
        for run in range(a.runs):
            for lib in (a.vs_lib, None):
                env = {k: v for k, v in os.environ.items() if k != "CNNACC_LIB_PATH"}
                if lib:
                    env["CNNACC_LIB_PATH"] = os.path.abspath(lib)
                cmd = [sys.executable, os.path.abspath(__file__), "--scan-rates", "--frames", str(a.frames), "--seconds",
                       str(a.seconds)]
                out = subprocess.run(cmd, env=env, capture_output=True, text=True, check=True).stdout
                d = {**json.loads(out.strip().splitlines()[-1]), "run": run, "library": lib or "this tree"}
                lines.append(d)
                print(json.dumps(d), flush=True)
        return write(a, lines)
    import ctypes as c
    import torch
    if os.environ.get("CNNACC_LIB_PATH"):               # another build may predate some of this tree's symbols
        other = c.CDLL(os.environ["CNNACC_LIB_PATH"])
        for name in [k for k in fc._lib.SYMBOLS if not hasattr(other, k)]:
            fc._lib.SYMBOLS.pop(name)
    acc = fc.CNNAccelerator()
    acc.load_weights(os.path.join(ROOT, "tests", "golden", "weights.bin"))
    acc.set_shifts(7, 10, 11)
    acc.load_classifier(*inputs.make_fc())
    host = fc.alloc_host((a.frames, H, W, 3))
    host[:] = inputs.make_frames(("smooth", 1), 1, H, W)
    t = torch.from_numpy(host).cuda()
    d = {"card": card(), "frame": [H, W], "frames": a.frames}
    for stride in (64, 8):
        d[f"dev_us_per_frame_s{stride}"] = event_ms(lambda: acc.scan_frames(t, stride), a.seconds) / a.frames * 1e3
        d[f"host_frames_per_s_s{stride}"] = wall_rate(lambda: acc.scan_frames(host, stride), a.seconds) * a.frames
    print(json.dumps(d), flush=True)


VGA_LEVELS = [(640, 480), (512, 384), (320, 240), (256, 192)]
P1080_LEVELS = [(1536, 864), (1280, 720), (1024, 576), (768, 432), (512, 288), (256, 144)]


def profile_split(acc, fn, n, reps=5):
    """us per frame of fn's kernels by part (torch.profiler CUDA kernel times, a pass of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    split = {}
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if us <= 0:
            continue
        name = e.key
        part = ("gray" if "gray_full_kernel" in name else "level_resize" if "pyramid_levels_kernel" in name
                else "window_tail" if "ScanWindows" in name else "merge" if "merge" in name
                else "conv" if "fused" in name else "other")
        split[part] = split.get(part, 0.0) + us / reps / n
    return split, sorted({e.key for e in prof.key_averages()})


def pyramid(a, acc, host, emit):
    """scan_pyramid beside detect_regions on the same rectangles, host-fed and device-resident, alternated twice in this
    run; the 1080p six-level set; the device-time split and per-level conv; batch 1."""
    import torch
    dev = torch.device("cuda", 0)
    t = torch.from_numpy(host[:a.dev_frames]).to(dev)
    nd = a.dev_frames
    for where, frames, n, measure in (("host_fed", host, a.frames, lambda fn: 1.0 / wall_rate(fn, a.seconds)),
                                      ("device_resident", t, nd, lambda fn: event_ms(fn, a.seconds) / 1e3)):
        secs = {}
        for rep in range(2):
            for stride in (8, 16, 32):
                secs.setdefault(("scan_pyramid", stride), []).append(measure(lambda: acc.scan_pyramid(frames, VGA_LEVELS, stride)))
                if stride in (16, 32) and where == "device_resident":
                    k = min(n, 64)                              # detect_regions converts and convolves every window on its own
                    reg = fc.pyramid_windows(k, H, W, VGA_LEVELS, stride)
                    secs.setdefault(("detect_regions", stride), []).append(
                        measure(lambda: acc.detect_regions(frames[:k], reg)) * n / k)
        for (path, stride), v in secs.items():
            per = len(fc.pyramid_windows(1, H, W, VGA_LEVELS, stride))
            emit({"what": where, "path": path, "levels": VGA_LEVELS, "stride": stride, "windows_per_frame": per, "s_runs": v,
                  "frames_per_s": n / min(v), "windows_per_s": n * per / min(v), "us_per_frame": min(v) / n * 1e6})
        if where == "device_resident":
            for stride in (16, 32):
                emit({"what": where, "ratio": "scan_pyramid/detect_regions (frames/s), same rectangles", "stride": stride,
                      "value": min(secs[("detect_regions", stride)]) / min(secs[("scan_pyramid", stride)])})
    split, kernels = profile_split(acc, lambda: acc.scan_pyramid_objects(t, VGA_LEVELS, 16), nd)
    emit({"what": "device_split", "path": "scan_pyramid_objects", "levels": VGA_LEVELS, "stride": 16, "score_min": 0.0,
          "frames": nd, "us_per_frame": split, "kernels": kernels})
    gray = acc.preprocess_pyramid(t, VGA_LEVELS)
    o = 0
    for w, h in VGA_LEVELS:
        g = gray[:, o:o + w * h].reshape(nd, h, w).contiguous()
        o += w * h
        emit({"what": "device_split", "path": "run_batch of one level's gray", "level": [w, h],
              "us_per_frame": event_ms(lambda: acc.run_batch(g), a.seconds) / nd * 1e3})
    del gray, g, t
    torch.cuda.synchronize()
    # 1920x1080 frames, six levels at stride 16
    n_hd = max(1, min(a.dev_frames // 8, 128))
    hd = fc.alloc_host((n_hd, 1080, 1920, 3))
    hd[:] = inputs.make_frames(("smooth", 3), 1, 1080, 1920)
    td = torch.from_numpy(hd).to(dev)
    per = len(fc.pyramid_windows(1, 1080, 1920, P1080_LEVELS, 16))
    for where, frames, measure in (("host_fed", hd, lambda fn: 1.0 / wall_rate(fn, a.seconds)),
                                   ("device_resident", td, lambda fn: event_ms(fn, a.seconds) / 1e3)):
        v = [measure(lambda: acc.scan_pyramid(frames, P1080_LEVELS, 16)) for _ in range(2)]
        emit({"what": where, "path": "scan_pyramid", "frame": [1080, 1920], "levels": P1080_LEVELS, "stride": 16,
              "windows_per_frame": per, "s_runs": v, "frames_per_s": n_hd / min(v), "us_per_frame": min(v) / n_hd * 1e6})
    split, kernels = profile_split(acc, lambda: acc.scan_pyramid_objects(td, P1080_LEVELS, 16), n_hd)
    emit({"what": "device_split", "path": "scan_pyramid_objects", "frame": [1080, 1920], "levels": P1080_LEVELS, "stride": 16,
          "score_min": 0.0, "frames": n_hd, "us_per_frame": split, "kernels": kernels})
    del td
    torch.cuda.synchronize()
    one = np.ascontiguousarray(host[:1])
    one_hd = np.ascontiguousarray(hd[:1])
    batch1(emit, "scan_pyramid_vga_stride16", lambda: acc.scan_pyramid(one, VGA_LEVELS, 16))
    batch1(emit, "scan_pyramid_objects_vga_stride16", lambda: acc.scan_pyramid_objects(one, VGA_LEVELS, 16))
    batch1(emit, "scan_pyramid_1080p_stride16", lambda: acc.scan_pyramid(one_hd, P1080_LEVELS, 16))
    batch1(emit, "scan_frames_vga_stride16", lambda: acc.scan_frames(one, 16))


if __name__ == "__main__":
    main()
