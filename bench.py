#!/usr/bin/env python3
"""bench.py -- throughput of the conv-stack hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the conv stack (128x128 u8 -> 64x16x16 u8, shipped weights.bin, shifts 2/4/6)
over one batch of B synthetic images per GPU -- B = 4096 by default, BASELINE.json's configs[1].  The steps walk
round-robin over enough independent buffer pairs to exceed 2 GiB, so no step finds its data in L2.  `value` is
images/s with the batches already resident in HBM; `e2e` is the same work through the C ABI with pinned HOST buffers
(every step's H2D + D2H inside the timed region): the streaming form of the call (cnnacc_run_batch_async / cnnacc_wait_batch,
four host batches in flight), with the plain synchronous cnnacc_run_batch loop next to it (`e2e.synchronous_call_images_per_s`).  `extra` adds the north_star's batch-65536 throughput, the full pipeline
(configs[2]) and the batch-1 latency.
N > 1: launched by torchrun, one rank per GPU, batch sharded by rank with no data-path collective (weak
scaling: B images per GPU); times are CUDA-event times, max over ranks.
`--impl reference` times the reference's own arm_cnn.c (oracle/_ref, one process per host core because
its static scratch buffers make it non-re-entrant) on the same workload; where oracle/_ref/arm_cnn.so is not built it
times the C restatement oracle/cnn_oracle.c instead, and `cpu_baseline.kind` / `sample` say which.
`--dump-outputs DIR` writes the features the last timed step computed (rank 0's shard) to DIR/features.npy as float32,
so that two builds can be compared output for output: the inputs depend only on the arguments.

Beside the contract line's `value` / `e2e` / `roofline` / `cpu_baseline` the line carries, at every N:
  `sustained`  >= 2 s of back-to-back conv-stack launches with the clocks / power / throttle reasons seen inside them;
  `stream_1m`  BASELINE configs[3]: 2^20 images sharded over the ranks (strong scaling), device-resident, through
               infer_batch in 65536-image chunks (tail inside the conv kernel: 44 B of predictions per image), predictions
               copied by every GPU into ITS slice of one pinned host array shared by the ranks, spot-checked on rank 0
               against the oracle; plus the same call fed from pinned host images (H2D inside the timed region).
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

OPS_PER_IMAGE = 2 * 40_108_032          # 2 x MACs, arm_benchmark.py:237 summed over the three layers
BYTES_PER_IMAGE = 16384 + 16384         # algorithmic HBM traffic: image in + features out
PRED_BYTES = 4 + 6 * 4 + 16             # cls i32 + 6 probs f32 + bbox 4 x i32 (SURVEY.md 8e)
STREAM_IMAGES = 1 << 20                 # BASELINE configs[3]: the "1M-image stream"
STREAM_CHUNK = 65536
SHIFTS = (2, 4, 6)
METRIC = "images/s, bit-exact int8 conv stack (128x128 -> 64x16x16)"


# ------------------------------------------------------------------------------------------------
# pieces that are unit-tested on CPU (tests/test_bench_cpu.py)
# ------------------------------------------------------------------------------------------------
def shard_range(n_total, rank, world):
    """Contiguous range [lo, hi) of a global batch owned by `rank` (SURVEY.md 8e)."""
    lo = (n_total * rank) // world
    hi = (n_total * (rank + 1)) // world
    return lo, hi


def reduce_max(value, dist):
    """MAX over ranks of a python float (identity when torch.distributed is not initialised)."""
    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return value
    import torch
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor([value], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_counts(count, dist):
    """Gather one integer per rank to every rank (used to total the images processed)."""
    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return [count]
    import torch
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor([count], dtype=torch.int64, device=dev)
    out = [torch.zeros_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return [int(o.item()) for o in out]


DUMP_IMAGES = 512                       # 512 x 64x16x16 float32 = 32 MiB


def dump_outputs(out_dir, feats):
    """--dump-outputs: `feats` (torch u8 [n,64,16,16]) -> out_dir/features.npy, float32.  A batch of more than DUMP_IMAGES
    images is sampled at fixed, seeded, sorted image indices, so runs with the same --batch dump the same images."""
    import torch
    n = feats.shape[0]
    idx = np.arange(n) if n <= DUMP_IMAGES else np.sort(np.random.default_rng(0).choice(n, DUMP_IMAGES, replace=False))
    sample = feats[torch.from_numpy(idx).to(feats.device)].cpu().numpy().astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "features.npy"), sample)
    return idx


def ncu_dram_bytes_per_image(kernel_tag="conv"):
    """dram__bytes_read.sum + dram__bytes_write.sum per image of the conv-stack launch, read from the NEWEST committed
    `ncu --set full` summary of that kernel under profiles/ (tools/ncu_summary.py writes the "DRAM traffic per launch"
    line).  Returns (bytes_per_image, file name) or (None, None)."""
    import glob
    import re
    best = None
    for path in glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_summary.txt")):
        name = os.path.basename(path)
        m = re.match(r"r(\d+)_", name)
        if not m:
            continue
        text = open(path).read()
        if "conv_stack_fused_kernel" not in text or ("tail" in name) != (kernel_tag == "tail"):
            continue
        t = re.search(r"DRAM traffic per launch: [\d,]+ B = ([\d,]+) B/image", text)
        if t:
            key = (int(m.group(1)), os.path.getmtime(path), name)
            if best is None or key > best[0]:
                best = (key, int(t.group(1).replace(",", "")), name)
    return (best[1], best[2]) if best else (None, None)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  NVML in a thread (a query takes well under a millisecond,
    so even a few-millisecond region gets samples); `nvidia-smi -lms` as the fallback (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []          # nvidia-smi fallback: (t, csv line)
        self.samples = []        # NVML: (t, sm_mhz, reasons bitmask)
        self.smax = None
        self._stop = False
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid_order = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if uuid_order and all(tok.strip().isdigit() for tok in uuid_order.split(",")):
                idx = int(uuid_order.split(",")[self.gpu])
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.nvml = (pynvml, h)
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll(self):
        pynvml, h = self.nvml
        while not self._stop:
            try:
                mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    rs = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    rs = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.samples.append((time.time(), mhz, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t_begin, t_end):
        if self.nvml is not None:
            self._stop = True
            self.thread.join(timeout=1.0)
            inreg = [(m, r) for ts, m, r in self.samples if t_begin <= ts <= t_end]
            if not inreg:                                     # region shorter than one poll: take the nearest sample
                near = sorted(self.samples, key=lambda x: abs(x[0] - 0.5 * (t_begin + t_end)))[:1]
                inreg = [(m, r) for _, m, r in near]
            reasons = sorted({name for _, r in inreg for name, bit in self.REASONS if r & bit})
            return {"sm_mhz": statistics.median([m for m, _ in inreg]) if inreg else None, "sm_max_mhz": self.smax,
                    "reasons": reasons, "samples": len(inreg), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            in_region = t_begin <= ts <= t_end + 0.1
            try:
                if in_region:
                    sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            if in_region:
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# reference arm: arm_cnn.c on the host cores
# ------------------------------------------------------------------------------------------------
# what the CPU arm timed, by the `kind` _ref_worker reports
CPU_PROGRAMS = {"reference": "the reference's own arm_cnn.c (oracle/_ref/arm_cnn.so)",
                "port": "oracle/cnn_oracle.c, the C restatement of arm_cnn.c (oracle/_ref/arm_cnn.so is not built)"}


def _ref_worker(args):
    """One process = one private mapping of the reference .so (static buffers => never threads)."""
    seed, n_images, weights, shifts, seconds = args
    import oracle
    lib = oracle.load_ref()
    kind = "reference"
    if lib is None:
        lib, kind = oracle.load_port(), "port"
    rng = np.random.default_rng(seed)
    imgs = rng.integers(0, 256, (max(n_images, 1), 128, 128), dtype=np.uint8)
    infer = (lambda im: oracle.ref_infer(lib, im, weights, shifts)) if kind == "reference" else \
            (lambda im: oracle.port_infer(lib, im, weights, shifts))
    infer(imgs[0])                                  # warm the code/data paths
    done, t0 = 0, time.perf_counter()
    if seconds is not None:
        while time.perf_counter() - t0 < seconds:
            infer(imgs[done % len(imgs)])
            done += 1
    else:
        for i in range(n_images):
            infer(imgs[i])
            done += 1
    return done, time.perf_counter() - t0, kind


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_reference_rate(weights, cores, seconds=None, images_per_core=None):
    """images/s of the reference CPU path over `cores` processes; returns (rate, kind, images, wall_s)."""
    jobs = [(1000 + c, images_per_core or 8, weights, SHIFTS, seconds) for c in range(cores)]
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_ref_worker, jobs)
    wall = time.perf_counter() - t0
    rate = sum(d / t for d, t, _ in res)
    return rate, res[0][2], sum(d for d, _, _ in res), wall


def numpy_port_ms(weights, reps=3):
    """ms per image of the numpy restatement (oracle/np_oracle.py), the reference's own slow path
    (dump_arm_features.numpy_infer); reported once beside the C rate, median of `reps`."""
    from oracle import np_oracle
    kern = np_oracle.unpack_weights(weights)
    img = np.random.default_rng(7).integers(0, 256, (128, 128), dtype=np.uint8)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        np_oracle.infer(img, kern, tuple(SHIFTS))
        ts.append(time.perf_counter() - t0)
    return 1000.0 * sorted(ts)[len(ts) // 2]


def run_reference_arm(args, weights):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per_core = 32                                    # bounded sample: cores x 32 images per step
    for _ in range(args.warmup):
        cpu_reference_rate(weights, cores, images_per_core=2)
    rates, total_imgs, t_total = [], 0, 0.0
    kind = "reference"
    for _ in range(args.steps):
        rate, kind, imgs, wall = cpu_reference_rate(weights, cores, images_per_core=per_core)
        rates.append(rate)
        total_imgs += imgs
        t_total += imgs / rate
    value = total_imgs / t_total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8*s8->s32", "data": "synthetic",
        "config": ours_config(args.batch, args.gpus, False),       # the same keys and values as our arm's line
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": kind,
                         "sample": f"{CPU_PROGRAMS[kind]} on the host CPU, {cores} processes x {per_core} images per step (a bounded "
                                   f"sample of the batch), {total_imgs} images in all, gcc -O3 (the reference's own flags)",
                         "cpu_model": _cpu_model()},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
_ORIG_AFFINITY = None


def ours_config(batch, world, direct, nbuf=None):
    """`config` of the JSON line -- identical for both arms (the reference arm samples the same workload)."""
    if nbuf is None:
        nbuf = max(2, -(-(2 << 30) // (batch * BYTES_PER_IMAGE)))
    return {"workload": f"configs[1]: 3-layer int8 conv stack, batch {batch} synthetic 128x128 images per GPU per step, "
                        "bit-exact vs arm_cnn.c",
            "batch_per_gpu": batch, "weights": "shipped weights.bin", "shifts": list(SHIFTS),
            "kernel_path": "direct per-layer" if direct else "fused",
            "l2_policy": "inputs larger than L2: %d buffer pairs walked round-robin, %d MiB in+out in total"
                         % (nbuf, nbuf * batch * BYTES_PER_IMAGE >> 20),
            "parallelism": f"batch-sharded x{world}, no collective"}


class NvmlWindow:
    """SM clock / power / throttle reasons of one GPU sampled in a thread while a measurement runs."""

    def __init__(self, gpu_index, period=0.005):
        self.samples, self._stop, self.thread, self.h, self.period = [], False, None, None, period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            self.h = None

    def __enter__(self):
        if self.h is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        return self

    def _poll(self):
        while not self._stop:
            try:
                self.samples.append((time.time(), float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)),
                                     self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0,
                                     int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception:
                pass
            time.sleep(self.period)

    def __exit__(self, *exc):
        self._stop = True
        if self.thread is not None:
            self.thread.join(timeout=1.0)

    def summary(self, t0, t1):
        s = [x for x in self.samples if t0 <= x[0] <= t1]
        if not s:
            return {"sm_mhz": None, "power_w_max": None, "reasons": ["nvml unavailable"], "samples": 0}
        bits = 0
        for x in s:
            bits |= x[3]
        return {"sm_mhz": statistics.median(x[1] for x in s), "sm_mhz_min": min(x[1] for x in s),
                "power_w_max": max(x[2] for x in s), "samples": len(s),
                "reasons": sorted(name for name, bit in ClockSampler.REASONS if bits & bit)}


def create_shared_predictions(path, n_images):
    """Rank 0: the file behind the ONE host array every rank's GPU copies its predictions into (SURVEY.md 8e)."""
    with open(path, "wb") as f:
        f.truncate(n_images * PRED_BYTES)


def map_shared_predictions(path, n_images):
    """Every rank: map the file -> (raw bytes, cls [n] i32, probs [n,6] f32, bbox [n,4] i32), all views of one mapping laid out
    array after array; a rank writes rows shard_range(n, rank, world) of each."""
    shm = np.memmap(path, dtype=np.uint8, mode="r+", shape=(n_images * PRED_BYTES,))
    cls = shm[:n_images * 4].view(np.int32)
    probs = shm[n_images * 4:n_images * 28].view(np.float32).reshape(n_images, 6)
    bbox = shm[n_images * 28:].view(np.int32).reshape(n_images, 4)
    return shm, cls, probs, bbox


def oracle_spot_check(images, cls, probs, bbox, weights, fc_w, fc_b):
    """Predictions of `images` (numpy [m,128,128]) against the oracle (conv stack: liboracle.so; classifier / box: the numpy
    restatement).  Returns (checked, mismatches)."""
    import oracle
    from oracle import np_oracle
    port = oracle.load_port()
    feats = oracle.port_infer_batch(port, images, weights, SHIFTS)
    bad = 0
    for i in range(len(images)):
        c, p, logits, _ = np_oracle.classify_vec(feats[i], fc_w, fc_b)
        if c != cls[i]:
            top2 = np.sort(logits)[-2:]
            bad += not (top2[1] - top2[0] <= 1e-5 * np.abs(logits).max())
            continue
        bad += not (np.abs(p - probs[i]).max() <= 1e-5 and tuple(int(v) for v in bbox[i]) == np_oracle.bbox_vec(feats[i], c, fc_w)[0])
    return len(images), int(bad)


def run_stream_1m(acc, fc, torch, ddist, rank, world, local, weights, gen):
    """BASELINE configs[3] (see the module docstring).  Strong scaling: 2^20 images in total at every N."""
    import inputs
    fw, fb = inputs.make_fc()
    acc.load_classifier(fw, fb)
    lo, hi = shard_range(STREAM_IMAGES, rank, world)
    n = hi - lo
    imgs = torch.randint(0, 256, (n, 128, 128), dtype=torch.uint8, device="cuda", generator=gen)
    # one host array for the whole job: a /dev/shm file mapped by every rank and page-locked in each (cudaHostRegister), so
    # every GPU copies its predictions straight into its slice and rank 0 reads the gathered result without another copy
    tag = os.environ.get("MASTER_PORT", str(os.getppid() if world > 1 else os.getpid()))
    path = f"/dev/shm/cnnacc_stream_{tag}.bin"
    total = STREAM_IMAGES * PRED_BYTES
    if rank == 0:
        create_shared_predictions(path, STREAM_IMAGES)
    if ddist is not None:
        ddist.barrier()
    shm, h_cls, h_probs, h_bbox = map_shared_predictions(path, STREAM_IMAGES)
    unregister = fc.register_host(shm)
    t_cls, t_probs, t_bbox = (torch.from_numpy(a[lo:hi]) for a in (h_cls, h_probs, h_bbox))
    stream = torch.cuda.Stream(device=local)
    acc.use_stream(stream.cuda_stream)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def one_pass():
        with torch.cuda.stream(stream):
            ev0.record(stream)
            for c0 in range(0, n, STREAM_CHUNK):
                c1 = min(n, c0 + STREAM_CHUNK)
                cls, probs, bbox = acc.infer_batch(imgs[c0:c1])
                t_cls[c0:c1].copy_(cls, non_blocking=True)
                t_probs[c0:c1].copy_(probs, non_blocking=True)
                t_bbox[c0:c1].copy_(bbox, non_blocking=True)
            ev1.record(stream)
        ev1.synchronize()
        return ev0.elapsed_time(ev1)

    one_pass()
    passes = 3
    if ddist is not None:
        ddist.barrier()
    torch.cuda.synchronize()
    l0 = acc.launch_count
    with NvmlWindow(local) as nv:
        t0 = time.time()
        ms = sum(one_pass() for _ in range(passes)) / passes
        t1 = time.time()
    launches = (acc.launch_count - l0) // passes
    ms = reduce_max(ms, ddist)
    if ddist is not None:
        ddist.barrier()
    # rank 0 checks gathered predictions of every rank's slice against the oracle (the images come back from that rank)
    pick = np.linspace(0, n - 1, 16).astype(np.int64)
    sample = imgs[torch.from_numpy(pick).cuda()].cpu()
    if ddist is not None:                                # 16 images per rank travel to rank 0 for the check (not timed)
        allg = [torch.empty_like(sample, device="cuda") for _ in range(world)]
        ddist.all_gather(allg, sample.cuda())
        samples = [g.cpu().numpy() for g in allg]
    else:
        samples = [sample.numpy()]
    out = None
    if rank == 0:
        checked = bad = 0
        for r in range(world):
            rlo, rhi = shard_range(STREAM_IMAGES, r, world)
            idx = rlo + np.linspace(0, rhi - rlo - 1, 16).astype(np.int64)
            c, b = oracle_spot_check(samples[r], h_cls[idx], h_probs[idx], h_bbox[idx], weights, fw, fb)
            checked, bad = checked + c, bad + b
        out = {"images": STREAM_IMAGES, "chunk": STREAM_CHUNK, "images_per_gpu": n, "scaling": "strong",
               "ms": ms, "images_per_s": STREAM_IMAGES / (ms / 1e3), "passes": passes, "gpu_launches_per_pass_per_gpu": launches,
               "pipeline": "infer_batch: conv stack + classifier / CAM-box tail inside one kernel, 44 B of predictions per image to HBM",
               "gather": "every GPU copies its predictions (D2H inside the timed region) into its slice of ONE host array: "
                         "a /dev/shm mapping page-locked in each rank (cnnacc_register_host); no collective",
               "prediction_bytes": total, "oracle_spot_check": {"checked": checked, "mismatches": bad},
               "clocks": nv.summary(t0, t1), "time": "CUDA events on each rank's stream, max over ranks, mean of the passes"}
    # the same call fed from pinned HOST images (H2D inside the timed region; only predictions come back)
    acc.use_stream(None)
    nh = min(n, STREAM_CHUNK)
    h_imgs = fc.alloc_host((nh, 128, 128), np.uint8)
    h_imgs[:] = imgs[:nh].cpu().numpy()
    acc.infer_batch(h_imgs)
    if ddist is not None:
        ddist.barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        got = acc.infer_batch(h_imgs)
    dt = reduce_max(time.perf_counter() - t0, ddist)
    if rank == 0:
        out["host_fed"] = {"images_per_s": world * 3 * nh / dt, "batch_per_gpu": nh, "h2d_bytes_per_call": nh * 16384,
                           "d2h_bytes_per_call": nh * PRED_BYTES,
                           "matches_stream": bool(np.array_equal(got[0], h_cls[lo:lo + nh]) and np.array_equal(got[2], h_bbox[lo:lo + nh]))}
    del imgs
    unregister()
    del t_cls, t_probs, t_bbox, h_cls, h_probs, h_bbox, shm
    if ddist is not None:
        ddist.barrier()
    if rank == 0:
        try:
            os.unlink(path)
        except OSError:
            pass
    return out


def bind_to_gpu_numa_node(gpu_index):
    """Pin this rank to the CPUs NVML reports as local to its GPU, so the pinned host buffers of the e2e leg (and the
    copy-issuing thread) sit on the socket the GPU's PCIe root hangs off.  One process per GPU, as a deployment would run
    it.  Returns a short description for the JSON line; CNNACC_BENCH_AFFINITY=0 turns it off."""
    if os.environ.get("CNNACC_BENCH_AFFINITY", "1") == "0" or not hasattr(os, "sched_setaffinity"):
        return "off"
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        global _ORIG_AFFINITY
        _ORIG_AFFINITY = os.sched_getaffinity(0)
        cpus &= _ORIG_AFFINITY
        if not cpus:
            return "none reported"
        os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} cpus local to gpu {gpu_index} ({min(cpus)}-{max(cpus)})"
    except Exception as e:                           # NVML missing or restricted: run unbound
        return f"unavailable ({type(e).__name__})"


def synthetic_batches(torch, nb, nbuf, rank):
    """The timed loop's `nbuf` device-resident batches of `nb` images from a generator seeded by the rank: the same images on
    every run, and the first k batches do not depend on nbuf.  Returns (generator, batches); later legs draw on."""
    g = torch.Generator(device="cuda")
    g.manual_seed(1234 + rank)
    return g, [torch.randint(0, 256, (nb, 128, 128), dtype=torch.uint8, device="cuda", generator=g) for _ in range(nbuf)]


def run_ours(args, weights):
    import torch
    import torch.distributed as dist
    import fpga_cnn_b200 as fc

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (ours): no CUDA device; there is no CPU fallback. Use --impl reference for the CPU arm.")
    torch.cuda.set_device(local)
    affinity = bind_to_gpu_numa_node(local)          # before any pinned allocation: first touch decides the NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ddist = dist if world > 1 else None

    B = args.batch                                   # images per GPU per step (weak scaling)
    acc = fc.CNNAccelerator(device=local)
    acc.load_weights(weights)
    acc.set_shifts(*SHIFTS)
    stream = torch.cuda.Stream(device=local)
    acc.use_stream(stream.cuda_stream)

    # Synthetic device-resident input: this rank's shard of a world*B image batch, in `nbuf` independent buffer pairs
    # that the timed loop walks round-robin.  Together they are >= 2 GiB, far beyond the 126 MB L2, so no step finds
    # its images (or the lines it will write) in cache.
    lo, hi = shard_range(B * world, rank, world)
    nb = hi - lo
    nbuf = max(2, -(-(2 << 30) // (nb * BYTES_PER_IMAGE)))
    g, imgs = synthetic_batches(torch, nb, nbuf, rank)
    feats = [torch.empty((nb, 64, 16, 16), dtype=torch.uint8, device="cuda") for _ in range(nbuf)]
    torch.cuda.synchronize()

    def barrier():
        if ddist is not None:
            ddist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ----------------------------------------------------------------
    for w in range(args.warmup):
        acc.run_batch(imgs[w % nbuf], out=feats[w % nbuf], direct=args.direct)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.05)
    launches0 = acc.launch_count
    barrier()
    t_begin = time.time()
    acc.timer_start()
    for st in range(args.steps):
        acc.run_batch(imgs[st % nbuf], out=feats[st % nbuf], direct=args.direct)
    ms = acc.timer_stop()
    barrier()
    t_end = time.time()
    launches = acc.launch_count - launches0
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, feats[(args.steps - 1) % nbuf])
    ms = reduce_max(ms, ddist)
    total_images = sum(gather_counts(nb, ddist)) * args.steps
    value = total_images / (ms / 1000.0)

    # ---- sustained: >= 2 s of back-to-back launches of the same step, clocks / power / throttle reasons sampled inside ----
    step_s = ms / args.steps / 1e3
    sus_steps = max(args.steps, int(args.sustained_s / step_s) + 1)
    barrier()
    with NvmlWindow(local) as nv:
        t0s = time.time()
        acc.timer_start()
        for st in range(sus_steps):
            acc.run_batch(imgs[st % nbuf], out=feats[st % nbuf], direct=args.direct)
        sus_ms = acc.timer_stop()
        t1s = time.time()
    sus_ms = reduce_max(sus_ms, ddist)
    sustained = {"images_per_s": sum(gather_counts(nb, ddist)) * sus_steps / (sus_ms / 1e3), "seconds": sus_ms / 1e3, "steps": sus_steps,
                 "clocks": nv.summary(t0s + min(0.3, 0.25 * (t1s - t0s)), t1s)}
    int8_peak_tops, int8_peak_ms = acc.probe_int8_peak(50.0)       # tcgen05 kind::i8 N=256 on every SM, measured in this run

    # ---- end to end through the C ABI with pinned host buffers -------------------------------------
    Be = min(B, args.e2e_batch)
    h_imgs = fc.alloc_host((Be, 128, 128), np.uint8)
    h_feats = fc.alloc_host((Be, 64, 16, 16), np.uint8)
    h_imgs[:] = imgs[0][:Be].cpu().numpy()
    acc.use_stream(None)
    for _ in range(max(1, min(args.warmup, 3))):
        acc.run_batch(h_imgs, out=h_feats, direct=args.direct)
    e2e_steps = max(1, args.steps)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        acc.run_batch(h_imgs, out=h_feats, direct=args.direct)       # synchronous: returns when feats are on the host
    e2e_sync_s = reduce_max(time.perf_counter() - t0, ddist)
    e2e_sync_value = world * Be * e2e_steps / e2e_sync_s
    # The streaming form of the same call (cnnacc_run_batch_async / cnnacc_wait_batch): four host batches in flight, so the first
    # H2D and the last D2H of a step overlap its neighbours'.  Every step still copies its own inputs in and its own features
    # out inside the timed region; the region ends when the last step's features are on the host.
    e2e_depth = 1 if args.direct else 4
    if e2e_depth > 1:
        h_in2 = [h_imgs] + [fc.alloc_host((Be, 128, 128), np.uint8) for _ in range(e2e_depth - 1)]
        h_out2 = [h_feats] + [fc.alloc_host((Be, 64, 16, 16), np.uint8) for _ in range(e2e_depth - 1)]
        for x in h_in2[1:]:
            x[:] = h_imgs

        def streamed(steps):
            pend = []
            for st in range(steps):
                pend.append(acc.run_batch_async(h_in2[st % e2e_depth], out=h_out2[st % e2e_depth]))
                if len(pend) >= e2e_depth:
                    acc.wait_batch(pend.pop(0))
            while pend:
                acc.wait_batch(pend.pop(0))

        streamed(max(e2e_depth, min(args.warmup, 3)))
        for y in h_out2[1:]:
            y[:] = 0
        barrier()
        t0 = time.perf_counter()
        streamed(e2e_steps)
        e2e_s = reduce_max(time.perf_counter() - t0, ddist)
        e2e_value = world * Be * e2e_steps / e2e_s
        e2e_streams_ok = all(np.array_equal(y, h_out2[0]) for y in h_out2[1:min(e2e_depth, e2e_steps)])
    else:
        e2e_s, e2e_value, e2e_streams_ok = e2e_sync_s, e2e_sync_value, True
    acc.use_stream(stream.cuda_stream)
    acc.run_batch(imgs[0], out=feats[0], direct=args.direct)
    acc.synchronize()
    ok = bool(np.array_equal(h_feats[:64], feats[0][:64].cpu().numpy()))
    # The ceiling of that leg on THIS box with THIS many ranks copying at once: the same bytes per step as plain concurrent
    # cudaMemcpyAsync H2D + D2H on two streams (torch copies, no kernels), all ranks together, max over ranks.
    t_h_in, t_h_out = torch.from_numpy(h_imgs), torch.from_numpy(h_feats)
    d_in, d_out = imgs[0][:Be], feats[0][:Be]
    s_in, s_out = torch.cuda.Stream(device=local), torch.cuda.Stream(device=local)

    def raw_copies(reps):
        for _ in range(reps):
            with torch.cuda.stream(s_in):
                d_in.copy_(t_h_in, non_blocking=True)
            with torch.cuda.stream(s_out):
                t_h_out.copy_(d_out, non_blocking=True)
        s_in.synchronize()
        s_out.synchronize()

    raw_copies(2)
    barrier()
    t0 = time.perf_counter()
    raw_copies(e2e_steps)
    raw_s = reduce_max(time.perf_counter() - t0, ddist)
    raw_ceiling = world * Be * e2e_steps / raw_s
    h_feats[:] = 0
    acc.use_stream(None)
    acc.run_batch(h_imgs, out=h_feats, direct=args.direct)      # (the probe overwrote h_feats with d_out: restore a real result)
    acc.use_stream(stream.cuda_stream)

    # ---- BASELINE configs[3]: the sharded 1M-image stream through the full pipeline, at every N ----
    del imgs[1:], feats[1:]
    torch.cuda.empty_cache()
    stream_1m = None if args.no_stream else run_stream_1m(acc, fc, torch, ddist, rank, world, local, weights, g)
    acc.use_stream(stream.cuda_stream)

    # ---- secondary measurements (rank 0 only, N = 1): north_star batch, full pipeline, batch-1 latency ----
    extra = {}
    if world == 1 and not args.quick:
        import inputs
        big = 65536
        bi = [torch.randint(0, 256, (big, 128, 128), dtype=torch.uint8, device="cuda", generator=g) for _ in range(2)]
        bf = [torch.empty((big, 64, 16, 16), dtype=torch.uint8, device="cuda") for _ in range(2)]
        for i in range(3):
            acc.run_batch(bi[i % 2], out=bf[i % 2], direct=args.direct)
        torch.cuda.synchronize()
        acc.timer_start()
        for i in range(6):
            acc.run_batch(bi[i % 2], out=bf[i % 2], direct=args.direct)
        extra["conv_stack_batch65536_images_per_s"] = 6 * big / (acc.timer_stop() / 1000.0)      # the north_star's target condition
        fw, fb = inputs.make_fc()
        acc.load_classifier(fw, fb)
        for i in range(2):
            acc.infer_batch(bi[i % 2], direct=args.direct)
        torch.cuda.synchronize()
        acc.timer_start()
        for i in range(4):
            acc.infer_batch(bi[i % 2], direct=args.direct)
        extra["full_pipeline_batch65536_images_per_s"] = 4 * big / (acc.timer_stop() / 1000.0)   # configs[2]: tail inside the conv kernel
        acc.infer_batch(bi[0], two_kernels=True)
        torch.cuda.synchronize()
        acc.timer_start()
        for i in range(4):
            acc.infer_batch(bi[i % 2], two_kernels=True)
        extra["full_pipeline_two_kernels_images_per_s"] = 4 * big / (acc.timer_stop() / 1000.0)   # A/B: features through HBM
        acc.infer_batch(bi[0], direct=args.direct, bbox="upsampled")
        torch.cuda.synchronize()
        acc.timer_start()
        for i in range(2):
            acc.infer_batch(bi[i % 2], direct=args.direct, bbox="upsampled")
        # the same with Classifier.get_cam_bbox's box (PIL-bilinear upsampled CAM) instead of bbox_vec's
        extra["full_pipeline_upsampled_bbox_images_per_s"] = 2 * big / (acc.timer_stop() / 1000.0)
        del bi, bf
        big5 = torch.randint(0, 256, (1024, 512, 512), dtype=torch.uint8, device="cuda", generator=g)     # configs[4]: 512x512, conv stack only
        out5 = torch.empty((1024, 64, 64, 64), dtype=torch.uint8, device="cuda")
        acc.run_batch(big5, out=out5)
        torch.cuda.synchronize()
        acc.timer_start()
        for _ in range(3):
            acc.run_batch(big5, out=out5)
        extra["conv_stack_512x512_images_per_s"] = 3 * 1024 / (acc.timer_stop() / 1000.0)   # 25 overlapping windows per image
        del big5, out5
        acc.use_stream(None)
        one = h_imgs[0].copy()
        lat, lat_c = [], []
        for i in range(2200):
            t0 = time.perf_counter()
            _, conv_ms, read_ms = acc.infer_one(one)
            lat.append((time.perf_counter() - t0) * 1e3)
            lat_c.append(conv_ms + read_ms)
        lat, lat_c = sorted(lat[200:]), sorted(lat_c[200:])
        extra["batch1_latency_ms"] = {"p50": lat[len(lat) // 2], "p99": lat[int(len(lat) * 0.99)], "iterations": len(lat),
                                      "path": "CNNAccelerator.infer_one: host image in, host features out, zero-copy kernel",
                                      "inside_the_c_call_p50": lat_c[len(lat_c) // 2], "inside_the_c_call_p99": lat_c[int(len(lat_c) * 0.99)]}
        # the real-time loop body for camera-sized frames (realtime_detect.py:582-598): pre-process + conv + classify + box
        acc.use_stream(stream.cuda_stream)           # device-resident leg: launches and timer events on one explicit stream
        vga = torch.randint(0, 256, (1024, 480, 640, 3), dtype=torch.uint8, device="cuda", generator=g)
        acc.preprocess(vga[:64])
        torch.cuda.synchronize()
        acc.timer_start()
        for _ in range(4):
            acc.preprocess(vga)
        extra["preprocess_vga_frames_per_s"] = 4 * 1024 / (acc.timer_stop() / 1000.0)      # device-resident 640x480 BGR frames
        del vga
        acc.use_stream(None)
        frames = fc.alloc_host((64, 480, 640, 3), np.uint8)
        frames[:] = np.random.default_rng(9).integers(0, 256, frames.shape, dtype=np.uint8)
        lat = []
        for i in range(330):
            t0 = time.perf_counter()
            acc.detect_frames(frames[i % 64:i % 64 + 1])
            lat.append((time.perf_counter() - t0) * 1e3)
        lat = sorted(lat[30:])
        extra["detect_frame_vga_latency_ms"] = {"p50": lat[len(lat) // 2], "p99": lat[int(len(lat) * 0.99)], "iterations": len(lat),
                                                "path": "CNNAccelerator.detect_frames: one 640x480 BGR host frame in, class / probs / box out"}
        del frames
        frames = fc.alloc_host((256, 480, 640, 3), np.uint8)      # 225 MiB: the staging ring, steady state
        frames[:] = np.random.default_rng(10).integers(0, 256, frames.shape, dtype=np.uint8)
        acc.detect_frames(frames)
        t0 = time.perf_counter()
        for _ in range(5):
            acc.detect_frames(frames)
        dt = time.perf_counter() - t0
        extra["detect_frames_vga_host_frames_per_s"] = 5 * 256 / dt
        extra["detect_frames_vga_host_h2d_gbs"] = 5 * frames.nbytes / dt / 1e9

    # ---- roofline of the dominant kernel (the conv-stack launch) -------------------------------------
    peaks = load_peaks()
    # The conv-stack launch dominates the step (fused path: exactly one launch per step), so its average
    # launch duration is ms / steps, measured with CUDA events on the launching stream.
    kernel_ms = ms / args.steps
    int8_peak = 2.0 * peaks["bf16_tflops"]
    achieved_tops = nb * OPS_PER_IMAGE / (kernel_ms / 1e3) / 1e12
    sus_tops = nb * OPS_PER_IMAGE / (sus_ms / sus_steps / 1e3) / 1e12
    dram_per_image, dram_file = ncu_dram_bytes_per_image()
    roofline = {
        "bound": "tensor", "achieved": achieved_tops, "peak": int8_peak, "unit": "TOP/s", "frac": achieved_tops / int8_peak,
        "traffic": None if (args.direct or dram_per_image is None) else nb * dram_per_image,
        "traffic_note": f"ncu dram__bytes_read+write per image ({dram_per_image} B, profiles/{dram_file}) x images per launch",
        "peak_note": f"int8 dense peak taken as 2 x {peaks['source']} bf16 burst ({peaks['bf16_tflops']} TF/s); nominal 4500 TOP/s; "
                     "peak_int8_measured = tcgen05.mma kind::i8 M128 N256 K32 back to back on every SM for 50 ms in THIS run",
        "peak_int8_measured": int8_peak_tops, "frac_of_int8_measured": achieved_tops / int8_peak_tops,
        "achieved_sustained": sus_tops, "frac_sustained": sus_tops / (2.0 * peaks["bf16_tflops_sustained"]),
        "frac_sustained_of_int8_measured": sus_tops / int8_peak_tops,
        "peak_sustained": 2.0 * peaks["bf16_tflops_sustained"],
        "algorithmic_ops_per_launch": nb * OPS_PER_IMAGE,
        "algorithmic_bytes_per_launch": nb * BYTES_PER_IMAGE,
        "hbm_achieved_gbs": nb * BYTES_PER_IMAGE / (kernel_ms / 1e3) / 1e9,
        "hbm_peak_gbs": peaks["hbm_gbs"],
        "kernel_ms": kernel_ms,
    }

    if rank == 0:
        if _ORIG_AFFINITY is not None:
            os.sched_setaffinity(0, _ORIG_AFFINITY)  # the CPU baseline uses every core the process was given
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            rate, kind, n_img, wall = cpu_reference_rate(weights, cores, seconds=2.0)
            rate1, _, n1, _ = cpu_reference_rate(weights, 1, seconds=1.0)
            cpu = {"value": rate, "unit": "images/s", "cores": cores, "kind": kind,
                   "sample": f"{CPU_PROGRAMS[kind]}: {n_img} images of the same workload in a 2 s window, one process per core, gcc -O3",
                   "single_core_images_per_s": rate1, "single_core_ms_per_image": 1000.0 / rate1 if rate1 else None,
                   "numpy_port_ms_per_image": numpy_port_ms(weights), "cpu_model": _cpu_model()}
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8*s8->s32", "data": "synthetic",
            "config": ours_config(B, world, args.direct, nbuf),
            "clocks": clocks,
            "sustained": sustained,
            "stream_1m": stream_1m,
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": Be * 16384, "d2h_bytes_per_step": Be * 16384,
                    "batch": Be, "steps": e2e_steps, "host_buffers": "pinned (cnnacc_alloc_host)", "cpu_affinity": affinity,
                    "matches_device_run": ok and e2e_streams_ok,
                    "api": ("cnnacc_run_batch_async + cnnacc_wait_batch, %d host batches in flight" % e2e_depth) if e2e_depth > 1 else "cnnacc_run_batch",
                    "batches_in_flight": e2e_depth, "synchronous_call_images_per_s": e2e_sync_value,
                    "raw_copy_ceiling_images_per_s": raw_ceiling, "frac_of_raw_copy_ceiling": e2e_value / raw_ceiling,
                    "raw_copy_ceiling_note": f"the same {Be * 16384} B H2D + {Be * 16384} B D2H per step as plain concurrent cudaMemcpyAsync on two "
                                             f"streams from the same pinned buffers, no kernels, all {world} rank(s) at once, max over ranks: "
                                             f"{raw_ceiling * 16384 / 1e9 / world:.1f} GB/s per direction per GPU"},
            "gpu_launches": launches,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096, help="images per GPU per step (BASELINE.json configs[1])")
    ap.add_argument("--e2e-batch", type=int, default=4096)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--direct", action="store_true", help="time the generic per-layer kernels instead of the fused one")
    ap.add_argument("--quick", action="store_true", help="skip the secondary measurements")
    ap.add_argument("--no-stream", action="store_true", help="skip the 1M-image stream block")
    ap.add_argument("--sustained-s", type=float, default=2.2, help="length of the sustained leg in seconds")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's features (rank 0's shard, at most %d images) to DIR/features.npy" % DUMP_IMAGES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    weights = np.fromfile(os.path.join(ROOT, "tests", "golden", "weights.bin"), dtype=np.uint8)
    if args.impl == "reference":
        run_reference_arm(args, weights)
    else:
        run_ours(args, weights)


if __name__ == "__main__":
    main()
