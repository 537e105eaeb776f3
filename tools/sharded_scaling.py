"""How the sharded host-batch calls (MultiAccelerator / cnnacc_*_sharded) scale over the GPUs of one box.

One process.  For N = 1 .. visible GPUs, on pinned host batches far larger than L2 (default 2^18 images = 4 GiB in):
  * sharded infer_batch images/s (H2D only: 16 KiB in, 44 B back), run_batch images/s (16 KiB each way), detect_frames
    frames/s at 640x480 (900 KiB in);
  * a raw-copy ceiling measured in the same run: the same bytes moved as plain concurrent cudaMemcpyAsync copies (torch
    copy_(non_blocking=True) from / to the same pinned buffers, every device at once), H2D only and both directions; every
    rate is also given as a fraction of its ceiling;
  * at N = 1 the sharded call against a plain CNNAccelerator call on the same data.
Then a sweep of the batch size n at N = 2 (two GPUs, or two handles on GPU 0 when there is one): one member against two, the
crossover that sets kMinShardBytes (csrc/shard_plan.h).  Host wall clock around calls that return once the results are on the
host; each figure repeats its call for at least --seconds.  One JSON line per N / per sweep point, also written to --out.

    python tools/sharded_scaling.py [--images 262144] [--frames 4096] [--seconds 2] [--out FILE]
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

PIECE = 64 << 20          # raw copies move 64 MiB pieces


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return [l.strip() for l in r.stdout.splitlines() if l.strip()] or [r.stderr.strip()]


def rate(fn, units, seconds):
    """units / s over back-to-back calls of fn for at least `seconds` (after one warm-up call)."""
    fn()
    calls, t0 = 0, time.perf_counter()
    while True:
        fn()
        calls += 1
        dt = time.perf_counter() - t0
        if calls >= 3 and dt >= seconds:
            return calls * units / dt


def pinned_fill(shape, seed):
    """Pinned host array filled with seeded images, tiled from a 64 MiB block (content does not change the work)."""
    a = fc.alloc_host(shape)
    flat = a.reshape(-1)
    block = np.random.default_rng(seed).integers(0, 256, min(flat.size, PIECE), dtype=np.uint8)
    for i in range(0, flat.size, block.size):
        flat[i:i + block.size] = block[:flat.size - i]
    return a


class RawCopies:
    """Plain concurrent copies of [N shards of] a pinned buffer to / from every device of the member set."""

    def __init__(self, torch, devices):
        self.torch = torch
        self.devices = sorted(set(devices))
        self.d_in = {d: torch.empty(PIECE, dtype=torch.uint8, device=f"cuda:{d}") for d in self.devices}
        self.d_out = {d: torch.empty(PIECE, dtype=torch.uint8, device=f"cuda:{d}") for d in self.devices}
        self.s_in = {d: torch.cuda.Stream(device=d) for d in self.devices}
        self.s_out = {d: torch.cuda.Stream(device=d) for d in self.devices}

    def run(self, h_in, h_out, members_devices):
        """h_in / h_out: flat uint8 torch views of pinned host memory (h_out None = H2D only), cut like the shard plan."""
        torch = self.torch
        k, nbytes = len(members_devices), h_in.numel()
        jobs = []
        for i, d in enumerate(members_devices):
            lo, hi = nbytes * i // k, nbytes * (i + 1) // k
            jobs.append([(d, p, min(p + PIECE, hi)) for p in range(lo, hi, PIECE)])
        for step in range(max(len(j) for j in jobs)):
            for j in jobs:
                if step < len(j):
                    d, a, b = j[step]
                    with torch.cuda.stream(self.s_in[d]):
                        self.d_in[d][:b - a].copy_(h_in[a:b], non_blocking=True)
                    if h_out is not None:
                        with torch.cuda.stream(self.s_out[d]):
                            h_out[a:b].copy_(self.d_out[d][:b - a], non_blocking=True)
        for d in self.devices:
            self.s_in[d].synchronize()
            self.s_out[d].synchronize()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--images", type=int, default=1 << 18)
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--max-gpus", type=int, default=0, help="0 = every visible GPU")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (there is no CPU fallback)")
    n_gpus = torch.cuda.device_count() if a.max_gpus <= 0 else min(a.max_gpus, torch.cuda.device_count())
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    cards = card()
    wt = np.fromfile(os.path.join(ROOT, "tests", "golden", "weights.bin"), dtype=np.uint8)
    fc_w, fc_b = inputs.make_fc()
    n, nf = a.images, a.frames
    imgs = pinned_fill((n, 128, 128), 1)
    feats = fc.alloc_host((n, 64, 16, 16))
    frames = pinned_fill((nf, 480, 640, 3), 2)
    t_imgs, t_feats, t_frames = (torch.from_numpy(x.reshape(-1)) for x in (imgs, feats, frames))
    raw = RawCopies(torch, range(n_gpus))

    def group(devices):
        m = fc.MultiAccelerator(devices)
        m.load_weights(wt)
        m.load_classifier(fc_w, fc_b)
        return m

    for N in range(1, n_gpus + 1):
        devs = list(range(N))
        m = group(devs)
        ceil_h2d = rate(lambda: raw.run(t_imgs, None, devs), n, a.seconds)
        ceil_both = rate(lambda: raw.run(t_imgs, t_feats, devs), n, a.seconds)
        ceil_frames = rate(lambda: raw.run(t_frames, None, devs), nf, a.seconds)
        infer = rate(lambda: m.infer_batch(imgs), n, a.seconds)
        run = rate(lambda: m.run_batch(imgs, out=feats), n, a.seconds)
        detect = rate(lambda: m.detect_frames(frames), nf, a.seconds)
        rec = {"N": N, "devices": devs, "cards": cards, "images": n, "frames": nf,
               "infer_batch_images_per_s": infer, "infer_frac_of_h2d_ceiling": infer / ceil_h2d,
               "run_batch_images_per_s": run, "run_frac_of_both_directions_ceiling": run / ceil_both,
               "detect_frames_per_s": detect, "detect_frac_of_h2d_ceiling": detect / ceil_frames,
               "raw_h2d_ceiling_images_per_s": ceil_h2d, "raw_h2d_GBps": ceil_h2d * 16384 / 1e9,
               "raw_both_directions_ceiling_images_per_s": ceil_both, "raw_both_GBps_per_direction": ceil_both * 16384 / 1e9,
               "raw_h2d_ceiling_frames_per_s": ceil_frames}
        if N == 1:
            plain = m.members[0]
            rec["plain_infer_batch_images_per_s"] = rate(lambda: plain.infer_batch(imgs), n, a.seconds)
            rec["plain_run_batch_images_per_s"] = rate(lambda: plain.run_batch(imgs, out=feats), n, a.seconds)
            rec["sharded_over_plain_infer"] = infer / rec["plain_infer_batch_images_per_s"]
            rec["sharded_over_plain_run"] = run / rec["plain_run_batch_images_per_s"]
        emit(rec)
        m.close()

    if a.no_sweep:
        return
    # one member against two on the same batch, alternating, median of the per-call times
    devs = [0, 1] if n_gpus >= 2 else [0, 0]
    m = group(devs)
    one = m.members[0]
    begin = np.zeros(4, np.int64)
    for k in range(0, 17):
        b = 1 << k
        x, y = imgs[:b], feats[:b]
        used = fc.load().cnnacc_shard_plan_host(b, 2, 16384, begin.ctypes.data_as(ctypes.c_void_p), 4)
        for name, f1, f2 in (("infer_batch", lambda: one.infer_batch(x), lambda: m.infer_batch(x)),
                             ("run_batch", lambda: one.run_batch(x, out=y), lambda: m.run_batch(x, out=y))):
            f1(); f2()
            t1, t2 = [], []
            t_end = time.perf_counter() + max(0.3, a.seconds / 4)
            while len(t1) < 5 or time.perf_counter() < t_end:
                for f, ts in ((f1, t1), (f2, t2)):
                    t0 = time.perf_counter(); f(); ts.append(time.perf_counter() - t0)
            s1, s2 = float(np.median(t1)), float(np.median(t2))
            emit({"sweep": name, "devices": devs, "cards": cards, "n": b, "bytes_in": b * 16384, "members_used": used,
                  "one_member_us": s1 * 1e6, "two_members_us": s2 * 1e6, "speedup": s1 / s2, "calls": len(t1)})


if __name__ == "__main__":
    main()
