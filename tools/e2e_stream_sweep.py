"""Streaming host-buffer calls (run_batch_async / wait_batch): throughput against the number of batches in flight."""
import os, sys, time, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import fpga_cnn_b200 as fc
wt = np.fromfile(os.path.join(ROOT, "tests/golden/weights.bin"), dtype=np.uint8)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
steps = max(12, (40 * 4096) // B)
a = fc.CNNAccelerator(device=0); a.load_weights(wt)
nb = 5
xs = [fc.alloc_host((B, 128, 128), np.uint8) for _ in range(nb)]
ys = [fc.alloc_host((B, 64, 16, 16), np.uint8) for _ in range(nb)]
xs[0][:] = np.random.default_rng(1).integers(0, 256, xs[0].shape, dtype=np.uint8)
for x in xs[1:]: x[:] = xs[0]
def sync_loop(n):
    for _ in range(n): a.run_batch(xs[0], out=ys[0])
def streamed(n, depth):
    pend = []
    for s in range(n):
        pend.append(a.run_batch_async(xs[s % depth], out=ys[s % depth]))
        if len(pend) >= depth: a.wait_batch(pend.pop(0))
    while pend: a.wait_batch(pend.pop(0))
sync_loop(3)
t0 = time.perf_counter(); sync_loop(steps); dt = time.perf_counter() - t0
res = [f"batch={B}: synchronous {steps * B / dt / 1e6:.3f}"]
for depth in (2, 3, 4, 5):
    streamed(depth + 2, depth)
    t0 = time.perf_counter(); streamed(steps, depth); dt = time.perf_counter() - t0
    res.append(f"depth{depth} {steps * B / dt / 1e6:.3f}")
assert all(np.array_equal(y, ys[0]) for y in ys[1:])
print("  ".join(res) + "  M img/s")
