"""Host-fed infer_batch (H2D of the images + 44 B of predictions back) against a plain H2D copy of the same pinned buffer."""
import os, sys, time, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import fpga_cnn_b200 as fc, inputs
wt = np.fromfile(os.path.join(ROOT, "tests/golden/weights.bin"), dtype=np.uint8)
acc = fc.CNNAccelerator(device=0); acc.load_weights(wt); acc.load_classifier(*inputs.make_fc())
n = 65536
h = fc.alloc_host((n, 128, 128), np.uint8); h[:] = np.random.default_rng(1).integers(0, 256, h.shape, dtype=np.uint8)
d = torch.empty((n, 128, 128), dtype=torch.uint8, device="cuda"); th = torch.from_numpy(h)
for piece in (n, 2048):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(3):
        for i in range(0, n, piece): d[i:i + piece].copy_(th[i:i + piece], non_blocking=True)
    torch.cuda.synchronize(); dt = time.perf_counter() - t0
    print(f"plain H2D, {piece * 16384 >> 20} MiB pieces: {3 * n * 16384 / dt / 1e9:.1f} GB/s = {3 * n / dt / 1e6:.2f} M img/s")
acc.infer_batch(h)
for rep in range(2):
    t0 = time.perf_counter()
    for _ in range(3): acc.infer_batch(h)
    dt = time.perf_counter() - t0
    print(f"infer_batch host-fed: {3 * n / dt / 1e6:.2f} M img/s = {3 * n * 16384 / dt / 1e9:.1f} GB/s")
t0 = time.perf_counter()
for _ in range(3): acc.infer_batch(h, two_kernels=True)
dt = time.perf_counter() - t0
print(f"  two kernels: {3 * n / dt / 1e6:.2f} M img/s")
# ---- the same pipeline rebuilt from torch pieces: which part costs the H2D rate? ----
sA, sK, sD = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
piece = 2048
slots = [torch.empty((piece, 128, 128), dtype=torch.uint8, device="cuda") for _ in range(4)]
hp = torch.empty((n, 6), dtype=torch.float32).pin_memory()
def emu(kernel, d2h):
    evk = [None] * 4
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for rep in range(3):
        for ci, i in enumerate(range(0, n, piece)):
            sl = slots[ci % 4]
            with torch.cuda.stream(sA):
                if evk[ci % 4] is not None: sA.wait_event(evk[ci % 4])
                sl.copy_(th[i:i + piece], non_blocking=True)
                ev = torch.cuda.Event(); ev.record(sA)
            if kernel:
                sK.wait_event(ev)
                acc.use_stream(sK.cuda_stream)
                cls, probs, bbox = acc.infer_batch(sl)
                e2 = torch.cuda.Event(); e2.record(sK); evk[ci % 4] = e2
                if d2h:
                    sD.wait_event(e2)
                    with torch.cuda.stream(sD): hp[i:i + piece].copy_(probs, non_blocking=True)
    torch.cuda.synchronize(); dt = time.perf_counter() - t0
    acc.use_stream(None)
    return 3 * n / dt / 1e6
print(f"emulated ring, H2D only: {emu(False, False):.2f} M img/s; + kernel: {emu(True, False):.2f}; + kernel + D2H of probs: {emu(True, True):.2f}")
x = torch.empty((piece, 128, 128), dtype=torch.uint8, device="cuda")
def emu_busy():      # H2D while an unrelated conv kernel stream keeps the SMs busy
    acc.use_stream(sK.cuda_stream)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for rep in range(3):
        for ci, i in enumerate(range(0, n, piece)):
            with torch.cuda.stream(sA): slots[ci % 4].copy_(th[i:i + piece], non_blocking=True)
            acc.infer_batch(x); acc.infer_batch(x); acc.infer_batch(x)
    torch.cuda.synchronize(); dt = time.perf_counter() - t0
    acc.use_stream(None)
    return 3 * n / dt / 1e6
print(f"H2D with independent kernels running all the time: {emu_busy():.2f} M img/s")
