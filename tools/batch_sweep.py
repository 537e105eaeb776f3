import sys
sys.path[:0] = ['.', 'tests']
import numpy as np, torch
import fpga_cnn_b200 as fc
wt = np.fromfile('tests/golden/weights.bin', dtype=np.uint8)
acc = fc.CNNAccelerator(device=0); acc.load_weights(wt)
for B in (4096, 16384, 65536):
    nbuf = max(2, (2 << 30) // (B * 32768))
    ins = [torch.randint(0, 256, (B, 128, 128), dtype=torch.uint8, device='cuda') for _ in range(nbuf)]
    outs = [torch.empty((B, 64, 16, 16), dtype=torch.uint8, device='cuda') for _ in range(nbuf)]
    for i in range(nbuf): acc.run_batch(ins[i], out=outs[i])
    acc.synchronize()
    steps = max(20, nbuf * 2)
    acc.timer_start()
    for s in range(steps): acc.run_batch(ins[s % nbuf], out=outs[s % nbuf])
    ms = acc.timer_stop()
    print(f"batch {B}: {nbuf} rotating buffers, {steps} steps: {ms/steps*1e3:.1f} us/step, {B*steps/ms/1e3:.3f} M img/s")
    del ins, outs
