import os, sys, time
sys.path[:0] = [os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests')]
import numpy as np
import fpga_cnn_b200 as fc
wt = np.fromfile(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden', 'weights.bin'), dtype=np.uint8)
acc = fc.CNNAccelerator(device=0); acc.load_weights(wt)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
h_imgs = fc.alloc_host((B, 128, 128), np.uint8); h_feats = fc.alloc_host((B, 64, 16, 16), np.uint8)
h_imgs[:] = np.random.default_rng(0).integers(0, 256, h_imgs.shape, dtype=np.uint8)
for _ in range(2): acc.run_batch(h_imgs, out=h_feats)
t0 = time.perf_counter()
for _ in range(20): acc.run_batch(h_imgs, out=h_feats)
dt = (time.perf_counter() - t0) / 20
print(f'batch {B}:', f'{B/dt/1e6:.3f} M img/s', f'{2*B*16384/dt/1e9:.1f} GB/s both ways')
