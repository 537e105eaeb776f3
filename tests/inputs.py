"""Seeded synthetic inputs shared by tests/, tests/golden/make_golden.py, bench.py and smoke().

Everything is integer arithmetic on numpy Generators so the same seeds give the same bytes in
the build container and on the GPU box.  Shapes follow SURVEY.md 8(d).
"""
import numpy as np

NUM_WEIGHT_BYTES = 23184


def tb_image(H=128, W=128):
    """sim/top/tb.v:522-527 stimulus: pixel[i] = (i*13 + 5) % 256."""
    i = np.arange(H * W, dtype=np.int64)
    return ((i * 13 + 5) % 256).astype(np.uint8).reshape(H, W)


def smooth_images(seed, n, H=128, W=128):
    """Low-frequency images: integer bilinear upsample of a coarse random grid + small noise."""
    rng = np.random.default_rng(seed)
    step = 16
    gh, gw = H // step + 1, W // step + 1
    grid = rng.integers(0, 256, (n, gh, gw)).astype(np.int64)
    ys, xs = np.arange(H), np.arange(W)
    y0, fy = ys // step, ys % step
    x0, fx = xs // step, xs % step
    a = grid[:, y0][:, :, x0]
    b = grid[:, y0][:, :, x0 + 1]
    c = grid[:, y0 + 1][:, :, x0]
    d = grid[:, y0 + 1][:, :, x0 + 1]
    fy = fy[None, :, None]
    fx = fx[None, None, :]
    top = a * (step - fx) + b * fx
    bot = c * (step - fx) + d * fx
    img = (top * (step - fy) + bot * fy) // (step * step)
    img = img + rng.integers(-6, 7, img.shape)
    return np.clip(img, 0, 255).astype(np.uint8)


def make_images(kind, n, H=128, W=128):
    """kind: 'tb' | ('rng', seed) | ('smooth', seed) | ('const', value)."""
    if kind == "tb":
        return np.broadcast_to(tb_image(H, W), (n, H, W)).copy()
    tag, arg = kind
    if tag == "rng":
        return np.random.default_rng(arg).integers(0, 256, (n, H, W), dtype=np.uint8)
    if tag == "smooth":
        return smooth_images(arg, n, H, W)
    if tag == "const":
        return np.full((n, H, W), arg, dtype=np.uint8)
    if tag == "bright":                         # 160..255: keeps the early layers near saturation (24-bit wrap cases)
        return np.random.default_rng(arg).integers(160, 256, (n, H, W), dtype=np.uint8)
    raise ValueError(kind)


def pack_weights(kernels):
    """[k0 (16,1,3,3), k1 (32,16,3,3), k2 (64,32,3,3)] int -> weights.bin bytes, file order [layer][ob][ic][c16][tap9]
    (the inverse of parse_kernels, arm_cnn.c:43-59; the writer is train_cnn.py:174-195)."""
    out = []
    for k in kernels:
        oc, ic = k.shape[:2]
        raw = np.asarray(k, dtype=np.int8).reshape(oc // 16, 16, ic, 3, 3).transpose(0, 2, 1, 3, 4)
        out.append(np.ascontiguousarray(raw).reshape(-1).view(np.uint8))
    w = np.concatenate(out)
    assert w.size == NUM_WEIGHT_BYTES
    return w


def make_weights(kind, shipped=None):
    """kind: 'shipped' | 'identity' | ('rng', seed) | ('const', byte) | ('sparse', seed) | ('acc24', seed) | 'acc24_extreme' |
    ('ternary', seed)."""
    if kind == "shipped":
        assert shipped is not None and shipped.size == NUM_WEIGHT_BYTES
        return np.array(shipped, dtype=np.uint8)
    if kind == "identity":                      # tb.v:501-513: all zero except byte 4 (core 0, centre tap) = 1
        w = np.zeros(NUM_WEIGHT_BYTES, dtype=np.uint8)
        w[4] = 1
        return w
    if kind == "acc24_extreme":                 # every layer-2 sum of an interior pixel is +-288*127*255 = +-9.33 M: beyond 2^23
        k2 = np.where((np.arange(64) % 2 == 0)[:, None, None, None], 127, -127) * np.ones((64, 32, 3, 3), dtype=np.int64)
        return pack_weights([np.full((16, 1, 3, 3), 127), np.full((32, 16, 3, 3), 127), k2])
    tag, arg = kind
    if tag == "ternary":                        # weights in {-1, 0, 1}: with shifts near (1,3,3) every layer's sums straddle 2^shift
        rng = np.random.default_rng(arg)
        return pack_weights([rng.integers(-1, 2, s) for s in ((16, 1, 3, 3), (32, 16, 3, 3), (64, 32, 3, 3))])
    if tag == "acc24":                          # large same-sign layer-2 kernels on near-saturated inputs: sums straddle 2^23
        rng = np.random.default_rng(arg)
        k0 = rng.integers(64, 128, (16, 1, 3, 3))
        k1 = rng.integers(rng.integers(70, 125, (32, 1, 1, 1)), 128, (32, 16, 3, 3))
        sign = np.where(np.arange(64) % 3 == 2, -1, 1)[:, None, None, None]
        k2 = sign * rng.integers(rng.integers(100, 127, (64, 1, 1, 1)), 128, (64, 32, 3, 3))
        return pack_weights([k0, k1, k2])
    if tag == "rng":                            # full range: bytes 0..255 == s8 -128..127
        return np.random.default_rng(arg).integers(0, 256, NUM_WEIGHT_BYTES, dtype=np.uint8)
    if tag == "const":
        return np.full(NUM_WEIGHT_BYTES, arg, dtype=np.uint8)
    if tag == "sparse":                         # mostly zero taps (exercises the kv==0 skip, arm_cnn.c:101)
        rng = np.random.default_rng(arg)
        w = rng.integers(0, 256, NUM_WEIGHT_BYTES, dtype=np.uint8)
        w[rng.random(NUM_WEIGHT_BYTES) < 0.8] = 0
        return w
    raise ValueError(kind)


def make_fc(seed=1234, n_cls=6):
    """Seeded (n_cls,1024) f32 classifier (the shipped fc_weight.npy is the stale (6,64) GAP one)."""
    rng = np.random.default_rng(seed)
    w = (rng.standard_normal((n_cls, 1024)) * 0.1).astype(np.float32)
    b = (rng.standard_normal(n_cls) * 0.1).astype(np.float32)
    return w, b


# 128x128 cases pinned by tests/golden/conv_cases.npz (outputs produced by the reference itself).
CONV_CASES = [
    dict(name="tb_identity", weights="identity", images="tb", n=1, shifts=(0, 0, 0), dump=True),
    dict(name="tb_shipped_default", weights="shipped", images="tb", n=1, shifts=(2, 4, 6), tail=True),
    dict(name="rng_shipped_default", weights="shipped", images=("rng", 0), n=8, shifts=(2, 4, 6), tail=True),
    dict(name="rng_shipped_mid", weights="shipped", images=("rng", 1), n=8, shifts=(7, 10, 11), dump=True, tail=True),
    dict(name="rng_random_mid", weights=("rng", 7), images=("rng", 2), n=4, shifts=(9, 12, 13), dump=True, tail=True),
    dict(name="shipped_shift0", weights="shipped", images=("rng", 3), n=2, shifts=(0, 0, 0)),
    dict(name="shipped_shift31", weights="shipped", images=("rng", 4), n=2, shifts=(31, 31, 31)),
    dict(name="smooth_shipped", weights="shipped", images=("smooth", 5), n=6, shifts=(6, 9, 10), tail=True),
    dict(name="smooth_random", weights=("rng", 11), images=("smooth", 6), n=4, shifts=(8, 12, 13), tail=True),
    dict(name="max_pos_weights", weights=("const", 0x7F), images=("const", 255), n=1, shifts=(11, 14, 15)),
    dict(name="min_neg_weights", weights=("const", 0x80), images=("rng", 8), n=1, shifts=(0, 0, 0)),
    dict(name="sparse_weights", weights=("sparse", 9), images=("rng", 10), n=3, shifts=(5, 7, 8), tail=True),
    dict(name="mixed_shifts", weights=("rng", 12), images=("smooth", 13), n=3, shifts=(3, 13, 9)),
]

# 24-bit wrapping accumulator (cnnacc_set_accumulator_bits(24)): outputs produced by the reference's own bit-accurate model,
# training/train_cnn.py:101-116 fpga_conv_layer, through tests/golden/make_acc24_golden.py -> acc24_cases.npz.  Weights stay
# within +-127 (that function clamps them).  The *_wrap cases are built so that layer 2 really leaves the 24-bit range.
ACC24_CASES = [
    dict(name="acc24_extreme", weights="acc24_extreme", images=("const", 255), n=1, shifts=(0, 0, 15), wraps=True),
    dict(name="acc24_wrap_a", weights=("acc24", 31), images=("bright", 32), n=3, shifts=(0, 14, 15), wraps=True),
    dict(name="acc24_wrap_b", weights=("acc24", 33), images=("bright", 34), n=3, shifts=(0, 13, 16), wraps=True),
    dict(name="acc24_wrap_smooth", weights=("acc24", 35), images=("smooth", 36), n=2, shifts=(0, 14, 15), wraps=True),
    dict(name="acc24_shipped_nowrap", weights="shipped", images=("rng", 1), n=4, shifts=(7, 10, 11), wraps=False),
    dict(name="acc24_sparse_nowrap", weights=("sparse", 9), images=("rng", 10), n=2, shifts=(5, 7, 8), wraps=False, clamp127=True),
]

# generic H x W cases (oracle = arm_benchmark.arm_conv_layer; arm_cnn.c is 128x128 only)
HW_CASES = [
    dict(name="hw_256x256", weights="shipped", images=("rng", 20), H=256, W=256, shifts=(7, 10, 11)),
    dict(name="hw_64x32", weights=("rng", 21), images=("rng", 22), H=64, W=32, shifts=(9, 12, 13)),
    dict(name="hw_512x512", weights="shipped", images=("smooth", 23), H=512, W=512, shifts=(6, 9, 10)),
]


# Workloads on which a one-LSB error shows.  Every layer ends in >> shift and a clip to 0..255, so an accumulator that is off
# by one changes an output byte only when its sum sits next to a multiple of 2^shift and its byte is not clipped: with the
# shipped weights at shifts (7,10,11) a +1 on every layer-2 accumulator changes about one final byte in 10 000.  Weights in
# {-1, 0, 1} at shifts near (1,3,3) keep 30-70 % of every layer's bytes strictly inside (0, 255) and let such a +1 change
# 3-25 % of the final bytes; tests/test_exposure_cpu.py measures both with the numpy oracle and holds every entry to them.
# images: (kind, count) pieces in order; more: the kind that workload_images() draws further images (or other sizes) from.
# acc24_wrap runs with 24-bit accumulators and is built to wrap, not to expose one LSB: a wrapped layer-2 sum is at least
# 2^24 - 9.4 M = 7.4 M away from zero, so only shifts of 15 and up give bytes inside (0, 255), and a +1 crosses a multiple of
# 2^15 once in 32 768 sums.  Its test is that the wraps happen and move many final bytes.
EXPOSED_WORKLOADS = [
    dict(name="tern_rng", weights=("ternary", 1), shifts=(1, 3, 3), images=[(("rng", 5), 32)], more=("rng", 105)),
    dict(name="tern_smooth", weights=("ternary", 2), shifts=(1, 3, 4), images=[(("smooth", 6), 32)], more=("smooth", 106)),
    dict(name="tern_tb", weights=("ternary", 3), shifts=(1, 3, 3), images=[("tb", 1), (("smooth", 7), 31)], more=("rng", 107)),
    dict(name="acc24_wrap", weights=("acc24", 31), shifts=(0, 14, 15), images=[(("bright", 32), 16)], more=("bright", 132),
         acc_bits=24),
]


def shift_triple_draws(trials=8):
    """Seeded random shift triples, each with its own ternary weights and image kind (smooth for every third trial, else
    uniform): shifts drawn from the ranges where those weights' sums reach 2^shift at every layer, so that each draw keeps
    its bytes informative (tests/test_exposure_cpu.py holds every draw to the EXPOSED_WORKLOADS criteria).
    -> [(name, weights kind, shifts, images kind)]."""
    rng = np.random.default_rng(77)
    out = []
    for t in range(trials):
        sh = (int(rng.integers(1, 3)), int(rng.integers(3, 5)), int(rng.integers(3, 5)))
        out.append((f"triple{t}", ("ternary", 500 + t), sh, ("smooth", 600 + t) if t % 3 == 0 else ("rng", 600 + t)))
    return out


def all_zero_triples(trials=4):
    """Seeded shift triples of 24..31 at every layer with full-range weights: no sum reaches 2^24 (32*9*255*128 = 9.4 M), so
    every byte of every layer is 0.  -> [(weights kind, shifts, images kind)]."""
    rng = np.random.default_rng(78)
    return [(("rng", 520 + t) if t % 2 else ("const", 0x7F), tuple(int(v) for v in rng.integers(24, 32, 3)),
             ("rng", 620 + t) if t % 2 else ("const", 255)) for t in range(trials)]


def workload_images(w, n=None, H=128, W=128):
    """The images of an EXPOSED_WORKLOADS entry: its own pieces for n = None; the first n of them, followed by further images
    of kind w["more"] (drawn 512 at a time) when n is larger; at any other size n images of kind w["more"]."""
    if (H, W) != (128, 128):
        return make_images(w["more"], n, H, W)
    own = np.concatenate([make_images(kind, k) for kind, k in w["images"]])
    if n is None or n <= len(own):
        return own[:n]
    tag, seed = w["more"]
    extra = [make_images((tag, seed * 1000 + b), min(512, n - len(own) - 512 * b)) for b in range(-(-(n - len(own)) // 512))]
    return np.concatenate([own] + extra)


def make_features(kind, n):
    """Synthetic (n,64,256) u8 feature maps for the classifier / CAM tail.
    kind: ('rng', seed) full range | ('low', seed) small values | ('saturated', seed) some channels all 255 |
          ('blob', seed) a few bright blobs on a dark map | ('sparse', seed) mostly zero | 'zeros' | 'full'."""
    if kind == "zeros":
        return np.zeros((n, 64, 256), dtype=np.uint8)
    if kind == "full":
        return np.full((n, 64, 256), 255, dtype=np.uint8)
    tag, seed = kind
    rng = np.random.default_rng(seed)
    f = rng.integers(0, 256, (n, 64, 256), dtype=np.uint8)
    if tag == "rng":
        return f
    if tag == "low":
        return (f >> 4).astype(np.uint8)
    if tag == "saturated":
        for i in range(n):
            f[i, rng.choice(64, size=int(rng.integers(1, 40)), replace=False)] = 255
        return f
    if tag == "sparse":
        f[rng.random(f.shape) < 0.95] = 0
        return f
    if tag == "blob":
        out = np.zeros((n, 64, 16, 16), dtype=np.int64)
        yy, xx = np.mgrid[0:16, 0:16]
        for i in range(n):
            for _ in range(int(rng.integers(1, 4))):
                cy, cx, r = rng.integers(0, 16), rng.integers(0, 16), rng.integers(1, 6)
                amp = rng.integers(40, 256, 64)
                out[i] += amp[:, None, None] * ((yy - cy) ** 2 + (xx - cx) ** 2 <= r * r)
        return np.clip(out + (f.reshape(n, 64, 16, 16) >> 5), 0, 255).astype(np.uint8).reshape(n, 64, 256)
    raise ValueError(kind)


# Classifier.get_cam_bbox cases pinned by tests/golden/cam_cases.npz (tests/golden/make_cam_golden.py)
CAM_CASES = [
    dict(name="cam_rng", features=("rng", 40), n=6),
    dict(name="cam_low", features=("low", 41), n=4),
    dict(name="cam_saturated", features=("saturated", 42), n=6),
    dict(name="cam_blob", features=("blob", 43), n=8),
    dict(name="cam_sparse", features=("sparse", 44), n=4),
    dict(name="cam_zeros", features="zeros", n=1),
    dict(name="cam_full", features="full", n=1),
]


def make_frames(kind, n, h, w):
    """Synthetic (n,h,w,3) u8 BGR camera frames.  kind: ('rng', seed) | ('smooth', seed) | ('edges', seed)."""
    tag, seed = kind
    rng = np.random.default_rng(seed)
    if tag == "rng":
        return rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    if tag == "smooth":
        hh, ww = -(-h // 16) * 16, -(-w // 16) * 16
        return np.stack([smooth_images(seed * 3 + c, n, hh, ww)[:, :h, :w] for c in range(3)], axis=-1)
    if tag == "edges":                              # saturated blocks: exercises rounding ties and 0 / 255 extremes
        blocks = rng.integers(0, 2, (n, -(-h // 7), -(-w // 5), 3), dtype=np.uint8) * 255
        return np.repeat(np.repeat(blocks, 7, axis=1), 5, axis=2)[:, :h, :w].copy()
    raise ValueError(kind)


# pre-processing cases pinned by tests/golden/prep_cases.npz (tests/golden/make_prep_golden.py; cv2 4.13.0)
PREP_CASES = [
    dict(name="vga_rng", frames=("rng", 50), n=2, h=480, w=640),            # the reference's camera size (realtime_detect.py:151)
    dict(name="vga_smooth", frames=("smooth", 51), n=2, h=480, w=640),
    dict(name="vga_edges", frames=("edges", 52), n=2, h=480, w=640),
    dict(name="portrait_720", frames=("rng", 53), n=1, h=1280, w=720),      # h > w branch, fractional scale 5.625
    dict(name="square_300", frames=("smooth", 54), n=1, h=300, w=300),      # no crop, scale 2.34
    dict(name="x2_256", frames=("edges", 55), n=2, h=256, w=320),           # integer scale 2: (sum + 2) >> 2
    dict(name="x3_384", frames=("edges", 56), n=2, h=384, w=384),           # integer scale 3: rint(sum * (1/9))
    dict(name="x6_768", frames=("rng", 57), n=1, h=768, w=1024),            # integer scale 6
    dict(name="x1_128", frames=("rng", 58), n=1, h=128, w=160),             # scale 1: gray only
    dict(name="odd_131", frames=("rng", 59), n=1, h=131, w=200),            # scale just above 1
]


# load_image_any cases pinned by tests/golden/pil_cases.npz (tests/golden/make_pil_golden.py runs the reference's own function on
# PNG files written from these arrays).  kind: 'L' | 'RGB' | 'RGBA'.
PIL_CASES = [
    dict(name="pil_rgb_vga", mode="RGB", images=("smooth", 80), h=480, w=640),
    dict(name="pil_rgb_rng_small", mode="RGB", images=("rng", 81), h=100, w=37),          # both dimensions enlarged
    dict(name="pil_l_256", mode="L", images=("rng", 82), h=256, w=256),                   # scale 2
    dict(name="pil_l_same", mode="L", images=("rng", 83), h=128, w=128),                  # size already right: a copy
    dict(name="pil_rgb_same", mode="RGB", images=("rng", 84), h=128, w=128),              # gray conversion only
    dict(name="pil_l_w128", mode="L", images=("smooth", 85), h=333, w=128),               # vertical pass only
    dict(name="pil_rgb_h128", mode="RGB", images=("rng", 86), h=128, w=300),              # horizontal pass only
    dict(name="pil_rgba_big", mode="RGBA", images=("smooth", 87), h=1000, w=1500),        # 127-tap windows
    dict(name="pil_l_strip", mode="L", images=("rng", 88), h=17, w=2000),                 # enlarge one way, shrink the other
    dict(name="pil_rgb_odd", mode="RGB", images=("edges", 89), h=129, w=127),             # ratios just off 1, saturated blocks
]


def make_pil_image(case):
    """Seeded decoded image of a PIL case: (h,w) for 'L', (h,w,3) 'RGB', (h,w,4) 'RGBA'."""
    ch = {"L": 1, "RGB": 3, "RGBA": 4}[case["mode"]]
    tag, seed = case["images"]
    h, w = case["h"], case["w"]
    if tag == "edges":
        planes = [make_frames(("edges", seed), 1, h, w)[0][..., c % 3] for c in range(ch)]
    elif tag == "smooth":
        hh, ww = -(-h // 16) * 16, -(-w // 16) * 16
        planes = [smooth_images(seed * 5 + c, 1, hh, ww)[0, :h, :w] for c in range(ch)]
    elif tag == "stripes":                          # saturated 0 / 255 diagonal stripes: the largest swings of the filter sums
        rng = np.random.default_rng(seed)
        yy, xx = np.ogrid[:h, :w]
        planes = [((((xx + yy * int(rng.integers(1, 4))) // int(rng.integers(1, 4))) % 2) * 255).astype(np.uint8)
                  for _ in range(ch)]
    elif tag == "const":                            # ('const', value): every pixel of every channel; 255 gives the largest sums
        planes = [np.full((h, w), seed, dtype=np.uint8) for _ in range(ch)]
    else:
        planes = [np.random.default_rng(seed * 5 + c).integers(0, 256, (h, w), dtype=np.uint8) for c in range(ch)]
    return planes[0] if ch == 1 else np.ascontiguousarray(np.stack(planes, axis=-1))


def _resample_pil_cases():
    """load_image_any at the edges of its domain, pinned by tests/golden/resample_edges.npz (make_resample_edges_golden.py runs
    Pillow itself).  Image.resize runs the vertical pass first when H > 100 W, so both sides of that switch are here for several
    widths (H is capped at the 32768 the loader accepts, so W = 328 has only 32768x328, which runs horizontal first), in every
    mode, plus the extreme shapes and both orientations of a strip."""
    cases, seed = [], 1000
    def add(h, w, mode, tag):
        nonlocal seed
        content = ("const", 255) if tag == "full" else (tag, seed)
        cases.append(dict(name=f"pil_{h}x{w}_{mode}_{tag}", mode=mode, images=content, h=h, w=w))
        seed += 1
    for w in (2, 3, 7, 64, 129, 327, 328):
        for h in sorted({min(100 * w, 32768), min(100 * w + 1, 32768)}):
            for mode, tag in (("L", "rng"), ("L", "stripes"), ("L", "full"), ("RGB", "rng"), ("RGBA", "stripes")):
                add(h, w, mode, tag)
    for h, w in ((1, 1), (1, 2), (2, 1), (1, 32768), (32768, 1), (3, 32768), (32768, 5), (32768, 128), (128, 32768)):
        add(h, w, "L", "rng")
    for h, w, mode, tag in ((3, 32768, "RGB", "rng"), (32768, 5, "RGB", "rng"), (32768, 5, "L", "full"),
                            (17, 2000, "L", "rng"), (2000, 17, "L", "rng"), (17, 2000, "RGB", "stripes"), (2000, 17, "RGB", "stripes")):
        add(h, w, mode, tag)
    return cases


RESAMPLE_PIL_CASES = _resample_pil_cases()

# centre-crop pre-processing at the large crop sides, pinned by tests/golden/resample_edges.npz (cv2 4.13.0): integer scales
# k = 9, 16, 32, 63, 64 (k != 2^j: the rounded 1/(k*k)), fractional sides up to 65 taps, 4K frames (one per 16 MiB staging
# chunk) and 8192x8192 frames (201 MB, above the 64 MiB latency path)
RESAMPLE_AREA_CASES = [
    dict(name="area_k9_1152", frames=("rng", 1200), n=2, h=1152, w=1300),
    dict(name="area_k16_2048", frames=("edges", 1201), n=1, h=2100, w=2048),
    dict(name="area_k32_4096", frames=("rng", 1202), n=1, h=4096, w=4096),
    dict(name="area_k63_8064", frames=("edges", 1203), n=1, h=8064, w=8100),
    dict(name="area_k64_8192", frames=("rng", 1204), n=1, h=8192, w=8192),
    dict(name="area_k64_8192_edges", frames=("edges", 1205), n=1, h=8192, w=8192),
    dict(name="area_1081", frames=("rng", 1206), n=2, h=1081, w=1500),
    dict(name="area_2047", frames=("edges", 1207), n=2, h=2047, w=2047),
    dict(name="area_2049", frames=("rng", 1208), n=1, h=2200, w=2049),
    dict(name="area_4095", frames=("edges", 1209), n=1, h=4095, w=4200),
    dict(name="area_4097", frames=("rng", 1210), n=1, h=4097, w=4097),
    dict(name="area_8191", frames=("edges", 1211), n=1, h=8191, w=8191),
    dict(name="area_4k", frames=("rng", 1212), n=3, h=2160, w=3840),
    dict(name="area_4k_edges", frames=("edges", 1213), n=2, h=2160, w=3840),
]


def make_area_frames(name):
    """The seeded frames of the RESAMPLE_AREA_CASES case `name`."""
    c = next(c for c in RESAMPLE_AREA_CASES if c["name"] == name)
    return make_frames(c["frames"], c["n"], c["h"], c["w"])


AREA_LARGE_SIDES = (1081, 1152, 2047, 2048, 2049, 4095, 4096, 4097, 8064, 8191, 8192)


def corner_regions(frame, fh, fw, sides=AREA_LARGE_SIDES):
    """(frame, x, y, side) for every side at the four corners of the frame."""
    return np.array([(frame, x, y, s) for s in sides for x, y in ((0, 0), (fw - s, 0), (0, fh - s), (fw - s, fh - s))], np.int32)


# regions of the 8192x8192 frames of area_k64_8192 and area_k64_8192_edges (201 MB each: one frame per staging chunk): every
# large side at the four corners of the first, three odd sides on the second
REGIONS_8192 = np.concatenate([corner_regions(0, 8192, 8192),
                               np.array([(1, 1, 8192 - 8191, 8191), (1, 8192 - 4097, 3, 4097), (1, 2049, 4000, 2049)], np.int32)])


# several regions of the frames of area_4k (frame 1 unreferenced), through host staging of one 4K frame per chunk
REGIONS_4K = np.array([(0, 0, 0, 2160), (0, 3840 - 2049, 111, 2049), (0, 1000, 2160 - 1081, 1081), (0, 3840 - 128, 2160 - 128, 128),
                       (0, 1680, 1, 2047), (2, 17, 3, 2047), (2, 3840 - 1152, 0, 1152), (2, 1500, 50, 2048), (2, 0, 2160 - 129, 129),
                       (2, 1792, 1008, 1152)], np.int32)


def make_training_set(seed=90, n=300, n_cls=6, noise=0.35):
    """Seeded (n,1024) f32 pooled-feature vectors in 0..1 with class structure + labels, for the classifier trainer
    (retrain_classifier.train_linear_classifier); noisy enough that validation accuracy moves during training."""
    rng = np.random.default_rng(seed)
    templates = (rng.random((n_cls, 1024)) < 0.08).astype(np.float32) * rng.uniform(0.3, 0.9, (n_cls, 1024)).astype(np.float32)
    labels = rng.integers(0, n_cls, n).astype(np.int64)
    x = templates[labels] * rng.uniform(0.2, 1.0, (n, 1)).astype(np.float32) + noise * rng.random((n, 1024)).astype(np.float32)
    return np.clip(x, 0.0, 1.0).astype(np.float32), labels
