"""Seeded rectangles (h, w, 3) u8 BGR for the rectangle region calls, pinned against cv2 4.13.0 by tests/golden/rect_cases.npz
(tests/golden/make_rect_golden.py).  They cover every row of OpenCV's INTER_AREA choice for an (h, w) source (csrc/regions.cuh):
copy, the 2x2 integer path, other integer pairs (kx, ky) = (w/128, h/128), one axis integer and the other fractional in both
orientations, both fractional, and the extremes of 128..8192 a side."""
import numpy as np


def _case(name, h, w, content, seed):
    return dict(name=name, h=h, w=w, content=content, seed=seed)


RECT_CASES = [
    _case("copy_128x128", 128, 128, "rng", 1),
    _case("k2x2_256x256", 256, 256, "stripes", 2),
    _case("k2x2_256x256_small", 256, 256, "small", 3),
    # integer pairs kx x ky, as (h, w) = (128 ky, 128 kx): rint(float(sum) * (1.f / (kx ky)))
    _case("k1x2_256x128", 256, 128, "small", 4),
    _case("k1x2_256x128_rng", 256, 128, "rng", 5),
    _case("k2x1_128x256", 128, 256, "small", 6),
    _case("k1x4_512x128", 512, 128, "stripes", 7),
    _case("k4x1_128x512", 128, 512, "small", 8),
    _case("k3x5_640x384", 640, 384, "small", 9),
    _case("k3x5_640x384_rng", 640, 384, "rng", 10),
    _case("k5x3_384x640", 384, 640, "stripes", 11),
    _case("k64x1_128x8192", 128, 8192, "small", 12),
    # one axis integer, the other fractional (the integer axis takes the table), both orientations
    _case("mix_200x384", 200, 384, "rng", 13),
    _case("mix_384x200", 384, 200, "small", 14),
    _case("mix_128x129", 128, 129, "stripes", 15),
    _case("mix_129x128", 129, 128, "rng", 16),
    _case("mix_129x8192", 129, 8192, "rng", 17),
    _case("mix_8192x129", 8192, 129, "small", 18),
    # both axes fractional
    _case("frac_200x300", 200, 300, "small", 19),
    _case("frac_333x1000", 333, 1000, "stripes", 20),
    _case("frac_1079x1919", 1079, 1919, "rng", 21),
    # extremes
    _case("k1x64_8192x128", 8192, 128, "stripes", 22),
    _case("frac_8191x8191", 8191, 8191, "rng", 23),
]


def make_rect(case):
    """The case's (h, w, 3) u8 BGR content: 'rng' uniform bytes, 'stripes' saturated 0 / 255 blocks of 3x2 pixels,
    'small' values 0..3 (gray 0..3: many products land exactly on .5, where rint's ties-to-even rule decides)."""
    h, w, kind = case["h"], case["w"], case["content"]
    rng = np.random.default_rng(case["seed"])
    if kind == "rng":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "stripes":
        blocks = rng.integers(0, 2, (-(-h // 3), -(-w // 2), 1), dtype=np.uint8) * 255
        return np.repeat(np.repeat(np.repeat(blocks, 3, axis=0), 2, axis=1), 3, axis=2)[:h, :w].copy()
    if kind == "small":
        return np.repeat(rng.integers(0, 4, (h, w, 1), dtype=np.uint8), 3, axis=2)
    raise ValueError(kind)


def pack_rects(cases, fh, fw):
    """Places the cases at odd offsets in frames of fh x fw, shelf by shelf, tallest first, two pixels apart.
    -> (n_frames, regions (R, 5) int32 (frame, x, y, w, h) in the order of `cases`)."""
    odd = lambda v: v | 1
    order = sorted(range(len(cases)), key=lambda i: -cases[i]["h"])
    regions = np.zeros((len(cases), 5), np.int32)
    frame, x, y, shelf = 0, 1, 1, 0
    for i in order:
        h, w = cases[i]["h"], cases[i]["w"]
        assert h + 2 <= fh and w + 2 <= fw
        if x + w > fw:                                          # next shelf
            x, y, shelf = 1, odd(y + shelf + 2), 0
        if y + h > fh:                                          # next frame
            frame, x, y, shelf = frame + 1, 1, 1, 0
        regions[i] = (frame, x, y, w, h)
        x, shelf = odd(x + w + 2), max(shelf, h)
    return frame + 1, regions
