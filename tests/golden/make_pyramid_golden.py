#!/usr/bin/env python3
"""Generate tests/golden/pyramid_cases.npz by running OpenCV directly.  Build container only.

    python tests/golden/make_pyramid_golden.py

A pyramid level (w, h) of a frame is
    cv2.resize(cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY), (w, h), interpolation=cv2.INTER_AREA)
and OpenCV picks its INTER_AREA arithmetic from both scales fw/w and fh/h.  These lines run single-threaded on the seeded
frames of PYRAMID_CASES (content from tests/rect_inputs.py make_rect).  The inputs are regenerated from their seeds at test
time; an output of at most 64 KiB is stored as it is, a larger one as its SHA-256, so the archive stays small.  Before
writing, asserts that the numpy restatement (tests/pyramid_oracle.py resize_area) reproduces every output.  The archive is
written with fixed member timestamps, so a rerun with the same library version reproduces it byte for byte.
"""
import hashlib
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pyramid_oracle  # noqa: E402
import rect_inputs  # noqa: E402
from make_resample_edges_golden import write_npz  # noqa: E402

OUT = os.path.join(HERE, "pyramid_cases.npz")
INLINE_MAX = 64 << 10


def _case(name, fh, fw, w, h, content, seed):
    return dict(name=name, fh=fh, fw=fw, w=w, h=h, content=content, seed=seed)


# (w, h) levels of (fh, fw) frames: every row of OpenCV's choice, one axis integer and the other fractional in both
# orientations, sizes where S / D differs from 1 / (D / S) in double (the tables must use S / D), 49x axes, and large
# frames
PYRAMID_CASES = [
    _case("copy_vga", 480, 640, 640, 480, "rng", 1),
    _case("k2x2_vga", 480, 640, 320, 240, "stripes", 2),
    _case("k2x2_vga_small", 480, 640, 320, 240, "small", 3),
    _case("k4x2_vga", 480, 640, 160, 240, "small", 4),
    _case("k5x5_720p", 720, 1280, 256, 144, "rng", 5),
    _case("k1x2_tall", 256, 128, 128, 128, "small", 6),
    _case("frac_vga_1.25", 480, 640, 512, 384, "rng", 7),
    _case("frac_vga_1.25_small", 480, 640, 512, 384, "small", 8),
    _case("frac_vga_2.5", 480, 640, 256, 192, "stripes", 9),
    _case("frac_720p_1.25", 720, 1280, 1024, 576, "rng", 10),
    _case("mix_x2_y1.25", 480, 640, 320, 384, "rng", 11),
    _case("mix_x1.25_y2", 480, 640, 512, 240, "small", 12),
    _case("mix_x1_yfrac", 300, 256, 256, 224, "stripes", 13),
    _case("frac_1000x750", 750, 1000, 800, 592, "rng", 14),
    _case("recip_0", 160, 0, 0, 128, "rng", 15),
    _case("recip_1", 160, 0, 0, 128, "small", 16),
    _case("recip_2", 160, 0, 0, 128, "stripes", 17),
    _case("recip_3", 160, 0, 0, 128, "rng", 18),
    _case("1080p_1536x864", 1080, 1920, 1536, 864, "rng", 19),
    _case("1080p_768x432", 1080, 1920, 768, 432, "small", 20),
    _case("4k_2560x1440", 2160, 3840, 2560, 1440, "rng", 21),
    _case("tall_8192x136", 8192, 136, 128, 6144, "rng", 22),
    _case("wide_144x8192", 144, 8192, 5120, 128, "stripes", 23),
    _case("k1x64_8192x128", 8192, 128, 128, 128, "small", 24),
    # a 49x axis: 1.0 / (1.0 / 49) != 49 in double, so OpenCV takes the table there although 49 is an integer
    _case("k49_x_256x6272", 256, 6272, 128, 128, "rng", 25),
    _case("k49_y_6272x256", 6272, 256, 128, 128, "rng", 26),
    _case("k49_x_480x6272", 480, 6272, 128, 240, "rng", 27),
    _case("k49x49_6272", 6272, 6272, 128, 128, "small", 28),
]


def _recip_pairs(count):
    """The first `count` (S, D) with D a multiple of 16 in 128..S, S < 2000, where S / D != 1 / (D / S) in double, D spread out."""
    out = []
    for D in (208, 400, 592, 1104):
        for S in range(D + 1, 2000):
            if S / D != 1.0 / (D / S) and S % D:
                out.append((S, D))
                break
    assert len(out) >= count
    return out[:count]


def cases():
    """PYRAMID_CASES with the recip_k rows filled from _recip_pairs (x axis S -> D)."""
    pairs = _recip_pairs(4)
    out = []
    for c in PYRAMID_CASES:
        c = dict(c)
        if c["name"].startswith("recip_") and c["fw"] == 0:
            S, D = pairs[int(c["name"][-1])]
            c["fw"], c["w"] = S, D
        out.append(c)
    return out


def make_frame(c):
    return rect_inputs.make_rect(dict(h=c["fh"], w=c["fw"], content=c["content"], seed=c["seed"]))


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    cv2.setNumThreads(1)
    out = {"cv2_version": np.array(cv2.__version__)}
    for c in cases():
        frame = make_frame(c)
        got = cv2.resize(cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY), (c["w"], c["h"]), interpolation=cv2.INTER_AREA)
        assert got.shape == (c["h"], c["w"]) and got.dtype == np.uint8
        assert np.array_equal(got, pyramid_oracle.level_gray(frame, c["w"], c["h"])), c["name"]
        out[c["name"]] = got if got.size <= INLINE_MAX else np.array(digest(got))
        print(f"{c['name']:22s} {c['fh']}x{c['fw']} -> {c['w']}x{c['h']} {c['content']:8s} mean {got.mean():6.1f}")
    write_npz(OUT, out)
    print("wrote pyramid_cases.npz", os.path.getsize(OUT), "bytes; cv2", cv2.__version__)


if __name__ == "__main__":
    main()
