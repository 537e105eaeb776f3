#!/usr/bin/env python3
"""Generate tests/golden/rect_cases.npz by running OpenCV directly.  Build container only.

    python tests/golden/make_rect_golden.py

A rectangle region (frame, x, y, w, h) pre-processes to
    cv2.resize(cv2.cvtColor(rect, cv2.COLOR_BGR2GRAY), (128, 128), interpolation=cv2.INTER_AREA)
and OpenCV picks its INTER_AREA arithmetic from both scales w/128 and h/128.  These lines run single-threaded on the seeded
rectangles of tests/rect_inputs.py RECT_CASES.  Only the 128x128 outputs and the library version are stored; the inputs are
regenerated from their seeds at test time.  Before writing, asserts that the numpy restatement (tests/rect_oracle.py
preprocess_rect) reproduces every output.  The archive is written with fixed member timestamps, so a rerun with the same
library version reproduces it byte for byte.
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import rect_inputs  # noqa: E402
import rect_oracle  # noqa: E402
from make_resample_edges_golden import write_npz  # noqa: E402

OUT = os.path.join(HERE, "rect_cases.npz")


def main():
    cv2.setNumThreads(1)
    out = {"cv2_version": np.array(cv2.__version__)}
    for case in rect_inputs.RECT_CASES:
        rect = rect_inputs.make_rect(case)
        got = cv2.resize(cv2.cvtColor(rect, cv2.COLOR_BGR2GRAY), (128, 128), interpolation=cv2.INTER_AREA)
        assert got.shape == (128, 128) and got.dtype == np.uint8
        assert np.array_equal(got, rect_oracle.preprocess_rect(rect)), case["name"]
        out[case["name"]] = got
        print(f"{case['name']:24s} {case['h']}x{case['w']} {case['content']:8s} mean {got.mean():6.1f}")
    write_npz(OUT, out)
    print("wrote rect_cases.npz", os.path.getsize(OUT), "bytes; cv2", cv2.__version__)


if __name__ == "__main__":
    main()
