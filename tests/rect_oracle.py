"""numpy restatement of OpenCV's BGR2GRAY + INTER_AREA on an (h, w) rectangle, the pre-processing of the rectangle region
calls (CNNACC_FLAG_RECTS, csrc/regions.cuh).  Test infrastructure only.  It builds on oracle/np_oracle.py (area_tab =
computeResizeAreaTab, bgr_to_gray) and, for squares, equals np_oracle.resize_area_u8 (tests/test_rect_regions_cpu.py)."""
import numpy as np

from oracle import np_oracle


def resize_area_rect_u8(src, d=128):
    """cv2.resize(src, (d,d), interpolation=INTER_AREA) for an (h, w) u8 image with h, w >= d.  OpenCV picks the path from
    both scales: integer box sums when h and w are both multiples of d, else ResizeArea with separate x and y tables, where
    an integer axis takes the table too (k taps of float(1/k), accumulated per tap).  Pinned against cv2 4.13.0 by
    tests/golden/rect_cases.npz (tests/golden/make_rect_golden.py)."""
    src = np.asarray(src, dtype=np.uint8)
    H, W = src.shape
    assert H >= d and W >= d
    if H == d and W == d:
        return src.copy()
    if H % d == 0 and W % d == 0:                    # ResizeAreaFast: exact integer box sums
        ky, kx = H // d, W // d
        tot = src.astype(np.int64).reshape(d, ky, d, kx).sum(axis=(1, 3))
        if kx == 2 and ky == 2:
            return ((tot + 2) >> 2).astype(np.uint8)
        sc = np.float32(1.0) / np.float32(kx * ky)
        return np.clip(np.rint(tot.astype(np.float32) * sc), 0, 255).astype(np.uint8)
    xtab, ytab = np_oracle.area_tab(W, d), np_oracle.area_tab(H, d)      # ResizeArea: float accumulation, horizontal first
    Sf = src.astype(np.float32)
    buf = np.zeros((H, d), dtype=np.float32)
    for dx, sx, a in xtab:
        buf[:, dx] = buf[:, dx] + Sf[:, sx] * a
    out = np.zeros((d, d), dtype=np.float32)
    first = np.ones(d, dtype=bool)
    for dy, sy, b in ytab:
        out[dy] = b * buf[sy] if first[dy] else out[dy] + b * buf[sy]
        first[dy] = False
    return np.clip(np.rint(out), 0, 255).astype(np.uint8)


def preprocess_rect(rect, d=128):
    """An (h,w,3) u8 BGR rectangle -> (128,128) u8: cv2.cvtColor(BGR2GRAY) then INTER_AREA (resize_area_rect_u8).  The gray
    conversion runs in row blocks, so an 8192-row rectangle needs no GB temporaries."""
    gray = np.concatenate([np_oracle.bgr_to_gray(rect[i:i + 1024]) for i in range(0, rect.shape[0], 1024)])
    return resize_area_rect_u8(gray, d)
