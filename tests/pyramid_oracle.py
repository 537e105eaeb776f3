"""numpy restatement of the pyramid calls (include/cnnacc.h, cnnacc_preprocess_pyramid / cnnacc_scan_pyramid): OpenCV's
BGR2GRAY + INTER_AREA to a level of any size (w, h), the window rectangles and their checks, and the scan of every level.
TEST INFRASTRUCTURE.  resize_area generalises rect_oracle.resize_area_rect_u8 from 128x128 to (w, h); it is pinned against
cv2 4.13.0 by tests/golden/pyramid_cases.npz (tests/golden/make_pyramid_golden.py)."""
import numpy as np

import scan_oracle
from oracle import np_oracle


def fast_axis(S, D):
    """OpenCV's integer-path test on one axis: 1 / (D / S) in double within DBL_EPSILON of an integer.  False for S = 49 D,
    where 1.0 / (1.0 / 49) != 49."""
    scale = 1.0 / (D / S)
    return abs(scale - np.rint(scale)) < np.finfo(np.float64).eps


def resize_area(src, w, h):
    """cv2.resize(src, (w, h), interpolation=INTER_AREA) for an (H, W) u8 image with H >= h and W >= w.  OpenCV picks the path
    from both scales: a copy at the same size, integer box sums when both axes pass fast_axis (2x2: (sum + 2) >> 2, else
    rint(float(sum) * (1.f / (kx ky)))), else ResizeArea with x taps computeResizeAreaTab(W -> w) and y taps (H -> h), where
    an integer axis takes the table too.  The tables use scale = S / D (np_oracle.area_tab)."""
    src = np.asarray(src, dtype=np.uint8)
    H, W = src.shape
    assert H >= h and W >= w
    if (H, W) == (h, w):
        return src.copy()
    if fast_axis(H, h) and fast_axis(W, w):          # ResizeAreaFast: exact integer box sums
        ky, kx = H // h, W // w
        tot = src.astype(np.int64).reshape(h, ky, w, kx).sum(axis=(1, 3))
        if kx == 2 and ky == 2:
            return ((tot + 2) >> 2).astype(np.uint8)
        sc = np.float32(1.0) / np.float32(kx * ky)
        return np.clip(np.rint(tot.astype(np.float32) * sc), 0, 255).astype(np.uint8)
    xtab, ytab = np_oracle.area_tab(W, w), np_oracle.area_tab(H, h)      # ResizeArea: float accumulation, horizontal first
    Sf = src.astype(np.float32)
    buf = np.zeros((H, w), dtype=np.float32)
    for dx, sx, a in xtab:
        buf[:, dx] = buf[:, dx] + Sf[:, sx] * a
    out = np.zeros((h, w), dtype=np.float32)
    first = np.ones(h, dtype=bool)
    for dy, sy, b in ytab:
        out[dy] = b * buf[sy] if first[dy] else out[dy] + b * buf[sy]
        first[dy] = False
    return np.clip(np.rint(out), 0, 255).astype(np.uint8)


def gray(frame):
    """Full-resolution BGR2GRAY in row blocks, so an 8192-row frame needs no GB temporaries."""
    return np.concatenate([np_oracle.bgr_to_gray(frame[i:i + 1024]) for i in range(0, frame.shape[0], 1024)])


def level_gray(frame, w, h):
    return resize_area(gray(frame), w, h)


def preprocess(frames, levels):
    """[F][sum of h * w]: every level of every frame, frame-major, then level."""
    return np.stack([np.concatenate([resize_area(gray(f), w, h).ravel() for w, h in levels]) for f in frames])


def level_ok(fh, fw, w, h, stride=None):
    """The header's level rule; with a stride also that every window's frame rectangle is in whole pixels."""
    if not (128 <= fh <= 8192 and 128 <= fw <= 8192):
        return False
    if w % 16 or h % 16 or not (128 <= w <= fw and 128 <= h <= fh):
        return False
    if stride is None:
        return True
    if stride < 8 or stride % 8:
        return False
    return all((128 * S) % D == 0 and all((o * S) % D == 0 for o in scan_oracle.origins(D, stride))
               for S, D in ((fw, w), (fh, h)))


def windows(n_frames, fh, fw, levels, stride):
    """(R, 5) int32 frame rectangles (frame, x fw / w, y fh / h, 128 fw / w, 128 fh / h), frame-major, then level, then y,
    then x; None where the call is refused."""
    if not 1 <= len(levels) <= 16 or not all(level_ok(fh, fw, w, h, stride) for w, h in levels):
        return None
    one = [(x * fw // w, y * fh // h, 128 * fw // w, 128 * fh // h)
           for w, h in levels for y in scan_oracle.origins(h, stride) for x in scan_oracle.origins(w, stride)]
    return np.array([(f,) + r for f in range(n_frames) for r in one], np.int32).reshape(-1, 5)


def level_windows(n_frames, w, h, stride):
    """The (frame, x, y, 128) windows of one level in level pixels, frame-major."""
    return scan_oracle.windows(n_frames, h, w, stride)


def scan(frames, levels, weights, shifts, fc_w, fc_b, stride, acc_bits=32):
    """-> (cls, probs, logits, bbox) over all windows in window order: scan_oracle's tail on each level's window maps."""
    kern = np_oracle.unpack_weights(weights)
    parts = []
    for f in frames:
        for w, h in levels:
            m = np_oracle.infer(level_gray(f, w, h), kern, shifts, H=h, W=w, acc_bits=acc_bits).reshape(1, 64, h // 8, w // 8)
            parts.append(scan_oracle.window_maps(m, level_windows(1, w, h, stride)))
    return scan_oracle.tail(np.concatenate(parts), fc_w, fc_b)
