"""The numpy restatement of the scanning calls (tests/scan_oracle.py) against np_oracle's per-image path, and the window
order and count the library and the Python wrapper use.  Workloads are inputs.EXPOSED_WORKLOADS' ternary ones, where a
one-LSB error or a window cut one cell off shows."""
import numpy as np
import pytest

import fpga_cnn_b200 as fc
import inputs
import scan_oracle
from oracle import np_oracle

TERNARY = [w for w in inputs.EXPOSED_WORKLOADS if w["name"].startswith("tern")]


def _frames(w, n, fh, fw, seed):
    tag = w["more"][0]
    return inputs.make_frames((tag if tag in ("rng", "smooth") else "rng", seed), n, fh, fw)


@pytest.mark.parametrize("w", TERNARY, ids=lambda w: w["name"])
def test_128_frames_are_the_per_image_path(w):
    """On a 128x128 frame the one window is the frame: preprocess -> infer -> tail."""
    frames = _frames(w, 3, 128, 128, 31)
    wt = inputs.make_weights(w["weights"])
    fw_, fb = inputs.make_fc()
    wins, wmaps, cls, probs, logits, box = scan_oracle.scan(frames, wt, w["shifts"], fw_, fb, 64)
    assert wins.tolist() == [[f, 0, 0, 128] for f in range(3)]
    kern = np_oracle.unpack_weights(wt)
    for f in range(3):
        feat = np_oracle.infer(np_oracle.preprocess_bgr(frames[f]), kern, w["shifts"])
        assert np.array_equal(wmaps[f].reshape(64, 256), feat)
        c, p, lg, _ = np_oracle.classify_vec(feat, fw_, fb)
        assert cls[f] == c and np.array_equal(probs[f], p) and np.array_equal(logits[f], lg)
        assert tuple(box[f]) == np_oracle.bbox_vec(feat, c, fw_)[0]


@pytest.mark.parametrize("w", TERNARY, ids=lambda w: w["name"])
def test_window_interior_is_the_crop(w):
    """A window's inner 14x14 cells are the conv stack of its 128x128 gray crop; its outer ring is exactly on the sides where
    the window's edge is the frame's edge, and differs elsewhere (the crop is zero-padded there, the frame is not).  Windows
    at odd and even cell offsets and flush with both far edges."""
    fh, fw = 144, 272
    frames = _frames(w, 1, fh, fw, 32)
    wt = inputs.make_weights(w["weights"])
    kern = np_oracle.unpack_weights(wt)
    maps = scan_oracle.frame_maps(frames, wt, w["shifts"])
    gray = np_oracle.bgr_to_gray(frames[0])
    seen = set()
    for y in (0, 8, 16):
        for x in (0, 8, 16, 72, 144):
            win = scan_oracle.window_maps(maps, [(0, x, y, 128)])[0]
            crop = np_oracle.infer(gray[y:y + 128, x:x + 128], kern, w["shifts"]).reshape(64, 16, 16)
            top, bottom, left, right = y == 0, y + 128 == fh, x == 0, x + 128 == fw
            rows = [0] * top + list(range(1, 15)) + [15] * bottom
            cols = [0] * left + list(range(1, 15)) + [15] * right
            exact = np.ix_(range(64), rows, cols)
            assert np.array_equal(win[exact], crop[exact]), (x, y)
            # a side inside the frame: its 14 cells between the corners differ somewhere
            for name, sl, edge in (("top", np.s_[:, 0, 1:15], top), ("bottom", np.s_[:, 15, 1:15], bottom),
                                   ("left", np.s_[:, 1:15, 0], left), ("right", np.s_[:, 1:15, 15], right)):
                assert edge or not np.array_equal(win[sl], crop[sl]), (x, y, name)
            seen.add(((x // 8) % 2, y == 0, y + 128 == fh, x + 128 == fw))
    assert {s[0] for s in seen} == {0, 1} and any(s[2] for s in seen) and any(s[3] for s in seen)


@pytest.mark.parametrize("fh,fw", [(128, 128), (144, 272), (480, 640), (720, 1280), (8192, 128), (2160, 3840)])
@pytest.mark.parametrize("stride", [8, 16, 24, 64, 120, 128])
def test_window_order_and_count(fh, fw, stride):
    wins = scan_oracle.windows(2, fh, fw, stride) if fh * fw <= 1280 * 720 else None
    per = scan_oracle.count(fh, stride) * scan_oracle.count(fw, stride)
    assert per == len(scan_oracle.origins(fh, stride)) * len(scan_oracle.origins(fw, stride))
    assert fc.CNNAccelerator._scan_windows(fh, fw, stride) == per
    if wins is not None:
        assert np.array_equal(wins, fc.grid_regions(2, fh, fw, 128, stride))
        assert len(wins) == 2 * per


def test_window_count_examples():
    assert scan_oracle.count(640, 64) * scan_oracle.count(480, 64) == 63        # the VGA tile grid
    assert scan_oracle.count(640, 8) * scan_oracle.count(480, 8) == 2925
    assert scan_oracle.count(3840, 8) * scan_oracle.count(2160, 8) == 118575    # beyond the merge's 16384 per frame
    assert scan_oracle.origins(480, 120) == [0, 120, 240, 352]                   # flush window added
    assert scan_oracle.origins(384, 128) == [0, 128, 256]                        # flush window already there
