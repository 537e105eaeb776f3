"""The reference helpers of tests/scan_reference.py on the CPU: row bands stitched back into whole-frame oracle maps, and
window selections that hold every flush window."""
import numpy as np
import pytest

import inputs
import oracle
import scan_oracle
import scan_reference as sr
from oracle import np_oracle

TERNARY = [w for w in inputs.EXPOSED_WORKLOADS if w["name"].startswith("tern")]


def _whole(gray, wt, shifts, bits):
    H, W = gray.shape
    if bits == 32:
        return oracle.port_infer_batch(oracle.load_port(), gray[None], wt, shifts, H, W).reshape(64, H // 8, W // 8)
    return np_oracle.infer(gray, np_oracle.unpack_weights(wt), shifts, H=H, W=W, acc_bits=24).reshape(64, H // 8, W // 8)


# (H, W, band heights): bands that do not divide H, a frame lower than the band (one band), a band of one 16-row group with
# neighbours on both sides, and the last band a single group
BAND_CASES_32 = [(400, 272, (48, 80, 112, 16)), (128, 272, (160, 128)), (272, 144, (256, 96)), (720, 160, (256, 704))]
BAND_CASES_24 = [(208, 144, (48, 80, 112)), (128, 144, (256,))]


@pytest.mark.parametrize("H,W,heights", BAND_CASES_32, ids=lambda c: str(c))
def test_stitched_bands_equal_whole_frame_32(shipped_weights, H, W, heights):
    for wt, shifts in ((shipped_weights, (7, 10, 10)), (inputs.make_weights(TERNARY[0]["weights"]), TERNARY[0]["shifts"])):
        gray = inputs.make_images(("smooth", H + W), 1, H, W)[0]
        want = _whole(gray, wt, shifts, 32)
        assert ((want > 0) & (want < 255)).mean() > 0.25
        for band in heights:
            assert np.array_equal(sr.oracle_maps(gray, wt, shifts, 32, band=band, workers=4), want), band
        assert np.array_equal(sr.oracle_maps(np.stack([gray, gray[::-1]]), wt, shifts, 32, band=heights[0], workers=4),
                              np.stack([want, _whole(np.ascontiguousarray(gray[::-1]), wt, shifts, 32)]))


@pytest.mark.parametrize("H,W,heights", BAND_CASES_24, ids=lambda c: str(c))
def test_stitched_bands_equal_whole_frame_24(H, W, heights):
    w = TERNARY[1]
    wt = inputs.make_weights(w["weights"])
    gray = inputs.make_images(("smooth", H * W), 1, H, W)[0]
    want = _whole(gray, wt, w["shifts"], 24)
    assert ((want > 0) & (want < 255)).mean() > 0.25
    for band in heights:
        assert np.array_equal(sr.oracle_maps(gray, wt, w["shifts"], 24, band=band, workers=4), want), band


def test_bands_cover_every_row_once():
    for H in (128, 144, 400, 720, 864, 8192):
        for band in (16, 48, 256):
            rows = np.zeros(H, int)
            for r0, r1, a, b in sr.bands(H, band):
                rows[r0:r1] += 1
                assert a == max(0, r0 - 16) and b == min(H, r1 + 16) and (b - a) % 16 == 0
            assert (rows == 1).all(), (H, band)


# (h, w, stride): the served level sizes, the wide and tall strips, sides where (side - 128) % stride is 0 (no flush window)
SELECT_CASES = [(720, 1280, 8), (2160, 3840, 64), (128, 8192, 8), (8192, 128, 8), (8192, 8192, 64), (864, 1536, 16),
                (1440, 2560, 64), (720, 1280, 16), (480, 640, 8), (480, 640, 16), (256, 144, 16), (640, 720, 16), (240, 1280, 16)]


@pytest.mark.parametrize("h,w,stride", SELECT_CASES, ids=lambda c: str(c))
def test_selection_holds_every_flush_window(h, w, stride):
    ny, nx = scan_oracle.count(h, stride), scan_oracle.count(w, stride)
    idx = sr.select_windows(h, w, stride)
    assert len(np.unique(idx)) == len(idx) and idx.min() >= 0 and idx.max() < ny * nx
    flush = sr.flush_windows(h, w, stride)
    assert flush <= set(idx.tolist()), sorted(flush - set(idx.tolist()))[:5]
    assert {0, nx - 1, (ny - 1) * nx, ny * nx - 1} <= set(idx.tolist())
    if ny * nx > sr.ALL_WINDOWS:
        assert len(idx) < ny * nx
        row = {i - (ny // 2) * nx for i in idx.tolist() if i // nx == ny // 2}
        assert any(all(x + k in row for k in range(16)) for x in row), "16 consecutive windows of one row"
    if (w - 128) % stride:                                # the header's rule: a last column flush with the right edge
        assert scan_oracle.origins(w, stride)[-1] == w - 128 and flush
