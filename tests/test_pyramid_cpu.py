"""CPU-side checks of the pyramid calls: the numpy restatement of a level's gray (tests/pyramid_oracle.py) against cv2 4.13.0
(tests/golden/pyramid_cases.npz), the window rectangles and every refusal through cnnacc_pyramid_windows_host against the
restatement, the level table of the issue through pyramid_levels, the identity level against scan_oracle, and the merge of
pyramid windows through cnnacc_merge_regions_host against the rectangle merge restatement."""
import ctypes
import os
import sys

import numpy as np
import pytest

import fpga_cnn_b200 as fc
import inputs
import pyramid_oracle
import scan_oracle
import test_rect_regions_cpu as rect

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_pyramid_golden as golden  # noqa: E402

GOLDEN = os.path.join(HERE, "golden", "pyramid_cases.npz")
TERNARY = [w for w in inputs.EXPOSED_WORKLOADS if w["name"].startswith("tern")]


@pytest.fixture(scope="module")
def lib():
    fc.build()
    return fc.load()


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


# ---- a level's gray ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", golden.cases(), ids=lambda c: c["name"])
def test_restatement_equals_opencv_golden(case):
    gold = np.load(GOLDEN)
    assert str(gold["cv2_version"]) == "4.13.0"
    got = pyramid_oracle.level_gray(golden.make_frame(case), case["w"], case["h"])
    want = gold[case["name"]]
    if want.dtype.kind == "U":
        assert golden.digest(got) == str(want)
    else:
        assert np.array_equal(got, want)


def test_golden_covers_every_path():
    kinds = set()
    for c in golden.cases():
        fw, fh, w, h = c["fw"], c["fh"], c["w"], c["h"]
        ix, iy = fw % w == 0, fh % h == 0
        kinds.add("copy" if (fw, fh) == (w, h) else "2x2" if (fw, fh) == (2 * w, 2 * h) else "int" if ix and iy
                  else "x_int" if ix else "y_int" if iy else "frac")
        if c["name"].startswith("recip_"):
            assert fw / w != 1.0 / (w / fw)
    assert kinds == {"copy", "2x2", "int", "x_int", "y_int", "frac"}
    assert max(max(c["fh"], c["fw"]) for c in golden.cases()) == 8192
    assert any(c["fw"] == 49 * c["w"] for c in golden.cases()) and any(c["fh"] == 49 * c["h"] for c in golden.cases())


def test_fast_axis_is_opencvs_test():
    # integer downscales 1..64 all take the integer path except 49, where 1.0 / (1.0 / 49) != 49 in double
    assert [k for k in range(1, 65) if not pyramid_oracle.fast_axis(128 * k, 128)] == [49]
    assert not pyramid_oracle.fast_axis(6272, 128) and not pyramid_oracle.fast_axis(640, 512)


def test_restatement_at_128_is_the_rectangle_one():
    rng = np.random.default_rng(5)
    for h, w in ((200, 384), (256, 256), (129, 300), (512, 128)):
        src = rng.integers(0, 256, (h, w), dtype=np.uint8)
        import rect_oracle
        assert np.array_equal(pyramid_oracle.resize_area(src, 128, 128), rect_oracle.resize_area_rect_u8(src))


# ---- windows and refusals -----------------------------------------------------------------------------------------------------

def windows_host(lib, fh, fw, levels, stride, cap=None):
    lv = np.ascontiguousarray(np.asarray(levels, np.int32).reshape(-1, 2))
    per = lib.cnnacc_pyramid_windows_host(fh, fw, _p(lv) if len(lv) else None, len(lv), stride, None, 0)
    if per < 0:
        return per, None
    out = np.full((per, 5), -9, np.int32)
    assert lib.cnnacc_pyramid_windows_host(fh, fw, _p(lv), len(lv), stride, _p(out), per if cap is None else cap) == per
    return per, out


SETS = [
    ((480, 640), [(640, 480), (512, 384), (320, 240), (256, 192)]),
    ((720, 1280), [(1280, 720), (1024, 576), (512, 288), (256, 144)]),
    ((1080, 1920), [(1536, 864), (1280, 720), (1024, 576), (768, 432), (512, 288), (256, 144)]),
    ((750, 1000), [(640, 480), (320, 240), (800, 400)]),        # scale 25/16: whole pixels from stride 16 on
    ((480, 640), [(640, 240), (320, 480), (128, 128)]),           # anisotropic
    ((144, 272), [(272, 144), (128, 128)]),
    ((8192, 128), [(128, 8192), (128, 4096), (128, 128)]),
    ((130, 260), [(256, 128)]),                                    # one window position per axis
]


@pytest.mark.parametrize("stride", [8, 16, 24, 32, 64, 120])
@pytest.mark.parametrize("size,levels", SETS, ids=[f"{s[0][0]}x{s[0][1]}_{len(s[1])}" for s in SETS])
def test_windows_host_equals_restatement(lib, size, levels, stride):
    fh, fw = size
    want = pyramid_oracle.windows(1, fh, fw, levels, stride)
    per, got = windows_host(lib, fh, fw, levels, stride)
    if want is None:
        assert per == fc._lib.ERR_ARG
        with pytest.raises(ValueError):
            fc.pyramid_windows(2, fh, fw, levels, stride)
        return
    assert per == len(want) and np.array_equal(got, want)
    two = fc.pyramid_windows(2, fh, fw, levels, stride)
    assert np.array_equal(two, pyramid_oracle.windows(2, fh, fw, levels, stride))
    # each level's windows in level pixels are scan_frames' windows of a frame of the level's size
    k = 0
    for w, h in levels:
        lw = scan_oracle.windows(1, h, w, stride)
        r = got[k:k + len(lw)]
        assert np.array_equal(r[:, 1] * w, lw[:, 1] * fw) and np.array_equal(r[:, 2] * h, lw[:, 2] * fh)
        k += len(lw)
    assert k == per


def test_issue_table_through_pyramid_levels():
    table = {(480, 640): ([(640, 480), (512, 384), (320, 240), (256, 192)], 5070, 1333),
             (720, 1280): ([(1280, 720), (1024, 576), (512, 288), (256, 144)], 18396, 4720),
             (1080, 1920): ([(1536, 864), (1280, 720), (1024, 576), (768, 432), (512, 288), (256, 144)], 38016, 9723)}
    for (fh, fw), (levels, n8, n16) in table.items():
        assert fc.pyramid_levels(fh, fw, 8) == levels and fc.pyramid_levels(fh, fw, 16) == levels
        assert len(fc.pyramid_windows(1, fh, fw, levels, 8)) == n8
        assert len(fc.pyramid_windows(1, fh, fw, levels, 16)) == n16
    assert 38016 > fc._lib.MERGE_MAX_PER_FRAME >= 9723


def test_pyramid_levels_are_admissible():
    for fh, fw in ((480, 640), (1080, 1920), (750, 1000), (2160, 3840), (128, 128), (131, 257)):
        for stride in (8, 16, 48):
            lv = fc.pyramid_levels(fh, fw, stride)
            assert lv == sorted(lv, reverse=True)
            assert all(w * fh == h * fw and pyramid_oracle.level_ok(fh, fw, w, h, stride) for w, h in lv)
            want = [(w, w * fh // fw) for w in range(fw - fw % 16, 127, -16) if (w * fh) % fw == 0
                    and pyramid_oracle.level_ok(fh, fw, w, w * fh // fw, stride)]
            assert lv == want


REFUSED = {
    "fh_127": (127, 640, [(128, 128)], 8),
    "fw_8193": (480, 8193, [(128, 128)], 8),
    "no_levels": (480, 640, [], 8),
    "17_levels": (480, 640, [(128, 128)] * 17, 8),
    "w_not_16": (480, 640, [(520, 384)], 8),
    "h_not_16": (480, 640, [(512, 388)], 8),
    "w_127": (480, 640, [(112, 240)], 8),
    "h_below_128": (480, 640, [(320, 112)], 8),
    "upscale_w": (480, 640, [(656, 480)], 8),
    "upscale_h": (480, 640, [(640, 496)], 8),
    "size_not_whole": (480, 640, [(448, 336)], 8),            # 128 * 640 / 448
    "origin_not_whole": (720, 1280, [(768, 432)], 8),         # x = 8: 8 * 5 / 3
    "stride_0": (480, 640, [(320, 240)], 0),
    "stride_7": (480, 640, [(320, 240)], 7),
    "stride_12": (480, 640, [(320, 240)], 12),
    "stride_neg": (480, 640, [(320, 240)], -8),
}


@pytest.mark.parametrize("name", sorted(REFUSED))
def test_refusals(lib, name):
    fh, fw, levels, stride = REFUSED[name]
    assert pyramid_oracle.windows(1, fh, fw, levels, stride) is None
    per, _ = windows_host(lib, fh, fw, levels, stride)
    assert per == fc._lib.ERR_ARG, name


def test_actual_origins_are_checked_not_the_stride(lib):
    """A 144x144 level of 153x153 frames (scale 17/16) has origins 0, 16 at stride 24: both whole (0, 17), though 24 * 17/16
    is not, so it is accepted; at stride 8 the origin 8 -> 8.5 refuses it.  A 128x128 level has the one origin 0 at every
    stride."""
    assert windows_host(lib, 153, 153, [(144, 144)], 24)[0] == 4
    assert windows_host(lib, 153, 153, [(144, 144)], 16)[0] == 4
    assert windows_host(lib, 153, 153, [(144, 144)], 8)[0] == fc._lib.ERR_ARG
    assert np.array_equal(windows_host(lib, 153, 153, [(144, 144)], 24)[1][:, 1:3], [[0, 0], [17, 0], [0, 17], [17, 17]])
    for stride in (8, 24, 40, 1024):
        per, r = windows_host(lib, 136, 136, [(128, 128)], stride)
        assert per == 1 and r.tolist() == [[0, 0, 0, 136, 136]]
        assert pyramid_oracle.windows(1, 136, 136, [(128, 128)], stride) is not None


def test_small_cap_and_null_levels(lib):
    lv = np.array([[320, 240]], np.int32)
    out = np.zeros((100, 5), np.int32)
    per = lib.cnnacc_pyramid_windows_host(480, 640, _p(lv), 1, 64, None, 0)
    assert per > 1
    assert lib.cnnacc_pyramid_windows_host(480, 640, _p(lv), 1, 64, _p(out), per - 1) == fc._lib.ERR_ARG
    assert lib.cnnacc_pyramid_windows_host(480, 640, None, 1, 64, None, 0) == fc._lib.ERR_ARG


# ---- the identity level -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("w", TERNARY, ids=lambda w: w["name"])
def test_identity_level_is_scan_oracle(w):
    frames = inputs.make_frames(("rng", 41), 2, 144, 272)
    wt = inputs.make_weights(w["weights"])
    fw_, fb = inputs.make_fc()
    got = pyramid_oracle.scan(frames, [(272, 144)], wt, w["shifts"], fw_, fb, 16)
    want = scan_oracle.scan(frames, wt, w["shifts"], fw_, fb, 16)[2:]
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    assert np.array_equal(pyramid_oracle.preprocess(frames, [(272, 144)]).reshape(2, 144, 272),
                          np.stack([np.asarray(pyramid_oracle.gray(f)) for f in frames]))
    assert np.array_equal(pyramid_oracle.windows(2, 144, 272, [(272, 144)], 16)[:, :3],
                          scan_oracle.windows(2, 144, 272, 16)[:, :3])


# ---- the merge on pyramid windows -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(4))
def test_merge_of_pyramid_windows_equals_restatement(lib, seed):
    rng = np.random.default_rng(seed)
    (fh, fw), levels = SETS[seed % 4]
    stride = (16, 32, 16, 16)[seed]
    n = 3
    reg = pyramid_oracle.windows(n, fh, fw, levels, stride)
    assert reg is not None
    R = len(reg)
    b1 = rng.integers(-5, 120, (R, 2))
    bbox = np.concatenate([b1, b1 + rng.integers(-3, 70, (R, 2))], 1).astype(np.int32)
    scores = rng.random(R, np.float32) if seed % 2 else rng.choice(np.float32([0.0, 0.25, 0.5, 1.0]), R)
    cls = rng.integers(0, 6, R).astype(np.int32)
    for agnostic, max_det, iou_max, score_min in ((False, 100, 0.5, 0.3), (True, 1024, 0.3, 0.0), (False, 5, 0.1, 0.5)):
        rc, got = rect._merge_host(lib, reg, scores, cls, bbox, n, score_min, iou_max, max_det, agnostic, fc._lib.FLAG_RECTS)
        assert rc == 0
        rect.sq.assert_same(got, rect.restate(reg, scores, cls, bbox, n, score_min, iou_max, max_det, agnostic),
                            (seed, agnostic, max_det))
    # region_boxes_to_frame maps the boxes exactly: the merge's 1/128-pixel boxes are its values times 128
    clipped = np.clip(bbox, 0, 127)
    assert np.array_equal(fc.region_boxes_to_frame(reg, clipped) * 128, rect.frame_boxes(reg, clipped))
