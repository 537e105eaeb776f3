"""The two resampling front ends at the edges of their domains, on the CPU: the numpy restatements (oracle/np_oracle.py)
reproduce every output of tests/golden/resample_edges.npz, which Pillow 12.2.0 and cv2 4.13.0 computed directly
(tests/golden/make_resample_edges_golden.py); Image.resize's pass order, checked against Pillow itself where it imports; and
the host staging plan for frames of 16 MiB and more."""
import ctypes
import os

import numpy as np
import pytest

import fpga_cnn_b200 as fc
import inputs
from oracle import np_oracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "resample_edges.npz")
CHUNK_BYTES = 16 << 20


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def oracle_preprocess(frame):
    """np_oracle.preprocess_bgr, with the gray conversion done in row blocks to keep an 8192x8192 frame's temporaries small."""
    h, w = frame.shape[:2]
    s = min(h, w)
    crop = frame[(h - s) // 2:(h - s) // 2 + s, (w - s) // 2:(w - s) // 2 + s]
    gray = np.concatenate([np_oracle.bgr_to_gray(crop[i:i + 1024]) for i in range(0, s, 1024)])
    return np_oracle.resize_area_u8(gray)


def horizontal_first(gray):
    """Pillow's arithmetic with the horizontal pass always first (the order before the tall-image rule)."""
    return np_oracle.pil_resize_bicubic_u8(np_oracle.pil_resize_bicubic_u8(gray, gray.shape[0], 128))


def test_fixture_records_the_library_versions(golden):
    assert str(golden["pillow_version"]) == "12.2.0" and str(golden["cv2_version"]) == "4.13.0"
    names = {c["name"] for c in inputs.RESAMPLE_PIL_CASES} | {c["name"] for c in inputs.RESAMPLE_AREA_CASES}
    assert len(names) == len(inputs.RESAMPLE_PIL_CASES) + len(inputs.RESAMPLE_AREA_CASES)
    assert names | {"pillow_version", "cv2_version", "regions_8192", "regions_4k"} == set(golden.files)


@pytest.mark.parametrize("case", inputs.RESAMPLE_PIL_CASES, ids=lambda c: c["name"])
def test_oracle_reproduces_loader_fixtures(case, golden):
    arr = inputs.make_pil_image(case)
    want = golden[case["name"]]
    assert want.shape == (128, 128) and want.dtype == np.uint8
    assert np.array_equal(np_oracle.load_image_array(arr), want.reshape(-1))


def test_tall_fixtures_tell_the_pass_orders_apart(golden):
    """The fixtures pin the order: on every vertical-first case of random content, horizontal-first gives other pixels."""
    tall = [c for c in inputs.RESAMPLE_PIL_CASES if np_oracle.pil_vertical_first(c["h"], c["w"])]
    assert {(c["h"], c["w"]) for c in tall} >= {(201, 2), (301, 3), (701, 7), (6401, 64), (12901, 129), (32701, 327), (32768, 5)}
    assert not any(np_oracle.pil_vertical_first(h, w) for h, w in [(200, 2), (12900, 129), (32768, 328), (128, 32768)])
    for c in tall:
        if c["w"] in (1, 128) or c["images"][0] != "rng":
            continue                                # one pass only, or flat / periodic content: the orders can agree
        gray = np_oracle.pil_to_l(inputs.make_pil_image(c))
        differ = int((horizontal_first(gray) != golden[c["name"]]).sum())
        assert differ > 0, c["name"]


@pytest.mark.parametrize("case", inputs.RESAMPLE_AREA_CASES, ids=lambda c: c["name"])
def test_oracle_reproduces_area_fixtures(case, golden):
    frames = inputs.make_area_frames(case["name"])
    want = golden[case["name"]]
    assert want.shape == (case["n"], 128, 128)
    for i, f in enumerate(frames):
        assert np.array_equal(oracle_preprocess(f), want[i]), i


@pytest.mark.parametrize("key,frames,regions", [
    ("regions_8192", ("area_k64_8192", "area_k64_8192_edges"), inputs.REGIONS_8192),
    ("regions_4k", ("area_4k",), inputs.REGIONS_4K)])
def test_oracle_reproduces_region_fixtures(key, frames, regions, golden):
    fr = np.concatenate([inputs.make_area_frames(n) for n in frames])
    want = golden[key]
    assert want.shape == (len(regions), 128, 128)
    for i, (f, x, y, s) in enumerate(regions):
        assert np.array_equal(oracle_preprocess(fr[f, y:y + s, x:x + s]), want[i]), tuple(regions[i])


def test_pass_order_against_pillow():
    """A dense sweep around H = 100 W straight against Pillow: the switch to vertical-first sits exactly at H = 100 W + 1."""
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(11)
    shapes = [(h, w) for w in range(1, 41) for h in range(100 * w - 2, 100 * w + 3)]
    shapes += [(h, w) for w in (64, 100, 128, 129, 200, 327) for h in (100 * w, 100 * w + 1)]
    shapes += [(32768, 327), (32768, 328), (3000, 2), (2, 3000), (32768, 1), (1, 32768), (101, 1), (129, 1), (12800, 128)]
    n_vertical_first = 0
    for h, w in shapes:
        a = rng.integers(0, 256, (h, w), dtype=np.uint8)
        want = np.asarray(Image.fromarray(a, "L").resize((128, 128)))
        assert np.array_equal(np_oracle.pil_resize_bicubic_u8(a), want), (h, w)
        n_vertical_first += np_oracle.pil_vertical_first(h, w)
    assert n_vertical_first >= 80
    for h, w, mode in ((201, 2, "RGB"), (1001, 10, "RGBA"), (200, 2, "RGBA"), (6401, 64, "RGB")):
        a = rng.integers(0, 256, (h, w, len(mode)), dtype=np.uint8)
        want = np.asarray(Image.fromarray(a, mode).convert("L").resize((128, 128)))
        assert np.array_equal(np_oracle.load_image_array(a).reshape(128, 128), want), (h, w, mode)


def _plan(lib, regions, n_frames, fh, fw, cap=1000):
    reg = np.ascontiguousarray(np.asarray(regions, np.int32).reshape(-1, 4))
    chunks = np.full((cap, 4), -7, np.int64)
    m = lib.cnnacc_region_plan_host(reg.ctypes.data_as(ctypes.c_void_p), len(reg), n_frames, fh, fw,
                                    chunks.ctypes.data_as(ctypes.c_void_p), cap)
    assert m >= 1
    return [tuple(int(v) for v in c) for c in chunks[:m]]


def test_staging_plan_of_large_frames():
    """Frames above 16 MiB are staged one per chunk: 4K (24.9 MB) and 8192x8192 (201 MB) centre crops, and the region
    lists of the GPU tests, where an unreferenced frame is never staged."""
    fc.build()
    lib = fc.load()
    for fh, fw in ((2160, 3840), (8192, 8192), (2365, 2365)):
        assert fh * fw * 3 > CHUNK_BYTES
        s = min(fh, fw)
        reg = [(f, (fw - s) // 2, (fh - s) // 2, s) for f in range(5)]
        assert _plan(lib, reg, 5, fh, fw) == [(f, f + 1, f, f + 1) for f in range(5)]
    assert _plan(lib, inputs.REGIONS_4K, 3, 2160, 3840) == [(0, 1, 0, 5), (2, 3, 5, 10)]
    n0 = int((inputs.REGIONS_8192[:, 0] == 0).sum())
    assert _plan(lib, inputs.REGIONS_8192, 2, 8192, 8192) == [(0, 1, 0, n0), (1, 2, n0, len(inputs.REGIONS_8192))]
