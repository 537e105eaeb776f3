"""CPU-side checks of the rectangle region calls (CNNACC_FLAG_RECTS): the numpy restatement of OpenCV's INTER_AREA on an
(h, w) source against cv2 4.13.0 (tests/golden/rect_cases.npz) and against the square restatement, the refusals and the
staging plan through cnnacc_rect_plan_host, the merge of rectangles through cnnacc_merge_regions_host against a numpy
restatement with (w, h), grid_rects, region_boxes_to_frame on (R, 5), and what the Python wrapper sends to the library."""
import ctypes
import os

import numpy as np
import pytest

import fpga_cnn_b200 as fc
import rect_inputs
import rect_oracle
import test_detect_objects_cpu as sq
from oracle import np_oracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rect_cases.npz")
VGA = (480, 640)


@pytest.fixture(scope="module")
def lib():
    fc.build()
    return fc.load()


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


# ---- pre-processing: the restatement -------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", rect_inputs.RECT_CASES, ids=lambda c: c["name"])
def test_restatement_equals_opencv_golden(case):
    gold = np.load(GOLDEN)
    assert str(gold["cv2_version"]) == "4.13.0"
    assert np.array_equal(rect_oracle.preprocess_rect(rect_inputs.make_rect(case)), gold[case["name"]])


def test_golden_covers_every_path():
    paths = set()
    for c in rect_inputs.RECT_CASES:
        h, w = c["h"], c["w"]
        if h % 128 or w % 128:
            paths.add("frac_" + ("both" if h % 128 and w % 128 else "one"))
        else:
            paths.add({1: "copy", 4: "2x2" if h == w else "int"}.get(h * w // 128 ** 2, "int"))
    assert paths == {"copy", "2x2", "int", "frac_one", "frac_both"}


@pytest.mark.parametrize("side", [128, 129, 200, 256, 333, 384, 512, 640, 1000, 1152])
def test_restatement_of_squares_is_the_square_one(side):
    rng = np.random.default_rng(side)
    for g in (rng.integers(0, 256, (side, side), dtype=np.uint8), rng.integers(0, 4, (side, side), dtype=np.uint8)):
        assert np.array_equal(rect_oracle.resize_area_rect_u8(g), np_oracle.resize_area_u8(g))


# ---- refusals and the staging plan -----------------------------------------------------------------------------------------

def _plan(lib, regions, n_frames, fh=VGA[0], fw=VGA[1], cap=100000, rects=True):
    k = 5 if rects else 4
    reg = np.ascontiguousarray(np.asarray(regions, np.int32).reshape(-1, k))
    chunks = np.full((cap, 4), -7, np.int64)
    fn = lib.cnnacc_rect_plan_host if rects else lib.cnnacc_region_plan_host
    m = fn(_p(reg), len(reg), n_frames, fh, fw, _p(chunks), cap)
    return m, chunks[:max(m, 0)]


BAD_RECTS = {
    "frame_negative": [(-1, 0, 0, 128, 128)],
    "frame_too_big": [(0, 0, 0, 128, 128), (3, 0, 0, 128, 128)],
    "w_small": [(0, 0, 0, 127, 200)],
    "h_small": [(0, 0, 0, 200, 127)],
    "w_big": [(0, 0, 0, 8193, 128)],
    "h_big": [(0, 0, 0, 128, 8193)],
    "x_negative": [(0, -1, 0, 128, 128)],
    "y_negative": [(0, 0, -1, 128, 128)],
    "x_past_edge": [(0, 385, 0, 256, 128)],
    "y_past_edge": [(0, 0, 225, 128, 256)],
    "w_past_edge": [(0, 0, 0, 641, 128)],
    "h_past_edge": [(0, 0, 0, 128, 481)],
    "decreasing": [(1, 0, 0, 128, 200), (0, 0, 0, 200, 128)],
    "overflow_x": [(0, 2 ** 31 - 100, 0, 200, 128)],
    "overflow_y": [(0, 0, 2 ** 31 - 100, 128, 200)],
}


@pytest.mark.parametrize("name", sorted(BAD_RECTS))
def test_refusals(lib, name):
    assert _plan(lib, BAD_RECTS[name], 3)[0] == fc._lib.ERR_ARG       # the check the real calls run (test_rect_regions_gpu.py)


def test_rect_edges_accepted(lib):
    ok = [(0, 0, 0, 640, 480), (0, 0, 0, 8192 // 16, 128), (1, 0, 352, 640, 128), (1, 512, 0, 128, 480), (2, 511, 351, 129, 129),
          (2, 0, 0, 128, 128)]
    m, chunks = _plan(lib, ok, 3)
    assert m == 1 and tuple(chunks[0]) == (0, 3, 0, 6)
    assert _plan(lib, [(0, 0, 0, 8192, 8192)], 1, 8192, 8192)[0] == 1
    assert _plan(lib, [(0, 0, 0, 128, 8192)], 1, 8192, 128)[0] == 1
    assert _plan(lib, np.zeros((0, 5), np.int32), 3)[0] == 0
    assert lib.cnnacc_rect_plan_host(None, 1, 3, 480, 640, _p(np.zeros(4, np.int64)), 1) == fc._lib.ERR_ARG


def test_plan_depends_only_on_frame_indices(lib):
    """The plan of rectangles is the plan of squares on the same frames (and that of squares written as rectangles)."""
    rng = np.random.default_rng(8)
    counts = rng.integers(0, 5, 120)
    counts[30:37] = 0
    counts[50] = 2500
    f = np.repeat(np.arange(120), counts)
    n = len(f)
    w, h = rng.integers(128, 641, n), rng.integers(128, 481, n)
    x, y = rng.integers(0, 641 - w), rng.integers(0, 481 - h)
    rects = np.stack([f, x, y, w, h], 1)
    s = np.minimum(w, h)
    squares = np.stack([f, x, y, s], 1)
    m, chunks = _plan(lib, rects, 120)
    assert m > 1
    m_sq, chunks_sq = _plan(lib, squares, 120, rects=False)
    assert m == m_sq and np.array_equal(chunks, chunks_sq)
    m_ws, chunks_ws = _plan(lib, np.stack([f, x, y, s, s], 1), 120)
    assert m_ws == m and np.array_equal(chunks_ws, chunks)
    assert np.array_equal(chunks[:, 2], np.r_[0, chunks[:-1, 3]]) and chunks[-1, 3] == n


# ---- the merge ------------------------------------------------------------------------------------------------------------

def frame_boxes(regions, bbox):
    """Boxes in 1/128 frame pixels as int64 (X1, Y1, X2, Y2) for rectangles: X = 128 x + clamp(bx) w, Y = 128 y + clamp(by) h."""
    b = np.clip(np.asarray(bbox, np.int64).reshape(-1, 4), 0, 127)
    reg = np.asarray(regions, np.int64).reshape(-1, 5)
    x, y, w, h = reg[:, 1:2], reg[:, 2:3], reg[:, 3:4], reg[:, 4:5]
    return np.concatenate([128 * x + b[:, 0:1] * w, 128 * y + b[:, 1:2] * h, 128 * x + b[:, 2:3] * w, 128 * y + b[:, 3:4] * h], 1)


def restate(regions, scores, cls, bbox, n_frames, score_min, iou_max, max_det, agnostic):
    """tests/test_detect_objects_cpu.py's restatement of the merge with each region's (w, h) in place of its side."""
    regions = np.asarray(regions, np.int32).reshape(-1, 5)
    scores, cls = np.asarray(scores, np.float32), np.asarray(cls, np.int32)
    B = frame_boxes(regions, bbox)
    im = np.float64(np.float32(iou_max))
    D = max_det
    n_det = np.zeros(n_frames, np.int32)
    d_reg, d_cls = np.full((n_frames, D), -1, np.int32), np.full((n_frames, D), -1, np.int32)
    d_score, d_box = np.zeros((n_frames, D), np.float32), np.zeros((n_frames, D, 4), np.float32)
    for f in range(n_frames):
        kept = []
        for r in sq.ranked_candidates(np.flatnonzero(regions[:, 0] == f), scores, score_min):
            if len(kept) >= D:
                break
            k = np.array(kept, np.int64)
            if not agnostic:
                k = k[cls[k] == cls[r]]
            if len(k) and (sq.iou(B[r], B[k]) > im).any():
                continue
            kept.append(r)
        n = len(kept)
        n_det[f] = n
        d_reg[f, :n], d_cls[f, :n], d_score[f, :n] = kept, cls[kept], scores[kept]
        d_box[f, :n] = (B[kept] / 128.0).astype(np.float32)
    return n_det, d_reg, d_cls, d_score, d_box


def _merge_host(lib, regions, scores, cls, bbox, n_frames, score_min, iou_max, max_det, agnostic, flags):
    scores, cls = np.ascontiguousarray(scores, np.float32), np.ascontiguousarray(cls, np.int32)
    bbox = np.ascontiguousarray(np.asarray(bbox, np.int32).reshape(-1, 4))
    D = max(int(max_det), 1)
    out = (np.full(n_frames, -9, np.int32), np.full((n_frames, D), -9, np.int32), np.full((n_frames, D), -9, np.int32),
           np.full((n_frames, D), -9, np.float32), np.full((n_frames, D, 4), -9, np.float32))
    flags |= fc._lib.FLAG_CLASS_AGNOSTIC if agnostic else 0
    rc = lib.cnnacc_merge_regions_host(_p(regions), len(regions), n_frames, _p(scores), _p(cls), _p(bbox), score_min, iou_max,
                                       max_det, *[_p(a) for a in out], flags)
    return rc, out


def as_rects(case, orient):
    """A square case of test_detect_objects_cpu.py as rectangles: 'wide' doubles x and w, 'tall' doubles y and h (a region
    whose doubled side would pass 8192 keeps its square).  Scaling one axis of every box by 2 scales every area by 2, so
    ties and IoU exactly at iou_max stay exact."""
    reg = case["regions"].astype(np.int64)
    f, x, y, s = reg.T
    k = np.where(2 * s <= 8192, 2, 1)
    if orient == "wide":
        rects = np.stack([f, x * k, y, s * k, s], 1)
    elif orient == "tall":
        rects = np.stack([f, x, y * k, s, s * k], 1)
    else:
        rects = np.stack([f, x, y, s, s], 1)
    return {**case, "regions": rects.astype(np.int32).reshape(-1, 5)}


def random_rect_case(seed, n_frames, max_per_frame, n_cls=5, max_det=100, agnostic=False, iou_max=0.5, score_min=0.2):
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, max_per_frame + 1, n_frames)
    f = np.repeat(np.arange(n_frames), counts)
    n = len(f)
    w, h = rng.choice([128, 160, 256, 300, 384, 640], n), rng.choice([128, 129, 200, 256, 480, 8192], n)
    regions = np.stack([f, rng.integers(0, 641, n), rng.integers(0, 481, n), w, h], 1)
    b1 = rng.integers(-5, 120, (n, 2))
    bbox = np.concatenate([b1, b1 + rng.integers(-3, 70, (n, 2))], 1)
    scores = rng.choice(np.float32([0.0, 0.25, 0.5, 1.0]), n) if seed % 2 else rng.random(n, np.float32)
    return dict(regions=regions.astype(np.int32), scores=scores, cls=rng.integers(0, n_cls, n).astype(np.int32),
                bbox=bbox.astype(np.int32), n_frames=n_frames, score_min=score_min, iou_max=iou_max, max_det=max_det,
                agnostic=agnostic)


RECT_CASES = {f"{name}_{o}": as_rects(c, o) for name, c in sq.CASES.items() if not name.startswith("random")
              for o in ("wide", "tall")}
RECT_CASES.update({f"random_rect_{s}": random_rect_case(s, (50, 30, 20)[s], (400, 2000, 100)[s], agnostic=s == 2,
                                                        max_det=(100, 1024, 5)[s]) for s in range(3)})


def test_rect_cases_keep_the_boundaries():
    assert restate(**RECT_CASES["iou_half_kept_wide"])[0][0] == 4
    assert restate(**RECT_CASES["iou_half_suppressed_tall"])[0][0] == 2
    assert restate(**RECT_CASES["max_det_1024_tall"])[0][0] == 1024
    assert len(RECT_CASES["full_frame_wide"]["regions"]) == 16385
    n, reg, *_ = restate(**RECT_CASES["signed_zero_nan_wide"])
    assert list(reg[0, :n[0]]) == [4, 0, 1, 3, 6]
    r = RECT_CASES["random_rect_1"]["regions"]
    assert (r[:, 3] != r[:, 4]).mean() > 0.5


@pytest.mark.parametrize("name", sorted(RECT_CASES))
def test_merge_regions_host_equals_restatement(lib, name):
    c = RECT_CASES[name]
    rc, got = _merge_host(lib, c["regions"], c["scores"], c["cls"], c["bbox"], c["n_frames"], c["score_min"], c["iou_max"],
                          c["max_det"], c["agnostic"], fc._lib.FLAG_RECTS)
    assert rc == 0
    sq.assert_same(got, restate(**c), name)


@pytest.mark.parametrize("name", sorted(sq.CASES))
def test_squares_as_rects_merge_as_squares(lib, name):
    c = sq.CASES[name]
    r = as_rects(c, "square")
    args = lambda d: (d["scores"], d["cls"], d["bbox"], d["n_frames"], d["score_min"], d["iou_max"], d["max_det"], d["agnostic"])
    rc, got = _merge_host(lib, np.ascontiguousarray(r["regions"]), *args(r), fc._lib.FLAG_RECTS)
    rc_sq, want = _merge_host(lib, np.ascontiguousarray(c["regions"]), *args(c), 0)
    assert rc == rc_sq == 0
    sq.assert_same(got, want, name)


MERGE_BAD = {"frame_negative": [(-1, 0, 0, 128, 128), (1, 0, 0, 128, 128)],
             "frame_too_big": [(0, 0, 0, 128, 128), (2, 0, 0, 128, 128)],
             "decreasing": [(1, 0, 0, 128, 128), (0, 0, 0, 128, 128)],
             "w_small": [(0, 0, 0, 127, 128), (1, 0, 0, 128, 128)], "h_small": [(0, 0, 0, 128, 127), (1, 0, 0, 128, 128)],
             "w_big": [(0, 0, 0, 8193, 128), (1, 0, 0, 128, 128)], "h_big": [(0, 0, 0, 128, 8193), (1, 0, 0, 128, 128)],
             "x_negative": [(0, -1, 0, 128, 200), (1, 0, 0, 128, 128)], "y_negative": [(0, 0, -1, 200, 128), (1, 0, 0, 128, 128)]}


@pytest.mark.parametrize("name", sorted(MERGE_BAD))
def test_merge_refusals(lib, name):
    ok = dict(scores=np.full(2, 0.5, np.float32), cls=np.zeros(2, np.int32), bbox=np.tile(np.int32([0, 0, 9, 9]), (2, 1)),
              n_frames=2, score_min=0.0, iou_max=0.5, max_det=10, agnostic=False)
    good = np.array([(0, 0, 0, 128, 8192), (1, 2 ** 31 - 1, 2 ** 31 - 1, 8192, 128)], np.int32)   # no frame size to check
    rc, _ = _merge_host(lib, good, *ok.values(), fc._lib.FLAG_RECTS)
    assert rc == 0
    rc, _ = _merge_host(lib, np.array(MERGE_BAD[name], np.int32), *ok.values(), fc._lib.FLAG_RECTS)
    assert rc == fc._lib.ERR_ARG


# ---- Python helpers -------------------------------------------------------------------------------------------------------

def test_grid_rects_aspect_grid():
    g = fc.grid_rects(2, 480, 640, [(128, 128), (256, 128), (128, 256)], 64)
    assert g.dtype == np.int32 and g.ndim == 2 and g.shape[1] == 5
    per = len(g) // 2
    assert (g[:per, 0] == 0).all() and (g[per:, 0] == 1).all() and np.array_equal(g[per:, 1:], g[:per, 1:])   # frame-major
    f0 = g[:per]
    sizes = [tuple(s) for s in f0[:, 3:]]
    assert sizes == sorted(sizes, key=[(128, 128), (256, 128), (128, 256)].index)                            # sizes in order
    counts = {s: sizes.count(s) for s in set(sizes)}
    assert counts == {(128, 128): 9 * 7, (256, 128): 7 * 7, (128, 256): 9 * 5}
    wide = f0[(f0[:, 3] == 256)]
    assert sorted(set(wide[:, 1])) == list(range(0, 385, 64)) and sorted(set(wide[:, 2])) == list(range(0, 321, 64)) + [352]
    tall = f0[(f0[:, 4] == 256)]
    assert sorted(set(tall[:, 1])) == list(range(0, 513, 64)) and sorted(set(tall[:, 2])) == list(range(0, 193, 64)) + [224]
    sq_part = f0[:63]
    assert np.array_equal(sq_part[:, [0, 1, 2, 3]], fc.grid_regions(1, 480, 640, 128, 64))
    assert (np.lexsort((sq_part[:, 1], sq_part[:, 2])) == np.arange(63)).all()        # within a size: y, then x


@pytest.mark.parametrize("fh,fw,sizes,strides", [(480, 640, [(200, 130), (129, 479)], (50, 33)),
                                                 (300, 700, (700, 128), [(1, 1)]),
                                                 (720, 1280, [(1280, 128), (128, 720)], [(100, 64), (64, 100)])])
def test_grid_rects_cover_every_pixel(fh, fw, sizes, strides):
    g = fc.grid_rects(2, fh, fw, sizes, strides)
    sizes = np.asarray(sizes).reshape(-1, 2)
    st = np.broadcast_to(np.asarray(strides).reshape(-1, 2), sizes.shape)
    for (w, h), (sx, sy) in zip(sizes, st):
        t = g[(g[:, 0] == 1) & (g[:, 3] == w) & (g[:, 4] == h)]
        cover = np.zeros((fh, fw), bool)
        for _, x, y, _, _ in t:
            assert 0 <= x and x + w <= fw and 0 <= y and y + h <= fh
            cover[y:y + h, x:x + w] = True
        assert cover.all() and len(set(map(tuple, t[:, 1:3].tolist()))) == len(t)
        xs, ys = sorted(set(t[:, 1].tolist())), sorted(set(t[:, 2].tolist()))
        assert xs[-1] == fw - w and ys[-1] == fh - h
        assert all(b - a <= sx for a, b in zip(xs, xs[1:])) and all(b - a <= sy for a, b in zip(ys, ys[1:]))


def test_grid_rects_equals_grid_regions_for_squares():
    want = fc.grid_regions(3, 480, 640, [128, 200, 333], [64, 100, 150])
    got = fc.grid_rects(3, 480, 640, [(128, 128), (200, 200), (333, 333)], [(64, 64), (100, 100), (150, 150)])
    assert np.array_equal(got[:, :4], want) and np.array_equal(got[:, 4], want[:, 3])


def test_grid_rects_rejections():
    for sizes, strides in (((641, 128), 64), ((128, 481), 64), ((128, 128), 0), ((128, 128), (64, 0)),
                           ([(128, 128), (256, 128)], [(64, 64)] * 3)):
        with pytest.raises(ValueError):
            fc.grid_rects(1, 480, 640, sizes, strides)


def test_region_boxes_to_frame_rects():
    reg = np.array([(0, 10, 20, 256, 128), (3, 100, 7, 128, 384), (1, 5, 6, 333, 129)], np.int32)
    box = np.array([(0, 0, 127, 127), (10, 20, 30, 40), (1, 2, 3, 4)], np.int32)
    got = fc.region_boxes_to_frame(reg, box)
    assert got.dtype == np.float64 and got.shape == (3, 4)
    want = np.array([[10, 20, 10 + 254, 20 + 127], [110, 7 + 60, 130, 7 + 120],
                     [5 + 333 / 128, 6 + 2 * 129 / 128, 5 + 3 * 333 / 128, 6 + 4 * 129 / 128]])
    assert np.array_equal(got, want)
    sqr = np.array([(0, 10, 20, 256), (3, 100, 7, 333)], np.int32)
    assert np.array_equal(fc.region_boxes_to_frame(np.c_[sqr, sqr[:, 3]], box[:2]), fc.region_boxes_to_frame(sqr, box[:2]))
    # its float32 cast is the merge's box, bit for bit
    c = RECT_CASES["random_rect_0"]
    inside = (c["bbox"] >= 0).all(1) & (c["bbox"] <= 127).all(1)
    want = fc.region_boxes_to_frame(c["regions"][inside], c["bbox"][inside]).astype(np.float32)
    got = (frame_boxes(c["regions"][inside], c["bbox"][inside]) / 128.0).astype(np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


# ---- what the wrapper sends -----------------------------------------------------------------------------------------------

class _Lib:
    """Records every library call: name, arguments and the int32 region records behind the region pointer."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def call(*args):
            if name in ("cnnacc_detect_regions", "cnnacc_preprocess_regions", "cnnacc_detect_objects"):
                p, n = args[5], args[6]
            else:                                                      # cnnacc_merge_regions
                p, n = args[1], args[2]
            if name in ("cnnacc_detect_objects", "cnnacc_merge_regions"):  # no detections: det_region -1
                n_frames = args[2] if name == "cnnacc_detect_objects" else args[3]
                det_region = ctypes.cast(args[11], ctypes.POINTER(ctypes.c_int32))
                np.ctypeslib.as_array(det_region, shape=(n_frames * args[9],))[:] = -1
            k = 5 if args[-1] & fc._lib.FLAG_RECTS else 4
            recs = np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_int32)), shape=(n, k)).copy() if n else None
            self.calls.append((name, recs, args[-1]))
            return 0
        return call


class _Recorder(fc.CNNAccelerator):
    def __init__(self):                                    # no cnnacc_create: nothing here touches a GPU
        self._n_cls = 3
        self._h = None
        self._libc = _Lib()

    def _check(self, rc):
        assert rc == 0


@pytest.mark.parametrize("k", [4, 5])
def test_wrapper_sends_records_and_flag(k):
    acc = _Recorder()
    rng = np.random.default_rng(k)
    reg = fc.grid_rects(3, 300, 300, [(128, 200), (256, 128)], 50)
    reg = reg[:, :4] if k == 4 else reg
    perm = rng.permutation(len(reg))
    shuffled = reg[perm].astype(np.int64)
    frames = np.zeros((3, 300, 300, 3), np.uint8)
    acc.detect_regions(frames, shuffled, return_gray=True)
    acc.preprocess_regions(frames, shuffled)
    acc.detect_objects(frames, shuffled)
    acc.merge_regions(shuffled, np.zeros(len(reg), np.int32), np.zeros(len(reg), np.float32), np.zeros((len(reg), 4), np.int32), 3)
    names = [c[0] for c in acc._libc.calls]
    assert names == ["cnnacc_detect_regions", "cnnacc_preprocess_regions", "cnnacc_detect_objects", "cnnacc_merge_regions"]
    for name, recs, flags in acc._libc.calls:
        assert bool(flags & fc._lib.FLAG_RECTS) == (k == 5), name
        assert recs.shape == (len(reg), k)
        assert np.array_equal(recs, shuffled[np.argsort(shuffled[:, 0], kind="stable")]), name    # grouped by frame, stably


def test_wrapper_refuses_other_shapes():
    acc = _Recorder()
    frames = np.zeros((1, 300, 300, 3), np.uint8)
    for bad in (np.zeros((2, 3), np.int32), np.zeros((2, 6), np.int32), np.zeros(5, np.int32), np.zeros((2, 5), np.float32),
                [(0, 0, 0, 128, 2 ** 31)]):
        with pytest.raises(ValueError):
            acc.detect_regions(frames, bad)
        with pytest.raises(ValueError):
            acc.detect_objects(frames, bad)
    assert acc._libc.calls == []
    cls, probs, box = acc.detect_regions(frames, np.zeros((0, 5), np.int32))
    assert cls.shape == (0,) and probs.shape == (0, 3) and box.shape == (0, 4)
