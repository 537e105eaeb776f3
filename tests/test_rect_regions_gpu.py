"""Rectangle regions (frame, x, y, w, h) on the GPU (CNNACC_FLAG_RECTS): the pre-processing equals cv2 4.13.0
(tests/golden/rect_cases.npz) and the numpy restatement byte for byte, the predictions equal infer_batch on that gray128,
w == h rectangles equal the square calls on every output, detect_objects equals the merge restatement applied to
detect_regions' own outputs, on host arrays (latency and staged paths) and CUDA tensors, and refusals launch nothing."""
import ctypes
import os

import numpy as np
import pytest

import inputs
import rect_inputs
import rect_oracle
from test_detect_objects_cpu import assert_same
from test_rect_regions_cpu import BAD_RECTS, MERGE_BAD, restate

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rect_cases.npz")


@pytest.fixture(scope="module")
def fc():
    import fpga_cnn_b200
    return fpga_cnn_b200


@pytest.fixture(scope="module")
def acc(fc, shipped_weights):
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    a.load_classifier(*inputs.make_fc())
    yield a
    a.close()


def _vp(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _cpu(x):
    return tuple(t.cpu().numpy() if hasattr(t, "cpu") else t for t in x)


def crops(frames, reg):
    return [frames[f, y:y + h, x:x + w] for f, x, y, w, h in reg]


def vga_rects(fc, n_frames, seed, n_random=30):
    """The aspect grid (128x128, 256x128, 128x256 at stride 64) plus seeded random rectangles on every frame, frame-major."""
    rng = np.random.default_rng(seed)
    grid = fc.grid_rects(n_frames, 480, 640, [(128, 128), (256, 128), (128, 256)], 64)
    w, h = rng.integers(128, 641, n_frames * n_random), rng.integers(128, 481, n_frames * n_random)
    f = np.repeat(np.arange(n_frames), n_random)
    rnd = np.stack([f, rng.integers(0, 641 - w), rng.integers(0, 481 - h), w, h], 1).astype(np.int32)
    return np.concatenate([grid, rnd])


def test_preprocess_regions_equals_opencv_golden(fc, acc):
    """Every case of rect_inputs at an odd offset, all paths in one call: three 8500x8200 frames hold them all."""
    import torch
    gold = np.load(GOLDEN)
    cases = rect_inputs.RECT_CASES
    nf, reg = rect_inputs.pack_rects(cases, 8500, 8200)
    assert nf == 3 and (reg[:, 1] % 2 == 1).all() and (reg[:, 2] % 2 == 1).all()
    frames = np.random.default_rng(31).integers(0, 256, (nf, 8500, 8200, 3), dtype=np.uint8)
    for c, (f, x, y, w, h) in zip(cases, reg):
        frames[f, y:y + h, x:x + w] = rect_inputs.make_rect(c)
    want = np.stack([gold[c["name"]] for c in cases])
    perm = np.random.default_rng(32).permutation(len(reg))
    got = acc.preprocess_regions(frames, reg[perm])
    assert np.array_equal(got, want[perm])
    for i, c in enumerate(cases[:-1]):                                # the restatement too (the 8191 square: CPU test)
        assert np.array_equal(rect_oracle.preprocess_rect(crops(frames, reg[i:i + 1])[0]), want[i]), c["name"]
    t = torch.from_numpy(frames).cuda()
    got = acc.preprocess_regions(t, reg)
    assert got.is_cuda and np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("bbox", ["vec", "upsampled"])
def test_detect_regions_equals_infer_batch(fc, acc, bbox):
    import torch
    frames = inputs.make_frames(("smooth", 1300), 4, 480, 640)
    frames[2] = inputs.make_frames(("rng", 1301), 1, 480, 640)[0]
    reg = vga_rects(fc, 4, 1302)
    perm = np.random.default_rng(1303).permutation(len(reg))
    sh = reg[perm]
    gray_want = np.stack([rect_oracle.preprocess_rect(q) for q in crops(frames, sh)])
    t = torch.from_numpy(frames).cuda()
    for logits in (False, True):
        want = acc.infer_batch(gray_want, bbox=bbox, logits=logits) + (gray_want,)
        got = acc.detect_regions(frames, sh, bbox=bbox, logits=logits, return_gray=True)           # staged host path
        assert_same(got, want, ("host", logits))
        small = acc.detect_regions(frames, sh[:40], bbox=bbox, logits=logits, return_gray=True)    # latency path
        assert_same(small, tuple(a[:40] for a in want), ("small", logits))
        dev = acc.detect_regions(t, sh, bbox=bbox, logits=logits, return_gray=True)
        assert all(d.is_cuda for d in dev)
        assert_same(_cpu(dev), want, ("device", logits))


def test_rects_with_equal_sides_equal_squares(fc, acc):
    import torch
    frames = inputs.make_frames(("smooth", 1400), 3, 480, 640)
    frames[1] = inputs.make_frames(("edges", 1401), 1, 480, 640)[0]
    sq = fc.grid_regions(3, 480, 640, [480, 256, 200, 129, 128], [160, 128, 100, 61, 64])
    sq = sq[np.random.default_rng(1402).permutation(len(sq))]
    rc = np.c_[sq, sq[:, 3]]
    t = torch.from_numpy(frames).cuda()
    for f in (frames, t):
        for bbox, logits in (("vec", False), ("upsampled", True)):
            assert_same(_cpu(acc.detect_regions(f, rc, bbox=bbox, logits=logits, return_gray=True)),
                        _cpu(acc.detect_regions(f, sq, bbox=bbox, logits=logits, return_gray=True)), (bbox, logits))
        kw = dict(score_min=0.2, iou_max=0.4, max_det=50)
        assert_same(_cpu(acc.detect_objects(f, rc, **kw)), _cpu(acc.detect_objects(f, sq, **kw)))
    assert np.array_equal(acc.preprocess_regions(frames, rc), acc.preprocess_regions(frames, sq))


def _expected(acc, frames, reg, bbox="vec", logits=False, score_min=0.0, iou_max=0.5, max_det=100, agnostic=False):
    cls, probs, box = _cpu(acc.detect_regions(frames, reg, bbox=bbox, logits=logits))
    scores = probs[np.arange(len(cls)), cls]
    return restate(reg, scores, cls, box, len(frames), score_min, iou_max, max_det, agnostic), box


def test_detect_objects_equals_restatement_of_detect_regions(fc, acc):
    import torch
    frames = inputs.make_frames(("smooth", 1500), 5, 480, 640)
    frames[3] = inputs.make_frames(("rng", 1501), 1, 480, 640)[0]
    reg = vga_rects(fc, 5, 1502)
    reg = reg[reg[:, 0] != 1]                                            # a frame without regions
    reg = reg[np.random.default_rng(1503).permutation(len(reg))]
    t = torch.from_numpy(frames).cuda()
    for bbox, logits, agnostic, iou_max, max_det in (("vec", False, False, 0.5, 100), ("upsampled", True, True, 0.3, 7)):
        cls, probs, box = acc.detect_regions(frames, reg, bbox=bbox, logits=logits)
        scores = probs[np.arange(len(cls)), cls]
        score_min = float(np.median(scores))
        want = restate(reg, scores, cls, box, len(frames), score_min, iou_max, max_det, agnostic)
        kw = dict(score_min=score_min, iou_max=iou_max, max_det=max_det, class_agnostic=agnostic, bbox=bbox, logits=logits)
        got = acc.detect_objects(frames, reg, **kw)
        assert_same(got, want, ("host", bbox))
        assert_same(_cpu(acc.detect_objects(t, reg, **kw)), want, ("device", bbox))
        n_det, region, *_, det_box = got
        assert n_det[1] == 0 and (n_det > 0).sum() >= 3
        for f in range(len(frames)):                                     # boxes: region_boxes_to_frame's, as float32
            kept = region[f, :n_det[f]]
            b = np.clip(box[kept], 0, 127)
            assert np.array_equal(det_box[f, :n_det[f]], fc.region_boxes_to_frame(reg[kept], b).astype(np.float32))
        few = reg[np.isin(reg[:, 0], [0, 4])][:50]                       # latency path
        want_few, _ = _expected(acc, frames, few, bbox, logits, score_min, iou_max, max_det, agnostic)
        assert_same(acc.detect_objects(frames, few, **kw), want_few, ("small", bbox))
    # the merge alone on the same predictions, host and device
    cls, probs, box = acc.detect_regions(frames, reg)
    scores = probs[np.arange(len(cls)), cls]
    want = restate(reg, scores, cls, box, len(frames), 0.3, 0.5, 100, False)
    assert_same(acc.merge_regions(reg, cls, scores, box, len(frames), score_min=0.3), want)
    tm = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (cls, scores, box)]
    assert_same(_cpu(acc.merge_regions(reg, *tm, len(frames), score_min=0.3)), want)


def test_device_path_frame_across_chunk_edge(fc, acc):
    """3 frames x 10 000 rectangles: the device path's 16384-region pieces end at frame edges."""
    import torch
    rng = np.random.default_rng(16)
    frames = inputs.make_frames(("smooth", 1600), 3, 480, 640)
    w, h = rng.choice([128, 160, 256, 300], 30000), rng.choice([128, 129, 200, 384], 30000)
    reg = np.stack([np.repeat(np.arange(3), 10000), rng.integers(0, 641 - w), rng.integers(0, 481 - h), w, h], 1).astype(np.int32)
    want, _ = _expected(acc, frames, reg, max_det=300, iou_max=0.4)
    got = acc.detect_objects(torch.from_numpy(frames).cuda(), reg, max_det=300, iou_max=0.4)
    assert_same(_cpu(got), want)
    assert (want[0] > 0).all()


def test_refusals_launch_nothing(fc, acc):
    frames = np.zeros((3, 480, 640, 3), np.uint8)
    R = fc._lib.FLAG_RECTS
    D = 16
    n_det, det_reg, det_cls = np.zeros(3, np.int32), np.zeros((3, D), np.int32), np.zeros((3, D), np.int32)
    det_score, det_box = np.zeros((3, D), np.float32), np.zeros((3, D, 4), np.float32)
    dets = [_vp(a) for a in (n_det, det_reg, det_cls, det_score, det_box)]
    n0 = acc.launch_count
    for name, bad in sorted(BAD_RECTS.items()):
        reg = np.ascontiguousarray(bad, np.int32)
        n = len(reg)
        gray = np.zeros((n, 128, 128), np.uint8)
        cls, probs, box = np.zeros(n, np.int32), np.zeros((n, 6), np.float32), np.zeros((n, 4), np.int32)
        L = acc._libc
        assert L.cnnacc_preprocess_regions(acc._h, _vp(frames), 3, 480, 640, _vp(reg), n, _vp(gray), R) == fc._lib.ERR_ARG, name
        assert L.cnnacc_detect_regions(acc._h, _vp(frames), 3, 480, 640, _vp(reg), n, _vp(gray), _vp(probs), _vp(cls), _vp(box),
                                       R) == fc._lib.ERR_ARG, name
        assert L.cnnacc_detect_objects(acc._h, _vp(frames), 3, 480, 640, _vp(reg), n, 0.0, 0.5, D, *dets, R) == fc._lib.ERR_ARG, name
        if name != "decreasing":                                          # the wrapper groups regions by frame itself
            with pytest.raises(ValueError):
                acc.detect_regions(frames, bad)
    sc, cl, bb = np.zeros(2, np.float32), np.zeros(2, np.int32), np.zeros((2, 4), np.int32)
    for name, bad in sorted(MERGE_BAD.items()):
        reg = np.ascontiguousarray(bad, np.int32)
        assert acc._libc.cnnacc_merge_regions(acc._h, _vp(reg), 2, 2, _vp(sc), _vp(cl), _vp(bb), 0.0, 0.5, D, *dets,
                                              R) == fc._lib.ERR_ARG, name
        if name != "decreasing":
            with pytest.raises(ValueError):
                acc.merge_regions(bad, cl, sc, bb, 2)
    assert acc.launch_count == n0
