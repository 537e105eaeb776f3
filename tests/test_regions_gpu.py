"""Region calls on the GPU (csrc/regions.cuh, cnnacc_detect_regions / cnnacc_preprocess_regions): every region's outputs
equal those of the centre-crop path for that square cut out as a frame of its own, and the pre-processing equals OpenCV
through the numpy restatement (oracle/np_oracle.py).  u8 / i32 outputs and fp32 probabilities must match exactly."""
import ctypes
import os

import numpy as np
import pytest

import inputs
from oracle import np_oracle
from test_regions_cpu import BAD_REGIONS

pytestmark = pytest.mark.gpu


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
    return a.ctypes.data_as(ctypes.c_void_p)


def detect_frames_c(fc, acc, frames, bbox="vec", logits=False):
    """cnnacc_detect_frames with every flag the region call takes -> (cls, probs, bbox, gray)."""
    frames = np.ascontiguousarray(frames)
    n = len(frames)
    flags = (fc._lib.FLAG_BBOX_UPSAMPLED if bbox == "upsampled" else 0) | (fc._lib.FLAG_LOGITS if logits else 0)
    cls, probs = np.empty(n, np.int32), np.empty((n, 6), np.float32)
    box, gray = np.empty((n, 4), np.int32), np.empty((n, 128, 128), np.uint8)
    acc._check(acc._libc.cnnacc_detect_frames(acc._h, _vp(frames), n, frames.shape[1], frames.shape[2], _vp(gray), _vp(probs),
                                              _vp(cls), _vp(box), flags))
    return cls, probs, box, gray


def squares(frames, regions):
    return [frames[f, y:y + s, x:x + s] for f, x, y, s in regions]


def assert_same(got, want, what=""):
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.dtype == w.dtype and g.shape == w.shape, (what, i)
        assert np.array_equal(g.view(np.uint8), w.view(np.uint8)), (what, i)


@pytest.mark.parametrize("h,w", [(480, 640), (720, 1280), (1280, 720), (300, 300)])
def test_centre_regions_equal_detect_frames(fc, acc, h, w):
    frames = inputs.make_frames(("smooth", h + 3 * w), 3, h, w)
    frames[1] = inputs.make_frames(("edges", h), 1, h, w)[0]
    s = min(h, w)
    reg = np.array([(f, (w - s) // 2, (h - s) // 2, s) for f in range(3)], np.int32)
    for bbox in ("vec", "upsampled"):
        for logits in (False, True):
            got = acc.detect_regions(frames, reg, bbox=bbox, logits=logits, return_gray=True)
            assert_same(got, detect_frames_c(fc, acc, frames, bbox, logits), (h, w, bbox, logits))


def _check_against_squares(fc, acc, frames, reg, bbox="vec"):
    cls, probs, box, gray = acc.detect_regions(frames, reg, bbox=bbox, return_gray=True)
    sq = squares(frames, reg)
    for i, q in enumerate(sq):
        assert np.array_equal(gray[i], np_oracle.preprocess_bgr(q)), (i, tuple(reg[i]))
    for side in sorted(set(reg[:, 3].tolist())):                       # detect_frames on the extracted squares, by side
        idx = np.flatnonzero(reg[:, 3] == side)
        want = detect_frames_c(fc, acc, np.stack([sq[i] for i in idx]), bbox)
        assert_same((cls[idx], probs[idx], box[idx], gray[idx]), want, side)
    return cls


def test_grid_and_pyramid_over_vga(fc, acc):
    frames = inputs.make_frames(("smooth", 200), 3, 480, 640)
    frames[2] = inputs.make_frames(("rng", 201), 1, 480, 640)[0]
    grid = fc.grid_regions(1, 480, 640, 128, 64)
    pyr = fc.grid_regions(1, 480, 640, [480, 240, 128], [240, 120, 64])
    pyr[:, 0] = 1
    extra = np.array([(2, 640 - 479, 1, 479), (2, 0, 480 - 333, 333), (2, 640 - 200, 480 - 200, 200), (2, 7, 0, 129),
                      (2, 640 - 256, 0, 256), (2, 0, 0, 384)], np.int32)
    reg = np.concatenate([grid, pyr, extra])
    _check_against_squares(fc, acc, frames, reg)
    _check_against_squares(fc, acc, frames, reg[::7], bbox="upsampled")


def test_every_path_in_one_call(fc, acc):
    """Sides 128 (copy), 256 (2x2), 384 / 768 (k x k) and fractional ones in one launch, touching all four edges."""
    fh, fw = 800, 1024
    frames = inputs.make_frames(("rng", 300), 2, fh, fw)
    frames[1] = inputs.make_frames(("edges", 301), 1, fh, fw)[0]
    reg = []
    for f in range(2):
        for s in (128, 256, 384, 768, 129, 200, 333, 479):
            reg += [(f, 0, 0, s), (f, fw - s, fh - s, s), (f, fw - s, 0, s), (f, 0, fh - s, s), (f, (fw - s) // 3, (fh - s) // 2, s)]
    _check_against_squares(fc, acc, frames, np.array(reg, np.int32))


def test_cpu_chain(fc, acc):
    from oracle import load_port, port_infer
    port = load_port()
    fw_, fb_ = inputs.make_fc()
    wt = np.fromfile(os.path.join(os.path.dirname(__file__), "golden", "weights.bin"), dtype=np.uint8)
    frames = inputs.make_frames(("smooth", 400), 2, 480, 640)
    reg = np.array([(0, 0, 0, 480), (0, 512, 352, 128), (1, 100, 50, 333), (1, 3, 4, 200)], np.int32)
    cls, probs, box, gray = acc.detect_regions(frames, reg, return_gray=True)
    for i, q in enumerate(squares(frames, reg)):
        g = np_oracle.preprocess_bgr(q)
        assert np.array_equal(gray[i], g)
        f = port_infer(port, g, wt, (7, 10, 11))
        c, p, _, _ = np_oracle.classify_vec(f, fw_, fb_)
        assert c == cls[i] and np.abs(p - probs[i]).max() <= 1e-5
        assert np_oracle.bbox_vec(f, c, fw_)[0] == tuple(box[i])
    cls_u, _, box_u = acc.detect_regions(frames, reg, bbox="upsampled")
    assert np.array_equal(cls_u, cls)
    assert np.array_equal(box_u, acc.cam_bbox_batch(acc.run_batch(gray).reshape(len(reg), 64, 256), cls))


def test_host_staging_equals_small_calls(fc, acc):
    n = 72
    frames = inputs.make_frames(("smooth", 500), n, 480, 640)
    rng = np.random.default_rng(7)
    tiles = fc.grid_regions(1, 480, 640, [128, 160, 333], [16, 40, 60])
    counts = rng.integers(0, 5, n)
    counts[[0, 1, 30, 31, 32, n - 1]] = 0                              # unreferenced leading, gap and trailing frames
    counts[40] = 1100                                                  # more than one launch of a chunk holds
    reg = np.array([(f, *tiles[rng.integers(len(tiles)), 1:]) for f in range(n) for _ in range(counts[f])], np.int32)
    assert len(reg) > 64
    got = acc.detect_regions(frames, reg, return_gray=True)
    parts = [acc.detect_regions(frames, reg[i:i + 64], return_gray=True) for i in range(0, len(reg), 64)]
    want = [np.concatenate([p[k] for p in parts]) for k in range(4)]
    assert_same(got, want)
    assert_same((acc.preprocess_regions(frames, reg),), (got[3],))
    for i in rng.choice(len(reg), 12, replace=False):
        f, x, y, s = reg[i]
        assert np.array_equal(got[3][i], np_oracle.preprocess_bgr(frames[f, y:y + s, x:x + s])), i


def test_device_pointers(fc, acc):
    import torch
    frames = inputs.make_frames(("smooth", 600), 4, 480, 640)
    regs = [fc.grid_regions(4, 480, 640, 128, 64)[::5], fc.grid_regions(4, 480, 640, [240, 333], [120, 100]),
            np.array([(3, 0, 0, 480), (0, 1, 2, 129)], np.int32)]
    regs += [r[np.random.default_rng(i).permutation(len(r))] for i, r in enumerate(regs)]   # unsorted as well
    want = [acc.detect_regions(frames, r, bbox="upsampled", return_gray=True) for r in regs]
    t = torch.from_numpy(frames).cuda()
    torch.cuda.synchronize()
    torch.cuda._sleep(100_000_000)          # keep the stream busy: every call below is queued before any of them runs
    got = [acc.detect_regions(t, r, bbox="upsampled", return_gray=True) for r in regs]
    g2 = acc.preprocess_regions(t, regs[0])
    torch.cuda.synchronize()
    for k, (g, w) in enumerate(zip(got, want)):
        assert_same([x.cpu().numpy() for x in g], w, k)
    assert np.array_equal(g2.cpu().numpy(), want[0][3])


def test_refusals_launch_nothing(fc, acc, shipped_weights):
    frames = np.zeros((3, 480, 640, 3), np.uint8)
    probs, cls = np.zeros((8, 6), np.float32), np.zeros(8, np.int32)
    box, gray = np.zeros((8, 4), np.int32), np.zeros((8, 128, 128), np.uint8)
    for name, bad in sorted(BAD_REGIONS.items()):
        reg = np.array(bad, np.int32)
        n0 = acc.launch_count
        for call in (lambda: acc._libc.cnnacc_detect_regions(acc._h, _vp(frames), 3, 480, 640, _vp(reg), len(reg), _vp(gray),
                                                             _vp(probs), _vp(cls), _vp(box), 0),
                     lambda: acc._libc.cnnacc_preprocess_regions(acc._h, _vp(frames), 3, 480, 640, _vp(reg), len(reg), _vp(gray), 0)):
            with pytest.raises(ValueError):
                acc._check(call())
        if name != "decreasing":                                   # the wrapper sorts by frame, so that one cannot reach it
            with pytest.raises(ValueError):
                acc.detect_regions(frames, reg)
        assert acc.launch_count == n0, name
    ok = np.array([(0, 0, 0, 128)], np.int32)
    n0 = acc.launch_count
    for args in ((None, 3, _vp(ok), 1), (_vp(frames), 3, None, 1)):    # NULL frames / regions
        rc = acc._libc.cnnacc_detect_regions(acc._h, args[0], args[1], 480, 640, args[2], args[3], None, _vp(probs), _vp(cls),
                                             _vp(box), 0)
        assert rc == fc._lib.ERR_ARG
    assert acc._libc.cnnacc_detect_regions(acc._h, None, 0, 480, 640, None, 0, None, None, None, None, 0) == 0
    assert acc.launch_count == n0
    c, p, b, g = acc.detect_regions(frames, np.zeros((0, 4), np.int32), return_gray=True)
    assert c.shape == (0,) and p.shape == (0, 6) and b.shape == (0, 4) and g.shape == (0, 128, 128)
    bare = fc.CNNAccelerator()                                         # no weights, then no classifier: -4
    try:
        args = (_vp(frames), 3, 480, 640, _vp(ok), 1, None, _vp(probs), _vp(cls), _vp(box), 0)
        assert bare._libc.cnnacc_detect_regions(bare._h, *args) == fc._lib.ERR_STATE
        bare.load_weights(shipped_weights)
        assert bare._libc.cnnacc_detect_regions(bare._h, *args) == fc._lib.ERR_STATE
        assert bare.launch_count == 0
    finally:
        bare.close()
