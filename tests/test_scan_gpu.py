"""The scanning calls on the GPU (cnnacc_scan_frames / cnnacc_scan_objects): every window's predictions equal classify_batch
on that window cut out of run_batch's feature map of the frame's gray, bit for bit, on the shipped weights and the exposed
ternary workloads at both accumulator widths; the numpy restatement (tests/scan_oracle.py) end to end; 128x128 frames
against detect_regions and detect_frames; host arrays against CUDA tensors on every path; scan_objects against merge_regions
on scan_frames' outputs; refusals that launch nothing; and bounded device memory over repeated calls."""
import ctypes

import numpy as np
import pytest

import inputs
import scan_oracle
from oracle import np_oracle
from test_detect_objects_cpu import assert_same

pytestmark = pytest.mark.gpu

STRIDES = [8, 16, 24, 64, 120, 128]
SIZES = [(128, 128), (144, 272), (480, 640), (720, 1280), (8192, 128)]
TERNARY = [w for w in inputs.EXPOSED_WORKLOADS if w["name"].startswith("tern")]
CONFIGS = [("shipped", "shipped", (7, 10, 11), bits) for bits in (32, 24)] + \
          [(w["name"], w["weights"], w["shifts"], bits) for w in TERNARY for bits in (32, 24)]
LOGIT_RTOL = 1e-5
PROB_ATOL = 1e-5


@pytest.fixture(scope="module")
def fc():
    import fpga_cnn_b200
    fpga_cnn_b200.load()
    return fpga_cnn_b200


@pytest.fixture(scope="module")
def acc(fc, shipped_weights):
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    a.load_classifier(*inputs.make_fc())
    yield a
    a.close()


@pytest.fixture
def shipped(acc, shipped_weights):
    """acc with the shipped weights at shifts (7, 10, 11) and 32-bit accumulators (tests that reconfigure it restore this)."""
    acc.load_weights(shipped_weights)
    acc.set_shifts(7, 10, 11)
    acc.set_accumulator_bits(32)
    return acc


def configure(acc, shipped_weights, weights, shifts, bits):
    acc.load_weights(shipped_weights if weights == "shipped" else inputs.make_weights(weights))
    acc.set_shifts(*shifts)
    acc.set_accumulator_bits(bits)


def _np(x):
    return tuple(np.asarray(t.cpu()) if hasattr(t, "cpu") else t for t in x)


def frames_of(n, fh, fw, seed):
    """Uniform frames for odd seeds, smooth ones for even seeds."""
    return inputs.make_frames(("rng" if seed % 2 else "smooth", seed), n, fh, fw)


def reference(fc, acc, frames, stride, logits=False, maps=None):
    """classify_batch(run_batch(gray)[window slices]) -> (cls, probs, bbox)."""
    n, fh, fw, _ = frames.shape
    if maps is None:
        maps = acc.run_batch(np.stack([np_oracle.bgr_to_gray(f) for f in frames]))
    wm = scan_oracle.window_maps(maps, fc.grid_regions(n, fh, fw, 128, stride))
    return acc.classify_batch(np.ascontiguousarray(wm), logits=logits)


# ---- classify equality ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("fh,fw", SIZES, ids=lambda s: str(s))
@pytest.mark.parametrize("name,weights,shifts,bits", CONFIGS, ids=[f"{c[0]}-{c[3]}" for c in CONFIGS])
def test_scan_equals_classify_of_window_maps(fc, acc, shipped_weights, name, weights, shifts, bits, fh, fw):
    configure(acc, shipped_weights, weights, shifts, bits)
    n = 2 if fh * fw <= 480 * 640 else 1
    frames = frames_of(n, fh, fw, 40 + len(name) + bits)
    maps = acc.run_batch(np.stack([np_oracle.bgr_to_gray(f) for f in frames]))
    for stride in STRIDES:
        for logits in (False, True):
            want = reference(fc, acc, frames, stride, logits, maps)
            assert_same(acc.scan_frames(frames, stride, logits=logits), want, (stride, logits))
            assert len(want[0]) == n * scan_oracle.count(fh, stride) * scan_oracle.count(fw, stride)


# ---- the numpy restatement end to end -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("bits", [32, 24])
@pytest.mark.parametrize("w", TERNARY, ids=lambda w: w["name"])
def test_scan_against_restatement(fc, acc, shipped_weights, w, bits):
    configure(acc, shipped_weights, w["weights"], w["shifts"], bits)
    fw_, fb = inputs.make_fc()
    checked = 0
    for (fh, fwd), stride in (((128, 128), 64), ((144, 272), 8), ((256, 384), 24)):
        frames = frames_of(2, fh, fwd, 50 + bits)
        _, _, cls_r, prob_r, logit_r, box_r = scan_oracle.scan(frames, inputs.make_weights(w["weights"]), w["shifts"], fw_, fb, stride, bits)
        for logits in (False, True):
            cls, probs, box = _np(acc.scan_frames(frames, stride, logits=logits))
            assert len(cls) == len(cls_r)
            for i in range(len(cls)):
                scale = np.abs(logit_r[i]).max()
                if cls[i] != cls_r[i]:
                    top2 = np.sort(logit_r[i])[-2:]
                    assert top2[1] - top2[0] <= LOGIT_RTOL * scale, (fh, fwd, stride, i)
                    continue
                if logits:
                    assert np.abs(probs[i] - logit_r[i]).max() <= LOGIT_RTOL * scale, (fh, fwd, stride, i)
                else:
                    assert np.abs(probs[i] - prob_r[i]).max() <= PROB_ATOL, (fh, fwd, stride, i)
                assert tuple(box[i]) == tuple(box_r[i]), (fh, fwd, stride, i)
                checked += 1
    assert checked > 400


# ---- 128x128 frames: the same computation as the per-region and per-frame calls ----------------------------------------------

def test_128_frames_equal_detect_regions_and_detect_frames(fc, shipped):
    frames = frames_of(5, 128, 128, 61)
    reg = np.array([(f, 0, 0, 128) for f in range(5)], np.int32)
    for logits in (False, True):
        got = shipped.scan_frames(frames, 64, logits=logits)
        assert_same(got, shipped.detect_regions(frames, reg, logits=logits), logits)
    assert_same(shipped.scan_frames(frames, 8), shipped.detect_frames(frames))


# ---- input types and paths ----------------------------------------------------------------------------------------------------

def test_host_and_device_paths(fc, shipped):
    import torch
    one = frames_of(1, 480, 640, 71)                                    # latency path
    many = np.ascontiguousarray(frames_of(60, 480, 640, 72))            # 60 VGA frames = 4 staging chunks of 18
    pinned = fc.alloc_host(many.shape)
    pinned[:] = many
    for frames, strides in ((one, (8, 64)), (many, (64, 16)), (pinned, (24,))):
        t = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
        for stride in strides:
            want = reference(fc, shipped, np.asarray(frames), stride)
            assert_same(shipped.scan_frames(frames, stride), want, ("host", len(frames), stride))
            got = shipped.scan_frames(t, stride)
            assert all(g.is_cuda for g in got)
            assert_same(_np(got), want, ("device", len(frames), stride))


def test_4k_frame(fc, shipped):
    """2160x3840 (24.9 MB, staged alone): stride 64 against the reference, stride 8 (118 575 windows) host against device."""
    import torch
    frames = frames_of(1, 2160, 3840, 81)
    t = torch.from_numpy(frames).cuda()
    want = reference(fc, shipped, frames, 64)
    assert_same(shipped.scan_frames(frames, 64), want)
    assert_same(_np(shipped.scan_frames(t, 64)), want)
    host = shipped.scan_frames(frames, 8)
    assert len(host[0]) == 118575
    assert_same(_np(shipped.scan_frames(t, 8)), host)


# ---- merging ---------------------------------------------------------------------------------------------------------------

def test_scan_objects_equals_merge_of_scan_frames(fc, shipped):
    import torch
    runs = 0
    for n, fh, fw, stride in ((3, 480, 640, 64), (3, 480, 640, 16), (2, 480, 640, 8), (4, 144, 272, 8)):
        frames = frames_of(n, fh, fw, 90 + stride)
        t = torch.from_numpy(frames).cuda()
        reg = fc.grid_regions(n, fh, fw, 128, stride)
        for logits in (False, True):
            cls, probs, box = shipped.scan_frames(frames, stride, logits=logits)
            scores = probs[np.arange(len(cls)), cls]
            for score_min, agnostic, max_det, iou_max in ((-np.inf if logits else 0.0, False, 100, 0.5),
                                                          (float(np.percentile(scores, 97)), False, 1024, 0.3),
                                                          (float(np.median(scores)), True, 1, 0.5),
                                                          (float(np.median(scores)), True, 1024, 0.1)):
                kw = dict(score_min=score_min, iou_max=iou_max, max_det=max_det, class_agnostic=agnostic)
                want = shipped.merge_regions(reg, cls, scores, box, n, **kw)
                what = (n, fh, fw, stride, logits, score_min, agnostic, max_det)
                assert_same(shipped.scan_objects(frames, stride, logits=logits, **kw), want, what + ("host",))
                got = shipped.scan_objects(t, stride, logits=logits, **kw)
                assert all(g.is_cuda for g in got)
                assert_same(_np(got), want, what + ("device",))
                runs += 1
    assert runs == 32


# ---- refusals ----------------------------------------------------------------------------------------------------------------

def _vp(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def test_refusals_launch_nothing(fc, shipped, shipped_weights):
    L = fc._lib
    acc = shipped
    buf = np.zeros((2, 2160, 3840, 3), np.uint8)
    probs, cls, box = np.zeros((300000, 6), np.float32), np.zeros(300000, np.int32), np.zeros((300000, 4), np.int32)
    dets = [np.zeros(2, np.int32), np.zeros((2, 1024), np.int32), np.zeros((2, 1024), np.int32), np.zeros((2, 1024), np.float32),
            np.zeros((2, 1024, 4), np.float32)]

    def scan(n=1, fh=480, fw=640, stride=64, flags=0):
        return acc._libc.cnnacc_scan_frames(acc._h, _vp(buf), n, fh, fw, stride, _vp(probs), _vp(cls), _vp(box), flags)

    def objects(n=1, fh=480, fw=640, stride=64, flags=0, iou_max=0.5, max_det=10, outs=dets):
        return acc._libc.cnnacc_scan_objects(acc._h, _vp(buf), n, fh, fw, stride, 0.0, iou_max, max_det, *[_vp(a) for a in outs],
                                             flags)
    n0 = acc.launch_count
    bad = [dict(n=-1), dict(fh=1080, fw=1920), dict(fh=112, fw=640), dict(fh=480, fw=8208), dict(fh=136), dict(fw=200),
           dict(stride=0), dict(stride=7), dict(stride=12), dict(stride=-8)]
    bad += [dict(flags=f) for f in (L.FLAG_BBOX_UPSAMPLED, L.FLAG_RECTS, L.FLAG_DIRECT, L.FLAG_KEEP_MAPS, L.FLAG_TWO_KERNELS)]
    for kw in bad:
        assert scan(**kw) == L.ERR_ARG, kw
        assert objects(**kw) == L.ERR_ARG, kw
    assert objects(fh=2160, fw=3840, stride=8) == L.ERR_ARG                 # 118 575 windows per frame
    for kw in (dict(max_det=0), dict(max_det=1025), dict(iou_max=float("nan")), dict(iou_max=1.5), dict(outs=[None] + dets[1:])):
        assert objects(**kw) == L.ERR_ARG, kw
    assert scan(n=0) == L.OK and objects(n=0) == L.OK
    for stride in (0, 7, 12):
        with pytest.raises(ValueError):
            acc.scan_frames(buf[:1, :480, :640], stride)
    with pytest.raises(ValueError):
        acc.scan_frames(np.zeros((1, 1080, 1920, 3), np.uint8))
    with pytest.raises(ValueError):
        acc.scan_objects(buf[:1], 8)
    assert acc.launch_count == n0
    bare = fc.CNNAccelerator()                                          # no weights, then no classifier: -4
    try:
        for _ in range(2):
            assert bare._libc.cnnacc_scan_frames(bare._h, _vp(buf), 1, 480, 640, 64, _vp(probs), _vp(cls), _vp(box), 0) == L.ERR_STATE
            assert bare._libc.cnnacc_scan_objects(bare._h, _vp(buf), 1, 480, 640, 64, 0.0, 0.5, 10, *[_vp(a) for a in dets], 0) == \
                L.ERR_STATE
            bare.load_weights(shipped_weights)
        assert bare.launch_count == 0
    finally:
        bare.close()


# ---- resources -----------------------------------------------------------------------------------------------------------------

def test_repeated_calls_hold_device_memory(fc, shipped):
    import torch
    sets = [frames_of(8, 480, 640, 101), frames_of(2, 720, 1280, 102)]
    tensors = [torch.from_numpy(f).cuda() for f in sets]

    def cycle():
        out = []
        for f, t in zip(sets, tensors):
            out.append(shipped.scan_frames(f, 16))
            out.append(_np(shipped.scan_frames(t, 16)))
            out.append(shipped.scan_objects(f, 64, score_min=0.2))
            out.append(_np(shipped.scan_objects(t, 64, score_min=0.2)))
        torch.cuda.synchronize()
        return out
    first = cycle()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(3):
        again = cycle()
    assert free0 - torch.cuda.mem_get_info()[0] < (64 << 20)
    for a, b in zip(first, again):
        assert_same(a, b)
