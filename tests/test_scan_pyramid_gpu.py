"""The pyramid calls on the GPU (cnnacc_preprocess_pyramid / cnnacc_scan_pyramid / cnnacc_scan_pyramid_objects): level gray
equal to cv2 (tests/golden/pyramid_cases.npz) and to the numpy restatement; every window's predictions equal classify_batch
on that window cut out of run_batch's feature map of the level's gray, bit for bit, on the shipped weights and the exposed
ternary workloads at both accumulator widths; a single identity level equal to scan_frames; scan_pyramid_objects against
merge_regions on the windows' frame rectangles; host arrays against CUDA tensors; refusals that launch nothing; bounded
device memory over repeated calls."""
import ctypes
import os
import sys

import numpy as np
import pytest

import inputs
import pyramid_oracle
import scan_oracle
from test_detect_objects_cpu import assert_same

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_pyramid_golden as golden  # noqa: E402

pytestmark = pytest.mark.gpu

TERNARY = [w for w in inputs.EXPOSED_WORKLOADS if w["name"].startswith("tern")]
CONFIGS = [("shipped", "shipped", (7, 10, 11), bits) for bits in (32, 24)] + \
          [(w["name"], w["weights"], w["shifts"], bits) for w in TERNARY for bits in (32, 24)]
LOGIT_RTOL = 1e-5
PROB_ATOL = 1e-5
VGA = [(640, 480), (512, 384), (320, 240), (256, 192)]
P720 = [(1280, 720), (1024, 576), (512, 288), (256, 144)]
P1080 = [(1536, 864), (1280, 720), (1024, 576), (768, 432), (512, 288), (256, 144)]
# (fh, fw, levels, stride): VGA, 720p, 1080p, 1000x750 at stride 16, anisotropic levels
SCANS = [(480, 640, VGA, 16), (720, 1280, P720, 32), (1080, 1920, P1080, 64), (750, 1000, [(640, 480), (320, 240)], 16),
         (480, 640, [(640, 240), (320, 480), (128, 128)], 24)]


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
    return inputs.make_frames(("rng" if seed % 2 else "smooth", seed), n, fh, fw)


def level_slices(gray, levels):
    """[F][sum h*w] -> per level [F][h][w]."""
    out, o = [], 0
    for w, h in levels:
        out.append(gray[:, o:o + w * h].reshape(-1, h, w))
        o += w * h
    return out


def reference(fc, acc, frames, levels, stride, logits=False):
    """classify_batch(run_batch(level gray)[window slices]) over all windows in window order -> (cls, probs, bbox)."""
    n = len(frames)
    per_level = []
    for (w, h), g in zip(levels, level_slices(np.asarray(acc.preprocess_pyramid(frames, levels)), levels)):
        maps = acc.run_batch(np.ascontiguousarray(g))
        wm = scan_oracle.window_maps(maps, scan_oracle.windows(n, h, w, stride))
        per_level.append(tuple(np.asarray(a) for a in acc.classify_batch(np.ascontiguousarray(wm), logits=logits)))
    counts = [len(scan_oracle.origins(h, stride)) * len(scan_oracle.origins(w, stride)) for w, h in levels]
    out = []
    for k in range(3):                                  # reorder level-major -> frame-major, then level
        parts = [p[k].reshape((n, c) + p[k].shape[1:]) for p, c in zip(per_level, counts)]
        out.append(np.concatenate(parts, axis=1).reshape((-1,) + per_level[0][k].shape[1:]))
    return tuple(out)


# ---- level gray -----------------------------------------------------------------------------------------------------------------

def test_preprocess_pyramid_equals_golden_and_restatement(fc, shipped):
    import torch
    gold = np.load(os.path.join(HERE, "golden", "pyramid_cases.npz"))
    for c in golden.cases():
        frame = golden.make_frame(c)[None]
        got = shipped.preprocess_pyramid(frame, [(c["w"], c["h"])])[0].reshape(c["h"], c["w"])
        want = gold[c["name"]]
        if want.dtype.kind == "U":
            assert golden.digest(got) == str(want), c["name"]
        else:
            assert np.array_equal(got, want), c["name"]
        dev = shipped.preprocess_pyramid(torch.from_numpy(frame).cuda(), [(c["w"], c["h"])])
        assert dev.is_cuda and np.array_equal(dev.cpu().numpy()[0].reshape(c["h"], c["w"]), got), c["name"]
    for fh, fw, levels, _ in SCANS:                      # several levels in one call, odd frame count
        frames = frames_of(3, fh, fw, 5)
        assert np.array_equal(shipped.preprocess_pyramid(frames, levels), pyramid_oracle.preprocess(frames, levels)), (fh, fw)
    odd = frames_of(1, 131, 257, 7)                     # n * fh * fw not a multiple of 4: the gray kernel's tail
    assert np.array_equal(shipped.preprocess_pyramid(odd, [(256, 128), (128, 128)]),
                          pyramid_oracle.preprocess(odd, [(256, 128), (128, 128)]))


# ---- classify equality ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("fh,fw,levels,stride", SCANS, ids=[f"{s[0]}x{s[1]}_{len(s[2])}_{s[3]}" for s in SCANS])
@pytest.mark.parametrize("name,weights,shifts,bits", CONFIGS, ids=[f"{c[0]}-{c[3]}" for c in CONFIGS])
def test_scan_pyramid_equals_classify_of_level_windows(fc, acc, shipped_weights, name, weights, shifts, bits, fh, fw, levels,
                                                       stride):
    configure(acc, shipped_weights, weights, shifts, bits)
    frames = frames_of(2 if fh * fw <= 720 * 1280 else 1, fh, fw, 40 + len(name) + bits)
    for logits in (False, True):
        want = reference(fc, acc, frames, levels, stride, logits)
        assert_same(acc.scan_pyramid(frames, levels, stride, logits=logits), want, (stride, logits))
        assert len(want[0]) == len(fc.pyramid_windows(len(frames), fh, fw, levels, stride))


def test_identity_level_is_scan_frames(fc, shipped):
    for fh, fw, stride in ((480, 640, 8), (144, 272, 24), (720, 1280, 64)):
        frames = frames_of(2, fh, fw, 21)
        for logits in (False, True):
            assert_same(shipped.scan_pyramid(frames, [(fw, fh)], stride, logits=logits), shipped.scan_frames(frames, stride, logits=logits))
        assert_same(shipped.scan_pyramid_objects(frames, [(fw, fh)], stride, score_min=0.2),
                    shipped.scan_objects(frames, stride, score_min=0.2))


def test_scan_pyramid_against_restatement(fc, acc, shipped_weights):
    """End to end against the numpy restatement (a supplement to the bit-exact classify_batch comparison above): a window's
    class may differ only where its top two logits tie within LOGIT_RTOL; elsewhere box and probabilities agree."""
    w = TERNARY[0]
    configure(acc, shipped_weights, w["weights"], w["shifts"], 32)
    fw_, fb = inputs.make_fc()
    frames = frames_of(1, 300, 640, 3)
    levels = [(512, 240), (320, 240), (256, 128)]
    cls_r, prob_r, logit_r, box_r = pyramid_oracle.scan(frames, levels, inputs.make_weights(w["weights"]), w["shifts"], fw_, fb, 32)
    cls, probs, box = acc.scan_pyramid(frames, levels, 32)
    assert len(cls) == len(cls_r) == len(fc.pyramid_windows(1, 300, 640, levels, 32))
    checked = 0
    for i in range(len(cls)):
        scale = np.abs(logit_r[i]).max()
        if cls[i] != cls_r[i]:
            top2 = np.sort(logit_r[i])[-2:]
            assert top2[1] - top2[0] <= LOGIT_RTOL * scale, i
            continue
        assert np.abs(probs[i] - prob_r[i]).max() <= PROB_ATOL, i
        assert tuple(box[i]) == tuple(box_r[i]), i
        checked += 1
    assert checked > 0.99 * len(cls)


# ---- merging ---------------------------------------------------------------------------------------------------------------------

def test_scan_pyramid_objects_equals_merge_regions(fc, shipped):
    import torch
    runs = 0
    for n, fh, fw, levels, stride in ((2, 480, 640, VGA, 16), (1, 1080, 1920, P1080, 16), (3, 480, 640, [(640, 240), (320, 480)], 32)):
        frames = frames_of(n, fh, fw, 90 + stride)
        t = torch.from_numpy(frames).cuda()
        reg = fc.pyramid_windows(n, fh, fw, levels, stride)
        for logits in (False, True):
            cls, probs, box = shipped.scan_pyramid(frames, levels, stride, logits=logits)
            scores = probs[np.arange(len(cls)), cls]
            for score_min, agnostic, max_det, iou_max in ((-np.inf if logits else 0.0, False, 100, 0.5),
                                                          (float(np.percentile(scores, 97)), False, 1024, 0.3),
                                                          (float(np.median(scores)), True, 1024, 0.1)):
                kw = dict(score_min=score_min, iou_max=iou_max, max_det=max_det, class_agnostic=agnostic)
                want = shipped.merge_regions(reg, cls, scores, box, n, **kw)
                what = (n, fh, fw, stride, logits, score_min, agnostic, max_det)
                assert_same(shipped.scan_pyramid_objects(frames, levels, stride, logits=logits, **kw), want, what + ("host",))
                got = shipped.scan_pyramid_objects(t, levels, stride, logits=logits, **kw)
                assert all(g.is_cuda for g in got)
                assert_same(_np(got), want, what + ("device",))
                runs += 1
    assert runs == 18


# ---- input types and paths ------------------------------------------------------------------------------------------------------

def test_host_and_device_paths(fc, shipped):
    import torch
    one = frames_of(1, 480, 640, 71)                                    # latency path
    many = np.ascontiguousarray(frames_of(40, 480, 640, 72))            # several 16 MiB staging chunks
    big = frames_of(1, 2160, 3840, 73)                                  # 4K: staged alone
    for frames, levels, stride in ((one, VGA, 8), (many, VGA, 32), (big, [(2560, 1440), (1280, 720)], 64)):
        t = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
        host = shipped.scan_pyramid(frames, levels, stride)
        got = shipped.scan_pyramid(t, levels, stride)
        assert all(g.is_cuda for g in got)
        assert_same(_np(got), host, (len(frames), stride))
        g_host = shipped.preprocess_pyramid(frames, levels)
        assert np.array_equal(shipped.preprocess_pyramid(t, levels).cpu().numpy(), g_host)
    want = reference(fc, shipped, many[:3], VGA, 32)
    n3 = len(want[0])
    assert_same(tuple(a[:n3] for a in shipped.scan_pyramid(many, VGA, 32)), want)


def test_frames_of_more_than_a_prediction_block(fc, shipped):
    """A pyramid frame may have more windows than a host-pointer prediction block (2^20): 8192x8192 frames with the levels
    8192x8192 and 4096x4096 at stride 8 have 1 265 090 windows each.  The host path then takes one frame per block; its
    predictions equal the device path's, which runs one frame per piece, for one frame (the latency path) and for two (one
    block each)."""
    import torch
    levels = [(8192, 8192), (4096, 4096)]
    per = len(fc.pyramid_windows(1, 8192, 8192, levels, 8))
    assert per == 1265090 > 1 << 20
    frames = np.random.default_rng(11).integers(0, 256, (2, 8192, 8192, 3), dtype=np.uint8)
    for n in (1, 2):
        host = shipped.scan_pyramid(frames[:n], levels, 8)
        assert len(host[0]) == n * per
        dev = _np(shipped.scan_pyramid(torch.from_numpy(frames[:n]).cuda(), levels, 8))
        assert_same(host, dev, n)
    # the last level's windows against classify_batch on its map (a slice, to keep the reference small)
    g = shipped.preprocess_pyramid(frames[1:], [(4096, 4096)]).reshape(1, 4096, 4096)
    maps = shipped.run_batch(g)
    wins = scan_oracle.windows(1, 4096, 4096, 8)[:20000]
    want = shipped.classify_batch(np.ascontiguousarray(scan_oracle.window_maps(maps, wins)))
    first = per + (per - len(scan_oracle.windows(1, 4096, 4096, 8)))      # frame 1, level 1
    assert_same(tuple(a[first:first + len(wins)] for a in host), want)


# ---- refusals ------------------------------------------------------------------------------------------------------------------

def _vp(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def test_refusals_launch_nothing(fc, shipped, shipped_weights):
    L = fc._lib
    acc = shipped
    buf = np.zeros((2, 2160, 3840, 3), np.uint8)
    probs, cls, box = np.zeros((300000, 6), np.float32), np.zeros(300000, np.int32), np.zeros((300000, 4), np.int32)
    gray = np.zeros(2 * 2160 * 3840 * 2, np.uint8)
    dets = [np.zeros(2, np.int32), np.zeros((2, 1024), np.int32), np.zeros((2, 1024), np.int32), np.zeros((2, 1024), np.float32),
            np.zeros((2, 1024, 4), np.float32)]

    def lv(levels):
        return np.ascontiguousarray(np.asarray(levels, np.int32).reshape(-1, 2))

    def scan(n=1, fh=480, fw=640, levels=VGA, stride=16, flags=0):
        a = lv(levels)
        return acc._libc.cnnacc_scan_pyramid(acc._h, _vp(buf), n, fh, fw, _vp(a) if len(a) else None, len(a), stride, _vp(probs),
                                             _vp(cls), _vp(box), flags)

    def objects(n=1, fh=480, fw=640, levels=VGA, stride=16, flags=0, iou_max=0.5, max_det=10, outs=dets):
        a = lv(levels)
        return acc._libc.cnnacc_scan_pyramid_objects(acc._h, _vp(buf), n, fh, fw, _vp(a) if len(a) else None, len(a), stride, 0.0,
                                                     iou_max, max_det, *[_vp(o) for o in outs], flags)

    def prep(n=1, fh=480, fw=640, levels=VGA, flags=0):
        a = lv(levels)
        return acc._libc.cnnacc_preprocess_pyramid(acc._h, _vp(buf), n, fh, fw, _vp(a) if len(a) else None, len(a), _vp(gray), flags)

    n0 = acc.launch_count
    level_bad = [dict(fh=127), dict(fw=8193), dict(levels=[]), dict(levels=[(128, 128)] * 17), dict(levels=[(520, 384)]),
                 dict(levels=[(512, 388)]), dict(levels=[(112, 240)]), dict(levels=[(656, 480)]), dict(levels=[(640, 496)])]
    scan_bad = level_bad + [dict(n=-1), dict(levels=[(448, 336)]), dict(fh=720, fw=1280, levels=[(768, 432)], stride=8),
                            dict(stride=0), dict(stride=7), dict(stride=12), dict(stride=-8)]
    scan_bad += [dict(flags=f) for f in (L.FLAG_BBOX_UPSAMPLED, L.FLAG_RECTS, L.FLAG_DIRECT, L.FLAG_KEEP_MAPS, L.FLAG_TWO_KERNELS)]
    for kw in scan_bad:
        assert scan(**kw) == L.ERR_ARG, kw
        assert objects(**kw) == L.ERR_ARG, kw
    for kw in level_bad + [dict(n=-1), dict(flags=L.FLAG_RECTS)]:
        assert prep(**kw) == L.ERR_ARG, kw
    assert objects(fh=1080, fw=1920, levels=P1080, stride=8) == L.ERR_ARG            # 38 016 windows per frame
    assert scan(fh=1080, fw=1920, levels=P1080, stride=8, n=0) == L.OK
    for kw in (dict(max_det=0), dict(max_det=1025), dict(iou_max=float("nan")), dict(outs=[None] + dets[1:])):
        assert objects(**kw) == L.ERR_ARG, kw
    a = lv(VGA)
    assert acc._libc.cnnacc_scan_pyramid(acc._h, None, 1, 480, 640, _vp(a), 4, 16, _vp(probs), _vp(cls), _vp(box), 0) == L.ERR_ARG
    assert scan(n=0) == L.OK and objects(n=0) == L.OK and prep(n=0) == L.OK
    with pytest.raises(ValueError):
        acc.scan_pyramid(buf[:1, :480, :640], [(448, 336)], 16)
    with pytest.raises(ValueError):
        acc.scan_pyramid_objects(buf[:1, :1080, :1920], P1080, 8)
    assert acc.launch_count == n0
    bare = fc.CNNAccelerator()                                          # no weights, then no classifier: -4
    try:
        for _ in range(2):
            assert bare._libc.cnnacc_scan_pyramid(bare._h, _vp(buf), 1, 480, 640, _vp(a), 4, 16, _vp(probs), _vp(cls), _vp(box),
                                                  0) == L.ERR_STATE
            assert bare._libc.cnnacc_scan_pyramid_objects(bare._h, _vp(buf), 1, 480, 640, _vp(a), 4, 16, 0.0, 0.5, 10,
                                                          *[_vp(o) for o in dets], 0) == L.ERR_STATE
            bare.load_weights(shipped_weights)
        assert bare.launch_count == 0
    finally:
        bare.close()


# ---- resources -----------------------------------------------------------------------------------------------------------------

def test_repeated_calls_hold_device_memory(fc, shipped):
    import torch
    sets = [(frames_of(8, 480, 640, 101), VGA), (frames_of(2, 1080, 1920, 102), P1080)]
    tensors = [torch.from_numpy(f).cuda() for f, _ in sets]

    def cycle():
        out = []
        for (f, levels), t in zip(sets, tensors):
            out.append(shipped.scan_pyramid(f, levels, 16))
            out.append(_np(shipped.scan_pyramid(t, levels, 16)))
            out.append(shipped.scan_pyramid_objects(f, levels, 16, score_min=0.2))
            out.append(_np(shipped.scan_pyramid_objects(t, levels, 16, score_min=0.2)))
            out.append((shipped.preprocess_pyramid(f, levels),))
        torch.cuda.synchronize()
        return out
    first = cycle()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(3):
        again = cycle()
    assert free0 - torch.cuda.mem_get_info()[0] < (64 << 20)
    for a, b in zip(first, again):
        for x, y in zip(a, b):
            assert np.array_equal(np.asarray(x), np.asarray(y))
