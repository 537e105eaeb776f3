"""The merge of region detections on the GPU (csrc/region_merge.cuh, cnnacc_detect_objects / cnnacc_merge_regions): every
output equals the numpy restatement of tests/test_detect_objects_cpu.py exactly, for merge_regions on the CPU cases and for
detect_objects against the restatement applied to detect_regions' own outputs, across the internal chunk edges of both the
device-pointer and the host-pointer paths."""
import ctypes

import numpy as np
import pytest

import inputs
from test_detect_objects_cpu import CASES, REFUSAL_OK, REFUSALS, assert_same, restate
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
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _cpu(x):
    return tuple(t.cpu().numpy() if hasattr(t, "cpu") else t for t in x)


def merge_args(c):
    return dict(score_min=c["score_min"], iou_max=c["iou_max"], max_det=c["max_det"], class_agnostic=c["agnostic"])


@pytest.mark.parametrize("name", sorted(CASES))
def test_merge_regions_equals_restatement(fc, acc, name):
    import torch
    c = CASES[name]
    want = restate(**c)
    got = acc.merge_regions(c["regions"], c["cls"], c["scores"], c["bbox"], c["n_frames"], **merge_args(c))
    assert_same(got, want, (name, "host"))
    t = [torch.from_numpy(np.ascontiguousarray(c[k])).cuda() for k in ("cls", "scores", "bbox")]
    got = acc.merge_regions(c["regions"], *t, c["n_frames"], **merge_args(c))
    assert all(g.is_cuda for g in got)
    assert_same(_cpu(got), want, (name, "device"))


def expected(acc, frames, reg, bbox="vec", logits=False, score_min=0.0, iou_max=0.5, max_det=100, agnostic=False):
    """The restatement applied to detect_regions' own outputs, in the caller's region order."""
    cls, probs, box = _cpu(acc.detect_regions(frames, reg, bbox=bbox, logits=logits))
    scores = probs[np.arange(len(cls)), cls]
    return restate(reg, scores, cls, box, len(frames), score_min, iou_max, max_det, agnostic), scores


def test_detect_objects_equals_restatement_of_detect_regions(fc, acc):
    import torch
    frames = inputs.make_frames(("smooth", 700), 5, 480, 640)
    frames[3] = inputs.make_frames(("rng", 701), 1, 480, 640)[0]
    grid = fc.grid_regions(5, 480, 640, 128, 64)
    pyr = fc.grid_regions(5, 480, 640, [480, 240, 128], [240, 120, 64])
    grid, pyr = grid[grid[:, 0] != 1], pyr[pyr[:, 0] != 4]            # frames without regions
    t = torch.from_numpy(frames).cuda()
    rng = np.random.default_rng(9)
    runs, empties = 0, []
    for reg in (grid, pyr, np.concatenate([grid, pyr])[rng.permutation(len(grid) + len(pyr))]):
        for bbox, logits, agnostic, iou_max, max_det in (("vec", False, False, 0.5, 100), ("upsampled", False, True, 0.3, 5),
                                                         ("vec", True, False, 0.1, 1024), ("upsampled", True, True, 0.7, 40)):
            cls, probs, box = acc.detect_regions(frames, reg, bbox=bbox, logits=logits)
            scores = probs[np.arange(len(cls)), cls]
            score_min = float(np.median(scores))                      # about half the regions are candidates
            want = restate(reg, scores, cls, box, len(frames), score_min, iou_max, max_det, agnostic)
            kw = dict(score_min=score_min, iou_max=iou_max, max_det=max_det, class_agnostic=agnostic, bbox=bbox, logits=logits)
            assert_same(acc.detect_objects(frames, reg, **kw), want, (len(reg), bbox, logits, "host"))
            got = acc.detect_objects(t, reg, **kw)
            assert all(g.is_cuda for g in got)
            assert_same(_cpu(got), want, (len(reg), bbox, logits, "device"))
            empty = sorted(set(range(len(frames))) - set(reg[:, 0].tolist()))   # grid: frame 1, pyramid: frame 4, mixed: none
            assert (want[0][empty] == 0).all() and (want[0] > 0).sum() >= 3
            empties.append(empty)
            runs += 1
    assert runs == 12 and empties[0] == [1] and empties[4] == [4]


def test_device_path_frame_across_chunk_edge(fc, acc):
    """3 frames x 10 000 regions: the device path runs 16384 regions per piece, so its pieces must end at frame edges."""
    import torch
    rng = np.random.default_rng(12)
    frames = inputs.make_frames(("smooth", 800), 3, 480, 640)
    side = rng.choice([128, 160, 200], 30000)
    reg = np.stack([np.repeat(np.arange(3), 10000), rng.integers(0, 641 - side), rng.integers(0, 481 - side), side], 1).astype(np.int32)
    want, _ = expected(acc, frames, reg, max_det=300, iou_max=0.4)
    got = acc.detect_objects(torch.from_numpy(frames).cuda(), reg, max_det=300, iou_max=0.4)
    assert_same(_cpu(got), want)


def test_host_path_frame_across_prediction_block(fc, acc):
    """About 1.06 M regions (128-side stride-4 grid, 11 481 per VGA frame, 92 frames): frame 91 straddles region 2^20, where
    the host path of detect_regions ends a prediction block; detect_objects ends its blocks at frame edges instead."""
    host = fc.alloc_host((92, 480, 640, 3))
    host[:] = inputs.make_frames(("smooth", 900), 92, 480, 640)
    reg = fc.grid_regions(92, 480, 640, 128, 4)
    per = len(reg) // 92
    assert per == 11481 and 91 * per < 2 ** 20 < 92 * per
    cls, probs, box = acc.detect_regions(host, reg)
    scores = probs[np.arange(len(cls)), cls]
    score_min = float(np.median(scores))                              # about half the regions are candidates
    kw = dict(score_min=score_min, iou_max=0.5, max_det=100)
    got = acc.detect_objects(host, reg, **kw)
    alone = acc.detect_objects(host[91:92], reg[reg[:, 0] == 91] - [91, 0, 0, 0], **kw)
    alone = (alone[0], np.where(alone[1] >= 0, alone[1] + 91 * per, -1).astype(np.int32)) + alone[2:]
    assert_same([a[91:92] for a in got], alone)
    for f in (0, 90, 91):
        sel = slice(f * per, (f + 1) * per)
        want = restate(reg[sel] - [f, 0, 0, 0], scores[sel], cls[sel], box[sel], 1, score_min, 0.5, 100, False)
        want = (want[0], np.where(want[1] >= 0, want[1] + f * per, -1).astype(np.int32)) + want[2:]
        assert_same([a[f:f + 1] for a in got], want, f)
    assert got[0][91] > 0 and got[0].sum() > 0


def test_queued_device_calls(fc, acc):
    import torch
    frames = inputs.make_frames(("smooth", 1000), 4, 480, 640)
    regs = [fc.grid_regions(4, 480, 640, 128, 64)[::3], fc.grid_regions(4, 480, 640, [240, 333], [120, 100]),
            np.array([(3, 0, 0, 480), (0, 1, 2, 129)], np.int32)]
    regs += [r[np.random.default_rng(i).permutation(len(r))] for i, r in enumerate(regs)]
    want = [acc.detect_objects(frames, r, bbox="upsampled", iou_max=0.2, max_det=7) for r in regs]
    c = CASES["random_2"]
    want_m = restate(**c)
    t = torch.from_numpy(frames).cuda()
    tm = [torch.from_numpy(np.ascontiguousarray(c[k])).cuda() for k in ("cls", "scores", "bbox")]
    torch.cuda.synchronize()
    torch.cuda._sleep(100_000_000)          # keep the stream busy: every call below is queued before any of them runs
    got = []
    for r in regs:
        got.append(acc.detect_objects(t, r, bbox="upsampled", iou_max=0.2, max_det=7))
        got.append(acc.merge_regions(c["regions"], *tm, c["n_frames"], **merge_args(c)))
    torch.cuda.synchronize()
    for k, w in enumerate(want):
        assert_same(_cpu(got[2 * k]), w, k)
        assert_same(_cpu(got[2 * k + 1]), want_m, k)


def _det_buffers(n_frames, max_det):
    return (np.zeros(n_frames, np.int32), np.zeros((n_frames, max_det), np.int32), np.zeros((n_frames, max_det), np.int32),
            np.zeros((n_frames, max_det), np.float32), np.zeros((n_frames, max_det, 4), np.float32))


def test_refusals_launch_nothing(fc, acc, shipped_weights):
    import torch
    frames = np.zeros((3, 480, 640, 3), np.uint8)
    out = _det_buffers(3, 1024)

    def detect(reg, iou_max=0.5, max_det=10, outs=out, flags=0, frames_p=_vp(frames)):
        reg = np.ascontiguousarray(reg, np.int32)
        return acc._libc.cnnacc_detect_objects(acc._h, frames_p, 3, 480, 640, _vp(reg), len(reg), 0.0, iou_max, max_det,
                                               *[_vp(a) if isinstance(a, np.ndarray) else a for a in outs], flags)
    n0 = acc.launch_count
    for name, bad in sorted(BAD_REGIONS.items()):                     # what detect_regions refuses
        assert detect(bad) == fc._lib.ERR_ARG, name
    ok = [(0, 0, 0, 128), (2, 5, 5, 200)]
    for kw in (dict(max_det=0), dict(max_det=1025), dict(iou_max=float("nan")), dict(iou_max=-0.1), dict(iou_max=1.5)):
        assert detect(ok, **kw) == fc._lib.ERR_ARG, kw
    assert detect(ok, outs=(None,) + out[1:]) == fc._lib.ERR_ARG          # n_det is required
    assert detect(np.tile([1, 0, 0, 128], (16385, 1))) == fc._lib.ERR_ARG
    with pytest.raises(ValueError):
        acc.detect_objects(frames, ok, max_det=0)
    with pytest.raises(ValueError):
        acc.detect_objects(frames, ok, iou_max=2.0)
    for name, bad in sorted(REFUSALS.items()):                        # what merge_regions refuses
        c = {**REFUSAL_OK, **bad}
        reg = np.ascontiguousarray(c["regions"], np.int32)
        sc, cl, bb = [np.ascontiguousarray(c[k], dt) for k, dt in (("scores", np.float32), ("cls", np.int32), ("bbox", np.int32))]
        o = _det_buffers(c["n_frames"], 1024)
        rc = acc._libc.cnnacc_merge_regions(acc._h, _vp(reg), len(reg), c["n_frames"], _vp(sc), _vp(cl), _vp(bb), 0.0, c["iou_max"],
                                            c["max_det"], *[_vp(a) for a in o], 0)
        assert rc == fc._lib.ERR_ARG, name
    # misaligned device pointers
    t = torch.from_numpy(frames).cuda()
    dev = [torch.zeros(3 * 1024 * 4 + 4, dtype=torch.float32, device="cuda") for _ in range(5)]
    p = lambda x, off=0: ctypes.c_void_p(x.data_ptr() + off)
    outs = [p(d) for d in dev]
    assert detect(ok, outs=outs[:4] + [p(dev[4], 4)], flags=fc._lib.FLAG_DEVICE_PTRS, frames_p=p(t)) == fc._lib.ERR_ARG
    assert detect(ok, outs=[p(dev[0], 2)] + outs[1:], flags=fc._lib.FLAG_DEVICE_PTRS, frames_p=p(t)) == fc._lib.ERR_ARG
    assert acc.launch_count == n0
    bare = fc.CNNAccelerator()                                         # no weights, then no classifier: -4
    try:
        reg = np.array(ok, np.int32)
        args = (_vp(frames), 3, 480, 640, _vp(reg), 2, 0.0, 0.5, 10, *[_vp(a) for a in out], 0)
        assert bare._libc.cnnacc_detect_objects(bare._h, *args) == fc._lib.ERR_STATE
        bare.load_weights(shipped_weights)
        assert bare._libc.cnnacc_detect_objects(bare._h, *args) == fc._lib.ERR_STATE
        assert bare.launch_count == 0
        # the merge alone needs neither
        c = CASES["duplicates"]
        assert_same(bare.merge_regions(c["regions"], c["cls"], c["scores"], c["bbox"], c["n_frames"]), restate(**c))
    finally:
        bare.close()


def test_no_regions_gives_empty_frames(fc, acc):
    import torch
    frames = inputs.make_frames(("smooth", 1100), 2, 480, 640)
    empty = np.zeros((0, 4), np.int32)
    for f in (frames, torch.from_numpy(frames).cuda()):
        n_det, region, cls, score, box = _cpu(acc.detect_objects(f, empty, max_det=3))
        assert (n_det == 0).all() and (region == -1).all() and (cls == -1).all() and (score == 0).all() and (box == 0).all()
        assert region.shape == (2, 3) and box.shape == (2, 3, 4)
