"""One host batch over several handles (cnnacc_*_sharded / MultiAccelerator): byte-identical to one handle, every shard edge
covered, and the refusals that launch nothing.  Two member sets: two handles on GPU 0 (always; exercises every slicing and
threading path) and every visible GPU (skipped below two)."""
import ctypes

import numpy as np
import pytest

import inputs
import oracle

pytestmark = pytest.mark.gpu

SHIFTS = (7, 10, 11)
CAP = 16


@pytest.fixture(scope="module")
def fc():
    import fpga_cnn_b200 as fc_
    fc_.load()
    return fc_


@pytest.fixture(scope="module", params=["gpu0x2", "all"])
def devices(request):
    import torch
    if request.param == "gpu0x2":
        return [0, 0]
    if torch.cuda.device_count() < 2:
        pytest.skip("fewer than two GPUs visible")
    return list(range(torch.cuda.device_count()))


def _configure(acc, wt, fc_w, fc_b):
    acc.load_weights(wt)
    acc.set_shifts(*SHIFTS)
    acc.load_classifier(fc_w, fc_b)


@pytest.fixture(scope="module")
def multi(fc, devices, shipped_weights):
    m = fc.MultiAccelerator(devices)
    _configure(m, shipped_weights, *inputs.make_fc())
    yield m
    m.close()


@pytest.fixture(scope="module")
def single(fc, shipped_weights):
    a = fc.CNNAccelerator(device=0)
    _configure(a, shipped_weights, *inputs.make_fc())
    yield a
    a.close()


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def _plan(fc, n, k, unit):
    begin = np.zeros(CAP, np.int64)
    m = fc.load().cnnacc_shard_plan_host(n, k, unit, _p(begin), CAP)
    assert m >= 1
    return m, [int(v) for v in begin[:m + 1]]


def _threshold(fc, k, unit):
    """Smallest n that the plan spreads over all k members."""
    lo, hi = 1, 1 << 40
    while lo < hi:
        mid = (lo + hi) // 2
        if _plan(fc, mid, k, unit)[0] >= k:
            hi = mid
        else:
            lo = mid + 1
    return lo


def _counts(m):
    return [a.launch_count for a in m.members]


def _hs(members):
    return (ctypes.c_void_p * len(members))(*[a._h.value for a in members])


def test_run_batch_equals_one_handle_and_the_oracle(fc, multi, single, shipped_weights):
    k = len(multi.members)
    n = max(10_007, _threshold(fc, k, 16384) + 7)
    imgs = inputs.make_images(("rng", 700), n)
    before = _counts(multi)
    got = multi.run_batch(imgs)
    assert all(b > a for a, b in zip(before, _counts(multi))), "every member must have run a shard"
    want = single.run_batch(imgs)
    assert got.shape == want.shape and np.array_equal(got, want)
    m, begin = _plan(fc, n, k, 16384)
    assert m == k
    edges = sorted({i for lo, hi in zip(begin, begin[1:]) for i in (lo, hi - 1)})
    port = oracle.load_port()
    ref = oracle.port_infer_batch(port, imgs[edges], shipped_weights, SHIFTS)
    assert np.array_equal(got.reshape(n, 64, 256)[edges], ref)


@pytest.mark.parametrize("kw", [dict(), dict(bbox="upsampled"), dict(logits=True)], ids=["vec", "upsampled", "logits"])
def test_infer_batch_equals_one_handle(fc, multi, single, kw):
    k = len(multi.members)
    n = max(4099, _threshold(fc, k, 16384) + 3)
    imgs = inputs.make_images(("smooth", 701), n)
    got, want = multi.infer_batch(imgs, **kw), single.infer_batch(imgs, **kw)
    for g, w in zip(got, want):
        assert g.dtype == w.dtype and g.shape == w.shape and np.array_equal(g, w)


def test_detect_frames_equals_one_handle(fc, multi, single):
    k = len(multi.members)
    n = max(150, _threshold(fc, k, 480 * 640 * 3) + 3)          # > 64 frames a shard: the staged ring path, not the small one
    frames = inputs.make_frames(("smooth", 702), n, 480, 640)
    for bbox in ("vec", "upsampled"):
        got, want = multi.detect_frames(frames, bbox=bbox, return_gray=True), single.detect_frames(frames, bbox=bbox, return_gray=True)
        for g, w in zip(got, want):
            assert g.shape == w.shape and np.array_equal(g, w)


def _sharded_infer(fc, multi, imgs, n_cls):
    """The C call straight on sentinel-filled outputs."""
    n = len(imgs)
    probs = np.full((n, n_cls), -1234.5, np.float32)
    cls = np.full(n, -7, np.int32)
    box = np.full((n, 4), -7, np.int32)
    failed = ctypes.c_int(99)
    rc = fc.load().cnnacc_infer_batch_sharded(_hs(multi.members), len(multi.members), _p(imgs), n, _p(probs), _p(cls), _p(box),
                                              0, ctypes.byref(failed))
    assert rc == 0 and failed.value == -1, (rc, failed.value)
    return cls, probs, box


def test_shard_edges(fc, multi, single):
    """n = 0, 1, k-1, k, k+1 and one image either side of the point where a second member joins; sentinel-filled outputs."""
    k = len(multi.members)
    thr = _threshold(fc, 2, 16384)                                   # first n that uses two members
    n_cls = multi.members[0]._n_cls
    for n in sorted({0, 1, max(k - 1, 0), k, k + 1, max(thr - 1, 0), thr}):
        imgs = inputs.make_images(("rng", 710 + n), n)
        before = _counts(multi)
        got = _sharded_infer(fc, multi, imgs, n_cls)
        used = sum(b != a for a, b in zip(before, _counts(multi)))
        assert used == (0 if n == 0 else _plan(fc, n, k, 16384)[0]), (n, used)
        if n == thr - 1:
            assert used == 1
        if n == thr:
            assert used == 2
        want = single.infer_batch(imgs)
        for g, w in zip(got, want):
            assert np.array_equal(g, w), n
        feats = np.full((n, 64, 16, 16), 0xA5, np.uint8)
        multi.run_batch(imgs, out=feats)
        assert np.array_equal(feats, single.run_batch(imgs)), n


@pytest.mark.parametrize("H,W,n_min", [(256, 256, 37), (64, 64, 301)], ids=["256x256_windows", "64x64_per_layer"])
def test_run_batch_other_sizes(fc, multi, single, H, W, n_min):
    k = len(multi.members)
    n = max(n_min, _threshold(fc, k, H * W) + 3)
    imgs = inputs.make_images(("rng", 720 + H), n, H, W)
    got = multi.run_batch(imgs)
    assert got.shape == (n, 64, H // 8, W // 8) and np.array_equal(got, single.run_batch(imgs))


def test_pinned_and_pageable_inputs_agree(fc, multi, single):
    k = len(multi.members)
    n = max(2051, _threshold(fc, k, 16384) + 1)
    pageable = inputs.make_images(("smooth", 730), n)
    pinned = fc.alloc_host(pageable.shape)
    pinned[:] = pageable
    out = fc.alloc_host((n, 64, 16, 16))
    assert np.array_equal(multi.run_batch(pinned, out=out), multi.run_batch(pageable))
    assert np.array_equal(out, single.run_batch(pageable))
    for g, w in zip(multi.infer_batch(pinned), multi.infer_batch(pageable)):
        assert np.array_equal(g, w)


def test_cuda_tensors_go_to_a_member(fc, multi):
    import torch
    x = torch.zeros((4, 128, 128), dtype=torch.uint8, device="cuda:0")
    with pytest.raises(ValueError, match=r"members\[i\]"):
        multi.run_batch(x)
    with pytest.raises(ValueError, match=r"members\[i\]"):
        multi.infer_batch(x)


def test_refusals_launch_nothing(fc, devices, shipped_weights):
    """Argument and configuration errors are found before any member starts: no member launches a kernel."""
    lib = fc.load()
    fc_w, fc_b = inputs.make_fc()
    n = 300
    imgs = inputs.make_images(("rng", 740), n)
    feats = np.zeros((n, 64, 16, 16), np.uint8)
    with fc.MultiAccelerator(devices) as m:
        _configure(m, shipped_weights, fc_w, fc_b)
        k = len(m.members)
        c0 = _counts(m)

        def run(hs, k_, flags=0):
            failed = ctypes.c_int(99)
            rc = lib.cnnacc_run_batch_sharded(hs, k_, _p(imgs), n, 128, 128, _p(feats), flags, ctypes.byref(failed))
            return rc, failed.value

        a0 = m.members[0]
        assert run(_hs([a0, m.members[1], a0]), 3) == (fc._lib.ERR_ARG, 2)              # the same handle twice
        assert "same handle" in lib.cnnacc_last_error(a0._h).decode()
        assert run(_hs(m.members), 0) == (fc._lib.ERR_ARG, -1)
        for flag in (fc._lib.FLAG_DEVICE_PTRS, fc._lib.FLAG_KEEP_MAPS):
            assert run(_hs(m.members), k, flag) == (fc._lib.ERR_ARG, 0)
        assert _counts(m) == c0

        # member 1 configured unlike member 0
        for wrong, right, what in ((lambda: m.members[1].set_shifts(2, 4, 6), lambda: m.members[1].set_shifts(*SHIFTS), "shifts"),
                                   (lambda: m.members[1].set_accumulator_bits(24), lambda: m.members[1].set_accumulator_bits(32), "accumulator"),
                                   (lambda: m.members[1].load_weights(inputs.make_weights(("rng", 7))),
                                    lambda: m.members[1].load_weights(shipped_weights), "weights"),
                                   (lambda: m.members[1].load_classifier(fc_w * 2, fc_b), lambda: m.members[1].load_classifier(fc_w, fc_b),
                                    "classifier")):
            wrong()
            c0 = _counts(m)
            if what != "classifier":                      # run_batch does not use the classifier
                assert run(_hs(m.members), k) == (fc._lib.ERR_ARG, 1)
                with pytest.raises(ValueError, match=f"member 1 .*{what}"):
                    m.run_batch(imgs)
            with pytest.raises(ValueError, match=f"member 1 .*{what}"):
                m.infer_batch(imgs)
            with pytest.raises(ValueError, match=f"member 1 .*{what}"):
                m.detect_frames(np.zeros((3, 480, 640, 3), np.uint8))
            assert _counts(m) == c0, what
            right()
        assert np.array_equal(m.run_batch(imgs), m.members[0].run_batch(imgs))

    # member 1 without a classifier: the prediction calls refuse with -4, run_batch still runs
    with fc.MultiAccelerator(devices) as m:
        m.load_weights(shipped_weights)
        m.members[0].load_classifier(fc_w, fc_b)
        c0 = _counts(m)
        with pytest.raises(RuntimeError, match=r"cnnacc error -4: member 1 .*classifier not loaded"):
            m.infer_batch(imgs)
        failed = ctypes.c_int(99)
        probs = np.zeros((n, 6), np.float32)
        assert lib.cnnacc_infer_batch_sharded(_hs(m.members), k, _p(imgs), n, _p(probs), None, None, 0,
                                              ctypes.byref(failed)) == fc._lib.ERR_STATE and failed.value == 1
        assert _counts(m) == c0
        m.run_batch(imgs)
