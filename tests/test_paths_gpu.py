"""Every entry point that computes features or predictions, against the oracle, on the workloads where a one-LSB error shows
(inputs.EXPOSED_WORKLOADS; tests/test_exposure_cpu.py measures what each can see), at 32- and 24-bit accumulator width.

References: oracle.port_infer_batch (the C port) for 32-bit features, np_oracle.infer(acc_bits=24) for 24-bit ones, and
np_oracle.classify_vec / bbox_vec / get_cam_bbox for predictions on the oracle's features.  Tolerances are test_tail_gpu.py's:
probabilities within 1e-5, logits within 1e-5 * max|logit|, the same argmax except where the reference's top two logits are
closer than that, boxes exact.
"""
import multiprocessing as mp

import numpy as np
import pytest

import inputs
import oracle
from oracle import np_oracle

pytestmark = pytest.mark.gpu

PROB_ATOL = 1e-5
LOGIT_RTOL = 1e-5
N_MANY = {32: 3000, 24: 1200}    # host calls this long go through the staging ring in ramped chunks (the 24-bit numpy reference
                                 # costs about 0.1 s an image)
N_PRED = 100                     # > 64: host prediction calls go through the staging ring
WS = 16384                       # images per feature-workspace chunk of a device-pointer prediction call
CASES = [(w, bits) for w in inputs.EXPOSED_WORKLOADS for bits in (32, 24)]
IDS = [f"{w['name']}-{bits}" for w, bits in CASES]


def _features_job(job):
    imgs, wt, sh, bits, H, W = job
    if bits == 32:
        return oracle.port_infer_batch(oracle.load_port(), imgs, wt, sh, H, W)
    kern = np_oracle.unpack_weights(wt)
    return np.stack([np_oracle.infer(im, kern, sh, H, W, acc_bits=24) for im in imgs])


def reference(wt, sh, bits, imgs, H=128, W=128):
    """(n, 64, H/8*W/8) u8 oracle features, on a process pool for large n."""
    n = len(imgs)
    workers = max(1, min(mp.cpu_count(), 32, n // 16))
    if workers == 1:
        return _features_job((imgs, wt, sh, bits, H, W))
    b = np.linspace(0, n, workers + 1).astype(int)
    with mp.get_context("fork").Pool(workers) as pool:
        return np.concatenate(pool.map(_features_job, [(imgs[b[i]:b[i + 1]], wt, sh, bits, H, W) for i in range(workers)]))


def pred_reference(feats, fw, fb):
    """Per image: (cls, probs, logits, bbox_vec box, get_cam_bbox box) of the oracle."""
    out = []
    for f in feats.reshape(-1, 64, 256):
        c, p, logits, _ = np_oracle.classify_vec(f, fw, fb)
        out.append((c, p, logits, np_oracle.bbox_vec(f, c, fw)[0], np_oracle.get_cam_bbox(f, c, fw)[1]))
    return out


def check_predictions(got, ref, bbox, logits, what):
    cls, probs, box = (np.asarray(a.cpu() if hasattr(a, "cpu") else a) for a in got)
    assert cls.shape == (len(ref),), what
    for i, (c, p, lg, box_vec, box_up) in enumerate(ref):
        scale = np.abs(lg).max()
        if cls[i] != c:
            top2 = np.sort(lg)[-2:]
            assert top2[1] - top2[0] <= LOGIT_RTOL * scale, f"{what}: argmax differs on image {i}"
            continue
        if logits:
            assert np.abs(probs[i] - lg).max() <= LOGIT_RTOL * scale, f"{what}: logits of image {i}"
        else:
            assert np.abs(probs[i] - p).max() <= PROB_ATOL, f"{what}: probabilities of image {i}"
        assert tuple(box[i]) == (box_up if bbox == "upsampled" else box_vec), f"{what}: box of image {i}"


def same(got, want, what):
    got = np.asarray(got.cpu() if hasattr(got, "cpu") else got).reshape(want.shape)
    bad = int((got != want).sum())
    assert bad == 0, f"{what}: {bad} bytes differ, first at {np.argwhere(got != want)[:3].tolist()}"


@pytest.fixture(scope="module")
def fc():
    import fpga_cnn_b200 as fc_
    fc_.load()
    return fc_


@pytest.fixture(scope="module")
def acc(fc):
    a = fc.CNNAccelerator()
    a.load_classifier(*inputs.make_fc())
    yield a
    a.close()


_cache = {}


def configure(a, w, bits):
    a.load_weights(inputs.make_weights(w["weights"]))
    a.set_shifts(*w["shifts"])
    a.set_accumulator_bits(bits)


def many(w, bits):
    """N_MANY[bits] images of the workload (its own first) and their oracle features, computed once per module run."""
    key = (w["name"], bits)
    if key not in _cache:
        imgs = inputs.workload_images(w, N_MANY[bits])
        _cache[key] = imgs, reference(inputs.make_weights(w["weights"]), w["shifts"], bits, imgs)
    return _cache[key]


def preds(w, bits):
    key = (w["name"], bits, "pred")
    if key not in _cache:
        imgs, feats = many(w, bits)
        _cache[key] = pred_reference(feats[:N_PRED], *inputs.make_fc())
    return _cache[key]


# ---- features ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_run_batch_host_and_device(w, bits, fc, acc):
    """Host arrays at n = 1 (latency path), 64, 65 (the first call through the staging ring), N_MANY (ramped chunks); a CUDA
    tensor; the per-layer kernels (direct=True)."""
    import torch
    configure(acc, w, bits)
    imgs, want = many(w, bits)
    for n in (1, 64, 65, len(imgs)):
        same(acc.run_batch(imgs[:n]), want[:n], f"host n={n}")
    same(acc.run_batch(torch.from_numpy(imgs).cuda()), want, "CUDA tensor")
    same(acc.run_batch(imgs[:300], direct=True), want[:300], "direct")


@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_run_batch_async(w, bits, fc, acc):
    """Several host batches in flight through one staging ring, waited for in submission order and out of it."""
    configure(acc, w, bits)
    imgs, want = many(w, bits)
    n = len(imgs)
    cuts = np.cumsum([0, n // 4, 1, 64, 65, n // 2, n - n // 4 - n // 2 - 130])
    ins = []
    for a0, a1 in zip(cuts[:-1], cuts[1:]):
        h = fc.alloc_host((a1 - a0, 128, 128))
        h[:] = imgs[a0:a1]
        ins.append(h)
    tickets = [acc.run_batch_async(h) for h in ins]
    outs = {i: acc.wait_batch(tickets[i]) for i in (3, 0, 5, 1, 2, 4)}
    for i, (a0, a1) in enumerate(zip(cuts[:-1], cuts[1:])):
        same(outs[i], want[a0:a1], f"async batch {i}")


@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_register_protocol(w, bits, acc):
    """load_image / start_inference / read_feature_map: all 112 BRAM channels of three images (layers 0 and 1 too)."""
    configure(acc, w, bits)
    kern = np_oracle.unpack_weights(inputs.make_weights(w["weights"]))
    for img in inputs.workload_images(w)[:3]:
        f2, l0, l1 = np_oracle.infer(img, kern, w["shifts"], return_all=True, acc_bits=bits)
        acc.load_image(img)
        acc.start_inference()
        assert acc.wait_done(10.0) >= 0
        for ch in range(16):
            same(acc.read_feature_map(ch, 4096), l0[ch].reshape(-1), f"layer 0 channel {ch}")
        for ch in range(32):
            same(acc.read_feature_map(16 + ch, 1024), l1[ch].reshape(-1), f"layer 1 channel {ch}")
        same(acc.read_layer2_output(), f2, "layer 2")


@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_infer_one_distinct_images_in_sequence(w, bits, acc):
    """The zero-copy batch-1 path: 300 different images one after another, each against its own oracle result, so features
    read before the kernel's store has landed (the previous image's) show."""
    configure(acc, w, bits)
    imgs, want = many(w, bits)
    for i in range(300):
        feat = acc.infer_one(imgs[i])[0]
        same(feat, want[i], f"infer_one image {i}")


@pytest.mark.parametrize("w", inputs.EXPOSED_WORKLOADS, ids=lambda w: w["name"])
def test_cnn_infer_symbol(w, fc):
    """cnn_infer through ARMEngine (realtime_detect.py:422-436).  Its process-wide handle always accumulates in 32 bits."""
    imgs, want = many(w, 32)
    eng = fc.ARMEngine(inputs.make_weights(w["weights"]), shifts=w["shifts"])
    for i in range(40):
        same(eng.run(imgs[i])[0], want[i], f"cnn_infer image {i}")


@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_multi_accelerator(w, bits, fc):
    """MultiAccelerator over two handles on one GPU: run_batch, infer_batch and detect_frames, sharded."""
    imgs, want = many(w, bits)
    with fc.MultiAccelerator([0, 0]) as m:
        m.load_weights(inputs.make_weights(w["weights"]))
        m.set_shifts(*w["shifts"])
        m.set_accumulator_bits(bits)
        m.load_classifier(*inputs.make_fc())
        same(m.run_batch(imgs), want, "sharded run_batch")
        check_predictions(m.infer_batch(imgs[:300], bbox="upsampled"), pred_reference(want[:300], *inputs.make_fc()),
                          "upsampled", False, "sharded infer_batch")
        frames = inputs.make_frames(("smooth", 900), 64, 144, 176)
        check_predictions(m.detect_frames(frames), _frames_reference(frames, w, bits), "vec", False, "sharded detect_frames")


# ---- sizes ------------------------------------------------------------------------------------------------------------
WINDOW_SIZES = [(128, 144), (144, 128), (128, 8192), (8192, 128), (400, 208)]
PER_LAYER_SIZES = [(16, 16), (16, 8192), (8192, 16), (48, 80), (112, 1024)]


@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_sizes(w, bits, acc):
    """Overlapping 128x128 windows (both sides >= 128) and the per-layer kernels (a side below 128) against the oracle's
    H x W form."""
    configure(acc, w, bits)
    wt = inputs.make_weights(w["weights"])
    for H, W in WINDOW_SIZES + PER_LAYER_SIZES:
        n = 1 if H * W > 200000 else 2
        imgs = inputs.workload_images(w, n, H, W)
        got = acc.run_batch(imgs)
        assert got.shape == (n, 64, H // 8, W // 8)
        same(got.reshape(n, 64, -1), reference(wt, w["shifts"], bits, imgs, H, W), f"{H}x{W}")


# ---- predictions ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_infer_batch_every_form(w, bits, acc):
    """infer_batch on host arrays and CUDA tensors, bbox 'vec' and 'upsampled', probabilities and logits, through the tail
    inside the conv kernel, the per-layer kernels (direct) and the features-in tail kernel (two_kernels)."""
    import torch
    configure(acc, w, bits)
    imgs, _ = many(w, bits)
    ref = preds(w, bits)
    x_host = imgs[:N_PRED]
    x_dev = torch.from_numpy(x_host).cuda()
    for x, kind in ((x_host, "host"), (x_dev, "device")):
        for bbox in ("vec", "upsampled"):
            for logits in (False, True):
                for mode in ("fused", "direct", "two_kernels"):
                    got = acc.infer_batch(x, bbox=bbox, logits=logits, direct=mode == "direct", two_kernels=mode == "two_kernels")
                    check_predictions(got, ref, bbox, logits, f"{kind} {bbox} logits={logits} {mode}")


@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_tail_calls_on_oracle_features(w, bits, acc):
    """classify_batch, cam_bbox_batch and pool_features on the oracle's features."""
    configure(acc, w, bits)
    _, feats = many(w, bits)
    feats = feats[:N_PRED]
    ref = preds(w, bits)
    for bbox in ("vec", "upsampled"):
        for logits in (False, True):
            check_predictions(acc.classify_batch(feats, bbox=bbox, logits=logits), ref, bbox, logits, f"classify_batch {bbox} {logits}")
    cls = np.array([r[0] for r in ref], np.int32)
    assert [tuple(b) for b in acc.cam_bbox_batch(feats, cls)] == [r[4] for r in ref]
    assert np.array_equal(acc.pool_features(feats), np_oracle.pool_bins(feats))


def _frames_reference(frames, w, bits):
    gray = np.stack([np_oracle.preprocess_bgr(f) for f in frames])
    return pred_reference(reference(inputs.make_weights(w["weights"]), w["shifts"], bits, gray), *inputs.make_fc())


@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_detect_frames_and_regions(w, bits, acc):
    """detect_frames (centre crop, gray, INTER_AREA, conv stack, tail) against preprocess_bgr followed by the oracle, and
    detect_regions on square regions of the same frames."""
    configure(acc, w, bits)
    frames = inputs.make_frames(("smooth", 901), 4, 300, 420)
    for bbox in ("vec", "upsampled"):
        check_predictions(acc.detect_frames(frames, bbox=bbox), _frames_reference(frames, w, bits), bbox, False, f"detect_frames {bbox}")
    regions = np.array([(0, 0, 0, 300), (1, 420 - 128, 300 - 128, 128), (2, 17, 33, 200), (3, 100, 0, 256)], np.int32)
    crops = np.stack([np_oracle.preprocess_bgr(frames[f, y:y + s, x:x + s]) for f, x, y, s in regions])
    ref = pred_reference(reference(inputs.make_weights(w["weights"]), w["shifts"], bits, crops), *inputs.make_fc())
    check_predictions(acc.detect_regions(frames, regions, bbox="upsampled"), ref, "upsampled", False, "detect_regions")


# ---- device-pointer calls longer than one feature workspace -----------------------------------------------------------
@pytest.mark.parametrize("w,bits", CASES, ids=IDS)
def test_device_infer_batch_across_workspace_chunks(w, bits, acc):
    """2 * 16384 + 3 images on device pointers: the forms that need the feature workspace (upsampled, direct, two_kernels)
    run it in three chunks.  Each equals the same handle's host-pointer result; the chunk edges and a strided sample equal
    the oracle."""
    import torch
    configure(acc, w, bits)
    n = 2 * WS + 3
    kind = w["more"] if w["more"][0] in ("rng", "bright") else ("rng", 910)
    imgs = inputs.make_images(kind, n)
    idx = np.unique(np.concatenate([np.arange(WS - 1, WS + 3), np.arange(2 * WS - 1, n), np.arange(0, n, 1999)]))
    ref = pred_reference(reference(inputs.make_weights(w["weights"]), w["shifts"], bits, imgs[idx]), *inputs.make_fc())
    x = torch.from_numpy(imgs).cuda()
    for bbox, direct, two in (("upsampled", False, False), ("vec", True, False), ("vec", False, True), ("upsampled", False, True)):
        what = f"bbox={bbox} direct={direct} two_kernels={two}"
        dev = [t.cpu().numpy() for t in acc.infer_batch(x, bbox=bbox, direct=direct, two_kernels=two)]
        host = acc.infer_batch(imgs, bbox=bbox, direct=direct, two_kernels=two)
        for d, h in zip(dev, host):
            assert np.array_equal(d, h), f"{what}: device != host at {np.flatnonzero((d != h).reshape(n, -1).any(axis=1))[:5]}"
        check_predictions([a[idx] for a in dev], ref, bbox, False, what)
