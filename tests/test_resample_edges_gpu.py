"""The two resampling front ends on the GPU at the edges of their domains, byte for byte against outputs Pillow 12.2.0 and
cv2 4.13.0 computed directly (tests/golden/resample_edges.npz, tests/golden/make_resample_edges_golden.py):

* cnnacc_image_to_gray128 (csrc/pil_resize.cuh) on both sides of Image.resize's switch to the vertical pass first
  (H > 100 W), on 1-pixel and 32768-pixel sides, in modes L / RGB / RGBA, in batches of 1 and 3, from host arrays and from
  torch CUDA tensors;
* the centre-crop pre-processing (preprocess_bgr_kernel) and detect_frames at crop sides 1081 .. 8192, on 4K frames (one
  per staging chunk) and 8192x8192 frames (above the 64 MiB latency path), from host and device pointers;
* the region kernel (preprocess_regions_kernel) on every large side at the corners of an 8192x8192 frame and on a 4K frame;
* the per-handle table caches, switched between calls that are all queued before any of them runs.
u8 / i32 outputs and fp32 probabilities must match exactly."""
import ctypes
import os

import numpy as np
import pytest

import inputs

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "resample_edges.npz")


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


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


def _pil_groups():
    groups = {}
    for c in inputs.RESAMPLE_PIL_CASES:
        groups.setdefault((c["h"], c["w"], c["mode"]), []).append(c)
    return groups


PIL_GROUPS = _pil_groups()


def assert_same(got, want, what=""):
    assert len(got) == len(want), what
    for i, (g, w) in enumerate(zip(got, want)):
        g = g.cpu().numpy() if hasattr(g, "cpu") else g
        assert g.dtype == w.dtype and g.shape == w.shape, (what, i)
        assert np.array_equal(g.view(np.uint8), w.view(np.uint8)), (what, i, int((g != w).sum()))


@pytest.mark.parametrize("key", list(PIL_GROUPS), ids=lambda k: f"{k[0]}x{k[1]}_{k[2]}")
def test_image_to_gray128_edges(acc, golden, key):
    """Every case alone, then a batch of 3 with an all-zero image (whose output is exactly 0) between two cases, then the
    group's cases together: host arrays and torch CUDA tensors."""
    import torch
    cases = PIL_GROUPS[key]
    imgs = [inputs.make_pil_image(c) for c in cases]
    want = [golden[c["name"]] for c in cases]
    zero = np.zeros_like(imgs[0])
    batches = [([i], [imgs[i]]) for i in range(len(cases))]
    batches.append(([len(cases) - 1, None, 0], [imgs[-1], zero, imgs[0]]))
    if len(cases) == 3:
        batches.append(([0, 1, 2], imgs))
    for idx, batch in batches:
        x = np.stack(batch)
        exp = np.stack([want[i] if i is not None else np.zeros((128, 128), np.uint8) for i in idx])
        got = acc.image_to_gray128(x)
        assert got.shape == (len(idx), 128, 128)
        assert_same(got, exp, ("host", key, idx))
        assert_same(acc.image_to_gray128(torch.from_numpy(x).cuda()), exp, ("torch", key, idx))


def _detect_frames_dev(fc, acc, t):
    """cnnacc_detect_frames with device pointers on torch's current stream -> (cls, probs, bbox, gray) tensors."""
    import torch
    n = t.shape[0]
    new = lambda shape, dt: torch.empty(shape, dtype=dt, device=t.device)
    cls, probs, box, gray = new((n,), torch.int32), new((n, 6), torch.float32), new((n, 4), torch.int32), new((n, 128, 128), torch.uint8)
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    with acc._on_stream_of(t):
        acc._check(acc._libc.cnnacc_detect_frames(acc._h, p(t), n, t.shape[1], t.shape[2], p(gray), p(probs), p(cls), p(box),
                                                  fc._lib.FLAG_DEVICE_PTRS))
    return cls, probs, box, gray


@pytest.mark.parametrize("case", inputs.RESAMPLE_AREA_CASES, ids=lambda c: c["name"])
def test_preprocess_and_detect_frames_edges(fc, acc, golden, case):
    import torch
    frames = inputs.make_area_frames(case["name"])
    want = golden[case["name"]]
    assert_same(acc.preprocess(frames), want, "host")
    t = torch.from_numpy(frames).cuda()
    assert_same(acc.preprocess(t), want, "device")
    pred = acc.infer_batch(want)                                   # the conv stack and tail on the fixture's gray images
    cls, probs, box, gray = acc.detect_frames(frames, return_gray=True)
    assert_same((cls, probs, box, gray), (*pred, want), "detect_frames host")
    assert_same(_detect_frames_dev(fc, acc, t), (*pred, want), "detect_frames device")


def test_regions_at_the_corners_of_8192_frames(fc, acc, golden):
    """Every large side at the four corners of one 8192x8192 frame and three odd sides on a second, in one call: host staging
    (one 201 MB frame per chunk), device pointers, and detect_regions against infer_batch on the fixture's gray images."""
    import torch
    frames = np.concatenate([inputs.make_area_frames("area_k64_8192"), inputs.make_area_frames("area_k64_8192_edges")])
    reg, want = inputs.REGIONS_8192, golden["regions_8192"]
    assert_same(acc.preprocess_regions(frames, reg), want, "host")
    t = torch.from_numpy(frames).cuda()
    assert_same(acc.preprocess_regions(t, reg), want, "device")
    pred = acc.infer_batch(want)
    assert_same(acc.detect_regions(frames, reg, return_gray=True), (*pred, want), "detect host")
    perm = np.random.default_rng(3).permutation(len(reg))
    assert_same(acc.detect_regions(t, reg[perm], return_gray=True), tuple(x[perm] for x in (*pred, want)), "detect device")


def test_regions_of_4k_frames_through_host_staging(acc, golden):
    frames = inputs.make_area_frames("area_4k")
    reg, want = inputs.REGIONS_4K, golden["regions_4k"]
    assert_same(acc.preprocess_regions(frames, reg), want)
    pred = acc.infer_batch(want)
    assert_same(acc.detect_regions(frames, reg, return_gray=True), (*pred, want))
    perm = np.random.default_rng(4).permutation(len(reg))
    assert_same(acc.detect_regions(frames, reg[perm], return_gray=True), tuple(x[perm] for x in (*pred, want)))


def test_table_caches_switch_between_queued_calls(acc, golden):
    """Crop sides and loader sizes alternate on one handle in device-pointer calls, each queued behind a sleep kernel: a call
    that replaced the handle's INTER_AREA or Pillow tables without waiting for the device would change them under the kernel
    of the call before it.  Every result equals the fixture."""
    import torch
    sides = ["area_1081", "area_k9_1152", "area_2047", "area_1081", "area_4095", "area_k16_2048", "area_2047", "area_1081"]
    loads = ["pil_201x2_L_rng", "pil_200x2_L_rng", "pil_2000x17_L_rng", "pil_17x2000_L_rng", "pil_201x2_L_rng",
             "pil_6401x64_RGB_rng", "pil_6400x64_RGB_rng", "pil_2000x17_L_rng"]
    frames = {n: torch.from_numpy(inputs.make_area_frames(n)).cuda() for n in set(sides)}
    pil = {c["name"]: c for c in inputs.RESAMPLE_PIL_CASES}
    imgs = {n: torch.from_numpy(inputs.make_pil_image(pil[n])[None].copy()).cuda() for n in set(loads)}
    torch.cuda.synchronize()
    got = []
    for s, l in zip(sides, loads):
        torch.cuda._sleep(20_000_000)
        got.append((s, acc.preprocess(frames[s])))
        torch.cuda._sleep(20_000_000)
        got.append((l, acc.image_to_gray128(imgs[l])))
    torch.cuda.synchronize()
    for k, (name, g) in enumerate(got):
        w = golden[name]
        assert_same(g, w if w.ndim == 3 else w[None], (k, name))
