"""The scanning calls against the oracle at the frame sizes they serve, and across the edges where a call is cut into pieces.

tests/test_scan_gpu.py and tests/test_scan_pyramid_gpu.py compare every window with classify_batch on run_batch's map of
the frame or level: both are this library's kernels, so a fault of the window-tiled conv at a large size would be in the
call and in its reference alike.  Here the reference is the oracle (tests/scan_reference.py): the C port at 32 bits and
the numpy oracle at 24 bits, on row bands of the whole frame or level, and np_oracle's tail on the windows.

  * run_batch's whole maps at 864x1536, 720x1280, 1440x2560, 2160x3840, 128x8192 and 8192x8192, and every level map of
    the pyramid cases;
  * scan_frames at 720x1280 / 8, 2160x3840 / 64, 128x8192 / 8 and 8192x8192 / 64, scan_pyramid on 1080p, 4K, VGA with a
    128x128 level and an anisotropic set, with probabilities and with logits;
  * calls long enough to cross at least two piece edges (device pointers) or staging-chunk and prediction-block edges
    (host pointers) and to end in a partial piece, against the same frames in calls of at most one piece, against
    merge_regions on their own predictions, and against the oracle on the frames either side of every edge.

Workloads: the shipped weights and the ternary EXPOSED_WORKLOADS at 32 bits; the ternary ones at 24 bits up to 1280x720.
Each case holds its oracle maps and windows to scan_reference.assert_exposed, so none passes on saturated bytes."""
import numpy as np
import pytest

import inputs
import pyramid_oracle
import scan_oracle
import scan_reference as sr
from test_detect_objects_cpu import assert_same
from test_paths_gpu import same

pytestmark = pytest.mark.gpu

# The shipped weights at shifts (7, 10, 10): at (7, 10, 11) the seeded classifier puts every window of these frames in one
# class.  tern_tb takes classifier seed 8 for the same reason.
SHIPPED = dict(name="shipped", weights="shipped", shifts=(7, 10, 10), fc_seed=1234)
TERNARY = [dict(name=w["name"], weights=w["weights"], shifts=w["shifts"], fc_seed=8 if w["name"] == "tern_tb" else 1234)
           for w in inputs.EXPOSED_WORKLOADS if w["name"].startswith("tern")]
MAX_24 = 720 * 1280                 # the numpy oracle's 24-bit conv is affordable up to 1280x720 frames and levels
MIN_INSIDE = 0.35                   # share of oracle map bytes strictly inside (0, 255); the CPU oracle gives 0.41 .. 0.53

VGA = [(640, 480), (512, 384), (320, 240), (256, 192)]
P1080 = [(1536, 864), (1280, 720), (1024, 576), (768, 432), (512, 288), (256, 144)]


def configs(max_px):
    """(workload, bits) pairs for a case of at most max_px pixels per frame or level."""
    out = [(w, 32) for w in [SHIPPED] + TERNARY]
    return out + ([(w, 24) for w in TERNARY] if max_px <= MAX_24 else [])


def params(cases, px):
    """(workload, bits) x cases, the 24-bit configurations only where px(case) <= MAX_24, and their ids."""
    out = [(w, bits) + tuple(c) for c in cases for w, bits in configs(px(c))]
    return out, [f"{p[0]['name']}-{p[1]}-" + "x".join(str(v) for v in p[2:4]) + f"-{len(p[4]) if len(p) > 5 else ''}s{p[-1]}"
                 for p in out]


@pytest.fixture(scope="module")
def fc():
    import fpga_cnn_b200
    fpga_cnn_b200.load()
    return fpga_cnn_b200


@pytest.fixture(scope="module")
def acc(fc):
    a = fc.CNNAccelerator()
    yield a
    a.close()


def weights_of(w, shipped_weights):
    return shipped_weights if w["weights"] == "shipped" else inputs.make_weights(w["weights"])


def configure(acc, shipped_weights, w, bits):
    acc.load_weights(weights_of(w, shipped_weights))
    acc.set_shifts(*w["shifts"])
    acc.set_accumulator_bits(bits)
    acc.load_classifier(*inputs.make_fc(w["fc_seed"]))


def _np(x):
    return tuple(np.asarray(t.cpu()) if hasattr(t, "cpu") else t for t in x)


_frames = {}


def frame(fh, fw):
    """One smooth BGR frame per size, shared by every workload (an 8192x8192 one takes seconds to make)."""
    if (fh, fw) not in _frames:
        _frames[(fh, fw)] = inputs.make_frames(("smooth", fh + fw), 1, fh, fw)
    return _frames[(fh, fw)]


def level_reference(gray, w, bits, shipped_weights, stride, seed=0, all_windows=sr.ALL_WINDOWS):
    """Oracle maps [F][64][h/8][w/8] of F gray images (F, h, w), the windows to check (indices into one image's windows)
    and the oracle's predictions on them, image-major."""
    F, h, wd = gray.shape
    maps = sr.oracle_maps(gray, weights_of(w, shipped_weights), w["shifts"], bits)
    if not stride:
        return maps, None, []
    idx = sr.select_windows(h, wd, stride, seed, all_windows)
    ref = []
    for f in range(F):
        ref += sr.tail(sr.level_windows(maps[f], h, wd, stride, idx), *inputs.make_fc(w["fc_seed"]))
    return maps, idx, ref


# ---- whole maps and scan_frames -------------------------------------------------------------------------------------------

FRAME_CASES = [(864, 1536, None), (720, 1280, 8), (1440, 2560, None), (2160, 3840, 64), (128, 8192, 8), (8192, 8192, 64)]


def frame_reference(w, bits, shipped_weights, fh, fw, stride):
    """-> (frames [1][fh][fw][3], gray, oracle maps [64][fh/8][fw/8], checked windows, their oracle predictions)."""
    frames = frame(fh, fw)
    gray = pyramid_oracle.gray(frames[0])
    maps, idx, ref = level_reference(gray[None], w, bits, shipped_weights, stride)
    what = (w["name"], bits, fh, fw, stride)
    if stride:
        sr.assert_exposed(maps, ref, MIN_INSIDE, what)
    else:
        assert ((maps > 0) & (maps < 255)).mean() >= MIN_INSIDE, what
    return frames, gray, maps[0], idx, ref


FRAME_PARAMS, FRAME_IDS = params(FRAME_CASES, lambda c: c[0] * c[1])


@pytest.mark.parametrize("w,bits,fh,fw,stride", FRAME_PARAMS, ids=FRAME_IDS)
def test_run_batch_and_scan_frames_vs_oracle(fc, acc, shipped_weights, w, bits, fh, fw, stride):
    """run_batch's whole map of the frame's gray equals the oracle's; scan_frames' windows (all of them, or the selection
    on large frames) equal the oracle's tail on that map."""
    configure(acc, shipped_weights, w, bits)
    frames, gray, maps, idx, ref = frame_reference(w, bits, shipped_weights, fh, fw, stride)
    same(acc.run_batch(gray[None]), maps[None], f"run_batch {fh}x{fw}")
    if stride is None:
        return
    for logits in (False, True):
        got = acc.scan_frames(frames, stride, logits=logits)
        assert len(got[0]) == scan_oracle.count(fh, stride) * scan_oracle.count(fw, stride)
        sr.check_windows(got, idx, ref, logits, f"scan_frames {fh}x{fw} stride {stride} logits={logits}")


# ---- scan_pyramid ---------------------------------------------------------------------------------------------------------

PYRAMID_CASES = [(1080, 1920, P1080, 16), (2160, 3840, [(2560, 1440), (1280, 720)], 64), (480, 640, VGA + [(128, 128)], 16),
                 (720, 1280, [(640, 720), (1280, 240)], 16)]


def pyramid_reference(w, bits, shipped_weights, frames, levels, stride, all_windows=sr.ALL_WINDOWS):
    """-> (level gray [F][sum h*w], per level oracle maps [F][64][h/8][w/8], rows into the call's windows, the oracle's
    predictions for those rows) for frames [F][fh][fw][3]."""
    F = len(frames)
    lv_gray = pyramid_oracle.preprocess(frames, levels)
    counts = [scan_oracle.count(h, stride) * scan_oracle.count(wd, stride) for wd, h in levels]
    per, first = sum(counts), np.cumsum([0] + counts)
    level_maps, rows, refs, o = [], [], [], 0
    for l, (wd, h) in enumerate(levels):
        g = lv_gray[:, o:o + wd * h].reshape(F, h, wd)
        o += wd * h
        maps, idx, ref = level_reference(g, w, bits, shipped_weights, stride, seed=l, all_windows=all_windows)
        level_maps.append(maps)
        rows.append((np.arange(F)[:, None] * per + first[l] + idx[None]).ravel())
        refs.append(ref)
    ref = [r for part in refs for r in part]
    sr.assert_exposed(np.concatenate([m.ravel() for m in level_maps]), ref, MIN_INSIDE, (w["name"], bits, frames.shape, levels,
                                                                                          stride))
    return lv_gray, level_maps, np.concatenate(rows), ref


PYRAMID_PARAMS, PYRAMID_IDS = params(PYRAMID_CASES, lambda c: max(wd * h for wd, h in c[2]))


@pytest.mark.parametrize("w,bits,fh,fw,levels,stride", PYRAMID_PARAMS, ids=PYRAMID_IDS)
def test_scan_pyramid_vs_oracle(fc, acc, shipped_weights, w, bits, fh, fw, levels, stride):
    """preprocess_pyramid equals the numpy INTER_AREA levels (pinned to cv2), run_batch of every level equals the oracle's
    map, and scan_pyramid's windows equal the oracle's tail on those maps."""
    configure(acc, shipped_weights, w, bits)
    frames = frame(fh, fw)
    lv_gray, level_maps, rows, ref = pyramid_reference(w, bits, shipped_weights, frames, levels, stride)
    assert np.array_equal(acc.preprocess_pyramid(frames, levels), lv_gray)
    o = 0
    for (wd, h), maps in zip(levels, level_maps):
        same(acc.run_batch(np.ascontiguousarray(lv_gray[:, o:o + wd * h].reshape(1, h, wd))), maps, f"run_batch level {wd}x{h}")
        o += wd * h
    for logits in (False, True):
        got = acc.scan_pyramid(frames, levels, stride, logits=logits)
        assert len(got[0]) == len(fc.pyramid_windows(1, fh, fw, levels, stride))
        sr.check_windows(got, rows, ref, logits, f"scan_pyramid {fh}x{fw} {levels} stride {stride} logits={logits}")


# ---- piece and block edges ------------------------------------------------------------------------------------------------

PRED_BLOCK = 1 << 20                # host pointers: predictions come back in frame-aligned blocks of up to 2^20 windows
STAGE = 16 << 20                    # host pointers: frames are staged in chunks of 16 MiB (a larger frame alone)
WORKSPACE = 256 << 20               # device pointers: pieces whose gray and feature workspaces are at most 256 MiB each


def piece_frames(fh, fw, levels, per):
    """Frames per device-pointer piece: min(256 MiB / max(plane + resized levels, level pixels), 2^20 / windows per frame)."""
    resized = sum(wd * h for wd, h in levels if (wd, h) != (fw, fh))
    return min(WORKSPACE // max(fh * fw + resized, sum(wd * h for wd, h in levels)), PRED_BLOCK // per)


def host_cuts(n, fh, fw, per):
    """-> (block edges, staging chunks (f0, f1)) of a host-pointer call of n frames: chunks restart at every block."""
    bf, fpc = max(PRED_BLOCK, per) // per, min(n, max(1, STAGE // (fh * fw * 3)))
    blocks = list(range(0, n, bf)) + [n]
    return blocks, [(f0, min(f0 + fpc, fb)) for fa, fb in zip(blocks, blocks[1:]) for f0 in range(fa, fb, fpc)], fpc


def distinct_frames(n, fh, fw, seed):
    """n frames, each its own: one of eight smooth frames rolled by an offset drawn from the frame's own seed, so a
    prediction or detection put on the wrong frame shows."""
    base = inputs.make_frames(("smooth", seed), 8, fh, fw)
    out = np.empty((n, fh, fw, 3), np.uint8)
    for f in range(n):
        r = np.random.default_rng(seed * 100000 + f)
        out[f] = np.roll(base[f % 8], (int(r.integers(fh)), int(r.integers(fw))), axis=(0, 1))
    return out


# (call, fh, fw, levels, stride, windows per frame, frames per device piece).  The VGA pyramid carries a 128x128 level, so
# with at least one SM's worth of frames per piece that level's conv launches may overlap (csrc/pdl_chain.h).
EDGE_CASES = [("frames", 480, 640, [(640, 480)], 8, 2925, 358),
              ("pyramid", 480, 640, VGA + [(128, 128)], 8, 5071, 206),
              ("pyramid", 1080, 1920, P1080, 16, 9723, 49)]


@pytest.mark.parametrize("kind,fh,fw,levels,stride,want_per,want_piece", EDGE_CASES,
                         ids=[f"{c[0]}_{c[1]}x{c[2]}_{len(c[3])}_{c[4]}" for c in EDGE_CASES])
def test_calls_across_piece_and_block_edges(fc, acc, shipped_weights, kind, fh, fw, levels, stride, want_per, want_piece):
    """2 pieces + 3 frames in one call, on host arrays and CUDA tensors, predictions and detections, sized from the
    restated constants above and asserted to straddle the edges it claims."""
    import torch
    w = SHIPPED
    configure(acc, shipped_weights, w, 32)
    if kind == "frames":
        windows = lambda n: fc.grid_regions(n, fh, fw, 128, stride)                                         # noqa: E731
        scan = lambda x: acc.scan_frames(x, stride)                                                          # noqa: E731
        objects = lambda x, **kw: acc.scan_objects(x, stride, **kw)                                         # noqa: E731
    else:
        windows = lambda n: fc.pyramid_windows(n, fh, fw, levels, stride)                                   # noqa: E731
        scan = lambda x: acc.scan_pyramid(x, levels, stride)                                                 # noqa: E731
        objects = lambda x, **kw: acc.scan_pyramid_objects(x, levels, stride, **kw)                         # noqa: E731
    per = len(windows(1))
    piece = piece_frames(fh, fw, levels, per)
    assert (per, piece) == (want_per, want_piece)
    n = 2 * piece + 3
    starts = list(range(0, n, piece))
    assert len(starts) == 3 and n % piece, "device pointers: two piece edges, a partial last piece"
    blocks, chunks, fpc = host_cuts(n, fh, fw, per)
    assert len(chunks) >= 3 and chunks[-1][1] - chunks[-1][0] < fpc, "host pointers: staging-chunk edges, a partial last chunk"
    if fh * fw <= 640 * 480:
        assert len(blocks) - 1 >= 3 and n % (blocks[1] - blocks[0]), "host pointers: two block edges, a partial last block"
    if (128, 128) in levels:
        assert piece >= torch.cuda.get_device_properties(0).multi_processor_count
    frames = distinct_frames(n, fh, fw, 7)
    t = torch.from_numpy(frames).cuda()
    cut = piece * 2 // 3                                   # reference calls: one piece each, cut off the big call's edges

    # predictions: host == device == the same frames in one-piece calls, concatenated
    host = scan(frames)
    assert len(host[0]) == n * per
    assert_same(_np(scan(t)), host, "device")
    parts = [_np(scan(t[f0:f0 + cut])) for f0 in range(0, n, cut)]
    assert_same(host, tuple(np.concatenate([p[k] for p in parts]) for k in range(3)), "one-piece calls")

    # detections: == merge_regions on the call's own predictions, == one-piece calls with region indices shifted
    cls, probs, box = host
    scores = probs[np.arange(len(cls)), cls]
    kw = dict(score_min=float(np.percentile(scores, 90)), iou_max=0.3, max_det=64)
    want = acc.merge_regions(windows(n), cls, scores, box, n, **kw)
    assert (want[0] > 0).mean() > 0.9 and len(np.unique(want[2][want[2] >= 0])) >= 2
    assert_same(objects(frames, **kw), want, "objects host")
    assert_same(_np(objects(t, **kw)), want, "objects device")
    pieces = []
    for f0 in range(0, n, cut):
        d = list(_np(objects(t[f0:f0 + cut], **kw)))
        d[1] = np.where(d[1] >= 0, d[1] + f0 * per, d[1]).astype(np.int32)
        pieces.append(d)
    assert_same(want, tuple(np.concatenate([p[k] for p in pieces]) for k in range(5)), "objects in one-piece calls")

    # the oracle on the frames either side of every piece and block edge, and on the last frame
    edges = sorted({f for s in starts[1:] + blocks[1:-1] for f in (s - 1, s)} | {n - 1})
    _, _, rows, ref = pyramid_reference(w, 32, shipped_weights, frames[edges], levels, stride, all_windows=1024)
    f_of = rows // per
    rows = np.asarray(edges)[f_of] * per + rows % per
    sr.check_windows(host, rows, ref, False, f"{kind} {fh}x{fw} frames {edges}")
