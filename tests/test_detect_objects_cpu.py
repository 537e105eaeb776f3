"""CPU-side checks of the merge of region detections (csrc/region_merge.h): a plain numpy restatement of the rule, checked
against brute-force invariants, and cnnacc_merge_regions_host equal to it byte for byte on ties, IoU boundaries, signed zeros
and NaN scores, class-agnostic merging, max_det limits, empty frames, full frames, out-of-range boxes and seeded random sets;
every refusal; and the Python wrapper's mapping of region indices back to the caller's order."""
import ctypes

import numpy as np
import pytest

import fpga_cnn_b200 as fc


@pytest.fixture(scope="module")
def lib():
    fc.build()
    return fc.load()


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


# ---- the restatement ----------------------------------------------------------------------------------------------------

def frame_boxes(regions, bbox):
    """Boxes in 1/128 frame pixels as int64 (X1, Y1, X2, Y2), after clamping to the 128 grid."""
    b = np.clip(np.asarray(bbox, np.int64).reshape(-1, 4), 0, 127)
    reg = np.asarray(regions, np.int64).reshape(-1, 4)
    x, y, s = reg[:, 1:2], reg[:, 2:3], reg[:, 3:4]
    return np.concatenate([128 * x + b[:, 0:1] * s, 128 * y + b[:, 1:2] * s, 128 * x + b[:, 2:3] * s, 128 * y + b[:, 3:4] * s], 1)


def area(B):
    return np.maximum(B[..., 2] - B[..., 0], 0) * np.maximum(B[..., 3] - B[..., 1], 0)


def iou(A, B):
    """IoU of box A against each of boxes B: float64 division of exact int64 areas, 0 when the union is 0."""
    iw = np.minimum(A[2], B[:, 2]) - np.maximum(A[0], B[:, 0])
    ih = np.minimum(A[3], B[:, 3]) - np.maximum(A[1], B[:, 1])
    inter = np.maximum(iw, 0) * np.maximum(ih, 0)
    uni = area(A) + area(B) - inter
    out = np.zeros(len(B))
    np.divide(inter.astype(np.float64), uni.astype(np.float64), out=out, where=uni != 0)
    return out


def ranked_candidates(idx, scores, score_min):
    """Region indices of a frame that are candidates, by score descending then index ascending (-0.0 == +0.0, no NaN)."""
    s = scores[idx]
    cand = idx[s >= np.float32(score_min)]
    return cand[np.lexsort((cand, -(scores[cand].astype(np.float64) + 0.0)))]


def restate(regions, scores, cls, bbox, n_frames, score_min, iou_max, max_det, agnostic):
    """The merge rule in numpy -> (n_det, region, cls, score, box) as the library lays them out."""
    regions = np.asarray(regions, np.int32).reshape(-1, 4)
    scores, cls = np.asarray(scores, np.float32), np.asarray(cls, np.int32)
    B = frame_boxes(regions, bbox)
    im = np.float64(np.float32(iou_max))
    D = max_det
    n_det = np.zeros(n_frames, np.int32)
    d_reg, d_cls = np.full((n_frames, D), -1, np.int32), np.full((n_frames, D), -1, np.int32)
    d_score, d_box = np.zeros((n_frames, D), np.float32), np.zeros((n_frames, D, 4), np.float32)
    for f in range(n_frames):
        kept = []
        for r in ranked_candidates(np.flatnonzero(regions[:, 0] == f), scores, score_min):
            if len(kept) >= D:
                break
            k = np.array(kept, np.int64)
            if not agnostic:
                k = k[cls[k] == cls[r]]
            if len(k) and (iou(B[r], B[k]) > im).any():
                continue
            kept.append(r)
        n = len(kept)
        n_det[f] = n
        d_reg[f, :n], d_cls[f, :n], d_score[f, :n] = kept, cls[kept], scores[kept]
        d_box[f, :n] = (B[kept] / 128.0).astype(np.float32)
    return n_det, d_reg, d_cls, d_score, d_box


def merge_host(lib, regions, scores, cls, bbox, n_frames, score_min, iou_max, max_det, agnostic, flags=0):
    regions = np.ascontiguousarray(np.asarray(regions, np.int32).reshape(-1, 4))
    scores, cls = np.ascontiguousarray(scores, np.float32), np.ascontiguousarray(cls, np.int32)
    bbox = np.ascontiguousarray(np.asarray(bbox, np.int32).reshape(-1, 4))
    D = max(int(max_det), 1)
    out = (np.full(n_frames, -9, np.int32), np.full((n_frames, D), -9, np.int32), np.full((n_frames, D), -9, np.int32),
           np.full((n_frames, D), -9, np.float32), np.full((n_frames, D, 4), -9, np.float32))
    flags |= fc._lib.FLAG_CLASS_AGNOSTIC if agnostic else 0
    rc = lib.cnnacc_merge_regions_host(_p(regions), len(regions), n_frames, _p(scores), _p(cls), _p(bbox), score_min, iou_max,
                                       max_det, *[_p(a) for a in out], flags)
    return rc, out


def assert_same(got, want, what=""):
    for i, (g, w) in enumerate(zip(got, want)):
        g, w = np.asarray(g), np.asarray(w)
        assert g.dtype == w.dtype and g.shape == w.shape, (what, i, g.dtype, w.dtype, g.shape, w.shape)
        assert np.array_equal(g.view(np.uint8), w.view(np.uint8)), (what, i)


# ---- the cases (tests/test_detect_objects_gpu.py runs the same ones on the device) --------------------------------------

def _case(regions, scores, cls, bbox, n_frames, score_min=0.0, iou_max=0.5, max_det=100, agnostic=False):
    return dict(regions=np.asarray(regions, np.int32).reshape(-1, 4), scores=np.asarray(scores, np.float32),
                cls=np.asarray(cls, np.int32), bbox=np.asarray(bbox, np.int32).reshape(-1, 4), n_frames=n_frames,
                score_min=score_min, iou_max=iou_max, max_det=max_det, agnostic=agnostic)


def random_case(seed, n_frames, max_per_frame, n_cls=6, max_det=100, agnostic=False, iou_max=0.5, score_min=0.2):
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, max_per_frame + 1, n_frames)
    counts[rng.choice(n_frames, max(1, n_frames // 10), replace=False)] = 0
    f = np.repeat(np.arange(n_frames), counts)
    n = len(f)
    side = rng.choice([128, 160, 200, 256, 333, 480], n)
    x, y = rng.integers(0, 641, n), rng.integers(0, 481, n)
    regions = np.stack([f, x, y, side], 1)
    b1 = rng.integers(-5, 120, (n, 2))
    b2 = b1 + rng.integers(-3, 70, (n, 2))
    bbox = np.concatenate([b1, b2], 1)
    scores = rng.choice(np.float32([0.0, 0.25, 0.5, 0.75, 1.0]), n) if seed % 2 else rng.random(n, np.float32)
    return _case(regions, scores, rng.integers(0, n_cls, n), bbox, n_frames, score_min, iou_max, max_det, agnostic)


def cases():
    half = np.nextafter(np.float32(0.5), np.float32(0))
    c = {}
    # the same region four times in each of two classes: exact score ties, broken by region index
    reg = [(0, 10, 20, 256)] * 8 + [(1, 0, 0, 128)] * 3
    c["duplicates"] = _case(reg, [0.5] * 8 + [0.9] * 3, [1, 2] * 4 + [0, 0, 0], [(10, 10, 90, 90)] * 8 + [(0, 0, 127, 127)] * 3, 2)
    # IoU exactly 1/2: kept at iou_max = 0.5, suppressed just below it
    reg = [(0, 0, 0, 128), (0, 0, 0, 128), (0, 64, 32, 256), (0, 64, 32, 256)]
    box = [(0, 0, 60, 60), (0, 20, 60, 80), (0, 0, 30, 30), (0, 10, 30, 40)]
    c["iou_half_kept"] = _case(reg, [0.9, 0.8, 0.7, 0.6], [0, 0, 1, 1], box, 1, iou_max=0.5)
    c["iou_half_suppressed"] = _case(reg, [0.9, 0.8, 0.7, 0.6], [0, 0, 1, 1], box, 1, iou_max=float(half))
    # signed zeros, NaN, -inf and a score equal to score_min
    nan = np.float32("nan")
    reg = [(0, 0, 0, 128)] * 8
    sc = [-0.0, 0.0, nan, -0.0, 0.25, np.float32(-np.inf), 0.0, nan]
    box = [(i * 10, 0, i * 10 + 9, 9) for i in range(8)]
    c["signed_zero_nan"] = _case(reg, sc, [0] * 8, box, 1, score_min=0.0)
    c["signed_zero_nan_neg_min"] = _case(reg, sc, [0] * 8, box, 1, score_min=-np.inf)
    c["score_equals_min"] = _case(reg, [0.25, 0.2500001, 0.2499999, 0.25, 1, 0, 0.25, 0.3], [0] * 8, box, 1, score_min=0.25)
    # overlapping boxes of different classes: kept per class, merged class-agnostic
    reg = [(0, 0, 0, 128)] * 6
    box = [(0, 0, 100, 100), (2, 2, 100, 100), (4, 4, 100, 100), (0, 0, 99, 99), (50, 50, 127, 127), (52, 50, 127, 127)]
    for ag in (False, True):
        c[f"classes_agnostic_{ag}"] = _case(reg, [0.9, 0.8, 0.7, 0.6, 0.5, 0.4], [0, 1, 2, 0, 1, 1], box, 1, agnostic=ag)
    # max_det 1, and 1024 of 1100 disjoint boxes (merge_regions has no frame size: regions far apart)
    c["max_det_1"] = _case(reg, [0.1, 0.9, 0.5, 0.9, 0.2, 0.3], [0, 1, 2, 0, 1, 1], box, 1, max_det=1)
    n = 1100
    reg = np.stack([np.zeros(n, int), np.arange(n) * 200, np.zeros(n, int), np.full(n, 128)], 1)
    c["max_det_1024"] = _case(reg, np.linspace(0, 1, n)[::-1], np.zeros(n), np.tile([0, 0, 127, 127], (n, 1)), 1, max_det=1024)
    # frames without regions before, between and after
    reg = [(2, 0, 0, 128), (2, 5, 5, 200), (4, 0, 0, 128)]
    c["empty_frames"] = _case(reg, [0.5, 0.6, 0.7], [1, 1, 1], [(0, 0, 50, 50), (0, 0, 50, 50), (1, 1, 2, 2)], 7)
    c["no_regions"] = _case(np.zeros((0, 4)), [], [], np.zeros((0, 4)), 3)
    # out-of-range box coordinates are clamped; inverted boxes have zero area (union 0 between two of them)
    reg = [(0, 0, 0, 128), (0, 0, 0, 128), (0, 0, 0, 256), (0, 0, 0, 256), (0, 3, 4, 8192)]
    box = [(-50, -1, 300, 128), (0, 0, 127, 127), (90, 90, 10, 10), (90, 90, 10, 10), (-2**31, 2**31 - 1, 2**31 - 1, -2**31)]
    c["out_of_range_boxes"] = _case(reg, [0.5, 0.4, 0.9, 0.8, 0.7], [0, 0, 0, 0, 0], box, 1, iou_max=0.0)
    # 16384 regions in one frame: a stride-8 grid of 128-side tiles with jittered boxes
    rng = np.random.default_rng(11)
    xs, ys = np.meshgrid(np.arange(128) * 8, np.arange(128) * 8)
    reg = np.stack([np.zeros(16384, int), xs.ravel(), ys.ravel(), np.full(16384, 128)], 1)
    b1 = rng.integers(0, 40, (16384, 2))
    c["full_frame"] = _case(np.concatenate([reg, [(1, 0, 0, 128)]]), rng.random(16385, np.float32),
                            rng.integers(0, 3, 16385), np.concatenate([np.concatenate([b1, b1 + 80], 1), [(0, 0, 1, 1)]]), 2,
                            max_det=1024, iou_max=0.3)
    for seed in range(4):
        c[f"random_{seed}"] = random_case(seed, (200, 60, 40, 40)[seed], (3000, 3000, 400, 400)[seed], agnostic=seed == 3,
                                          max_det=(100, 300, 1024, 7)[seed], iou_max=(0.5, 0.3, 0.7, 0.45)[seed])
    return c


CASES = cases()


# ---- the restatement against brute force ---------------------------------------------------------------------------------

@pytest.mark.parametrize("name", sorted(CASES))
def test_restatement_invariants(name):
    c = CASES[name]
    reg, sc, cl = c["regions"], c["scores"], c["cls"]
    n_det, d_reg, d_cls, d_score, d_box = restate(**c)
    B = frame_boxes(reg, c["bbox"])
    im = np.float64(np.float32(c["iou_max"]))
    for f in range(c["n_frames"]):
        kept = d_reg[f, :n_det[f]]
        assert (d_reg[f, n_det[f]:] == -1).all() and (d_cls[f, n_det[f]:] == -1).all()
        assert (d_score[f, n_det[f]:] == 0).all() and (d_box[f, n_det[f]:] == 0).all()
        assert (reg[kept, 0] == f).all() and np.array_equal(d_cls[f, :n_det[f]], cl[kept])
        for i, r in enumerate(kept):                       # no two kept boxes of a class overlap beyond iou_max
            others = kept[i + 1:]
            if not c["agnostic"]:
                others = others[cl[others] == cl[r]]
            assert not (iou(B[r], B[others]) > im).any(), (f, r)
        ranked = list(ranked_candidates(np.flatnonzero(reg[:, 0] == f), sc, c["score_min"]))
        kept_set = set(kept.tolist())
        rank = {r: i for i, r in enumerate(ranked)}
        kept_rank = np.array([rank[r] for r in kept], np.int64)
        assert (np.diff(kept_rank) > 0).all()                                        # kept in rank order
        full_at = kept_rank[-1] if n_det[f] == c["max_det"] else len(ranked)
        for pos, r in enumerate(ranked):                   # every dropped candidate was suppressed, or max_det was reached
            if r in kept_set or pos > full_at:
                continue
            before = kept[kept_rank < pos].astype(np.int64)
            if not c["agnostic"]:
                before = before[cl[before] == cl[r]]
            assert len(before) and (iou(B[r], B[before]) > im).any(), (f, r)
        not_cand = np.flatnonzero(reg[:, 0] == f)
        not_cand = not_cand[~(sc[not_cand] >= np.float32(c["score_min"]))]
        assert not set(not_cand.tolist()) & set(kept.tolist())


def test_restatement_boundary_cases():
    assert restate(**CASES["iou_half_kept"])[0][0] == 4
    assert restate(**CASES["iou_half_suppressed"])[0][0] == 2
    n, reg, *_ = restate(**CASES["duplicates"])
    assert list(reg[0, :n[0]]) == [0, 1] and list(reg[1, :n[1]]) == [8]      # ties: the lowest index wins
    n, reg, *_ = restate(**CASES["signed_zero_nan"])
    assert list(reg[0, :n[0]]) == [4, 0, 1, 3, 6]                            # +0.0 and -0.0 tie; NaN and -inf never candidates
    assert list(restate(**CASES["signed_zero_nan_neg_min"])[1][0, :6]) == [4, 0, 1, 3, 6, 5]
    assert restate(**CASES["max_det_1024"])[0][0] == 1024
    assert restate(**CASES["classes_agnostic_False"])[0][0] > restate(**CASES["classes_agnostic_True"])[0][0]
    n, reg, *_ = restate(**CASES["empty_frames"])
    assert list(n) == [0, 0, 2, 0, 1, 0, 0]
    n, reg, cls, score, box = restate(**CASES["out_of_range_boxes"])
    assert list(reg[0, :n[0]]) == [2, 3, 4, 0] and (box[0, 3] == [0, 0, 127, 127]).all()


def test_boxes_equal_region_boxes_to_frame():
    c = CASES["random_0"]
    inside = (c["bbox"] >= 0).all(1) & (c["bbox"] <= 127).all(1)
    want = fc.region_boxes_to_frame(c["regions"][inside], c["bbox"][inside]).astype(np.float32)
    got = (frame_boxes(c["regions"][inside], c["bbox"][inside]) / 128.0).astype(np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


# ---- the library's CPU replay against the restatement ----------------------------------------------------------------------

@pytest.mark.parametrize("name", sorted(CASES))
def test_merge_regions_host_equals_restatement(lib, name):
    c = CASES[name]
    rc, got = merge_host(lib, **c)
    assert rc == 0
    assert_same(got, restate(**c), name)


def test_null_optional_outputs(lib):
    c = CASES["random_1"]
    reg, sc, cl, bb = c["regions"], c["scores"], c["cls"], c["bbox"]
    n_det = np.zeros(c["n_frames"], np.int32)
    assert lib.cnnacc_merge_regions_host(_p(reg), len(reg), c["n_frames"], _p(sc), _p(cl), _p(bb), 0.2, 0.3, 300, _p(n_det),
                                         None, None, None, None, 0) == 0
    assert np.array_equal(n_det, restate(**c)[0])


def _refusal_args():
    ok = dict(regions=[(0, 0, 0, 128), (1, 5, 5, 200)], scores=[0.5, 0.5], cls=[0, 0], bbox=[(0, 0, 9, 9)] * 2, n_frames=2,
              score_min=0.0, iou_max=0.5, max_det=10, agnostic=False)
    bad = {"max_det_0": dict(max_det=0), "max_det_1025": dict(max_det=1025), "iou_nan": dict(iou_max=float("nan")),
           "iou_negative": dict(iou_max=-0.1), "iou_above_1": dict(iou_max=1.5),
           "frame_negative": dict(regions=[(-1, 0, 0, 128), (1, 0, 0, 128)]),
           "frame_too_big": dict(regions=[(0, 0, 0, 128), (2, 0, 0, 128)]),
           "decreasing": dict(regions=[(1, 0, 0, 128), (0, 0, 0, 128)]), "side_small": dict(regions=[(0, 0, 0, 127), (1, 0, 0, 128)]),
           "side_big": dict(regions=[(0, 0, 0, 8193), (1, 0, 0, 128)]), "x_negative": dict(regions=[(0, -1, 0, 128), (1, 0, 0, 128)]),
           "y_negative": dict(regions=[(0, 0, -1, 128), (1, 0, 0, 128)])}
    n = 16385
    bad["frame_over_16384"] = dict(regions=np.tile([0, 0, 0, 128], (n, 1)), scores=np.zeros(n), cls=np.zeros(n),
                                   bbox=np.zeros((n, 4)), n_frames=1)
    return ok, bad


REFUSAL_OK, REFUSALS = _refusal_args()


@pytest.mark.parametrize("name", sorted(REFUSALS))
def test_refusals(lib, name):
    rc, _ = merge_host(lib, **{**REFUSAL_OK, **REFUSALS[name]})
    assert rc == fc._lib.ERR_ARG


def test_refusals_of_pointers_and_flags(lib):
    rc, _ = merge_host(lib, **REFUSAL_OK)
    assert rc == 0
    assert merge_host(lib, **REFUSAL_OK, flags=fc._lib.FLAG_DEVICE_PTRS)[0] == fc._lib.ERR_ARG
    reg = np.array(REFUSAL_OK["regions"], np.int32)
    sc, cl, bb = np.zeros(2, np.float32), np.zeros(2, np.int32), np.zeros((2, 4), np.int32)
    nd = np.zeros(2, np.int32)
    call = lambda *a: lib.cnnacc_merge_regions_host(*a, 0.0, 0.5, 10, *[None] * 5, 0)
    assert lib.cnnacc_merge_regions_host(_p(reg), 2, 2, _p(sc), _p(cl), _p(bb), 0.0, 0.5, 10, None, None, None, None, None, 0) \
        == fc._lib.ERR_ARG                                                    # n_det is required
    args = [_p(reg), 2, 2, _p(sc), _p(cl), _p(bb)]
    for i in (0, 3, 4, 5):                                                    # NULL regions / scores / cls / bbox
        a = list(args)
        a[i] = None
        assert lib.cnnacc_merge_regions_host(*a, 0.0, 0.5, 10, _p(nd), None, None, None, None, 0) == fc._lib.ERR_ARG
    assert lib.cnnacc_merge_regions_host(_p(reg), 2, -1, _p(sc), _p(cl), _p(bb), 0.0, 0.5, 10, _p(nd), None, None, None, None,
                                         0) == fc._lib.ERR_ARG
    assert call(None, 0, 0, None, None, None) == fc._lib.ERR_ARG             # n_det NULL even for an empty call
    assert lib.cnnacc_merge_regions_host(None, 0, 0, None, None, None, 0.0, 0.5, 10, _p(nd), None, None, None, None, 0) == 0


# ---- the wrapper's region order --------------------------------------------------------------------------------------------

class _Recorder(fc.CNNAccelerator):
    """A CNNAccelerator without a device whose merge call is the CPU replay."""

    def __init__(self):
        self._libc = fc.load()
        self._h = None
        self.sent = None

    def _check(self, rc):
        fc._lib.check(rc)


def test_wrapper_maps_regions_back_to_the_callers_order(lib):
    c = random_case(21, 12, 60)
    acc = _Recorder()
    libc = acc._libc

    class Shim:                                    # route the device call to the host replay
        def __getattr__(self, name):
            return getattr(libc, name)

        @staticmethod
        def cnnacc_merge_regions(h, *a):
            return libc.cnnacc_merge_regions_host(*a)
    acc._libc = Shim()
    perm = np.random.default_rng(4).permutation(len(c["regions"]))
    shuffled = {**c, **{k: c[k][perm] for k in ("regions", "scores", "cls", "bbox")}}
    got = acc.merge_regions(shuffled["regions"], shuffled["cls"], shuffled["scores"], shuffled["bbox"], c["n_frames"],
                            score_min=c["score_min"], iou_max=c["iou_max"], max_det=c["max_det"])
    # the restatement on the caller's own (ungrouped) order: indices and tie-breaks are the caller's
    assert_same(got, restate(**shuffled))
    assert (got[0] > 0).any() and len(np.unique(shuffled["scores"])) < len(perm)      # ties present
    with pytest.raises(ValueError):
        acc.merge_regions(c["regions"], c["cls"], c["scores"], c["bbox"], c["n_frames"], max_det=0)
