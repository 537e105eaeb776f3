"""CPU-side checks of the region calls: the INTER_AREA taps the kernel computes (cnnacc_area_tab_host), the staging plan of
the host-pointer path (csrc/region_plan.h through cnnacc_region_plan_host), the refusals, and the pure-numpy helpers and
sort / unsort of the Python wrapper."""
import ctypes

import numpy as np
import pytest

import fpga_cnn_b200 as fc
from oracle import np_oracle

TAPS = 80
VGA = (480, 640)
VGA_BYTES = 480 * 640 * 3
CHUNK_BYTES = 16 << 20


@pytest.fixture(scope="module")
def lib():
    fc.build()
    return fc.load()


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _tab(lib, side):
    start, cnt = np.zeros(128, np.int32), np.zeros(128, np.int32)
    alpha = np.full((128, TAPS), -1, np.float32)
    taps = lib.cnnacc_area_tab_host(side, _p(start), _p(cnt), _p(alpha), TAPS)
    assert taps >= 1, side
    return taps, start, cnt, alpha


def _oracle_rows(side):
    rows = [[] for _ in range(128)]
    for d, s, a in np_oracle.area_tab(side, 128):
        rows[d].append((s, a))
    return rows


@pytest.mark.parametrize("sides", [range(128, 4097), [4099, 4500, 5000, 6001, 6143, 7777, 8000, 8190, 8191, 8192]],
                         ids=["128-4096", "to-8192"])
def test_area_taps_equal_opencv_table(lib, sides):
    for side in sides:
        taps, start, cnt, alpha = _tab(lib, side)
        assert taps == cnt.max()
        if side % 128 == 0:                                  # integer scales: k taps of weight 1 (kernels sum integers)
            k = side // 128
            assert (cnt == k).all() and (start == np.arange(128) * k).all() and (alpha[:, :k] == 1).all(), side
            continue
        for d, row in enumerate(_oracle_rows(side)):
            assert cnt[d] == len(row) and start[d] == row[0][0], (side, d)
            assert [s for s, _ in row] == list(range(start[d], start[d] + cnt[d])), (side, d)
            want = np.array([a for _, a in row], np.float32)
            assert np.array_equal(alpha[d, :cnt[d]].view(np.uint32), want.view(np.uint32)), (side, d)
            assert (alpha[d, cnt[d]:] == 0).all()


def test_area_tab_refusals(lib):
    start, cnt = np.zeros(128, np.int32), np.zeros(128, np.int32)
    alpha = np.zeros((128, TAPS), np.float32)
    for side in (127, 0, -5, 8193):
        assert lib.cnnacc_area_tab_host(side, _p(start), _p(cnt), _p(alpha), TAPS) == fc._lib.ERR_ARG
    assert lib.cnnacc_area_tab_host(8191, _p(start), _p(cnt), _p(alpha), 8) == fc._lib.ERR_ARG     # 65 taps do not fit 8
    assert lib.cnnacc_area_tab_host(8191, _p(start), _p(cnt), _p(alpha), TAPS) == 65


def _plan(lib, regions, n_frames, fh=VGA[0], fw=VGA[1], cap=100000):
    reg = np.ascontiguousarray(np.asarray(regions, np.int32).reshape(-1, 4))
    chunks = np.full((cap, 4), -7, np.int64)
    m = lib.cnnacc_region_plan_host(_p(reg), len(reg), n_frames, fh, fw, _p(chunks), cap)
    return m, chunks[:max(m, 0)]


def _check_plan(regions, chunks, frame_bytes):
    regions = np.asarray(regions).reshape(-1, 4)
    n = len(regions)
    assert chunks[0, 2] == 0 and chunks[-1, 3] == n
    assert (chunks[1:, 2] == chunks[:-1, 3]).all() and (chunks[:, 3] > chunks[:, 2]).all()   # every region exactly once
    staged = []
    for f0, f1, r0, r1 in chunks:
        fr = regions[r0:r1, 0]
        assert fr.min() == f0 and fr.max() == f1 - 1                 # the staged range is first .. last referenced frame
        assert set(range(f0, f1)) <= set(fr.tolist())                # and every staged frame is referenced
        assert (f1 - f0) * frame_bytes <= max(CHUNK_BYTES, frame_bytes)
        staged += list(range(f0, f1))
    return staged


def test_plan_stages_referenced_frames_once(lib):
    rng = np.random.default_rng(5)
    # 90 VGA frames: none on the first 5, the last 7 and a gap 40..44; uneven counts; frame 20 with 3000 regions
    counts = np.zeros(90, int)
    counts[5:83] = rng.integers(0, 4, 78)
    counts[40:45] = 0
    counts[20] = 3000
    counts[21] = 1
    g = fc.grid_regions(1, 480, 640, [128, 200, 333], [16, 50, 40])
    regions = []
    for f, c in enumerate(counts):
        for i in range(c):
            regions.append((f, *g[i % len(g), 1:]))
    regions = np.array(regions, np.int32)
    m, chunks = _plan(lib, regions, 90)
    assert m >= 1
    staged = _check_plan(regions, chunks, VGA_BYTES)
    referenced = sorted(set(regions[:, 0].tolist()))
    assert staged == referenced                                        # each referenced frame once; no other frame
    assert 0 not in staged and 89 not in staged and 42 not in staged
    big = [c for c in chunks if c[0] <= 20 < c[1]]
    assert len(big) == 1 and big[0][3] - big[0][2] >= 3000             # split over launches, never re-staged


def test_plan_of_one_region_per_frame_is_the_frame_chunks(lib):
    for fh, fw in ((480, 640), (128, 128), (1080, 1920), (4096, 4096)):
        n = 300
        fb = fh * fw * 3
        side = min(fh, fw)
        reg = np.array([(f, (fw - side) // 2, (fh - side) // 2, side) for f in range(n)], np.int32)
        m, chunks = _plan(lib, reg, n, fh, fw)
        per = max(1, CHUNK_BYTES // fb)
        want = [(i, min(n, i + per)) for i in range(0, n, per)]
        assert [(int(a), int(b)) for a, b in chunks[:, :2]] == want and (chunks[:, :2] == chunks[:, 2:]).all()


def test_plan_capacity_and_empty(lib):
    reg = np.array([(f, 0, 0, 128) for f in range(100)], np.int32)
    m, _ = _plan(lib, reg, 100)
    assert m == 6                                                      # 18 VGA frames per 16 MiB chunk
    assert _plan(lib, reg, 100, cap=5)[0] == fc._lib.ERR_ARG
    assert _plan(lib, np.zeros((0, 4), np.int32), 3)[0] == 0
    assert lib.cnnacc_region_plan_host(None, 0, 3, 480, 640, _p(np.zeros(4, np.int64)), 1) == 0
    assert lib.cnnacc_region_plan_host(None, 1, 3, 480, 640, _p(np.zeros(4, np.int64)), 1) == fc._lib.ERR_ARG


BAD_REGIONS = {
    "frame_negative": [(-1, 0, 0, 128)],
    "frame_too_big": [(0, 0, 0, 128), (3, 0, 0, 128)],
    "side_small": [(0, 0, 0, 127)],
    "side_big": [(0, 0, 0, 8193)],
    "x_negative": [(0, -1, 0, 128)],
    "y_negative": [(0, 0, -1, 128)],
    "x_past_edge": [(0, 513, 0, 128)],
    "y_past_edge": [(0, 0, 353, 128)],
    "side_past_edge": [(0, 0, 0, 481)],
    "decreasing": [(1, 0, 0, 128), (0, 0, 0, 128)],
    "overflow": [(0, 2 ** 31 - 100, 0, 200)],
}


@pytest.mark.parametrize("name", sorted(BAD_REGIONS))
def test_refusals(lib, name):
    reg = np.array(BAD_REGIONS[name], np.int32)
    assert _plan(lib, reg, 3)[0] == fc._lib.ERR_ARG              # the check the real calls run (tests/test_regions_gpu.py)


def test_region_edges_accepted(lib):
    ok = [(0, 0, 0, 480), (0, 160, 0, 480), (1, 512, 352, 128), (2, 0, 0, 128), (2, 511, 351, 129)]
    m, chunks = _plan(lib, ok, 3)
    assert m == 1 and tuple(chunks[0]) == (0, 3, 0, 5)


def test_grid_regions_vga_and_pyramid():
    g = fc.grid_regions(2, 480, 640, 128, 64)
    assert g.dtype == np.int32 and g.shape == (126, 4)
    assert (g[:63, 0] == 0).all() and (g[63:, 0] == 1).all()          # frame-major
    xs, ys = sorted(set(g[:63, 1])), sorted(set(g[:63, 2]))
    assert xs == list(range(0, 513, 64)) and ys == list(range(0, 321, 64)) + [352]   # flush edge only where missing
    p = fc.grid_regions(1, 480, 640, [480, 240, 128], [240, 120, 64])
    assert len(p) == 2 + 15 + 63
    assert [tuple(r) for r in p[:2]] == [(0, 0, 0, 480), (0, 160, 0, 480)]
    assert (p[:2, 3] == 480).all() and (p[2:17, 3] == 240).all() and (p[17:, 3] == 128).all()   # sides in the given order


@pytest.mark.parametrize("fh,fw,sides,strides", [(480, 640, [128, 200, 333], [64, 100, 150]), (300, 300, [128, 300], [7, 1]),
                                                 (720, 1280, [129, 719], [128, 1000])])
def test_grid_regions_cover_every_pixel(fh, fw, sides, strides):
    g = fc.grid_regions(3, fh, fw, sides, strides)
    assert (np.diff(g[:, 0]) >= 0).all()
    for side, stride in zip(sides, strides):
        t = g[(g[:, 0] == 1) & (g[:, 3] == side)]
        cover = np.zeros((fh, fw), bool)
        for _, x, y, s in t:
            assert 0 <= x and x + s <= fw and 0 <= y and y + s <= fh
            cover[y:y + s, x:x + s] = True
        assert cover.all(), (side, stride)
        assert len(set(map(tuple, t[:, 1:3].tolist()))) == len(t)
        rows = sorted(set(t[:, 2].tolist()))
        assert rows[0] == 0 and rows[-1] == fh - side
        assert all(b - a <= stride for a, b in zip(rows, rows[1:]))


def test_grid_regions_rejects_oversized_tiles():
    with pytest.raises(ValueError):
        fc.grid_regions(1, 480, 640, 481, 64)
    with pytest.raises(ValueError):
        fc.grid_regions(1, 480, 640, [128, 256], [64, 64, 64])


def test_region_boxes_to_frame():
    reg = np.array([(0, 10, 20, 128), (3, 100, 7, 256), (1, 5, 6, 333)], np.int32)
    box = np.array([(0, 0, 127, 127), (10, 20, 30, 40), (1, 2, 3, 4)], np.int32)
    got = fc.region_boxes_to_frame(reg, box)
    assert got.dtype == np.float64
    want = np.array([[10, 20, 137, 147], [120, 47, 160, 87],
                     [5 + 333 / 128, 6 + 2 * 333 / 128, 5 + 3 * 333 / 128, 6 + 4 * 333 / 128]])
    assert np.array_equal(got, want)


class _Recorder(fc.CNNAccelerator):
    """A CNNAccelerator without a device: the library call is replaced by one that records the regions it is given and
    writes, for each, values derived from the region itself."""

    def __init__(self):                                    # no cnnacc_create: nothing here touches a GPU
        self._n_cls = 3
        self.calls = []

    def _call_regions(self, frames_p, nf, fh, fw, reg, gray_p, outs_p, detect, flags):
        self.calls.append(reg.copy())
        n = len(reg)
        view = lambda p, ct, shape: np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ct)), shape=shape)
        key = reg[:, 0] * 100000 + reg[:, 1] * 100 + reg[:, 2]
        if detect:
            view(outs_p[0], ctypes.c_int32, (n,))[:] = key
            view(outs_p[1], ctypes.c_float, (n, 3))[:] = reg[:, 3:4]
            view(outs_p[2], ctypes.c_int32, (n, 4))[:] = reg
        if gray_p is not None:
            view(gray_p, ctypes.c_uint8, (n, 128, 128))[:] = (key % 251)[:, None, None]


def test_wrapper_sorts_by_frame_and_restores_the_callers_order():
    acc = _Recorder()
    rng = np.random.default_rng(3)
    reg = np.array([(f, x, y, 128 + x) for f in range(6) for x in range(4) for y in range(3)], np.int64)
    reg = reg[rng.permutation(len(reg))]
    frames = np.zeros((6, 300, 300, 3), np.uint8)
    cls, probs, box, gray = acc.detect_regions(frames, reg, return_gray=True)
    sent = acc.calls[-1]
    assert sent.dtype == np.int32 and sent.flags.c_contiguous
    assert (np.diff(sent[:, 0]) >= 0).all()
    same_frame = [sent[sent[:, 0] == f].tolist() for f in range(6)]
    assert same_frame == [reg[reg[:, 0] == f].tolist() for f in range(6)]    # stable within a frame
    assert np.array_equal(box, reg) and np.array_equal(cls, reg[:, 0] * 100000 + reg[:, 1] * 100 + reg[:, 2])
    assert np.array_equal(probs[:, 0], reg[:, 3]) and np.array_equal(gray[:, 5, 7], cls % 251)
    g = acc.preprocess_regions(frames, reg)
    assert np.array_equal(g, gray)
    acc.detect_regions(frames, sent)
    assert np.array_equal(acc.calls[-1], sent)                                 # already grouped: passed unchanged


def test_wrapper_rejects_malformed_region_arrays():
    acc = _Recorder()
    frames = np.zeros((1, 200, 200, 3), np.uint8)
    for bad in (np.zeros((3, 3), np.int32), np.zeros(4, np.int32), np.zeros((2, 4), np.float32), [(0, 0, 0, 2 ** 31)]):
        with pytest.raises(ValueError):
            acc.detect_regions(frames, bad)
    cls, probs, box = acc.detect_regions(frames, np.zeros((0, 4), np.int32))
    assert cls.shape == (0,) and probs.shape == (0, 3) and box.shape == (0, 4)
