"""Oracle references for the scanning calls at the frame sizes they serve (tests/test_scan_reference_gpu.py).  TEST
INFRASTRUCTURE.

  oracle_maps      the oracle's [64][h/8][w/8] feature maps of whole frames or levels: oracle.port_infer_batch at 32 bits,
                   np_oracle.infer(acc_bits=24) at 24, cut into row bands that run on a process pool and are stitched back
  select_windows   which windows of a level to check where checking all of them costs too much in the numpy tail
  check_windows    a call's predictions against the oracle's tail on those windows (test_paths_gpu.check_predictions)
  assert_exposed   that a case can fail at all: informative map bytes, several classes, boxes other than the full window

An output cell o of the conv stack depends on input rows 8o-7 .. 8o+14 and on the zero padding at the image border
(csrc/tiling.cuh).  A band of whole 16-row groups computed with 16 rows (2 cells) of frame above and below it, clipped at the
frame edge, therefore holds the whole-frame oracle's cells once those 2 halo cells are dropped on each inner side:
tests/test_scan_reference_cpu.py checks the stitched maps against the whole-frame oracle."""
import multiprocessing as mp

import numpy as np

import oracle
import scan_oracle
from oracle import np_oracle
from test_paths_gpu import check_predictions

BAND = 256                 # rows per band (a multiple of 16)
HALO = 16                  # rows of frame on each side of a band: 2 output cells
ALL_WINDOWS = 4096         # levels with at most this many windows are checked at every window
N_RANDOM = 384             # seeded random windows on larger levels, on top of the structured ones
FULL_BOX = (0, 0, 127, 127)


def bands(H, band=BAND):
    """[(r0, r1, a, b)]: output rows [r0, r1) of a frame of H rows, computed from input rows [a, b)."""
    assert band % 16 == 0 and H % 16 == 0
    return [(r0, min(H, r0 + band), max(0, r0 - HALO), min(H, r0 + band + HALO)) for r0 in range(0, H, band)]


def _maps_job(job):
    slab, weights, shifts, bits = job
    h, w = slab.shape
    if bits == 32:
        m = oracle.port_infer_batch(oracle.load_port(), slab[None], weights, shifts, h, w)
    else:
        m = np_oracle.infer(slab, np_oracle.unpack_weights(weights), shifts, H=h, W=w, acc_bits=24)
    return m.reshape(64, h // 8, w // 8)


def oracle_maps(gray, weights, shifts, bits, band=BAND, workers=None):
    """[64][h/8][w/8] u8 oracle maps of an (h, w) gray image, or [F][64][h/8][w/8] of (F, h, w) images, at 32 or 24 bits.
    Every image is cut into row bands (bands()) that run on a `fork` pool of up to 32 processes."""
    g = np.asarray(gray, dtype=np.uint8)
    one = g.ndim == 2
    g = g.reshape((-1,) + g.shape[-2:])
    F, H, W = g.shape
    jobs, where = [], []
    for f in range(F):
        for r0, r1, a, b in bands(H, band):
            jobs.append((np.ascontiguousarray(g[f, a:b]), weights, tuple(shifts), bits))
            where.append((f, r0, r1, a))
    n = min(workers or mp.cpu_count(), 32, len(jobs))
    if n <= 1:
        parts = [_maps_job(j) for j in jobs]
    else:
        with mp.get_context("fork").Pool(n) as pool:
            parts = pool.map(_maps_job, jobs, chunksize=1)
    out = np.empty((F, 64, H // 8, W // 8), np.uint8)
    for (f, r0, r1, a), m in zip(where, parts):
        out[f, :, r0 // 8:r1 // 8] = m[:, (r0 - a) // 8:(r1 - a) // 8]
    return out[0] if one else out


def tile_seams(n_out):
    """The first output cell of every conv tile but the first along a map side of n_out cells (cnnacc_tile_plan_host)."""
    import ctypes
    import fpga_cnn_b200 as fc
    g, s, e = (np.zeros(80, np.int32) for _ in range(3))
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)      # noqa: E731
    k = fc._lib.load().cnnacc_tile_plan_host(int(n_out), p(g), p(s), p(e), 80)
    assert k >= 1, n_out
    return [int(v) for v in s[1:k]]


def select_windows(h, w, stride, seed=0, all_windows=ALL_WINDOWS, n_random=N_RANDOM):
    """Indices, in the level's window order (y, then x), of the windows of an h x w level at `stride` to check.  Every window
    when there are at most `all_windows`; else the four corners, the whole last row and last column (the windows made flush
    with the far edges), 16 consecutive x origins of one row (at stride 8 they are 16 consecutive cells: every byte shift of
    the tail's 16-byte row gather), for every conv tile seam along x (y) a window with that seam near its middle, the seams
    paired along the diagonal, and n_random seeded random windows."""
    ys, xs = scan_oracle.origins(h, stride), scan_oracle.origins(w, stride)
    ny, nx = len(ys), len(xs)
    if ny * nx <= all_windows:
        return np.arange(ny * nx)
    sel = {(0, 0), (0, nx - 1), (ny - 1, 0), (ny - 1, nx - 1)}
    sel.update((ny - 1, ix) for ix in range(nx))
    sel.update((iy, nx - 1) for iy in range(ny))
    x0 = max(0, min(nx - 16, nx // 2 - 8))
    sel.update((ny // 2, ix) for ix in range(x0, min(nx, x0 + 16)))

    def straddling(origins, seams):
        cells = np.asarray(origins) // 8
        return [int(np.argmin(np.abs(cells + 8 - s))) for s in seams]
    sx, sy = straddling(xs, tile_seams(w // 8)), straddling(ys, tile_seams(h // 8))
    sel.update((ny // 3, ix) for ix in sx)
    sel.update((iy, nx // 3) for iy in sy)
    sel.update(zip(sy, sx))
    idx = {iy * nx + ix for iy, ix in sel}
    idx.update(np.random.default_rng(seed).choice(ny * nx, min(n_random, ny * nx), replace=False).tolist())
    return np.array(sorted(idx), np.int64)


def flush_windows(h, w, stride):
    """Indices of the windows whose origin is clamped to the far edge on either axis (the header's flush windows)."""
    ys, xs = scan_oracle.origins(h, stride), scan_oracle.origins(w, stride)
    nx = len(xs)
    return {iy * nx + ix for iy, y in enumerate(ys) for ix, x in enumerate(xs) if (h - 128) % stride and y == h - 128 or
            (w - 128) % stride and x == w - 128}


def level_windows(maps, h, w, stride, idx):
    """[len(idx)][64][16][16]: windows idx of one level's map [64][h/8][w/8]."""
    wins = scan_oracle.windows(1, h, w, stride)[idx]
    return scan_oracle.window_maps(maps[None], wins)


def tail(wmaps, fc_w, fc_b):
    """The oracle's predictions on window maps -> [(cls, probs, logits, bbox_vec box, None)] as check_predictions takes."""
    cls, probs, logits, box = scan_oracle.tail(wmaps, fc_w, fc_b)
    return [(int(c), p, lg, tuple(int(v) for v in b), None) for c, p, lg, b in zip(cls, probs, logits, box)]


def check_windows(got, rows, ref, logits, what):
    """got: a call's (cls, probs, bbox) over all its windows; rows: the windows ref describes."""
    cls, probs, box = (np.asarray(a.cpu() if hasattr(a, "cpu") else a) for a in got)
    check_predictions((cls[rows], probs[rows], box[rows]), ref, "vec", logits, what)


def assert_exposed(maps, ref, min_inside, what):
    """A case that cannot fail passes vacuously: hold its oracle maps to min_inside bytes strictly inside (0, 255), and its
    checked windows to at least two classes and to boxes that are not all the full window."""
    inside = float(((maps > 0) & (maps < 255)).mean())
    assert inside >= min_inside, f"{what}: {inside:.3f} of the map bytes inside (0, 255)"
    assert len({r[0] for r in ref}) >= 2, f"{what}: every checked window has class {ref[0][0]}"
    assert any(r[3] != FULL_BOX for r in ref), f"{what}: every checked box is the full window"
