"""CPU-side checks of the sharded host-batch calls: the shard plan (csrc/shard_plan.h through cnnacc_shard_plan_host) and the
refusals that need no GPU."""
import ctypes

import numpy as np
import pytest

import fpga_cnn_b200 as fc

CAP = 16


@pytest.fixture(scope="module")
def lib():
    fc.build()
    return fc.load()


def _plan(lib, n, n_handles, unit_bytes):
    begin = np.full(CAP, -7, np.int64)
    m = lib.cnnacc_shard_plan_host(n, n_handles, unit_bytes, begin.ctypes.data_as(ctypes.c_void_p), CAP)
    assert m >= 1, (n, n_handles, unit_bytes, m)
    assert (begin[m + 1:] == -7).all()                   # writes begin[0 .. m] only
    return m, [int(v) for v in begin[:m + 1]]


def min_shard_bytes(lib):
    """kMinShardBytes, recovered from the plan: with unit_bytes = 1 two members are used from n = 2 * kMinShardBytes on."""
    lo, hi = 1, 1 << 40
    while lo < hi:
        mid = (lo + hi) // 2
        if _plan(lib, mid, 2, 1)[0] == 2:
            hi = mid
        else:
            lo = mid + 1
    return lo // 2


def test_plans_cover_every_call_once(lib):
    k = min_shard_bytes(lib)
    assert k >= 1 and _plan(lib, 2 * k - 1, 2, 1)[0] == 1
    rng = np.random.default_rng(0)
    ns = list(range(0, 3000)) + [int(v) for v in rng.integers(3000, 1 << 31, 200)] + [(1 << 31) - 1, 1 << 31]
    for unit in (1, 4096, 16384, 65536, 640 * 480 * 3):
        for n in ns:
            for n_handles in range(1, 9):
                m, begin = _plan(lib, n, n_handles, unit)
                assert m == min(n_handles, max(1, n * unit // k)), (n, n_handles, unit, m)
                assert begin[0] == 0 and begin[-1] == n
                sizes = np.diff(begin)
                assert (sizes >= 0).all()                                   # ascending, contiguous, [0, n) exactly once
                assert sizes.max() - sizes.min() <= 1, (n, n_handles, unit, begin)
                assert begin == [n * i // m for i in range(m + 1)]          # bench.py's shard_range
                if n == 0:
                    assert m == 1 and begin == [0, 0]


def test_plan_rejects_bad_arguments(lib):
    begin = np.zeros(CAP, np.int64)
    p = begin.ctypes.data_as(ctypes.c_void_p)
    assert lib.cnnacc_shard_plan_host(-1, 2, 16384, p, CAP) < 0
    assert lib.cnnacc_shard_plan_host(10, 0, 16384, p, CAP) < 0
    assert lib.cnnacc_shard_plan_host(10, -3, 16384, p, CAP) < 0
    assert lib.cnnacc_shard_plan_host(10, 2, 0, p, CAP) < 0
    assert lib.cnnacc_shard_plan_host(10, 2, 16384, None, CAP) < 0
    n = 1 << 30                                                             # uses all 8 members: needs 9 entries
    assert lib.cnnacc_shard_plan_host(n, 8, 16384, p, 8) < 0
    assert lib.cnnacc_shard_plan_host(n, 8, 16384, p, 9) == 8
    assert lib.cnnacc_shard_plan_host(0, 8, 16384, p, 1) < 0 and lib.cnnacc_shard_plan_host(0, 8, 16384, p, 2) == 1


def test_sharded_calls_refuse_missing_members(lib):
    img = np.zeros((4, 128, 128), np.uint8)
    out = np.zeros((4, 64, 16, 16), np.uint8)
    probs = np.zeros((4, 16), np.float32); cls = np.zeros(4, np.int32); box = np.zeros((4, 4), np.int32)
    frames = np.zeros((4, 480, 640, 3), np.uint8); gray = np.zeros((4, 128, 128), np.uint8)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    empty = (ctypes.c_void_p * 1)()
    for hs, k in ((None, 2), (empty, 0), (empty, -1), (empty, 1)):          # NULL array, no members, a NULL member
        failed = ctypes.c_int(99)
        assert lib.cnnacc_run_batch_sharded(hs, k, p(img), 4, 128, 128, p(out), 0, ctypes.byref(failed)) == fc._lib.ERR_ARG
        assert failed.value == (0 if k == 1 else -1)
        assert lib.cnnacc_infer_batch_sharded(hs, k, p(img), 4, p(probs), p(cls), p(box), 0, None) == fc._lib.ERR_ARG
        assert lib.cnnacc_detect_frames_sharded(hs, k, p(frames), 4, 480, 640, p(gray), p(probs), p(cls), p(box), 0,
                                                None) == fc._lib.ERR_ARG


def test_multi_accelerator_needs_a_gpu(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CUDA device"):
        fc.MultiAccelerator()
    with pytest.raises(RuntimeError, match="no CUDA device"):
        fc.MultiAccelerator([0, 0])
