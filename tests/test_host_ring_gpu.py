"""Host-pointer calls that reuse a staging slot: more chunks than the ring's four slots, so every slot is taken a second time
and its "slot free" wait is on the path.  Each call's result must equal calls of at most one chunk each (or the
device-pointer call), and the call must launch exactly one kernel per chunk (two with upsampled boxes from images)."""
import numpy as np
import pytest

import inputs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def acc(shipped_weights):
    import fpga_cnn_b200 as fc
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    a.load_classifier(*inputs.make_fc(seed=11))
    yield a
    a.close()


def _launches(acc, fn, *args, **kw):
    before = acc.launch_count
    out = fn(*args, **kw)
    return out, acc.launch_count - before


def _pieces(n, step):
    return [(i, min(i + step, n)) for i in range(0, n, step)]


def test_pool_features_reuses_slots(acc):
    n = 9000                                                          # 5 chunks of <= 2048
    feats = inputs.make_features(("rng", 90), n)
    got, launches = _launches(acc, acc.pool_features, feats)
    assert launches == 5
    want = np.concatenate([acc.pool_features(feats[a:b]) for a, b in _pieces(n, 2048)])
    assert np.array_equal(got, want)


def test_cam_bbox_batch_reuses_slots(acc):
    n = 16500                                                         # 5 chunks of <= 4096
    feats = inputs.make_features(("blob", 91), n)
    cls = np.random.default_rng(91).integers(0, 6, n).astype(np.int32)
    (box, cam), launches = _launches(acc, acc.cam_bbox_batch, feats, cls, return_cam=True)
    assert launches == 5
    parts = [acc.cam_bbox_batch(feats[a:b], cls[a:b], return_cam=True) for a, b in _pieces(n, 4096)]
    assert np.array_equal(box, np.concatenate([p[0] for p in parts]))
    assert np.array_equal(cam, np.concatenate([p[1] for p in parts]))


@pytest.mark.parametrize("bbox, per_chunk", [("vec", 1), ("upsampled", 2)])
def test_infer_batch_host_reuses_slots(acc, bbox, per_chunk):
    import torch
    n = 10000                                                         # 5 chunks of <= 2048
    imgs = inputs.make_images(("rng", 92), n)
    (cls, probs, box), launches = _launches(acc, acc.infer_batch, imgs, bbox=bbox)
    assert launches == 5 * per_chunk
    cls_d, probs_d, box_d = acc.infer_batch(torch.from_numpy(imgs).cuda(), bbox=bbox)
    assert np.array_equal(cls, cls_d.cpu().numpy())
    assert np.array_equal(probs, probs_d.cpu().numpy())
    assert np.array_equal(box, box_d.cpu().numpy())


def test_classify_and_bbox_batch_host_reuse_slots(acc):
    import torch
    n = 10000                                                         # 5 chunks of <= 2048
    feats = inputs.make_features(("rng", 93), n)
    (cls, probs, box), launches = _launches(acc, acc.classify_batch, feats)
    assert launches == 5
    cls_d, probs_d, box_d = acc.classify_batch(torch.from_numpy(feats).cuda())
    assert np.array_equal(cls, cls_d.cpu().numpy())
    assert np.array_equal(probs, probs_d.cpu().numpy())
    assert np.array_equal(box, box_d.cpu().numpy())
    given = np.random.default_rng(93).integers(0, 6, n).astype(np.int32)   # CNNACC_FLAG_CLS_GIVEN: classes go in per chunk
    box_g, launches = _launches(acc, acc.bbox_batch, feats, given)
    assert launches == 5
    assert np.array_equal(box_g, np.concatenate([acc.bbox_batch(feats[a:b], given[a:b]) for a, b in _pieces(n, 2048)]))
