"""Every CUDA resource a handle grows is released with it: handles that run calls touching every workspace, staging slot,
prediction block, descriptor buffer and table are created and closed several times over, and each cycle gives the same
bytes and launch count as the first while device memory returns to where it started."""
import numpy as np
import pytest

import inputs

pytestmark = pytest.mark.gpu

CYCLES = 4


@pytest.fixture(scope="module")
def fc():
    import fpga_cnn_b200
    return fpga_cnn_b200


@pytest.fixture(scope="module")
def data(fc):
    frames = inputs.make_frames(("rng", 7), 3, 480, 640)
    regions = fc.grid_regions(3, 480, 640, (128, 256), (64, 128))
    return dict(
        # 512 host images of 512x512 through the per-layer kernels: ~190 MiB of map workspaces, ~250 MiB of staging slots
        big=inputs.make_images(("rng", 3), 512, 512, 512),
        imgs=inputs.make_images(("rng", 4), 300),
        feats=inputs.make_features(("rng", 5), 300),
        prep=[inputs.make_frames(("smooth", 6), 2, 160, 200), inputs.make_frames(("rng", 8), 2, 300, 256)],
        pil=[np.random.default_rng(9).integers(0, 256, (2, 100, 150), dtype=np.uint8),
             np.random.default_rng(10).integers(0, 256, (1, 300, 200, 3), dtype=np.uint8)],
        frames=frames, regions=regions)


def _np(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def run_cycle(fc, weights, d):
    """One handle from creation to close -> (named array outputs, launch count)."""
    import torch
    a = fc.CNNAccelerator()
    out = {}
    try:
        a.load_weights(weights)
        a.load_classifier(*inputs.make_fc())
        out["run_direct_512"] = a.run_batch(d["big"], direct=True)
        for name, x in (("infer_300", d["imgs"]), ("infer_40", d["imgs"][:40])):
            for k, v in zip(("cls", "probs", "bbox"), a.infer_batch(x)):
                out[f"{name}_{k}"] = v
        out["pool"] = a.pool_features(d["feats"])
        out["cam_bbox"], out["cam"] = a.cam_bbox_batch(d["feats"], out["infer_300_cls"], return_cam=True)
        for i, f in enumerate(d["prep"]):
            out[f"prep_{i}"] = a.preprocess(f)
        for i, im in enumerate(d["pil"]):
            out[f"pil_{i}"] = a.image_to_gray128(im)
        frames_t = torch.from_numpy(d["frames"]).cuda()
        for kind, fr in (("host", d["frames"]), ("dev", frames_t)):
            for k, v in zip(("cls", "probs", "bbox", "gray"), a.detect_regions(fr, d["regions"], return_gray=True)):
                out[f"regions_{kind}_{k}"] = _np(v)
            for k, v in enumerate(a.detect_objects(fr, d["regions"], score_min=0.2)):
                out[f"objects_{kind}_{k}"] = _np(v)
        del frames_t
        cls, probs = out["regions_host_cls"], out["regions_host_probs"]
        merged = a.merge_regions(d["regions"], cls, probs[np.arange(len(cls)), cls], out["regions_host_bbox"], len(d["frames"]),
                                 score_min=0.2)
        for k, v in enumerate(merged):
            out[f"merge_{k}"] = v
        out["async"] = np.array(a.wait_batch(a.run_batch_async(np.ascontiguousarray(d["imgs"][:200]))))
        out["one"] = a.infer_one(d["imgs"][0])[0]
        a.probe_int8_peak(1.0)                          # its timing varies from run to run: only its launches are compared
        launches = a.launch_count
    finally:
        a.close()
    return out, launches


def test_handle_resources_released_every_cycle(fc, shipped_weights, data):
    import torch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    first, launches0 = run_cycle(fc, shipped_weights, data)
    for c in range(1, CYCLES):
        got, launches = run_cycle(fc, shipped_weights, data)
        assert launches == launches0, c
        assert got.keys() == first.keys()
        for k in first:
            same = got[k].dtype == first[k].dtype and got[k].shape == first[k].shape and got[k].tobytes() == first[k].tobytes()
            assert same, (c, k)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    assert free0 - torch.cuda.mem_get_info()[0] < (64 << 20)      # the calls above grow ~0.5 GiB of buffers per handle
