#!/usr/bin/env python3
"""Generate tests/golden/resample_edges.npz by running Pillow and OpenCV directly.  Build container only.

    python tests/golden/make_resample_edges_golden.py

The two resampling front ends at the edges of their domains:
  * load_image_any (pynq_inference.py:414-425) is `Image.open(path).convert('L').resize((128, 128))`; these lines run on
    lossless PNG files written from the seeded images of tests/inputs.py RESAMPLE_PIL_CASES.
  * the capture loop's pre-processing (realtime_detect.py:582-591) is centre-crop, cv2.cvtColor(BGR2GRAY),
    cv2.resize(INTER_AREA), as in make_prep_golden.py; it runs single-threaded on the seeded frames of RESAMPLE_AREA_CASES, on
    the squares of inputs.REGIONS_8192 and inputs.REGIONS_4K.
Only the 128x128 outputs and the library versions are stored; the inputs are regenerated from their seeds at test time.
Before writing, asserts that the numpy restatement (oracle/np_oracle.py) reproduces every output.  The archive is written
with fixed member timestamps, so a rerun with the same library versions reproduces it byte for byte.
"""
import io
import os
import sys
import tempfile
import zipfile

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import inputs  # noqa: E402
from oracle import np_oracle  # noqa: E402
from make_prep_golden import reference_preprocess  # noqa: E402

OUT = os.path.join(HERE, "resample_edges.npz")


def oracle_preprocess(frame):
    """np_oracle.preprocess_bgr with the gray conversion done in row blocks (an 8192x8192 frame needs no GB temporaries)."""
    h, w = frame.shape[:2]
    s = min(h, w)
    crop = frame[(h - s) // 2:(h - s) // 2 + s, (w - s) // 2:(w - s) // 2 + s]
    gray = np.concatenate([np_oracle.bgr_to_gray(crop[i:i + 1024]) for i in range(0, s, 1024)])
    return np_oracle.resize_area_u8(gray)


def region_outputs(frames, regions, fn):
    return np.stack([fn(np.ascontiguousarray(frames[f, y:y + s, x:x + s])) for f, x, y, s in regions])


def write_npz(path, arrays):
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_DEFLATED) as z:
        for key in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(arrays[key]), allow_pickle=False)
            info = zipfile.ZipInfo(key + ".npy", date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            z.writestr(info, buf.getvalue())


def main():
    import PIL
    from PIL import Image
    cv2.setNumThreads(1)
    out = {"pillow_version": np.array(PIL.__version__), "cv2_version": np.array(cv2.__version__)}
    with tempfile.TemporaryDirectory() as tmp:
        for case in inputs.RESAMPLE_PIL_CASES:
            arr = inputs.make_pil_image(case)
            path = os.path.join(tmp, "img.png")
            Image.fromarray(arr, case["mode"]).save(path)
            got = np.array(Image.open(path).convert("L").resize((128, 128)), dtype=np.uint8)
            assert got.shape == (128, 128)
            assert np.array_equal(got.reshape(-1), np_oracle.load_image_array(arr)), case["name"]
            out[case["name"]] = got
            print(f"{case['name']:32s} mean {got.mean():6.1f}")
    for case in inputs.RESAMPLE_AREA_CASES:
        frames = inputs.make_frames(case["frames"], case["n"], case["h"], case["w"])
        got = np.stack([reference_preprocess(np.ascontiguousarray(f)) for f in frames])
        for i, f in enumerate(frames):
            assert np.array_equal(got[i], oracle_preprocess(f)), (case["name"], i)
        out[case["name"]] = got
        print(f"{case['name']:32s} {case['h']}x{case['w']} n={case['n']} mean {got.mean():6.1f}")
    big = np.concatenate([inputs.make_area_frames("area_k64_8192"), inputs.make_area_frames("area_k64_8192_edges")])
    out["regions_8192"] = region_outputs(big, inputs.REGIONS_8192, reference_preprocess)
    assert np.array_equal(out["regions_8192"], region_outputs(big, inputs.REGIONS_8192, oracle_preprocess))
    del big
    uhd = inputs.make_area_frames("area_4k")
    out["regions_4k"] = region_outputs(uhd, inputs.REGIONS_4K, reference_preprocess)
    assert np.array_equal(out["regions_4k"], region_outputs(uhd, inputs.REGIONS_4K, oracle_preprocess))
    write_npz(OUT, out)
    print("wrote resample_edges.npz", os.path.getsize(OUT), "bytes; Pillow", PIL.__version__, "cv2", cv2.__version__)


if __name__ == "__main__":
    main()
