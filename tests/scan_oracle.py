"""numpy restatement of cnnacc_scan_frames (include/cnnacc.h): gray at full resolution, the conv stack once per frame at
fh x fw, then classify_vec / bbox_vec on the 16x16 window of the frame's feature map at (x/8, y/8).  TEST INFRASTRUCTURE.
tests/test_scan_cpu.py pins it against np_oracle's per-image path; tests/test_scan_gpu.py compares the library with it."""
import numpy as np

from oracle import np_oracle


def origins(side, stride):
    """Window origins along one side: 0, stride, 2 stride, ... plus one flush with the far edge when that is missing."""
    pos = list(range(0, side - 128 + 1, stride))
    if pos[-1] != side - 128:
        pos.append(side - 128)
    return pos


def count(side, stride):
    """The header's rule for nx (ny): (side - 128) / stride + 1 + ((side - 128) % stride != 0)."""
    return (side - 128) // stride + 1 + int((side - 128) % stride != 0)


def windows(n_frames, fh, fw, stride):
    """(R, 4) int32 (frame, x, y, 128), frame-major, then y, then x."""
    return np.array([(f, x, y, 128) for f in range(n_frames) for y in origins(fh, stride) for x in origins(fw, stride)],
                    np.int32).reshape(-1, 4)


def frame_maps(frames, weights, shifts, acc_bits=32):
    """[F][64][fh/8][fw/8] u8: np_oracle.infer of each frame's full-resolution gray."""
    kern = np_oracle.unpack_weights(weights)
    _, fh, fw, _ = frames.shape
    return np.stack([np_oracle.infer(np_oracle.bgr_to_gray(f), kern, shifts, H=fh, W=fw, acc_bits=acc_bits)
                     .reshape(64, fh // 8, fw // 8) for f in frames])


def window_maps(maps, wins):
    """[R][64][16][16]: the window (f, x, y) of each row of `wins` cut out of its frame's map."""
    return np.stack([maps[f, :, y // 8:y // 8 + 16, x // 8:x // 8 + 16] for f, x, y, _ in wins])


def tail(wmaps, fc_w, fc_b):
    """classify_vec + bbox_vec per map -> (cls [R], probs [R, n_cls], logits [R, n_cls], bbox [R, 4])."""
    cls, probs, logits, boxes = [], [], [], []
    for m in wmaps.reshape(-1, 64, 256):
        c, p, lg, _ = np_oracle.classify_vec(m, fc_w, fc_b)
        cls.append(c)
        probs.append(p)
        logits.append(lg)
        boxes.append(np_oracle.bbox_vec(m, c, fc_w)[0])
    return np.array(cls, np.int32), np.array(probs), np.array(logits), np.array(boxes, np.int32).reshape(-1, 4)


def scan(frames, weights, shifts, fc_w, fc_b, stride, acc_bits=32):
    """-> (windows (R, 4), window maps [R][64][16][16], cls, probs, logits, bbox) for frames [F][fh][fw][3]."""
    n, fh, fw, _ = frames.shape
    wins = windows(n, fh, fw, stride)
    wmaps = window_maps(frame_maps(frames, weights, shifts, acc_bits), wins)
    return (wins, wmaps) + tail(wmaps, fc_w, fc_b)
