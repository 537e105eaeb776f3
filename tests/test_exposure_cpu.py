"""What the byte-exact GPU tests can see: for every workload of inputs.EXPOSED_WORKLOADS and every draw of
inputs.shift_triple_draws(), the numpy oracle shows that an accumulator off by one changes final output bytes.

Every layer ends in >> shift, a clip to 0..255 and a 2x2 max, so a wrong accumulator is only visible when its sum sits next
to a multiple of 2^shift, it is the maximum of its pool window and its byte is not clipped -- and then only if the changed
byte moves a later layer's sum across such a multiple too.  Per workload this file asserts:
  * at every layer at least 30 % of the pooled bytes are strictly inside (0, 255);
  * adding 1 to every accumulator of layer L changes at least 3 % of the final bytes, for L = 0, 1, 2;
  * adding 1 to the accumulators of ONE spatial position of layer L (every output channel there, the shape of a bad halo
    column, parity plane or half-slab) changes a final byte in at least one image, for each position tried: corners, borders,
    the middle rows (pooled row 32 of layer 0 is where the kernel hands act1 from its top to its bottom half) and columns 15,
    16, 31, 32.
A GPU path whose output equals the oracle's on these workloads therefore has no such error.  CPU only.
"""
import numpy as np
import pytest

import inputs
from oracle import np_oracle

MIN_INSIDE = 0.30
MIN_CHANGED = 0.03


def _acc(x, kern):
    """(N,ic,H,W) u8 -> (N,oc,H,W) int64 accumulators of the 3x3 same/zero-pad conv.  float32 GEMMs are exact here: every
    partial sum is an integer below 32*9*255*128 = 9.4 M < 2^24."""
    N, ic, H, W = x.shape
    xp = np.zeros((N, ic, H + 2, W + 2), np.float32)
    xp[:, :, 1:-1, 1:-1] = x
    k = kern.astype(np.float32)
    acc = np.zeros((N, kern.shape[0], H, W), np.float32)
    for dy in range(3):
        for dx in range(3):
            acc += np.einsum("oi,nihw->nohw", k[:, :, dy, dx], xp[:, :, dy:dy + H, dx:dx + W], optimize=True)
    return acc.astype(np.int64)


def _pool(acc, shift):
    y = np.clip(acc >> shift, 0, 255)
    N, oc, H, W = y.shape
    return y.reshape(N, oc, H // 2, 2, W // 2, 2).max(axis=(3, 5)).astype(np.uint8)


def _layer_acc(x, kern, acc_bits):
    a = _acc(x, kern)
    return ((a + (1 << 23)) % (1 << 24)) - (1 << 23) if acc_bits == 24 else a


def _forward(imgs, kern, shifts, acc_bits=32):
    """-> accumulators (after the 24-bit wrap, before the shift) and pooled bytes of every layer."""
    x, accs, outs = imgs[:, None], [], []
    for L in range(3):
        accs.append(_layer_acc(x, kern[L], acc_bits))
        x = _pool(accs[-1], shifts[L])
        outs.append(x)
    return accs, outs


def _downstream(x, kern, shifts, L, acc_bits):
    """Pooled bytes of layer L -> final bytes."""
    for l in range(L + 1, 3):
        x = _pool(_layer_acc(x, kern[l], acc_bits), shifts[l])
    return x


def _positions(S):
    rows = sorted({0, 1, S // 2 - 2, S // 2 - 1, S // 2, S // 2 + 1, S - 2, S - 1})
    cols = sorted({0, 1, 15, 16, 31, 32, S - 2, S - 1} & set(range(S)))
    return [(y, x) for y in rows for x in cols]


def exposure(imgs, wt, shifts, acc_bits=32):
    """-> (inside fraction per layer, final bytes changed by +1 on all of layer L, per layer L: positions whose +1 no image
    shows, the final bytes)."""
    kern = np_oracle.unpack_weights(wt)
    accs, outs = _forward(imgs, kern, shifts, acc_bits)
    final = outs[2]
    inside = [float(((o > 0) & (o < 255)).mean()) for o in outs]
    changed = [float((_downstream(_pool(accs[L] + 1, shifts[L]), kern, shifts, L, acc_bits) != final).mean()) for L in range(3)]
    blind = []
    for L in range(3):
        S = accs[L].shape[2]
        missed = []
        for y, x in _positions(S):
            y0, x0 = y & ~1, x & ~1
            win = accs[L][:, :, y0:y0 + 2, x0:x0 + 2].copy()
            win[:, :, y - y0, x - x0] += 1
            new = np.clip(win.reshape(len(imgs), -1, 4).max(axis=2) >> shifts[L], 0, 255).astype(np.uint8)
            seen = False
            for i in np.flatnonzero((new != outs[L][:, :, y // 2, x // 2]).any(axis=1)):
                m = outs[L][i:i + 1].copy()
                m[0, :, y // 2, x // 2] = new[i]
                if (_downstream(m, kern, shifts, L, acc_bits) != final[i:i + 1]).any():
                    seen = True
                    break
            if not seen:
                missed.append((y, x))
        blind.append(missed)
    return inside, changed, blind, final


def test_batched_forward_is_the_oracle():
    """The batched restatement above is np_oracle.infer, at both accumulator widths."""
    for w in inputs.EXPOSED_WORKLOADS:
        imgs = inputs.workload_images(w)[:2]
        kern = np_oracle.unpack_weights(inputs.make_weights(w["weights"]))
        bits = w.get("acc_bits", 32)
        got = _forward(imgs, kern, w["shifts"], bits)[1][2]
        for i in range(2):
            assert np.array_equal(got[i].reshape(64, 256), np_oracle.infer(imgs[i], kern, w["shifts"], acc_bits=bits)), w["name"]


def _lsb_cases():
    cases = [(w["name"], w["weights"], w["shifts"], inputs.workload_images(w)) for w in inputs.EXPOSED_WORKLOADS
             if w.get("acc_bits", 32) == 32]
    cases += [(name, wk, sh, inputs.make_images(ik, 40)) for name, wk, sh, ik in inputs.shift_triple_draws()]
    return cases


@pytest.mark.parametrize("case", _lsb_cases(), ids=lambda c: c[0])
def test_one_lsb_errors_show(case):
    name, wk, shifts, imgs = case
    inside, changed, blind, _ = exposure(imgs, inputs.make_weights(wk), shifts)
    print(f"{name} shifts {shifts}: inside (0,255) {['%.2f' % v for v in inside]}, "
          f"final bytes changed by +1 at L0/L1/L2 {['%.1f %%' % (100 * v) for v in changed]}")
    assert min(inside) >= MIN_INSIDE, inside
    assert min(changed) >= MIN_CHANGED, changed
    assert not any(blind), blind


def test_24_bit_workload_wraps_and_stays_informative():
    """acc24_wrap: many layer-2 sums leave the 24-bit range, the wrapped results differ from the 32-bit ones in many final
    bytes, and the final bytes (and layer 1's) stay informative.  The other workloads' sums stay below 2^23, so their 24-bit
    results equal the 32-bit ones and their 24-bit runs are the one-LSB tests of the 24-bit kernels."""
    w = next(w for w in inputs.EXPOSED_WORKLOADS if w["name"] == "acc24_wrap")
    imgs = inputs.workload_images(w)
    wt = inputs.make_weights(w["weights"])
    kern = np_oracle.unpack_weights(wt)
    accs32, outs32 = _forward(imgs, kern, w["shifts"], 32)
    _, outs24 = _forward(imgs, kern, w["shifts"], 24)
    wrapped = float((np.abs(accs32[2]) >= (1 << 23)).mean())
    moved = float((outs24[2] != outs32[2]).mean())
    inside = [float(((o > 0) & (o < 255)).mean()) for o in outs24]
    print(f"acc24_wrap: layer-2 sums beyond 2^23 {100 * wrapped:.1f} %, final bytes moved by the wrap {100 * moved:.1f} %, "
          f"inside (0,255) {['%.2f' % v for v in inside]}")
    assert wrapped >= 0.2 and moved >= 0.2
    assert inside[1] >= MIN_INSIDE and inside[2] >= MIN_INSIDE
    for v in inputs.EXPOSED_WORKLOADS:
        if v.get("acc_bits", 32) == 32:
            a = _forward(inputs.workload_images(v), np_oracle.unpack_weights(inputs.make_weights(v["weights"])), v["shifts"])[0]
            assert max(int(np.abs(x).max()) for x in a) < (1 << 23), v["name"]


def test_all_zero_triples_are_all_zero():
    """The draws of test_conv_gpu.py's test_shifts_that_zero_every_output: with shifts of 24..31 at every layer no byte of
    any layer can be non-zero (the largest sum, 32*9*255*128 = 9.4 M, is below 2^24)."""
    for wk, sh, ik in inputs.all_zero_triples():
        imgs = inputs.make_images(ik, 2)
        kern = np_oracle.unpack_weights(inputs.make_weights(wk))
        assert min(sh) >= 24 and not any(np_oracle.infer(imgs[i], kern, sh).any() for i in range(2))
