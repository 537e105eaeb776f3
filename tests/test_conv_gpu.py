"""Parity of the CUDA conv stack with the oracle, through the C ABI.  Bit-exact (integer path)."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import inputs
import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fc():
    import fpga_cnn_b200 as fc_
    fc_.load()
    return fc_


@pytest.fixture(scope="module")
def acc(fc, shipped_weights):
    a = fc.CNNAccelerator(device=0)
    a.load_weights(shipped_weights)
    yield a
    a.close()


@pytest.fixture(scope="module")
def port():
    return oracle.load_port()


@pytest.mark.parametrize("direct", [False, True], ids=["fused", "direct"])
@pytest.mark.parametrize("case", inputs.CONV_CASES, ids=lambda c: c["name"])
def test_golden_cases(case, direct, acc, shipped_weights, conv_golden):
    wt = inputs.make_weights(case["weights"], shipped_weights)
    acc.load_weights(wt)
    acc.set_shifts(*case["shifts"])
    imgs = inputs.make_images(case["images"], case["n"])
    got = acc.run_batch(imgs, direct=direct)
    assert got.shape == (case["n"], 64, 16, 16)
    assert np.array_equal(got.reshape(case["n"], 64, 256), conv_golden[case["name"]])


@pytest.mark.parametrize("case", [c for c in inputs.CONV_CASES if c.get("dump")], ids=lambda c: c["name"])
def test_intermediate_maps_via_register_protocol(case, acc, shipped_weights, conv_golden):
    """load_image / start / wait / read_feature_map over BRAM channels 0-111 (pynq_inference.py:209-286)."""
    acc.load_weights(inputs.make_weights(case["weights"], shipped_weights))
    acc.set_shifts(*case["shifts"])
    img = inputs.make_images(case["images"], 1)[0]
    acc.load_image(img)
    acc.start_inference()
    assert acc.wait_done(10.0) >= 0
    assert (acc.read_reg(0x04) >> 1) & 1
    l0, l1 = conv_golden[case["name"] + "__l0"], conv_golden[case["name"] + "__l1"]
    for ch in (0, 7, 15):
        assert np.array_equal(acc.read_feature_map(ch, 4096), l0[ch].reshape(-1))
    for ch in (16, 33, 47):
        assert np.array_equal(acc.read_feature_map(ch, 1024), l1[ch - 16].reshape(-1))
    assert np.array_equal(acc.read_layer2_output(), conv_golden[case["name"]][0])
    # dump_fpga_features-style register pokes (write 0x20 / 0x24, read 0x28)
    acc.write_reg(0x20, 48 + 5); acc.write_reg(0x24, 100)
    assert acc.read_reg(0x28) == conv_golden[case["name"]][0][5, 100]


@pytest.mark.parametrize("direct", [False, True], ids=["fused", "direct"])
def test_random_batch_vs_oracle(direct, acc, port, shipped_weights):
    rng = np.random.default_rng(5)
    for trial in range(4):
        wt = shipped_weights if trial % 2 == 0 else inputs.make_weights(("rng", 300 + trial))
        sh = (7, 10, 11) if trial % 2 == 0 else (9, 12, 13)
        n = int(rng.integers(1, 70))
        imgs = inputs.make_images(("rng", 400 + trial), n)
        acc.load_weights(wt)
        acc.set_shifts(*sh)
        got = acc.run_batch(imgs, direct=direct).reshape(n, 64, 256)
        want = oracle.port_infer_batch(port, imgs, wt, sh)
        assert np.array_equal(got, want), f"trial {trial}: {np.argwhere(got != want)[:5]}"


@pytest.mark.parametrize("n", [1, 2, 3, 147, 148, 149, 295, 296, 297, 445])
def test_batch_sizes_around_the_sm_count(n, acc, port, shipped_weights):
    """The fused kernel is persistent (one CTA per SM, images strided by CTA): CTAs with 1, 2, 3 and 4 images, the
    2-deep input prefetch and the cross-image pipeline hand-offs all have to line up at every batch size."""
    acc.load_weights(shipped_weights)
    acc.set_shifts(7, 10, 11)
    imgs = inputs.make_images(("rng", 1000 + n), n)
    got = acc.run_batch(imgs).reshape(n, 64, 256)
    assert np.array_equal(got, oracle.port_infer_batch(port, imgs, shipped_weights, (7, 10, 11)))


def test_random_shift_triples(acc, port):
    """Random per-layer shifts, each drawn where its layer's sums reach 2^shift for the draw's ternary weights, so every layer
    keeps informative bytes and a one-LSB error shows (inputs.shift_triple_draws; test_exposure_cpu.py holds each draw to it)."""
    for name, wk, sh, ik in inputs.shift_triple_draws():
        wt = inputs.make_weights(wk)
        imgs = inputs.make_images(ik, 40)
        acc.load_weights(wt)
        acc.set_shifts(*sh)
        got = acc.run_batch(imgs).reshape(40, 64, 256)
        want = oracle.port_infer_batch(port, imgs, wt, sh)
        assert np.array_equal(got, want), (name, sh, int((got != want).sum()))


def test_shifts_that_zero_every_output(acc):
    """Shifts of 24..31 at every layer (the top of the 5-bit AXI register field, pynq_inference.py:226-229): every byte is 0."""
    for wk, sh, ik in inputs.all_zero_triples():
        acc.load_weights(inputs.make_weights(wk))
        acc.set_shifts(*sh)
        got = acc.run_batch(inputs.make_images(ik, 40))
        assert not got.any(), sh


@pytest.mark.parametrize("case", inputs.HW_CASES, ids=lambda c: c["name"])
def test_generic_sizes(case, acc, shipped_weights, conv_golden):
    acc.load_weights(inputs.make_weights(case["weights"], shipped_weights))
    acc.set_shifts(*case["shifts"])
    img = inputs.make_images(case["images"], 1, case["H"], case["W"])
    got = acc.run_batch(img)
    assert np.array_equal(got.reshape(64, -1), conv_golden[case["name"]])


@pytest.mark.parametrize("H,W", [(128, 256), (144, 208), (384, 128), (240, 336), (512, 512)])
def test_tiled_windows_vs_oracle_and_direct(H, W, acc, port, shipped_weights):
    """Sizes above 128x128 run as overlapping 128x128 windows through the fused kernel (csrc/tiling.cuh): every output
    must equal the oracle's full-image result (halo recompute, image-border padding) and the per-layer kernels'."""
    n = 3
    for wt, sh, kind in ((shipped_weights, (7, 10, 11), ("rng", 31)), (inputs.make_weights(("rng", 32)), (9, 12, 13), ("smooth", 33))):
        acc.load_weights(wt)
        acc.set_shifts(*sh)
        imgs = inputs.make_images(kind, n, H, W)
        got = acc.run_batch(imgs)
        assert got.shape == (n, 64, H // 8, W // 8)
        want = oracle.port_infer_batch(port, imgs, wt, sh, H, W)
        assert np.array_equal(got.reshape(n, 64, -1), want), np.argwhere(got.reshape(n, 64, -1) != want)[:5]
        assert np.array_equal(acc.run_batch(imgs, direct=True), got)


def test_fused_equals_direct_at_scale(acc, shipped_weights):
    """Full-size property check: the fused kernel and the per-layer kernels agree on 4096 images (config 2)."""
    acc.load_weights(shipped_weights)
    acc.set_shifts(7, 10, 11)
    imgs = inputs.make_images(("rng", 77), 4096)
    a = acc.run_batch(imgs)
    b = acc.run_batch(imgs, direct=True)
    assert np.array_equal(a, b)


def test_ten_thousand_images_vs_oracle(acc, port, shipped_weights):
    """The north_star gate: 10 000 synthetic images, 100 % byte-equal vs the oracle (multi-process on the host)."""
    import multiprocessing as mp
    n = 10000
    acc.load_weights(shipped_weights)
    got = {}
    imgs = inputs.make_images(("rng", 1234), n)
    for sh in ((2, 4, 6), (7, 10, 11)):
        acc.set_shifts(*sh)
        got[sh] = acc.run_batch(imgs).reshape(n, 64, 256)
    workers = min(mp.cpu_count(), 32)
    bounds = np.linspace(0, n, workers + 1).astype(int)
    for sh in got:
        jobs = [(imgs[bounds[i]:bounds[i + 1]], shipped_weights, sh) for i in range(workers)]
        with mp.get_context("fork").Pool(workers) as pool:
            parts = pool.map(_oracle_chunk, jobs)
        want = np.concatenate(parts)
        bad = np.flatnonzero((got[sh] != want).reshape(n, -1).any(axis=1))
        assert bad.size == 0, f"shifts {sh}: {bad.size} images differ, first {bad[:5]}"


def _oracle_chunk(job):
    imgs, wt, sh = job
    return oracle.port_infer_batch(oracle.load_port(), imgs, wt, sh)


def test_drop_in_cnn_infer_symbol(fc, shipped_weights, conv_golden):
    """The reference's ARMEngine.run body against libcnnacc.so (realtime_detect.py:422-436)."""
    eng = fc.ARMEngine(shipped_weights, shifts=(7, 10, 11))
    imgs = inputs.make_images(("rng", 1), 3)
    for i in range(3):
        feat, conv_ms, read_ms = eng.run(imgs[i])
        assert feat.shape == (64, 256) and feat.dtype == np.uint8 and read_ms == 0.0
        assert np.array_equal(feat, conv_golden["rng_shipped_mid"][i])


def test_engine_run_surface(fc, shipped_weights, conv_golden):
    eng = fc.B200Engine(shipped_weights, shifts=(2, 4, 6))
    imgs = inputs.make_images(("rng", 0), 2)
    for i in range(2):
        feat, conv_ms, read_ms = eng.run(imgs[i].reshape(128, 128))
        assert np.array_equal(feat, conv_golden["rng_shipped_default"][i]) and conv_ms > 0 and read_ms > 0


def test_error_conventions(fc, shipped_weights):
    a = fc.CNNAccelerator()
    with pytest.raises(RuntimeError):
        a.run_batch(np.zeros((1, 128, 128), np.uint8))          # weights not loaded
    with pytest.raises(AssertionError):
        a.load_weights(np.zeros(100, np.uint8))                 # pynq_inference.py:189
    a.load_weights(shipped_weights)
    with pytest.raises(AssertionError):
        a.load_image(np.zeros(100, np.uint8))                   # pynq_inference.py:214
    with pytest.raises(ValueError):
        a.set_shifts(2, 4, 32)
    with pytest.raises(ValueError):
        a.run_batch(np.zeros((1, 100, 128), np.uint8))
    n0 = a.launch_count
    for out in (np.zeros(2 * 16384, np.float32),                 # the right element count, of the wrong dtype
                np.zeros(4 * 16384, np.uint8)[::2]):             # a strided view over a buffer large enough for 2*16384
        with pytest.raises(ValueError):
            a.run_batch(np.zeros((2, 128, 128), np.uint8), out=out)
    assert a.launch_count == n0
    with pytest.raises(RuntimeError):
        a.start_inference()                                      # no image loaded
    assert a.run_batch(np.zeros((0, 128, 128), np.uint8)).shape == (0, 64, 16, 16)   # empty batch
    a.close()


def test_device_pointer_path_with_torch(fc, shipped_weights, conv_golden):
    import torch
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    a.use_stream(torch.cuda.current_stream().cuda_stream)
    imgs = torch.from_numpy(inputs.make_images(("rng", 1), 8)).cuda()
    out = a.run_batch(imgs)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().reshape(8, 64, 256), conv_golden["rng_shipped_mid"])
    n0 = a.launch_count
    with pytest.raises(ValueError):
        a.run_batch(imgs.float())
    assert a.launch_count == n0
    a.close()


def test_handle_lifecycle_and_mixed_call_sizes(fc, port, shipped_weights):
    """Handles are created and destroyed repeatedly, two live side by side, and one handle sees call sizes that grow, shrink
    and switch between the latency path, the staging ring and device pointers -- every result still byte-equal to the oracle."""
    import torch
    imgs = inputs.make_images(("rng", 31), 700)
    want = oracle.port_infer_batch(port, imgs, shipped_weights, (7, 10, 11)).reshape(700, 64, 16, 16)
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(6):
        a, b = fc.CNNAccelerator(), fc.CNNAccelerator()
        for h in (a, b):
            h.load_weights(shipped_weights)
            h.set_shifts(7, 10, 11)
        for n in (1, 700, 3, 65, 64, 300, 2):
            got = (a if n % 2 else b).run_batch(imgs[:n])
            assert np.array_equal(got, want[:n]), n
        t = torch.from_numpy(imgs[:130]).cuda()
        assert np.array_equal(a.run_batch(t).cpu().numpy(), want[:130])
        a.close()
        b.close()
    torch.cuda.synchronize()
    assert free0 - torch.cuda.mem_get_info()[0] < (64 << 20)          # nothing substantial leaked across 12 handles


def test_two_host_threads_two_handles(fc, port, shipped_weights):
    """One handle per host thread (INTEGRATION.md section 5): concurrent run_batch calls do not disturb each other."""
    import threading
    imgs = [inputs.make_images(("rng", 40 + i), 400) for i in range(2)]
    want = [oracle.port_infer_batch(port, im, shipped_weights, (2, 4, 6)).reshape(400, 64, 16, 16) for im in imgs]
    accs = [fc.CNNAccelerator() for _ in range(2)]
    for a in accs:
        a.load_weights(shipped_weights)
    bad = []

    def work(i):
        for _ in range(10):
            if not np.array_equal(accs[i].run_batch(imgs[i]), want[i]):
                bad.append(i)

    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for a in accs:
        a.close()
    assert not bad


@pytest.mark.parametrize("direct", [False, True], ids=["fused", "direct"])
@pytest.mark.parametrize("case", inputs.ACC24_CASES, ids=lambda c: c["name"])
def test_acc24_mode_vs_trainer_fixtures(case, direct, fc, shipped_weights, acc24_golden):
    """cnnacc_set_accumulator_bits(24): byte-equal to the reference's own bit-accurate model (train_cnn.fpga_conv_layer,
    fixtures from tests/golden/make_acc24_golden.py) on wrapping and non-wrapping cases; the default mode is untouched."""
    wt = inputs.make_weights(case["weights"], shipped_weights)
    if case.get("clamp127"):
        wt = inputs.pack_weights([np.maximum(k, -127) for k in oracle.np_oracle.unpack_weights(wt)])
    imgs = inputs.make_images(case["images"], case["n"])
    a = fc.CNNAccelerator()
    a.load_weights(wt)
    a.set_shifts(*case["shifts"])
    assert a.get_accumulator_bits() == 32
    plain = a.run_batch(imgs, direct=direct).reshape(case["n"], 64, 256)
    assert np.array_equal(plain, oracle.port_infer_batch(oracle.load_port(), imgs, wt, case["shifts"]))
    a.set_accumulator_bits(24)
    assert a.get_accumulator_bits() == 24
    got = a.run_batch(imgs, direct=direct).reshape(case["n"], 64, 256)
    assert np.array_equal(got, acc24_golden[case["name"]]), np.argwhere(got != acc24_golden[case["name"]])[:5]
    assert np.array_equal(got, plain) != case["wraps"]
    with pytest.raises(ValueError):
        a.set_accumulator_bits(16)
    a.set_accumulator_bits(32)
    assert np.array_equal(a.run_batch(imgs, direct=direct).reshape(case["n"], 64, 256), plain)
    a.close()


def test_acc24_random_vs_oracle_incl_windows(fc):
    """More wrapping inputs than the fixtures hold, against the pinned numpy restatement, plus a 256x128 image through the
    window mode (the wrap sits in the shared layer-2 epilogue)."""
    a = fc.CNNAccelerator()
    a.set_accumulator_bits(24)
    for seed in (71, 72):
        wt = inputs.make_weights(("acc24", seed))
        kern = oracle.np_oracle.unpack_weights(wt)
        a.load_weights(wt)
        a.set_shifts(0, 14, 15)
        imgs = inputs.make_images(("bright", seed + 10), 5)
        got = a.run_batch(imgs).reshape(5, 64, 256)
        for i in range(5):
            assert np.array_equal(got[i], oracle.np_oracle.infer(imgs[i], kern, (0, 14, 15), acc_bits=24)), (seed, i)
        big = inputs.make_images(("bright", seed + 20), 1, 256, 128)
        want = oracle.np_oracle.infer(big[0], kern, (0, 14, 15), H=256, W=128, acc_bits=24)
        assert np.array_equal(a.run_batch(big).reshape(64, -1), want)
        assert np.array_equal(a.run_batch(big, direct=True).reshape(64, -1), want)
    a.close()


def test_torch_call_is_ordered_on_the_current_stream(fc, port, shipped_weights):
    """Device-pointer calls run on torch's current stream unless use_stream() chose one: producer -> run_batch -> .cpu()
    needs no explicit synchronisation, on the default stream and on a side stream."""
    import torch
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    base = inputs.make_images(("rng", 90), 2048)
    want = oracle.port_infer_batch(port, base[:64], shipped_weights, (7, 10, 11)).reshape(64, 64, 16, 16)
    for stream in (None, torch.cuda.Stream()):
        ctx = torch.cuda.stream(stream) if stream is not None else torch.cuda.stream(torch.cuda.current_stream())
        with ctx:
            for rep in range(3):
                t = torch.from_numpy(base).cuda(non_blocking=True)
                t = (t ^ 0xFF) ^ 0xFF                     # a torch kernel produces the input on the current stream
                got = a.run_batch(t).cpu()                # no use_stream, no synchronize
                assert np.array_equal(got.numpy()[:64], want)
                cls_f = a.run_batch(t[:64].clone())
                assert np.array_equal(cls_f.cpu().numpy(), want)
    with pytest.raises(ValueError):
        a.run_batch(torch.zeros((2, 128, 128), dtype=torch.uint8, device="cuda"), out=torch.zeros(5, dtype=torch.uint8, device="cuda"))
    a.close()


def test_direct_path_at_the_largest_size(fc, port, shipped_weights):
    """8192 x 8192 is the largest size the API accepts: layer 0 of the per-layer path has 256 x 256 = 65 536 tiles, one more
    than gridDim.y allows (the tile index now shares gridDim.x with the image index).  Per-layer kernels == window mode on
    the whole image, and the top-left corner == the oracle on a crop (outputs 0..13 only see pixels 0..119)."""
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    img = inputs.make_images(("rng", 55), 1, 8192, 8192)
    direct = a.run_batch(img, direct=True)
    assert direct.shape == (1, 64, 1024, 1024)
    assert np.array_equal(direct, a.run_batch(img))
    corner = oracle.port_infer_batch(port, np.ascontiguousarray(img[:, :128, :128]), shipped_weights, (7, 10, 11)).reshape(64, 16, 16)
    assert np.array_equal(direct[0, :, :14, :14], corner[:, :14, :14])
    a.close()


def test_predictions_into_a_shared_registered_mapping(fc, port, shipped_weights, tmp_path):
    """bench.py's stream_1m pattern: a file mapping page-locked with cnnacc_register_host receives the predictions of
    device-resident chunks by plain async copies; they equal the host-pointer call's."""
    import torch
    n = 3000
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    a.load_classifier(*inputs.make_fc())
    imgs = inputs.make_images(("rng", 56), n)
    want_cls, want_probs, want_box = a.infer_batch(imgs)
    path = "/dev/shm/cnnacc_test_%d.bin" % os.getpid()
    with open(path, "wb") as f:
        f.truncate(n * 44)
    try:
        shm = np.memmap(path, dtype=np.uint8, mode="r+", shape=(n * 44,))
        unregister = fc.register_host(shm)
        h_cls = torch.from_numpy(shm[:n * 4].view(np.int32))
        h_probs = torch.from_numpy(shm[n * 4:n * 28].view(np.float32).reshape(n, 6))
        h_box = torch.from_numpy(shm[n * 28:].view(np.int32).reshape(n, 4))
        t = torch.from_numpy(imgs).cuda()
        for c0 in range(0, n, 1024):
            cls, probs, box = a.infer_batch(t[c0:c0 + 1024])
            h_cls[c0:c0 + 1024].copy_(cls, non_blocking=True)
            h_probs[c0:c0 + 1024].copy_(probs, non_blocking=True)
            h_box[c0:c0 + 1024].copy_(box, non_blocking=True)
        torch.cuda.synchronize()
        assert np.array_equal(h_cls.numpy(), want_cls) and np.array_equal(h_probs.numpy(), want_probs) and np.array_equal(h_box.numpy(), want_box)
        unregister()
        del h_cls, h_probs, h_box, shm
    finally:
        os.unlink(path)
    a.close()


def test_back_to_back_launches_with_and_without_dependencies(fc, port, shipped_weights):
    """Consecutive device-pointer run_batch calls are launched with programmatic stream serialisation and skip the wait for
    their predecessor only when the host can show them independent.  Dependent patterns must still be ordered: the same output
    buffer written twice (last writer wins), an output buffer that aliases the previous input, many rotating buffers, small
    grids in between, and two handles sharing a stream."""
    import torch
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    st = torch.cuda.Stream()
    a.use_stream(st.cuda_stream)
    n = 1500
    host = [inputs.make_images(("rng", 700 + i), n) for i in range(4)]
    want = [oracle.port_infer_batch(port, im, shipped_weights, (7, 10, 11)).reshape(n, 64, 16, 16) for im in host]
    with torch.cuda.stream(st):
        x = [torch.from_numpy(im).cuda() for im in host]
        outs = [torch.empty((n, 64, 16, 16), dtype=torch.uint8, device="cuda") for _ in range(4)]
        shared = torch.empty((n, 64, 16, 16), dtype=torch.uint8, device="cuda")
        for rep in range(20):
            for i in range(4):                       # independent: rotating inputs and outputs
                a.run_batch(x[i], out=outs[i])
            for i in range(4):                       # WAW: one output buffer, last writer must win
                a.run_batch(x[i], out=shared)
            a.run_batch(x[0][:7], out=outs[0][:7])   # a small grid in the chain
            a.run_batch(x[1], out=outs[1])
        st.synchronize()
        for i in range(4):
            assert np.array_equal(outs[i].cpu().numpy(), want[i]), i
        assert np.array_equal(shared.cpu().numpy(), want[3])
        # RAW through an aliased buffer: the second launch reads what the first wrote (features reinterpreted as images)
        chain_in = torch.from_numpy(host[0][:148 * 4]).cuda()
        mid = torch.empty((148 * 4, 64, 16, 16), dtype=torch.uint8, device="cuda")
        for rep in range(10):
            a.run_batch(chain_in, out=mid)
            second = a.run_batch(mid.view(148 * 4, 128, 128))
        st.synchronize()
        mid_h = mid.cpu().numpy()
        assert np.array_equal(mid_h, want[0][:148 * 4])
        want2 = oracle.port_infer_batch(port, mid_h.reshape(148 * 4, 128, 128), shipped_weights, (7, 10, 11)).reshape(-1, 64, 16, 16)
        assert np.array_equal(second.cpu().numpy(), want2)
        # two handles on one stream: the second handle's launch reads the first handle's output
        b = fc.CNNAccelerator()
        b.load_weights(shipped_weights)
        b.set_shifts(7, 10, 11)
        b.use_stream(st.cuda_stream)
        for rep in range(10):
            a.run_batch(chain_in, out=mid)
            third = b.run_batch(mid.view(148 * 4, 128, 128))
            a.run_batch(x[2], out=outs[2])
        st.synchronize()
        assert np.array_equal(third.cpu().numpy(), want2) and np.array_equal(outs[2].cpu().numpy(), want[2])
        b.close()
    a.close()


def test_asynchronous_host_batches(fc, port, shipped_weights):
    """cnnacc_run_batch_async / cnnacc_wait_batch: a stream of host batches through one staging ring.  Every batch equals the
    oracle whatever the submission depth, the wait order, the batch sizes (slot growth in mid-stream) and the calls mixed in."""
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    a.set_shifts(7, 10, 11)
    sizes = [300, 300, 300, 1200, 1, 300, 2048, 300, 300, 300, 700, 300]           # 12 > CNNACC_MAX_PENDING batches in flight
    h_in = [fc.alloc_host((n, 128, 128)) for n in sizes]
    h_out = [fc.alloc_host((n, 64, 16, 16)) for n in sizes]
    for i, n in enumerate(sizes):
        h_in[i][:] = inputs.make_images(("rng", 7000 + i), n)
        h_out[i][:] = 0xEE
    want = [oracle.port_infer_batch(port, x, shipped_weights, (7, 10, 11)) for x in h_in]
    tickets = [a.run_batch_async(x, out=y) for x, y in zip(h_in, h_out)]           # all submitted before any wait
    assert tickets == list(range(len(sizes)))
    for i in (5, 0, 11, 3):                                                         # any order; older ones are complete by then
        out = a.wait_batch(tickets[i])
        assert out is h_out[i]
    a.synchronize()
    for i, n in enumerate(sizes):
        assert np.array_equal(h_out[i].reshape(n, 64, 256), want[i]), i
    # depth-2 streaming loop (the bench's e2e leg), a synchronous call and a device-pointer call in mid-stream, 512x512 batches
    import torch
    prev = None
    for rep in range(6):
        i = rep % 3
        h_out[i][:] = 0
        t = a.run_batch_async(h_in[i], out=h_out[i])
        if rep == 2:
            got = a.run_batch(h_in[4])                                              # synchronous: drains the ring first
            assert np.array_equal(got.reshape(1, 64, 256), want[4])
        if rep == 4:
            d = a.run_batch(torch.from_numpy(np.ascontiguousarray(h_in[4])).cuda())
            assert np.array_equal(d.cpu().numpy().reshape(1, 64, 256), want[4])
        if prev is not None:
            j, tp = prev
            assert np.array_equal(a.wait_batch(tp).reshape(-1, 64, 256), want[j]), rep
        prev = (i, t)
    assert np.array_equal(a.wait_batch(prev[1]).reshape(-1, 64, 256), want[prev[0]])
    big = fc.alloc_host((3, 512, 512))
    big[:] = np.random.default_rng(9).integers(0, 256, big.shape, dtype=np.uint8)
    tb = [a.run_batch_async(big) for _ in range(2)]
    outs = [a.wait_batch(t) for t in tb]
    assert outs[0].shape == (3, 64, 64, 64) and np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], a.run_batch(big))
    # argument errors: unknown ticket, sizes that need the per-layer workspaces, arrays that would need a copy
    with pytest.raises(ValueError):
        a.wait_batch(10 ** 6)
    with pytest.raises(ValueError):
        a.run_batch_async(np.zeros((2, 64, 64), np.uint8))
    with pytest.raises(ValueError):
        a.run_batch_async(np.zeros((2, 128, 256), np.uint8)[:, :, ::2])
    t0 = a.run_batch_async(np.zeros((0, 128, 128), np.uint8))                      # empty batch: a ticket that is complete
    assert a.wait_batch(t0).shape == (0, 64, 16, 16)
    a.close()


def test_misaligned_device_pointers_are_refused(fc, shipped_weights):
    """Device pointers feed TMA descriptors and 128-bit accesses: a misaligned one is a ValueError, not a faulted context."""
    import torch
    a = fc.CNNAccelerator()
    a.load_weights(shipped_weights)
    w, b = inputs.make_fc()
    a.load_classifier(w, b)
    raw = torch.zeros(3 * 16384 + 64, dtype=torch.uint8, device="cuda")
    good = raw[:2 * 16384].view(2, 128, 128)
    bad = raw[4:4 + 2 * 16384].view(2, 128, 128)                        # contiguous, 4 bytes off
    n0 = a.launch_count
    with pytest.raises(ValueError):
        a.run_batch(bad)
    with pytest.raises(ValueError):
        a.run_batch(good, out=torch.zeros(2 * 16384 + 16, dtype=torch.uint8, device="cuda")[8:8 + 2 * 16384].view(2, 64, 16, 16))
    with pytest.raises(ValueError):
        a.infer_batch(bad)
    with pytest.raises(ValueError):
        a.classify_batch(bad.view(2, 64, 256))
    assert a.launch_count == n0
    assert a.run_batch(good).shape == (2, 64, 16, 16)                    # the context is intact
    a.synchronize()
    a.close()


def test_bench_dump_is_the_last_timed_step(port, shipped_weights, tmp_path):
    """bench.py --dump-outputs: features.npy holds what the last of --steps timed steps computed from its seeded batch."""
    import torch
    import bench
    nb, steps = bench.DUMP_IMAGES, 3
    r = subprocess.run([sys.executable, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"),
                        "--steps", str(steps), "--warmup", "0", "--batch", str(nb), "--quick", "--no-stream", "--no-cpu-baseline",
                        "--sustained-s", "0", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    got = np.load(tmp_path / "features.npy")
    assert got.dtype == np.float32 and got.shape == (nb, 64, 16, 16)
    _, batches = bench.synthetic_batches(torch, nb, steps, 0)
    want = oracle.port_infer_batch(port, batches[steps - 1].cpu().numpy(), shipped_weights, bench.SHIFTS)
    assert np.array_equal(got.reshape(nb, 64, 256), want)
