"""Host-side mirror of the reference's engine objects, backed by libcnnacc.so on a B200.

Same call surface as the reference (file:line under /root/reference/software/):

  CNNAccelerator      pynq_inference.py:95-286   load_weights / load_image / set_shifts / start_inference /
                                                 wait_done / read_feature_map / read_layer2_output / write_reg / read_reg
  B200Engine.run      realtime_detect.py:313-363 FPGAEngine.run(gray128) -> (feat (64,256) u8, conv_ms, read_ms)
  load_arm_cnn_lib    realtime_detect.py:369-392 returns a CDLL whose cnn_infer is the drop-in GPU symbol, so the
                                                 reference's ARMEngine.run body works unchanged on it
  classify_vec        realtime_detect.py:68-82   (idx, name, conf, probs)
  bbox_vec            realtime_detect.py:85-116  (x1, y1, x2, y2)

plus the batch entry points the reference has no analogue for: run_batch, classify_batch, infer_batch.
There is no CPU fallback and no simulation mode: without the CUDA library / a B200 the constructor raises.
"""
import contextlib
import ctypes
import os
import time
import weakref

import numpy as np

from . import _lib

# constants with the reference's names (pynq_inference.py:61-89, realtime_detect.py:33-37)
REG_CONTROL, REG_STATUS = 0x00, 0x04
REG_OUTPUT_CH, REG_OUTPUT_ADDR, REG_OUTPUT_DATA, REG_RELU_SHIFTS = 0x20, 0x24, 0x28, 0x28
L2_NUM_CHANNELS, L2_SIZE, L2_CH_OFFSET = 64, 256, 48
SHIFT_L0, SHIFT_L1, SHIFT_L2 = 2, 4, 6
NUM_WEIGHT_BYTES, NUM_IMAGE_BYTES = 23184, 16384
IMG, N_CH, FM, CH_OFF = 128, 64, 256, 48
NAMES = ['airplane', 'cat', 'zebra', 'bus', 'bicycle', 'donut']


def _is_torch_cuda(x):
    return hasattr(x, "data_ptr") and getattr(x, "is_cuda", False)


def _vp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _item_bytes(x):
    """Bytes per item of a batch [N, ...] (also for N == 0)."""
    n = 1
    for d in x.shape[1:]:
        n *= int(d)
    return n if len(x.shape) >= 2 else -1


def register_host(array):
    """Page-lock a host array the caller owns (e.g. an np.memmap of a /dev/shm file shared by the per-GPU processes) so the
    copy engines can write into it directly.  Returns a callable that unregisters it."""
    lib = _lib.load()
    a = np.asarray(array)
    _lib.check(lib.cnnacc_register_host(ctypes.c_void_p(a.ctypes.data), a.nbytes))
    return lambda: lib.cnnacc_unregister_host(ctypes.c_void_p(a.ctypes.data))


def alloc_host(shape, dtype=np.uint8):
    """Page-locked host array the copy engines stream from (the role of pynq.allocate, realtime_detect.py:293,301)."""
    lib = _lib.load()
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    p = ctypes.c_void_p()
    _lib.check(lib.cnnacc_alloc_host(max(nbytes, 1), ctypes.byref(p)))
    buf = (ctypes.c_uint8 * max(nbytes, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    weakref.finalize(buf, lib.cnnacc_free_host, ctypes.c_void_p(p.value))
    return arr


class CNNAccelerator:
    """The accelerator object: load weights.bin, run image(s), read back the 64x16x16 features."""

    def __init__(self, bitstream_path=None, device=0):
        # bitstream_path is accepted for signature compatibility (pynq_inference.py:98) and ignored:
        # the "overlay" is libcnnacc.so.
        self._libc = _lib.load()
        self._h = ctypes.c_void_p()
        _lib.check(self._libc.cnnacc_create(int(device), ctypes.byref(self._h)))
        self.device = int(device)
        self._out_ch = 0
        self._out_addr = 0
        self._n_cls = 0
        self._user_stream = 0
        self._pending = {}
        self._one_ms = (ctypes.byref(ctypes.c_float()), ctypes.byref(ctypes.c_float()))
        self._finalizer = weakref.finalize(self, self._libc.cnnacc_destroy, self._h)

    # -- helpers ---------------------------------------------------------------------------------
    def _check(self, rc):
        _lib.check(rc, self._h)

    def close(self):
        self._finalizer()

    @property
    def launch_count(self):
        return int(self._libc.cnnacc_launch_count(self._h))

    def use_stream(self, cuda_stream_ptr):
        """Launch on a caller-owned CUDA stream (e.g. torch.cuda.current_stream().cuda_stream); 0/None = own stream."""
        self._user_stream = int(cuda_stream_ptr or 0)
        self._check(self._libc.cnnacc_set_stream(self._h, ctypes.c_void_p(self._user_stream)))

    @contextlib.contextmanager
    def _on_stream_of(self, *tensors):
        """Device-pointer calls are asynchronous.  Unless the caller chose a stream with use_stream(), run them on torch's
        CURRENT stream of the tensors' device, so they are ordered after the ops that produced the inputs and before the ops
        that consume the outputs (a `.cpu()` right after the call is then safe)."""
        import torch
        for t in tensors:
            if t is not None and t.get_device() != self.device:
                raise ValueError(f"tensor is on cuda:{t.get_device()}, this accelerator is on cuda:{self.device}")
        if self._user_stream:
            yield
            return
        ptr = torch.cuda.current_stream(self.device).cuda_stream or 1       # 0 = legacy default stream = cudaStreamLegacy (0x1)
        self._check(self._libc.cnnacc_set_stream(self._h, ctypes.c_void_p(ptr)))
        try:
            yield
        finally:
            self._check(self._libc.cnnacc_set_stream(self._h, ctypes.c_void_p(0)))

    def synchronize(self):
        self._check(self._libc.cnnacc_synchronize(self._h))

    def timer_start(self):
        """CUDA-event timer on the handle's stream: pair it with use_stream(...) when timing calls on torch tensors (without
        use_stream those run on torch's current stream, not on the handle's own)."""
        self._check(self._libc.cnnacc_timer_start(self._h))

    def timer_stop(self):
        ms = ctypes.c_float()
        self._check(self._libc.cnnacc_timer_stop(self._h, ctypes.byref(ms)))
        return ms.value

    # -- reference surface: pynq_inference.CNNAccelerator --------------------------------------------
    def load_weights(self, weights_path):
        """pynq_inference.py:186-207.  Accepts a path or a 23184-byte array."""
        weights = np.fromfile(weights_path, dtype=np.uint8) if isinstance(weights_path, (str, os.PathLike)) \
            else np.ascontiguousarray(weights_path, dtype=np.uint8).reshape(-1)
        assert len(weights) == NUM_WEIGHT_BYTES, f"Expected {NUM_WEIGHT_BYTES} weights, got {len(weights)}"
        self._check(self._libc.cnnacc_load_weights(self._h, _vp(weights), weights.size))

    def load_image(self, image):
        """pynq_inference.py:209-224."""
        if isinstance(image, (str, os.PathLike)):
            image = np.fromfile(image, dtype=np.uint8)
        image = np.ascontiguousarray(image, dtype=np.uint8).reshape(-1)
        assert len(image) == NUM_IMAGE_BYTES, f"Expected {NUM_IMAGE_BYTES} pixels, got {len(image)}"
        self._check(self._libc.cnnacc_load_image(self._h, _vp(image), image.size))

    def set_shifts(self, s0=SHIFT_L0, s1=SHIFT_L1, s2=SHIFT_L2):
        """pynq_inference.py:226-229.  Values outside 0..31 raise ValueError instead of being masked."""
        self._check(self._libc.cnnacc_set_shifts(self._h, int(s0), int(s1), int(s2)))

    def get_shifts(self):
        s = (ctypes.c_int * 3)()
        self._check(self._libc.cnnacc_get_shifts(self._h, s))
        return tuple(s)

    def set_accumulator_bits(self, bits=32):
        """32 = arm_cnn.c's int32 accumulator (default, the parity target); 24 = the PL accumulator / the trainer's bit-accurate
        model (rtl/core/accumulator.v:15, training/train_cnn.py:101-116): sums wrap to 24-bit two's complement before the pool."""
        self._check(self._libc.cnnacc_set_accumulator_bits(self._h, int(bits)))

    def get_accumulator_bits(self):
        return int(self._libc.cnnacc_get_accumulator_bits(self._h))

    def probe_int8_peak(self, target_ms=50.0):
        """Dense int8 tensor-core ceiling of this GPU measured now (tcgen05.mma kind::i8 N=256 on every SM) -> (TOP/s, ms)."""
        tops, ms = ctypes.c_double(), ctypes.c_double()
        self._check(self._libc.cnnacc_probe_int8_peak(self._h, float(target_ms), ctypes.byref(tops), ctypes.byref(ms)))
        return tops.value, ms.value

    def start_inference(self):
        """pynq_inference.py:231-234."""
        self._check(self._libc.cnnacc_start(self._h))

    def wait_done(self, timeout=10.0):
        """pynq_inference.py:236-251: returns elapsed seconds, raises TimeoutError."""
        t0 = time.time()
        rc = self._libc.cnnacc_wait(self._h, int(timeout * 1e6))
        if rc == _lib.ERR_TIMEOUT:
            st = self._libc.cnnacc_status(self._h)
            raise TimeoutError(f"Timed out after {timeout}s (busy={st & 1}, done={(st >> 1) & 1}, layer={(st >> 2) & 3})")
        self._check(rc)
        return time.time() - t0

    def read_feature_map(self, channel, num_values):
        """pynq_inference.py:253-265 over the 112-channel feature-BRAM map (0-15 L0, 16-47 L1, 48-111 L2)."""
        values = np.zeros(num_values, dtype=np.uint8)
        self._check(self._libc.cnnacc_read_feature_map(self._h, int(channel), int(num_values), _vp(values)))
        return values

    def read_layer2_output(self):
        """pynq_inference.py:267-286 -> (64, 256) uint8."""
        features = np.zeros((L2_NUM_CHANNELS, L2_SIZE), dtype=np.uint8)
        self._check(self._libc.cnnacc_read_features(self._h, _vp(features), L2_NUM_CHANNELS, L2_CH_OFFSET))
        return features

    def write_reg(self, offset, value):
        """Register-file view used by dump_fpga_features.py:42-88 (writes 0x20/0x24, reads 0x28)."""
        value = int(value)
        if offset == REG_CONTROL:
            if value & 0x1:
                self.start_inference()
        elif offset == REG_OUTPUT_CH:
            self._out_ch = value & 0x7F
        elif offset == REG_OUTPUT_ADDR:
            self._out_addr = value & 0xFFF
        elif offset == REG_RELU_SHIFTS:
            self.set_shifts(value & 0x1F, (value >> 5) & 0x1F, (value >> 10) & 0x1F)

    def read_reg(self, offset):
        if offset == REG_STATUS:
            st = self._libc.cnnacc_status(self._h)
            if st < 0:
                self._check(st)
            return st
        if offset == REG_OUTPUT_DATA:
            depth = 4096 if self._out_ch < 16 else (1024 if self._out_ch < 48 else 256)
            if self._out_ch >= 112 or self._out_addr >= depth:
                return 0
            return int(self.read_feature_map(self._out_ch, self._out_addr + 1)[self._out_addr])
        return 0

    # -- batch entry points -----------------------------------------------------------------------
    def run_batch(self, images, out=None, direct=False):
        """images [N,H,W] u8 (numpy, host) or a torch CUDA tensor -> features [N,64,H/8,W/8] u8 of the same kind."""
        flags = _lib.FLAG_DIRECT if direct else 0
        if _is_torch_cuda(images):
            import torch
            assert images.dtype == torch.uint8 and images.is_contiguous() and images.dim() == 3
            n, H, W = images.shape
            if out is None:
                out = torch.empty((n, 64, H // 8, W // 8), dtype=torch.uint8, device=images.device)
            elif not (_is_torch_cuda(out) and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() == n * 64 * (H // 8) * (W // 8)):
                raise ValueError("out must be a contiguous CUDA uint8 tensor of n*64*(H/8)*(W/8) elements")
            with self._on_stream_of(images, out):
                self._check(self._libc.cnnacc_run_batch(self._h, ctypes.c_void_p(images.data_ptr()), n, H, W,
                                                        ctypes.c_void_p(out.data_ptr()), flags | _lib.FLAG_DEVICE_PTRS))
            return out
        images = np.ascontiguousarray(images, dtype=np.uint8)
        if images.ndim != 3:
            raise ValueError("images must be [N,H,W]")
        n, H, W = images.shape
        if out is None:
            out = np.empty((n, 64, H // 8, W // 8), dtype=np.uint8)
        self._check(self._libc.cnnacc_run_batch(self._h, _vp(images), n, H, W, _vp(out), flags))
        return out

    def run_batch_async(self, images, out=None):
        """Queue one HOST batch (images [N,H,W] u8, C-contiguous, ideally from alloc_host) and return a ticket at once;
        wait_batch(ticket) returns the features.  Batches complete in order and overlap each other's copies (cnnacc.h:
        cnnacc_run_batch_async).  `images` and `out` must not be touched until the ticket was waited for."""
        if not (isinstance(images, np.ndarray) and images.dtype == np.uint8 and images.flags.c_contiguous and images.ndim == 3):
            raise ValueError("images must be a C-contiguous uint8 numpy array [N,H,W] (no implicit copy: the call returns before it is read)")
        n, H, W = images.shape
        if out is None:
            out = alloc_host((n, 64, H // 8, W // 8), np.uint8)
        elif not (isinstance(out, np.ndarray) and out.dtype == np.uint8 and out.flags.c_contiguous and out.size == n * 64 * (H // 8) * (W // 8)):
            raise ValueError("out must be a C-contiguous uint8 numpy array of n*64*(H/8)*(W/8) elements")
        ticket = ctypes.c_int64(-1)
        self._check(self._libc.cnnacc_run_batch_async(self._h, _vp(images), n, H, W, _vp(out), 0, ctypes.byref(ticket)))
        self._pending[ticket.value] = (images, out)          # keep both alive while the copy engines use them
        for t in [t for t in self._pending if t <= ticket.value - 4 * _lib.MAX_PENDING]:
            del self._pending[t]                             # never waited for, and complete for a long time (cnnacc.h)
        return ticket.value

    def wait_batch(self, ticket):
        """Block until the batch behind `ticket` is complete -> its features array."""
        self._check(self._libc.cnnacc_wait_batch(self._h, int(ticket)))
        return self._pending.pop(ticket, (None, None))[1]

    def load_classifier(self, fc_w, fc_b):
        fc_w = np.ascontiguousarray(fc_w, dtype=np.float32)
        fc_b = np.ascontiguousarray(fc_b, dtype=np.float32)
        if fc_w.ndim != 2 or fc_w.shape[1] != 1024 or fc_b.shape != (fc_w.shape[0],):
            raise ValueError(f"classifier must be (n_cls,1024)+(n_cls,), got {fc_w.shape} {fc_b.shape}")
        self._check(self._libc.cnnacc_load_classifier(self._h, _vp(fc_w), _vp(fc_b), fc_w.shape[0]))
        self._n_cls = fc_w.shape[0]

    def _predict(self, fn, x, direct=False, bbox="vec", logits=False, two_kernels=False):
        if bbox not in ("vec", "upsampled"):
            raise ValueError("bbox must be 'vec' (realtime_detect.bbox_vec) or 'upsampled' (Classifier.get_cam_bbox)")
        flags = (_lib.FLAG_DIRECT if direct else 0) | (_lib.FLAG_BBOX_UPSAMPLED if bbox == "upsampled" else 0) | \
                (_lib.FLAG_LOGITS if logits else 0) | (_lib.FLAG_TWO_KERNELS if two_kernels else 0)
        if self._n_cls == 0:
            raise RuntimeError("classifier not loaded")
        if _is_torch_cuda(x):
            import torch
            # the kernels read each item through 128-bit loads / a TMA box: shape, dtype and layout must be exact
            if x.dtype != torch.uint8 or not x.is_contiguous() or _item_bytes(x) != 16384:
                raise ValueError("expected a contiguous CUDA uint8 tensor of [N,128,128] images or [N,64,256] features")
            n = x.shape[0]
            probs = torch.empty((n, self._n_cls), dtype=torch.float32, device=x.device)
            cls = torch.empty((n,), dtype=torch.int32, device=x.device)
            bbox = torch.empty((n, 4), dtype=torch.int32, device=x.device)
            with self._on_stream_of(x):
                self._check(fn(self._h, ctypes.c_void_p(x.data_ptr()), n, ctypes.c_void_p(probs.data_ptr()),
                               ctypes.c_void_p(cls.data_ptr()), ctypes.c_void_p(bbox.data_ptr()),
                               flags | _lib.FLAG_DEVICE_PTRS))
            return cls, probs, bbox
        x = np.ascontiguousarray(x, dtype=np.uint8)
        if _item_bytes(x) != 16384:
            raise ValueError("expected [N,128,128] images or [N,64,256] features")
        n = x.shape[0]
        probs = np.empty((n, self._n_cls), dtype=np.float32)
        cls = np.empty((n,), dtype=np.int32)
        bbox = np.empty((n, 4), dtype=np.int32)
        self._check(fn(self._h, _vp(x), n, _vp(probs), _vp(cls), _vp(bbox), flags))
        return cls, probs, bbox

    def classify_batch(self, features, bbox="vec", logits=False):
        """features [N,64,256] (or [N,64,16,16]) u8 -> (cls [N] i32, probs [N,n_cls] f32, bbox [N,4] i32).
        bbox='vec': realtime_detect.bbox_vec; bbox='upsampled': pynq_inference.Classifier.get_cam_bbox.
        logits=True: the second element holds the raw logits W.pooled + b (realtime_detect.py:79) instead of the softmax."""
        return self._predict(self._libc.cnnacc_classify_batch, features, bbox=bbox, logits=logits)

    def pool_features(self, features):
        """features [N,64,256] u8 -> [N,1024] f32 spatial-bin pooled, /255 (retrain_classifier.py:188-205): the trainer's input."""
        x = np.ascontiguousarray(features, dtype=np.uint8)
        if _item_bytes(x) != 16384:
            raise ValueError("expected [N,64,256] features")
        n = x.shape[0]
        out = np.empty((n, 1024), dtype=np.float32)
        self._check(self._libc.cnnacc_pool_features(self._h, _vp(x), n, _vp(out), 0))
        return out

    def cam_bbox_batch(self, features, cls, return_cam=False):
        """Classifier.get_cam_bbox (pynq_inference.py:349-408) for given classes: features [N,64,256] u8 + cls [N] i32
        -> bbox [N,4] i32 (x1,y1,x2,y2), and with return_cam the upsampled maps [N,128,128] u8 (cam_full = maps/255)."""
        if self._n_cls == 0:
            raise RuntimeError("classifier not loaded")
        x = np.ascontiguousarray(features, dtype=np.uint8)
        cls = np.ascontiguousarray(cls, dtype=np.int32)
        n = x.shape[0] if x.ndim else -1
        if _item_bytes(x) != 16384 or cls.shape != (n,):
            raise ValueError("expected [N,64,256] features and [N] classes")
        bbox = np.empty((n, 4), dtype=np.int32)
        cam = np.empty((n, 128, 128), dtype=np.uint8) if return_cam else None
        self._check(self._libc.cnnacc_cam_bbox_batch(self._h, _vp(x), n, _vp(cls), _vp(bbox), _vp(cam) if return_cam else None, 0))
        return (bbox, cam) if return_cam else bbox

    def bbox_batch(self, features, cls):
        """bbox_vec for given classes: features [N,64,256] u8 + cls [N] i32 -> bbox [N,4] i32 (host arrays)."""
        if self._n_cls == 0:
            raise RuntimeError("classifier not loaded")
        x = np.ascontiguousarray(features, dtype=np.uint8)
        cls = np.ascontiguousarray(cls, dtype=np.int32)
        n = x.shape[0] if x.ndim else -1
        if _item_bytes(x) != 16384 or cls.shape != (n,):
            raise ValueError("expected [N,64,256] features and [N] classes")
        bbox = np.empty((n, 4), dtype=np.int32)
        self._check(self._libc.cnnacc_classify_batch(self._h, _vp(x), n, None, _vp(cls), _vp(bbox), _lib.FLAG_CLS_GIVEN))
        return bbox

    def infer_batch(self, images, direct=False, bbox="vec", logits=False, two_kernels=False):
        """images [N,128,128] u8 -> (cls, probs, bbox).  The classifier / CAM-box tail runs inside the conv-stack kernel on
        the feature map still in shared memory: only 44 B of predictions per image reach HBM.  two_kernels=True is the A/B
        path: features to a workspace, then the features-in tail kernel."""
        return self._predict(self._libc.cnnacc_infer_batch, images, direct, bbox, logits, two_kernels)

    def preprocess(self, frames):
        """realtime_detect.py:582-591 for a batch: frames [N,h,w,3] u8 BGR -> [N,128,128] u8 (centre-crop, BGR2GRAY,
        INTER_AREA), bit-identical to cv2 4.13.  numpy in -> numpy out; torch CUDA tensor in -> torch CUDA tensor out."""
        if _is_torch_cuda(frames):
            import torch
            if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8 or not frames.is_contiguous():
                raise ValueError("expected a contiguous [N,h,w,3] uint8 tensor")
            n, fh, fw = frames.shape[:3]
            out = torch.empty((n, 128, 128), dtype=torch.uint8, device=frames.device)
            with self._on_stream_of(frames):
                self._check(self._libc.cnnacc_preprocess_bgr(self._h, ctypes.c_void_p(frames.data_ptr()), n, fh, fw,
                                                             ctypes.c_void_p(out.data_ptr()), _lib.FLAG_DEVICE_PTRS))
            return out
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        if frames.ndim != 4 or frames.shape[3] != 3:
            raise ValueError("expected [N,h,w,3] BGR frames")
        n, fh, fw = frames.shape[:3]
        out = np.empty((n, 128, 128), dtype=np.uint8)
        self._check(self._libc.cnnacc_preprocess_bgr(self._h, _vp(frames), n, fh, fw, _vp(out), 0))
        return out

    def image_to_gray128(self, images):
        """The arithmetic of pynq_inference.load_image_any (:414-425) for decoded images of one size: [N,H,W] (mode L),
        [N,H,W,3] (RGB) or [N,H,W,4] (RGBA) u8 -> [N,128,128] u8 = PIL convert('L').resize((128,128)), bit-identical to
        Pillow 12.2 (integer luma, default BICUBIC resampler).  numpy in -> numpy out; torch CUDA tensor in -> tensor out."""
        if _is_torch_cuda(images):
            import torch
            if images.dtype != torch.uint8 or not images.is_contiguous() or images.dim() not in (3, 4):
                raise ValueError("expected a contiguous uint8 tensor [N,H,W] or [N,H,W,C]")
            n, H, W = images.shape[:3]
            C = images.shape[3] if images.dim() == 4 else 1
            out = torch.empty((n, 128, 128), dtype=torch.uint8, device=images.device)
            with self._on_stream_of(images):
                self._check(self._libc.cnnacc_image_to_gray128(self._h, ctypes.c_void_p(images.data_ptr()), n, H, W, C,
                                                               ctypes.c_void_p(out.data_ptr()), _lib.FLAG_DEVICE_PTRS))
            return out
        images = np.ascontiguousarray(images, dtype=np.uint8)
        if images.ndim not in (3, 4):
            raise ValueError("expected [N,H,W] or [N,H,W,C] images")
        n, H, W = images.shape[:3]
        C = images.shape[3] if images.ndim == 4 else 1
        out = np.empty((n, 128, 128), dtype=np.uint8)
        self._check(self._libc.cnnacc_image_to_gray128(self._h, _vp(images), n, H, W, C, _vp(out), 0))
        return out

    def detect_frames(self, frames, bbox="vec", return_gray=False):
        """The loop body of realtime_detect.py:582-598 for a batch of camera frames [N,h,w,3] u8 BGR (host array):
        preprocess -> conv stack -> classify -> CAM box on the GPU.  -> (cls, probs, bbox[, gray128])."""
        if bbox not in ("vec", "upsampled"):
            raise ValueError("bbox must be 'vec' or 'upsampled'")
        if self._n_cls == 0:
            raise RuntimeError("classifier not loaded")
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        if frames.ndim != 4 or frames.shape[3] != 3:
            raise ValueError("expected [N,h,w,3] BGR frames")
        n, fh, fw = frames.shape[:3]
        probs = np.empty((n, self._n_cls), dtype=np.float32)
        cls = np.empty((n,), dtype=np.int32)
        box = np.empty((n, 4), dtype=np.int32)
        gray = np.empty((n, 128, 128), dtype=np.uint8) if return_gray else None
        self._check(self._libc.cnnacc_detect_frames(self._h, _vp(frames), n, fh, fw, _vp(gray) if return_gray else None,
                                                    _vp(probs), _vp(cls), _vp(box),
                                                    _lib.FLAG_BBOX_UPSAMPLED if bbox == "upsampled" else 0))
        return (cls, probs, box, gray) if return_gray else (cls, probs, box)

    def detect_regions(self, frames, regions, bbox="vec", logits=False, return_gray=False):
        """detect_frames on caller-chosen square regions: frames [F,h,w,3] u8 BGR (numpy, or a contiguous CUDA uint8 tensor run
        on torch's current stream), regions (R,4) integers (frame, x, y, side) in any order, side 128..8192, inside its
        frame.  Region r's results are those detect_frames gives for frames[f][y:y+side, x:x+side] as a frame of its own; its
        box is in that square's 128x128 coordinates (region_boxes_to_frame maps it to frame pixels).
        -> (cls [R], probs [R,n_cls], bbox [R,4][, gray128 [R,128,128]]) in the order of `regions`, numpy or torch like frames."""
        if bbox not in ("vec", "upsampled"):
            raise ValueError("bbox must be 'vec' or 'upsampled'")
        if self._n_cls == 0:
            raise RuntimeError("classifier not loaded")
        flags = (_lib.FLAG_BBOX_UPSAMPLED if bbox == "upsampled" else 0) | (_lib.FLAG_LOGITS if logits else 0)
        return self._regions(frames, regions, True, return_gray, flags)

    def preprocess_regions(self, frames, regions):
        """preprocess on caller-chosen square regions (see detect_regions) -> gray128 [R,128,128] u8 in the order of `regions`."""
        return self._regions(frames, regions, False, True, 0)[0]

    def _regions(self, frames, regions, detect, want_gray, flags):
        reg = np.asarray(regions)
        if reg.ndim != 2 or reg.shape[1] != 4 or not (reg.size == 0 or np.issubdtype(reg.dtype, np.integer)):
            raise ValueError("regions must be an (R, 4) integer array of (frame, x, y, side)")
        reg = reg.astype(np.int64)
        if reg.size and (reg.min() < -2 ** 31 or reg.max() >= 2 ** 31):
            raise ValueError("region values must fit int32")
        order = np.argsort(reg[:, 0], kind="stable")         # the library takes regions grouped by frame
        shuffled = bool((order != np.arange(len(order))).any())
        reg = np.ascontiguousarray(reg[order], dtype=np.int32)
        n = reg.shape[0]
        nc = self._n_cls
        if _is_torch_cuda(frames):
            import torch
            if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8 or not frames.is_contiguous():
                raise ValueError("expected a contiguous [F,h,w,3] uint8 tensor")
            nf, fh, fw = frames.shape[:3]
            new = lambda shape, dt: torch.empty(shape, dtype=dt, device=frames.device)
            gray = new((n, 128, 128), torch.uint8) if want_gray else None
            outs = (new((n,), torch.int32), new((n, nc), torch.float32), new((n, 4), torch.int32)) if detect else ()
            ptr = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
            with self._on_stream_of(frames):
                self._call_regions(ptr(frames), nf, fh, fw, reg, ptr(gray), [ptr(t) for t in outs], detect,
                                   flags | _lib.FLAG_DEVICE_PTRS)
            res = outs + ((gray,) if want_gray else ())
            if shuffled:
                inv = torch.from_numpy(np.argsort(order)).to(frames.device)
                res = tuple(t[inv] for t in res)
            return res
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        if frames.ndim != 4 or frames.shape[3] != 3:
            raise ValueError("expected [F,h,w,3] BGR frames")
        nf, fh, fw = frames.shape[:3]
        gray = np.empty((n, 128, 128), dtype=np.uint8) if want_gray else None
        outs = (np.empty((n,), np.int32), np.empty((n, nc), np.float32), np.empty((n, 4), np.int32)) if detect else ()
        self._call_regions(_vp(frames), nf, fh, fw, reg, _vp(gray) if want_gray else None, [_vp(a) for a in outs], detect, flags)
        res = outs + ((gray,) if want_gray else ())
        if shuffled:
            inv = np.argsort(order)
            res = tuple(a[inv] for a in res)
        return res

    def _call_regions(self, frames_p, nf, fh, fw, reg, gray_p, outs_p, detect, flags):
        if detect:
            cls_p, probs_p, box_p = outs_p
            self._check(self._libc.cnnacc_detect_regions(self._h, frames_p, nf, fh, fw, _vp(reg), reg.shape[0], gray_p,
                                                         probs_p, cls_p, box_p, flags))
        else:
            self._check(self._libc.cnnacc_preprocess_regions(self._h, frames_p, nf, fh, fw, _vp(reg), reg.shape[0], gray_p, flags))

    def infer_one(self, gray128):
        """One image, lowest latency.  -> (feat (64,256) u8, conv_ms, read_ms)."""
        img = gray128 if (type(gray128) is np.ndarray and gray128.dtype == np.uint8 and gray128.flags.c_contiguous) \
            else np.ascontiguousarray(gray128, dtype=np.uint8)
        assert img.size == NUM_IMAGE_BYTES
        feat = np.empty((N_CH, FM), dtype=np.uint8)
        c, r = self._one_ms                     # two c_floats kept for the life of the object (the latency path is host-bound)
        rc = self._libc.cnnacc_infer_one(self._h, img.ctypes.data, feat.ctypes.data, c, r)
        if rc:
            self._check(rc)
        return feat, c._obj.value, r._obj.value


def _tile_origins(size, side, stride):
    pos = list(range(0, size - side + 1, stride))
    if pos[-1] != size - side:
        pos.append(size - side)                              # one tile flush with the far edge
    return pos


def grid_regions(n_frames, fh, fw, sides, strides):
    """Regions (frame, x, y, side) tiling every frame of a [n_frames, fh, fw, 3] batch at each side: tiles at x = 0, stride,
    2 stride, ... plus one flush with the right edge (x = fw - side) when that position is missing, the same for y.  `sides`
    and `strides` are ints or equal-length sequences.  Frame-major (frame, then side in the given order, then y, then x): the
    order CNNAccelerator.detect_regions hands to the library unchanged.  -> (R, 4) int32."""
    sides = [int(s) for s in np.atleast_1d(sides)]
    strides = [int(s) for s in np.atleast_1d(strides)]
    if len(strides) == 1:
        strides = strides * len(sides)
    if len(strides) != len(sides):
        raise ValueError("sides and strides must have the same length")
    per_frame = []
    for side, stride in zip(sides, strides):
        if side < 1 or side > min(fh, fw) or stride < 1:
            raise ValueError(f"side {side} / stride {stride} does not fit a {fh}x{fw} frame")
        for y in _tile_origins(fh, side, stride):
            for x in _tile_origins(fw, side, stride):
                per_frame.append((x, y, side))
    tiles = np.array(per_frame, dtype=np.int32).reshape(-1, 3)
    out = np.empty((int(n_frames), len(tiles), 4), dtype=np.int32)
    out[:, :, 0] = np.arange(int(n_frames), dtype=np.int32)[:, None]
    out[:, :, 1:] = tiles[None]
    return out.reshape(-1, 4)


def region_boxes_to_frame(regions, bbox):
    """Boxes of detect_regions (x1, y1, x2, y2 on the region's 128x128 grid) in frame pixels: x + b * side / 128 for x1 and
    x2, y + b * side / 128 for y1 and y2, as float64.  This is the one mapping the library documents; it merges nothing
    (no NMS).  -> (R, 4) float64."""
    reg = np.asarray(regions, dtype=np.float64).reshape(-1, 4)
    b = np.asarray(bbox, dtype=np.float64).reshape(-1, 4)
    scale = reg[:, 3:4] / 128.0
    origin = np.concatenate([reg[:, 1:3], reg[:, 1:3]], axis=1)
    return origin + b * scale


class MultiAccelerator:
    """One host batch over several GPUs in one call: a CNNAccelerator per entry of `devices` (None = every visible GPU; a
    device may repeat), run through the cnnacc_*_sharded calls.  Each call cuts the batch into contiguous shards, runs shard
    i on member i's own thread and returns once every prediction / feature is in the host arrays -- the same values, byte for
    byte, as one CNNAccelerator.  Host arrays from alloc_host() are pinned for every GPU; ordinary numpy arrays work, slowly.

    Configuration (load_weights, set_shifts, set_accumulator_bits, load_classifier) goes to every member.  Everything that
    stays per device -- torch tensors, run_batch_async tickets, the register protocol -- is on `.members[i]`."""

    def __init__(self, devices=None):
        if devices is None:
            import torch
            devices = list(range(torch.cuda.device_count())) or [0]     # [0]: no GPU -> CNNAccelerator raises "no CUDA device"
        devices = [int(d) for d in devices]
        if not devices:
            raise ValueError("devices must name at least one GPU")
        self._libc = _lib.load()
        self.members = []
        try:
            for d in devices:
                self.members.append(CNNAccelerator(device=d))
        except BaseException:
            self.close()
            raise
        self._hs = (ctypes.c_void_p * len(self.members))(*[m._h.value for m in self.members])

    def close(self):
        for m in self.members:
            m.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _call(self, fn, *args):
        failed = ctypes.c_int(-1)
        rc = fn(self._hs, len(self.members), *args, ctypes.byref(failed))
        i = failed.value
        if rc != _lib.OK and 0 <= i < len(self.members):
            _lib.check(rc, self.members[i]._h, prefix=f"member {i} (cuda:{self.members[i].device}): ")
        _lib.check(rc)

    @staticmethod
    def _host_only(x):
        if _is_torch_cuda(x):
            raise ValueError("MultiAccelerator takes host arrays; run a CUDA tensor on the accelerator of its GPU, .members[i]")

    # -- configuration, broadcast to every member ----------------------------------------------------------------------
    def load_weights(self, weights_path):
        for m in self.members:
            m.load_weights(weights_path)

    def set_shifts(self, s0=SHIFT_L0, s1=SHIFT_L1, s2=SHIFT_L2):
        for m in self.members:
            m.set_shifts(s0, s1, s2)

    def set_accumulator_bits(self, bits=32):
        for m in self.members:
            m.set_accumulator_bits(bits)

    def load_classifier(self, fc_w, fc_b):
        for m in self.members:
            m.load_classifier(fc_w, fc_b)

    # -- sharded host-batch calls: same arguments and results as CNNAccelerator's for host arrays -----------------------
    def run_batch(self, images, out=None, direct=False):
        """images [N,H,W] u8 (host) -> features [N,64,H/8,W/8] u8."""
        self._host_only(images)
        images = np.ascontiguousarray(images, dtype=np.uint8)
        if images.ndim != 3:
            raise ValueError("images must be [N,H,W]")
        n, H, W = images.shape
        if out is None:
            out = np.empty((n, 64, H // 8, W // 8), dtype=np.uint8)
        elif not (isinstance(out, np.ndarray) and out.dtype == np.uint8 and out.flags.c_contiguous and out.size == n * 64 * (H // 8) * (W // 8)):
            raise ValueError("out must be a C-contiguous uint8 numpy array of n*64*(H/8)*(W/8) elements")
        self._call(self._libc.cnnacc_run_batch_sharded, _vp(images), n, H, W, _vp(out), _lib.FLAG_DIRECT if direct else 0)
        return out

    def _n_cls(self):
        n_cls = self.members[0]._n_cls
        if n_cls == 0:
            raise RuntimeError("classifier not loaded")
        return n_cls

    def infer_batch(self, images, direct=False, bbox="vec", logits=False, two_kernels=False):
        """images [N,128,128] u8 (host) -> (cls [N] i32, probs [N,n_cls] f32, bbox [N,4] i32)."""
        self._host_only(images)
        if bbox not in ("vec", "upsampled"):
            raise ValueError("bbox must be 'vec' (realtime_detect.bbox_vec) or 'upsampled' (Classifier.get_cam_bbox)")
        flags = (_lib.FLAG_DIRECT if direct else 0) | (_lib.FLAG_BBOX_UPSAMPLED if bbox == "upsampled" else 0) | \
                (_lib.FLAG_LOGITS if logits else 0) | (_lib.FLAG_TWO_KERNELS if two_kernels else 0)
        n_cls = self._n_cls()
        x = np.ascontiguousarray(images, dtype=np.uint8)
        if _item_bytes(x) != 16384:
            raise ValueError("expected [N,128,128] images")
        n = x.shape[0]
        probs = np.empty((n, n_cls), dtype=np.float32)
        cls = np.empty((n,), dtype=np.int32)
        box = np.empty((n, 4), dtype=np.int32)
        self._call(self._libc.cnnacc_infer_batch_sharded, _vp(x), n, _vp(probs), _vp(cls), _vp(box), flags)
        return cls, probs, box

    def detect_frames(self, frames, bbox="vec", return_gray=False):
        """Camera frames [N,h,w,3] u8 BGR (host) -> (cls, probs, bbox[, gray128]), as CNNAccelerator.detect_frames."""
        self._host_only(frames)
        if bbox not in ("vec", "upsampled"):
            raise ValueError("bbox must be 'vec' or 'upsampled'")
        n_cls = self._n_cls()
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        if frames.ndim != 4 or frames.shape[3] != 3:
            raise ValueError("expected [N,h,w,3] BGR frames")
        n, fh, fw = frames.shape[:3]
        probs = np.empty((n, n_cls), dtype=np.float32)
        cls = np.empty((n,), dtype=np.int32)
        box = np.empty((n, 4), dtype=np.int32)
        gray = np.empty((n, 128, 128), dtype=np.uint8) if return_gray else None
        self._call(self._libc.cnnacc_detect_frames_sharded, _vp(frames), n, fh, fw, _vp(gray) if return_gray else None,
                   _vp(probs), _vp(cls), _vp(box), _lib.FLAG_BBOX_UPSAMPLED if bbox == "upsampled" else 0)
        return (cls, probs, box, gray) if return_gray else (cls, probs, box)


class B200Engine:
    """FPGAEngine's surface (realtime_detect.py:246-363): run(gray128) -> (feat, conv_ms, read_ms)."""

    def __init__(self, weights=None, shifts=(SHIFT_L0, SHIFT_L1, SHIFT_L2), device=0, clib=None):
        self.acc = CNNAccelerator(device=device)
        if weights is not None:
            self.acc.load_weights(weights)
        self.acc.set_shifts(*shifts)

    def run(self, gray128):
        feat, conv_ms, read_ms = self.acc.infer_one(np.asarray(gray128).flatten().astype(np.uint8))
        return feat.copy(), conv_ms, read_ms


def load_arm_cnn_lib():
    """realtime_detect.py:369-392: a CDLL exposing cnn_infer with argtypes=[c_void_p]*4 -- here the GPU symbol."""
    lib = ctypes.CDLL(_lib.LIB_PATH)
    lib.cnn_infer.argtypes = [ctypes.c_void_p] * 4
    lib.cnn_infer.restype = ctypes.c_int
    return lib


class ARMEngine:
    """realtime_detect.py:398-436 with the C library swapped for libcnnacc.so; run() body follows the reference."""

    def __init__(self, weights_bin, shifts=(SHIFT_L0, SHIFT_L1, SHIFT_L2)):
        self.wt = np.fromfile(weights_bin, dtype=np.uint8) if isinstance(weights_bin, (str, os.PathLike)) \
            else np.ascontiguousarray(weights_bin, dtype=np.uint8)
        self.shifts_arr = np.array(shifts, dtype=np.int32)
        self.output_buf = np.zeros(N_CH * FM, dtype=np.uint8)
        self.clib = load_arm_cnn_lib()

    def run(self, gray128):
        img = np.asarray(gray128).flatten().astype(np.uint8)
        t0 = time.time()
        rc = self.clib.cnn_infer(img.ctypes.data_as(ctypes.c_void_p), self.wt.ctypes.data_as(ctypes.c_void_p),
                                 self.shifts_arr.ctypes.data_as(ctypes.c_void_p),
                                 self.output_buf.ctypes.data_as(ctypes.c_void_p))
        if rc != 0:
            raise RuntimeError(f"cnn_infer returned {rc}")
        conv_ms = (time.time() - t0) * 1000
        return self.output_buf.reshape(N_CH, FM).copy(), conv_ms, 0.0


class Classifier:
    """pynq_inference.py:292-408 on the GPU: classify((64,256) u8) -> (class_index, class_name, confidence, probabilities)
    and get_cam_bbox(features, class_idx) -> (cam_full, (x1, y1, x2, y2)).

    The reference takes the exact-integer bin mean and then divides by 255; the tail kernel computes S/4080 in one
    rounding, which is the same fp32 value.  Weights must be (num_classes, 1024) -- the (6,64) GAP file the reference
    ships does not fit its own classify() either (SURVEY.md 2.4)."""

    def __init__(self, fc_weight_path, fc_bias_path, classes_path=None, device=0):
        import json
        load = lambda x: np.load(x) if isinstance(x, (str, os.PathLike)) else np.asarray(x)
        self.weight = np.ascontiguousarray(load(fc_weight_path), dtype=np.float32)
        self.bias = np.ascontiguousarray(load(fc_bias_path), dtype=np.float32)
        self.num_classes = self.weight.shape[0]
        self.class_names = None
        if classes_path and os.path.exists(classes_path):
            with open(classes_path) as f:
                self.class_names = json.load(f)
        self._acc = CNNAccelerator(device=device)
        self._acc.load_classifier(self.weight, self.bias)     # ValueError unless (n_cls, 1024) + (n_cls,)

    def classify(self, features):
        cls, probs, _ = self._acc.classify_batch(np.asarray(features, dtype=np.uint8).reshape(1, 64, 256))
        idx = int(cls[0])
        name = self.class_names[idx] if self.class_names else str(idx)
        return idx, name, float(probs[0, idx]), probs[0]

    def get_cam_bbox(self, features, class_idx, img_size=128):
        """pynq_inference.py:349-408 -> (cam_full (128,128) f32 in 0..1, (x1, y1, x2, y2))."""
        if img_size != 128:
            raise ValueError("img_size is 128 (IMG_SIZE, pynq_inference.py:72)")
        bbox, cam = self._acc.cam_bbox_batch(np.asarray(features, dtype=np.uint8).reshape(1, 64, 256),
                                             np.array([class_idx], dtype=np.int32), return_cam=True)
        return cam[0].astype(np.float32) / 255.0, tuple(int(v) for v in bbox[0])


def load_features(path):
    """Read a feature dump written by dump_features or by the reference's dumpers (retrain_classifier.py:155-158):
    -> (features (N,64,256) u8, labels (N,), names, shifts or None)."""
    data = np.load(path, allow_pickle=False)
    return (data["features"], data["labels"], list(data["names"]) if "names" in data else None,
            tuple(int(v) for v in data["shifts"]) if "shifts" in data else None)


def dump_features(acc, images, labels, names, output, shifts=None):
    """The .npz the reference's feature dumpers write (dump_arm_features.py:162-170, dump_fpga_features.py:116-120):
    features (N,64,256) u8, labels, names, shifts.  `images` is [N,128,128] u8; one batched call instead of a loop."""
    images = np.ascontiguousarray(images, dtype=np.uint8)
    if shifts is not None:
        acc.set_shifts(*shifts)
    feats = acc.run_batch(images).reshape(len(images), N_CH, FM)
    np.savez(output, features=feats, labels=np.array(labels), names=list(names), shifts=np.array(acc.get_shifts()))
    return feats


_tail_acc = {}


def _tail_accelerator(fc_w, fc_b, device=0):
    key = (device, fc_w.shape, fc_w.tobytes(), fc_b.tobytes())
    acc = _tail_acc.get("acc")
    if acc is None:
        acc = _tail_acc["acc"] = CNNAccelerator(device=device)
    if _tail_acc.get("key") != key:
        acc.load_classifier(fc_w, fc_b)
        _tail_acc["key"] = key
    return acc


def classify_vec(feat_flat, fc_w, fc_b, names=NAMES):
    """realtime_detect.py:68-82 on the GPU: (64,256) u8 -> (idx, name, conf, probs)."""
    fc_w = np.ascontiguousarray(fc_w, dtype=np.float32)
    fc_b = np.ascontiguousarray(fc_b, dtype=np.float32)
    acc = _tail_accelerator(fc_w, fc_b)
    cls, probs, _ = acc.classify_batch(np.asarray(feat_flat, dtype=np.uint8).reshape(1, 64, 256))
    i = int(cls[0])
    return i, names[i], float(probs[0, i]), probs[0]


def bbox_vec(feat_flat, cls_idx, fc_w, fc_b=None):
    """realtime_detect.py:85-116 on the GPU: bbox of the CAM of class cls_idx."""
    fc_w = np.ascontiguousarray(fc_w, dtype=np.float32)
    fc_b = np.zeros(fc_w.shape[0], np.float32) if fc_b is None else np.ascontiguousarray(fc_b, dtype=np.float32)
    acc = _tail_accelerator(fc_w, fc_b)
    feats = np.ascontiguousarray(feat_flat, dtype=np.uint8).reshape(1, 64, 256)
    bbox = acc.bbox_batch(feats, np.array([cls_idx], dtype=np.int32))
    return tuple(int(v) for v in bbox[0])


_loader_acc = {}


def load_image_any(image_path, acc=None):
    """pynq_inference.load_image_any (:414-425): `.bin` -> the 16384 raw bytes; any other format -> decoded by PIL on the host
    (file parsing stays there), then convert('L') + resize((128,128)) on the GPU, bit-identical to Pillow.  -> (16384,) u8.
    Modes other than L / RGB / RGBA (palette, CMYK, 16-bit ...) are first converted to 'L' by PIL itself."""
    ext = os.path.splitext(image_path)[1].lower()
    if ext == '.bin':
        image = np.fromfile(image_path, dtype=np.uint8)
        if len(image) != 128 * 128:
            raise ValueError(f"Expected 16384 bytes, got {len(image)}")
        return image
    from PIL import Image
    img = Image.open(image_path)
    if img.mode not in ("L", "RGB", "RGBA"):
        img = img.convert("L")
    arr = np.asarray(img, dtype=np.uint8)
    if acc is None:
        acc = _loader_acc.get("acc")
        if acc is None:
            acc = _loader_acc["acc"] = CNNAccelerator()
    return acc.image_to_gray128(arr[None]).reshape(-1)


def train_linear_classifier(features, labels, num_classes, lr=0.01, epochs=1000, val_split=0.2, verbose=True, device=0):
    """retrain_classifier.train_linear_classifier (:24-124) with the arithmetic on the GPU: softmax cross-entropy with
    class-balanced sample weights and L2 regularisation, SGD with momentum 0.9, learning rate halved every 300 epochs, the
    weights with the best validation accuracy (checked at epoch 1 and every 100) returned as (W (C,D), b (C,)).

    `features` is (N, D) float32 -- the pooled (N,1024) vectors of CNNAccelerator.pool_features -- `labels` (N,) int.  The
    shuffle / split / initialisation use numpy's RandomState(42) exactly as the reference does, so both start from the same
    point; every step afterwards is the same fp32 operation in the same order (torch on CUDA instead of numpy), so the result
    differs only by summation order inside the matrix products."""
    import torch
    dev = torch.device("cuda", device)
    features = np.ascontiguousarray(features, dtype=np.float32)
    labels = np.asarray(labels)
    N, D = features.shape
    rng = np.random.RandomState(42)
    indices = rng.permutation(N)
    n_val = max(1, int(N * val_split))
    val_idx, train_idx = indices[:n_val], indices[n_val:]
    y_train_np, y_val_np = labels[train_idx], labels[val_idx]
    class_counts = np.bincount(y_train_np, minlength=num_classes).astype(np.float32)
    class_counts = np.maximum(class_counts, 1)
    class_weights = (1.0 / class_counts)
    class_weights = class_weights / class_weights.sum() * num_classes
    W0 = rng.randn(D, num_classes).astype(np.float32) * 0.01
    hi = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False                 # plain fp32 products, as numpy
    try:
        X_train = torch.from_numpy(features[train_idx]).to(dev)
        X_val = torch.from_numpy(features[val_idx]).to(dev)
        y_train = torch.from_numpy(y_train_np.astype(np.int64)).to(dev)
        y_val = torch.from_numpy(y_val_np.astype(np.int64)).to(dev)
        sample_weights = torch.from_numpy(class_weights.astype(np.float32)).to(dev)[y_train]
        W = torch.from_numpy(W0).to(dev)
        b = torch.zeros(num_classes, dtype=torch.float32, device=dev)
        vW, vb = torch.zeros_like(W), torch.zeros_like(b)
        momentum, reg_lambda = 0.9, 0.001
        N_t = y_train.numel()
        rows = torch.arange(N_t, device=dev)
        best_val_acc, best_W, best_b = 0, W.clone(), b.clone()
        for epoch in range(epochs):
            logits = X_train @ W + b
            logits = logits - logits.max(dim=1, keepdim=True).values
            exp_logits = torch.exp(logits)
            probs = exp_logits / exp_logits.sum(dim=1, keepdim=True)
            want_loss = verbose and ((epoch + 1) % 100 == 0 or epoch == 0)
            if want_loss:
                loss = (-(torch.log(probs[rows, y_train] + 1e-10)) * sample_weights).mean() + 0.5 * reg_lambda * (W * W).sum()
            dlogits = probs.clone()
            dlogits[rows, y_train] -= 1
            dlogits *= sample_weights[:, None]
            dlogits /= N_t
            dW = X_train.T @ dlogits + reg_lambda * W
            db = dlogits.sum(dim=0)
            vW = momentum * vW - lr * dW
            vb = momentum * vb - lr * db
            W += vW
            b += vb
            if (epoch + 1) % 100 == 0 or epoch == 0:
                train_acc = float(((X_train @ W + b).argmax(dim=1) == y_train).float().mean()) * 100
                val_acc = float(((X_val @ W + b).argmax(dim=1) == y_val).float().mean()) * 100
                if val_acc > best_val_acc:
                    best_val_acc, best_W, best_b = val_acc, W.clone(), b.clone()
                if verbose:
                    print(f"  Epoch {epoch+1:4d}: loss={float(loss):.4f} train={train_acc:.1f}% val={val_acc:.1f}%")
            if (epoch + 1) % 300 == 0:
                lr *= 0.5
        return best_W.T.contiguous().cpu().numpy(), best_b.cpu().numpy()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = hi
